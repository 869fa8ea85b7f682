/*
 * a1mpc.h -- C ABI of the B200-native batched convex-MPC QP engine.
 *
 * Drop-in boundary for the hot path of ShuoYangRobotics/A1-QP-MPC-Controller:
 *   ConvexMpc            (src/a1_cpp/src/ConvexMpc.h:22-94,  ConvexMpc.cpp:7-260)
 *   A1RobotControl::compute_grf, MPC branch (src/a1_cpp/src/A1RobotControl.cpp:446-562)
 *   A1RobotControl::compute_grf, QP  branch (src/a1_cpp/src/A1RobotControl.cpp:377-445)
 *   OsqpEigen::Solver set-up / solve / getSolution call sites
 *                        (A1RobotControl.cpp:416-439, 522-555; test/test_mpc.cpp:131-151)
 *
 * Plain C, no Eigen / STL / torch types.  Every function returns 0 on success and a negative
 * A1MPC_E* code on failure; a1mpc_last_error() gives the message of the calling thread's last
 * failure.  A handle owns one CUDA device + one stream + scratch; it is NOT thread-safe,
 * distinct handles are independent.  There is no CPU fallback: without a usable CUDA device
 * a1mpc_create() fails with A1MPC_ENODEVICE.
 *
 * Batch layout: every per-QP field is batch-major SoA ("field-major, QP index fastest"):
 * element (field f, QP b) of an array documented as [F][B] lives at  base[f * ld + b]  where
 * ld is the `ld` member of the struct (ld >= B; ld == B for a dense batch).  This is what makes
 * a warp's loads coalesced on the device.
 */
#ifndef A1MPC_H_
#define A1MPC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define A1MPC_VERSION 100

/* error codes */
#define A1MPC_OK          0
#define A1MPC_EINVAL     -1   /* bad argument / unsupported configuration            */
#define A1MPC_ENODEVICE  -2   /* no usable CUDA device (there is no CPU fallback)    */
#define A1MPC_ECUDA      -3   /* CUDA runtime error, see a1mpc_last_error()          */
#define A1MPC_ENOMEM     -4
#define A1MPC_ENCCL      -5   /* NCCL not loadable / NCCL error                      */

/* per-QP status written by the solve kernels */
#define A1MPC_STATUS_OPTIMAL     0  /* KKT certificate verified in-kernel (exact active set)  */
#define A1MPC_STATUS_IPM_ONLY    1  /* interior-point iterate returned, finisher not verified */
#define A1MPC_STATUS_MAXITER     2  /* iteration cap hit before the IPM tolerance             */
#define A1MPC_STATUS_NUMERICAL   3  /* non-positive pivot / NaN in the inputs                 */
#define A1MPC_STATUS_NO_CONTACT  4  /* no stance foot: all forces are zero by the constraints */

#define A1MPC_MAX_HORIZON 20

typedef struct a1mpc_handle a1mpc_handle;

/* Batch-uniform configuration; mirrors the constants of the reference.
 *   horizon          PLAN_HORIZON                      (A1Params.h:26)            10 | 20
 *   dt               mpc_dt                            (A1RobotControl.cpp:462)
 *   mu,fz_min,fz_max friction pyramid and fz bounds    (ConvexMpc.cpp:8, 223-224)
 *   mass, inertia    robot_mass, a1_trunk_inertia      (A1CtrlStates.h:40-43), row-major
 *   q[13], r[12]     q_weights, r_weights (un-doubled; the engine applies the factor 2 of
 *                    ConvexMpc.cpp:20,41)
 *   max_iter, tol    solver controls; 0 selects the defaults (40, 1e-9 switch-over mu)
 *   precision        64: every array of the boundary is fp64 (the reference's arithmetic type).
 *                    32: BASELINE config 3's "fp32" -- the floating-point arrays of the HOT-PATH boundary (a1mpc_solve_batch,
 *                        a1mpc_solve_batch_warm, a1mpc_solve_batch_ext, a1mpc_solve_batch_ext_warm: x0, rot, foot, ref, normals
 *                        in; f_body, u_full out) hold float instead of double, 224 instead of 440 bytes per QP; they are
 *                        declared `double*` below and
 *                        reinterpreted.  The arithmetic in between stays fp64 with the in-kernel KKT certificate: the reduced
 *                        systems have condition numbers of 1e5 (N=10) .. 1e6 (N=20), an fp32 factorisation cannot certify
 *                        1e-4 N, and the only fp32-input tensor-core MMA (tf32, 10-bit mantissa) breaks down on 85 % of the
 *                        QPs (profiles/r01_notes.md).  Accuracy contract: the returned forces are the exact optimum of the QP
 *                        posed by the fp32-rounded inputs, rounded to fp32 -- |f - f*(rounded inputs)| <= 1e-4 N + 1 fp32 ulp.
 *                        The parity / neighbouring entry points (build_qp, qp_mats, solve_dense, grf_qp, torques, plan,
 *                        kinematics, EKF) are fp64 whatever this field says.
 */
typedef struct a1mpc_config {
  int    horizon;
  int    precision;      /* 64 | 32 (fp32 arrays at the hot-path boundary, see above)  */
  double dt;
  double mu, fz_min, fz_max;
  double mass;
  double inertia[9];
  double q[13];
  double r[12];
  int    max_iter;
  double tol;
} a1mpc_config;

/* Fills cfg with the reference launch defaults (config/gazebo_a1_mpc.yaml:6-72,
 * a1_ctrl.launch:2-3): N=10, dt=0.0025, mu=0.3, fz in [0,180], mass 12, gazebo weights. */
void a1mpc_default_config(a1mpc_config* cfg);

/* Inputs of A1RobotControl::compute_grf's MPC branch, i.e. the A1CtrlStates fields it reads
 * (A1RobotControl.cpp:452-488, 498-503; A1CtrlStates.h:347-413).  Pointers are ALL host or ALL
 * device (detected with cudaPointerGetAttributes).
 *   x0      [12][B]  root_euler(3), root_pos(3), root_ang_vel(3), root_lin_vel(3)  (world)
 *   rot     [9][B]   root_rot_mat, row-major
 *   foot    [12][B]  foot_pos_abs, leg-major: FL(x,y,z), FR, RL, RR  (A1CtrlStates.h:399)
 *   ref     [9][B]   root_euler_d[0], root_euler_d[1], root_ang_vel_d(3), root_lin_vel_d(3, body),
 *                    root_pos_d[2]
 *   contact [B]      bit i set = state.contacts[i]   (leg order FL,FR,RL,RR)
 */
typedef struct a1mpc_inputs {
  const double*   x0;
  const double*   rot;
  const double*   foot;
  const double*   ref;
  const uint32_t* contact;
  size_t          ld;
} a1mpc_inputs;

/* Outputs.  f_body is what compute_grf returns (A1RobotControl.cpp:555-563): R^T * u[3i:3i+3],
 * first horizon step, leg-major.  status is mandatory; iters and u_full may be NULL.
 *   f_body [12][B]   status [B]   iters [B] (IPM iterations + 100*finisher rounds)
 *   u_full [12*N][B] world-frame solution over the whole horizon (OsqpEigen getSolution()) */
typedef struct a1mpc_outputs {
  double*  f_body;
  int32_t* status;
  int32_t* iters;
  double*  u_full;
  size_t   ld;
} a1mpc_outputs;

/* ---- life cycle --------------------------------------------------------------------------- */
int  a1mpc_create(a1mpc_handle** out, const a1mpc_config* cfg, int device);
int  a1mpc_destroy(a1mpc_handle* h);
const char* a1mpc_last_error(void);
int  a1mpc_device_count(void);

/* ---- the hot path: replaces compute_grf's MPC branch for B robots -------------------------- */
/* One call = build (linearise, condense, Hessian, gradient) + QP solve + force extraction for
 * every QP of the batch.  Host pointers: cudaMemcpy2DAsync straight from / to the caller's arrays (pinned memory from
 * a1mpc_host_alloc makes them truly asynchronous DMA; pageable memory works and is staged by the driver), solve, D2H,
 * then one stream synchronise: the call is synchronous.  Device pointers: enqueued on the handle's stream, asynchronous
 * (use a1mpc_sync).  ALL arrays of one call must live on the same side (checked: A1MPC_EINVAL on a mix). */
int  a1mpc_solve_batch(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_outputs* out);

/* ---- device-resident warm start across control ticks (SURVEY 8f.3) --------------------------------------------------
 * The reference keeps ONE OsqpEigen::Solver alive and warm-starts every tick from the previous solution
 * (A1RobotControl.h:67, A1RobotControl.cpp:522-538).  Here the state that is worth keeping is the optimal ACTIVE FACE of
 * every robot: a1mpc_solve_batch_warm first runs the exact active-face finisher on the faces stored in `warm` by the
 * previous call (a few reduced factorisations, no interior-point iteration when they still verify -- KKT-certified like
 * every OPTIMAL result) and falls back to the cold path per robot otherwise; it then stores the new faces.  Results are
 * the same optimum either way (the QP is strictly convex).
 *   warm   DEVICE buffer of a1mpc_warm_bytes(h, B) bytes (a1mpc_device_alloc), owned by the caller, one slot per batch
 *          index b; a1mpc_warm_reset (or zero bytes) = no guess.  A robot whose stance feet changed starts cold.
 *   shift  how many horizon steps the stored faces move towards "now" (0: the problem is re-posed relative to the
 *          current state every tick, as compute_grf does; 1: references fixed in absolute time).
 * in / out as in a1mpc_solve_batch (host or device).  Horizon 10 only in this round (A1MPC_EINVAL otherwise). */
size_t a1mpc_warm_bytes(const a1mpc_handle* h, int B);
int  a1mpc_warm_reset(a1mpc_handle* h, void* warm, int B);
int  a1mpc_solve_batch_warm(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_outputs* out, void* warm, int shift);

/* ---- BASELINE config 4: an EXTENSION beyond the reference (which keeps one contact pattern over the horizon,
 * ConvexMpc.cpp:226-245, and world-z friction pyramids) ------------------------------------------------ */
/*   contact_sched [N][B]  contact mask of every horizon step (batch-major, ld of `in`), or NULL = in->contact everywhere
 *   normals       [12][B] terrain normal per foot (world frame, normalised by the engine), or NULL = world z.
 * With normals the friction pyramid and the fz bounds act in each foot's terrain frame; the returned forces are
 * world/body-frame as in a1mpc_solve_batch.  Restrictions: normals need r[3i] == r[3i+1] == r[3i+2] per foot (a rotated
 * diagonal R would not be diagonal), normal z-components must be positive. */
typedef struct a1mpc_inputs_ext {
  const uint32_t* contact_sched;
  const double*   normals;
} a1mpc_inputs_ext;
int  a1mpc_solve_batch_ext(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_inputs_ext* ext, const a1mpc_outputs* out);

/* ---- warm start across control ticks for the extended call ---------------------------------------------------------
 * a1mpc_solve_batch_ext with the device-resident warm start of a1mpc_solve_batch_warm: the same arguments, host / device
 * rules, precision and outputs as a1mpc_solve_batch_ext, and `warm` / `shift` as for a1mpc_solve_batch_warm (same buffer
 * format, a1mpc_warm_bytes / a1mpc_warm_reset; a slot written by either warm call may be read by the other).  Horizons 10
 * and 20.  ext NULL or without schedule and normals: exactly a1mpc_solve_batch_warm.
 * Guesses are per foot-step, not per robot: a change of stance feet does not force a cold start.  Foot-step (s, leg) starts
 * from the face stored at (min(s + shift, N - 1), leg); a foot-step that is not in contact gets the swing face whatever the
 * slot holds.  Only OPTIMAL results store faces; NUMERICAL, NO_CONTACT and uncertified robots store "no guess".
 *   shift  1 is the natural setting with a1mpc_update_plan_batch, which advances every schedule by one horizon step per tick
 *          (step st of the plan is the gait at counter + st * speed); a1mpc_solve_batch_warm's compute_grf-style 0 applies to a
 *          pattern that is re-posed every tick.  Any shift gives the same optimum; a misaligned one only costs hits. */
int  a1mpc_solve_batch_ext_warm(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_inputs_ext* ext, const a1mpc_outputs* out,
                                void* warm, int shift);

/* ---- ConvexMpc members, for parity with the reference class (ConvexMpc.h:87-93) ----------- */
/* Dense QP data exactly as ConvexMpc::calculate_qp_mats leaves it after compute_grf drove it
 * (constant B_d over the horizon, A1RobotControl.cpp:498-514).  QP-major outputs:
 *   H [B][12N][12N] row-major (hessian, densified), g [B][12N] (gradient),
 *   lb, ub [B][20N] (ConvexMpc.cpp:223-245; +-1e30 = OsqpEigen::INFTY).  Any may be NULL. */
int  a1mpc_build_qp_batch(a1mpc_handle* h, int B, const a1mpc_inputs* in,
                          double* H, double* g, double* lb, double* ub);

/* ConvexMpc::calculate_qp_mats for caller-supplied discrete models (the public API allows a
 * different B_d per step: test/test_mpc.cpp:106-122).  QP-major inputs:
 *   A_d [B][13][13] row-major, B_d_list [B][13N][12] row-major (B_mat_d_list),
 *   x0 [B][13] (mpc_states), x_d [B][13N] (mpc_states_d);  outputs as above. */
int  a1mpc_qp_mats_batch(a1mpc_handle* h, int B, const double* A_d, const double* B_d_list,
                         const double* x0, const double* x_d, double* H, double* g);
/* The same call with the intermediate public members of ConvexMpc as well (ConvexMpc.h:77-78, ConvexMpc.cpp:181-202):
 *   A_qp [B][13N][13] (rows 13i.. = A_d^(i+1)),  B_qp [B][13N][12N] (block (i,j) = A_d^(i-j) B_d[j], j <= i, zero above).
 * Any output may be NULL (at least one must not be). */
int  a1mpc_qp_rollout_batch(a1mpc_handle* h, int B, const double* A_d, const double* B_d_list,
                            const double* x0, const double* x_d, double* A_qp, double* B_qp, double* H, double* g);

/* OsqpEigen::Solver replacement for the MPC QP (A1RobotControl.cpp:522-555):
 *   min 1/2 u'Hu + g'u  s.t. the friction pyramid of ConvexMpc.cpp:46-58 with the contact
 *   pattern `contact` (constant over the horizon).  H [B][12N][12N], g [B][12N] QP-major,
 *   u [B][12N] out (getSolution()), status [B]. */
int  a1mpc_solve_dense_batch(a1mpc_handle* h, int B, const double* H, const double* g,
                             const uint32_t* contact, double* u, int32_t* status);

/* ---- compute_grf's QP branch (stance_leg_control_type == 0), A1RobotControl.cpp:377-445 ---- */
/* 12-variable instantaneous GRF QP, batched.  All arrays QP-major:
 *   root_acc [B][6]  desired wrench (A1RobotControl.cpp:379-391, caller-computed PD + gravity)
 *   rot_z [B][9], rot [B][9]  root_rot_mat_z, root_rot_mat (row-major); foot [B][12] leg-major
 *   contact [B];  f_body [B][12] out;  status [B] out.
 * Constants Q=diag(1,1,1,400,400,100), R=1e-3, mu=0.7, F in [0,180] (A1RobotControl.cpp:11-15). */
int  a1mpc_grf_qp_batch(a1mpc_handle* h, int B, const double* root_acc, const double* rot_z,
                        const double* rot, const double* foot, const uint32_t* contact,
                        double* f_body, int32_t* status);

/* ---- the step right after the path (SURVEY 8f.1): A1RobotControl::compute_joint_torques ------------- */
/* A1RobotControl.cpp:289-319, batched, batch-major SoA like a1mpc_solve_batch (ld = B), host or device pointers:
 *   f_grf   [12][B]  foot_forces_grf, leg-major (the f_body output of a1mpc_solve_batch can be passed as is)
 *   f_kin   [12][B]  foot_forces_kin, leg-major (swing-leg PD force, A1RobotControl.cpp:286)
 *   jac     [36][B]  the four 3x3 diagonal blocks of j_foot, leg-major then row-major (A1CtrlStates.h:409)
 *   contact [B]      bit i = contacts[i]
 *   km_foot[3], torques_gravity[12]: batch-uniform (A1CtrlStates.h:122,129), ALWAYS HOST arrays (read by the call itself, also when
 *                    the batch arrays are device pointers)
 *   tau     [12][B]  in/out: stance legs  J^T (-f_grf),  swing legs  J^-1 (km_foot .* f_kin)  (partial-pivot LU),
 *                    + torques_gravity; an entry whose result is NaN keeps its previous value (:314-317). */
int  a1mpc_joint_torques_batch(a1mpc_handle* h, int B, const double* f_grf, const double* f_kin, const double* jac,
                               const uint32_t* contact, const double* km_foot, const double* torques_gravity, double* tau);

/* ---- upstream producers of the path's inputs (SURVEY 8f.4) ------------------------------------------------------ */
/* Leg forward kinematics and Jacobian: A1Kinematics::fk / jac (legKinematics/A1Kinematics.cpp:7-18; bodies :39-131) with the
 * per-tick derived quantities of GazeboA1ROS.cpp:264-279, batched.  Batch-major SoA (ld = B), host or device pointers:
 *   joint_pos [12][B] leg-major (FL, FR, RL, RR) x (hip, thigh, calf); joint_vel [12][B] (NULL: no velocities)
 *   rot [9][B] root_rot_mat row-major (NULL: no *_abs outputs)
 *   rho_opt [12] = 4 legs x (cx, cy, cz) contact offset; rho_fix [20] = 4 legs x (leg_offset_x, leg_offset_y, motor_offset,
 *   upper_leg_length, lower_leg_length) (GazeboA1ROS.cpp:76-97): HOST arrays, batch-uniform
 *   out (any may be NULL): foot_pos_rel [12][B]; jac [36][B] = the four 3x3 blocks of j_foot, leg-major then row-major (the
 *   layout a1mpc_joint_torques_batch takes); foot_vel_rel [12][B] = J dq; foot_pos_abs [12][B] = R foot_pos_rel (the `foot`
 *   input of a1mpc_solve_batch); foot_vel_abs [12][B]. */
int  a1mpc_leg_kinematics_batch(a1mpc_handle* h, int B, const double* joint_pos, const double* joint_vel, const double* rot,
                                const double* rho_opt, const double* rho_fix, double* foot_pos_rel, double* jac, double* foot_vel_rel,
                                double* foot_pos_abs, double* foot_vel_abs);

/* A1BasicEKF (A1BasicEKF.cpp), batched: 18 states (position, velocity, four foot positions), 28 measurements, orientation
 * taken from the IMU.  The filter state lives on the device: a1mpc_ekf_bytes(B) bytes (a1mpc_device_alloc), per robot 342
 * doubles = x[18], P[18][18] row-major.
 *   a1mpc_ekf_init_batch    A1BasicEKF::init_state (:56-68): P = 3 I, x = (0, 0, 0.09, 0, 0, 0, R fk_i + pos)
 *   a1mpc_ekf_update_batch  A1BasicEKF::update_estimation (:70-164) with the constructor's C, Q, R (:7-53; noise constants of
 *                           A1BasicEKF.h:16-21): contact estimate from movement_mode / foot_force, process update, measurement,
 *                           S = C Pbar C' + R, x and P update, position-drift cut (:144-148)
 *   batch-major SoA inputs (ld = B), host or device: movement_mode [B], imu_acc [3][B], imu_ang_vel [3][B], rot [9][B],
 *   foot_pos_rel [12][B], foot_vel_rel [12][B], foot_force [4][B]
 *   out (any may be NULL): root_pos [3][B] (= estimated_root_pos), root_lin_vel [3][B], estimated_contacts [B] (bit i = leg i),
 *   status [B]: 0, or A1MPC_STATUS_NUMERICAL when S is not positive definite / not finite (that robot's state is untouched). */
size_t a1mpc_ekf_bytes(int B);
int  a1mpc_ekf_init_batch(a1mpc_handle* h, int B, void* ekf_state, const double* foot_pos_rel, const double* rot);
int  a1mpc_ekf_update_batch(a1mpc_handle* h, int B, void* ekf_state, double dt, int assume_flat_ground, const uint32_t* movement_mode,
                            const double* imu_acc, const double* imu_ang_vel, const double* rot, const double* foot_pos_rel,
                            const double* foot_vel_rel, const double* foot_force, double* root_pos, double* root_lin_vel,
                            uint32_t* estimated_contacts, int32_t* status);

/* ---- the step right before the path (SURVEY 8f.2): A1RobotControl::update_plan ------------------------ */
/* Gait counters -> planned contacts, and the Raibert foothold targets (A1RobotControl.cpp:148-202), batched; plus what the
 * reference does not do: the planned contact mask of every horizon step (it freezes the current pattern,
 * ConvexMpc.cpp:226-245), in the [N][B] layout a1mpc_solve_batch_ext takes.  Batch-major SoA (ld = B), host or device:
 *   gait_counter [4][B] in/out; gait_counter_speed [4][B]; movement_mode [B] (0 standstill: all feet planned in contact and
 *   the counters reset to the trot offsets 0,120,120,0 -- A1CtrlStates.h:322-326);
 *   lin_vel [3][B] root_lin_vel (world); lin_vel_d [3][B] root_lin_vel_d; rot_z [9][B], rot [9][B], root_pos [3][B];
 *   out: plan_contacts [B]; contact_sched [N][B] (step i = i plan ticks ahead; may be NULL);
 *        foot_pos_target_rel / _abs / _world [12][B] leg-major (any may be NULL). */
typedef struct a1mpc_gait_params {
  double counter_per_gait;      /* 240  (A1CtrlStates.h:23)  */
  double counter_per_swing;     /* 120  (A1CtrlStates.h:24)  */
  double control_dt;            /* MAIN_UPDATE_FREQUENCY / 1000 (A1CtrlStates.h:332) */
  double default_foot_pos[12];  /* 3 x NUM_LEG row-major (A1CtrlStates.h:45-47) */
  double foot_delta_x_limit, foot_delta_y_limit;   /* A1Params.h:44-45 */
  int    horizon;               /* steps of contact_sched */
} a1mpc_gait_params;
int  a1mpc_update_plan_batch(a1mpc_handle* h, int B, const a1mpc_gait_params* gp, double* gait_counter, const double* gait_counter_speed,
                             const uint32_t* movement_mode, const double* lin_vel, const double* lin_vel_d, const double* rot_z,
                             const double* rot, const double* root_pos, uint32_t* plan_contacts, uint32_t* contact_sched,
                             double* foot_pos_target_rel, double* foot_pos_target_abs, double* foot_pos_target_world);

/* ---- device memory, stream and timing helpers (so hosts need no CUDA headers) -------------- */
int  a1mpc_device_alloc(a1mpc_handle* h, size_t bytes, void** ptr);
int  a1mpc_device_free(a1mpc_handle* h, void* ptr);
int  a1mpc_host_alloc(a1mpc_handle* h, size_t bytes, void** ptr);   /* pinned */
int  a1mpc_host_free(a1mpc_handle* h, void* ptr);
int  a1mpc_memcpy_h2d(a1mpc_handle* h, void* dst, const void* src, size_t bytes);  /* async on the stream */
int  a1mpc_memcpy_d2h(a1mpc_handle* h, void* dst, const void* src, size_t bytes);  /* async on the stream */
int  a1mpc_sync(a1mpc_handle* h);
int  a1mpc_event_create(a1mpc_handle* h, void** ev);
int  a1mpc_event_destroy(a1mpc_handle* h, void* ev);
int  a1mpc_event_record(a1mpc_handle* h, void* ev);                  /* on the handle's stream */
int  a1mpc_event_elapsed_ms(a1mpc_handle* h, void* start, void* stop, float* ms); /* syncs on stop */
/* number of kernels this handle has launched since creation (bench.py's gpu_launches) */
int64_t a1mpc_launch_count(const a1mpc_handle* h);
/* measured peak of the fp64 FMA pipe on this device, TFLOP/s (dependent-free DFMA stream) */
int  a1mpc_measure_fp64_peak(a1mpc_handle* h, double* tflops);
/* Per-class kernel timing for roofline reports: between begin and end every a1mpc_solve_batch records a
 * CUDA-event pair around each class kernel ON THE STREAM THAT KERNEL RUNS ON (up to max_calls calls).
 * end() synchronises and returns the summed device time in ms of the kernels for 1,2,3,4 stance feet. */
int  a1mpc_profile_begin(a1mpc_handle* h, int max_calls);
int  a1mpc_profile_end(a1mpc_handle* h, double* ms_per_class4, int* calls);
/* writes one buffer larger than L2 (flushes L2 between timed iterations when asked to) */
int  a1mpc_flush_l2(a1mpc_handle* h);

/* ---- optional final collect across GPUs (SURVEY 8e): all-gather of f_body over NCCL ------- */
/* NCCL is dlopen'ed at first use; without it these return A1MPC_ENCCL and nothing else in the
 * library depends on it.  unique_id is a 128-byte ncclUniqueId produced on rank 0. */
int  a1mpc_nccl_unique_id(void* unique_id128);
int  a1mpc_nccl_init(a1mpc_handle* h, int nranks, int rank, const void* unique_id128);
/* gathers f_local [12][B_local] (device) from every rank into f_all [nranks][12][B_local].  Asynchronous: the collective runs on
 * the handle's collect stream after everything enqueued so far and overlaps later solves; a1mpc_sync and a1mpc_event_record
 * wait for it.  Do not overwrite f_local / read f_all before one of them. */
int  a1mpc_allgather_forces(a1mpc_handle* h, const double* f_local, double* f_all, int B_local);

/* ---- fused final collect (SURVEY 2.3 last row / 8e): the solve kernels store the forces into every GPU's gathered buffer -------
 * One process per GPU.  Each rank allocates its gathered buffer f_all [nranks][B_local][12] (QP-major: the 12 body-frame forces of a
 * robot are contiguous, leg-major -- NOT the batch-major layout of f_body / ncclAllGather) with a1mpc_peer_gather_create, which
 * returns a 64-byte CUDA IPC handle; the ranks exchange the handles (any transport: the caller's MPI / torch.distributed / files)
 * and map each other's buffers with a1mpc_peer_gather_connect.  From then on every a1mpc_solve_batch / _warm call with device
 * pointers and B == B_local ALSO stores the 12 forces of every QP, straight from the solve kernels' epilogue, into block [rank] of
 * every rank's buffer (one contiguous 96-byte peer store per QP and rank over NVLink / NVSwitch -- no collective call, no extra pass
 * over the data) and then
 * publishes the call's sequence number to every rank.  a1mpc_peer_gather_wait enqueues, on the handle's collect stream (forked after
 * everything enqueued so far, so that later solves are not held back by a slower peer; a1mpc_sync and a1mpc_event_record join
 * it, exactly like the NCCL collect), a wait until the forces of this rank's latest call number have arrived from ALL ranks
 * (the ranks must make the same sequence of calls).
 * Semantics: "latest value" -- a rank that runs ahead overwrites its block with its next call's forces; callers that must consume
 * call k everywhere before any rank starts call k+1 add their own barrier.  precision 32: the buffer holds float.
 * The wait itself is a stream memory operation (cuStreamWaitValue64 on this rank's flag array: no SM is occupied); where the driver
 * refuses it, or with A1MPC_PEER_WAIT_KERNEL=1, a one-warp polling kernel with a ~2 s cap is used instead, and a peer that never
 * arrives is then reported by a1mpc_peer_gather_status (0 = fine, r+1 = rank r timed out) instead of hanging the stream.
 * Needs peer access between the GPUs (same NVLink domain) and CUDA IPC between the processes; A1MPC_ECUDA otherwise -- the NCCL
 * all-gather above remains available as the portable path. */
int  a1mpc_peer_gather_create(a1mpc_handle* h, int nranks, int rank, int B_local, void* ipc_handle64);
int  a1mpc_peer_gather_connect(a1mpc_handle* h, const void* all_handles /* nranks x 64 bytes, rank order */);
int  a1mpc_peer_gather_buffer(a1mpc_handle* h, double** f_all);
int  a1mpc_peer_gather_wait(a1mpc_handle* h);
int  a1mpc_peer_gather_status(a1mpc_handle* h, int* timed_out_rank_plus_1);
int  a1mpc_peer_gather_destroy(a1mpc_handle* h);

/* ---- synthetic workload generator (SURVEY 8d), host-side, deterministic ------------------- */
/* Fills host SoA arrays (ld = B) with the trot-gait state distribution of the benchmark.
 * config_id: 2 = trot narrow noise (configs 2,3,5), 4 = wide noise (config 4's state noise).
 * seed = 0xA1C0FFEE + config_id + `stream` (use the rank / batch index as stream). */
int  a1mpc_gen_states(int config_id, uint64_t stream, int B, double* x0, double* rot, double* foot,
                      double* ref, uint32_t* contact);
/* config-4 extras for the same (config_id, stream, B): per-step schedules [N][B] drawn from trot / bound / rotary gallop at
 * a random phase of a 16-step period, and per-foot normals [12][B] = z tilted by N(0,0.2) rad about a random horizontal axis */
int  a1mpc_gen_schedule(int config_id, uint64_t stream, int B, int horizon, uint32_t* contact_sched, double* normals);

#ifdef __cplusplus
}
#endif
#endif /* A1MPC_H_ */
