// a1mpc_internal.h -- host-side glue between the translation units of liba1mpc.so
#pragma once
#include <cuda_runtime.h>
#include "a1mpc_device.cuh"

namespace a1mpc {

struct ClassLaunch {
  int wpc = 1;
  size_t smem = 0;
  int max_ctas = 0;  // resident CTAs on the whole device (persistent grid size)
  bool supported = false;
};

// fused path (a1mpc_solve_n10.cu / a1mpc_solve_n20.cu)
cudaError_t fused_setup_n10(int sm_count, ClassLaunch (&cls)[5]);
cudaError_t fused_setup_n20(int sm_count, ClassLaunch (&cls)[5]);
void fused_launch_n10(int ns, const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out);
void fused_launch_n20(int ns, const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out);
// warm-started variant of the N = 10 classes (a1mpc_solve_batch_warm); set up by fused_setup_n10
void fused_launch_n10_warm(int ns, const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count,
                           const DevOutputs& out, uint32_t* warm, int shift);
// extended path (per-step contact schedules + terrain normals), a1mpc_solve_ext.cu.  `cw` / warm != nullptr: the warm-started
// kernels of a1mpc_solve_batch_ext_warm (their own occupancy, launched with the ClassLaunch that setup filled for them)
cudaError_t ext_setup(int horizon, int sm_count, ClassLaunch& c, ClassLaunch& cw);
void ext_launch(int horizon, const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out,
                uint32_t* warm = nullptr, int shift = 0);
// compacted two-stance-feet-per-step class of the extended path (a1mpc_sched.cuh; N = 10)
cudaError_t sched2_setup(int sm_count, ClassLaunch& c, ClassLaunch& cw);
void sched2_launch(const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out,
                   uint32_t* warm = nullptr, int shift = 0);
cudaError_t build_dense_launch(const DevParams& P, const DevInputs& in, int B, double* H, double* g, double* lb, double* ub, cudaStream_t st);

// QP-major side entry points (a1mpc_dense.cu)
cudaError_t dense_setup(int horizon);
// scratch: (4*B + 8) ints
cudaError_t dense_qp_mats_launch(const DevParams& P, int B, const double* A_d, const double* B_d_list, const double* x0, const double* x_d,
                                 double* H, double* g, double* A_qp, double* B_qp, cudaStream_t st);
// returns cudaErrorInvalidValue for configurations whose factor does not fit (N=20 with >2 stance feet)
cudaError_t dense_solve_launch(const DevParams& P, int sm_count, int B, const double* H, const double* g, const uint32_t* contact, double* u,
                               int32_t* status, int* scratch, cudaStream_t st, int* nlaunch);
cudaError_t grf_qp_launch(int sm_count, int B, const double* root_acc, const double* rot_z, const double* rot, const double* foot,
                          const uint32_t* contact, double* f_body, int32_t* status, int* scratch, cudaStream_t st, int* nlaunch);

}  // namespace a1mpc
