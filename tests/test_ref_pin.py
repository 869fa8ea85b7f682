"""The oracle pinned to the REFERENCE'S OWN compiled code (CPU tests, no GPU).

tests/golden/convexmpc_v1.npz was produced by oracle/_ref/libref_mpc.so: the reference's ConvexMpc.cpp, A1RobotControl.cpp, A1BasicEKF.cpp
and utils/Utils.cpp compiled unmodified against the header stand-ins of oracle/ref_shim/ (tests/golden/make_ref_golden.py).  These tests
hold the oracle restatement (oracle/a1mpc_oracle.cpp) to those vectors -- every row of SURVEY 8(a) that the reference computes itself --
and to what the reference build returned on states of their own (tests/golden/ref_live_v1.npz).
Tolerances: products of ~1e2 terms accumulated in a different order agree to a few ulp: 1e-14 relative (measured <= 2e-15);
bounds, the pyramid matrix and contact plans: exact.
"""
import numpy as np

import a1mpc
from common import load_ref_golden, load_ref_live, ref_cfg_kwargs
from oracle import oracle_py as O

N = 10
IU = np.triu_indices(12 * N)


def _relerr(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def _batch(G, sel):
    return O.Batch(G["mpc_x0"][sel].T, G["mpc_rot"][sel].T, G["mpc_foot"][sel].T, G["mpc_ref"][sel].T, G["mpc_contact"][sel])


def test_oracle_build_matches_reference_golden(built):
    """P0, rows a1-a10: H (full for 9 states, diag + 8-column sketch for all 41), g, lb, ub, the pyramid matrix, x0 / x_d packing"""
    G = load_ref_golden()
    V = G["probe_V"]
    worst = dict(H=0.0, HV=0.0, g=0.0, xd=0.0)
    for w in range(3):
        sel = np.nonzero(G["mpc_weights"] == w)[0]
        cfg = O.make_config(**ref_cfg_kwargs(G, w))
        ob = _batch(G, sel)
        for k, i in enumerate(sel):
            H, g, A, lb, ub = O.build_qp(cfg, ob, k)
            assert np.array_equal(A, G["Ac"]) and np.array_equal(lb, G["mpc_lb"][i]) and np.array_equal(ub, G["mpc_ub"][i])
            if i < G["mpc_Hfull_triu"].shape[0]:
                worst["H"] = max(worst["H"], _relerr(H[IU], G["mpc_Hfull_triu"][i]))
            worst["HV"] = max(worst["HV"], _relerr(H @ V, G["mpc_HV"][i]), _relerr(np.diag(H), G["mpc_Hdiag"][i]))
            worst["g"] = max(worst["g"], _relerr(g, G["mpc_g"][i]))
            ro = O.rollout(cfg, ob, k)
            assert np.array_equal(ro["mpc_states"], G["mpc_mpc_states"][i])
            worst["xd"] = max(worst["xd"], _relerr(ro["mpc_states_d"], G["mpc_mpc_states_d"][i]))
    assert worst["H"] <= 1e-14 and worst["HV"] <= 1e-14 and worst["g"] <= 1e-14 and worst["xd"] <= 1e-15, worst


def test_oracle_rollout_matches_reference_golden(built):
    """rows a3-a6: A_d, B_d, A_qp, B_qp as the reference's ConvexMpc members hold them"""
    G = load_ref_golden()
    for k, i in enumerate(G["roll_idx"]):
        cfg = O.make_config(**ref_cfg_kwargs(G, int(G["mpc_weights"][i])))
        ro = O.rollout(cfg, _batch(G, [i]), 0)
        for name in ("A_d", "B_d_list", "A_qp", "B_qp"):
            assert _relerr(ro[name], G["roll_" + name][k]) <= 1e-14, name
            assert np.array_equal(ro[name] == 0, G["roll_" + name][k] == 0), name   # same sparsity pattern (block lower triangle)


def test_oracle_general_rollout_matches_reference_golden(built):
    """ConvexMpc::calculate_qp_mats with a different B_d every step, driven in the order of test/test_mpc.cpp:106-125"""
    G = load_ref_golden()
    for k in range(G["step_A_d"].shape[0]):
        cfg = O.make_config(**ref_cfg_kwargs(G, int(G["step_weights"][k])))
        H, g = O.qp_mats(cfg, G["step_A_d"][k], G["step_B_d_list"][k], G["step_x0"][k], G["step_x_d"][k])
        assert _relerr(H[IU], G["step_H_triu"][k]) <= 1e-14 and _relerr(g, G["step_g"][k]) <= 1e-14


def test_oracle_forces_match_reference_compute_grf(built):
    """rows a11-a12 end to end: the reference's compute_grf (its QP solved to eps 1e-11 by the OSQP-algorithm restatement) against the
    oracle's exact solve of its own build: <= 1e-5 N (the stored forces carry the ADMM tolerance), P1's gate is 1e-4 N"""
    G = load_ref_golden()
    worst = 0.0
    for w in range(3):
        sel = np.nonzero(G["mpc_weights"] == w)[0]
        cfg = O.make_config(**ref_cfg_kwargs(G, w))
        f, info = O.compute_grf_batch(cfg, _batch(G, sel), O.MODE_EXACT, nthreads=4)
        assert (info[:, 1] == 1).all()
        worst = max(worst, float(np.abs(f.T - G["mpc_f_body"][sel]).max()))
        # velocity command in the world frame, a state write-back of compute_grf (A1RobotControl.cpp:470)
        for k, i in enumerate(sel):
            Rm = G["mpc_rot"][i].reshape(3, 3)
            assert np.abs(Rm @ G["mpc_ref"][i][5:8] - G["mpc_vd_world"][i]).max() <= 1e-15
    assert worst <= 1e-5, worst
    # the reference's only standalone driver: known answer of test/test_mpc.cpp (printed there, never checked)
    assert abs(G["mpc_f_body"][0][2] - 42.7901021118) < 1e-6 and abs(G["mpc_f_body"][0][1] + 12.8370306335) < 1e-6


def _root_acc(x0, rot, ref12, gains, mass):
    """A1RobotControl.cpp:325-333, 380-392 (the PD law in front of the single-step QP)"""
    e, p, w, v = x0[0:3], x0[3:6], x0[6:9], x0[9:12]
    Rm = rot.reshape(3, 3)
    ed, pd, vd, wd = ref12[0:3], ref12[3:6], ref12[6:9], ref12[9:12]
    err = ed - e
    if err[2] > 3.1415926 * 1.5:
        err[2] = ed[2] - 3.1415926 * 2 - e[2]
    elif err[2] < -3.1415926 * 1.5:
        err[2] = ed[2] + 3.1415926 * 2 - e[2]
    kpl, kdl, kpa, kda = gains[0:3], gains[3:6], gains[6:9], gains[9:12]
    acc = np.zeros(6)
    acc[0:3] = kpl * (pd - p) + Rm @ (kdl * (vd - Rm.T @ v))
    acc[3:6] = kpa * err + kda * (wd - Rm.T @ w)
    acc[2] += mass * 9.8
    return acc


def test_oracle_grf_qp_matches_reference_golden(built):
    """BASELINE config 1: the 12-variable QP exactly as compute_grf's QP branch hands it to OsqpEigen (A1RobotControl.cpp:377-445)"""
    G = load_ref_golden()
    mass = float(G["w0"][0])
    for k in range(G["grf_P"].shape[0]):
        acc = _root_acc(G["grf_x0"][k].copy(), G["grf_rot"][k], G["grf_ref12"][k], G["grf_gains"][k], mass)
        rz = G["grf_rot_z"][k].reshape(3, 3)
        foot = G["grf_foot"][k].reshape(4, 3)
        Minv = np.zeros((6, 12))
        for i in range(4):
            r = foot[i]
            S = np.array([[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]])
            Minv[0:3, 3 * i:3 * i + 3] = np.eye(3)
            Minv[3:6, 3 * i:3 * i + 3] = rz.T @ S
        Q = np.diag([1.0, 1.0, 1.0, 400.0, 400.0, 100.0])
        assert _relerr(Minv.T @ Q @ Minv + 1e-3 * np.eye(12), G["grf_P"][k]) <= 1e-14
        assert _relerr(-Minv.T @ Q @ acc, G["grf_q"][k]) <= 1e-13
        f, info = O.grf_qp_single(acc, G["grf_rot_z"][k], G["grf_rot"][k], G["grf_foot"][k], int(G["grf_contact"][k]), O.MODE_EXACT)
        # the stored forces carry the ADMM tolerance of the stand-in solver along this QP's flat directions (measured 2e-5 N)
        assert info[1] == 1 and np.abs(f - G["grf_f_body"][k]).max() <= 1e-4


def test_oracle_joint_torques_update_plan_match_reference_golden(built):
    """SURVEY 8f.1, 8f.2: compute_joint_torques (A1RobotControl.cpp:289-319) and update_plan (:148-202)"""
    G = load_ref_golden()
    for k in range(G["tau_tau"].shape[0]):
        t = O.joint_torques(G["tau_f_grf"][k], G["tau_f_kin"][k], G["tau_jac"][k], int(G["tau_contact"][k]), G["tau_km"][k], G["tau_grav"][k], G["tau_tau_prev"][k])
        assert np.abs(t - G["tau_tau"][k]).max() <= 1e-12 * max(1.0, np.abs(G["tau_tau"][k]).max()), k
    gp = a1mpc.default_gait_params(horizon=N)
    assert [gp.counter_per_gait, gp.counter_per_swing, gp.control_dt] == list(G["plan_params"]) and \
        np.array_equal(np.array(list(gp.default_foot_pos)).reshape(3, 4).T.reshape(-1), G["plan_default_foot_pos"])   # axis-major there, leg-major here
    for k in range(G["plan_gc_in"].shape[0]):
        gc, plan, sched, trel, tabs, tw = O.update_plan(gp, int(G["plan_mode"][k]), G["plan_gc_in"][k], G["plan_gcs"][k], G["plan_lin_vel"][k], G["plan_lin_vel_d"][k],
                                                        G["plan_rot_z"][k], G["plan_rot"][k], G["plan_root_pos"][k])
        assert np.array_equal(gc, G["plan_gc_out"][k]) and plan == int(G["plan_plan"][k]), k
        assert np.abs(trel - G["plan_trel"][k]).max() <= 1e-15 and np.abs(tabs - G["plan_tabs"][k]).max() <= 1e-15 and np.abs(tw - G["plan_tworld"][k]).max() <= 2e-15


def test_oracle_ekf_matches_reference_golden(built):
    """SURVEY 8f.4: A1BasicEKF over 30 ticks, each side carrying its own state (x, P compared every tick)"""
    G = load_ref_golden()
    x, P = O.ekf_init(G["ekf_fpr0"], G["ekf_rot"])
    assert np.abs(x - G["ekf_x_init"]).max() <= 1e-15 and np.array_equal(P, G["ekf_P_init"])
    for t in range(G["ekf_x"].shape[0]):
        x, P, pos, vel, ec, rc = O.ekf_update(x, P, 0.0025, 1, int(G["ekf_mode"][t]), G["ekf_acc"][t], G["ekf_gyro"][t], G["ekf_rot"], G["ekf_fpr"][t], G["ekf_fvr"][t], G["ekf_force"][t])
        assert rc == 0 and ec == int(G["ekf_ec"][t])
        assert np.abs(x - G["ekf_x"][t]).max() <= 1e-11 and np.abs(P - G["ekf_P"][t]).max() <= 1e-11, t
        assert np.abs(pos - G["ekf_pos"][t]).max() <= 1e-11 and np.abs(vel - G["ekf_vel"][t]).max() <= 1e-11


# --------------------------------------------------------------------------------------------------------------------------
# what the reference build (oracle/_ref) returned on inputs of these tests' own, stored in tests/golden/ref_live_v1.npz
# (tests/golden/make_ref_live_golden.py)
# --------------------------------------------------------------------------------------------------------------------------
def test_golden_file_is_what_the_reference_build_produces(built):
    """a few entries of the committed file, re-run through the reference build: bit-identical"""
    G = load_ref_golden()
    L = load_ref_live()
    assert np.array_equal(L["golden_A"], G["Ac"])
    for k, i in enumerate(L["golden_idx"]):
        assert np.array_equal(L["golden_g"][k], G["mpc_g"][i]) and np.array_equal(L["golden_lb"][k], G["mpc_lb"][i])
        assert np.array_equal(L["golden_Hdiag"][k], G["mpc_Hdiag"][i])
        assert np.array_equal(L["golden_mpc_states_d"][k], G["mpc_mpc_states_d"][i]) and np.array_equal(L["golden_f_body"][k], G["mpc_f_body"][i])


def test_oracle_equals_reference_build_on_fresh_states(built):
    """(a) of the verdict's definition of done: oracle build == reference build on 48 generator states apart from the ones of
    convexmpc_v1.npz, both weight sets (the Hessian through diag(H) and H @ v)"""
    G = load_ref_golden()
    L = load_ref_live()
    v = G["probe_V"][:, 0]
    worst = dict(H=0.0, g=0.0, f=0.0)
    for w in np.unique(L["fresh_weights"]):
        sel = np.nonzero(L["fresh_weights"] == w)[0]
        cfg = O.make_config(**ref_cfg_kwargs(G, int(w)))
        ob = O.Batch(L["fresh_x0"][sel].T, L["fresh_rot"][sel].T, L["fresh_foot"][sel].T, L["fresh_ref"][sel].T, L["fresh_contact"][sel])
        fo, info = O.compute_grf_batch(cfg, ob, O.MODE_EXACT, nthreads=4)
        for b, i in enumerate(sel):
            H, g, A, lb, ub = O.build_qp(cfg, ob, b)
            assert np.array_equal(A, G["Ac"]) and np.array_equal(lb, L["fresh_lb"][i]) and np.array_equal(ub, L["fresh_ub"][i])
            worst["H"] = max(worst["H"], _relerr(np.diag(H), L["fresh_Hdiag"][i]), _relerr(H @ v, L["fresh_Hv"][i]))
            worst["g"] = max(worst["g"], _relerr(g, L["fresh_g"][i]))
            worst["f"] = max(worst["f"], float(np.abs(fo[:, b] - L["fresh_f_body"][i]).max()))
    # forces: the reference's QP is solved by the ADMM stand-in (eps 1e-11), which leaves up to ~3e-5 N along flat directions of the
    # wide-noise / hardware-weight QPs; 1e-4 N is the P1 gate
    assert worst["H"] <= 1e-14 and worst["g"] <= 1e-14 and worst["f"] <= 1e-4, worst


def test_reference_compute_grf_warm_started_ticks_and_default_osqp(built):
    """the persistent solver path (A1RobotControl.cpp:522-538: initSolver once, update* afterwards) gives the same forces on the third
    tick as on the first; and with OSQP's DEFAULT tolerance the reference's own answer is far from the optimum (P2, reported)"""
    G = load_ref_golden()
    L = load_ref_live()
    i = int(L["ticks_idx"])
    a, b, d = L["ticks_f1"], L["ticks_f3"], L["ticks_f_default_osqp"]
    assert np.array_equal(a, b) and np.array_equal(a, G["mpc_f_body"][i])
    assert np.abs(d - a).max() > 1e-3
    f, info = O.compute_grf_batch(O.make_config(**ref_cfg_kwargs(G, int(G["mpc_weights"][i]))), _batch(G, [i]), O.MODE_EXACT, nthreads=1)
    assert info[0, 1] == 1 and np.abs(f[:, 0] - a).max() <= 1e-5 and np.abs(d - f[:, 0]).max() > 1e-3


def test_reference_standalone_driver_runs_and_prints_the_known_answer(built):
    """oracle/_ref/ref_test_mpc = the reference's test/test_mpc.cpp, main() and all, compiled unmodified: what it printed, and the
    oracle on the same state"""
    f = load_ref_live()["test_mpc_printed"]          # 3 x 4, printed as the reference prints foot_forces_grf
    assert abs(f[2, 0] - 42.7901) < 1e-3 and abs(f[2, 2] - 42.7901) < 1e-3 and abs(f[1, 0] + 12.837) < 1e-3
    assert np.abs(f[:, 1]).max() < 1e-6 and np.abs(f[:, 3]).max() < 1e-6      # swing legs FR, RR
    ocfg, ob = O.test_mpc_fixture()
    fo, info = O.compute_grf_batch(ocfg, ob, O.MODE_EXACT, nthreads=1)
    assert np.abs(fo[:, 0].reshape(4, 3).T - f).max() < 1e-3
