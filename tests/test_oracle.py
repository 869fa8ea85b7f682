"""CPU tests of the oracle (test infrastructure) against the committed golden fixtures and against
itself (two independent solvers + KKT certificates).  No GPU."""
import numpy as np
import pytest

from common import golden_groups, load_golden, obatch


@pytest.fixture(scope="module")
def O(built):
    from oracle import oracle_py
    return oracle_py


def test_test_mpc_fixture_known_answer(O):
    """the state of the reference's only standalone driver (test/test_mpc.cpp:15-91) against the surveyor's
    independently derived optimum (SURVEY.md Appendix C)"""
    cfg, ob = O.test_mpc_fixture()
    f, info, u = O.compute_grf_batch(cfg, ob, O.MODE_EXACT, want_u=True)
    ka = load_golden()["test_mpc_fixture"]["survey_known_answer"]
    assert np.allclose(f[0:3, 0], ka["FL"], atol=2e-10) and np.allclose(f[6:9, 0], ka["RL"], atol=2e-10)
    assert np.abs(f[3:6, 0]).max() == 0 and np.abs(f[9:12, 0]).max() == 0      # swing feet pinned to zero
    fz = u[0].reshape(10, 4, 3)[:, 0, 2]
    assert np.allclose(fz, [42.790, 45.687, 47.351, 47.826, 47.060, 44.906, 41.114, 35.317, 29.772, 18.588], atol=6e-4)
    H, g, A, lb, ub = O.build_qp(cfg, ob, 0)
    assert abs(0.5 * u[0] @ H @ u[0] + g @ u[0] - (-1.364844425490e-01)) < 1e-12
    assert info[0, 1] == 1 and info[0, 2] < 1e-15


def test_exact_reproduces_golden(O):
    for hz, w, wk, st, f_gold in golden_groups():
        cfg = O.make_config(horizon=hz, **wk)
        f, info = O.compute_grf_batch(cfg, obatch(O, st), O.MODE_EXACT)
        assert (info[:, 1] == 1).all()
        assert np.abs(f - f_gold).max() <= 1e-9
        # certificates on the literal 12N-variable problem
        assert info[:, 2].max() <= 1e-12 and info[:, 3].max() <= 1e-9 and info[:, 4].max() <= 1e-9


def test_osqp_restatement_converges_to_the_same_point(O):
    """second, independent method: the OSQP algorithm (the reference's solver) run to eps 1e-11"""
    hz, w, wk, st, f_gold = golden_groups()[0]
    cfg = O.make_config(horizon=hz, **wk)
    sl = slice(0, 6)
    f, info = O.compute_grf_batch(cfg, obatch(O, st, sl), O.MODE_OSQP_TIGHT)
    assert (info[:, 1] == 1).all()
    assert np.abs(f - f_gold[:, sl]).max() <= 1e-5


def test_osqp_default_is_far_from_converged(O):
    """P2 (reported, not gated): the shipped controller runs OSQP at eps 1e-3 and stops early"""
    hz, w, wk, st, f_gold = golden_groups()[0]
    cfg = O.make_config(horizon=hz, **wk)
    f, info = O.compute_grf_batch(cfg, obatch(O, st), O.MODE_OSQP_DEFAULT)
    assert (info[:, 0] <= 4000).all() and (info[:, 0] % 25 == 0).all()     # terminates on a check_termination multiple
    d = np.abs(f - f_gold).max(axis=0)
    assert d.max() > 1e-3


def test_literal_build_structure(O):
    """facts the CUDA kernels rely on, checked on the literal restatement: H symmetric positive definite,
    H == T0 (x) G0 + T1 (x) G1 + 2R (A_c^3 = 0, constant B_d), bounds pattern, pyramid matrix"""
    hz, w, wk, st, _ = golden_groups()[0]
    cfg = O.make_config(horizon=hz, **wk)
    N = hz
    H, g, A, lb, ub = O.build_qp(cfg, obatch(O, st), 2)
    assert np.abs(H - H.T).max() <= 1e-18 + 1e-15 * np.abs(H).max()
    assert np.linalg.eigvalsh(H).min() >= 2 * min(wk["r"]) * (1 - 1e-6)
    T0 = np.array([[N - max(a, b) for b in range(N)] for a in range(N)], float)
    T1 = np.array([[sum((i - a) * (i - b) for i in range(max(a, b), N)) for b in range(N)] for a in range(N)], float)
    Hb = H.reshape(N, 12, N, 12)
    G1 = (Hb[N - 2, :, N - 2] - 2 * Hb[N - 1, :, N - 1] + np.diag(2 * np.array(wk["r"])))  # T1[N-2,N-2]=1, T0 diff = 1
    G0 = Hb[N - 1, :, N - 1] - np.diag(2 * np.array(wk["r"]))                               # T0[N-1,N-1]=1, T1=0
    Hk = np.einsum("ab,ij->aibj", T0, G0) + np.einsum("ab,ij->aibj", T1, G1)
    Hk = Hk.reshape(12 * N, 12 * N) + np.diag(np.tile(2 * np.array(wk["r"]), N))
    assert np.abs(Hk - H).max() <= 1e-13 * np.abs(H).max()
    # pyramid rows (ConvexMpc.cpp:46-58) and bounds (:223-245)
    assert A.shape == (20 * N, 12 * N) and (A != 0).sum() == 9 * 4 * N
    assert np.allclose(A[0:5, 0:3], [[1, 0, .3], [1, 0, -.3], [0, 1, .3], [0, 1, -.3], [0, 0, 1]])
    c = [(int(st["contact"][2]) >> i) & 1 for i in range(4)]
    assert np.allclose(ub[4:20:5], 180.0 * np.array(c)) and (lb[4::5] == 0).all()
    assert (ub[0::5] == 1e30).all() and (lb[1::5] == -1e30).all()


def test_qp_mats_general_equals_driven_build(O):
    """ConvexMpc::calculate_qp_mats fed with the same A_d / B_d every step reproduces compute_grf's build"""
    hz, w, wk, st, _ = golden_groups()[0]
    cfg = O.make_config(horizon=hz, **wk)
    b = 1
    H, g, A, lb, ub = O.build_qp(cfg, obatch(O, st), b)
    from gpu_helpers import discrete_model
    Ad, Bd, x0, xd = discrete_model(cfg, st, b)
    H2, g2 = O.qp_mats(cfg, Ad, np.tile(Bd, (hz, 1)), x0, xd)
    assert np.abs(H2 - H).max() <= 1e-15 * np.abs(H).max() and np.abs(g2 - g).max() <= 1e-14 * np.abs(g).max()


def test_grf_qp_single_two_methods(O):
    """config 1: 12-variable instantaneous GRF QP, standing, four feet (A1RobotControl.cpp:377-445)"""
    rot = np.eye(3).ravel()
    foot = np.array([.17, .15, -.3, .17, -.15, -.3, -.17, .15, -.3, -.17, -.15, -.3])
    acc = np.array([5.0, -3.0, 12.0 * 9.8 + 20.0, 2.0, -1.0, 0.5])
    f, info = O.grf_qp_single(acc, rot, rot, foot, 0b1111, O.MODE_EXACT)
    ft, _ = O.grf_qp_single(acc, rot, rot, foot, 0b1111, O.MODE_OSQP_TIGHT)
    assert info[1] == 1 and np.abs(f - ft).max() <= 1e-6
    assert abs(f[2::3].sum() - acc[2]) < 1.0          # supports the weight (soft, Q_z = 100 vs R = 1e-3)
    f2, _ = O.grf_qp_single(acc, rot, rot, foot, 0b0101, O.MODE_EXACT)
    assert np.abs(f2[3:6]).max() == 0 and np.abs(f2[9:12]).max() == 0


def test_config4_extension_oracle_two_methods(O, built):
    """per-step contact schedule + terrain normals (extension beyond the reference): exact solver vs OSQP-algorithm run tight,
    and the extension with nothing to extend equals the plain path"""
    import a1mpc
    B = 12
    st = a1mpc.gen_states(B, 4, 5)
    sched, normals = a1mpc.gen_schedule(B, 10, 4, 5)
    assert sched.shape == (10, B) and np.abs(np.linalg.norm(normals.reshape(4, 3, B), axis=1) - 1).max() < 1e-14
    cfg = O.make_config()
    f, info = O.compute_grf_batch_ext(cfg, obatch(O, st), sched, normals, O.MODE_EXACT, nthreads=4)
    ft, _ = O.compute_grf_batch_ext(cfg, obatch(O, st), sched, normals, O.MODE_OSQP_TIGHT, nthreads=4)
    assert (info[:, 1] == 1).all() and info[:, 2].max() <= 1e-12 and info[:, 3].max() <= 1e-9 and info[:, 4].max() <= 1e-9
    assert np.abs(f - ft).max() <= 1e-5
    f0, _ = O.compute_grf_batch(cfg, obatch(O, st), O.MODE_EXACT)
    f1, _ = O.compute_grf_batch_ext(cfg, obatch(O, st), None, None, O.MODE_EXACT)
    assert np.abs(f0 - f1).max() <= 1e-12
    # a foot that is in the air at step 0 gets exactly zero force
    air = np.array([[((int(sched[0, b]) >> leg) & 1) == 0 for b in range(B)] for leg in range(4)])
    assert np.abs(f.reshape(4, 3, B)[air.nonzero()[0], :, air.nonzero()[1]]).max() == 0


def test_neighbour_rows_oracle_sanity(O):
    """the restated update_plan / compute_joint_torques (the steps either side of the path) on hand-checkable inputs"""
    import a1mpc
    gp = a1mpc.default_gait_params(10)
    eye = np.eye(3).ravel()
    # standstill: all feet planned in contact, counters reset to the trot offsets (A1CtrlStates.h:322-326)
    gc, plan, sched, trel, tabs, tw = O.update_plan(gp, 0, [5, 6, 7, 8], [2, 2, 2, 2], [0, 0, 0], [0, 0, 0], eye, eye, [0, 0, 0.3])
    assert plan == 0b1111 and list(gc) == [0, 120, 120, 0] and (sched == 0b1111).all()
    assert np.allclose(trel.reshape(4, 3), [[.17, .15, -.35], [.17, -.15, -.35], [-.17, .15, -.35], [-.17, -.15, -.35]])
    assert np.allclose(tw.reshape(4, 3)[:, 2], -.35 + .3)
    # walking: FL/RR half a cycle ahead of FR/RL; counters advance by their speed and wrap at counter_per_gait
    gc, plan, sched, *_ = O.update_plan(gp, 1, [118, 238, 238, 118], [2, 2, 2, 2], [0, 0, 0], [0, 0, 0], eye, eye, [0, 0, 0.3])
    assert list(gc) == [120, 0, 0, 120] and plan == 0b1111
    assert sched[0] == 0b1111 and sched[1] == 0b0110 and (sched[1:] == 0b0110).all()      # FL, RR lift off one tick later
    # Raibert foothold saturates at FOOT_DELTA_X_LIMIT
    *_, trel, _, _ = O.update_plan(gp, 1, [0, 0, 0, 0], [2, 2, 2, 2], [5, 0, 0], [0, 0, 0], eye, eye, [0, 0, 0])
    assert np.allclose(trel.reshape(4, 3)[:, 0], [.27, .27, -.07, -.07])
    # torques: stance leg J^T(-f), swing leg J^-1 (km .* f_kin), + gravity compensation
    jac = np.tile((2 * np.eye(3)).ravel(), 4)
    f = np.arange(12.0); fk = np.ones(12) * 10
    tau = O.joint_torques(f, fk, jac, 0b0001, [0.1, 0.1, 0.1], np.zeros(12))
    assert np.allclose(tau[0:3], -2 * f[0:3]) and np.allclose(tau[3:], 0.5)


def test_kinematics_oracle_is_pinned_to_the_reference(O):
    """golden vectors generated from the REFERENCE's own A1Kinematics::fk / jac (tests/golden/make_kin_golden.py, built by
    `make -C oracle ref`); and 500 random draws against what that build returned for them (tests/golden/ref_live_v1.npz)"""
    from common import load_kin_golden, load_ref_live
    g = load_kin_golden()
    assert len(g["cases"]) >= 64
    for c in g["cases"]:
        p, J = O.leg_kinematics(c["q"], c["rho_opt"], c["rho_fix"])
        assert np.abs(p - np.array(c["p"])).max() <= 1e-14 and np.abs(J.reshape(9) - np.array(c["J"])).max() <= 1e-14
    L = load_ref_live()
    kin_p, kin_J = L["kin_p"], L["kin_J"]
    rng = np.random.default_rng(7)
    for k in range(500):
        q = rng.uniform(-2, 2, 3); ro = rng.normal(0, 0.05, 3); rf = rng.normal(0, 0.2, 5)
        p, J = O.leg_kinematics(q, ro, rf)
        assert np.abs(p - kin_p[k]).max() <= 1e-14 and np.abs(J - kin_J[k]).max() <= 1e-14


def test_ekf_oracle_sanity(O):
    """the dense restatement of A1BasicEKF: a robot standing still on flat ground converges to the true height and zero velocity"""
    rot = np.eye(3).reshape(9)
    fk = np.array([[0.18, 0.13, -0.3], [0.18, -0.13, -0.3], [-0.18, 0.13, -0.3], [-0.18, -0.13, -0.3]]).reshape(12)
    x, P = O.ekf_init(fk, rot)
    assert np.allclose(np.diag(P), 3.0) and abs(x[2] - 0.09) < 1e-15 and np.allclose(x[6:9], fk[0:3] + [0, 0, 0.09])
    for _ in range(400):
        x, P, pos, vel, ec, rc = O.ekf_update(x, P, 0.0025, 1, 0, [0, 0, 9.81], [0, 0, 0], rot, fk, np.zeros(12), [80] * 4)
        assert rc == 0 and ec == 0b1111
    assert abs(pos[2] - 0.3) < 2e-3 and np.abs(vel).max() < 1e-3
    assert np.allclose(P, P.T) and np.linalg.eigvalsh(P).min() > -1e-12
