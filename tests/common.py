import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_golden():
    with open(os.path.join(ROOT, "tests", "golden", "golden_v1.json")) as fh:
        return json.load(fh)


def golden_groups():
    """golden cases grouped by (horizon, weights) -> (cfg kwargs, state dict, f_body [12,B])"""
    g = load_golden()
    groups = {}
    for c in g["cases"]:
        groups.setdefault((c["horizon"], c["weights"]), []).append(c)
    out = []
    for (hz, w), cs in sorted(groups.items()):
        st = dict(x0=np.array([c["x0"] for c in cs]).T.copy(), rot=np.array([c["rot"] for c in cs]).T.copy(),
                  foot=np.array([c["foot"] for c in cs]).T.copy(), ref=np.array([c["ref"] for c in cs]).T.copy(),
                  contact=np.array([c["contact"] for c in cs], dtype=np.uint32))
        f = np.array([c["f_body"] for c in cs]).T.copy()
        out.append((hz, w, g["weights"][w], st, f))
    return out


def load_ref_golden():
    """vectors produced by the REFERENCE's own compiled sources (tests/golden/make_ref_golden.py)"""
    with np.load(os.path.join(ROOT, "tests", "golden", "convexmpc_v1.npz")) as z:
        return {k: z[k] for k in z.files}


def load_ref_live():
    """what the reference build returned on the inputs of the tests that compare with it (tests/golden/make_ref_live_golden.py)"""
    with np.load(os.path.join(ROOT, "tests", "golden", "ref_live_v1.npz")) as z:
        return {k: z[k] for k in z.files}


def ref_cfg_kwargs(G, w):
    """keyword arguments (mass, inertia, q, r) of weight set w of the reference golden file, for O.make_config / a1mpc.default_config"""
    v = G["w%d" % w]
    return dict(mass=float(v[0]), inertia=tuple(v[1:10]), q=tuple(v[10:23]), r=tuple(v[23:35]))


def obatch(O, st, sl=None):
    if sl is None:
        return O.Batch(st["x0"], st["rot"], st["foot"], st["ref"], st["contact"])
    return O.Batch(st["x0"][:, sl], st["rot"][:, sl], st["foot"][:, sl], st["ref"][:, sl], st["contact"][sl])


def check_feasible(f_world_u, mu, fzmax, contact, tol=1e-7):
    """u_full [12N,B] world-frame: friction pyramid and fz bounds (ConvexMpc.cpp:46-58, 223-245)"""
    n12, B = f_world_u.shape
    u = f_world_u.reshape(n12 // 12, 4, 3, B)
    fx, fy, fz = u[:, :, 0], u[:, :, 1], u[:, :, 2]
    c = np.array([[(int(m) >> leg) & 1 for m in contact] for leg in range(4)])[None]  # [1,4,B]
    assert (np.abs(fx) <= mu * fz + tol).all() and (np.abs(fy) <= mu * fz + tol).all()
    assert (fz >= -tol).all() and (fz <= fzmax * c + tol).all()


def load_kin_golden():
    """vectors produced by the REFERENCE's own A1Kinematics (tests/golden/make_kin_golden.py)"""
    with open(os.path.join(ROOT, "tests", "golden", "kinematics_v1.json")) as fh:
        return json.load(fh)


def estimation_scenario(B, seed=0):
    """synthetic joint states / IMU of B robots for the kinematics + EKF rows (SURVEY 8f.4); rho_fix of GazeboA1ROS.cpp:76-97"""
    rng = np.random.default_rng(seed)
    rho_fix = np.array([[0.1805, 0.047, 0.0838, 0.21, 0.21], [0.1805, -0.047, -0.0838, 0.21, 0.21],
                        [-0.1805, 0.047, 0.0838, 0.21, 0.21], [-0.1805, -0.047, -0.0838, 0.21, 0.21]])
    rho_opt = rng.normal(0, 0.01, (4, 3))
    q = np.tile(np.array([0.0, 0.8, -1.6] * 4)[:, None], (1, B)) + rng.normal(0, 0.3, (12, B))
    dq = rng.normal(0, 2.0, (12, B))

    def rotm(r, p, y):
        cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(y), np.sin(y)
        Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]]); Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
        Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
        return Rz @ Ry @ Rx
    rot = np.stack([rotm(*rng.normal(0, [0.05, 0.05, 1.0])).reshape(9) for _ in range(B)], axis=1)
    return rng, rho_opt, rho_fix, q, dq, rot


def check_kinematics(O, outs, q, dq, rot, rho_opt, rho_fix, tol=1e-12):
    fpr, jac, fvr, fpa, fva = outs
    B = q.shape[1]
    for b in range(B):
        R = rot[:, b].reshape(3, 3)
        for leg in range(4):
            p, J = O.leg_kinematics(q[3 * leg:3 * leg + 3, b], rho_opt[leg], rho_fix[leg])
            v = J @ dq[3 * leg:3 * leg + 3, b]
            sl = slice(3 * leg, 3 * leg + 3)
            assert np.abs(fpr[sl, b] - p).max() <= tol and np.abs(jac[9 * leg:9 * leg + 9, b].reshape(3, 3) - J).max() <= tol
            assert np.abs(fvr[sl, b] - v).max() <= 10 * tol and np.abs(fpa[sl, b] - R @ p).max() <= tol and np.abs(fva[sl, b] - R @ v).max() <= 10 * tol


def ekf_walk(O, B, ticks, kin, init, update, seed=0):
    """runs `ticks` filter updates of B robots through (kin, init, update) -- the GPU engine's or the emulator's -- next to the
    oracle, each side carrying its OWN state from tick to tick; returns the worst difference in x, P and the outputs"""
    rng, rho_opt, rho_fix, q, dq, rot = estimation_scenario(B, seed)
    fpr, jac, fvr, fpa, fva = kin(q, dq, rot, rho_opt.reshape(12), rho_fix.reshape(20))
    get_state = init(fpr, rot)
    xs = []; Ps = []
    for b in range(B):
        x, P = O.ekf_init(fpr[:, b], rot[:, b]); xs.append(x); Ps.append(P)
    dt = 0.0025
    worst = 0.0
    for tick in range(ticks):
        mode = (rng.random(B) < 0.8).astype(np.uint32)
        acc = rng.normal([0, 0, 9.81], 1.0, (B, 3)).T.copy(); gyro = rng.normal(0, 0.3, (3, B))
        q = q + dt * dq; dq = dq + rng.normal(0, 0.5, dq.shape)
        fpr, jac, fvr, fpa, fva = kin(q, dq, rot, rho_opt.reshape(12), rho_fix.reshape(20))
        force = rng.uniform(-20, 160, (4, B))
        flat = 1 if tick % 7 else 0
        pos, vel, ec, status = update(dt, flat, mode, acc, gyro, rot, fpr, fvr, force, tick)
        assert (status == 0).all(), status
        X, PP = get_state()
        for b in range(B):
            x, P, po, ve, eco, rc = O.ekf_update(xs[b], Ps[b], dt, flat, mode[b], acc[:, b], gyro[:, b], rot[:, b], fpr[:, b], fvr[:, b], force[:, b])
            assert rc == 0 and ec[b] == eco
            xs[b], Ps[b] = x, P
            worst = max(worst, np.abs(X[b] - x).max(), np.abs(PP[b] - P).max(), np.abs(pos[:, b] - po).max(), np.abs(vel[:, b] - ve).max())
    return worst
