"""Generates tests/golden/ref_live_v1.npz: what the reference build (oracle/_ref, `make -C oracle ref`) returns for the checks of
tests/test_ref_pin.py and tests/test_oracle.py that compare with it on inputs of their own, so that those checks run everywhere.

Contents (float64 unless noted):
  golden_*  entries golden_idx of convexmpc_v1.npz re-run through the reference's compute_grf: g, lb, diag(H), mpc_states_d, f_body;
            golden_A, the pyramid matrix (the same for every entry)
  fresh_*   48 generator states (16 each of config 2 / gazebo weights, config 4 / gazebo, config 4 / hardware; weights index into
            w0..w2 of convexmpc_v1.npz): inputs, and the reference's g, lb, ub, diag(H), H @ probe_V[:, 0] (probe_V of
            convexmpc_v1.npz) and f_body.  The full Hessians would not fit a small file: the sketch stands in for them.
  ticks_*   convexmpc_v1.npz entry ticks_idx through compute_grf on the first and the third tick of one persistent solver, and with
            OSQP's default tolerance
  test_mpc_printed  the 3 x 4 forces printed by the reference's standalone driver (oracle/_ref/ref_test_mpc), as printed
  kin_p, kin_J      A1Kinematics::fk / jac on the 500 random (q, rho_opt, rho_fix) that test_oracle.py draws from default_rng(7)
Run:  python tests/golden/make_ref_live_golden.py        (CPU only, needs the oracle/_ref build)
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "a1-qp-mpc-controller_b200")); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import a1mpc
from oracle import oracle_py as O
from oracle import ref_py as R
from common import load_ref_golden, ref_cfg_kwargs

GOLDEN_IDX = (0, 3, 30, 40)
FRESH = (("gazebo", 2, 501), ("gazebo", 4, 502), ("hardware", 4, 503))
FRESH_PER_STREAM = 16
TICKS_IDX = 5


def kinematics_inputs():
    """the draws of test_oracle.test_kinematics_oracle_is_pinned_to_the_reference, in its order"""
    rng = np.random.default_rng(7)
    out = []
    for _ in range(500):
        q = rng.uniform(-2, 2, 3); ro = rng.normal(0, 0.05, 3); rf = rng.normal(0, 0.2, 5)
        out.append((q, ro, rf))
    return out


def main():
    assert R.available(), "oracle/_ref/libref_mpc.so missing: run `make -C oracle ref` where the reference sources are present"
    G = load_ref_golden()
    out = {}

    golden = {k: [] for k in ("g", "lb", "Hdiag", "mpc_states_d", "f_body")}
    for i in GOLDEN_IDX:
        cfg = O.make_config(**ref_cfg_kwargs(G, int(G["mpc_weights"][i])))
        r = R.compute_grf(cfg, G["mpc_x0"][i], G["mpc_rot"][i], G["mpc_foot"][i], G["mpc_ref"][i], int(G["mpc_contact"][i]))
        P, q, A, l, u = r["qp"]
        if "golden_A" in out:
            assert np.array_equal(A, out["golden_A"])
        out["golden_A"] = A
        for k, v in zip(golden, (q, l, np.diag(P).copy(), r["mpc_states_d"], r["f_body"])):
            golden[k].append(v)
    out["golden_idx"] = np.array(GOLDEN_IDX, dtype=np.int32)
    for k, v in golden.items():
        out["golden_" + k] = np.stack(v)

    v = G["probe_V"][:, 0]
    fresh = {k: [] for k in ("x0", "rot", "foot", "ref", "contact", "weights", "g", "lb", "ub", "Hdiag", "Hv", "f_body")}
    for wname, cid, stream in FRESH:
        w = ["gazebo", "hardware"].index(wname)
        cfg = O.make_config(**ref_cfg_kwargs(G, w))
        st = a1mpc.gen_states(FRESH_PER_STREAM, cid, stream=stream)
        for b in range(FRESH_PER_STREAM):
            r = R.compute_grf(cfg, st["x0"][:, b], st["rot"][:, b], st["foot"][:, b], st["ref"][:, b], int(st["contact"][b]))
            P, q, A, l, u = r["qp"]
            assert np.array_equal(A, G["Ac"])
            for k, val in zip(fresh, (st["x0"][:, b], st["rot"][:, b], st["foot"][:, b], st["ref"][:, b], st["contact"][b], w,
                                      q, l, u, np.diag(P).copy(), P @ v, r["f_body"])):
                fresh[k].append(val)
    for k, val in fresh.items():
        out["fresh_" + k] = np.array(val, dtype=np.uint32 if k == "contact" else (np.int32 if k == "weights" else np.float64))

    i = TICKS_IDX
    cfg = O.make_config(**ref_cfg_kwargs(G, int(G["mpc_weights"][i])))
    args = (cfg, G["mpc_x0"][i], G["mpc_rot"][i], G["mpc_foot"][i], G["mpc_ref"][i], int(G["mpc_contact"][i]))
    out["ticks_idx"] = np.array(i, dtype=np.int32)
    out["ticks_f1"] = R.compute_grf(*args, ticks=1)["f_body"]
    out["ticks_f3"] = R.compute_grf(*args, ticks=3)["f_body"]
    out["ticks_f_default_osqp"] = R.compute_grf(*args, solver="default")["f_body"]

    txt = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "ref_test_mpc")], capture_output=True, text=True, timeout=60, check=True).stdout
    out["test_mpc_printed"] = np.array([[float(x) for x in ln.split()] for ln in txt.splitlines()[:3]])
    assert out["test_mpc_printed"].shape == (3, 4)

    kin = [O.ref_leg_kinematics(q, ro, rf) for q, ro, rf in kinematics_inputs()]
    out["kin_p"] = np.stack([p for p, J in kin])
    out["kin_J"] = np.stack([J for p, J in kin])

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_live_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote %s: %d arrays, %.0f KB" % (path, len(out), os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
