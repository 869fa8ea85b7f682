"""CPU tests of the C-ABI shared library: it loads, exports every symbol include/a1mpc.h declares, validates
arguments, and FAILS LOUDLY without a GPU (no CPU fallback).  No compute calls."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def a1(built):
    import a1mpc
    return a1mpc


def test_every_declared_symbol_is_exported(a1):
    hdr = open(os.path.join(ROOT, "include", "a1mpc.h")).read()
    declared = sorted(set(re.findall(r"\b(a1mpc_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 25
    lib = a1.lib()
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, missing
    assert sorted(set(a1.EXPORTS)) == declared


def test_struct_layout_matches_header(a1):
    # a1mpc_config: 2 ints, 5 doubles, 9+13+12 doubles, int (+pad), double
    assert C.sizeof(a1.Config) == 8 + 5 * 8 + 34 * 8 + 8 + 8
    assert C.sizeof(a1.Inputs) == 6 * 8 and C.sizeof(a1.Outputs) == 5 * 8
    assert C.sizeof(a1.InputsExt) == 2 * 8 and C.sizeof(a1.GaitParams) == 3 * 8 + 12 * 8 + 2 * 8 + 8


def test_default_config_is_the_launch_default(a1):
    c = a1.default_config()
    assert (c.horizon, c.dt, c.mu, c.fz_max, c.mass) == (10, 0.0025, 0.3, 180.0, 12.0)       # A1Params.h:26, ConvexMpc.cpp:8,224
    assert list(c.q) == [20, 10, 1, 0, 0, 420, .05, .05, .05, 30, 30, 10, 0]                  # gazebo_a1_mpc.yaml:40-56
    assert list(c.r) == [1e-7] * 12


def test_argument_validation_happens_before_the_device_probe(a1):
    h = C.c_void_p()
    for kw in (dict(horizon=7), dict(precision=16), dict(fz_min=1.0), dict(mu=0.0), dict(r=[0.0] * 12)):
        rc = a1.lib().a1mpc_create(C.byref(h), C.byref(a1.default_config(**kw)), 0)
        assert rc == -1 and a1.lib().a1mpc_last_error()


_NO_GPU_CHECK = """
import a1mpc
assert a1mpc.lib().a1mpc_device_count() == 0
try:
    a1mpc.Engine()
except a1mpc.A1MpcError as e:
    assert "no CUDA device" in str(e), e
else:
    raise AssertionError("Engine() without a device did not fail")
"""


def test_no_gpu_means_loud_failure_not_fallback(a1):
    """in a process that sees no device (an empty CUDA_VISIBLE_DEVICES hides the GPUs of a machine that has some)"""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", _NO_GPU_CHECK], cwd=os.path.join(ROOT, "a1-qp-mpc-controller_b200"), env=env,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr


def test_generator_is_deterministic_and_well_formed(a1):
    a = a1.gen_states(4096, 2, 5)
    b = a1.gen_states(4096, 2, 5)
    c = a1.gen_states(4096, 2, 6)
    for k in a:
        assert np.array_equal(a[k], b[k])
    assert not np.array_equal(a["x0"], c["x0"])
    R = a["rot"].T.reshape(-1, 3, 3)
    assert np.abs(R @ R.transpose(0, 2, 1) - np.eye(3)).max() < 1e-14
    frac = [(a["contact"] == m).mean() for m in (0b1001, 0b0110, 0b1111)]
    assert abs(frac[0] - .45) < .03 and abs(frac[1] - .45) < .03 and abs(frac[2] - .10) < .02
    assert a["x0"][5].min() >= 0.296 and a["x0"][5].max() <= 0.304
    w = a1.gen_states(4096, 4, 5)
    assert w["x0"][5].min() < 0.26 and w["x0"][5].max() > 0.31
    # the first 16 QPs of a batch do not depend on the batch size (per-QP substreams)
    s = a1.gen_states(16, 2, 5)
    assert np.array_equal(s["x0"], a["x0"][:, :16])


def test_every_binding_marshals_its_arguments(a1):
    """Every Engine method of a1mpc.py, driven with a NULL handle: the C entry points must reject it with A1MPC_EINVAL
    *after* ctypes has converted every argument against the declared prototype -- a wrong argument count or type in the
    binding shows up here (ctypes.ArgumentError / TypeError) instead of on the GPU box."""
    eng = a1.Engine.__new__(a1.Engine)
    eng.h, eng.cfg, eng.device = None, a1.default_config(), 0
    B = 4
    st = a1.gen_states(B, 2, 1)
    null = C.c_void_p(0)
    rng = np.random.default_rng(0)
    r = lambda *s: rng.standard_normal(s)
    calls = [
        lambda: eng.solve(st, want_u=True),
        lambda: eng.solve_warm(st, null),
        lambda: eng.warm_alloc(B),
        lambda: eng.solve_ext(st, np.full((10, B), 9, dtype=np.uint32), np.tile([0.0, 0.0, 1.0], 4)[:, None].repeat(B, 1)),
        lambda: eng.build_qp(st),
        lambda: eng.qp_mats(r(B, 13, 13), r(B, 130, 12), r(B, 13), r(B, 130)),
        lambda: eng.solve_dense(r(B, 120, 120), r(B, 120), np.full(B, 9, dtype=np.uint32)),
        lambda: eng.grf_qp(r(B, 6), r(B, 9), r(B, 9), r(B, 12), np.full(B, 15, dtype=np.uint32)),
        lambda: eng.leg_kinematics(r(12, B), r(12, B), r(9, B), r(12), r(20)),
        lambda: eng.ekf_alloc(B),
        lambda: eng.ekf_init(null, r(12, B), r(9, B)),
        lambda: eng.ekf_update(null, 0.0025, True, np.ones(B, dtype=np.uint32), r(3, B), r(3, B), r(9, B), r(12, B), r(12, B), r(4, B)),
        lambda: eng.ekf_state(null, B),
        lambda: eng.update_plan(a1.default_gait_params(10), r(4, B), r(4, B), np.ones(B, dtype=np.uint32), r(3, B), r(3, B), r(9, B), r(9, B), r(3, B)),
        lambda: eng.dalloc(64),
        lambda: eng.halloc(64),
    ]
    for i, call in enumerate(calls):
        with pytest.raises(a1.A1MpcError):
            call()
    assert a1.lib().a1mpc_warm_bytes(None, B) == 0 and a1.lib().a1mpc_ekf_bytes(B) == B * 342 * 8
    eng.h = None   # nothing to destroy
