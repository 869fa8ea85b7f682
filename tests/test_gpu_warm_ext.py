"""Warm start of the extended call (a1mpc_solve_batch_ext_warm) through the C ABI on the GPU: per-step contact schedules that
advance one step per tick, terrain normals, the previous tick's verified faces as the first guess per foot-step.  Same checks
as tests/test_emu_warm_ext.py runs on the CPU emulator (the emulator replay of the GPU suite has no extended warm call, hence
the skip under A1MPC_EMU_ENGINE)."""
import ctypes as C
import os

import numpy as np
import pytest

from common import obatch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(os.environ.get("A1MPC_EMU_ENGINE") == "1", reason="emulator twin: tests/test_emu_warm_ext.py")]

TOL_F = 1e-4      # N
SCALE = np.array([.02, .02, .02, .01, .01, .005, .1, .1, .1, .05, .05, .05])[:, None]


@pytest.fixture(scope="module")
def a1(built):
    import a1mpc
    return a1mpc


@pytest.fixture(scope="module")
def O(built):
    from oracle import oracle_py
    return oracle_py


def _plan(a1, B, N, T, seed):
    """N + T plan steps (tick t solves steps t .. t + N - 1); robots 0-63 have four feet down at step 2 and robots 64-127 lift a
    foot at step N + 1, so they move between the compacted and the general kernel"""
    base, normals = a1.gen_schedule(B, 20, 4, seed)
    plan = base[np.arange(N + T) % 16]
    plan[2, 0:64] = 0b1111
    plan[N + 1, 64:128] &= 0b0001
    plan[N + 1, 64:128] |= 0b0001
    return plan, normals


def _advance(st, rng, noise):
    x0 = st["x0"].copy()
    x0[3:6] += 0.0025 * st["x0"][9:12]
    x0[0:3] += 0.0025 * st["x0"][6:9]
    x0 += noise * rng.standard_normal(x0.shape) * SCALE
    return dict(st, x0=x0)


def _sub(st, idx):
    return {k: (v[idx] if k == "contact" else v[:, idx]) for k, v in st.items()}


def _ticks(a1, O, N, B, T, nsample, seed):
    eng = a1.Engine(a1.default_config(horizon=N))
    ocfg = O.make_config(horizon=N)
    plan, normals = _plan(a1, B, N, T, seed)
    st = a1.gen_states(B, 4, seed)
    rng = np.random.default_rng(seed)
    sample = np.sort(np.random.default_rng(seed + 1).choice(B, size=min(nsample, B), replace=False))
    warm = eng.warm_alloc(B)
    hits = []
    for t in range(T):
        sched = np.ascontiguousarray(plan[t:t + N])
        f, status, iters, u = eng.solve_ext_warm(st, warm, sched, normals, shift=1, want_u=True)
        assert (status == a1.STATUS_OPTIMAL).all(), (t, np.bincount(status))
        fo, _ = O.compute_grf_batch_ext(ocfg, obatch(O, _sub(st, sample)), sched[:, sample], normals[:, sample], mode=O.MODE_EXACT,
                                        nthreads=O.hardware_threads())
        assert np.abs(f[:, sample] - fo).max() <= TOL_F, (t, np.abs(f[:, sample] - fo).max())
        legs = (sched[:, None, :] >> (np.arange(12) // 3)[None, :, None]) & 1
        assert (u.reshape(N, 12, B)[legs == 0] == 0).all()
        fc, sc, itc = eng.solve_ext(st, sched, normals)                       # the cold call: same optimum
        assert (sc == a1.STATUS_OPTIMAL).all() and np.abs(f - fc).max() < 1e-7
        hits.append((iters % 100 == 0).mean())
        st = _advance(st, rng, 0.03)
    a1.lib().a1mpc_device_free(eng.h, warm)
    eng.close()
    return hits


def test_config4_size_advancing_schedules_n10(a1, O):
    """B = 16384, three ticks, a seeded sample of 4096 QPs per tick against the extended oracle, every status checked"""
    hits = _ticks(a1, O, 10, 16384, 3, 4096, 21)
    assert hits[0] == 0.0 and min(hits[1:]) > 0.5, hits


def test_advancing_schedules_n20(a1, O):
    hits = _ticks(a1, O, 20, 512, 3, 512, 22)
    assert hits[0] == 0.0 and hits[1] > 0.3, hits


def test_device_and_host_pointers_agree(a1):
    """the same two ticks through device pointers (asynchronous) and host pointers (mirrors): bit-identical outputs and slots"""
    B, N = 1024, 10
    eng = a1.Engine(a1.default_config(horizon=N))
    lib = a1.lib()
    plan, normals = _plan(a1, B, N, 2, 23)
    st = a1.gen_states(B, 4, 23)
    w_host, w_dev = eng.warm_alloc(B), eng.warm_alloc(B)
    d = a1.DeviceBatch(eng, B)
    dsched, dnorm = eng.dalloc(N * B * 4), eng.dalloc(12 * B * 8)
    nm = np.ascontiguousarray(normals)
    a1._check(lib.a1mpc_memcpy_h2d(eng.h, dnorm, nm.ctypes.data_as(C.c_void_p), nm.nbytes))
    for t in range(2):
        sched = np.ascontiguousarray(plan[t:t + N])
        fh, sh, ih = eng.solve_ext_warm(st, w_host, sched, normals, shift=1)
        d.upload(st)
        a1._check(lib.a1mpc_memcpy_h2d(eng.h, dsched, sched.ctypes.data_as(C.c_void_p), sched.nbytes))
        a1._check(lib.a1mpc_solve_batch_ext_warm(eng.h, B, C.byref(d.inp), C.byref(a1.InputsExt(dsched, dnorm)), C.byref(d.out), w_dev, 1))
        eng.sync()
        fd, sd = d.download()
        assert np.array_equal(fh, fd) and np.array_equal(sh, sd) and (sh == a1.STATUS_OPTIMAL).all()
        st = _advance(st, np.random.default_rng(t), 0.03)
    slots = []
    for w in (w_host, w_dev):
        a = np.zeros((B, 4 + 4 * N), dtype=np.uint32)
        a1._check(lib.a1mpc_memcpy_d2h(eng.h, a.ctypes.data_as(C.c_void_p), w, a.nbytes))
        slots.append(a)
    assert np.array_equal(slots[0], slots[1]) and (slots[0][:, 0] == 1).all()
    d.free()
    for p in (w_host, w_dev, dsched, dnorm):
        a1.lib().a1mpc_device_free(eng.h, p)
    eng.close()


def test_precision_32(a1, O):
    """fp32 boundary arrays: within 1e-4 N + 1 fp32 ulp of 180 N of the optimum of the fp32-rounded inputs (DESIGN.md §3)"""
    B, N = 1024, 10
    eng = a1.Engine(a1.default_config(horizon=N, precision=32))
    plan, normals = _plan(a1, B, N, 2, 24)
    st = a1.gen_states(B, 4, 24)
    warm = eng.warm_alloc(B)
    nm32 = normals.astype(np.float32).astype(np.float64)
    for t in range(2):
        sched = np.ascontiguousarray(plan[t:t + N])
        f, status, iters = eng.solve_ext_warm(st, warm, sched, normals, shift=1)
        st32 = {k: (v if k == "contact" else v.astype(np.float32).astype(np.float64)) for k, v in st.items()}
        fo, _ = O.compute_grf_batch_ext(O.make_config(horizon=N), obatch(O, st32), sched, nm32, mode=O.MODE_EXACT, nthreads=O.hardware_threads())
        assert f.dtype == np.float32 and (status == a1.STATUS_OPTIMAL).all()
        assert np.abs(f.astype(np.float64) - fo).max() <= 1e-4 + 1.5e-5
        st = _advance(st, np.random.default_rng(t), 0.03)
    a1.lib().a1mpc_device_free(eng.h, warm)
    eng.close()


def test_argument_errors(a1):
    st = a1.gen_states(8, 4, 1)
    sched, normals = a1.gen_schedule(8, 10, 4, 1)
    eng = a1.Engine(a1.default_config(horizon=10))
    warm = eng.warm_alloc(8)
    host = np.zeros(8 * 44, dtype=np.uint32)
    with pytest.raises(a1.A1MpcError, match="device memory"):
        eng.solve_ext_warm(st, host.ctypes.data_as(C.c_void_p), sched, normals)
    for shift in (-1, 11):
        with pytest.raises(a1.A1MpcError, match="shift out of range"):
            eng.solve_ext_warm(st, warm, sched, normals, shift=shift)
    a1.lib().a1mpc_device_free(eng.h, warm)
    eng.close()
    r = [1e-7] * 12
    r[4] = 2e-7
    eng = a1.Engine(a1.default_config(horizon=10, r=r))
    warm = eng.warm_alloc(8)
    with pytest.raises(a1.A1MpcError, match="isotropic"):
        eng.solve_ext_warm(st, warm, sched, normals)
    a1.lib().a1mpc_device_free(eng.h, warm)
    eng.close()
