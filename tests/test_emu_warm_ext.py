"""The warm start of the extended call (a1mpc_solve_batch_ext_warm) on the CPU block emulator: per-step contact schedules
and terrain normals, the previous tick's verified faces as the finisher's first guess per foot-step, routed like the library
(two-feet-per-step robots on the compacted kernel, everything else on the general 4-foot kernel).  Results must be the
cold optimum whatever the slot holds; the GPU twin is tests/test_gpu_warm_ext.py."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
from common import obatch  # noqa: E402

SCALE = np.array([.02, .02, .02, .01, .01, .005, .1, .1, .1, .05, .05, .05])[:, None]


@pytest.fixture(scope="module")
def E():
    import emu_py
    emu_py.lib()
    return emu_py


@pytest.fixture(scope="module")
def W(E):
    import emu_warm_ext
    emu_warm_ext.lib()
    return emu_warm_ext


@pytest.fixture(scope="module")
def a1(E):
    return E.a1mpc


@pytest.fixture(scope="module")
def O():
    from oracle import oracle_py
    oracle_py.lib()
    return oracle_py


def _plan(a1, B, N, T, seed):
    """a gait plan of N + T steps: tick t solves steps t .. t + N - 1 (what update_plan gives, one step per tick).  Robots 0-7
    have all four feet down at step 2 (general kernel until that step leaves the horizon, then compacted); robots 8-15 lift a
    foot at step N + 1 (compacted first, general from tick 2 on)."""
    base, normals = a1.gen_schedule(B, 20, 4, seed)
    plan = base[np.arange(N + T) % 16]          # the generator's gaits have a period of 16 steps
    plan[2, 0:8] = 0b1111
    plan[N + 1, 8:16] &= 0b0001
    plan[N + 1, 8:16] |= 0b0001
    return plan, normals


def _advance(st, rng, noise):
    x0 = st["x0"].copy()
    x0[3:6] += 0.0025 * st["x0"][9:12]
    x0[0:3] += 0.0025 * st["x0"][6:9]
    x0 += noise * rng.standard_normal(x0.shape) * SCALE
    return dict(st, x0=x0)


def _absent_u(u, sched):
    """u_full entries of foot-steps that are not in contact"""
    N, B = sched.shape
    legs = (sched[:, None, :] >> (np.arange(12) // 3)[None, :, None]) & 1
    return u.reshape(N, 12, B)[legs == 0]


def _factorisations(iters):
    return iters % 100 + iters // 100


def _ticks(W, a1, O, N, B, T, shift, noise=0.03, seed=4):
    cfg, ocfg = a1.default_config(horizon=N), O.make_config(horizon=N)
    plan, normals = _plan(a1, B, N, T, seed)
    st = a1.gen_states(B, 4, seed)
    rng = np.random.default_rng(seed)
    warm = np.zeros((B, 4 + 4 * N), dtype=np.uint32)
    rows = []
    for t in range(T):
        sched = np.ascontiguousarray(plan[t:t + N])
        f, status, iters, u, stats = W.solve(cfg, st, sched=sched, normals=normals, warm=warm, shift=shift, want_u=True, order=t % 3)
        fc, sc, itc, _ = W.solve(cfg, st, sched=sched, normals=normals, warm=np.zeros_like(warm), shift=shift)   # same kernels, no guess
        fo, info = O.compute_grf_batch_ext(ocfg, obatch(O, st), sched, normals, mode=O.MODE_EXACT, nthreads=4)
        assert (status == a1.STATUS_OPTIMAL).all() and (sc == a1.STATUS_OPTIMAL).all(), (t, np.bincount(status))
        assert np.abs(f - fo).max() < 1e-7, (t, np.abs(f - fo).max())
        assert (_absent_u(u, sched) == 0).all()
        assert (warm[:, 0] == 1).all() and (warm[:, 2] == N).all() and (warm[:, 1] == sched[0]).all()
        rows.append(dict(stats=stats, hit=(iters % 100 == 0).mean(), fact=_factorisations(iters).mean(), fact_cold=_factorisations(itc).mean()))
        st = _advance(st, rng, noise)
    return rows


def test_advancing_schedules_n10(E, W, a1, O):
    """five ticks, B = 96, noise 0.03, normals, 16 robots that move between the two extended kernels.  Emulator sweep (ticks
    1-4, profiles/r03_notes.md): 62-66 % hits, 7.2-7.7 factorisations per QP against 8.1-8.2 cold"""
    rows = _ticks(W, a1, O, 10, 96, 5, shift=1)
    assert rows[0]["hit"] == 0.0                                  # no guess yet
    assert rows[0]["stats"]["general"] == 8 and rows[2]["stats"]["general"] == 16 and rows[4]["stats"]["general"] == 8
    later = rows[1:]
    assert min(r["hit"] for r in later) > 0.5
    assert np.mean([r["fact"] for r in later]) < 0.97 * np.mean([r["fact_cold"] for r in later])


def test_advancing_schedules_n20(E, W, a1, O):
    """N = 20: every robot on the general kernel (a team of warps per QP).  Sweep: 62 % hits at tick 1"""
    rows = _ticks(W, a1, O, 20, 16, 3, shift=1)
    assert rows[0]["stats"]["compact"] == 0 and rows[1]["hit"] > 0.4


def test_shift_zero_is_misaligned_but_exact(E, W, a1, O):
    """shift = 0 on an advancing plan guesses step s from the previous tick's step s: few hits (sweep: 7-13 %), same optimum"""
    rows = _ticks(W, a1, O, 10, 48, 3, shift=0)
    assert max(r["hit"] for r in rows) < 0.5


def test_slot_shared_with_constant_pattern_call(E, W, a1, O):
    """a slot written by a1mpc_solve_batch_warm is a valid guess for a1mpc_solve_batch_ext_warm and the other way round: with
    a schedule that repeats the contact mask the two calls pose the same QP, so the faces verify"""
    B, N = 64, 10
    cfg, ocfg = a1.default_config(horizon=N), O.make_config(horizon=N)
    st = a1.gen_states(B, 2, 9)
    sched = np.ascontiguousarray(np.repeat(st["contact"][None, :], N, axis=0))
    rng = np.random.default_rng(9)
    st2 = _advance(st, rng, 0.03)
    fo2, _ = O.compute_grf_batch(ocfg, obatch(O, st2), mode=O.MODE_EXACT, nthreads=4)
    for first, second in (("plain", "ext"), ("ext", "plain")):
        warm = np.zeros((B, 4 + 4 * N), dtype=np.uint32)
        for which, s in ((first, st), (second, st2)):
            solve = (lambda *a, **k: W.solve(*a, sched=sched, **k)) if which == "ext" else E.solve
            f, status, iters, _ = solve(cfg, s, warm=warm, shift=0, order=2)
        assert (status == a1.STATUS_OPTIMAL).all() and np.abs(f - fo2).max() < 1e-7
        assert (iters % 100 == 0).mean() > 0.8, (first, second, (iters % 100 == 0).mean())


def test_garbage_slot_is_no_guess(E, W, a1, O):
    """valid-looking headers and a 2-bit field equal to 3 at one foot-step: no guess (cold path), exact results"""
    B, N = 24, 10
    cfg = a1.default_config(horizon=N)
    st = a1.gen_states(B, 4, 3)
    sched, normals = a1.gen_schedule(B, N, 4, 3)
    sched[:, :4] = 0b1111                          # general kernel for four of them
    warm = np.zeros((B, 4 + 4 * N), dtype=np.uint32)
    W.solve(cfg, st, sched=sched, normals=normals, warm=warm, shift=0)
    assert (warm[:, 0] == 1).all()
    leg = np.array([int(np.flatnonzero((int(sched[5, b]) >> np.arange(4)) & 1)[0]) for b in range(B)])
    warm[np.arange(B), 4 + 4 * 5 + leg] = 0b000111   # zx field = 3 at a foot-step in contact
    f, status, iters, _ = W.solve(cfg, st, sched=sched, normals=normals, warm=warm, shift=0)
    fo, _ = O.compute_grf_batch_ext(O.make_config(horizon=N), obatch(O, st), sched, normals, mode=O.MODE_EXACT, nthreads=4)
    assert (status == a1.STATUS_OPTIMAL).all() and np.abs(f - fo).max() < 1e-7
    assert ((iters % 100) > 0).all()


def test_bad_inputs_store_no_guess(E, W, a1, O):
    """NaN inputs (NUMERICAL) and robots without a foot in contact anywhere in the horizon (NO_CONTACT) leave w[0] = 0, on
    both extended kernels"""
    B, N = 32, 10
    cfg = a1.default_config(horizon=N)
    st = a1.gen_states(B, 4, 7)
    sched, normals = a1.gen_schedule(B, N, 4, 7)
    sched[:, 4:8] = 0b0111                         # general kernel
    warm = np.zeros((B, 4 + 4 * N), dtype=np.uint32)
    W.solve(cfg, st, sched=sched, normals=normals, warm=warm, shift=1)
    assert (warm[:, 0] == 1).all()
    sched[:, 0] = 0; sched[:, 4] = 0
    st["x0"][5, 1] = np.nan; st["x0"][5, 5] = np.nan
    f, status, iters, _ = W.solve(cfg, st, sched=sched, normals=normals, warm=warm, shift=1)
    assert status[0] == a1.STATUS_NO_CONTACT and status[4] == a1.STATUS_NO_CONTACT
    assert status[1] == a1.STATUS_NUMERICAL and status[5] == a1.STATUS_NUMERICAL
    assert (warm[[0, 1, 4, 5], 0] == 0).all() and np.abs(f[:, [0, 1, 4, 5]]).max() == 0
    ok = np.ones(B, dtype=bool); ok[[0, 1, 4, 5]] = False
    assert (status[ok] == a1.STATUS_OPTIMAL).all() and (warm[ok, 0] == 1).all()


def test_lane_order_does_not_matter(W, a1):
    B, N = 40, 10
    cfg = a1.default_config(horizon=N)
    plan, normals = _plan(a1, B, N, 2, 11)
    st = a1.gen_states(B, 4, 11)
    w0 = np.zeros((B, 4 + 4 * N), dtype=np.uint32)
    W.solve(cfg, st, sched=np.ascontiguousarray(plan[0:N]), normals=normals, warm=w0, shift=1)
    st2 = _advance(st, np.random.default_rng(1), 0.03)
    sched = np.ascontiguousarray(plan[1:N + 1])
    res = []
    for order in (0, 1, 2):
        w = w0.copy()
        res.append(W.solve(cfg, st2, sched=sched, normals=normals, warm=w, shift=1, order=order, want_u=True)[:4] + (w,))
    for other in res[1:]:
        for a, b in zip(res[0], other):
            assert np.array_equal(a, b)
