"""dev tool (tools/warm_bench.py --ext): closed-loop throughput of the warm-started extended call next to the cold one.

A ring of T = 32 control ticks is uploaded once per batch size and noise level: config-4 states (advanced by dt plus a random
walk of sensor-level noise), per-step contact schedules that advance one plan step per tick (the generator's gaits have a
period of 16 steps, so the ring closes on the schedule; the state jumps back once per lap) and terrain normals.  Four modes
on the same ring, alternated in rounds: cold / warm extended call (shift 1), and the constant-pattern pair a1mpc_solve_batch /
a1mpc_solve_batch_warm (shift 0) on the same states with each robot's first-step contact mask.  Per mode: ms per tick (device
events, median of the rounds), QPs/s, hit rate (no interior-point iteration) and factorisations per QP over one lap, and the
largest force difference to the cold call of the same kind at the last tick of that lap."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "a1-qp-mpc-controller_b200")); sys.path.insert(0, ROOT)
import a1mpc  # noqa: E402

N, T, ROUNDS = 10, 32, 3
SCALE = np.array([.02, .02, .02, .01, .01, .005, .1, .1, .1, .05, .05, .05])[:, None]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:   # the numbers below are still device-event timings; say that the card could not be read
        return "card not read (%s)" % e


class Ring:
    def __init__(self, eng, B, noise, seed=3):
        self.eng, self.B = eng, B
        lib = a1mpc.lib()
        rng = np.random.default_rng(seed)
        st = a1mpc.gen_states(B, 4, seed)
        base, normals = a1mpc.gen_schedule(B, 20, 4, seed)
        plan = np.ascontiguousarray(base[np.arange(T + N) % 16])
        self.dnorm = eng.dalloc(normals.nbytes)
        a1mpc._check(lib.a1mpc_memcpy_h2d(eng.h, self.dnorm, normals.ctypes.data_as(C.c_void_p), normals.nbytes))
        self.ticks, self.sched = [], []
        for t in range(T):
            sched = np.ascontiguousarray(plan[t:t + N])
            st = dict(st, contact=np.ascontiguousarray(sched[0]))
            d = a1mpc.DeviceBatch(eng, B); d.upload(st); self.ticks.append(d)
            ds = eng.dalloc(sched.nbytes)
            a1mpc._check(lib.a1mpc_memcpy_h2d(eng.h, ds, sched.ctypes.data_as(C.c_void_p), sched.nbytes))
            self.sched.append(ds)
            x0 = st["x0"].copy()
            x0[3:6] += 0.0025 * st["x0"][9:12]; x0[0:3] += 0.0025 * st["x0"][6:9]
            x0 += noise * rng.standard_normal(x0.shape) * SCALE
            st = dict(st, x0=x0)
        self.warm = {m: eng.warm_alloc(B) for m in ("warm_ext", "warm")}

    def call(self, mode, t):
        lib, d = a1mpc.lib(), self.ticks[t]
        if mode.endswith("ext"):
            ext = a1mpc.InputsExt(self.sched[t], self.dnorm)
            if mode == "warm_ext": rc = lib.a1mpc_solve_batch_ext_warm(self.eng.h, self.B, C.byref(d.inp), C.byref(ext), C.byref(d.out), self.warm[mode], 1)
            else: rc = lib.a1mpc_solve_batch_ext(self.eng.h, self.B, C.byref(d.inp), C.byref(ext), C.byref(d.out))
        elif mode == "warm": rc = lib.a1mpc_solve_batch_warm(self.eng.h, self.B, C.byref(d.inp), C.byref(d.out), self.warm[mode], 0)
        else: rc = lib.a1mpc_solve_batch(self.eng.h, self.B, C.byref(d.inp), C.byref(d.out))
        a1mpc._check(rc)

    def timed_lap(self, mode, laps):
        e0, e1 = self.eng.event(), self.eng.event()
        self.eng.sync(); self.eng.record(e0)
        for r in range(laps * T):
            self.call(mode, r % T)
        self.eng.record(e1); self.eng.sync()
        return self.eng.elapsed_ms(e0, e1) / (laps * T)

    def stats_lap(self, mode):
        """one more lap, results downloaded per tick: hit rate, factorisations per QP, statuses; forces of the last tick"""
        lib = a1mpc.lib()
        hit = fact = 0.0; bad = 0
        for t in range(T):
            self.call(mode, t)
            f, status = self.ticks[t].download()
            it = np.zeros(self.B, dtype=np.int32)
            a1mpc._check(lib.a1mpc_memcpy_d2h(self.eng.h, it.ctypes.data_as(C.c_void_p), self.ticks[t].iters, it.nbytes)); self.eng.sync()
            ok = status == a1mpc.STATUS_OPTIMAL
            bad += int((~ok).sum())
            hit += (it[ok] % 100 == 0).mean() / T; fact += (it[ok] % 100 + it[ok] // 100).mean() / T
        return hit, fact, bad, f


def main(sizes):
    print("# tools/warm_bench.py --ext   %s   N = %d, ring of %d ticks, %d alternated rounds of %d ticks per mode" % (card(), N, T, ROUNDS, 2 * T), flush=True)
    eng = a1mpc.Engine(a1mpc.default_config(horizon=N))
    modes = ("cold_ext", "warm_ext", "cold", "warm")
    for B in sizes:
        for noise in (0.03, 0.1):
            ring = Ring(eng, B, noise)
            for m in modes:                       # warm-up lap of every mode (module loads, first-touch of the slots)
                ring.timed_lap(m, 1)
            ms = {m: [] for m in modes}
            for _ in range(ROUNDS):
                for m in modes:
                    ms[m].append(ring.timed_lap(m, 2))
            res = {m: ring.stats_lap(m) for m in modes}
            for m in modes:
                hit, fact, bad, f = res[m]
                ref = res["cold_ext" if m.endswith("ext") else "cold"][3]
                t = float(np.median(ms[m]))
                print("B=%5d noise %.2f %-8s %7.3f ms/tick (rounds %s)  %6.2f M QPs/s  hits %5.1f %%  %5.2f factorisations/QP  not optimal %d  max|f - cold| %.1e N"
                      % (B, noise, m, t, " ".join("%.3f" % v for v in ms[m]), B / t * 1e-3, 100 * hit, fact, bad, np.abs(f - ref).max()), flush=True)
            for d in ring.ticks: d.free()
            for p in ring.sched + [ring.dnorm] + list(ring.warm.values()): a1mpc.lib().a1mpc_device_free(eng.h, p)
    eng.close()
