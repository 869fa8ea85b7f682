"""dev tool: closed-loop throughput of the device-resident warm start (a1mpc_solve_batch_warm) next to the cold path.
A ring of T consecutive control ticks (state advanced by dt plus a random walk of sensor-level noise) is uploaded once; the
timed loop walks the ring.  Not part of bench.py's contract (that measures independent QPs, i.e. the cold path).

    python tools/warm_bench.py [B] [noise]      constant contact pattern (a1mpc_solve_batch / _warm, shift 0)
    python tools/warm_bench.py --ext [B ...]    scheduled ticks: a1mpc_solve_batch_ext / _ext_warm (shift 1) with per-step
                                                schedules that advance one step per tick and terrain normals, at noise 0.03
                                                and 0.1, next to the constant-pattern pair on the same states"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "a1-qp-mpc-controller_b200")); sys.path.insert(0, ROOT)
import a1mpc

if "--ext" in sys.argv:
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import warm_bench_ext
    warm_bench_ext.main([int(a) for a in sys.argv[1:] if a != "--ext"] or [1024, 16384])
    sys.exit(0)

B = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
noise = float(sys.argv[2]) if len(sys.argv) > 2 else 0.1
T = 32
eng = a1mpc.Engine(a1mpc.default_config(horizon=10))
rng = np.random.default_rng(0)
st = a1mpc.gen_states(B, 2, 3)
scale = np.array([.02, .02, .02, .01, .01, .005, .1, .1, .1, .05, .05, .05])[:, None]
ticks = []
for t in range(T):
    d = a1mpc.DeviceBatch(eng, B); d.upload(st); ticks.append(d)
    st = {k: v.copy() for k, v in st.items()}
    st["x0"][3:6] += 0.0025 * st["x0"][9:12]; st["x0"][0:3] += 0.0025 * st["x0"][6:9]
    st["x0"] += noise * rng.standard_normal(st["x0"].shape) * scale
warm = eng.warm_alloc(B)
lib = a1mpc.lib()


def run(use_warm, reps):
    e0, e1 = eng.event(), eng.event()
    for t in range(T):   # warm-up lap
        if use_warm: a1mpc._check(lib.a1mpc_solve_batch_warm(eng.h, B, C.byref(ticks[t].inp), C.byref(ticks[t].out), warm, 0))
        else: eng.solve_ptrs(B, ticks[t].inp, ticks[t].out)
    eng.sync(); eng.record(e0)
    for r in range(reps):
        t = r % T
        if use_warm: a1mpc._check(lib.a1mpc_solve_batch_warm(eng.h, B, C.byref(ticks[t].inp), C.byref(ticks[t].out), warm, 0))
        else: eng.solve_ptrs(B, ticks[t].inp, ticks[t].out)
    eng.record(e1); eng.sync()
    return eng.elapsed_ms(e0, e1) / reps


for name, w in (("cold", False), ("warm", True)):
    ms = run(w, 4 * T)
    f, status = ticks[(4 * T - 1) % T].download()
    print("B=%d noise %.2f %s: %.3f ms/tick  %.0f QPs/s  optimal %.4f" % (B, noise, name, ms, B / ms * 1e3, (status == 0).mean()), flush=True)
