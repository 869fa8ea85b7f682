#!/usr/bin/env python
"""bench.py -- convex-MPC QPs/s of the B200 engine (and, with --impl reference, of the CPU restatement
of the reference path).  One JSON line on stdout (rank 0).

A "step" is one a1mpc_solve_batch over one batch of synthetic trot-gait states:
pack -> build (linearise + condense) -> QP solve -> force extraction, for B QPs per GPU.
Default workload = BASELINE.json configs[1]: trot gait, horizon N=10, batch 1024, fp64, per GPU.
Weak scaling: every rank solves its own B QPs (independent slices, no data-path collective); for N>1 the
12 foot forces of every rank are all-gathered over NCCL after each step (config 5's final collect).

Timing: CUDA events on the handle's stream around exactly K steps after W warm-up steps, barrier + device
synchronise on both sides, max over ranks.  Inputs rotate through a ring of distinct batches larger than L2.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "a1-qp-mpc-controller_b200"))
sys.path.insert(0, ROOT)

METRIC = "convex-MPC QPs/sec (N=10, batched)"
UNIT = "QPs/s"
L2_BYTES = 126e6
IN_BYTES_PER_QP = 42 * 8 + 4     # x0[12] rot[9] foot[12] ref[9] fp64 + contact mask
OUT_BYTES_PER_QP = 12 * 8 + 4    # f_body[12] fp64 + status
ALG_BYTES_PER_QP = IN_BYTES_PER_QP + OUT_BYTES_PER_QP   # 440 B (SURVEY 8d)
DUMP_BYTES = 60 * 1000 * 1000    # --dump-outputs: below 64 MB with the .npy headers


def algorithmic_flops(N, ns_hist, fact_by_class):
    """FLOPs per launch of one class kernel.
    algorithmic (SURVEY 8d): build counted as the reference formulates it + factorizations * (n^3/3 + 4 n^2 + 30 n), n = 3*NS*N
    executed: what this engine does instead -- closed-form build (two Gram blocks + gradient), and per factorization either the
              n x n Cholesky + two solve pairs (NS <= 2) or the 6N x 6N wrench-space core + block products (NS >= 3)"""
    build = 2 * 13 ** 3 * (N - 1) + 2 * 13 * 13 * 12 * N * (N - 1) / 2 + 2 * (12 * N) ** 2 * 13 * N + 2 * 13 * N * 13 + 2 * 12 * N * 13 * N
    total_alg = 0.0
    total_exec = 0.0
    for ns, cnt in ns_hist.items():
        if ns == 0 or cnt == 0:
            continue
        n = 3 * ns * N
        it = fact_by_class.get(ns, 0.0)
        total_alg += cnt * (build + it * (n ** 3 / 3.0 + 4.0 * n * n + 30.0 * n))
        A = 3 * ns
        build_exec = 2 * 2 * 6 * A * A + 2 * 12 * n + 40 * N * N
        if ns <= 2:
            per_fact = n ** 3 / 3.0 + 4.0 * n * n + 2 * (2 * N + 2 * A) * n + 30.0 * n
        else:
            nc = 6 * N
            kr = (N * (N + 1) / 2) * (2 * 6 * 6 * 6 + 2 * 36 * 3)
            per_fact = nc ** 3 / 3.0 + kr + 4.0 * nc * nc + 4 * (2 * N + 12) * 2 * nc + 2 * (18 + 18 + 18) * ns * N * 2 + 60.0 * n
        total_exec += cnt * (build_exec + it * per_fact)
    return total_alg, total_exec


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the GPU is under load (B200_PROFILING.md recipe)"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            p = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    """torch.distributed is plumbing only: barrier + MAX over ranks of the device-timed milliseconds"""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        else:
            dist_mod.init_process_group(backend="gloo")
        dist = dist_mod
    return rank, world, local, dist


def dist_barrier(dist):
    if dist is not None:
        dist.barrier()


def dist_max(dist, value):
    if dist is None:
        return value
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def dist_bcast_bytes(dist, payload, rank):
    if dist is None:
        return payload
    obj = [payload if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0)
    return obj[0]


def cpu_reference_rate(cfg_kw, config_id, nthreads, target_seconds, O):
    """reference path restated on CPU (dense build + OSQP-algorithm at default settings, cold start) on a bounded
    sample of the same synthetic workload (same generator, same distribution), sized for ~target_seconds"""
    ocfg = O.make_config(**cfg_kw)
    probe = 16 * nthreads
    st = O.gen_states(probe, config_id, stream=777)
    sec, _ = O.time_reference_path(ocfg, O.Batch(st["x0"], st["rot"], st["foot"], st["ref"], st["contact"]), nthreads)
    rate = probe / max(sec, 1e-9)
    S = int(max(probe, min(rate * target_seconds, 4e6)))
    st = O.gen_states(S, config_id, stream=778)
    sec, _ = O.time_reference_path(ocfg, O.Batch(st["x0"], st["rot"], st["foot"], st["ref"], st["contact"]), nthreads)
    return S / sec, S, sec


def dist_allgather_obj(dist, obj, world):
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


def setup_collect(a1mpc, eng, dist, n_gpus, rank, B, mode):
    """final collect of the forces.  "peer": the solve kernels store them straight into every rank's gathered buffer (CUDA IPC peer
    mappings, stores over NVLink; a1mpc_peer_gather_*) -- a per-step wait on the step flags is all that is enqueued; "nccl": one
    ncclAllGather per step on a side stream.  Returns (description, per-step function or None, error text or None)."""
    err = None
    if mode in ("auto", "peer"):
        hd = None
        try:
            hd = eng.peer_gather_create(n_gpus, rank, B)
        except Exception as e:
            err = str(e)
        handles = dist_allgather_obj(dist, hd, n_gpus)      # every rank takes part in both exchanges whatever happened locally
        ok = 0
        if all(x is not None for x in handles):
            try:
                eng.peer_gather_connect(handles)
                ok = 1
            except Exception as e:
                err = str(e)
        if all(dist_allgather_obj(dist, ok, n_gpus)):
            return ("fused: solve-kernel epilogue stores one 96-byte record per QP into every rank's buffer over NVLink (CUDA IPC peer memory) + step flags",
                    (lambda d: eng.peer_gather_wait()), None, eng.peer_gather_buffer())
        try:
            eng.peer_gather_destroy()
        except Exception:
            pass
        err = err or "a peer rank could not map the buffers"
        if mode == "peer":
            return "unavailable", None, err, None
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        if spec and spec.submodule_search_locations:
            cand = os.path.join(list(spec.submodule_search_locations)[0], "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ.setdefault("A1MPC_NCCL_LIB", cand)
        if not getattr(eng, "_nccl_ready", False):
            uid, uerr = None, None
            if rank == 0:
                try:
                    uid = a1mpc.nccl_unique_id()
                except Exception as e:      # still take part in the broadcast: the other ranks are waiting in it
                    uerr = str(e)
            uid, uerr = dist_bcast_bytes(dist, (uid, uerr), rank)
            if uid is None:
                raise RuntimeError(uerr)
            eng.nccl_init(n_gpus, rank, uid)
            eng._nccl_ready = True
        gbuf = eng.dalloc(n_gpus * 12 * B * 8)
        return "ncclAllGather of [12][B] forces per step" + (" (peer path unavailable: %s)" % err if err else ""), (lambda d: eng.allgather_forces(d.f_body, gbuf, B)), err, gbuf
    except Exception as e:
        return "unavailable", None, "%s; nccl: %s" % (err, e), None


def verify_collect(a1mpc, eng, dist, n_gpus, rank, B, d, gbuf, qp_major):
    """after one more step + wait: block [p] of every rank's gathered buffer must be rank p's own f_body, bit for bit"""
    eng.sync()
    dist_barrier(dist)
    f, _ = d.download()
    mine = int(np.ascontiguousarray(f).view(np.uint64).sum(dtype=np.uint64))
    sums = dist_allgather_obj(dist, mine, n_gpus)
    g = np.zeros((n_gpus, 12 * B), dtype=f.dtype)
    a1mpc._check(a1mpc.lib().a1mpc_memcpy_d2h(eng.h, g.ctypes.data, gbuf, g.nbytes))
    eng.sync()
    # block [rank] is batch-major [12][B] from ncclAllGather, QP-major [B][12] from the fused peer stores
    own = g[rank].reshape(12, B) if qp_major is False else g[rank].reshape(B, 12).T
    ok = all(int(np.ascontiguousarray(g[p]).view(np.uint64).sum(dtype=np.uint64)) == sums[p] for p in range(n_gpus)) and np.array_equal(own, f)
    return bool(all(dist_allgather_obj(dist, bool(ok), n_gpus)))


def timed_steps(eng, dist, step, K, W):
    """W warm-up + exactly K timed steps, CUDA events on the handle's stream, barrier + synchronise on both sides, max over ranks"""
    for i in range(W):
        step(i)
    eng.sync()
    dist_barrier(dist)
    e0, e1 = eng.event(), eng.event()
    eng.record(e0)
    for i in range(K):
        step(W + i)
    eng.record(e1)
    eng.sync()
    dist_barrier(dist)
    return dist_max(dist, eng.elapsed_ms(e0, e1)) / K


def dump_outputs(out_dir, d, rank, world):
    """what a caller of the timed path receives from one step -- forces [12, B] and status [B] of batch `d` -- as float64 .npy files,
    so that two builds run with the same arguments can be compared output for output.  Above DUMP_BYTES (shared by the ranks) a
    fixed, seeded sample of the QPs is written, with their indices in qp_index.npy.  Ranks other than 0 add _rank<r> to the names."""
    f, status = d.download()
    arrays = {"f_body": f.astype(np.float64), "status": status.astype(np.float64)}
    B = status.shape[0]
    keep_max = DUMP_BYTES // world // (14 * 8)        # f_body[12] + status + qp_index per sampled QP
    if B * 13 * 8 > DUMP_BYTES // world:
        keep = np.sort(np.random.default_rng(0).choice(B, keep_max, replace=False))
        arrays = {"f_body": arrays["f_body"][:, keep], "status": arrays["status"][keep], "qp_index": keep.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    suffix = "_rank%d" % rank if rank else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a))


def _status_hist(a1mpc, eng, d, B):
    st = np.zeros(B, dtype=np.int32)
    a1mpc._check(a1mpc.lib().a1mpc_memcpy_d2h(eng.h, st.ctypes.data, d.status, st.nbytes))
    eng.sync()
    return {int(k): int(v) for k, v in zip(*np.unique(st, return_counts=True))}


def subrecord_config3(a1mpc, local, K=20, W=3):
    """BASELINE configs[2]: trot, N = 20, batch 8192, precision 32 (fp32 boundary arrays, fp64 + certificate inside), 1 GPU.
    4 distinct device-resident batches, L2 flushed before every step (the flush, ~40 us, is inside the timed region: < 0.3 %)."""
    B, N = 8192, 20
    eng = a1mpc.Engine(a1mpc.default_config(horizon=N, precision=32), device=local)
    dev = []
    for r in range(4):
        d = a1mpc.DeviceBatch(eng, B, want_u=False, want_iters=False)
        d.upload(a1mpc.gen_states(B, 2, stream=3000 + r))
        dev.append(d)

    def step(i):
        eng.flush_l2()
        eng.solve_ptrs(B, dev[i % 4].inp, dev[i % 4].out)
    ms = timed_steps(eng, None, step, K, W)
    rec = {"workload": "trot gait convex MPC, horizon N=20 (240x240 condensed Hessian), batch 8192, precision 32 (BASELINE configs[2])",
           "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": K, "warmup": W, "dtype": "f64 arithmetic, f32 boundary arrays (224 B/QP)",
           "status_histogram": _status_hist(a1mpc, eng, dev[0], B), "cache": "4 distinct batches, L2 flushed before every step"}
    eng.close()
    return rec


def subrecord_config4(a1mpc, local, K=20, W=3):
    """BASELINE configs[3]: randomised contact schedules (trot / bound / rotary gallop) + terrain normals, batch 16384, fp64, 1 GPU
    (an extension beyond the reference; a1mpc_solve_batch_ext with device-resident arrays)."""
    import ctypes as C
    B, N = 16384, 10
    eng = a1mpc.Engine(a1mpc.default_config(horizon=N), device=local)
    dev = []
    for r in range(4):
        d = a1mpc.DeviceBatch(eng, B, want_u=False, want_iters=False)
        d.upload(a1mpc.gen_states(B, 4, stream=4000 + r))
        sched, normals = a1mpc.gen_schedule(B, N, 4, 4000 + r)
        d.sched = eng.dalloc(sched.nbytes); d.normals = eng.dalloc(normals.nbytes)
        a1mpc._check(a1mpc.lib().a1mpc_memcpy_h2d(eng.h, d.sched, sched.ctypes.data, sched.nbytes))
        a1mpc._check(a1mpc.lib().a1mpc_memcpy_h2d(eng.h, d.normals, normals.ctypes.data, normals.nbytes))
        eng.sync()
        d.ext = a1mpc.InputsExt(d.sched, d.normals)
        dev.append(d)

    def step(i):
        d = dev[i % 4]
        eng.flush_l2()
        a1mpc._check(a1mpc.lib().a1mpc_solve_batch_ext(eng.h, B, C.byref(d.inp), C.byref(d.ext), C.byref(d.out)))
    ms = timed_steps(eng, None, step, K, W)
    rec = {"workload": "randomised contact schedule (trot/bound/gallop) + terrain normals, horizon N=10, batch 16384, fp64 (BASELINE configs[3])",
           "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": K, "warmup": W, "dtype": "f64",
           "status_histogram": _status_hist(a1mpc, eng, dev[0], B), "cache": "4 distinct batches, L2 flushed before every step"}
    eng.close()
    return rec


def subrecord_config5(a1mpc, eng, dist, n_gpus, rank, collect_mode, K=30, W=3):
    """BASELINE configs[4]: N = 10 trot, 32768 QPs per GPU (262144 at 8 GPUs), all-gather of the [12][B] forces after every step.
    Every rank takes part (the collect is a collective); device time, max over ranks."""
    B = 32768
    dev = []
    for r in range(4):
        d = a1mpc.DeviceBatch(eng, B, want_u=False, want_iters=False)
        d.upload(a1mpc.gen_states(B, 2, stream=5000 + rank * 1000003 + r))
        dev.append(d)
    desc, fn, err, gbuf = ("none", None, None, None)
    if collect_mode:
        try:
            eng.peer_gather_destroy()
        except Exception:
            pass
        desc, fn, err, gbuf = setup_collect(a1mpc, eng, dist, n_gpus, rank, B, collect_mode)

    def step(i):
        d = dev[i % 4]
        eng.solve_ptrs(B, d.inp, d.out)
        if fn is not None:
            fn(d)
    ms = timed_steps(eng, dist, step, K, W)
    peer_status = None
    try:
        peer_status = eng.peer_gather_status()
    except Exception:
        pass
    verified = None
    if fn is not None:
        step(0)
        verified = verify_collect(a1mpc, eng, dist, n_gpus, rank, B, dev[0], gbuf, desc.startswith("fused"))
    rec = {"workload": "trot gait convex MPC, horizon N=10, batch 32768 per GPU = %d QPs per step, fp64 (BASELINE configs[4])" % (B * n_gpus),
           "value": n_gpus * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": K, "warmup": W, "dtype": "f64", "n_gpus": n_gpus,
           "final_collect": desc if fn is not None else ("none" if not collect_mode else "unavailable: %s" % err), "peer_wait_timeouts": peer_status, "final_collect_verified": verified,
           "status_histogram_rank0": _status_hist(a1mpc, eng, dev[0], B),
           "cache": "4 distinct batches per rank (4 x 11 MB in, outputs 3 MB): smaller than L2, the path is compute bound (440 B against ~1 MFLOP per QP)"}
    for d in dev:
        d.free()
    return rec


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm on all usable host cores, same metric/config.  kind "port": the oracle's
    literal restatement (dense ConvexMpc build + OSQP-algorithm).  The reference's own ConvexMpc.cpp does compile here (oracle/_ref,
    against the ref_shim header stand-ins) and pins the restatement, but its matrix products would run through the stand-in's plain
    loops instead of Eigen's vectorised kernels, and OSQP itself is absent -- timing that build would misstate the reference."""
    from oracle import oracle_py as O
    rank, world, local, dist = dist_setup(args.gpus)
    if rank != 0:
        return
    # threads = the cores this process can really use (cgroup quota / affinity), not hardware_concurrency
    nthreads, core_info = O.effective_cores()
    B = args.batch
    cfg_kw = dict(horizon=args.horizon)
    ocfg = O.make_config(**cfg_kw)
    # bounded sample per step so that warmup+steps end within a few minutes
    probe = 16 * nthreads
    stp = O.gen_states(probe, 2, 777)
    sec, _ = O.time_reference_path(ocfg, O.Batch(stp["x0"], stp["rot"], stp["foot"], stp["ref"], stp["contact"]), nthreads)
    rate = probe / max(sec, 1e-9)
    budget = 150.0 / max(1, args.steps + args.warmup)
    S = int(max(16 * nthreads, rate * min(budget, 4.0)))
    st = O.gen_states(S, 2, 778)
    ob = O.Batch(st["x0"], st["rot"], st["foot"], st["ref"], st["contact"])
    for _ in range(args.warmup):
        O.time_reference_path(ocfg, ob, nthreads)
    t = 0.0
    for _ in range(args.steps):
        sec, _ = O.time_reference_path(ocfg, ob, nthreads)
        t += sec
    value = S * args.steps / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "trot gait convex MPC, horizon N=%d, batch %d per GPU, fp64 (BASELINE configs[1])" % (args.horizon, B),
                       "sample_qps_per_step": S},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "cores_detail": core_info, "kind": "port",
                             "sample": "%d synthetic QPs (same generator/distribution as the workload) per step, dense ConvexMpc build + OSQP-algorithm restatement at OSQP defaults, cold start, one QP per task" % S},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=1024, help="QPs per GPU per step (configs[1]: 1024; config 5 shard: 32768)")
    ap.add_argument("--horizon", type=int, default=10)
    ap.add_argument("--config-id", type=int, default=2, help="2: trot narrow noise, 4: wide noise")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--collect", default="auto", choices=["auto", "peer", "nccl"], help="final collect for --gpus > 1")
    ap.add_argument("--ring", type=int, default=0, help="number of distinct input batches (0: enough to exceed L2)")
    ap.add_argument("--no-subrecords", action="store_true", help="skip the config3 / config4 / config5 sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the forces and statuses of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import a1mpc
    rank, world, local, dist = dist_setup(args.gpus)
    n_gpus = world if world > 1 else 1
    B, N, K, W = args.batch, args.horizon, args.steps, args.warmup
    cfg = a1mpc.default_config(horizon=N)
    eng = a1mpc.Engine(cfg, device=local)

    # ---- ring of distinct input batches, total bytes > L2 so that no step finds its inputs cached ----
    ring = max(2, int(np.ceil(1.05 * L2_BYTES / (IN_BYTES_PER_QP * B))))     # independent of --steps
    if args.ring > 0:
        ring = args.ring                                                       # profiler runs: a short ring, labelled as such
    dev, host = [], []
    for r in range(ring):
        st = a1mpc.gen_states(B, args.config_id, stream=rank * 1000003 + r)
        d = a1mpc.DeviceBatch(eng, B, want_u=False, want_iters=(r == 0))
        d.upload(st)
        dev.append(d)
        if r < 8:
            host.append(st)
    ring_bytes = ring * IN_BYTES_PER_QP * B

    # ---- final collect of the forces (config 5): fused peer stores, NCCL all-gather as the fallback ----
    collect_desc, collect_fn, collect_err, collect_buf = "none", None, None, None
    if n_gpus > 1 and not args.no_gather:
        collect_desc, collect_fn, collect_err, collect_buf = setup_collect(a1mpc, eng, dist, n_gpus, rank, B, args.collect)

    def step(i):
        d = dev[i % ring]
        eng.solve_ptrs(B, d.inp, d.out)
        if collect_fn is not None:
            collect_fn(d)

    # ---- warm-up ----
    for i in range(W):
        step(i)
    eng.sync()
    f0, status0 = dev[0].download()
    iters0 = np.zeros(B, dtype=np.int32)
    a1mpc._check(a1mpc.lib().a1mpc_memcpy_d2h(eng.h, iters0.ctypes.data, dev[0].iters, iters0.nbytes))
    eng.sync()

    # ---- timed region: exactly K steps ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # the fp64 FMA peak of this device (roofline denominator) is measured right here: a burst of dense DFMA that also
    # brings the SM clock out of idle before a short timed region
    fp64_peak = eng.fp64_peak_tflops()
    e0, e1 = eng.event(), eng.event()
    launches0 = eng.launches()
    eng.profile_begin(K)
    dist_barrier(dist)
    eng.sync()
    t_wall0 = time.time()
    eng.record(e0)
    for i in range(K):
        step(W + i)
    eng.record(e1)
    eng.sync()
    dist_barrier(dist)
    t_wall1 = time.time()
    ms_local = eng.elapsed_ms(e0, e1)
    class_ms, ncalls = eng.profile_end()
    launches = eng.launches() - launches0
    ms = dist_max(dist, ms_local)
    value = n_gpus * B * K / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dev[(W + K - 1) % ring], rank, n_gpus)     # before the passes below overwrite the ring's outputs

    collect_ok = None
    if collect_fn is not None:
        step(0)
        collect_ok = verify_collect(a1mpc, eng, dist, n_gpus, rank, B, dev[0], collect_buf, collect_desc.startswith("fused"))

    # ---- per-step latency distribution (p50 solve us), separate pass with a sync per step ----
    lat = []
    ea, eb = eng.event(), eng.event()
    for i in range(min(K, 300)):
        eng.record(ea)
        step(i)
        eng.record(eb)
        lat.append(eng.elapsed_ms(ea, eb) * 1e3)
    lat = np.array(lat)

    # ---- end to end through the public host-pointer call: pinned host inputs, H2D + solve + D2H each step ----
    hp = []
    for st in host:
        p = {k: eng.pinned_array(st[k].shape, st[k].dtype) for k in st}
        for k in st:
            p[k][...] = st[k]
        hp.append(p)
    f_pin = eng.pinned_array((12, B), np.float64)
    s_pin = eng.pinned_array((B,), np.int32)
    Ke = min(K, 400)

    def e2e_step(i):
        p = hp[i % len(hp)]
        inp = a1mpc.Inputs(p["x0"].ctypes.data, p["rot"].ctypes.data, p["foot"].ctypes.data, p["ref"].ctypes.data, p["contact"].ctypes.data, B)
        out = a1mpc.Outputs(f_pin.ctypes.data, s_pin.ctypes.data, None, None, B)
        eng.solve_ptrs(B, inp, out)

    for i in range(3):
        e2e_step(i)
    dist_barrier(dist)
    eng.sync()
    tw0 = time.time()
    eng.record(e0)
    for i in range(Ke):
        e2e_step(i)
    eng.record(e1)
    eng.sync()
    dist_barrier(dist)
    e2e_ms = dist_max(dist, eng.elapsed_ms(e0, e1))
    e2e_wall = time.time() - tw0
    e2e_value = n_gpus * B * Ke / (max(e2e_ms, 1e3 * 0) * 1e-3)
    clocks = sampler.stop(t_wall0, time.time()) if rank == 0 else None

    # ---- sub-records: the other BASELINE configs at their stated sizes (outside the headline's timed region) ----
    sub = {}
    if not args.no_subrecords and B == 1024 and N == 10:
        if n_gpus > 1:
            sub["config5"] = subrecord_config5(a1mpc, eng, dist, n_gpus, rank, args.collect if collect_fn is not None else None)
        elif rank == 0:
            sub["config3"] = subrecord_config3(a1mpc, local)
            sub["config4"] = subrecord_config4(a1mpc, local)

    if rank != 0:
        return
    # ---- the plugin-level call a user of the reference makes, with pageable memory (C++ shim, its own process) ----
    plugin = None
    exe = os.path.join(ROOT, "tests", "cpp", "bench_compute_grf")
    if n_gpus == 1 and not args.no_subrecords and os.path.exists(exe):
        try:
            eng.sync()
            r = subprocess.run([exe, str(B), "200", "5"], capture_output=True, text=True, timeout=120)
            plugin = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            plugin = {"unavailable": str(e)}
    # ---- roofline of the dominant kernel (most device time among the class kernels) ----
    ns_of = np.array([bin(int(c) & 15).count("1") for c in host[0]["contact"]])
    hist = {ns: int((ns_of == ns).sum()) for ns in range(5)}
    dom = int(np.argmax(class_ms)) + 1
    dom_ms = class_ms[dom - 1] / max(ncalls, 1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    dom_qps = hist.get(dom, 0)
    achieved_gbs = ALG_BYTES_PER_QP * dom_qps / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    it_by_class = {}
    for ns in range(1, 5):
        m = ns_of == ns
        if m.any():
            it_by_class[ns] = float(np.mean(iters0[m] % 100 + iters0[m] // 100))   # factorizations per QP
    fl_alg, fl_exec = algorithmic_flops(N, {dom: dom_qps}, it_by_class)
    traffic = None
    traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = tj.get("kernels", {}).get("solve_kernel<NS=%d,N=%d>@%d" % (dom, N, B))
        if ent:
            traffic = ent["dram_bytes_read"] + ent["dram_bytes_write"]
            traffic_src = "ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch of %s (%s; tools/make_traffic_json.py)" % (ent["ncu_kernel_name"], tj.get("source"))
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "solve_kernel<NS=%d,N=%d>" % (dom, N), "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved_gbs / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src,
                "algorithmic_bytes_per_qp": ALG_BYTES_PER_QP, "qps_per_launch": dom_qps, "kernel_ms": dom_ms,
                "note": "the path is fp64-pipe/latency bound (SURVEY 8d: ~1e4 FLOP/B), so the HBM fraction is small by construction; see roofline_fp64"}
    roofline_fp64 = {"bound": "fp64 pipes (DFMA + DMMA.8x8x4; the tensor and the vector fp64 peak of a B200 are about equal)", "kernel": roofline["kernel"], "unit": "TFLOP/s",
                     "achieved_algorithmic": fl_alg / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0,
                     "achieved_executed": fl_exec / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0,
                     "peak": fp64_peak, "peak_source": "measured in this run (a1mpc_measure_fp64_peak: dependent-free DFMA stream)",
                     "frac": (fl_exec / (dom_ms * 1e-3) / 1e12) / fp64_peak if dom_ms > 0 and fp64_peak > 0 else None,
                     "factorizations_per_qp": it_by_class}
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import oracle_py as O
        nthreads, core_info = O.effective_cores()
        v, S, sec = cpu_reference_rate(dict(horizon=N), args.config_id, nthreads, args.cpu_seconds, O)
        v1, S1, sec1 = cpu_reference_rate(dict(horizon=N), args.config_id, 1, 2.0, O)
        cpu = {"value": v, "unit": UNIT, "cores": nthreads, "cores_detail": core_info, "kind": "port",
               "sample": "%d synthetic QPs (same generator/distribution as the step batch) in %.1f s; dense ConvexMpc build + OSQP-algorithm restatement at OSQP defaults (eps 1e-3), cold start" % (S, sec),
               "single_thread_value": v1}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "trot gait convex MPC, horizon N=%d, batch %d per GPU, fp64 (BASELINE configs[1]%s)" % (N, B, "" if (B == 1024 and N == 10) else " variant"),
                       "horizon": N, "batch_per_gpu": B, "global_batch": B * n_gpus, "generator": "a1mpc_gen_states config_id=%d" % args.config_id,
                       "cache": "inputs rotate through a ring of %d distinct batches = %.0f MB %s L2 (126 MB)" % (ring, ring_bytes / 1e6, ">" if ring_bytes > L2_BYTES else "< (NOT larger than)"),
                       "stance_feet_histogram": hist,
                       "final_collect_verified": collect_ok,
                       "final_collect": (collect_desc if collect_fn is not None else ("none" if n_gpus == 1 or args.no_gather else "unavailable: %s" % collect_err))},
            "p50_solve_us": float(np.percentile(lat, 50)), "p99_solve_us": float(np.percentile(lat, 99)),
            "p50_solve_us_per_qp": float(np.percentile(lat, 50)) / B,
            "status_histogram": {int(k): int(v) for k, v in zip(*np.unique(status0, return_counts=True))},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": IN_BYTES_PER_QP * B, "d2h_bytes_per_step": OUT_BYTES_PER_QP * B,
                    "steps": Ke, "wall_s": e2e_wall},
            "gpu_launches": launches,
            "roofline": roofline, "roofline_fp64": roofline_fp64, "cpu_baseline": cpu, "clocks": clocks,
            "class_kernel_ms_per_step": {int(i + 1): float(class_ms[i] / max(ncalls, 1)) for i in range(4)}}
    line.update(sub)
    if plugin is not None:
        line["e2e_plugin_pageable"] = plugin
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
    try:
        import torch.distributed as _d
        if _d.is_available() and _d.is_initialized():
            _d.destroy_process_group()
    except Exception:
        pass
