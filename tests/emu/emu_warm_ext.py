"""ctypes binding of the extended warm start on the CPU block emulator (emu_warm_ext.cpp -> liba1mpc_emu_warm_ext.so).
TEST INFRASTRUCTURE: the device code of a1mpc_solve_batch_ext_warm compiled by g++ against cuda_emu.h, with the flags of
tests/emu/Makefile; rebuilt when a source is newer than the library."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

import emu_py

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(emu_py.ROOT, "a1-qp-mpc-controller_b200", "csrc")
_LIB = os.path.join(_HERE, "liba1mpc_emu_warm_ext.so")
_SRC = ["emu_warm_ext.cpp", "cuda_emu.cpp"]
_lib = None

a1mpc = emu_py.a1mpc


def lib():
    global _lib
    if _lib is None:
        deps = [os.path.join(_HERE, f) for f in _SRC + ["cuda_emu.h"]] + glob.glob(os.path.join(_CSRC, "*"))
        deps.append(os.path.join(emu_py.ROOT, "include", "a1mpc.h"))
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps):
            tmp = _LIB + ".%d.tmp" % os.getpid()
            subprocess.check_call(["g++", "-std=c++17", "-O1", "-mfma", "-march=x86-64-v3", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                                   "-Wno-attributes", "-o", tmp] + _SRC + ["-lpthread", "-l:libstdc++.so.6", "-lm"], cwd=_HERE)
            os.replace(tmp, _LIB)
        _lib = C.CDLL(_LIB)
    return _lib


def solve(cfg, st, warm, sched=None, normals=None, shift=1, compact=True, order=0, nthreads=8, want_u=False):
    """a1mpc_solve_batch_ext_warm on the emulator.  st: dict x0[12,B] rot[9,B] foot[12,B] ref[9,B] contact[B]; warm: host
    uint32 [B, 4 + 4N], updated in place.  Returns f_body[12,B], status[B], iters[B] (, u_full[12N,B]) and
    {"general": QPs on the general kernel, "compact": QPs on the compacted kernel}"""
    B = st["contact"].shape[0]
    assert warm.dtype == np.uint32 and warm.shape == (B, 4 + 4 * cfg.horizon) and warm.flags["C_CONTIGUOUS"]
    p = emu_py._p
    arrs = [np.ascontiguousarray(st[k], dtype=np.float64) for k in ("x0", "rot", "foot", "ref")]
    contact = np.ascontiguousarray(st["contact"], dtype=np.uint32)
    inp = a1mpc.Inputs(p(arrs[0]), p(arrs[1]), p(arrs[2]), p(arrs[3]), p(contact), B)
    f = np.zeros((12, B)); status = np.full(B, -7, dtype=np.int32); iters = np.zeros(B, dtype=np.int32)
    u = np.zeros((12 * cfg.horizon, B)) if want_u else None
    out = a1mpc.Outputs(p(f), p(status), p(iters), p(u), B)
    sc = np.ascontiguousarray(sched, dtype=np.uint32) if sched is not None else None
    nm = np.ascontiguousarray(normals, dtype=np.float64) if normals is not None else None
    queued = (C.c_int * 2)()
    rc = lib().emu_solve_ext_warm(C.byref(cfg), B, C.byref(inp), p(sc), p(nm), C.byref(out), p(warm), int(shift), int(compact), order, nthreads,
                                  queued)
    assert rc == 0, rc
    return (f, status, iters) + ((u,) if want_u else ()) + ({"general": int(queued[0]), "compact": int(queued[1])},)
