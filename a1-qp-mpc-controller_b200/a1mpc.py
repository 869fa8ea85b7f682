"""ctypes binding of liba1mpc.so (the C ABI in include/a1mpc.h).

This file is glue for tests/ and bench.py: it marshals numpy arrays to the C entry points and nothing
else.  There is no Python compute path and no fallback: if the shared library is missing or no B200 is
visible, construction fails loudly.  C++ hosts use include/a1mpc.h (or the ConvexMpcBatch /
A1RobotControlBatch shims under host/) directly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("A1MPC_LIB", os.path.join(_HERE, "liba1mpc.so"))   # A1MPC_LIB: developer A/B builds only

STATUS_OPTIMAL, STATUS_IPM_ONLY, STATUS_MAXITER, STATUS_NUMERICAL, STATUS_NO_CONTACT = 0, 1, 2, 3, 4

EXPORTS = [
    "a1mpc_default_config", "a1mpc_create", "a1mpc_destroy", "a1mpc_last_error", "a1mpc_device_count",
    "a1mpc_solve_batch", "a1mpc_warm_bytes", "a1mpc_warm_reset", "a1mpc_solve_batch_warm", "a1mpc_solve_batch_ext", "a1mpc_solve_batch_ext_warm", "a1mpc_build_qp_batch", "a1mpc_qp_mats_batch", "a1mpc_solve_dense_batch",
    "a1mpc_grf_qp_batch", "a1mpc_joint_torques_batch", "a1mpc_leg_kinematics_batch", "a1mpc_ekf_bytes", "a1mpc_ekf_init_batch", "a1mpc_ekf_update_batch", "a1mpc_update_plan_batch", "a1mpc_device_alloc", "a1mpc_device_free", "a1mpc_host_alloc", "a1mpc_host_free",
    "a1mpc_memcpy_h2d", "a1mpc_memcpy_d2h", "a1mpc_sync", "a1mpc_event_create", "a1mpc_event_destroy",
    "a1mpc_event_record", "a1mpc_event_elapsed_ms", "a1mpc_launch_count", "a1mpc_measure_fp64_peak",
    "a1mpc_flush_l2", "a1mpc_profile_begin", "a1mpc_profile_end", "a1mpc_nccl_unique_id", "a1mpc_nccl_init", "a1mpc_allgather_forces",
    "a1mpc_qp_rollout_batch", "a1mpc_peer_gather_create", "a1mpc_peer_gather_connect", "a1mpc_peer_gather_buffer", "a1mpc_peer_gather_wait", "a1mpc_peer_gather_status", "a1mpc_peer_gather_destroy", "a1mpc_gen_states", "a1mpc_gen_schedule",
]


class Config(C.Structure):
    _fields_ = [("horizon", C.c_int), ("precision", C.c_int), ("dt", C.c_double),
                ("mu", C.c_double), ("fz_min", C.c_double), ("fz_max", C.c_double),
                ("mass", C.c_double), ("inertia", C.c_double * 9),
                ("q", C.c_double * 13), ("r", C.c_double * 12),
                ("max_iter", C.c_int), ("tol", C.c_double)]


class Inputs(C.Structure):
    _fields_ = [("x0", C.c_void_p), ("rot", C.c_void_p), ("foot", C.c_void_p), ("ref", C.c_void_p),
                ("contact", C.c_void_p), ("ld", C.c_size_t)]


class GaitParams(C.Structure):
    _fields_ = [("counter_per_gait", C.c_double), ("counter_per_swing", C.c_double), ("control_dt", C.c_double),
                ("default_foot_pos", C.c_double * 12), ("foot_delta_x_limit", C.c_double), ("foot_delta_y_limit", C.c_double),
                ("horizon", C.c_int)]


def default_gait_params(horizon=10):
    """A1CtrlStates.h:23-24, 45-47, 332; A1Params.h:44-45"""
    g = GaitParams()
    g.counter_per_gait, g.counter_per_swing, g.control_dt = 240.0, 120.0, 0.0025
    g.default_foot_pos[:] = [0.17, 0.17, -0.17, -0.17, 0.15, -0.15, 0.15, -0.15, -0.35, -0.35, -0.35, -0.35]
    g.foot_delta_x_limit, g.foot_delta_y_limit, g.horizon = 0.1, 0.1, horizon
    return g


class InputsExt(C.Structure):
    _fields_ = [("contact_sched", C.c_void_p), ("normals", C.c_void_p)]


class Outputs(C.Structure):
    _fields_ = [("f_body", C.c_void_p), ("status", C.c_void_p), ("iters", C.c_void_p), ("u_full", C.c_void_p),
                ("ld", C.c_size_t)]


_lib = None


def lib():
    """loads liba1mpc.so; raises if it has not been built (python __graft_entry__.py build / make)"""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("liba1mpc.so is missing: run `make` (or __graft_entry__.build()) first; "
                               "there is no Python/CPU fallback for the engine")
        l = C.CDLL(LIB_PATH)
        l.a1mpc_last_error.restype = C.c_char_p
        l.a1mpc_launch_count.restype = C.c_int64
        l.a1mpc_warm_bytes.restype = C.c_size_t
        l.a1mpc_ekf_bytes.restype = C.c_size_t
        l.a1mpc_launch_count.argtypes = [C.c_void_p]
        for name in ("a1mpc_device_alloc", "a1mpc_host_alloc"):
            getattr(l, name).argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        for name in ("a1mpc_device_free", "a1mpc_host_free", "a1mpc_event_destroy", "a1mpc_event_record"):
            getattr(l, name).argtypes = [C.c_void_p, C.c_void_p]
        for name in ("a1mpc_memcpy_h2d", "a1mpc_memcpy_d2h"):
            getattr(l, name).argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        l.a1mpc_sync.argtypes = [C.c_void_p]
        l.a1mpc_flush_l2.argtypes = [C.c_void_p]
        l.a1mpc_peer_gather_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        l.a1mpc_peer_gather_connect.argtypes = [C.c_void_p, C.c_char_p]
        l.a1mpc_peer_gather_buffer.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        l.a1mpc_peer_gather_wait.argtypes = [C.c_void_p]
        l.a1mpc_peer_gather_status.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        l.a1mpc_peer_gather_destroy.argtypes = [C.c_void_p]
        l.a1mpc_destroy.argtypes = [C.c_void_p]
        l.a1mpc_event_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        l.a1mpc_event_elapsed_ms.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        l.a1mpc_solve_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(Inputs), C.POINTER(Outputs)]
        l.a1mpc_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(Config), C.c_int]
        l.a1mpc_default_config.argtypes = [C.POINTER(Config)]
        l.a1mpc_warm_bytes.argtypes = [C.c_void_p, C.c_int]
        l.a1mpc_warm_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        l.a1mpc_solve_batch_warm.argtypes = [C.c_void_p, C.c_int, C.POINTER(Inputs), C.POINTER(Outputs), C.c_void_p, C.c_int]
        l.a1mpc_leg_kinematics_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 10
        l.a1mpc_ekf_bytes.argtypes = [C.c_int]
        l.a1mpc_ekf_init_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        l.a1mpc_ekf_update_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_int] + [C.c_void_p] * 11
        l.a1mpc_solve_batch_ext.argtypes = [C.c_void_p, C.c_int, C.POINTER(Inputs), C.POINTER(InputsExt), C.POINTER(Outputs)]
        l.a1mpc_solve_batch_ext_warm.argtypes = [C.c_void_p, C.c_int, C.POINTER(Inputs), C.POINTER(InputsExt), C.POINTER(Outputs), C.c_void_p, C.c_int]
        l.a1mpc_gen_schedule.argtypes = [C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        l.a1mpc_build_qp_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(Inputs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.a1mpc_qp_mats_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 6
        l.a1mpc_qp_rollout_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
        l.a1mpc_solve_dense_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 5
        l.a1mpc_grf_qp_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 7
        l.a1mpc_joint_torques_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 7
        l.a1mpc_update_plan_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(GaitParams)] + [C.c_void_p] * 13
        l.a1mpc_gen_states.argtypes = [C.c_int, C.c_uint64, C.c_int] + [C.c_void_p] * 5
        l.a1mpc_measure_fp64_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        l.a1mpc_profile_begin.argtypes = [C.c_void_p, C.c_int]
        l.a1mpc_profile_end.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
        l.a1mpc_nccl_unique_id.argtypes = [C.c_void_p]
        l.a1mpc_nccl_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        l.a1mpc_allgather_forces.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        _lib = l
    return _lib


class A1MpcError(RuntimeError):
    pass


def _check(rc):
    if rc != 0:
        raise A1MpcError("a1mpc error %d: %s" % (rc, (lib().a1mpc_last_error() or b"").decode()))


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_config(**kw):
    c = Config()
    lib().a1mpc_default_config(C.byref(c))
    for k, v in kw.items():
        if k in ("inertia", "q", "r"):
            getattr(c, k)[:] = v
        else:
            setattr(c, k, v)
    return c


def gen_states(B, config_id=2, stream=0):
    """deterministic synthetic trot-gait batch (SURVEY 8d) -> dict of host SoA arrays"""
    x0 = np.zeros((12, B)); rot = np.zeros((9, B)); foot = np.zeros((12, B)); ref = np.zeros((9, B))
    contact = np.zeros(B, dtype=np.uint32)
    rc = lib().a1mpc_gen_states(config_id, stream, B, _p(x0), _p(rot), _p(foot), _p(ref), _p(contact))
    _check(rc)
    return dict(x0=x0, rot=rot, foot=foot, ref=ref, contact=contact)


def gen_schedule(B, horizon, config_id=4, stream=0):
    """config-4 extras: per-step contact schedule [N,B] and per-foot terrain normals [12,B]"""
    sched = np.zeros((horizon, B), dtype=np.uint32); normals = np.zeros((12, B))
    _check(lib().a1mpc_gen_schedule(config_id, stream, B, horizon, _p(sched), _p(normals)))
    return sched, normals


class DeviceBatch:
    """device-resident SoA inputs + outputs of one batch (ld = B)"""

    def __init__(self, eng, B, want_u=False, want_iters=True):
        self.eng, self.B = eng, B
        N = eng.cfg.horizon
        es = np.dtype(eng.ftype).itemsize
        self.x0 = eng.dalloc(12 * B * es); self.rot = eng.dalloc(9 * B * es); self.foot = eng.dalloc(12 * B * es)
        self.ref = eng.dalloc(9 * B * es); self.contact = eng.dalloc(B * 4)
        self.f_body = eng.dalloc(12 * B * es); self.status = eng.dalloc(B * 4)
        self.iters = eng.dalloc(B * 4) if want_iters else None
        self.u_full = eng.dalloc(12 * N * B * es) if want_u else None
        self.inp = Inputs(self.x0, self.rot, self.foot, self.ref, self.contact, B)
        self.out = Outputs(self.f_body, self.status, self.iters, self.u_full, B)

    def upload(self, st):
        e = self.eng
        for name in ("x0", "rot", "foot", "ref", "contact"):
            a = np.ascontiguousarray(st[name], dtype=(np.uint32 if name == "contact" else e.ftype))
            _check(lib().a1mpc_memcpy_h2d(e.h, getattr(self, name), _p(a), a.nbytes))
        e.sync()

    def download(self):
        e, B = self.eng, self.B
        f = np.zeros((12, B), dtype=e.ftype); status = np.zeros(B, dtype=np.int32)
        _check(lib().a1mpc_memcpy_d2h(e.h, _p(f), self.f_body, f.nbytes))
        _check(lib().a1mpc_memcpy_d2h(e.h, _p(status), self.status, status.nbytes))
        e.sync()
        return f, status

    def free(self):
        for name in ("x0", "rot", "foot", "ref", "contact", "f_body", "status", "iters", "u_full"):
            p = getattr(self, name)
            if p:
                lib().a1mpc_device_free(self.eng.h, p)
                setattr(self, name, None)


class Engine:
    """one handle = one B200 + one stream (a1mpc_create / a1mpc_destroy)"""

    def __init__(self, cfg=None, device=0):
        self.cfg = cfg if cfg is not None else default_config()
        h = C.c_void_p()
        _check(lib().a1mpc_create(C.byref(h), C.byref(self.cfg), device))
        self.h = h
        self.device = device

    @property
    def ftype(self):
        """element type of the hot-path boundary arrays (a1mpc_config::precision)"""
        return np.float32 if self.cfg.precision == 32 else np.float64

    def close(self):
        if self.h:
            lib().a1mpc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- hot path ----
    def solve(self, st, want_u=False):
        """host arrays in, host arrays out (H2D + kernels + D2H inside the call)"""
        B = st["x0"].shape[1]
        N = self.cfg.horizon
        ft = self.ftype     # float32 arrays at the boundary when cfg.precision == 32
        a = {k: np.ascontiguousarray(st[k], dtype=(np.uint32 if k == "contact" else ft)) for k in ("x0", "rot", "foot", "ref", "contact")}
        f = np.zeros((12, B), dtype=ft); status = np.zeros(B, dtype=np.int32); iters = np.zeros(B, dtype=np.int32)
        u = np.zeros((12 * N, B), dtype=ft) if want_u else None
        inp = Inputs(_p(a["x0"]), _p(a["rot"]), _p(a["foot"]), _p(a["ref"]), _p(a["contact"]), B)
        out = Outputs(_p(f), _p(status), _p(iters), _p(u), B)
        _check(lib().a1mpc_solve_batch(self.h, B, C.byref(inp), C.byref(out)))
        return (f, status, iters, u) if want_u else (f, status, iters)

    def warm_alloc(self, B):
        """device-resident warm-start state for B robots (no guess yet); free with a1mpc_device_free / Engine.dfree"""
        nbytes = lib().a1mpc_warm_bytes(self.h, B)
        p = self.dalloc(nbytes)
        _check(lib().a1mpc_warm_reset(self.h, p, B))
        return p

    def solve_warm(self, st, warm, shift=0):
        """a1mpc_solve_batch_warm: host arrays in/out, `warm` from warm_alloc (updated in place on the device)"""
        B = st["x0"].shape[1]
        a = {k: np.ascontiguousarray(st[k], dtype=(np.uint32 if k == "contact" else self.ftype)) for k in ("x0", "rot", "foot", "ref", "contact")}
        f = np.zeros((12, B), dtype=self.ftype); status = np.zeros(B, dtype=np.int32); iters = np.zeros(B, dtype=np.int32)
        inp = Inputs(_p(a["x0"]), _p(a["rot"]), _p(a["foot"]), _p(a["ref"]), _p(a["contact"]), B)
        out = Outputs(_p(f), _p(status), _p(iters), None, B)
        _check(lib().a1mpc_solve_batch_warm(self.h, B, C.byref(inp), C.byref(out), warm, int(shift)))
        return f, status, iters

    def solve_ext(self, st, sched=None, normals=None, want_u=False):
        """BASELINE config 4 (extension): per-step contact schedule [N,B] and/or terrain normals [12,B]"""
        B = st["x0"].shape[1]
        N = self.cfg.horizon
        ft = self.ftype
        a = {k: np.ascontiguousarray(st[k], dtype=(np.uint32 if k == "contact" else ft)) for k in ("x0", "rot", "foot", "ref", "contact")}
        sc = np.ascontiguousarray(sched, dtype=np.uint32) if sched is not None else None
        nm = np.ascontiguousarray(normals, dtype=ft) if normals is not None else None
        f = np.zeros((12, B), dtype=ft); status = np.zeros(B, dtype=np.int32); iters = np.zeros(B, dtype=np.int32)
        u = np.zeros((12 * N, B), dtype=ft) if want_u else None
        inp = Inputs(_p(a["x0"]), _p(a["rot"]), _p(a["foot"]), _p(a["ref"]), _p(a["contact"]), B)
        ext = InputsExt(_p(sc), _p(nm))
        out = Outputs(_p(f), _p(status), _p(iters), _p(u), B)
        _check(lib().a1mpc_solve_batch_ext(self.h, B, C.byref(inp), C.byref(ext), C.byref(out)))
        return (f, status, iters, u) if want_u else (f, status, iters)

    def solve_ext_warm(self, st, warm, sched=None, normals=None, shift=1, want_u=False):
        """a1mpc_solve_batch_ext_warm: solve_ext with the warm start of solve_warm (`warm` from warm_alloc, updated in place on
        the device); shift = 1 for schedules that advance one step per tick (update_plan)"""
        B = st["x0"].shape[1]
        N = self.cfg.horizon
        ft = self.ftype
        a = {k: np.ascontiguousarray(st[k], dtype=(np.uint32 if k == "contact" else ft)) for k in ("x0", "rot", "foot", "ref", "contact")}
        sc = np.ascontiguousarray(sched, dtype=np.uint32) if sched is not None else None
        nm = np.ascontiguousarray(normals, dtype=ft) if normals is not None else None
        f = np.zeros((12, B), dtype=ft); status = np.zeros(B, dtype=np.int32); iters = np.zeros(B, dtype=np.int32)
        u = np.zeros((12 * N, B), dtype=ft) if want_u else None
        inp = Inputs(_p(a["x0"]), _p(a["rot"]), _p(a["foot"]), _p(a["ref"]), _p(a["contact"]), B)
        ext = InputsExt(_p(sc), _p(nm))
        out = Outputs(_p(f), _p(status), _p(iters), _p(u), B)
        _check(lib().a1mpc_solve_batch_ext_warm(self.h, B, C.byref(inp), C.byref(ext), C.byref(out), warm, int(shift)))
        return (f, status, iters, u) if want_u else (f, status, iters)

    def solve_ptrs(self, B, inp, out):
        """raw a1mpc_solve_batch on caller-built Inputs/Outputs (host or device pointers)"""
        _check(lib().a1mpc_solve_batch(self.h, B, C.byref(inp), C.byref(out)))

    # ---- ConvexMpc parity members ----
    def build_qp(self, st):
        B = st["x0"].shape[1]
        N = self.cfg.horizon
        n, m = 12 * N, 20 * N
        a = {k: np.ascontiguousarray(st[k], dtype=(np.uint32 if k == "contact" else np.float64)) for k in ("x0", "rot", "foot", "ref", "contact")}
        H = np.zeros((B, n, n)); g = np.zeros((B, n)); lb = np.zeros((B, m)); ub = np.zeros((B, m))
        inp = Inputs(_p(a["x0"]), _p(a["rot"]), _p(a["foot"]), _p(a["ref"]), _p(a["contact"]), B)
        _check(lib().a1mpc_build_qp_batch(self.h, B, C.byref(inp), _p(H), _p(g), _p(lb), _p(ub)))
        return H, g, lb, ub

    def qp_mats(self, A_d, B_d_list, x0, x_d):
        A_d = np.ascontiguousarray(A_d, dtype=np.float64); B_d_list = np.ascontiguousarray(B_d_list, dtype=np.float64)
        x0 = np.ascontiguousarray(x0, dtype=np.float64); x_d = np.ascontiguousarray(x_d, dtype=np.float64)
        B = A_d.shape[0]
        n = 12 * self.cfg.horizon
        H = np.zeros((B, n, n)); g = np.zeros((B, n))
        _check(lib().a1mpc_qp_mats_batch(self.h, B, _p(A_d), _p(B_d_list), _p(x0), _p(x_d), _p(H), _p(g)))
        return H, g

    def qp_rollout(self, A_d, B_d_list, x0, x_d):
        """a1mpc_qp_rollout_batch: A_qp [B,13N,13], B_qp [B,13N,12N], H, g"""
        A_d = np.ascontiguousarray(A_d, dtype=np.float64); B_d_list = np.ascontiguousarray(B_d_list, dtype=np.float64)
        x0 = np.ascontiguousarray(x0, dtype=np.float64); x_d = np.ascontiguousarray(x_d, dtype=np.float64)
        B = A_d.shape[0]; N = self.cfg.horizon; n = 12 * N
        Aq = np.zeros((B, 13 * N, 13)); Bq = np.zeros((B, 13 * N, n)); H = np.zeros((B, n, n)); g = np.zeros((B, n))
        _check(lib().a1mpc_qp_rollout_batch(self.h, B, _p(A_d), _p(B_d_list), _p(x0), _p(x_d), _p(Aq), _p(Bq), _p(H), _p(g)))
        return Aq, Bq, H, g

    def solve_dense(self, H, g, contact):
        H = np.ascontiguousarray(H, dtype=np.float64); g = np.ascontiguousarray(g, dtype=np.float64)
        contact = np.ascontiguousarray(contact, dtype=np.uint32)
        B = H.shape[0]
        u = np.zeros((B, 12 * self.cfg.horizon)); status = np.zeros(B, dtype=np.int32)
        _check(lib().a1mpc_solve_dense_batch(self.h, B, _p(H), _p(g), _p(contact), _p(u), _p(status)))
        return u, status

    def grf_qp(self, root_acc, rot_z, rot, foot, contact):
        arrs = [np.ascontiguousarray(v, dtype=np.float64) for v in (root_acc, rot_z, rot, foot)]
        contact = np.ascontiguousarray(contact, dtype=np.uint32)
        B = arrs[0].shape[0]
        f = np.zeros((B, 12)); status = np.zeros(B, dtype=np.int32)
        _check(lib().a1mpc_grf_qp_batch(self.h, B, _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), _p(contact), _p(f), _p(status)))
        return f, status

    def joint_torques(self, f_grf, f_kin, jac, contact, km_foot, torques_gravity, tau_prev=None):
        """batch-major SoA [12,B], [12,B], [36,B], [B] -> tau [12,B]"""
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (f_grf, f_kin, jac, km_foot, torques_gravity)]
        contact = np.ascontiguousarray(contact, dtype=np.uint32)
        B = a[0].shape[1]
        tau = np.zeros((12, B)) if tau_prev is None else np.ascontiguousarray(tau_prev, dtype=np.float64).copy()
        _check(lib().a1mpc_joint_torques_batch(self.h, B, _p(a[0]), _p(a[1]), _p(a[2]), _p(contact), _p(a[3]), _p(a[4]), _p(tau)))
        return tau

    def leg_kinematics(self, joint_pos, joint_vel, rot, rho_opt, rho_fix):
        """a1mpc_leg_kinematics_batch, host arrays: [12,B], [12,B], [9,B], rho_opt[12], rho_fix[20] ->
        foot_pos_rel [12,B], jac [36,B], foot_vel_rel [12,B], foot_pos_abs [12,B], foot_vel_abs [12,B]"""
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (joint_pos, joint_vel, rot, rho_opt, rho_fix)]
        B = a[0].shape[1]
        outs = [np.zeros((12, B)), np.zeros((36, B)), np.zeros((12, B)), np.zeros((12, B)), np.zeros((12, B))]
        _check(lib().a1mpc_leg_kinematics_batch(self.h, B, *[_p(v) for v in a], *[_p(o) for o in outs]))
        return outs

    def ekf_alloc(self, B):
        """device-resident filter state of B robots (342 doubles each: x[18], P[18,18])"""
        return self.dalloc(lib().a1mpc_ekf_bytes(B))

    def ekf_init(self, ekf, foot_pos_rel, rot):
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (foot_pos_rel, rot)]
        _check(lib().a1mpc_ekf_init_batch(self.h, a[0].shape[1], ekf, _p(a[0]), _p(a[1])))

    def ekf_update(self, ekf, dt, assume_flat_ground, movement_mode, imu_acc, imu_ang_vel, rot, foot_pos_rel, foot_vel_rel, foot_force):
        """a1mpc_ekf_update_batch, host arrays -> root_pos [3,B], root_lin_vel [3,B], estimated_contacts [B], status [B]"""
        mm = np.ascontiguousarray(movement_mode, dtype=np.uint32)
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (imu_acc, imu_ang_vel, rot, foot_pos_rel, foot_vel_rel, foot_force)]
        B = mm.shape[0]
        pos = np.zeros((3, B)); vel = np.zeros((3, B)); ec = np.zeros(B, dtype=np.uint32); status = np.full(B, -7, dtype=np.int32)
        _check(lib().a1mpc_ekf_update_batch(self.h, B, ekf, C.c_double(dt), int(assume_flat_ground), _p(mm), *[_p(v) for v in a],
                                            _p(pos), _p(vel), _p(ec), _p(status)))
        return pos, vel, ec, status

    def ekf_state(self, ekf, B):
        """copy of the device-resident filter state: x [B,18], P [B,18,18]"""
        buf = np.zeros((B, 342))
        _check(lib().a1mpc_memcpy_d2h(self.h, _p(buf), ekf, buf.nbytes))
        _check(lib().a1mpc_sync(self.h))
        return buf[:, :18].copy(), buf[:, 18:].reshape(B, 18, 18).copy()

    def update_plan(self, gp, gait_counter, gait_counter_speed, movement_mode, lin_vel, lin_vel_d, rot_z, rot, root_pos):
        """A1RobotControl::update_plan batched; returns new gait_counter [4,B], plan_contacts [B], contact_sched [N,B],
        foot_pos_target_rel/abs/world [12,B]"""
        gc = np.ascontiguousarray(gait_counter, dtype=np.float64).copy()
        B = gc.shape[1]
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (gait_counter_speed, lin_vel, lin_vel_d, rot_z, rot, root_pos)]
        mode = np.ascontiguousarray(movement_mode, dtype=np.uint32)
        plan = np.zeros(B, dtype=np.uint32); sched = np.zeros((gp.horizon, B), dtype=np.uint32)
        trel = np.zeros((12, B)); tabs = np.zeros((12, B)); tw = np.zeros((12, B))
        _check(lib().a1mpc_update_plan_batch(self.h, B, C.byref(gp), _p(gc), _p(a[0]), _p(mode), _p(a[1]), _p(a[2]), _p(a[3]), _p(a[4]), _p(a[5]),
                                             _p(plan), _p(sched), _p(trel), _p(tabs), _p(tw)))
        return gc, plan, sched, trel, tabs, tw

    # ---- memory / timing helpers ----
    def dalloc(self, nbytes):
        p = C.c_void_p()
        _check(lib().a1mpc_device_alloc(self.h, nbytes, C.byref(p)))
        return p

    def halloc(self, nbytes):
        p = C.c_void_p()
        _check(lib().a1mpc_host_alloc(self.h, nbytes, C.byref(p)))
        return p

    def pinned_array(self, shape, dtype):
        """numpy view over pinned host memory (kept alive by the returned array's base object)"""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = self.halloc(max(nbytes, 8))
        buf = (C.c_char * nbytes).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
        return arr

    def sync(self):
        _check(lib().a1mpc_sync(self.h))

    def event(self):
        e = C.c_void_p()
        _check(lib().a1mpc_event_create(self.h, C.byref(e)))
        return e

    def record(self, ev):
        _check(lib().a1mpc_event_record(self.h, ev))

    def elapsed_ms(self, e0, e1):
        ms = C.c_float()
        _check(lib().a1mpc_event_elapsed_ms(self.h, e0, e1, C.byref(ms)))
        return float(ms.value)

    def launches(self):
        return int(lib().a1mpc_launch_count(self.h))

    def fp64_peak_tflops(self):
        v = C.c_double()
        _check(lib().a1mpc_measure_fp64_peak(self.h, C.byref(v)))
        return float(v.value)

    def profile_begin(self, max_calls):
        _check(lib().a1mpc_profile_begin(self.h, max_calls))

    def profile_end(self):
        ms = np.zeros(4); n = C.c_int()
        _check(lib().a1mpc_profile_end(self.h, _p(ms), C.byref(n)))
        return ms, int(n.value)

    def nccl_init(self, nranks, rank, uid_bytes):
        buf = C.create_string_buffer(bytes(uid_bytes), 128)
        _check(lib().a1mpc_nccl_init(self.h, nranks, rank, buf))

    def allgather_forces(self, f_local_ptr, f_all_ptr, B_local):
        _check(lib().a1mpc_allgather_forces(self.h, f_local_ptr, f_all_ptr, B_local))

    # ---- fused final collect over peer memory (one process per GPU) ----
    def peer_gather_create(self, nranks, rank, B_local):
        """allocates this rank's gathered buffer; returns the 64-byte CUDA IPC handle to hand to the other ranks"""
        hd = (C.c_char * 64)()
        _check(lib().a1mpc_peer_gather_create(self.h, int(nranks), int(rank), int(B_local), hd))
        return bytes(hd.raw)

    def peer_gather_connect(self, handles):
        """handles: the ranks' 64-byte handles in rank order (list of bytes)"""
        blob = b"".join(handles)
        _check(lib().a1mpc_peer_gather_connect(self.h, C.c_char_p(blob)))

    def peer_gather_buffer(self):
        p = C.c_void_p()
        _check(lib().a1mpc_peer_gather_buffer(self.h, C.byref(p)))
        return p

    def peer_gather_wait(self):
        _check(lib().a1mpc_peer_gather_wait(self.h))

    def peer_gather_status(self):
        v = C.c_int()
        _check(lib().a1mpc_peer_gather_status(self.h, C.byref(v)))
        return v.value

    def peer_gather_destroy(self):
        _check(lib().a1mpc_peer_gather_destroy(self.h))

    def flush_l2(self):
        _check(lib().a1mpc_flush_l2(self.h))


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    _check(lib().a1mpc_nccl_unique_id(buf))
    return bytes(buf.raw)
