// a1mpc_api.cu -- C ABI of the engine (include/a1mpc.h) over the sm_100a kernels.
// No CPU fallback anywhere in this file: every compute entry point launches CUDA kernels or fails.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <algorithm>
#include <initializer_list>

#include "a1mpc_internal.h"
#include "a1mpc_misc.cuh"
#include "a1mpc_estim.cuh"

using namespace a1mpc;

namespace {
thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(A1MPC_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
  } while (0)

}  // namespace

extern "C" void a1mpc_internal_nccl_destroy(void* comm);   // a1mpc_nccl.cpp
extern "C" void* a1mpc_internal_gather_begin(a1mpc_handle* h);
extern "C" void a1mpc_internal_gather_end(a1mpc_handle* h);

struct a1mpc_handle {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t side[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
  a1mpc_config cfg;
  DevParams P;
  a1mpc::ClassLaunch cls[5];  // index = number of stance feet
  a1mpc::ClassLaunch cls_ext;  // extended path (config 4)
  a1mpc::ClassLaunch cls_sched2;   // its compacted two-feet-per-step class (N = 10; A1MPC_EXT_COMPACT=0 disables it)
  a1mpc::ClassLaunch cls_ext_warm, cls_sched2_warm;   // the same two with the warm start (a1mpc_solve_batch_ext_warm)
  bool ext_compact = false;
  double* d_rec_ext = nullptr;
  size_t cap_ext = 0;
  uint32_t* d_sched = nullptr;
  double* d_normals = nullptr;
  size_t cap_ext_mirror = 0;
  // scratch sized for `cap` QPs
  size_t cap = 0;
  double* d_rec = nullptr;
  int* d_count = nullptr;
  // device mirrors for host-pointer calls
  double *d_x0 = nullptr, *d_rot = nullptr, *d_foot = nullptr, *d_ref = nullptr, *d_f = nullptr, *d_u = nullptr;
  uint32_t* d_contact = nullptr;
  int32_t *d_status = nullptr, *d_iters = nullptr;
  size_t cap_u = 0;
  // generic scratch for the QP-major side APIs
  void* d_side = nullptr;
  size_t side_bytes = 0;
  int* d_lists = nullptr;
  size_t lists_bytes = 0;
  double* d_flush = nullptr;
  size_t flush_elems = 0;
  int64_t launches = 0;
  // optional per-class kernel timing (bench roofline): event pairs on the class streams
  bool prof_on = false;
  int prof_cap = 0, prof_n = 0;
  std::vector<cudaEvent_t> prof_ev;  // [call][class 1..4][begin,end]
  // NCCL (dlopen'ed)
  void* nccl_lib = nullptr;
  void* nccl_comm = nullptr;
  cudaStream_t gather_stream = nullptr;   // the optional final collect runs here, overlapped with the next step's solve
  cudaEvent_t ev_gather_in = nullptr, ev_gather_done = nullptr;
  bool gather_pending = false;
  // fused final collect over peer memory (a1mpc_peer_gather_*)
  struct PeerGather {
    bool connected = false;
    int nranks = 0, rank = 0;
    size_t B = 0;
    void* local = nullptr;                 // this rank's allocation: [nranks][12][B] doubles, then nranks u64 step flags, then an int error word
    double* buf[MAX_PEERS] = {nullptr};    // every rank's gathered buffer as mapped into this process (buf[rank] == local)
    unsigned long long* flags[MAX_PEERS] = {nullptr};
    bool opened[MAX_PEERS] = {false};
    unsigned long long step = 0;
  } peer;
};

namespace {

int ensure_capacity(a1mpc_handle* h, size_t B, bool mirrors, bool want_u) {
  if (B > h->cap) {
    CK(cudaStreamSynchronize(h->stream));
    auto fr = [](void* p) { if (p) cudaFree(p); };
    fr(h->d_rec); fr(h->d_x0); fr(h->d_rot); fr(h->d_foot); fr(h->d_ref); fr(h->d_f); fr(h->d_contact); fr(h->d_status); fr(h->d_iters);
    fr(h->d_u);
    h->d_rec = h->d_x0 = h->d_rot = h->d_foot = h->d_ref = h->d_f = h->d_u = nullptr;
    h->d_contact = nullptr; h->d_status = h->d_iters = nullptr;
    h->cap_u = 0;
    size_t cap = 1024;
    while (cap < B) cap *= 2;
    h->cap = cap;
    CK(cudaMalloc(&h->d_rec, 4 * cap * REC_BYTES));
  }
  if (mirrors && !h->d_x0) {
    const size_t cap = h->cap;
    CK(cudaMalloc(&h->d_x0, 12 * cap * 8));
    CK(cudaMalloc(&h->d_rot, 9 * cap * 8));
    CK(cudaMalloc(&h->d_foot, 12 * cap * 8));
    CK(cudaMalloc(&h->d_ref, 9 * cap * 8));
    CK(cudaMalloc(&h->d_f, 12 * cap * 8));
    CK(cudaMalloc(&h->d_contact, cap * 4));
    CK(cudaMalloc(&h->d_status, cap * 4));
    CK(cudaMalloc(&h->d_iters, cap * 4));
  }
  if (mirrors && want_u && h->cap_u < h->cap) {
    if (h->d_u) cudaFree(h->d_u);
    CK(cudaMalloc(&h->d_u, (size_t)12 * h->cfg.horizon * h->cap * 8));
    h->cap_u = h->cap;
  }
  return A1MPC_OK;
}

int ensure_side(a1mpc_handle* h, size_t bytes) {
  if (bytes > h->side_bytes) {
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_side) cudaFree(h->d_side);
    h->d_side = nullptr;
    CK(cudaMalloc(&h->d_side, bytes));
    h->side_bytes = bytes;
  }
  return A1MPC_OK;
}

int ensure_lists(a1mpc_handle* h, size_t bytes) {
  if (bytes > h->lists_bytes) {
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_lists) cudaFree(h->d_lists);
    h->d_lists = nullptr;
    CK(cudaMalloc(&h->d_lists, bytes));
    h->lists_bytes = bytes;
  }
  return A1MPC_OK;
}

bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// true when the non-NULL pointers do not all live on the same side as `dev` says (a host pointer dereferenced by a kernel is a sticky
// fault for the whole CUDA context, so every entry point classifies every array it is given)
bool mixed_sides(bool dev, std::initializer_list<const void*> ptrs) {
  for (const void* q : ptrs)
    if (q && is_device_ptr(q) != dev) return true;
  return false;
}

// enqueue the fused path on device-resident SoA data
void attach_peers(a1mpc_handle* h, int B, DevOutputs& d) {
  d.npeer = 0; d.rank = 0; d.peer_ld = 0;
  for (int p = 0; p < MAX_PEERS; ++p) d.peer[p] = nullptr;
  if (h->peer.connected && (size_t)B == h->peer.B) {
    d.npeer = h->peer.nranks; d.rank = h->peer.rank; d.peer_ld = h->peer.B;
    for (int p = 0; p < h->peer.nranks; ++p) d.peer[p] = h->peer.buf[p];
  }
}

int peer_signal(a1mpc_handle* h, int B) {
  if (!(h->peer.connected && (size_t)B == h->peer.B)) return A1MPC_OK;
  PeerFlags pf;
  for (int p = 0; p < MAX_PEERS; ++p) pf.p[p] = h->peer.flags[p];
  h->peer.step++;
  peer_signal_kernel<<<1, 32, 0, h->stream>>>(pf, h->peer.nranks, h->peer.rank, h->peer.step);
  h->launches++;
  CK(cudaGetLastError());
  return A1MPC_OK;
}

int enqueue_solve(a1mpc_handle* h, int B, const DevInputs& din, const DevOutputs& dout_in, uint32_t* warm = nullptr, int shift = 0) {
  DevOutputs dout = dout_in;
  attach_peers(h, B, dout);
  CK(cudaMemsetAsync(h->d_count, 0, 16 * sizeof(int), h->stream));
  pack_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(din, B, h->d_rec, (int)h->cap, h->d_count, dout, h->cfg.horizon);
  h->launches++;
  CK(cudaEventRecord(h->ev_fork, h->stream));
  const int N = h->cfg.horizon;
  // heaviest class first, each class on its own stream so that the few long 4-stance solves overlap
  // the many short trot solves
  for (int ns = 4; ns >= 1; --ns) {
    cudaStream_t st = h->side[ns - 1];
    CK(cudaStreamWaitEvent(st, h->ev_fork, 0));
    const double* rec = h->d_rec + (size_t)(ns - 1) * h->cap * REC_DOUBLES;
    const bool prof = h->prof_on && h->prof_n < h->prof_cap;
    if (prof) CK(cudaEventRecord(h->prof_ev[((size_t)h->prof_n * 4 + (ns - 1)) * 2 + 0], st));
    if (!h->cls[ns].supported) unsupported_kernel<<<(B + 127) / 128, 128, 0, st>>>(rec, h->d_count, ns, dout, N);
    else if (N == 10 && warm) fused_launch_n10_warm(ns, h->cls[ns], st, B, h->P, rec, h->d_count, dout, warm, shift);
    else if (N == 10) fused_launch_n10(ns, h->cls[ns], st, B, h->P, rec, h->d_count, dout);
    else fused_launch_n20(ns, h->cls[ns], st, B, h->P, rec, h->d_count, dout);
    h->launches++;
    if (prof) CK(cudaEventRecord(h->prof_ev[((size_t)h->prof_n * 4 + (ns - 1)) * 2 + 1], st));
    CK(cudaEventRecord(h->ev_join[ns - 1], st));
    CK(cudaStreamWaitEvent(h->stream, h->ev_join[ns - 1], 0));
  }
  if (h->prof_on && h->prof_n < h->prof_cap) h->prof_n++;
  CK(cudaGetLastError());
  return peer_signal(h, B);   // fused collect: publish this call's step number to every rank (no-op when not connected)
}

int copy_rows(cudaStream_t st, void* dst, size_t dst_ld, const void* src, size_t src_ld, int rows, size_t B, size_t esz, cudaMemcpyKind kind) {
  CK(cudaMemcpy2DAsync(dst, dst_ld * esz, src, src_ld * esz, B * esz, rows, kind, st));
  return A1MPC_OK;
}

}  // namespace

extern "C" {

const char* a1mpc_last_error(void) { return g_err.c_str(); }

int a1mpc_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

void a1mpc_default_config(a1mpc_config* c) {
  std::memset(c, 0, sizeof(*c));
  c->horizon = 10;
  c->precision = 64;
  c->dt = 0.0025;
  c->mu = 0.3;
  c->fz_min = 0.0;
  c->fz_max = 180.0;
  c->mass = 12.0;
  c->inertia[0] = 0.0158533; c->inertia[4] = 0.0377999; c->inertia[8] = 0.0456542;
  const double q[13] = {20, 10, 1, 0, 0, 420, 0.05, 0.05, 0.05, 30, 30, 10, 0};
  for (int i = 0; i < 13; ++i) c->q[i] = q[i];
  for (int i = 0; i < 12; ++i) c->r[i] = 1e-7;
  c->max_iter = 0;
  c->tol = 0.0;
}

int a1mpc_create(a1mpc_handle** out, const a1mpc_config* cfg, int device) {
  if (!out || !cfg) return fail(A1MPC_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->horizon != 10 && cfg->horizon != 20) return fail(A1MPC_EINVAL, "horizon must be 10 or 20");
  if (cfg->precision != 64 && cfg->precision != 32) return fail(A1MPC_EINVAL, "precision must be 64 or 32 (see include/a1mpc.h)");
  if (!(cfg->fz_min == 0.0)) return fail(A1MPC_EINVAL, "fz_min must be 0 (the reference hard-codes it, ConvexMpc.cpp:223)");
  if (!(cfg->mu > 0.0) || !(cfg->fz_max > 0.0) || !(cfg->mass > 0.0) || !(cfg->dt > 0.0)) return fail(A1MPC_EINVAL, "mu, fz_max, mass, dt must be positive");
  for (int i = 0; i < 12; ++i)
    if (!(cfg->r[i] > 0.0)) return fail(A1MPC_EINVAL, "r weights must be positive (H must be positive definite)");
  for (int i = 0; i < 13; ++i)
    if (!(cfg->q[i] >= 0.0)) return fail(A1MPC_EINVAL, "q weights must be non-negative");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return fail(A1MPC_ENODEVICE, "no CUDA device available (this engine has no CPU fallback)");
  }
  if (device < 0 || device >= ndev) return fail(A1MPC_EINVAL, "device index out of range");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(A1MPC_ENODEVICE, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) + "; this library is built for sm_100a only");
  a1mpc_handle* h = new a1mpc_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->cfg = *cfg;
  DevParams& P = h->P;
  P.N = cfg->horizon;
  P.max_iter = cfg->max_iter > 0 ? cfg->max_iter : 40;
  P.dt = cfg->dt; P.mu = cfg->mu; P.fzmax = cfg->fz_max; P.mass = cfg->mass;
  P.mu_switch = cfg->tol > 0.0 ? cfg->tol : MU_SWITCH_DEFAULT;
  for (int i = 0; i < 9; ++i) P.inertia[i] = cfg->inertia[i];
  for (int i = 0; i < 13; ++i) P.q2[i] = 2.0 * cfg->q[i];
  for (int i = 0; i < 12; ++i) P.r2[i] = 2.0 * cfg->r[i];
  int rc = A1MPC_OK;
  auto bail = [&](int code) { a1mpc_destroy(h); return code; };
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(A1MPC_ECUDA, "stream create failed"));
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  for (int i = 0; i < 4; ++i) {
    // the classes with more stance feet take longer per QP: their CTAs are placed first
    const int prio = (i >= 2) ? prio_hi : prio_lo;
    if (cudaStreamCreateWithPriority(&h->side[i], cudaStreamNonBlocking, prio) != cudaSuccess) return bail(fail(A1MPC_ECUDA, "stream create failed"));
    if (cudaEventCreateWithFlags(&h->ev_join[i], cudaEventDisableTiming) != cudaSuccess) return bail(fail(A1MPC_ECUDA, "event create failed"));
  }
  if (cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess) return bail(fail(A1MPC_ECUDA, "event create failed"));
  if (cudaMalloc(&h->d_count, 16 * sizeof(int)) != cudaSuccess) return bail(fail(A1MPC_ENOMEM, "cudaMalloc failed"));
  {
    cudaError_t e = (cfg->horizon == 10) ? fused_setup_n10(h->sm_count, h->cls) : fused_setup_n20(h->sm_count, h->cls);
    if (e != cudaSuccess) return bail(fail(A1MPC_ECUDA, std::string("kernel setup: ") + cudaGetErrorString(e)));
    e = ext_setup(cfg->horizon, h->sm_count, h->cls_ext, h->cls_ext_warm);
    if (e != cudaSuccess) return bail(fail(A1MPC_ECUDA, std::string("ext kernel setup: ") + cudaGetErrorString(e)));
    {   // schedules with two stance feet in every step run on the compact direct kernel (a1mpc_sched.cuh): 2.5 M instead of 1.5 M
        // QPs/s end to end on a B200 at B = 16384 (profiles/r02a_call1_*.txt).  A1MPC_EXT_COMPACT=0 keeps everything on the general kernel (A/B).
      const char* ev = std::getenv("A1MPC_EXT_COMPACT");
      if (!(ev && ev[0] == '0') && cfg->horizon == 10) {
        e = sched2_setup(h->sm_count, h->cls_sched2, h->cls_sched2_warm);
        if (e != cudaSuccess) return bail(fail(A1MPC_ECUDA, std::string("compact ext kernel setup: ") + cudaGetErrorString(e)));
        h->ext_compact = true;
      }
    }
    e = dense_setup(cfg->horizon);
    if (e != cudaSuccess) return bail(fail(A1MPC_ECUDA, std::string("dense kernel setup: ") + cudaGetErrorString(e)));
  }
  (void)rc;
  *out = h;
  return A1MPC_OK;
}

int a1mpc_destroy(a1mpc_handle* h) {
  if (!h) return A1MPC_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->gather_stream) cudaStreamSynchronize(h->gather_stream);
  if (h->nccl_comm) { a1mpc_internal_nccl_destroy(h->nccl_comm); h->nccl_comm = nullptr; }   // before its streams go away
  a1mpc_peer_gather_destroy(h);
  auto fr = [](void* p) { if (p) cudaFree(p); };
  fr(h->d_rec); fr(h->d_count); fr(h->d_x0); fr(h->d_rot); fr(h->d_foot); fr(h->d_ref); fr(h->d_f); fr(h->d_u);
  fr(h->d_contact); fr(h->d_status); fr(h->d_iters); fr(h->d_side); fr(h->d_flush); fr(h->d_lists);
  fr(h->d_rec_ext); fr(h->d_sched); fr(h->d_normals);
  for (int i = 0; i < 4; ++i) {
    if (h->side[i]) cudaStreamDestroy(h->side[i]);
    if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
  }
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  if (h->gather_stream) { cudaStreamSynchronize(h->gather_stream); cudaStreamDestroy(h->gather_stream); cudaEventDestroy(h->ev_gather_in); cudaEventDestroy(h->ev_gather_done); }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return A1MPC_OK;
}

static int solve_batch_impl(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_outputs* out, uint32_t* warm, int shift) {
  if (!h || !in || !out) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  if (!in->x0 || !in->rot || !in->foot || !in->ref || !in->contact || !out->f_body || !out->status) return fail(A1MPC_EINVAL, "null input/output array");
  if (in->ld < (size_t)B || out->ld < (size_t)B) return fail(A1MPC_EINVAL, "ld < B");
  CK(cudaSetDevice(h->device));
  // every array of the call lives on the same side (a host pointer dereferenced by a kernel is a sticky fault for the whole context)
  const bool dev_in = is_device_ptr(in->x0), dev_out = is_device_ptr(out->f_body);
  const void* all_ptrs[] = {in->rot, in->foot, in->ref, in->contact, out->status, out->iters, out->u_full};
  bool mixed = (dev_in != dev_out);
  for (const void* q : all_ptrs) mixed = mixed || (q && is_device_ptr(q) != dev_in);
  if (mixed) return fail(A1MPC_EINVAL, "inputs and outputs must be all-host or all-device");
  const int f32 = (h->cfg.precision == 32) ? 1 : 0;   // fp32 arrays at the boundary, fp64 inside
  const size_t es = f32 ? 4 : 8;
  int rc;
  if (dev_in) {
    if ((rc = ensure_capacity(h, B, false, false))) return rc;
    DevInputs di{in->x0, in->rot, in->foot, in->ref, in->contact, in->ld, f32};
    DevOutputs dout{out->f_body, out->status, out->iters, out->u_full, out->ld, f32};
    return enqueue_solve(h, B, di, dout, warm, shift);
  }
  if ((rc = ensure_capacity(h, B, true, out->u_full != nullptr))) return rc;
  const size_t Bs = (size_t)B;
  if ((rc = copy_rows(h->stream, h->d_x0, Bs, in->x0, in->ld, 12, Bs, es, cudaMemcpyHostToDevice))) return rc;
  if ((rc = copy_rows(h->stream, h->d_rot, Bs, in->rot, in->ld, 9, Bs, es, cudaMemcpyHostToDevice))) return rc;
  if ((rc = copy_rows(h->stream, h->d_foot, Bs, in->foot, in->ld, 12, Bs, es, cudaMemcpyHostToDevice))) return rc;
  if ((rc = copy_rows(h->stream, h->d_ref, Bs, in->ref, in->ld, 9, Bs, es, cudaMemcpyHostToDevice))) return rc;
  CK(cudaMemcpyAsync(h->d_contact, in->contact, Bs * 4, cudaMemcpyHostToDevice, h->stream));
  DevInputs di{h->d_x0, h->d_rot, h->d_foot, h->d_ref, h->d_contact, Bs, f32};
  DevOutputs dout{h->d_f, h->d_status, out->iters ? h->d_iters : nullptr, out->u_full ? h->d_u : nullptr, Bs, f32};
  if ((rc = enqueue_solve(h, B, di, dout, warm, shift))) return rc;
  if ((rc = copy_rows(h->stream, out->f_body, out->ld, h->d_f, Bs, 12, Bs, es, cudaMemcpyDeviceToHost))) return rc;
  CK(cudaMemcpyAsync(out->status, h->d_status, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out->iters) CK(cudaMemcpyAsync(out->iters, h->d_iters, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out->u_full)
    if ((rc = copy_rows(h->stream, out->u_full, out->ld, h->d_u, Bs, 12 * h->cfg.horizon, Bs, es, cudaMemcpyDeviceToHost))) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return A1MPC_OK;
}

int a1mpc_solve_batch(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_outputs* out) { return solve_batch_impl(h, B, in, out, nullptr, 0); }

size_t a1mpc_warm_bytes(const a1mpc_handle* h, int B) {
  if (!h || B <= 0) return 0;
  return (size_t)B * (size_t)(WARM_HDR + 4 * h->cfg.horizon) * sizeof(uint32_t);
}

int a1mpc_warm_reset(a1mpc_handle* h, void* warm, int B) {
  if (!h || !warm || B <= 0) return fail(A1MPC_EINVAL, "null argument");
  if (!is_device_ptr(warm)) return fail(A1MPC_EINVAL, "warm must be device memory (a1mpc_device_alloc)");
  CK(cudaSetDevice(h->device));
  CK(cudaMemsetAsync(warm, 0, a1mpc_warm_bytes(h, B), h->stream));
  return A1MPC_OK;
}

int a1mpc_solve_batch_warm(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_outputs* out, void* warm, int shift) {
  if (!h || !warm) return fail(A1MPC_EINVAL, "null argument");
  if (h->cfg.horizon != 10) return fail(A1MPC_EINVAL, "warm start is implemented for horizon 10 (see include/a1mpc.h)");
  if (shift < 0 || shift > h->cfg.horizon) return fail(A1MPC_EINVAL, "shift out of range");
  CK(cudaSetDevice(h->device));
  if (!is_device_ptr(warm)) return fail(A1MPC_EINVAL, "warm must be device memory (a1mpc_device_alloc)");
  return solve_batch_impl(h, B, in, out, static_cast<uint32_t*>(warm), shift);
}

// the extended call, cold (warm == nullptr) or warm-started: argument checks, device mirrors and packing are shared, only
// the solve launches differ.  The caller has checked h, in, out and that ext carries a schedule or normals.
static int solve_ext_impl(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_inputs_ext* ext, const a1mpc_outputs* out, uint32_t* warm,
                          int shift) {
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  if (!in->x0 || !in->rot || !in->foot || !in->ref || !in->contact || !out->f_body || !out->status) return fail(A1MPC_EINVAL, "null input/output array");
  if (in->ld < (size_t)B || out->ld < (size_t)B) return fail(A1MPC_EINVAL, "ld < B");
  if (ext->normals)
    for (int i = 0; i < 4; ++i)
      if (h->cfg.r[3 * i] != h->cfg.r[3 * i + 1] || h->cfg.r[3 * i] != h->cfg.r[3 * i + 2])
        return fail(A1MPC_EINVAL, "terrain normals need isotropic r weights per foot (r[3i] == r[3i+1] == r[3i+2])");
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.horizon;
  const size_t Bs = (size_t)B;
  const bool dev = is_device_ptr(in->x0);
  {
    const void* all_ptrs[] = {in->rot, in->foot, in->ref, in->contact, out->f_body, out->status, out->iters, out->u_full, ext->contact_sched, ext->normals};
    for (const void* q : all_ptrs)
      if (q && is_device_ptr(q) != dev) return fail(A1MPC_EINVAL, "inputs and outputs must be all-host or all-device");
  }
  const int f32 = (h->cfg.precision == 32) ? 1 : 0;
  const size_t es = f32 ? 4 : 8;
  int rc;
  if ((rc = ensure_capacity(h, B, !dev, !dev && out->u_full != nullptr))) return rc;
  if (Bs > h->cap_ext) {
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_rec_ext) cudaFree(h->d_rec_ext);
    h->d_rec_ext = nullptr;
    CK(cudaMalloc(&h->d_rec_ext, 2 * h->cap * REC_EXT_BYTES));   // second half: queue of the compacted class
    h->cap_ext = h->cap;
  }
  DevInputs di{in->x0, in->rot, in->foot, in->ref, in->contact, in->ld, f32};
  DevOutputs dout{out->f_body, out->status, out->iters, out->u_full, out->ld, f32};
  const uint32_t* dsched = ext->contact_sched;
  const double* dnorm = ext->normals;
  if (!dev) {
    if (Bs > h->cap_ext_mirror) {
      CK(cudaStreamSynchronize(h->stream));
      if (h->d_sched) cudaFree(h->d_sched);
      if (h->d_normals) cudaFree(h->d_normals);
      h->d_sched = nullptr; h->d_normals = nullptr;
      CK(cudaMalloc(&h->d_sched, (size_t)A1MPC_MAX_HORIZON * h->cap * 4));
      CK(cudaMalloc(&h->d_normals, 12 * h->cap * 8));
      h->cap_ext_mirror = h->cap;
    }
    if ((rc = copy_rows(h->stream, h->d_x0, Bs, in->x0, in->ld, 12, Bs, es, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(h->stream, h->d_rot, Bs, in->rot, in->ld, 9, Bs, es, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(h->stream, h->d_foot, Bs, in->foot, in->ld, 12, Bs, es, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(h->stream, h->d_ref, Bs, in->ref, in->ld, 9, Bs, es, cudaMemcpyHostToDevice))) return rc;
    CK(cudaMemcpyAsync(h->d_contact, in->contact, Bs * 4, cudaMemcpyHostToDevice, h->stream));
    if (ext->contact_sched) {
      if ((rc = copy_rows(h->stream, h->d_sched, Bs, ext->contact_sched, in->ld, N, Bs, 4, cudaMemcpyHostToDevice))) return rc;
      dsched = h->d_sched;
    }
    if (ext->normals) {
      if ((rc = copy_rows(h->stream, h->d_normals, Bs, ext->normals, in->ld, 12, Bs, es, cudaMemcpyHostToDevice))) return rc;
      dnorm = h->d_normals;
    }
    di = DevInputs{h->d_x0, h->d_rot, h->d_foot, h->d_ref, h->d_contact, Bs, f32};
    dout = DevOutputs{h->d_f, h->d_status, out->iters ? h->d_iters : nullptr, out->u_full ? h->d_u : nullptr, Bs, f32};
  }
  attach_peers(h, -1, dout);   // the fused collect is wired to a1mpc_solve_batch / _warm only
  CK(cudaMemsetAsync(h->d_count, 0, 16 * sizeof(int), h->stream));
  const ClassLaunch& cls_ext = warm ? h->cls_ext_warm : h->cls_ext;
  if (h->ext_compact && dsched) {
    pack_ext2_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(di, dsched, dnorm, B, h->d_rec_ext, (int)h->cap_ext, h->d_count, dout, N);
    ext_launch(N, cls_ext, h->stream, B, h->P, h->d_rec_ext, h->d_count, dout, warm, shift);
    sched2_launch(warm ? h->cls_sched2_warm : h->cls_sched2, h->stream, B, h->P, h->d_rec_ext + h->cap_ext * REC_EXT_DOUBLES, h->d_count, dout,
                  warm, shift);
    h->launches += 3;
  } else {
    pack_ext_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(di, dsched, dnorm, B, h->d_rec_ext, h->d_count, dout, N);
    ext_launch(N, cls_ext, h->stream, B, h->P, h->d_rec_ext, h->d_count, dout, warm, shift);
    h->launches += 2;
  }
  if (warm) {
    warm_clear_idle_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(di.contact, dsched, di.ld, B, N, warm);
    h->launches++;
  }
  CK(cudaGetLastError());
  if (!dev) {
    if ((rc = copy_rows(h->stream, out->f_body, out->ld, h->d_f, Bs, 12, Bs, es, cudaMemcpyDeviceToHost))) return rc;
    CK(cudaMemcpyAsync(out->status, h->d_status, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
    if (out->iters) CK(cudaMemcpyAsync(out->iters, h->d_iters, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
    if (out->u_full)
      if ((rc = copy_rows(h->stream, out->u_full, out->ld, h->d_u, Bs, 12 * N, Bs, es, cudaMemcpyDeviceToHost))) return rc;
    CK(cudaStreamSynchronize(h->stream));
  }
  return A1MPC_OK;
}

int a1mpc_solve_batch_ext(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_inputs_ext* ext, const a1mpc_outputs* out) {
  if (!h || !in || !out) return fail(A1MPC_EINVAL, "null argument");
  if (!ext || (!ext->contact_sched && !ext->normals)) return a1mpc_solve_batch(h, B, in, out);
  return solve_ext_impl(h, B, in, ext, out, nullptr, 0);
}

int a1mpc_solve_batch_ext_warm(a1mpc_handle* h, int B, const a1mpc_inputs* in, const a1mpc_inputs_ext* ext, const a1mpc_outputs* out, void* warm,
                               int shift) {
  if (!h || !in || !out || !warm) return fail(A1MPC_EINVAL, "null argument");
  if (!ext || (!ext->contact_sched && !ext->normals)) return a1mpc_solve_batch_warm(h, B, in, out, warm, shift);
  if (shift < 0 || shift > h->cfg.horizon) return fail(A1MPC_EINVAL, "shift out of range");
  CK(cudaSetDevice(h->device));
  if (!is_device_ptr(warm)) return fail(A1MPC_EINVAL, "warm must be device memory (a1mpc_device_alloc)");
  return solve_ext_impl(h, B, in, ext, out, static_cast<uint32_t*>(warm), shift);
}

int a1mpc_build_qp_batch(a1mpc_handle* h, int B, const a1mpc_inputs* in, double* H, double* g, double* lb, double* ub) {
  if (!h || !in) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  if ((lb == nullptr) != (ub == nullptr)) return fail(A1MPC_EINVAL, "lb and ub must be given together");
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.horizon, n = 12 * N, m = 20 * N;
  const bool dev = is_device_ptr(in->x0);
  if (mixed_sides(dev, {in->rot, in->foot, in->ref, in->contact, H, g, lb, ub})) return fail(A1MPC_EINVAL, "inputs and outputs must be all-host or all-device");
  int rc;
  DevInputs di{in->x0, in->rot, in->foot, in->ref, in->contact, in->ld};
  double *dH = H, *dg = g, *dlb = lb, *dub = ub;
  if (!dev) {
    if ((rc = ensure_capacity(h, B, true, false))) return rc;
    const size_t Bs = (size_t)B;
    if ((rc = copy_rows(h->stream, h->d_x0, Bs, in->x0, in->ld, 12, Bs, 8, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(h->stream, h->d_rot, Bs, in->rot, in->ld, 9, Bs, 8, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(h->stream, h->d_foot, Bs, in->foot, in->ld, 12, Bs, 8, cudaMemcpyHostToDevice))) return rc;
    if ((rc = copy_rows(h->stream, h->d_ref, Bs, in->ref, in->ld, 9, Bs, 8, cudaMemcpyHostToDevice))) return rc;
    CK(cudaMemcpyAsync(h->d_contact, in->contact, Bs * 4, cudaMemcpyHostToDevice, h->stream));
    di = DevInputs{h->d_x0, h->d_rot, h->d_foot, h->d_ref, h->d_contact, Bs};
    const size_t bytes = Bs * ((size_t)n * n + n + 2 * m) * 8;
    if ((rc = ensure_side(h, bytes))) return rc;
    double* base = (double*)h->d_side;
    dH = H ? base : nullptr;
    dg = g ? base + Bs * n * n : nullptr;
    dlb = lb ? base + Bs * n * n + Bs * n : nullptr;
    dub = ub ? base + Bs * n * n + Bs * n + Bs * m : nullptr;
  }
  {
    cudaError_t e = build_dense_launch(h->P, di, B, dH, dg, dlb, dub, h->stream);
    if (e != cudaSuccess) return fail(A1MPC_ECUDA, std::string("build kernel: ") + cudaGetErrorString(e));
    h->launches++;
  }
  if (!dev) {
    const size_t Bs = (size_t)B;
    if (H) CK(cudaMemcpyAsync(H, dH, Bs * n * n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (g) CK(cudaMemcpyAsync(g, dg, Bs * n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (lb) CK(cudaMemcpyAsync(lb, dlb, Bs * m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (ub) CK(cudaMemcpyAsync(ub, dub, Bs * m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return A1MPC_OK;
}

static int qp_mats_impl(a1mpc_handle* h, int B, const double* A_d, const double* B_d_list, const double* x0, const double* x_d,
                        double* H, double* g, double* A_qp, double* B_qp) {
  if (!h || !A_d || !B_d_list || !x0 || !x_d || (!H && !g && !A_qp && !B_qp)) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.horizon, n = 12 * N;
  const bool dev = is_device_ptr(A_d);
  {
    const void* all_ptrs[] = {B_d_list, x0, x_d, H, g, A_qp, B_qp};
    for (const void* q : all_ptrs)
      if (q && is_device_ptr(q) != dev) return fail(A1MPC_EINVAL, "inputs and outputs must be all-host or all-device");
  }
  const size_t Bs = (size_t)B;
  const size_t szA = Bs * 169, szB = Bs * 13 * N * 12, szx0 = Bs * 13, szxd = Bs * 13 * N, szH = H ? Bs * n * n : 0, szg = g ? Bs * n : 0;
  const size_t szAq = A_qp ? Bs * 13 * N * 13 : 0, szBq = B_qp ? Bs * 13 * N * n : 0;
  const double *dA = A_d, *dB = B_d_list, *dx0 = x0, *dxd = x_d;
  double *dH = H, *dg = g, *dAq = A_qp, *dBq = B_qp;
  int rc;
  if (!dev) {
    if ((rc = ensure_side(h, (szA + szB + szx0 + szxd + szH + szg + szAq + szBq) * 8))) return rc;
    double* p = (double*)h->d_side;
    CK(cudaMemcpyAsync(p, A_d, szA * 8, cudaMemcpyHostToDevice, h->stream)); dA = p; p += szA;
    CK(cudaMemcpyAsync(p, B_d_list, szB * 8, cudaMemcpyHostToDevice, h->stream)); dB = p; p += szB;
    CK(cudaMemcpyAsync(p, x0, szx0 * 8, cudaMemcpyHostToDevice, h->stream)); dx0 = p; p += szx0;
    CK(cudaMemcpyAsync(p, x_d, szxd * 8, cudaMemcpyHostToDevice, h->stream)); dxd = p; p += szxd;
    if (H) { dH = p; p += szH; }
    if (g) { dg = p; p += szg; }
    if (A_qp) { dAq = p; p += szAq; }
    if (B_qp) { dBq = p; p += szBq; }
  }
  {
    cudaError_t e = dense_qp_mats_launch(h->P, B, dA, dB, dx0, dxd, dH, dg, dAq, dBq, h->stream);
    if (e != cudaSuccess) return fail(A1MPC_ECUDA, std::string("qp_mats kernel: ") + cudaGetErrorString(e));
    h->launches += 1;
  }
  if (!dev) {
    if (H) CK(cudaMemcpyAsync(H, dH, szH * 8, cudaMemcpyDeviceToHost, h->stream));
    if (g) CK(cudaMemcpyAsync(g, dg, szg * 8, cudaMemcpyDeviceToHost, h->stream));
    if (A_qp) CK(cudaMemcpyAsync(A_qp, dAq, szAq * 8, cudaMemcpyDeviceToHost, h->stream));
    if (B_qp) CK(cudaMemcpyAsync(B_qp, dBq, szBq * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return A1MPC_OK;
}

int a1mpc_qp_mats_batch(a1mpc_handle* h, int B, const double* A_d, const double* B_d_list, const double* x0, const double* x_d,
                        double* H, double* g) {
  if (!H && !g) return fail(A1MPC_EINVAL, "null argument");
  return qp_mats_impl(h, B, A_d, B_d_list, x0, x_d, H, g, nullptr, nullptr);
}

int a1mpc_qp_rollout_batch(a1mpc_handle* h, int B, const double* A_d, const double* B_d_list, const double* x0, const double* x_d,
                           double* A_qp, double* B_qp, double* H, double* g) {
  return qp_mats_impl(h, B, A_d, B_d_list, x0, x_d, H, g, A_qp, B_qp);
}

int a1mpc_solve_dense_batch(a1mpc_handle* h, int B, const double* H, const double* g, const uint32_t* contact, double* u, int32_t* status) {
  if (!h || !H || !g || !contact || !u || !status) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.horizon, n = 12 * N;
  const bool dev = is_device_ptr(H);
  if (mixed_sides(dev, {g, contact, u, status})) return fail(A1MPC_EINVAL, "inputs and outputs must be all-host or all-device");
  const size_t Bs = (size_t)B;
  const double *dH = H, *dg = g;
  const uint32_t* dc = contact;
  double* du = u;
  int32_t* ds = status;
  int rc;
  const size_t list_bytes = (4 * Bs + 8) * sizeof(int);
  if ((rc = ensure_lists(h, list_bytes))) return rc;
  if (!dev) {
    const size_t bytes = (Bs * n * n + 2 * Bs * n) * 8 + Bs * 8;
    if ((rc = ensure_side(h, bytes))) return rc;
    double* p = (double*)h->d_side;
    CK(cudaMemcpyAsync(p, H, Bs * n * n * 8, cudaMemcpyHostToDevice, h->stream)); dH = p; p += Bs * n * n;
    CK(cudaMemcpyAsync(p, g, Bs * n * 8, cudaMemcpyHostToDevice, h->stream)); dg = p; p += Bs * n;
    du = p; p += Bs * n;
    uint32_t* pc = (uint32_t*)p;
    CK(cudaMemcpyAsync(pc, contact, Bs * 4, cudaMemcpyHostToDevice, h->stream)); dc = pc;
    ds = (int32_t*)(pc + Bs);
  }
  {
    int nl = 0;
    cudaError_t e = dense_solve_launch(h->P, h->sm_count, B, dH, dg, dc, du, ds, h->d_lists, h->stream, &nl);
    if (e != cudaSuccess) return fail(A1MPC_ECUDA, std::string("dense solve kernels: ") + cudaGetErrorString(e));
    h->launches += nl;
  }
  if (!dev) {
    CK(cudaMemcpyAsync(u, du, Bs * n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(status, ds, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return A1MPC_OK;
}

int a1mpc_grf_qp_batch(a1mpc_handle* h, int B, const double* root_acc, const double* rot_z, const double* rot, const double* foot,
                       const uint32_t* contact, double* f_body, int32_t* status) {
  if (!h || !root_acc || !rot_z || !rot || !foot || !contact || !f_body || !status) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  CK(cudaSetDevice(h->device));
  const bool dev = is_device_ptr(root_acc);
  if (mixed_sides(dev, {rot_z, rot, foot, contact, f_body, status})) return fail(A1MPC_EINVAL, "inputs and outputs must be all-host or all-device");
  const size_t Bs = (size_t)B;
  const double *da = root_acc, *drz = rot_z, *dr = rot, *dfo = foot;
  const uint32_t* dc = contact;
  double* df = f_body;
  int32_t* ds = status;
  int rc;
  if ((rc = ensure_lists(h, (4 * Bs + 8) * sizeof(int)))) return rc;
  if (!dev) {
    if ((rc = ensure_side(h, Bs * (6 + 9 + 9 + 12 + 12) * 8 + Bs * 8))) return rc;
    double* p = (double*)h->d_side;
    CK(cudaMemcpyAsync(p, root_acc, Bs * 6 * 8, cudaMemcpyHostToDevice, h->stream)); da = p; p += Bs * 6;
    CK(cudaMemcpyAsync(p, rot_z, Bs * 9 * 8, cudaMemcpyHostToDevice, h->stream)); drz = p; p += Bs * 9;
    CK(cudaMemcpyAsync(p, rot, Bs * 9 * 8, cudaMemcpyHostToDevice, h->stream)); dr = p; p += Bs * 9;
    CK(cudaMemcpyAsync(p, foot, Bs * 12 * 8, cudaMemcpyHostToDevice, h->stream)); dfo = p; p += Bs * 12;
    df = p; p += Bs * 12;
    uint32_t* pc = (uint32_t*)p;
    CK(cudaMemcpyAsync(pc, contact, Bs * 4, cudaMemcpyHostToDevice, h->stream)); dc = pc;
    ds = (int32_t*)(pc + Bs);
  }
  {
    int nl = 0;
    cudaError_t e = grf_qp_launch(h->sm_count, B, da, drz, dr, dfo, dc, df, ds, h->d_lists, h->stream, &nl);
    if (e != cudaSuccess) return fail(A1MPC_ECUDA, std::string("grf_qp kernels: ") + cudaGetErrorString(e));
    h->launches += nl;
  }
  if (!dev) {
    CK(cudaMemcpyAsync(f_body, df, Bs * 12 * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(status, ds, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return A1MPC_OK;
}

int a1mpc_joint_torques_batch(a1mpc_handle* h, int B, const double* f_grf, const double* f_kin, const double* jac, const uint32_t* contact,
                              const double* km_foot, const double* torques_gravity, double* tau) {
  if (!h || !f_grf || !f_kin || !jac || !contact || !km_foot || !torques_gravity || !tau) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  CK(cudaSetDevice(h->device));
  const bool dev = is_device_ptr(f_grf);
  if (mixed_sides(dev, {f_kin, jac, contact, tau})) return fail(A1MPC_EINVAL, "batch arrays must be all-host or all-device (km_foot, torques_gravity: always host)");
  if (is_device_ptr(km_foot) || is_device_ptr(torques_gravity)) return fail(A1MPC_EINVAL, "km_foot and torques_gravity are host arrays (batch-uniform parameters)");
  const size_t Bs = (size_t)B;
  TorqueParams P;
  for (int i = 0; i < 3; ++i) P.km[i] = km_foot[i];
  for (int i = 0; i < 12; ++i) P.tg[i] = torques_gravity[i];
  const double *dg = f_grf, *dk = f_kin, *dj = jac;
  const uint32_t* dc = contact;
  double* dt = tau;
  int rc;
  if (!dev) {
    if ((rc = ensure_side(h, Bs * (12 + 12 + 36 + 12) * 8 + Bs * 4))) return rc;
    double* p = (double*)h->d_side;
    CK(cudaMemcpyAsync(p, f_grf, Bs * 12 * 8, cudaMemcpyHostToDevice, h->stream)); dg = p; p += Bs * 12;
    CK(cudaMemcpyAsync(p, f_kin, Bs * 12 * 8, cudaMemcpyHostToDevice, h->stream)); dk = p; p += Bs * 12;
    CK(cudaMemcpyAsync(p, jac, Bs * 36 * 8, cudaMemcpyHostToDevice, h->stream)); dj = p; p += Bs * 36;
    CK(cudaMemcpyAsync(p, tau, Bs * 12 * 8, cudaMemcpyHostToDevice, h->stream)); dt = p; p += Bs * 12;
    uint32_t* pc = (uint32_t*)p;
    CK(cudaMemcpyAsync(pc, contact, Bs * 4, cudaMemcpyHostToDevice, h->stream)); dc = pc;
  }
  joint_torques_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(B, dg, dk, dj, dc, P, dt);
  h->launches++;
  CK(cudaGetLastError());
  if (!dev) {
    CK(cudaMemcpyAsync(tau, dt, Bs * 12 * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return A1MPC_OK;
}

int a1mpc_update_plan_batch(a1mpc_handle* h, int B, const a1mpc_gait_params* gp, double* gait_counter, const double* gait_counter_speed,
                            const uint32_t* movement_mode, const double* lin_vel, const double* lin_vel_d, const double* rot_z,
                            const double* rot, const double* root_pos, uint32_t* plan_contacts, uint32_t* contact_sched,
                            double* t_rel, double* t_abs, double* t_world) {
  if (!h || !gp || !gait_counter || !gait_counter_speed || !movement_mode || !plan_contacts) return fail(A1MPC_EINVAL, "null argument");
  const bool want_t = t_rel || t_abs || t_world;
  if (want_t && (!lin_vel || !lin_vel_d || !rot_z || !rot || !root_pos)) return fail(A1MPC_EINVAL, "foothold targets need lin_vel, lin_vel_d, rot_z, rot, root_pos");
  if (B <= 0 || gp->horizon < 0 || gp->horizon > A1MPC_MAX_HORIZON) return fail(A1MPC_EINVAL, "bad B or horizon");
  CK(cudaSetDevice(h->device));
  GaitDev G;
  G.cpg = gp->counter_per_gait; G.cps = gp->counter_per_swing; G.cdt = gp->control_dt; G.dxl = gp->foot_delta_x_limit; G.dyl = gp->foot_delta_y_limit;
  for (int i = 0; i < 12; ++i) G.dfp[i] = gp->default_foot_pos[i];
  G.N = gp->horizon;
  const bool dev = is_device_ptr(gait_counter);
  const size_t Bs = (size_t)B;
  int rc;
  if (dev) {
    update_plan_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(B, G, gait_counter, gait_counter_speed, movement_mode, lin_vel, lin_vel_d, rot_z, rot, root_pos,
                                                                plan_contacts, contact_sched, t_rel, t_abs, t_world);
    h->launches++;
    CK(cudaGetLastError());
    return A1MPC_OK;
  }
  // host pointers: stage everything in one scratch allocation
  const size_t nd = Bs * (4 + 4 + 3 + 3 + 9 + 9 + 3 + 36), nu = Bs * (1 + 1 + (size_t)G.N);
  if ((rc = ensure_side(h, nd * 8 + nu * 4))) return rc;
  double* p = (double*)h->d_side;
  double* d_gc = p; p += 4 * Bs;
  double* d_gcs = p; p += 4 * Bs;
  double* d_lv = p; p += 3 * Bs;
  double* d_lvd = p; p += 3 * Bs;
  double* d_rz = p; p += 9 * Bs;
  double* d_r = p; p += 9 * Bs;
  double* d_pos = p; p += 3 * Bs;
  double* d_trel = p; p += 12 * Bs;
  double* d_tabs = p; p += 12 * Bs;
  double* d_tw = p; p += 12 * Bs;
  uint32_t* u = (uint32_t*)p;
  uint32_t* d_mode = u; u += Bs;
  uint32_t* d_plan = u; u += Bs;
  uint32_t* d_sched = u;
  CK(cudaMemcpyAsync(d_gc, gait_counter, 4 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_gcs, gait_counter_speed, 4 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(d_mode, movement_mode, Bs * 4, cudaMemcpyHostToDevice, h->stream));
  if (want_t) {
    CK(cudaMemcpyAsync(d_lv, lin_vel, 3 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_lvd, lin_vel_d, 3 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_rz, rot_z, 9 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_r, rot, 9 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_pos, root_pos, 3 * Bs * 8, cudaMemcpyHostToDevice, h->stream));
  }
  update_plan_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(B, G, d_gc, d_gcs, d_mode, d_lv, d_lvd, d_rz, d_r, d_pos, d_plan, contact_sched ? d_sched : nullptr,
                                                              t_rel ? d_trel : nullptr, t_abs ? d_tabs : nullptr, t_world ? d_tw : nullptr);
  h->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(gait_counter, d_gc, 4 * Bs * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(plan_contacts, d_plan, Bs * 4, cudaMemcpyDeviceToHost, h->stream));
  if (contact_sched) CK(cudaMemcpyAsync(contact_sched, d_sched, (size_t)G.N * Bs * 4, cudaMemcpyDeviceToHost, h->stream));
  if (t_rel) CK(cudaMemcpyAsync(t_rel, d_trel, 12 * Bs * 8, cudaMemcpyDeviceToHost, h->stream));
  if (t_abs) CK(cudaMemcpyAsync(t_abs, d_tabs, 12 * Bs * 8, cudaMemcpyDeviceToHost, h->stream));
  if (t_world) CK(cudaMemcpyAsync(t_world, d_tw, 12 * Bs * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return A1MPC_OK;
}

// ---- upstream producers of the path's inputs (SURVEY 8f.4) ---------------------------------------------------
}  // extern "C"
namespace {
// host-pointer mode of the side entry points: inputs are staged into h->d_side, outputs copied back after the kernel
struct Stage {
  a1mpc_handle* h;
  bool host;
  char* cur = nullptr;
  struct Out { void* host; const void* dev; size_t bytes; };
  std::vector<Out> outs;
  static size_t pad(size_t b) { return (b + 255) & ~(size_t)255; }
  template <class T>
  int in(const T*& p, size_t bytes) {
    if (!host || !p) return A1MPC_OK;
    CK(cudaMemcpyAsync(cur, p, bytes, cudaMemcpyHostToDevice, h->stream));
    p = reinterpret_cast<const T*>(cur);
    cur += pad(bytes);
    return A1MPC_OK;
  }
  template <class T>
  void out(T*& p, size_t bytes) {
    if (!host || !p) return;
    outs.push_back({p, cur, bytes});
    p = reinterpret_cast<T*>(cur);
    cur += pad(bytes);
  }
  int finish() {
    if (!host) return A1MPC_OK;
    for (const Out& o : outs) CK(cudaMemcpyAsync(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return A1MPC_OK;
  }
};
}  // namespace
extern "C" {

int a1mpc_leg_kinematics_batch(a1mpc_handle* h, int B, const double* joint_pos, const double* joint_vel, const double* rot,
                               const double* rho_opt, const double* rho_fix, double* foot_pos_rel, double* jac, double* foot_vel_rel,
                               double* foot_pos_abs, double* foot_vel_abs) {
  if (!h || !joint_pos || !rho_opt || !rho_fix) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  if ((foot_vel_rel || foot_vel_abs) && !joint_vel) return fail(A1MPC_EINVAL, "foot velocities need joint_vel");
  if ((foot_pos_abs || foot_vel_abs) && !rot) return fail(A1MPC_EINVAL, "body-aligned outputs need rot");
  CK(cudaSetDevice(h->device));
  const size_t Bs = (size_t)B;
  LegParams P;
  for (int i = 0; i < 12; ++i) P.rho_opt[i] = rho_opt[i];
  for (int i = 0; i < 20; ++i) P.rho_fix[i] = rho_fix[i];
  Stage st{h, !is_device_ptr(joint_pos)};
  int rc;
  if (st.host) {
    if ((rc = ensure_side(h, 8 * Stage::pad(36 * Bs * 8)))) return rc;
    st.cur = (char*)h->d_side;
  }
  if ((rc = st.in(joint_pos, 12 * Bs * 8))) return rc;
  if ((rc = st.in(joint_vel, 12 * Bs * 8))) return rc;
  if ((rc = st.in(rot, 9 * Bs * 8))) return rc;
  st.out(foot_pos_rel, 12 * Bs * 8); st.out(jac, 36 * Bs * 8); st.out(foot_vel_rel, 12 * Bs * 8);
  st.out(foot_pos_abs, 12 * Bs * 8); st.out(foot_vel_abs, 12 * Bs * 8);
  leg_kinematics_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(B, joint_pos, joint_vel, rot, P, foot_pos_rel, jac, foot_vel_rel, foot_pos_abs, foot_vel_abs);
  h->launches++;
  CK(cudaGetLastError());
  return st.finish();
}

size_t a1mpc_ekf_bytes(int B) { return B > 0 ? (size_t)B * EKF_STATE_DOUBLES * sizeof(double) : 0; }

int a1mpc_ekf_init_batch(a1mpc_handle* h, int B, void* ekf_state, const double* foot_pos_rel, const double* rot) {
  if (!h || !ekf_state || !foot_pos_rel || !rot) return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  CK(cudaSetDevice(h->device));
  if (!is_device_ptr(ekf_state)) return fail(A1MPC_EINVAL, "ekf_state must be device memory (a1mpc_device_alloc)");
  const size_t Bs = (size_t)B;
  Stage st{h, !is_device_ptr(foot_pos_rel)};
  int rc;
  if (st.host) {
    if ((rc = ensure_side(h, 2 * Stage::pad(12 * Bs * 8)))) return rc;
    st.cur = (char*)h->d_side;
  }
  if ((rc = st.in(foot_pos_rel, 12 * Bs * 8))) return rc;
  if ((rc = st.in(rot, 9 * Bs * 8))) return rc;
  ekf_init_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(B, static_cast<double*>(ekf_state), foot_pos_rel, rot);
  h->launches++;
  CK(cudaGetLastError());
  return st.finish();
}

int a1mpc_ekf_update_batch(a1mpc_handle* h, int B, void* ekf_state, double dt, int assume_flat_ground, const uint32_t* movement_mode,
                           const double* imu_acc, const double* imu_ang_vel, const double* rot, const double* foot_pos_rel,
                           const double* foot_vel_rel, const double* foot_force, double* root_pos, double* root_lin_vel,
                           uint32_t* estimated_contacts, int32_t* status) {
  if (!h || !ekf_state || !movement_mode || !imu_acc || !imu_ang_vel || !rot || !foot_pos_rel || !foot_vel_rel || !foot_force)
    return fail(A1MPC_EINVAL, "null argument");
  if (B <= 0) return fail(A1MPC_EINVAL, "B must be positive");
  if (!(dt > 0.0)) return fail(A1MPC_EINVAL, "dt must be positive");
  CK(cudaSetDevice(h->device));
  if (!is_device_ptr(ekf_state)) return fail(A1MPC_EINVAL, "ekf_state must be device memory (a1mpc_device_alloc)");
  static bool attr_set[64] = {};
  const size_t smem = (size_t)EKF_WPC * EKF_WARP_DOUBLES * sizeof(double);
  if (h->device < 64 && !attr_set[h->device]) {
    CK(cudaFuncSetAttribute(ekf_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[h->device] = true;
  }
  const size_t Bs = (size_t)B;
  Stage st{h, !is_device_ptr(imu_acc)};
  int rc;
  if (st.host) {
    if ((rc = ensure_side(h, 12 * Stage::pad(12 * Bs * 8)))) return rc;
    st.cur = (char*)h->d_side;
  }
  if ((rc = st.in(movement_mode, Bs * 4))) return rc;
  if ((rc = st.in(imu_acc, 3 * Bs * 8))) return rc;
  if ((rc = st.in(imu_ang_vel, 3 * Bs * 8))) return rc;
  if ((rc = st.in(rot, 9 * Bs * 8))) return rc;
  if ((rc = st.in(foot_pos_rel, 12 * Bs * 8))) return rc;
  if ((rc = st.in(foot_vel_rel, 12 * Bs * 8))) return rc;
  if ((rc = st.in(foot_force, 4 * Bs * 8))) return rc;
  st.out(root_pos, 3 * Bs * 8); st.out(root_lin_vel, 3 * Bs * 8); st.out(estimated_contacts, Bs * 4); st.out(status, Bs * 4);
  EkfParams P{dt, assume_flat_ground ? 1 : 0};
  int grid = (B + EKF_WPC - 1) / EKF_WPC;
  if (grid > h->sm_count * 2) grid = h->sm_count * 2;
  ekf_update_kernel<<<grid, 32 * EKF_WPC, smem, h->stream>>>(B, P, static_cast<double*>(ekf_state), movement_mode, imu_acc, imu_ang_vel, rot,
                                                             foot_pos_rel, foot_vel_rel, foot_force, root_pos, root_lin_vel, estimated_contacts, status);
  h->launches++;
  CK(cudaGetLastError());
  return st.finish();
}

// ---- helpers -------------------------------------------------------------------------------
int a1mpc_device_alloc(a1mpc_handle* h, size_t bytes, void** ptr) {
  if (!h || !ptr) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  if (cudaMalloc(ptr, bytes) != cudaSuccess) { cudaGetLastError(); return fail(A1MPC_ENOMEM, "cudaMalloc failed"); }
  return A1MPC_OK;
}
int a1mpc_device_free(a1mpc_handle* h, void* ptr) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaFree(ptr));
  return A1MPC_OK;
}
int a1mpc_host_alloc(a1mpc_handle* h, size_t bytes, void** ptr) {
  if (!h || !ptr) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  if (cudaMallocHost(ptr, bytes) != cudaSuccess) { cudaGetLastError(); return fail(A1MPC_ENOMEM, "cudaMallocHost failed"); }
  return A1MPC_OK;
}
int a1mpc_host_free(a1mpc_handle* h, void* ptr) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaFreeHost(ptr));
  return A1MPC_OK;
}
int a1mpc_memcpy_h2d(a1mpc_handle* h, void* dst, const void* src, size_t bytes) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
  return A1MPC_OK;
}
int a1mpc_memcpy_d2h(a1mpc_handle* h, void* dst, const void* src, size_t bytes) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
  return A1MPC_OK;
}
static int join_gather(a1mpc_handle* h) {
  if (h->gather_pending) {   // the compute stream (and everything timed on it) waits for the outstanding collect
    CK(cudaStreamWaitEvent(h->stream, h->ev_gather_done, 0));
    h->gather_pending = false;
  }
  return A1MPC_OK;
}

int a1mpc_sync(a1mpc_handle* h) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  { int rc = join_gather(h); if (rc) return rc; }
  CK(cudaStreamSynchronize(h->stream));
  return A1MPC_OK;
}
int a1mpc_event_create(a1mpc_handle* h, void** ev) {
  if (!h || !ev) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  cudaEvent_t e;
  CK(cudaEventCreate(&e));
  *ev = (void*)e;
  return A1MPC_OK;
}
int a1mpc_event_destroy(a1mpc_handle* h, void* ev) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaEventDestroy((cudaEvent_t)ev));
  return A1MPC_OK;
}
int a1mpc_event_record(a1mpc_handle* h, void* ev) {
  if (!h || !ev) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  { int rc = join_gather(h); if (rc) return rc; }
  CK(cudaEventRecord((cudaEvent_t)ev, h->stream));
  return A1MPC_OK;
}
int a1mpc_event_elapsed_ms(a1mpc_handle* h, void* start, void* stop, float* ms) {
  if (!h || !start || !stop || !ms) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaEventSynchronize((cudaEvent_t)stop));
  CK(cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop));
  return A1MPC_OK;
}
int64_t a1mpc_launch_count(const a1mpc_handle* h) { return h ? h->launches : 0; }

int a1mpc_measure_fp64_peak(a1mpc_handle* h, double* tflops) {
  if (!h || !tflops) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  const int threads = 256, blocks = h->sm_count * 8, iters = 1 << 16;
  int rc;
  if ((rc = ensure_side(h, (size_t)threads * blocks * 8))) return rc;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    CK(cudaEventRecord(e0, h->stream));
    fp64_peak_kernel<<<blocks, threads, 0, h->stream>>>((double*)h->d_side, iters);
    h->launches++;
    CK(cudaEventRecord(e1, h->stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * (double)iters * threads * blocks;
    if (rep > 0) best = std::max(best, fl / (ms * 1e-3) * 1e-12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops = best;
  return A1MPC_OK;
}

int a1mpc_profile_begin(a1mpc_handle* h, int max_calls) {
  if (!h || max_calls <= 0) return fail(A1MPC_EINVAL, "bad argument");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  while ((int)h->prof_ev.size() < max_calls * 8) {
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    h->prof_ev.push_back(e);
  }
  h->prof_cap = max_calls;
  h->prof_n = 0;
  h->prof_on = true;
  return A1MPC_OK;
}

int a1mpc_profile_end(a1mpc_handle* h, double* ms_per_class4, int* calls) {
  if (!h || !ms_per_class4) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  for (int k = 0; k < 4; ++k) ms_per_class4[k] = 0.0;
  for (int c = 0; c < h->prof_n; ++c)
    for (int k = 0; k < 4; ++k) {
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, h->prof_ev[((size_t)c * 4 + k) * 2], h->prof_ev[((size_t)c * 4 + k) * 2 + 1]));
      ms_per_class4[k] += ms;
    }
  if (calls) *calls = h->prof_n;
  h->prof_on = false;
  return A1MPC_OK;
}

int a1mpc_flush_l2(a1mpc_handle* h) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  if (!h->d_flush) {
    h->flush_elems = (size_t)256 * 1024 * 1024 / 8;  // 256 MiB > 126 MB L2
    if (cudaMalloc(&h->d_flush, h->flush_elems * 8) != cudaSuccess) { cudaGetLastError(); return fail(A1MPC_ENOMEM, "cudaMalloc failed"); }
  }
  flush_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>(h->d_flush, h->flush_elems, 1.0);
  h->launches++;
  CK(cudaGetLastError());
  return A1MPC_OK;
}

/* ---- fused final collect over peer memory (one process per GPU, CUDA IPC) ------------------------------------------------ */
int a1mpc_peer_gather_create(a1mpc_handle* h, int nranks, int rank, int B_local, void* ipc_handle64) {
  if (!h || !ipc_handle64 || nranks < 1 || nranks > MAX_PEERS || rank < 0 || rank >= nranks || B_local <= 0) return fail(A1MPC_EINVAL, "bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t");
  CK(cudaSetDevice(h->device));
  a1mpc_peer_gather_destroy(h);
  auto& pg = h->peer;
  const size_t fbytes = (size_t)nranks * 12 * (size_t)B_local * 8;
  const size_t bytes = fbytes + (size_t)MAX_PEERS * 8 + 64;
  CK(cudaMalloc(&pg.local, bytes));
  CK(cudaMemset(pg.local, 0, bytes));
  pg.nranks = nranks; pg.rank = rank; pg.B = (size_t)B_local; pg.step = 0;
  pg.buf[rank] = (double*)pg.local;
  pg.flags[rank] = (unsigned long long*)((char*)pg.local + fbytes);
  cudaIpcMemHandle_t hd;
  CK(cudaIpcGetMemHandle(&hd, pg.local));
  std::memcpy(ipc_handle64, &hd, 64);
  return A1MPC_OK;
}

int a1mpc_peer_gather_connect(a1mpc_handle* h, const void* all_handles) {
  if (!h || !all_handles) return fail(A1MPC_EINVAL, "null argument");
  auto& pg = h->peer;
  if (!pg.local) return fail(A1MPC_EINVAL, "a1mpc_peer_gather_create first");
  CK(cudaSetDevice(h->device));
  const size_t fbytes = (size_t)pg.nranks * 12 * pg.B * 8;
  for (int p = 0; p < pg.nranks; ++p) {
    if (p == pg.rank) continue;
    cudaIpcMemHandle_t hd;
    std::memcpy(&hd, (const char*)all_handles + 64 * (size_t)p, 64);
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(A1MPC_ECUDA, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(p) + "): " + cudaGetErrorString(e));
    pg.buf[p] = (double*)ptr;
    pg.flags[p] = (unsigned long long*)((char*)ptr + fbytes);
    pg.opened[p] = true;
  }
  pg.connected = true;
  return A1MPC_OK;
}

int a1mpc_peer_gather_buffer(a1mpc_handle* h, double** f_all) {
  if (!h || !f_all) return fail(A1MPC_EINVAL, "null argument");
  if (!h->peer.local) return fail(A1MPC_EINVAL, "a1mpc_peer_gather_create first");
  *f_all = (double*)h->peer.local;
  return A1MPC_OK;
}

int a1mpc_peer_gather_wait(a1mpc_handle* h) {
  if (!h) return fail(A1MPC_EINVAL, "null argument");
  auto& pg = h->peer;
  if (!pg.connected) return fail(A1MPC_EINVAL, "a1mpc_peer_gather_connect first");
  CK(cudaSetDevice(h->device));
  int* err = (int*)((char*)pg.local + (size_t)pg.nranks * 12 * pg.B * 8 + (size_t)MAX_PEERS * 8);
  // like the NCCL collect, the wait runs on the collect stream, forked after everything enqueued so far (this rank's signal included):
  // the next solve is not held back by a slower peer; a1mpc_sync / a1mpc_event_record join it.  (Measured with the wait on the
  // compute stream, 2 x B200, B = 1024: 0.456 ms per step against 0.414 without any collect -- every step then ends in lock-step with
  // the slowest rank; profiles/r02_notes.md.)
  cudaStream_t gs = (cudaStream_t)a1mpc_internal_gather_begin(h);
  if (!gs) return fail(A1MPC_ECUDA, "could not create the collect stream");
  // Preferred: stream memory operations (cuStreamWaitValue64, >=): the wait is done by the GPU's front end and occupies no SM.  A
  // spinning wait KERNEL sits on one SM for most of every step once the compute stream runs ahead, and since the persistent solve
  // kernels split their queue statically, one perturbed SM stretches the whole launch: measured +0.67 ms per 6.1 ms step at
  // 2 x 32768 QPs (profiles/r02_notes.md).  The kernel (polling every 5 us, ~2 s cap) remains as the fallback.
  typedef int (*wait_value_fn)(cudaStream_t, unsigned long long, unsigned long long, unsigned int);
  static wait_value_fn wait_value = nullptr;
  static bool looked_up = false;
  if (!looked_up) {
    looked_up = true;
    const char* ev = std::getenv("A1MPC_PEER_WAIT_KERNEL");
    if (!(ev && ev[0] == '1')) {
      void* fn = nullptr;
      cudaDriverEntryPointQueryResult qres;
      if (cudaGetDriverEntryPoint("cuStreamWaitValue64", &fn, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
        wait_value = (wait_value_fn)fn;
      else
        cudaGetLastError();
    }
  }
  bool done = false;
  if (wait_value) {
    done = true;
    for (int p = 0; p < pg.nranks && done; ++p)
      if (wait_value(gs, (unsigned long long)(uintptr_t)(pg.flags[pg.rank] + p), pg.step, 0u /* CU_STREAM_WAIT_VALUE_GEQ */) != 0) done = false;
    if (!done) { wait_value = nullptr; cudaGetLastError(); }   // not supported on this memory / driver: use the kernel from now on
    else h->launches += 0;
  }
  if (!done) {
    peer_wait_kernel<<<1, 32, 0, gs>>>(pg.flags[pg.rank], pg.nranks, pg.step, (long long)4e9 /* ~2 s */, err);
    h->launches++;
    CK(cudaGetLastError());
  }
  a1mpc_internal_gather_end(h);
  return A1MPC_OK;
}

int a1mpc_peer_gather_status(a1mpc_handle* h, int* timed_out_rank_plus_1) {
  if (!h || !timed_out_rank_plus_1) return fail(A1MPC_EINVAL, "null argument");
  auto& pg = h->peer;
  if (!pg.local) return fail(A1MPC_EINVAL, "a1mpc_peer_gather_create first");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaMemcpy(timed_out_rank_plus_1, (char*)pg.local + (size_t)pg.nranks * 12 * pg.B * 8 + (size_t)MAX_PEERS * 8, sizeof(int), cudaMemcpyDeviceToHost));
  return A1MPC_OK;
}

int a1mpc_peer_gather_destroy(a1mpc_handle* h) {
  if (!h) return A1MPC_OK;
  auto& pg = h->peer;
  if (!pg.local) return A1MPC_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (int p = 0; p < MAX_PEERS; ++p) {
    if (pg.opened[p] && pg.buf[p]) cudaIpcCloseMemHandle(pg.buf[p]);
    pg.opened[p] = false; pg.buf[p] = nullptr; pg.flags[p] = nullptr;
  }
  cudaFree(pg.local);
  pg.local = nullptr; pg.connected = false; pg.nranks = 0; pg.B = 0;
  return A1MPC_OK;
}

}  // extern "C"

// accessors for a1mpc_nccl.cpp (which must not see the handle layout)
extern "C" {
void* a1mpc_internal_stream(a1mpc_handle* h) { return (void*)h->stream; }
// forks the collect stream off the compute stream (everything enqueued so far is visible to the collective) and returns it
void* a1mpc_internal_gather_begin(a1mpc_handle* h) {
  if (!h->gather_stream) {
    if (cudaStreamCreateWithFlags(&h->gather_stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    cudaEventCreateWithFlags(&h->ev_gather_in, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_gather_done, cudaEventDisableTiming);
  }
  cudaEventRecord(h->ev_gather_in, h->stream);
  cudaStreamWaitEvent(h->gather_stream, h->ev_gather_in, 0);
  return (void*)h->gather_stream;
}
void a1mpc_internal_gather_end(a1mpc_handle* h) {
  cudaEventRecord(h->ev_gather_done, h->gather_stream);
  h->gather_pending = true;
}
int a1mpc_internal_device(a1mpc_handle* h) { return h->device; }
void** a1mpc_internal_nccl_slot(a1mpc_handle* h) { return &h->nccl_comm; }
void a1mpc_internal_set_error(const char* msg) { g_err = msg; }
}
