// emu_warm_ext.cpp -- a1mpc_solve_batch_ext_warm on the CPU block emulator of cuda_emu.h.  TEST INFRASTRUCTURE ONLY: the
// UNCHANGED device code of the extended warm start (solve_kernel_warm<4, N, ., 1, true>, solve_kernel_sched2_warm<10, 4>,
// warm_clear_idle_kernel) run as solve_ext_impl() of a1mpc_api.cu launches it: at N = 10 with a schedule, pack_ext2_kernel
// routes two-feet-per-step robots to the compacted kernel and everything else to the general one.  Built by
// tests/emu/emu_warm_ext.py into liba1mpc_emu_warm_ext.so, next to the emulator of emu_driver.cpp.
#define A1MPC_EMU 1
#include "cuda_emu.h"

#include <atomic>
#include <thread>

#include "../../a1-qp-mpc-controller_b200/csrc/a1mpc_misc.cuh"
#include "../../a1-qp-mpc-controller_b200/csrc/a1mpc_sched.cuh"

using namespace a1mpc;

namespace {

DevParams make_params(const a1mpc_config* cfg) {   // a1mpc_create() in a1mpc_api.cu
  DevParams P;
  P.N = cfg->horizon;
  P.max_iter = cfg->max_iter > 0 ? cfg->max_iter : 40;
  P.dt = cfg->dt; P.mu = cfg->mu; P.fzmax = cfg->fz_max; P.mass = cfg->mass;
  P.mu_switch = cfg->tol > 0.0 ? cfg->tol : MU_SWITCH_DEFAULT;
  for (int i = 0; i < 9; ++i) P.inertia[i] = cfg->inertia[i];
  for (int i = 0; i < 13; ++i) P.q2[i] = 2.0 * cfg->q[i];
  for (int i = 0; i < 12; ++i) P.r2[i] = 2.0 * cfg->r[i];
  return P;
}

// one persistent-grid launch of `nq` queued QPs, ~2 QPs per slot (exercises the queue and the CTA rendezvous), blocks spread
// over host threads
template <class Kernel>
void launch(int nq, int wpc, int threads, size_t smem, int order_mode, int nthreads, Kernel&& kernel) {
  if (nq == 0) return;
  const int grid = std::max(1, (nq + 2 * wpc - 1) / (2 * wpc));
  std::atomic<int> next{0};
  auto worker = [&]() {
    for (;;) {
      const int bx = next.fetch_add(1);
      if (bx >= grid) break;
      a1emu::run_block(a1emu::Dim3{(unsigned)bx, 0, 0}, a1emu::Dim3{(unsigned)grid, 1, 1}, threads, smem, order_mode, kernel);
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < std::max(1, nthreads); ++t) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
}

template <int N, int WPC>
void run_general(const DevParams& P, const double* rec, const int* count, const DevOutputs& out, int order_mode, int nthreads, uint32_t* warm,
                 int shift) {
  using G = Geo<4, N, 1>;
  launch(count[5], WPC, 32 * WPC * G::TW, G::smem_bytes(WPC), order_mode, nthreads,
         [&]() { solve_kernel_warm<4, N, WPC, 1, true>(P, rec, count, out, warm, shift); });
}

}  // namespace

extern "C" {

// Same contract as a1mpc_solve_batch_ext_warm with host pointers; `warm` is a host buffer of B * (4 + 4 * horizon) u32 (zero =
// no guess).  compact = 0: every robot on the general kernel (as A1MPC_EXT_COMPACT=0).  order_mode: lane order between
// collectives (0 ascending, 1 descending, 2 pseudo-random).  queued[0] / [1]: QPs served by the general / compacted kernel.
int emu_solve_ext_warm(const a1mpc_config* cfg, int B, const a1mpc_inputs* in, const uint32_t* sched, const double* normals, const a1mpc_outputs* o,
                       uint32_t* warm, int shift, int compact, int order_mode, int nthreads, int* queued) {
  if (cfg->horizon != 10 && cfg->horizon != 20) return -1;
  if ((!sched && !normals) || !warm || shift < 0 || shift > cfg->horizon) return -2;
  const DevParams P = make_params(cfg);
  const DevInputs din{in->x0, in->rot, in->foot, in->ref, in->contact, in->ld};
  const DevOutputs dout{o->f_body, o->status, o->iters, o->u_full, o->ld};
  const size_t cap = (size_t)B;
  int count[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // [0..7] class counts, [8..15] queue counters (next_qp)
  const bool two = compact && sched && cfg->horizon == 10;             // pack_ext2_kernel: compacted queue behind the first `cap` records
  std::vector<double> rec(cap * (two ? 2 : 1) * (size_t)REC_EXT_DOUBLES + 2);
  const int pb = 128, pgrid = (B + pb - 1) / pb;
  for (int bx = 0; bx < pgrid; ++bx)
    a1emu::run_block(a1emu::Dim3{(unsigned)bx, 0, 0}, a1emu::Dim3{(unsigned)pgrid, 1, 1}, pb, 0, 0, [&]() {
      if (two) pack_ext2_kernel(din, sched, normals, B, rec.data(), (int)cap, count, dout, cfg->horizon);
      else pack_ext_kernel(din, sched, normals, B, rec.data(), count, dout, cfg->horizon);
    });
  if (cfg->horizon == 10) run_general<10, A1MPC_WPC34>(P, rec.data(), count, dout, order_mode, nthreads, warm, shift);
  else run_general<20, 1>(P, rec.data(), count, dout, order_mode, nthreads, warm, shift);
  if (two) {
    const double* rec2 = rec.data() + cap * REC_EXT_DOUBLES;
    launch(count[6], 4, 32 * 4, SchedGeo<10>::smem_bytes(4), order_mode, nthreads,
           [&]() { solve_kernel_sched2_warm<10, 4>(P, rec2, count, dout, warm, shift); });
  }
  for (int bx = 0; bx < pgrid; ++bx)
    a1emu::run_block(a1emu::Dim3{(unsigned)bx, 0, 0}, a1emu::Dim3{(unsigned)pgrid, 1, 1}, pb, 0, 0,
                     [&]() { warm_clear_idle_kernel(in->contact, sched, in->ld, B, cfg->horizon, warm); });
  if (queued) { queued[0] = count[5]; queued[1] = count[6]; }
  return 0;
}

}  // extern "C"
