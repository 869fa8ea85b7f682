// a1mpc_solve_ext.cu -- the fused kernel for BASELINE config 4 (an extension beyond the reference, which has a constant
// contact pattern over the horizon and world-z friction pyramids): per-step contact schedules + per-foot terrain normals.
// It is the 4-foot wrench-space kernel with absent foot-steps pinned to zero (identity rows), forces solved in each
// foot's terrain frame.
#include "a1mpc_internal.h"
#include "a1mpc_sched.cuh"

namespace a1mpc {

// dynamic shared memory attribute + occupancy of one kernel: the persistent grid size of its launches
template <class K>
static cudaError_t setup_kernel(K* kernel, int threads, int sm_count, ClassLaunch& c) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem);
  if (e != cudaSuccess) return e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, c.smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorLaunchOutOfResources;
  c.max_ctas = occ * sm_count;
  c.supported = true;
  return cudaSuccess;
}

// N = 10: 4 warps per CTA like the other wrench-space classes (rendezvous before every factorisation); N = 20: one
template <int N>
constexpr int ext_wpc() { return (N == 10) ? A1MPC_WPC34 : 1; }

template <int N>
static cudaError_t setup_n(int sm_count, ClassLaunch& c, ClassLaunch& cw) {
  using G = Geo<4, N, 1>;
  constexpr int WPC = ext_wpc<N>();
  c.wpc = cw.wpc = WPC;
  c.smem = cw.smem = G::smem_bytes(WPC);
  cudaError_t e = setup_kernel(solve_kernel<4, N, WPC, 1, true>, 32 * WPC * G::TW, sm_count, c);
  if (e != cudaSuccess) return e;
  return setup_kernel(solve_kernel_warm<4, N, WPC, 1, true>, 32 * WPC * G::TW, sm_count, cw);
}

cudaError_t ext_setup(int horizon, int sm_count, ClassLaunch& c, ClassLaunch& cw) {
  return horizon == 10 ? setup_n<10>(sm_count, c, cw) : setup_n<20>(sm_count, c, cw);
}

static int persistent_grid(const ClassLaunch& c, int B) {
  int grid = (B + c.wpc - 1) / c.wpc;
  if (grid > c.max_ctas) grid = c.max_ctas;
  return grid < 1 ? 1 : grid;
}

template <int N>
static void launch_n(const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out,
                     uint32_t* warm, int shift) {
  constexpr int WPC = ext_wpc<N>();
  const int grid = persistent_grid(c, B), threads = 32 * WPC * Geo<4, N, 1>::TW;
  if (warm) solve_kernel_warm<4, N, WPC, 1, true><<<grid, threads, c.smem, st>>>(P, rec, count, out, warm, shift);
  else solve_kernel<4, N, WPC, 1, true><<<grid, threads, c.smem, st>>>(P, rec, count, out);
}

void ext_launch(int horizon, const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out,
                uint32_t* warm, int shift) {
  if (horizon == 10) launch_n<10>(c, st, B, P, rec, count, out, warm, shift);
  else launch_n<20>(c, st, B, P, rec, count, out, warm, shift);
}

cudaError_t sched2_setup(int sm_count, ClassLaunch& c, ClassLaunch& cw) {
  constexpr int WPC = 4;
  c.wpc = cw.wpc = WPC;
  c.smem = cw.smem = SchedGeo<10>::smem_bytes(WPC);
  cudaError_t e = setup_kernel(solve_kernel_sched2<10, WPC>, 32 * WPC, sm_count, c);
  if (e != cudaSuccess) return e;
  return setup_kernel(solve_kernel_sched2_warm<10, WPC>, 32 * WPC, sm_count, cw);
}

void sched2_launch(const ClassLaunch& c, cudaStream_t st, int B, const DevParams& P, const double* rec, const int* count, const DevOutputs& out,
                   uint32_t* warm, int shift) {
  const int grid = persistent_grid(c, B);
  if (warm) solve_kernel_sched2_warm<10, 4><<<grid, 32 * 4, c.smem, st>>>(P, rec, count, out, warm, shift);
  else solve_kernel_sched2<10, 4><<<grid, 32 * 4, c.smem, st>>>(P, rec, count, out);
}

}  // namespace a1mpc
