// a1mpc_sched.cuh -- BASELINE config 4, compacted: per-step contact schedules in which EVERY horizon step has exactly two stance
// feet (trot, bound, pace, any phase) are a 3*2*N-variable problem -- the size of the reference's trot problem -- although the
// two feet change from step to step.  The general extended kernel (solve_kernel<4,N,.,wrench,EXT>) carries all four legs and pins
// the absent foot-steps; this one eliminates them: H_compact = Sel' (T0 (x) G0 + T1 (x) G1 + 2R) Sel with the full 12 x 12 Gram
// blocks and a (step, leg) selection, solved by the direct 64 x 64 tensor-core core like the trot class.
// OPT-IN this round (A1MPC_EXT_COMPACT=1 in the environment of a1mpc_create): validated on the CPU emulator only.
// Include from a1mpc_solve_ext.cu and tests/emu (the kernel body is a1mpc_sched2_body.inc).
#pragma once
#include "a1mpc_device.cuh"

namespace a1mpc {

template <int N>
struct SchedGeo {
  using G2 = Geo<2, N, 0>;
  static constexpr int NPF = (12 * N + 7) / 8 * 8;        // a full (4-leg) vector
  // per-warp extras behind G2::WARP_DOUBLES (doubles)
  static constexpr int X_G = 0;                           // full gradient
  static constexpr int X_G0 = X_G + NPF;                  // 12 x 12 Gram blocks, all four legs
  static constexpr int X_G1 = X_G0 + 144;
  static constexpr int X_R2 = X_G1 + 144;
  static constexpr int X_VP0 = X_R2 + 12;
  static constexpr int X_VP1 = X_VP0 + NPF;
  static constexpr int X_VIN = X_VP1 + NPF;
  static constexpr int X_VOUT = X_VIN + NPF;
  static constexpr int X_LEG = X_VOUT + NPF;              // K ints: leg of foot-step k
  static constexpr int X_TOTAL = (X_LEG + (G2::K + 1) / 2 + 1) / 2 * 2;
  static constexpr int WARP_DOUBLES = G2::WARP_DOUBLES + X_TOTAL;
  static constexpr size_t smem_bytes(int wpc) { return (size_t)(G2::TAB_DOUBLES + wpc * WARP_DOUBLES) * 8; }
};

// vout = sgn * ((T0 (x) G0 + T1 (x) G1 + 2R) vin + gmul * g) on a hand-assembled context (the arithmetic of kron_matvec_impl)
template <int NS, int N>
__device__ __forceinline__ void kron_matvec_ctx(const Ctx<NS, N, 0>& c, const double* __restrict__ vin, double* __restrict__ vout, double sgn,
                                                double gmul) {
  using G = Geo<NS, N, 0>;
  constexpr int A = G::A;
  const int lane = c.lane;
#pragma unroll
  for (int t = 0; t < G::T; ++t) {
    const int i = lane + 32 * t;
    if (i < G::NV) {
      const int s = i / A, a = i - s * A;
      double p0 = 0.0, p1 = 0.0;
#pragma unroll
      for (int sp = 0; sp < N; ++sp) {
        const double x = vin[sp * A + a];
        p0 = fma(c.T0[sp * N + s], x, p0);
        p1 = fma(c.T1[sp * N + s], x, p1);
      }
      c.vp0[i] = p0;
      c.vp1[i] = p1;
    }
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < G::T; ++t) {
    const int i = lane + 32 * t;
    if (i < G::NV) {
      const int s = i / A, a = i - s * A;
      double acc = fma(c.R2[a], vin[i], gmul * c.g[i]);
#pragma unroll
      for (int ap = 0; ap < A; ++ap) {
        acc = fma(c.G0[a * A + ap], c.vp0[s * A + ap], acc);
        acc = fma(c.G1[a * A + ap], c.vp1[s * A + ap], acc);
      }
      vout[i] = sgn * acc;
    }
  }
  __syncwarp();
}

// Hessian provider of the compacted problem: foot-step k = 2 s + f is leg legmap[k] of step s
template <int N>
struct SchedHess {
  using G = Geo<2, N, 0>;
  static constexpr bool kronecker = false;
  Ctx<4, N, 0> cf;        // full-leg quantities (g, G0, G1, R2, vp0, vp1; everything else unused)
  const int* legmap;
  double* vinf;
  double* voutf;
  __device__ __forceinline__ void matvec(const Ctx<2, N, 0>& c, const double* vin, double* vout, double sgn, double gmul = 1.0) const {
    const int lane = c.lane;
    for (int i = lane; i < 12 * N; i += 32) vinf[i] = 0.0;
    __syncwarp();
    for (int i = lane; i < G::NV; i += 32) {
      const int k = i / 3, a = i - 3 * k;
      vinf[12 * (k >> 1) + 3 * legmap[k] + a] = vin[i];
    }
    __syncwarp();
    kron_matvec_ctx<4, N>(cf, vinf, voutf, sgn, gmul);
    for (int i = lane; i < G::NV; i += 32) {
      const int k = i / 3, a = i - 3 * k;
      vout[i] = voutf[12 * (k >> 1) + 3 * legmap[k] + a];
    }
    __syncwarp();
  }
  __device__ __forceinline__ void block(const Ctx<2, N, 0>& c, int k1, int k2, double (&h)[3][3]) const {
    const int s1 = k1 >> 1, s2 = k2 >> 1, l1 = legmap[k1], l2 = legmap[k2];
    const double t0 = c.T0[s1 * N + s2], t1 = c.T1[s1 * N + s2];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        const int ga = (3 * l1 + a) * 12 + 3 * l2 + b;
        h[a][b] = fma(t0, cf.G0[ga], t1 * cf.G1[ga]);
      }
    if (k1 == k2) {
#pragma unroll
      for (int a = 0; a < 3; ++a) h[a][a] += cf.R2[3 * l1 + a];
    }
  }
};

// records: the extended record of pack_ext_kernel (REC_EXT_DOUBLES), queue count[6]
template <int N, int WPC>
__global__ void __launch_bounds__(32 * WPC) solve_kernel_sched2(const __grid_constant__ DevParams P, const double* __restrict__ rec,
                                                                const int* __restrict__ count, DevOutputs out) {
  constexpr bool WARM = false;
  uint32_t* const warm = nullptr;
  const int shift = 0;
#include "a1mpc_sched2_body.inc"
}

// the same kernel with the device-resident warm start (a1mpc_solve_batch_ext_warm; the slot format of WARM_HDR)
template <int N, int WPC>
__global__ void __launch_bounds__(32 * WPC) solve_kernel_sched2_warm(const __grid_constant__ DevParams P, const double* __restrict__ rec,
                                                                     const int* __restrict__ count, DevOutputs out, uint32_t* __restrict__ warm,
                                                                     int shift) {
  constexpr bool WARM = true;
#include "a1mpc_sched2_body.inc"
}

}  // namespace a1mpc
