// a1mpc_misc.cuh -- non-template kernels; include from exactly one translation unit (a1mpc_api.cu)
#pragma once
#include "a1mpc_device.cuh"

namespace a1mpc {

// -------------------------------------------------------------------------------------------
// pack kernel: SoA batch -> per-class records.  Thread-per-QP, every load is a coalesced 64-bit
// batch-major access (32 consecutive QPs per warp instruction).
// -------------------------------------------------------------------------------------------
__global__ void pack_kernel(DevInputs in, int B, double* __restrict__ rec, int cap, int* __restrict__ count,
                            DevOutputs out, int horizon) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const uint32_t mask = in.contact[b] & 15u;
  const int ns = __popc(mask);
  if (ns == 0) {  // every foot is pinned to zero by fz in [0,0] (ConvexMpc.cpp:233,238)
    st_zero_forces(out, b);
    out.status[b] = A1MPC_STATUS_NO_CONTACT;
    if (out.iters) out.iters[b] = 0;
    if (out.u_full)
      for (int k = 0; k < 12 * horizon; ++k) st_out(out.u_full, (size_t)k * out.ld + b, 0.0, out.f32);
    return;
  }
  const int slot = atomicAdd(&count[ns], 1);
  double* r = rec + ((size_t)(ns - 1) * cap + slot) * REC_DOUBLES;
#pragma unroll
  for (int k = 0; k < 12; ++k) r[k] = ld_in(in.x0, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 9; ++k) r[12 + k] = ld_in(in.rot, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 12; ++k) r[21 + k] = ld_in(in.foot, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 9; ++k) r[33 + k] = ld_in(in.ref, (size_t)k * in.ld + b, in.f32);
  r[42] = __hiloint2double((int)mask, b);
  r[43] = 0.0;
}

// pack kernel of the extended path: one 464-byte record per QP (base record + per-step contact masks + unit normals)
__global__ void pack_ext_kernel(DevInputs in, const uint32_t* __restrict__ sched, const double* __restrict__ normals, int B,
                                double* __restrict__ rec, int* __restrict__ count, DevOutputs out, int horizon) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  unsigned long long s0 = 0ull, s1 = 0ull;
  for (int st = 0; st < horizon; ++st) {
    const unsigned long long m = (sched ? sched[(size_t)st * in.ld + b] : in.contact[b]) & 15u;
    if (st < 16) s0 |= m << (4 * st);
    else s1 |= m << (4 * (st - 16));
  }
  if (s0 == 0ull && s1 == 0ull) {
    st_zero_forces(out, b);
    out.status[b] = A1MPC_STATUS_NO_CONTACT;
    if (out.iters) out.iters[b] = 0;
    if (out.u_full)
      for (int k = 0; k < 12 * horizon; ++k) st_out(out.u_full, (size_t)k * out.ld + b, 0.0, out.f32);
    return;
  }
  const int slot = atomicAdd(&count[5], 1);
  double* r = rec + (size_t)slot * REC_EXT_DOUBLES;
#pragma unroll
  for (int k = 0; k < 12; ++k) r[k] = ld_in(in.x0, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 9; ++k) r[12 + k] = ld_in(in.rot, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 12; ++k) r[21 + k] = ld_in(in.foot, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 9; ++k) r[33 + k] = ld_in(in.ref, (size_t)k * in.ld + b, in.f32);
  r[42] = __hiloint2double((int)(s0 & 15ull), b);
  r[43] = 0.0;
  r[44] = __longlong_as_double((long long)s0);
  r[45] = __longlong_as_double((long long)s1);
  for (int leg = 0; leg < 4; ++leg) {
    double nx = 0.0, ny = 0.0, nz = 1.0;
    if (normals) {
      nx = ld_in(normals, (size_t)(3 * leg) * in.ld + b, in.f32); ny = ld_in(normals, (size_t)(3 * leg + 1) * in.ld + b, in.f32); nz = ld_in(normals, (size_t)(3 * leg + 2) * in.ld + b, in.f32);
      const double inv = rsqrt(nx * nx + ny * ny + nz * nz);
      nx *= inv; ny *= inv; nz *= inv;
      // a terrain normal must point out of the ground (nz > 0, include/a1mpc.h): anything else is poisoned here and comes back as
      // A1MPC_STATUS_NUMERICAL with zero forces from the solve kernel's input check instead of being clamped silently
      if (!(nz > 0.0)) { nx = ny = nz = __longlong_as_double(0x7ff8000000000000ll); }
    }
    r[46 + 3 * leg] = nx; r[47 + 3 * leg] = ny; r[48 + 3 * leg] = nz;
  }
}

// pack kernel of the extended path with the compacted class (A1MPC_EXT_COMPACT): schedules with exactly two stance feet in every
// horizon step go to queue 6 (records behind the first `cap` records), everything else to queue 5 as in pack_ext_kernel
__global__ void pack_ext2_kernel(DevInputs in, const uint32_t* __restrict__ sched, const double* __restrict__ normals, int B,
                                 double* __restrict__ rec, int cap, int* __restrict__ count, DevOutputs out, int horizon) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  unsigned long long s0 = 0ull, s1 = 0ull;
  bool two = true;
  for (int st = 0; st < horizon; ++st) {
    const unsigned long long m = (sched ? sched[(size_t)st * in.ld + b] : in.contact[b]) & 15u;
    two = two && (__popc((unsigned)m) == 2);
    if (st < 16) s0 |= m << (4 * st);
    else s1 |= m << (4 * (st - 16));
  }
  if (s0 == 0ull && s1 == 0ull) {
    st_zero_forces(out, b);
    out.status[b] = A1MPC_STATUS_NO_CONTACT;
    if (out.iters) out.iters[b] = 0;
    if (out.u_full)
      for (int k = 0; k < 12 * horizon; ++k) st_out(out.u_full, (size_t)k * out.ld + b, 0.0, out.f32);
    return;
  }
  const int slot = atomicAdd(&count[two ? 6 : 5], 1);
  double* r = rec + ((two ? (size_t)cap : (size_t)0) + (size_t)slot) * REC_EXT_DOUBLES;
#pragma unroll
  for (int k = 0; k < 12; ++k) r[k] = ld_in(in.x0, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 9; ++k) r[12 + k] = ld_in(in.rot, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 12; ++k) r[21 + k] = ld_in(in.foot, (size_t)k * in.ld + b, in.f32);
#pragma unroll
  for (int k = 0; k < 9; ++k) r[33 + k] = ld_in(in.ref, (size_t)k * in.ld + b, in.f32);
  r[42] = __hiloint2double((int)(s0 & 15ull), b);
  r[43] = 0.0;
  r[44] = __longlong_as_double((long long)s0);
  r[45] = __longlong_as_double((long long)s1);
  for (int leg = 0; leg < 4; ++leg) {
    double nx = 0.0, ny = 0.0, nz = 1.0;
    if (normals) {
      nx = ld_in(normals, (size_t)(3 * leg) * in.ld + b, in.f32); ny = ld_in(normals, (size_t)(3 * leg + 1) * in.ld + b, in.f32); nz = ld_in(normals, (size_t)(3 * leg + 2) * in.ld + b, in.f32);
      const double inv = rsqrt(nx * nx + ny * ny + nz * nz);
      nx *= inv; ny *= inv; nz *= inv;
      // a terrain normal must point out of the ground (nz > 0, include/a1mpc.h): anything else is poisoned here and comes back as
      // A1MPC_STATUS_NUMERICAL with zero forces from the solve kernel's input check instead of being clamped silently
      if (!(nz > 0.0)) { nx = ny = nz = __longlong_as_double(0x7ff8000000000000ll); }
    }
    r[46 + 3 * leg] = nx; r[47 + 3 * leg] = ny; r[48 + 3 * leg] = nz;
  }
}

// a1mpc_solve_batch_ext_warm: a robot with no foot in contact anywhere in the horizon never reaches a solve kernel (the pack
// kernels answer NO_CONTACT); its slot is marked "no guess" here, as the solve kernels do for every result that is not OPTIMAL
__global__ void warm_clear_idle_kernel(const uint32_t* __restrict__ contact, const uint32_t* __restrict__ sched, size_t ld, int B, int horizon,
                                       uint32_t* __restrict__ warm) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  uint32_t any = 0u;
  for (int st = 0; st < horizon; ++st) any |= (sched ? sched[(size_t)st * ld + b] : contact[b]) & 15u;
  if (any == 0u) warm[(size_t)b * (WARM_HDR + 4 * horizon)] = 0u;
}

// Classes whose factor does not fit in shared memory (N=20 with four stance feet in fp64):
// reported, never silently approximated.
__global__ void unsupported_kernel(const double* __restrict__ rec, const int* __restrict__ count, int cls, DevOutputs out, int horizon) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= count[cls]) return;
  const int b = __double2loint(rec[(size_t)q * REC_DOUBLES + 42]);
  st_zero_forces(out, b);
  out.status[b] = A1MPC_STATUS_NUMERICAL;
  if (out.iters) out.iters[b] = 0;
  if (out.u_full)
    for (int k = 0; k < 12 * horizon; ++k) st_out(out.u_full, (size_t)k * out.ld + b, 0.0, out.f32);
}

// compute_joint_torques (A1RobotControl.cpp:289-319): thread per QP, every access batch-major coalesced.  HBM bound:
// (12+12+36+12) fp64 + 4 B read, 12 fp64 written per QP = 676 B/QP.
struct TorqueParams { double km[3]; double tg[12]; };
__global__ void joint_torques_kernel(int B, const double* __restrict__ f_grf, const double* __restrict__ f_kin,
                                     const double* __restrict__ jac, const uint32_t* __restrict__ contact, TorqueParams P,
                                     double* __restrict__ tau) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const size_t ld = (size_t)B;
  const uint32_t mask = contact[b];
#pragma unroll
  for (int leg = 0; leg < 4; ++leg) {
    double J[9], t[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) J[k] = jac[(size_t)(9 * leg + k) * ld + b];
    if ((mask >> leg) & 1u) {   // stance: J^T * (-f)
      const double f0 = -f_grf[(size_t)(3 * leg) * ld + b], f1 = -f_grf[(size_t)(3 * leg + 1) * ld + b], f2 = -f_grf[(size_t)(3 * leg + 2) * ld + b];
#pragma unroll
      for (int a = 0; a < 3; ++a) t[a] = J[a] * f0 + J[3 + a] * f1 + J[6 + a] * f2;
    } else {                    // swing: solve J tau = km .* f_kin with partial pivoting (Eigen's jac.lu().solve)
      double r[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) r[a] = P.km[a] * f_kin[(size_t)(3 * leg + a) * ld + b];
      // column 0 pivot
      int p = 0;
      if (fabs(J[3]) > fabs(J[p * 3])) p = 1;
      if (fabs(J[6]) > fabs(J[p * 3])) p = 2;
      if (p != 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { const double x = J[k]; J[k] = J[3 * p + k]; J[3 * p + k] = x; }
        const double x = r[0]; r[0] = r[p]; r[p] = x;
      }
      double m1 = J[3] / J[0], m2 = J[6] / J[0];
      J[4] -= m1 * J[1]; J[5] -= m1 * J[2]; r[1] -= m1 * r[0];
      J[7] -= m2 * J[1]; J[8] -= m2 * J[2]; r[2] -= m2 * r[0];
      if (fabs(J[7]) > fabs(J[4])) {
        double x = J[4]; J[4] = J[7]; J[7] = x;
        x = J[5]; J[5] = J[8]; J[8] = x;
        x = r[1]; r[1] = r[2]; r[2] = x;
      }
      const double m3 = J[7] / J[4];
      J[8] -= m3 * J[5]; r[2] -= m3 * r[1];
      t[2] = r[2] / J[8];
      t[1] = (r[1] - J[5] * t[2]) / J[4];
      t[0] = (r[0] - J[1] * t[1] - J[2] * t[2]) / J[0];
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double v = t[a] + P.tg[3 * leg + a];
      if (v == v) tau[(size_t)(3 * leg + a) * ld + b] = v;   // "prevent nan" (:314-317)
    }
  }
}

// update_plan (A1RobotControl.cpp:148-202): thread per robot, batch-major coalesced.
struct GaitDev { double cpg, cps, cdt, dfp[12], dxl, dyl; int N; };
__global__ void update_plan_kernel(int B, GaitDev G, double* __restrict__ gc, const double* __restrict__ gcs, const uint32_t* __restrict__ mode,
                                   const double* __restrict__ lv, const double* __restrict__ lvd, const double* __restrict__ rz,
                                   const double* __restrict__ rot, const double* __restrict__ pos, uint32_t* __restrict__ plan,
                                   uint32_t* __restrict__ sched, double* __restrict__ t_rel, double* __restrict__ t_abs, double* __restrict__ t_world) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const size_t ld = (size_t)B;
  double c[4], sp[4];
  uint32_t m = 0;
  const bool walk = mode[b] != 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    sp[i] = gcs[(size_t)i * ld + b];
    if (!walk) {
      c[i] = (i == 1 || i == 2) ? 120.0 : 0.0;   // gait_counter_reset(), trot
      m |= 1u << i;
    } else {
      c[i] = fmod(gc[(size_t)i * ld + b] + sp[i], G.cpg);
      if (c[i] <= G.cps) m |= 1u << i;
    }
    gc[(size_t)i * ld + b] = c[i];
  }
  plan[b] = m;
  if (sched) {
    for (int st = 0; st < G.N; ++st) {
      uint32_t ms = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double ci = walk ? fmod(c[i] + (double)st * sp[i], G.cpg) : 0.0;
        if (!walk || ci <= G.cps) ms |= 1u << i;
      }
      sched[(size_t)st * ld + b] = ms;
    }
  }
  if (t_rel || t_abs || t_world) {
    double v[3], vd[3], Rz[9], R[9], p[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { v[k] = lv[(size_t)k * ld + b]; vd[k] = lvd[(size_t)k * ld + b]; p[k] = pos[(size_t)k * ld + b]; }
#pragma unroll
    for (int k = 0; k < 9; ++k) { Rz[k] = rz[(size_t)k * ld + b]; R[k] = rot[(size_t)k * ld + b]; }
    const double vr0 = Rz[0] * v[0] + Rz[3] * v[1] + Rz[6] * v[2], vr1 = Rz[1] * v[0] + Rz[4] * v[1] + Rz[7] * v[2];   // Rz^T v
    const double kf = sqrt(fabs(G.dfp[8]) / 9.8);   // default_foot_pos(2): third scalar of the 3 x 4 matrix = z of leg 0
    for (int i = 0; i < 4; ++i) {
      double dx = kf * (vr0 - vd[0]) + ((G.cps / sp[i]) * G.cdt) / 2.0 * vd[0];
      double dy = kf * (vr1 - vd[1]) + ((G.cps / sp[i]) * G.cdt) / 2.0 * vd[1];
      dx = fmin(fmax(dx, -G.dxl), G.dxl);
      dy = fmin(fmax(dy, -G.dyl), G.dyl);
      const double f[3] = {G.dfp[0 * 4 + i] + dx, G.dfp[1 * 4 + i] + dy, G.dfp[2 * 4 + i]};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const double fa = R[3 * a] * f[0] + R[3 * a + 1] * f[1] + R[3 * a + 2] * f[2];
        if (t_rel) t_rel[(size_t)(3 * i + a) * ld + b] = f[a];
        if (t_abs) t_abs[(size_t)(3 * i + a) * ld + b] = fa;
        if (t_world) t_world[(size_t)(3 * i + a) * ld + b] = fa + p[a];
      }
    }
  }
}

// fp64 FMA pipe peak probe: 8 independent dependent-free DFMA chains per thread
__global__ void fp64_peak_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, k = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, k); a1 = fma(a1, m, k); a2 = fma(a2, m, k); a3 = fma(a3, m, k);
    a4 = fma(a4, m, k); a5 = fma(a5, m, k); a6 = fma(a6, m, k); a7 = fma(a7, m, k);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

__global__ void flush_kernel(double* buf, size_t n, double v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) buf[i] = v;
}

// -------------------------------------------------------------------------------------------
// fused final collect (a1mpc_peer_gather_*): step flags between the GPUs of one job.  The forces themselves are stored by the
// solve kernels (st_forces); these two tiny kernels order them: after the solve kernels of call number `step` have completed on
// this GPU, lane p of peer_signal_kernel publishes `step` in slot [rank] of rank p's flag array (system-scope release: the
// kernel boundary before it has already made the peer stores visible); peer_wait_kernel spins (system-scope acquire loads) until
// every rank's slot of the LOCAL flag array has reached `step`, with a clock cap so that a dead peer cannot hang the GPU.
// -------------------------------------------------------------------------------------------
#ifndef A1MPC_EMU
struct PeerFlags { unsigned long long* p[MAX_PEERS]; };
__global__ void peer_signal_kernel(PeerFlags flags, int nranks, int rank, unsigned long long step) {
  const int lane = threadIdx.x;
  __threadfence_system();
  if (lane < nranks) {
    unsigned long long* dst = flags.p[lane] + rank;
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(step) : "memory");
  }
}
__global__ void peer_wait_kernel(const unsigned long long* __restrict__ local_flags, int nranks, unsigned long long step, long long max_cycles,
                                 int* __restrict__ err) {
  const int lane = threadIdx.x;
  if (lane < nranks) {
    const long long t0 = clock64();
    unsigned long long v;
    for (;;) {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(local_flags + lane) : "memory");
      if (v >= step) break;
      if (clock64() - t0 > max_cycles) { atomicExch(err, 1 + lane); break; }
      __nanosleep(5000);   // 5 us: a tighter poll only perturbs the solve CTA that shares this SM
    }
  }
  __threadfence_system();
}
#endif

}  // namespace a1mpc
