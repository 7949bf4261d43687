// solve_kernel_big.cuh -- the fused control() kernel for num_basis > 32 (sm_100a, FP64).
//
// The reference accepts any basis count (basis.cpp:48-77).  The warp-per-instance kernels (solve_kernel.cuh,
// solve_kernel_v2.cuh) keep an instance's nb x nb coefficient block in ONE warp's registers, which stops at
// nb = 32; this kernel gives an instance a whole CTA instead: the coefficient block is spread over the CTA's
// warps as DMMA accumulator strips, S = lamda .* (c_k - phi_k) goes through an L2-resident scratch row per
// resident CTA, and both contractions run on the FP64 tensor cores (mma.sync m8n8k4 -> DMMA.8x8x4) from order-major
// cos / sin tables of 32 states at a time: c_k as rank-32 updates of 8 x 64 coefficient strips (one strip per warp
// and pass), the metric gradient as the products of a warp's 8 coefficient rows with the x tables of 32 steps.
// Same arithmetic contract, parameter block, error bits and outputs as solve_kernel (read its header first); the
// rollout and the co-state pass are the same three warp scans, run by warp 0.
//
// Replaces, per instance: ErgodicControl::control() (ergodic_control.hpp:225-311) with Basis::trajCoeff
// (basis.cpp:109-120), gradErgodicMetric (:419-436), gradBarrier (:454-474), the backward RK4 (integrator.hpp:154-194,
// rhodot :65-69) and updateControl (:439-451).
#pragma once

#include "solve_kernel.cuh"

namespace eb
{
constexpr int kBigThreads = 256;
constexpr int kBigWarps = kBigThreads / 32;
constexpr int kBigMaxBasis = 128;  // EB_MAX_NUM_BASIS (ergodic_b200.h): tables of 32 states fit shared memory

// order-major tables: row = one order's cos / sin over the 32 states of a chunk; pitch 36 = 32 + 4 -> the DMMA
// fragment loads (8 rows x 4 states, or 4 rows x 8 states) touch every bank pair exactly twice: 2 wavefronts, the minimum
constexpr int kBigPitch = 36;
__host__ __device__ inline int big_tab_rows(int nb) { return (nb + 7) & ~7; }  // orders padded to whole 8-row tiles (zeros)
// shared memory (doubles): per-step records [4][npad], e_x | e_y [2][npad], the table region (four gradient tables
// [rows][36]; the two c_k tables alias the first two), the per-warp partial gradient sums [8][32][2], the metric partials
__host__ __device__ inline int big_tab_doubles(int nb) { return 4 * big_tab_rows(nb) * kBigPitch; }
inline size_t solve_big_smem_bytes(int nb, int N)
{
  const int npad = ((N + 31) / 32) * 32;
  return sizeof(double) * (size_t)(6 * npad + big_tab_doubles(nb) + 2 * 32 * kBigWarps + 16);
}

// cos(k pi u), sin(k pi u) started directly at order k0 (and k0 - 1): a recurrence never runs longer than a
// quarter of the orders
struct BigChain
{
  double ck, cm, sk, sm, two;
};
__device__ __forceinline__ BigChain big_chain_start(double u, int k0)
{
  BigChain c;
  double s1, c1;
  fast_sincospi(u, &s1, &c1);
  c.two = 2.0 * c1;
  fast_sincospi((double)k0 * u, &c.sk, &c.ck);
  fast_sincospi((double)(k0 - 1) * u, &c.sm, &c.cm);
  return c;
}
__device__ __forceinline__ void big_chain_step(BigChain& c)
{
  const double cn = fma(c.two, c.ck, -c.cm), sn = fma(c.two, c.sk, -c.sm);
  c.cm = c.ck;
  c.ck = cn;
  c.sm = c.sk;
  c.sk = sn;
}

template <int MODEL, bool PER_INST = false>
__global__ void __launch_bounds__(kBigThreads) solve_kernel_big(const SolveParams p, double* __restrict__ scratch)
{
  extern __shared__ __align__(16) double smem_big[];
  double* const smem = smem_big;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rounds = (p.N + 31) >> 5;
  const int npad = rounds * 32;
  const int nb = p.nb, K = nb * nb;
  double* const rec = smem;                 // [4][npad]: heading cos, sin; Fourier-frame x, y
  double* const exy = rec + 4 * npad;       // [2][npad]: e_x, e_y of every step
  double* const tab = exy + 2 * npad;       // table region
  double* const part = tab + big_tab_doubles(nb);  // [8 warps][32 steps][2]
  double* const mred = part + 2 * 32 * kBigWarps;  // [8] metric partials
  double* const S = scratch + (size_t)blockIdx.x * K;
  const int tabrows = big_tab_rows(nb), Tt = tabrows >> 3;  // 8 x 8 coefficient tiles per axis
  const int ntb = (Tt + 7) >> 3;                             // strips of up to 8 tiles per tile row
  const int nunits = Tt * ntb, npass = (nunits + kBigWarps - 1) / kBigWarps;
  const int T = p.M + p.N;
  const int kq = tabrows >> 2;  // table rows per builder segment (4 segments)

  grid_dependency_wait();
  for (int inst = blockIdx.x; inst < p.B; inst += gridDim.x)
  {
    const double* ut_in = p.ut_in + (size_t)inst * p.N * 3;
    double* ut_out = p.ut_out + (size_t)inst * p.N * 3;
    __syncthreads();  // the previous instance is done with shared memory

    // ---- forward rollout with the shifted controls (:233-237), warp 0 -----------------------------------------
    if (warp == 0)
    {
      RolloutCarry cy;
      const double xv = lane < 3 ? p.x[(size_t)inst * 3 + lane] : 0.0;
      if (p.pose_out && lane < 3) p.pose_out[(size_t)inst * 3 + lane] = xv;
      cy.x = __shfl_sync(kFull, xv, 0);
      cy.y = __shfl_sync(kFull, xv, 1);
      cy.th = __shfl_sync(kFull, xv, 2);
      fast_sincos(cy.th, &cy.sth, &cy.cth);
      for (int r = 0; r < rounds; r++)
      {
        const int i = r * 32 + lane;
        const bool valid = i < p.N;
        double u0 = 0.0, u1 = 0.0, u2 = 0.0;
        if (i + 1 < p.N)
        {  // shift left by one column, last column zero
          u0 = ut_in[(i + 1) * 3 + 0];
          u1 = ut_in[(i + 1) * 3 + 1];
          u2 = ut_in[(i + 1) * 3 + 2];
        }
        if (MODEL == kModelSimpleCart && !(fabs(u1 - 0.0) < 1.0e-12)) atomicOr(p.fault, 1);  // cart.hpp:167-170
        double xo, yo, tho, ce, se;
        rollout_round<MODEL>(p.dt, valid, lane, u0, u1, u2, cy, xo, yo, tho, ce, se);
        rec[0 * npad + i] = ce;
        rec[1 * npad + i] = se;
        rec[2 * npad + i] = xo - frame<PER_INST, kFrXmin>(p, inst);
        rec[3 * npad + i] = yo - frame<PER_INST, kFrYmin>(p, inst);
      }
    }
    __syncthreads();

    // ---- c_k = (1/T) sum_t cos(ky b y_t) cos(kx a x_t) over the sampled past states and the horizon
    //      (basis.cpp:109-120), S = lamda .* (c_k - phi_k) (:422), ergodic metric.  Order-major cosine tables of 32
    //      states at a time; a warp owns the 8 x 64 coefficient strip (ti, 8 tj) of a pass and runs 8 DMMA k-steps
    //      per chunk over it (fragments as in solve_kernel's coeff_chunk) -------------------------------------------
    double metric = 0.0;
    const int g = lane >> 2, q = lane & 3;
    double* const t_x = tab;                  // cos(kx a x_s)   [8 T][kBigPitch]
    double* const t_y = tab + tabrows * kBigPitch;  // cos(ky b y_s)
    for (int pass = 0; pass < npass; pass++)
    {
      const int unit = pass * kBigWarps + warp;
      const bool active = unit < nunits;
      const int ti = active ? unit / ntb : 0, tj0 = active ? 8 * (unit % ntb) : 0;
      const int ntj = active ? min(8, Tt - tj0) : 0;
      double acc[8][2];
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j][0] = acc[j][1] = 0.0;
      for (int s0 = 0; s0 < T; s0 += 32)
      {
        __syncthreads();  // the previous chunk's tables have been read
        {
          // table builders: thread = (state, axis, quarter of the orders)
          const int axis = warp & 1, seg = warp >> 1;
          const int s = s0 + lane;
          const bool valid = s < T;
          double coord = 0.0;
          if (valid)
          {
            if (s < p.M)
            {  // ReplayBuffer::sampleMemory (buffer.cpp:64-111)
              long long idx = s;
              if (p.idx_mode == 1)
                idx = p.mem_idx[(size_t)inst * p.batch_size + s];
              else if (p.idx_mode == 2)
              {
                const uint64_t r = mix64(mix64(p.seed + p.call * 0xD1B54A32D192ED03ull) ^
                                         ((uint64_t)inst * 0x9E3779B97F4A7C15ull + (uint64_t)s));
                idx = (long long)__umul64hi(r, (uint64_t)p.mem_count);
              }
              if ((unsigned long long)idx >= (unsigned long long)p.mem_count)
              {  // memory_.at() throws (buffer.cpp:84,103): fault bit 2 and a safe index
                atomicOr(p.fault, 2);
                idx = 0;
              }
              if (p.idx_mode != 0 && p.mem_idx_out && warp == 0 && pass == 0)
                p.mem_idx_out[(size_t)inst * p.batch_size + s] = (int)idx;
              const double* h = p.hist + ((size_t)idx * p.B + inst) * 3;
              coord = h[axis] - (axis ? frame<PER_INST, kFrYmin>(p, inst) : frame<PER_INST, kFrXmin>(p, inst));
            }
            else
              coord = rec[(2 + axis) * npad + (s - p.M)];
          }
          const double u = coord * (axis ? frame<PER_INST, kFrInvLy>(p, inst) : frame<PER_INST, kFrInvLx>(p, inst));
          const int k0 = seg * kq, k1 = min(tabrows, k0 + kq);
          double* const col = (axis ? t_y : t_x) + lane;
          BigChain ch = big_chain_start(u, k0);
          for (int k = k0; k < k1; k++)
          {
            col[k * kBigPitch] = (valid && k < nb) ? ch.ck : 0.0;  // states past the end and padding orders: zero
            big_chain_step(ch);
          }
        }
        __syncthreads();
        if (active)
        {
          const int ksteps = (min(32, T - s0) + 3) >> 2;
          const double* const fa = t_y + (8 * ti + g) * kBigPitch + q;
          const double* const fb = t_x + (8 * tj0 + g) * kBigPitch + q;
          for (int ks = 0; ks < ksteps; ks++)
          {
            const double a = fa[4 * ks];
            double b[8];
#pragma unroll
            for (int j = 0; j < 8; j++) b[j] = j < ntj ? fb[j * 8 * kBigPitch + 4 * ks] : 0.0;
#pragma unroll
            for (int j = 0; j < 8; j++)
              if (j < ntj) dmma884(acc[j][0], acc[j][1], a, b[j]);
          }
        }
      }
      if (active)
      {
        const double inv_t = 1.0 / (double)T;  // basis.cpp:119
        const int ky = 8 * ti + g;
#pragma unroll
        for (int j = 0; j < 8; j++)
#pragma unroll
          for (int e = 0; e < 2; e++)
          {
            const int kx = 8 * (tj0 + j) + 2 * q + e;
            if (j < ntj && ky < nb && kx < nb)
            {
              const int k = ky * nb + kx;
              const double c = __dmul_rn(inv_t, acc[j][e]);
              const double d = __dsub_rn(c, phik_at<PER_INST>(p, inst, K, k));
              const double sv = __ldg(p.lamk + k) * d;
              metric += sv * d;
              if (p.ck) p.ck[(size_t)inst * K + k] = c;
              S[k] = sv;
            }
          }
      }
    }
    metric = warp_sum(metric);
    if (lane == 0) mred[warp] = metric;
    __syncthreads();  // S is complete (global writes of this CTA are visible to it past the barrier)
    if (tid == 0 && p.metric)
    {
      double m = 0.0;
      for (int w8 = 0; w8 < kBigWarps; w8++) m += mred[w8];
      p.metric[inst] = m;
    }

    // ---- gradient of the ergodic metric (:419-436), 32 steps at a time: R1 = S (a_kx sin(kx a x_t)), R2 = S cos(kx a x_t)
    //      as DMMA products of the warp's 8 coefficient rows with the order-major x tables (4 tiles of 8 steps), then
    //      e_x = sum_ky cos(ky b y_t) R1[ky][t], e_y = sum_ky b_ky sin(ky b y_t) R2[ky][t]: fragment-wise product with
    //      the y tables, a shuffle reduction over the 8 row lanes, and a sum over the warps in index order ------------
    double* const t_asx = tab;
    double* const t_cx = tab + tabrows * kBigPitch;
    double* const t_cy = tab + 2 * tabrows * kBigPitch;
    double* const t_bsy = tab + 3 * tabrows * kBigPitch;
    const int gks = (nb + 3) >> 2;
    for (int r = 0; r < rounds; r++)
    {
      {
        const int axis = warp & 1, seg = warp >> 1;
        const int i = r * 32 + lane;
        const double coord = rec[(2 + axis) * npad + i];
        const double u = coord * (axis ? frame<PER_INST, kFrInvLy>(p, inst) : frame<PER_INST, kFrInvLx>(p, inst));
        const double f = axis ? frame<PER_INST, kFrBy>(p, inst) : frame<PER_INST, kFrAx>(p, inst);
        const int k0 = seg * kq, k1 = min(tabrows, k0 + kq);
        double* const tc = (axis ? t_cy : t_cx) + lane;
        double* const ts = (axis ? t_bsy : t_asx) + lane;
        BigChain ch = big_chain_start(u, k0);
        for (int k = k0; k < k1; k++)
        {
          tc[k * kBigPitch] = k < nb ? ch.ck : 0.0;
          ts[k * kBigPitch] = k < nb ? ((double)k * f) * ch.sk : 0.0;
          big_chain_step(ch);
        }
      }
      __syncthreads();
      {
        const int nnj = min(4, (min(32, p.N - r * 32) + 7) >> 3);  // 8-step tiles with at least one valid step
        double v[4][2], w[4][2];  // e_x, e_y partial sums of steps 8 nj + 2 q + e over this lane's rows
#pragma unroll
        for (int nj = 0; nj < 4; nj++) v[nj][0] = v[nj][1] = w[nj][0] = w[nj][1] = 0.0;
        for (int mi = warp; mi < Tt; mi += kBigWarps)
        {
          const int ky = 8 * mi + g;
          double R1[4][2], R2[4][2];
#pragma unroll
          for (int nj = 0; nj < 4; nj++) R1[nj][0] = R1[nj][1] = R2[nj][0] = R2[nj][1] = 0.0;
          const double* const srow = S + (size_t)min(ky, nb - 1) * nb;
          const bool row_ok = ky < nb;
          double a = (row_ok && q < nb) ? srow[q] : 0.0;
          for (int ks = 0; ks < gks; ks++)
          {
            const int kxn = 4 * (ks + 1) + q;
            const double a_next = (row_ok && kxn < nb) ? srow[kxn] : 0.0;  // next k-step's fragment, ahead of the DMMAs
            const double* const bs = t_asx + (4 * ks + q) * kBigPitch + g;
            const double* const bc = t_cx + (4 * ks + q) * kBigPitch + g;
#pragma unroll
            for (int nj = 0; nj < 4; nj++)
              if (nj < nnj)
              {
                dmma884(R1[nj][0], R1[nj][1], a, bs[8 * nj]);
                dmma884(R2[nj][0], R2[nj][1], a, bc[8 * nj]);
              }
            a = a_next;
          }
          // lane (g, q) holds R[ky = 8 mi + g][steps 8 nj + 2 q, + 1]: weight with the y tables
          const double* const yc = t_cy + ky * kBigPitch + 2 * q;
          const double* const ys = t_bsy + ky * kBigPitch + 2 * q;
#pragma unroll
          for (int nj = 0; nj < 4; nj++)
            if (nj < nnj)
            {
              const double2 c2 = *reinterpret_cast<const double2*>(yc + 8 * nj);
              const double2 s2 = *reinterpret_cast<const double2*>(ys + 8 * nj);
              v[nj][0] = fma(c2.x, R1[nj][0], v[nj][0]);
              v[nj][1] = fma(c2.y, R1[nj][1], v[nj][1]);
              w[nj][0] = fma(s2.x, R2[nj][0], w[nj][0]);
              w[nj][1] = fma(s2.y, R2[nj][1], w[nj][1]);
            }
        }
        // sum over the 8 row lanes (lane = 4 g + q): xor 4, 8, 16
#pragma unroll
        for (int nj = 0; nj < 4; nj++)
#pragma unroll
          for (int e = 0; e < 2; e++)
          {
            double sv = v[nj][e], sw = w[nj][e];
#pragma unroll
            for (int o = 4; o < 32; o <<= 1)
            {
              sv += __shfl_xor_sync(kFull, sv, o);
              sw += __shfl_xor_sync(kFull, sw, o);
            }
            if (g == 0)
            {
              part[(warp * 32 + 8 * nj + 2 * q + e) * 2 + 0] = sv;
              part[(warp * 32 + 8 * nj + 2 * q + e) * 2 + 1] = sw;
            }
          }
      }
      __syncthreads();  // also: the tables may be rebuilt
      if (tid < 64)
      {
        const int st = tid & 31, which = tid >> 5;
        double sum = 0.0;
        for (int w8 = 0; w8 < kBigWarps; w8++) sum += part[(w8 * 32 + st) * 2 + which];
        exy[which * npad + r * 32 + st] = -sum * p.w;  // times expl_weight (:433)
      }
    }
    __syncthreads();

    // ---- backward co-state pass and control update (:277, :439-451, integrator.hpp:154-194), warp 0 ----------
    if (warp == 0)
    {
      double r0c = 0.0, r1c = 0.0, r2c = 0.0;  // rho(T) = 0 (:203)
      for (int r = rounds - 1; r >= 0; r--)
      {
        const int i = r * 32 + lane;
        const bool valid = i < p.N;
        const double ce = rec[0 * npad + i], se = rec[1 * npad + i];
        const double xf = rec[2 * npad + i], yf = rec[3 * npad + i];
        const double ex = exy[i], ey = exy[npad + i];
        double u0 = 0.0, u1 = 0.0;
        if (i + 1 < p.N)
        {
          u0 = ut_in[(i + 1) * 3 + 0];
          u1 = ut_in[(i + 1) * 3 + 1];
        }
        // gradBarrier :454-474
        double bx = 0.0, byv = 0.0;
        bx += 2.0 * (double)(xf > frame<PER_INST, kFrLx>(p, inst) - p.beps) * (xf - (frame<PER_INST, kFrLx>(p, inst) - p.beps));
        byv += 2.0 * (double)(yf > frame<PER_INST, kFrLy>(p, inst) - p.beps) * (yf - (frame<PER_INST, kFrLy>(p, inst) - p.beps));
        bx += 2.0 * (double)(xf < p.beps) * (xf - p.beps);
        byv += 2.0 * (double)(yf < p.beps) * (yf - p.beps);
        bx *= p.bw;
        byv *= p.bw;
        // rhodot (:65-69): components 0 and 1 do not depend on rho
        const double k0 = valid ? (-ex - bx) : 0.0;
        const double k1 = valid ? (-ey - byv) : 0.0;
        const double inc0 = -(p.dt / 6.0 * (((k0 + 2.0 * k0) + 2.0 * k0) + k0));
        const double inc1 = -(p.dt / 6.0 * (((k1 + 2.0 * k1) + 2.0 * k1) + k1));
        const double suf0 = warp_scan_incl_rev(inc0, lane);
        const double suf1 = warp_scan_incl_rev(inc1, lane);
        double exc0 = __shfl_down_sync(kFull, suf0, 1), exc1 = __shfl_down_sync(kFull, suf1, 1);
        if (lane == 31) exc0 = exc1 = 0.0;
        const double r0p = r0c + exc0, r1p = r1c + exc1;  // rho before this (backward) step
        const double r0 = r0c + suf0, r1 = r1c + suf1;    // rho after it = rhot.col(i)
        double a02, a12;
        if (MODEL == kModelOmni)
        {  // omni.hpp:195-196
          a02 = -u0 * se - u1 * ce;
          a12 = u0 * ce - u1 * se;
        }
        else
        {  // cart.hpp:184-185
          a02 = -u0 * se;
          a12 = u0 * ce;
        }
        // component 2: k = -(A02 rho0 + A12 rho1) at the four RK4 stages
        const double k1_2 = -(a02 * r0p + a12 * r1p);
        const double r0s = r0p - p.dt * (0.5 * k0), r1s = r1p - p.dt * (0.5 * k1);
        const double k2_2 = -(a02 * r0s + a12 * r1s);
        const double r0e = r0p - p.dt * k0, r1e = r1p - p.dt * k1;
        const double k4_2 = -(a02 * r0e + a12 * r1e);
        const double inc2 = valid ? -(p.dt / 6.0 * (((k1_2 + 2.0 * k2_2) + 2.0 * k2_2) + k4_2)) : 0.0;
        const double r2 = r2c + warp_scan_incl_rev(inc2, lane);
        r0c = __shfl_sync(kFull, r0, 0);
        r1c = __shfl_sync(kFull, r1, 0);
        r2c = __shfl_sync(kFull, r2, 0);
        // updateControl: u = -Rinv * (B^T rho), clamped
        double bt0, bt1;
        if (MODEL == kModelOmni)
        {  // omni.hpp:208-210
          bt0 = ce * r0 + se * r1;
          bt1 = -se * r0 + ce * r1;
        }
        else
        {  // cart.hpp:196-202
          bt0 = ce * r0 + se * r1;
          bt1 = 0.0;
        }
        double un[3];
        bool finite = true;
#pragma unroll
        for (int c = 0; c < 3; c++)
        {
          const double v = -((p.Rinv[c + 0] * bt0 + p.Rinv[c + 3] * bt1) + p.Rinv[c + 6] * r2);
          finite &= fabs(v) <= 1.7976931348623157e308;  // false for NaN and Inf
          un[c] = clampd(v, p.umin[c], p.umax[c]);
          if (valid) ut_out[i * 3 + c] = un[c];
        }
        if (valid && !finite) atomicOr(p.fault, 4);  // NaN / Inf guard
        if (r == 0) publish_first_twist(p, inst, lane, un);
      }
    }
  }
}
}  // namespace eb
