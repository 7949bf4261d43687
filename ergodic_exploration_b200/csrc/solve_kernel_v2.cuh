// solve_kernel_v2.cuh -- the fused control() kernel for num_basis 13..24, re-laid to spare the SM's load/store
// data pipe (sm_100a, FP64).  Same arithmetic contract and the same parameter block as solve_kernel.cuh (read its
// header first: one warp per instance, lanes = time steps, warp-scan RK4, c_k on the FP64 tensor cores); here the
// metric gradient runs on the tensor cores too, and the DMMA operands are laid out to spare shared memory.
//
// ncu on the round-1 kernel (solve_kernel at nb 16..24, since retired; profiles/solve_c5_r02_lsu.txt): the FP64 pipe (DFMA and DMMA share it on B200) was
// 60 % busy while `l1tex__data_pipe_lsu_wavefronts` -- shared-memory loads / stores, shuffles and global accesses,
// ONE wavefront per cycle per SM for all four schedulers -- ran at 71 %, 84 % with the math removed: the kernel
// was bound by operand traffic through shared memory, not by arithmetic.  So this version trades a few DFMAs for
// wavefronts:
//  * c_k, Chebyshev-product tiles.  cos((8a+g) t) = 2 cos(8a t) cos(g t) - cos((8a-g) t), so the tile of orders
//    8a..8a+7 is accumulated as U_ab = sum_t (cy_g cy_8a)(cx_h cx_8b) from the fragments of orders 0..7 times one
//    scalar per state (one DMUL per fragment and k-step), and the true coefficients follow from
//    4 U_ab[g][h] = C[8a+g][8b+h] + C[8a-g][8b+h] + C[8a+g][8b-h] + C[8a-g][8b-h] by two passes of warp shuffles per
//    INSTANCE (rows, then columns).  The cosine tables shrink from nb rows per axis to 8 + (tiles - 1): 44 % fewer
//    table stores and fragment loads at nb = 16, 50 % at nb = 20.
//  * the table builders read their state's coordinate straight from the step records (lane = (axis, slot)), one
//    sincospi per lane and half-round, no shuffles; replay states load the one coordinate they need from HBM,
//    one half-round ahead of its use.
//  * metric gradient: the x tables are never written.  In R1 = (S a) SX, R2 = (b S) CX the B fragment of lane
//    (g, q) is sin / cos((4 ks + q) alpha x_t) for ITS time step t = g: orders of one residue mod 4, which the lane
//    generates in registers with a stride-4 three-term recurrence (v_{k+4} = 2 cos(4t) v_k - v_{k-4}).  Only the
//    two y tables go through shared memory (all 32 lanes build them: lane = (parity, cos|sin, slot)).
// tools/emu/emu_v2.py replays this lane-level data flow on the CPU against the plain formulas.
#pragma once

#include "solve_kernel.cuh"

namespace eb
{
// S (NB x NB) in shared memory: pitch = 4 or 12 (mod 16) -> conflict-free A-fragment loads
__host__ __device__ constexpr int s_pitch(int nb) { return nb % 8 == 0 ? nb + 4 : nb; }

// Instantiated for NB = 16, 20 and 24.
template <int NB>
struct Solve2Cfg
{
  static constexpr int kTiles = (NB + 7) / 8;
  static constexpr int kGks = (NB + 3) / 4;
  static constexpr int kRows = 8 + (kTiles - 1);           // c_k table rows per axis: orders 0..7, then 8, 16, 24
  static constexpr int kAxisStride = kRows * kTabStride;   // one axis' c_k table (pitch 20: conflict-free fragments)
  static constexpr int kCkDoubles = 2 * kAxisStride;
  static constexpr int kYStride = NB * 8 + 8;              // one y table (cos | sin), [ky][8 slots]; +8: 16 banks apart
  static constexpr int kYDoubles = 2 * kYStride;
  static constexpr int kSPitch = s_pitch(NB);
  static constexpr int kSDoubles = NB * kSPitch;
  static constexpr int kUnion = kCkDoubles > kYDoubles ? (kCkDoubles > kSDoubles ? kCkDoubles : kSDoubles) :
                                                         (kYDoubles > kSDoubles ? kYDoubles : kSDoubles);
  static constexpr int kStage = 64;                        // e_x | e_y of one round, handed to the time-step lanes
  static constexpr int kTabDoubles = kUnion + kStage;
  static constexpr int kFields = 8;                        // heading cos, sin; Fourier-frame x, y; cos, sin of a x; of b y
  static constexpr int kMinBlocks = NB <= 16 ? 6 : 4;
  static constexpr int kWideWarps = NB <= 16 ? 24 : 16;  // one CTA per SM for single-wave batches (see SolveCfg)
};

// per-step records are kept for the horizon rounded up to a half-round (16 steps)
__host__ __device__ inline int solve2_npad(int N) { return (N + 15) & ~15; }
template <int NB>
inline size_t solve2_smem_bytes(int N, int warps = kSolveWarps);

// One half-round (16 states) of the rank-T update of the c_k accumulators.  lane = (axis = lane / 16, slot = lane % 16)
// holds c1 = cos(pi * coordinate / l) of ITS axis of state `slot`; it runs the even / odd Chebyshev chains up to
// order 8, derives orders 16 and 24 by doubling, and writes its column of the axis table.  Then up to four DMMA
// k-steps: fragments of orders 0..7 (A0: y, B0: x), the per-state scalars cos(8a ..) and kTiles^2 tiles.
template <int NB>
__device__ __forceinline__ void coeff_half(double* __restrict__ tab, const int lane, const bool ok, const int left,
                                           const double c1, double (&acc)[(NB + 7) / 8][(NB + 7) / 8][2])
{
  using Cfg = Solve2Cfg<NB>;
  constexpr int TILES = Cfg::kTiles;
  const int g = lane >> 2, q = lane & 3;
  double* const mytab = tab + (lane >> 4) * Cfg::kAxisStride + (lane & 15);
  {
    const double v = c1;
    const double m = fma(4.0 * v, v, -2.0);
    // (T_{-2}, T_0) = (2 v^2 - 1, 1), (T_{-1}, T_1) = (v, v); states past the end give zero columns
    double em = ok ? fma(2.0 * v, v, -1.0) : 0.0, ek = ok ? 1.0 : 0.0;
    double om = ok ? v : 0.0, ok1 = om;
    __syncwarp();  // the previous half's fragment loads are done
#pragma unroll
    for (int k = 0; k < 8; k += 2)
    {
      mytab[k * kTabStride] = ek;
      mytab[(k + 1) * kTabStride] = ok1;
      const double en = fma(m, ek, -em), on = fma(m, ok1, -om);
      em = ek;
      ek = en;
      om = ok1;
      ok1 = on;
    }
    if (TILES > 1)
    {
      const double t8 = ek;  // T_8 (0 for a padded state)
      mytab[8 * kTabStride] = t8;
      if (TILES > 2)
      {
        const double t16 = ok ? fma(2.0 * t8, t8, -1.0) : 0.0;
        mytab[9 * kTabStride] = t16;
        if (TILES > 3) mytab[10 * kTabStride] = ok ? fma(2.0 * t16, t8, -t8) : 0.0;  // T_24 = 2 T_16 T_8 - T_8
      }
    }
  }
  __syncwarp();
  const double* const tabx = tab;
  const double* const taby = tab + Cfg::kAxisStride;
  const int ksteps = (min(left, kTabSlots) + 3) >> 2;
  for (int s = 0; s < ksteps; s++)
  {
    double a[TILES], b[TILES];
    const int col = 4 * s + q;
    a[0] = taby[g * kTabStride + col];
    b[0] = tabx[g * kTabStride + col];
#pragma unroll
    for (int t = 1; t < TILES; t++)
    {
      a[t] = a[0] * taby[(7 + t) * kTabStride + col];
      b[t] = b[0] * tabx[(7 + t) * kTabStride + col];
    }
#pragma unroll
    for (int ti = 0; ti < TILES; ti++)
#pragma unroll
      for (int tj = 0; tj < TILES; tj++) dmma_ck(acc[ti][tj][0], acc[ti][tj][1], a[ti], b[tj]);
  }
}

template <int NB>
inline size_t solve2_smem_bytes(int N, int warps)
{
  return sizeof(double) * warps * (size_t)(Solve2Cfg<NB>::kTabDoubles + Solve2Cfg<NB>::kFields * solve2_npad(N));
}

template <int MODEL, int NB, int WARPS = kSolveWarps, bool PER_INST = false>
__global__ void __launch_bounds__(WARPS * 32, WARPS == kSolveWarps ? Solve2Cfg<NB>::kMinBlocks : 1) solve_kernel2(const SolveParams p)
{
  using Cfg = Solve2Cfg<NB>;
  constexpr int TILES = Cfg::kTiles;
  constexpr int GKS = Cfg::kGks;
  static_assert(NB == 16 || NB == 20 || NB == 24, "solve_kernel2 serves num_basis 13..24 (template sizes 16, 20, 24)");
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rounds = (p.N + 31) >> 5;
  const int npad = solve2_npad(p.N);
  const int nb = p.nb, K = nb * nb;
  const int g = lane >> 2, q = lane & 3;

  const int inst = blockIdx.x * WARPS + warp;
  __shared__ WideIo<WARPS> wio;  // wide single-wave CTAs: poses in / first twists out as one segment (solve_kernel.cuh)
  grid_dependency_wait();  // programmatic dependent launch: see solve_kernel.cuh
  if constexpr (WideIo<WARPS>::kOn) wide_io_load(wio, p);
  if (inst >= p.B) return;

  double* const tab = smem + warp * (Cfg::kTabDoubles + Cfg::kFields * npad);
  double* const stage_ = tab + Cfg::kUnion;
  double* const rec = tab + Cfg::kTabDoubles;
  double* const Ssm = tab;  // S (NB x NB) aliases the tables between the c_k phase and the gradient

  double acc[TILES][TILES][2];
#pragma unroll
  for (int i = 0; i < TILES; i++)
#pragma unroll
    for (int j = 0; j < TILES; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

  // builder role of this lane: one axis of one state of a half-round
  const int axis = lane >> 4, slot = lane & 15;
  const double inv_l = axis ? frame<PER_INST, kFrInvLy>(p, inst) : frame<PER_INST, kFrInvLx>(p, inst);
  const double origin = axis ? frame<PER_INST, kFrYmin>(p, inst) : frame<PER_INST, kFrXmin>(p, inst);

  // ---- sampled past states (buffer.cpp:64-111), Fourier frame (:243-244) ----
  if (p.M > 0)
  {
    // the coordinate of half-round h + 1 is loaded while half-round h is contracted
    auto fetch = [&](const int base) -> double {
      const int j = base + slot;
      if (j >= p.M) return 0.0;
      long long idx = j;  // stored <= batch_size: all states, insertion order
      if (p.idx_mode == 1)
        idx = p.mem_idx[(size_t)inst * p.batch_size + j];
      else if (p.idx_mode == 2)
      {
        const uint64_t r = mix64(mix64(p.seed + p.call * 0xD1B54A32D192ED03ull) ^
                                 ((uint64_t)inst * 0x9E3779B97F4A7C15ull + (uint64_t)j));
        idx = (long long)__umul64hi(r, (uint64_t)p.mem_count);
      }
      if ((unsigned long long)idx >= (unsigned long long)p.mem_count)
      {  // buffer.cpp:84,103: memory_.at() throws; here: fault bit 2 (-> EB_ERR_OUT_OF_RANGE) and a safe index
        atomicOr(p.fault, 2);
        idx = 0;
      }
      if (p.idx_mode != 0 && p.mem_idx_out && axis == 0) p.mem_idx_out[(size_t)inst * p.batch_size + j] = (int)idx;
      if (p.hist_cos) return __ldg(p.hist_cos + ((size_t)idx * p.B + inst) * 2 + axis);  // the cached cosine itself
      return __ldg(p.hist + ((size_t)idx * p.B + inst) * 3 + axis);
    };
    double cur = fetch(0);
    for (int base = 0; base < p.M; base += kTabSlots)
    {
      const double nxt = base + kTabSlots < p.M ? fetch(base + kTabSlots) : 0.0;
      const bool ok = base + slot < p.M;
      const double c1 = p.hist_cos ? cur : fast_cospi((cur - origin) * inv_l);
      coeff_half<NB>(tab, lane, ok, p.M - base, c1, acc);
      cur = nxt;
    }
  }

  // ---- forward rollout with the shifted controls (:233-237) ----------------
  const double* ut_in = p.ut_in + (size_t)inst * p.N * 3;
  double* ut_out = p.ut_out + (size_t)inst * p.N * 3;
  RolloutCarry cy;
  {
    double xv = 0.0;
    if constexpr (WideIo<WARPS>::kOn)
      xv = lane < 3 ? wio.x[3 * warp + lane] : 0.0;
    else
      xv = lane < 3 ? p.x[(size_t)inst * 3 + lane] : 0.0;
    if (p.pose_out && lane < 3) p.pose_out[(size_t)inst * 3 + lane] = xv;
    cy.x = __shfl_sync(kFull, xv, 0);
    cy.y = __shfl_sync(kFull, xv, 1);
    cy.th = __shfl_sync(kFull, xv, 2);
    fast_sincos(cy.th, &cy.sth, &cy.cth);
  }
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
    if (i < npad)
    {
      rec[0 * npad + i] = ce;
      rec[1 * npad + i] = se;
      rec[2 * npad + i] = xo - frame<PER_INST, kFrXmin>(p, inst);
      rec[3 * npad + i] = yo - frame<PER_INST, kFrYmin>(p, inst);
    }
    __syncwarp();
    const int nvalid = min(32, p.N - r * 32);
#pragma unroll
    for (int h = 0; h < 2; h++)
    {
      const int left = nvalid - h * kTabSlots;  // valid states in this half (warp-uniform)
      if (left <= 0) break;
      const int si = r * 32 + h * kTabSlots + slot;  // the state this lane builds (one axis of it)
      const bool ok = slot < left;
      double sn = 0.0, cs = 1.0;
      if (ok) fast_sincospi(rec[(2 + axis) * npad + si] * inv_l, &sn, &cs);
      rec[(4 + 2 * axis) * npad + si] = cs;  // cos / sin of a x (axis 0) or b y (axis 1): the gradient reads them back
      rec[(5 + 2 * axis) * npad + si] = sn;
      coeff_half<NB>(tab, lane, ok, left, cs, acc);
    }
  }

  // ---- product tiles -> coefficients: rows, then columns (see the header) -----------------------
  __syncwarp();
#pragma unroll
  for (int a = 1; a < TILES; a++)
#pragma unroll
    for (int b = 0; b < TILES; b++)
#pragma unroll
      for (int e = 0; e < 2; e++)
      {
        const double other = __shfl_sync(kFull, acc[a - 1][b][e], 4 * ((8 - g) & 7) + q);
        if (g > 0) acc[a][b][e] = 2.0 * acc[a][b][e] - other;
      }
#pragma unroll
  for (int b = 1; b < TILES; b++)
#pragma unroll
    for (int a = 0; a < TILES; a++)
    {
      const double o0 = __shfl_sync(kFull, acc[a][b - 1][0], 4 * g + ((4 - q) & 3));
      const double o1 = __shfl_sync(kFull, acc[a][b - 1][1], 4 * g + (3 - q));
      if (q > 0) acc[a][b][0] = 2.0 * acc[a][b][0] - o0;
      acc[a][b][1] = 2.0 * acc[a][b][1] - o1;
    }

  // ---- c_k, S = lamda .* (c_k - phi_k) (:422), ergodic metric ---------------
  {
    const double inv_t = 1.0 / (double)(p.M + p.N);  // basis.cpp:119
    double metric = 0.0;
#pragma unroll
    for (int ti = 0; ti < TILES; ti++)
#pragma unroll
      for (int tj = 0; tj < TILES; tj++)
#pragma unroll
        for (int e = 0; e < 2; e++)
        {
          const int ky = 8 * ti + g, kx = 8 * tj + 2 * q + e;
          double s = 0.0;
          if (ky < nb && kx < nb)
          {
            const int k = ky * nb + kx;
            const double c = __dmul_rn(inv_t, acc[ti][tj][e]);
            const double d = __dsub_rn(c, phik_at<PER_INST>(p, inst, K, k));
            s = __ldg(p.lamk + k) * d;
            metric += s * d;
            if (p.ck) p.ck[(size_t)inst * K + k] = c;
          }
          if (ky < NB && kx < NB) Ssm[ky * Cfg::kSPitch + kx] = s;
        }
    if (p.metric)
    {
      metric = warp_sum(metric);
      if (lane == 0) p.metric[inst] = metric;
    }
  }
  __syncwarp();

  // S as A fragments, ONE copy for both bilinear forms: R1 = S (a_kx SX) and R2 = S CX share the A operand when the
  // order weight a_kx rides on the sin chain (B operand) and b_ky is applied to R2's rows in the epilogue
  double SF[TILES][GKS];
#pragma unroll
  for (int mi = 0; mi < TILES; mi++)
#pragma unroll
    for (int ks = 0; ks < GKS; ks++)
    {
      const int ky = 8 * mi + g, kx = 4 * ks + q;
      SF[mi][ks] = (ky < NB && kx < NB) ? Ssm[ky * Cfg::kSPitch + kx] : 0.0;
    }
  __syncwarp();  // S has been read: the table region is free for the y tables
  const double a4 = 4.0 * frame<PER_INST, kFrAx>(p, inst);  // a_kx advances by 4 a per k-step (kx = 4 ks + q)

  // ---- per round, last round first: metric gradient in 8-step tiles (:419-436), then the backward co-state
  //      pass and the control update of the same 32 steps (:277, :439-451) ----------------------------------
  double* const tyc = tab;                    // cos(ky b y_t), [ky][8]
  double* const tys = tab + Cfg::kYStride;    // sin(ky b y_t)
  // y-table builder role: lane = (parity of the orders, cos | sin, slot)
  const int ypar = lane >> 4, ycs = (lane >> 3) & 1, yslot = lane & 7;
  double* const myy = tab + ycs * Cfg::kYStride + ypar * 8 + yslot;

  double r0c = 0.0, r1c = 0.0, r2c = 0.0;  // rho(T) = 0 (:203)
  for (int r = rounds - 1; r >= 0; r--)
  {
    const int i = r * 32 + lane;
    const bool valid = i < p.N;
    const int left = p.N - r * 32;  // valid steps in this round (warp-uniform)
    const int ntiles = min(4, (left + 7) >> 3);
    for (int nj = 0; nj < ntiles; nj++)
    {
      const int t0 = r * 32 + 8 * nj;
      {
        // y tables of the tile: even / odd orders of cos (ycs = 0) or sin (ycs = 1), v_{k+2} = (4c^2 - 2) v_k - v_{k-2}
        const int t = t0 + yslot;
        const double c = rec[6 * npad + t], sn = rec[7 * npad + t];
        const double m = fma(4.0 * c, c, -2.0);
        double vm, v;
        if (ycs == 0)
        {
          vm = ypar ? c : fma(2.0 * c, c, -1.0);  // cos(-t) | cos(-2t)
          v = ypar ? c : 1.0;
        }
        else
        {
          vm = ypar ? -sn : -2.0 * sn * c;  // sin(-t) | sin(-2t)
          v = ypar ? sn : 0.0;
        }
        __syncwarp();  // the previous tile's y-fragment loads are done
#pragma unroll
        for (int k = 0; k < NB; k += 2)
        {
          myy[k * 8] = v;
          const double vn = fma(m, v, -vm);
          vm = v;
          v = vn;
        }
      }
      // x operands in registers: lane (g, q) needs cos / sin((4 ks + q) a x_t) of ITS step t = t0 + g
      double X, Xm, Z, Zm, m4;
      {
        const double c = rec[4 * npad + t0 + g], s = rec[5 * npad + t0 + g];
        const double c2 = fma(2.0 * c, c, -1.0), s2 = 2.0 * s * c;
        const double c3 = fma(2.0 * c, c2, -c), s3 = fma(2.0 * c, s2, -s);
        const double c4 = fma(2.0 * c2, c2, -1.0), s4 = 2.0 * s2 * c2;
        // orders q and q - 4:  q = 0: (1, c4 | 0, -s4)  1: (c, c3 | s, -s3)  2: (c2, c2 | s2, -s2)  3: (c3, c | s3, -s)
        X = q == 0 ? 1.0 : q == 1 ? c : q == 2 ? c2 : c3;
        Xm = q == 0 ? c4 : q == 1 ? c3 : q == 2 ? c2 : c;
        Z = q == 0 ? 0.0 : q == 1 ? s : q == 2 ? s2 : s3;
        Zm = -(q == 0 ? s4 : q == 1 ? s3 : q == 2 ? s2 : s);
        m4 = 2.0 * c4;
      }
      double R1[TILES][2], R2[TILES][2];
#pragma unroll
      for (int mi = 0; mi < TILES; mi++) R1[mi][0] = R1[mi][1] = R2[mi][0] = R2[mi][1] = 0.0;
      double akx = (double)q * frame<PER_INST, kFrAx>(p, inst);
#pragma unroll
      for (int ks = 0; ks < GKS; ks++)
      {
        const double za = akx * Z;  // a_kx sin(kx a x_t)
        akx += a4;
#pragma unroll
        for (int mi = 0; mi < TILES; mi++)
        {
          dmma_gr(R1[mi][0], R1[mi][1], SF[mi][ks], za);
          dmma_gr(R2[mi][0], R2[mi][1], SF[mi][ks], X);
        }
        if (ks + 1 < GKS)
        {
          const double xn = fma(m4, X, -Xm), zn = fma(m4, Z, -Zm);
          Xm = X;
          X = xn;
          Zm = Z;
          Z = zn;
        }
      }
      __syncwarp();  // the y tables of this tile are complete
      // lane (g, q) holds R[ky = 8 mi + g][slot 2q, 2q + 1]: weight with the y tables
      double v0 = 0.0, v1 = 0.0, w0 = 0.0, w1 = 0.0;  // e_x, e_y partial sums for slots 2q, 2q + 1
#pragma unroll
      for (int mi = 0; mi < TILES; mi++)
      {
        const int ky = 8 * mi + g;
        if ((TILES * 8 == NB) || (ky < NB))
        {
          const double2 cy2 = *reinterpret_cast<const double2*>(tyc + ky * 8 + 2 * q);
          const double2 sy2 = *reinterpret_cast<const double2*>(tys + ky * 8 + 2 * q);
          const double bky = (double)ky * frame<PER_INST, kFrBy>(p, inst);
          v0 = fma(cy2.x, R1[mi][0], v0);
          v1 = fma(cy2.y, R1[mi][1], v1);
          w0 = fma(sy2.x, bky * R2[mi][0], w0);
          w1 = fma(sy2.y, bky * R2[mi][1], w1);
        }
      }
      // sum over the 8 row lanes g (lane = 4 g + q) by recursive halving:
      //   xor 16: lanes g < 4 keep e_x, g >= 4 keep e_y;  xor 8: keep slot 2q (g & 2 == 0) or 2q + 1;  xor 4: full
      {
        const bool hi = (g & 4) != 0;
        const double s0 = hi ? v0 : w0, s1 = hi ? v1 : w1;  // what the partner keeps
        double k0 = hi ? w0 : v0, k1 = hi ? w1 : v1;
        k0 += __shfl_xor_sync(kFull, s0, 16);
        k1 += __shfl_xor_sync(kFull, s1, 16);
        const bool odd = (g & 2) != 0;
        double kk = odd ? k1 : k0;
        kk += __shfl_xor_sync(kFull, odd ? k0 : k1, 8);
        kk += __shfl_xor_sync(kFull, kk, 4);
        if ((g & 1) == 0) stage_[(hi ? 32 : 0) + 8 * nj + 2 * q + (odd ? 1 : 0)] = kk;
      }
    }
    __syncwarp();
    double ex = 0.0, ey = 0.0;
    if (lane < 8 * ntiles)
    {
      ex = stage_[lane];
      ey = stage_[32 + lane];
    }
    __syncwarp();  // the stage is free for the next round
    // dF/dx = -a sin(a x) cos(b y), dF/dy = -b cos(a x) sin(b y); times expl_weight (:433)
    ex = -ex * p.w;
    ey = -ey * p.w;

    const int ir = min(i, npad - 1);  // lanes past the records are not valid steps
    const double ce = rec[0 * npad + ir], se = rec[1 * npad + ir];
    const double xf = rec[2 * npad + ir], yf = rec[3 * npad + ir];
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
    // A = fdx(x_i, u_i): only A02, A12 are non-zero
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
    if (valid && !finite) atomicOr(p.fault, 4);  // NaN / Inf guard (SURVEY.md section 5)
    if (r == 0)
    {
      if constexpr (WideIo<WARPS>::kOn)
        wide_io_store(wio, p, lane, warp, un);
      else
        publish_first_twist(p, inst, lane, un);
    }
  }
}
}  // namespace eb
