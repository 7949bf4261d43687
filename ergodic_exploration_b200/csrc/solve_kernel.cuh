// solve_kernel.cuh -- one receding-horizon ergodic control() iteration for a
// batch of independent instances, fused into ONE kernel (sm_100a, FP64).
//
// Replaces, per instance, the body of ErgodicControl<ModelT>::control()
// (ergodic_control.hpp:225-311): the control shift (:233-234), the RK4 forward
// rollout (integrator.hpp:135-152,176-184), ReplayBuffer::sampleMemory
// (buffer.cpp:64-111), Basis::trajCoeff (basis.cpp:109-120), gradErgodicMetric
// (:419-436), gradBarrier (:454-474), the backward co-state RK4
// (integrator.hpp:154-174,186-194 with rhodot :65-69) and updateControl
// (:439-451), plus the ergodic metric sum_k lamda_k (c_k - phi_k)^2.
//
// Mapping.  One warp owns one instance; lanes are TIME STEPS.
//  * The 3-twist models have theta' = u2, so theta_i is a prefix sum of the
//    per-step increments and (x, y) are prefix sums of per-step RK4
//    displacements that depend only on theta: the "sequential" RK4 chain is
//    three warp-shuffle scans.  The co-state has the same structure backwards
//    (A^T rho only feeds rho_2), so it is three suffix scans.
//  * cos(k a x), sin(k a x) for k < nb come from one sincospi per state and the
//    Chebyshev three-term recurrence (error ~ k^2 eps, << 1e-9 for nb <= 32).
//  * c_k = (1/T) sum_t cos(ky b y_t) cos(kx a x_t) is a rank-T update of an
//    nb x nb matrix: lanes stage their cosine rows in shared memory, and the
//    warp contracts them with FP64 tensor-core tiles (mma.sync m8n8k4 ->
//    DMMA.8x8x4), accumulators in registers.
//  * the metric gradient is a pair of bilinear forms per step,
//    sx^T (a.S) cy and cx^T (S.b) sy: each lane evaluates them for its own time
//    step with S broadcast from shared memory, cos/sin rows of a kx block held in
//    registers.
//  * N > 1 GPUs: the first twists are published to every rank over NVLink peer
//    memory by this kernel itself (peer_gather.cuh).
// This kernel serves num_basis <= 12 and 25..32; 13..24 run solve_kernel2
// (solve_kernel_v2.cuh), which also puts the gradient on the tensor cores.
// Shared memory per warp: SolveCfg::kTabDoubles (the two c_k tables, S aliases
// them) + (4 or 8)*32*rounds doubles of per-step records.
#pragma once

#include "common.cuh"

namespace eb
{
constexpr int kModelSimpleCart = 0;
constexpr int kModelOmni = 1;
constexpr int kSolveWarps = 4;   // warps (instances in flight) per CTA
constexpr int kMaxPeers = 8;     // ranks of one NVSwitch box
constexpr int kPeerBuffers = 4;  // gathered buffers rotating by step (fused gather)
constexpr int kTabSlots = 16;    // time slots per coefficient chunk (half a round)
constexpr int kTabStride = 20;   // 16 slots + 4 pad: 20 % 16 == 4 -> conflict-free fragment loads

#ifdef EB_PHASE_TIMING
// debug build only: per-instance clock64() stamps at the phase boundaries
constexpr int kPhaseSlots = 16;
__device__ long long g_phase[65536 * kPhaseSlots];
#define EB_PHASE(idx)                                                                      \
  do                                                                                       \
  {                                                                                        \
    if (lane == 0 && inst < 65536) g_phase[inst * kPhaseSlots + (idx)] = clock64();        \
  } while (0)
#else
#define EB_PHASE(idx) do { } while (0)
#endif

#ifdef EB_DEBUG_DUMP
__device__ double g_dbg[4096 * 16];  // debug build only: per-step intermediates of instance 0
#endif

// Ablation timing (tools/ablate.sh; debug builds only, results are numerically WRONG): -DEB_ABL=<bits> removes a
// class of work from the fused kernel so that its marginal cost can be read off the kernel time.
//  1: c_k DMMAs -> integer xor of the operands   2: gradient DMMAs (solve_kernel2) -> xor   4: c_k table recurrences
//  + stores   8: sin/cos polynomials -> 2 flops   64: warp scans -> identity
//  128: solve_kernel returns at once (launch + drain cost of the grid)
#ifndef EB_ABL
#define EB_ABL 0
#endif
__device__ __forceinline__ void abl_xor(double& d0, double a, double b)
{
  d0 = __hiloint2double(__double2hiint(d0), __double2loint(d0) ^ __double2loint(a) ^ __double2hiint(b));
}
__device__ __forceinline__ void dmma_ck(double& d0, double& d1, double a, double b)
{
#if EB_ABL & 1
  abl_xor(d0, a, b);
#else
  dmma884(d0, d1, a, b);
#endif
}
__device__ __forceinline__ void dmma_gr(double& d0, double& d1, double a, double b)
{
#if EB_ABL & 2
  abl_xor(d0, a, b);
#else
  dmma884(d0, d1, a, b);
#endif
}

struct SolveParams
{
  int B, N, M, nb;
  int mem_count, batch_size, idx_mode;  // idx_mode: 0 identity, 1 from mem_idx, 2 device sampler
  double dt, lx, ly, inv_lx, inv_ly, ax, by, xmin, ymin, w;
  double Rinv[9], umin[3], umax[3], bw, beps;
  unsigned long long seed, call;
  const double* x;       // [B][3]
  double* pose_out;      // [B][3] or null: copy of x kept as pose_ (:227)
  const double* ut_in;   // [B][N][3]
  double* ut_out;        // [B][N][3]
  const double* hist;    // [cap][B][3]
  const double* hist_cos;  // [cap][B][2] or null: cos(pi (x - xmin) / lx), cos(pi (y - ymin) / ly) of every stored state,
                           // kept by the host side for the current Fourier frame (hist_cos_kernel)
  const int* mem_idx;    // [B][batch_size]
  int* mem_idx_out;      // [B][batch_size]
  const double* phik;    // [nb*nb]
  const double* lamk;    // [nb*nb]
  double* u0;            // [B][3]
  double* metric;        // [B] or null
  double* ck;            // [B][nb*nb] or null
  int* fault;
  // fused gather over NVLink peer memory (peer_gather.cuh): every rank's copy of the
  // gathered first twists, already offset to this rank's row block; 0 = off
  int n_peer;
  double* u0_peer[kMaxPeers];
  unsigned long long* flag_peer[kMaxPeers];  // this rank's slot in every rank's arrival flags
  unsigned long long flag_value;             // written there once all of this rank's rows have landed
  unsigned int* done_counter;                // warps of this launch that have published their row
  const unsigned long long* my_flags;        // this rank's own arrival flags [n_peer] ...
  unsigned long long need;                   // ... must all have reached this before the buffer is reused
  // num_basis > 32 (solve_kernel_big.cuh): one row of nb * nb doubles per resident CTA, and how many rows there are
  double* big_scratch;
  int big_rows;
  // per-instance targets (PER_INST kernels): Fourier frame of every instance [B][kFrDoubles]; phik is then [B][nb*nb]
  const double* frames;
};

// Layout of a per-instance frame record.  The derived values are computed by the same expressions as the shared
// frame's (eb_control_dev), so an instance whose frame equals the shared one sees the same bits.
enum FrameField
{
  kFrXmin,
  kFrYmin,
  kFrLx,
  kFrLy,
  kFrInvLx,
  kFrInvLy,
  kFrAx,
  kFrBy,
  kFrDoubles
};

// One value of the Fourier frame of `inst`: read at its use site (L1 serves the 64-byte record), never hoisted by hand
// across the kernel, so the per-instance kernels keep the shared ones' register budget.
template <bool PER_INST, int F>
__device__ __forceinline__ double frame(const SolveParams& p, const int inst)
{
  if constexpr (PER_INST)
    return __ldg(p.frames + (size_t)inst * kFrDoubles + F);
  else if constexpr (F == kFrXmin)
    return p.xmin;
  else if constexpr (F == kFrYmin)
    return p.ymin;
  else if constexpr (F == kFrLx)
    return p.lx;
  else if constexpr (F == kFrLy)
    return p.ly;
  else if constexpr (F == kFrInvLx)
    return p.inv_lx;
  else if constexpr (F == kFrInvLy)
    return p.inv_ly;
  else if constexpr (F == kFrAx)
    return p.ax;
  else
    return p.by;
}

// phi_k[k] of `inst`: the shared row, or the instance's own row of the [B][K] table
template <bool PER_INST>
__device__ __forceinline__ double phik_at(const SolveParams& p, const int inst, const int K, const int k)
{
  if constexpr (PER_INST)
    return __ldg(p.phik + (size_t)inst * K + k);
  else
    return __ldg(p.phik + k);
}

// The first twist of one instance: lanes 0..2 store one contiguous 24-byte segment (u0 may live in mapped host
// memory); with a peer group (N > 1 GPUs) the same row goes into every rank's gathered buffer.
__device__ __forceinline__ void publish_first_twist(const SolveParams& p, const int inst, const int lane, const double (&un)[3])
{
  const double a0 = __shfl_sync(kFull, un[0], 0), a1 = __shfl_sync(kFull, un[1], 0), a2 = __shfl_sync(kFull, un[2], 0);
  const double mine = lane == 0 ? a0 : (lane == 1 ? a1 : a2);
  if (lane < 3) p.u0[(size_t)inst * 3 + lane] = mine;
  if (p.n_peer > 0)
  {
    // The gather IS these stores: the row goes straight into every rank's gathered
    // buffer over NVLink (P2P stores, no separate collective, nothing to wait for
    // on this rank).  When the last warp of the launch has published its row, this
    // rank's arrival flag is raised on every peer (release at system scope).
    // Buffer reuse: this step's buffer was last written kPeerBuffers steps ago; a rank
    // reads a step's rows before it launches the next step, so once every rank has
    // FINISHED step (this - kPeerBuffers + 1) -- p.need, long past in a balanced run --
    // nobody can still be reading it.  Checked here, at the end of the warp's work.
    if (lane < p.n_peer)
      while (*(const volatile unsigned long long*)(p.my_flags + lane) < p.need) __nanosleep(100);
    __syncwarp();
    if (lane < 3)
    {
#pragma unroll
      for (int q = 0; q < kMaxPeers; q++)
        if (q < p.n_peer) p.u0_peer[q][(size_t)inst * 3 + lane] = mine;
    }
    // release at GPU scope into the arrival counter; the last warp's system-scope fence is
    // cumulative over every row it has thereby observed (PTX memory model: the gpu-scope
    // fence + counter increment of each warp synchronises with the last warp's read of the
    // counter, and causality order is transitive), so only that one warp pays for a system fence
    __threadfence();
    __syncwarp();
    if (lane == 0)
    {
      const unsigned int prev = atomicAdd(p.done_counter, 1u);
      if (prev == (unsigned int)p.B - 1u)
      {
        *p.done_counter = 0u;  // ready for the next launch on this stream
        __threadfence_system();
#pragma unroll
        for (int q = 0; q < kMaxPeers; q++)
          if (q < p.n_peer) *(volatile unsigned long long*)p.flag_peer[q] = p.flag_value;
      }
    }
  }
}

// Wide single-wave CTAs (one per SM, no peer group): the poses of the CTA's instances come in and their first twists go
// out as ONE contiguous segment each -- 3 coalesced requests per CTA instead of a 24-byte request per warp.  Both may
// live in page-locked HOST memory (eb_control_host's zero-copy path), where 4096 small PCIe requests cost 3 us (reads)
// and 6 us (writes) of a 23 us step.  The last warp of the CTA to finish writes the segment.
template <int WARPS>
struct WideIo
{
  static constexpr bool kOn = WARPS > kSolveWarps;
  double x[kOn ? 3 * WARPS : 1];
  double u0[kOn ? 3 * WARPS : 1];
  unsigned int arrived;
};

template <int WARPS>
__device__ __forceinline__ void wide_io_load(WideIo<WARPS>& io, const SolveParams& p)
{
  const int first = blockIdx.x * WARPS;
  const int cnt = min(WARPS, p.B - first);
  if ((int)threadIdx.x < 3 * cnt) io.x[threadIdx.x] = p.x[(size_t)first * 3 + threadIdx.x];
  if (threadIdx.x == 0) io.arrived = 0u;
  __syncthreads();  // every warp of the CTA is still here (the early exit of surplus warps comes after this)
}

template <int WARPS>
__device__ __forceinline__ void wide_io_store(WideIo<WARPS>& io, const SolveParams& p, const int lane, const int warp,
                                              const double (&un)[3])
{
  const double a0 = __shfl_sync(kFull, un[0], 0), a1 = __shfl_sync(kFull, un[1], 0), a2 = __shfl_sync(kFull, un[2], 0);
  if (lane < 3) io.u0[3 * warp + lane] = lane == 0 ? a0 : (lane == 1 ? a1 : a2);
  const int first = blockIdx.x * WARPS;
  const int cnt = min(WARPS, p.B - first);
  __syncwarp();
  unsigned int last = 0u;
  if (lane == 0)
  {
    __threadfence_block();  // release this warp's row ...
    last = atomicAdd(&io.arrived, 1u) == (unsigned int)(cnt - 1) ? 1u : 0u;
    __threadfence_block();  // ... and acquire the others' before the segment is read
  }
  if (__shfl_sync(kFull, last, 0))
    for (int i = lane; i < 3 * cnt; i += 32) p.u0[(size_t)first * 3 + i] = io.u0[i];
}

// Programmatic dependent launch (cudaLaunchAttributeProgrammaticStreamSerialization): wait for the kernel ahead in the
// stream to complete and flush, then let the kernel behind start placing its CTAs as this one's drain.  Both are no-ops
// for a launch without the attribute.
__device__ __forceinline__ void grid_dependency_wait()
{
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

template <int MODEL>
__device__ __forceinline__ void model_f(double u0, double u1, double c, double s, double& fx, double& fy)
{
  if (MODEL == kModelOmni)
  {  // omni.hpp:177-182
    fx = u0 * c - u1 * s;
    fy = u0 * s + u1 * c;
  }
  else
  {  // cart.hpp:172
    fx = u0 * c;
    fy = u0 * s;
  }
}

// Forward rollout of one round of 32 steps (integrator.hpp:135-152,176-184).
// In: controls of this lane's step, carries (state before the round's first
// step).  Out: post-step state of this lane's step and its heading cos/sin.
struct RolloutCarry
{
  double x, y, th, cth, sth;
};

template <int MODEL>
__device__ __forceinline__ void rollout_round(const double dt, const bool valid, const int lane, const double u0,
                                              const double u1, const double u2, RolloutCarry& cy, double& xo,
                                              double& yo, double& tho, double& ce, double& se)
{
  // theta: k1..k4 all equal u2, so the RK4 increment is (dt/6)*(u2+2u2+2u2+u2)
  const double dth = valid ? (dt / 6.0) * (((u2 + 2.0 * u2) + 2.0 * u2) + u2) : 0.0;
  const double inc = warp_scan_incl(dth, lane);
  double exc = __shfl_up_sync(kFull, inc, 1);
  if (lane == 0) exc = 0.0;
  const double th_before = cy.th + exc;
  tho = cy.th + inc;
  const double thm = th_before + dt * (0.5 * u2);  // k2, k3 stage heading
  double sm, cm;
  fast_sincos(tho, &se, &ce);  // k4 stage heading == post-step heading (to rounding)
  fast_sincos(thm, &sm, &cm);
  double cb = __shfl_up_sync(kFull, ce, 1), sb = __shfl_up_sync(kFull, se, 1);
  if (lane == 0)
  {
    cb = cy.cth;
    sb = cy.sth;
  }
  double k1x, k1y, k2x, k2y, k4x, k4y;
  model_f<MODEL>(u0, u1, cb, sb, k1x, k1y);
  model_f<MODEL>(u0, u1, cm, sm, k2x, k2y);
  model_f<MODEL>(u0, u1, ce, se, k4x, k4y);
  const double dx = valid ? (dt / 6.0) * (((k1x + 2.0 * k2x) + 2.0 * k2x) + k4x) : 0.0;
  const double dy = valid ? (dt / 6.0) * (((k1y + 2.0 * k2y) + 2.0 * k2y) + k4y) : 0.0;
  xo = cy.x + warp_scan_incl(dx, lane);
  yo = cy.y + warp_scan_incl(dy, lane);
  cy.x = __shfl_sync(kFull, xo, 31);
  cy.y = __shfl_sync(kFull, yo, 31);
  cy.th = __shfl_sync(kFull, tho, 31);
  cy.cth = __shfl_sync(kFull, ce, 31);
  cy.sth = __shfl_sync(kFull, se, 31);
}

// Rank-32 update of the nb x nb coefficient accumulators from one round of
// (up to) 32 states, in two half-rounds of 16 states.  The 32 lanes of the warp
// build the two cosine tables of a half-round together: lane (axis = lane / 16,
// slot = lane % 16) runs the Chebyshev recurrence of ONE axis of ONE state and
// writes its row transposed (tab[k][slot]); the even and odd orders are two
// independent chains, T_{k+2} = (4c^2 - 2) T_k - T_{k-2}.  Then the warp runs up
// to four DMMA k-steps over those 16 states.
template <int NB>
__device__ __forceinline__ void coeff_chunk(double* __restrict__ tabx, const int lane, const bool valid,
                                            const int nvalid, const double c1x, const double c1y,
                                            double (&acc)[(NB + 7) / 8][(NB + 7) / 8][2])
{
  constexpr int TILES = (NB + 7) / 8;
  static_assert(NB % 2 == 0, "NB must be even");
  const int g = lane >> 2, q = lane & 3;
  const double* taby = tabx + NB * kTabStride;
  double* const mytab = tabx + (lane >> 4) * (NB * kTabStride) + (lane & 15);  // this lane's axis table, its slot
#pragma unroll
  for (int h = 0; h < 2; h++)
  {
    const int left = nvalid - h * kTabSlots;  // valid states in this half (warp-uniform)
    if (left <= 0) break;
    {
      // state (lane % 16) of this half lives in lane 16 h + lane % 16
      const int src = 16 * h + (lane & 15);
      const double sx = __shfl_sync(kFull, c1x, src), sy = __shfl_sync(kFull, c1y, src);
      const bool ok = __shfl_sync(kFull, (int)valid, src) != 0;
      const double v = lane < 16 ? sx : sy;
      // (T_{-2}, T_0) = (2 v^2 - 1, 1), (T_{-1}, T_1) = (v, v); states past the end
      // of the trajectory give zero rows (the recurrence is homogeneous)
      const double m = fma(4.0 * v, v, -2.0);
      double em = ok ? fma(2.0 * v, v, -1.0) : 0.0, ek = ok ? 1.0 : 0.0;
      double om = ok ? v : 0.0, ok1 = om;
      __syncwarp();  // the previous half's fragment loads are done
#if EB_ABL & 4
      mytab[0] = ek + ok1 + em * m;
#else
#pragma unroll
      for (int k = 0; k < NB; k += 2)
      {
        mytab[k * kTabStride] = ek;
        mytab[(k + 1) * kTabStride] = ok1;
        const double en = fma(m, ek, -em), on = fma(m, ok1, -om);
        em = ek;
        ek = en;
        om = ok1;
        ok1 = on;
      }
#endif
    }
    __syncwarp();
    const int ksteps = (min(left, kTabSlots) + 3) >> 2;
    for (int s = 0; s < ksteps; s++)
    {
      double a[TILES], b[TILES];
#pragma unroll
      for (int t = 0; t < TILES; t++)
      {
        const int k = 8 * t + g;
        const bool in = (TILES * 8 == NB) || (k < NB);
        a[t] = in ? taby[k * kTabStride + 4 * s + q] : 0.0;
        b[t] = in ? tabx[k * kTabStride + 4 * s + q] : 0.0;
      }
#pragma unroll
      for (int ti = 0; ti < TILES; ti++)
#pragma unroll
        for (int tj = 0; tj < TILES; tj++) dmma_ck(acc[ti][tj][0], acc[ti][tj][1], a[ti], b[tj]);
    }
  }
}

// Per-NB tuning of the fused kernel.
//  * kRecompute: the per-step record keeps 4 fields (heading cos/sin, Fourier-frame
//    position) and the gradient pass re-evaluates sincospi of the position, instead
//    of 8 fields -- ~3 % more FP64 work for 2 KB (N <= 64) less shared memory per
//    warp, which buys resident warps where shared memory is the limiter.
//  * kBlock: the gradient's kx range is walked in blocks of kBlock orders so that
//    only 2 kBlock doubles of cos / sin rows are live in registers.
//  * kMinBlocks: resident CTAs per SM the register allocation is tuned for.
// Instantiated for NB = 8, 10, 12 and 32 (num_basis 13..24 run solve_kernel2).
template <int NB>
struct SolveCfg
{
  static constexpr bool kRecompute = NB >= 16;
  static constexpr int kFields = kRecompute ? 4 : 8;
  // per-warp table region: the two c_k tables (pitch 20, 16 slots); S (NB x NB, pitch NB) aliases it
  static constexpr int kSPitch = NB;
  static constexpr int kTabDoubles = 2 * NB * kTabStride;
  static constexpr int kBlock = NB <= 12 ? NB : 8;
  static constexpr int kMinBlocks = NB <= 10 ? 7 : NB <= 12 ? 6 : 4;
  // Single-wave batches (configs[1]: 4096 instances on 148 SMs) run ONE CTA per SM with this many warps: the SM's
  // instances then start together instead of behind 7 serial CTA launches (measured 34.9 -> 31.2 us at 4096 x nb 10)
  static constexpr int kWideWarps = NB <= 10 ? 28 : NB <= 12 ? 24 : 16;
  static_assert(NB <= 12 || NB == 32, "num_basis 13..24 run solve_kernel2");
  static_assert(NB % kBlock == 0, "kx blocks must tile NB");
};

inline size_t solve_smem_bytes(int tab_doubles, int fields, int rounds, int warps = kSolveWarps)
{
  return sizeof(double) * warps * (size_t)(tab_doubles + fields * 32 * rounds);
}

template <int MODEL, int NB, int WARPS = kSolveWarps, bool PER_INST = false>
__global__ void __launch_bounds__(WARPS * 32, WARPS == kSolveWarps ? SolveCfg<NB>::kMinBlocks : 1) solve_kernel(const SolveParams p)
{
  using Cfg = SolveCfg<NB>;
  constexpr int TILES = (NB + 7) / 8;
  constexpr int KB = Cfg::kBlock;
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rounds = (p.N + 31) >> 5;
  const int npad = rounds * 32;
  const int nb = p.nb, K = nb * nb;

  const int inst = blockIdx.x * WARPS + warp;
  __shared__ WideIo<WARPS> wio;
  grid_dependency_wait();  // programmatic dependent launch: nothing global is touched before the previous kernel is complete
  // the first round's controls do not depend on the pose: their HBM latency runs under the pose staging (which may be a
  // PCIe round trip on the zero-copy host path) instead of behind it
  double e_u0 = 0.0, e_u1 = 0.0, e_u2 = 0.0;
  if (inst < p.B && lane + 1 < p.N)
  {
    const double* e_in = p.ut_in + ((size_t)inst * p.N + lane + 1) * 3;
    e_u0 = e_in[0];
    e_u1 = e_in[1];
    e_u2 = e_in[2];
  }
  if constexpr (WideIo<WARPS>::kOn) wide_io_load(wio, p);
  if (inst >= p.B) return;
#if EB_ABL & 128
  if (lane < 3) p.u0[(size_t)inst * 3 + lane] = 0.0;  // ablation timing only: the launch itself
  return;
#endif
  EB_PHASE(0);

  // per-warp shared memory: the two cosine tables, then the per-step records
  double* tabx = smem + warp * (Cfg::kTabDoubles + Cfg::kFields * npad);
  double* rec = tabx + Cfg::kTabDoubles;
  double* Ssm = tabx;  // S (NB x NB) aliases the two tables (2*NB*20 doubles) once c_k is complete

  double acc[TILES][TILES][2];
#pragma unroll
  for (int i = 0; i < TILES; i++)
#pragma unroll
    for (int j = 0; j < TILES; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

  // ---- sampled past states (buffer.cpp:64-111), Fourier frame (:243-244) ----
  for (int base = 0; base < p.M; base += 32)
  {
    const int j = base + lane;
    const bool valid = j < p.M;
    double c1x = 1.0, c1y = 1.0;
    if (valid)
    {
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
      if (p.idx_mode != 0 && p.mem_idx_out) p.mem_idx_out[(size_t)inst * p.batch_size + j] = (int)idx;
      if (p.hist_cos)
      {  // cosines cached per stored state: 16 bytes in, no trig
        const double2 hc = *reinterpret_cast<const double2*>(p.hist_cos + ((size_t)idx * p.B + inst) * 2);
        c1x = hc.x;
        c1y = hc.y;
      }
      else
      {
        const double* h = p.hist + ((size_t)idx * p.B + inst) * 3;
        const double xf = h[0] - frame<PER_INST, kFrXmin>(p, inst), yf = h[1] - frame<PER_INST, kFrYmin>(p, inst);
        c1x = fast_cospi(xf * frame<PER_INST, kFrInvLx>(p, inst));
        c1y = fast_cospi(yf * frame<PER_INST, kFrInvLy>(p, inst));
      }
    }
    const int nvalid = min(32, p.M - base);
    coeff_chunk<NB>(tabx, lane, valid, nvalid, c1x, c1y, acc);
  }

  EB_PHASE(1);
  // ---- forward rollout with the shifted controls (:233-237) ----------------
  const double* ut_in = p.ut_in + (size_t)inst * p.N * 3;
  double* ut_out = p.ut_out + (size_t)inst * p.N * 3;
  RolloutCarry cy;
  {
    // one 24-byte request per warp (x may live in mapped host memory); wide CTAs: from the CTA's staged segment
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
    if (r == 0)
    {
      u0 = e_u0;
      u1 = e_u1;
      u2 = e_u2;
    }
    else if (i + 1 < p.N)
    {  // shift left by one column, last column zero
      u0 = ut_in[(i + 1) * 3 + 0];
      u1 = ut_in[(i + 1) * 3 + 1];
      u2 = ut_in[(i + 1) * 3 + 2];
    }
    if (MODEL == kModelSimpleCart && !(fabs(u1 - 0.0) < 1.0e-12)) atomicOr(p.fault, 1);  // cart.hpp:167-170
    double xo, yo, tho, ce, se;
    rollout_round<MODEL>(p.dt, valid, lane, u0, u1, u2, cy, xo, yo, tho, ce, se);
    const double xf = xo - frame<PER_INST, kFrXmin>(p, inst), yf = yo - frame<PER_INST, kFrYmin>(p, inst);
    rec[0 * npad + i] = ce;
    rec[1 * npad + i] = se;
    rec[2 * npad + i] = xf;
    rec[3 * npad + i] = yf;
    double ca, cb;
    if (Cfg::kRecompute)
    {
      ca = fast_cospi(xf * frame<PER_INST, kFrInvLx>(p, inst));
      cb = fast_cospi(yf * frame<PER_INST, kFrInvLy>(p, inst));
    }
    else
    {
      double sa, sb;
      fast_sincospi(xf * frame<PER_INST, kFrInvLx>(p, inst), &sa, &ca);
      fast_sincospi(yf * frame<PER_INST, kFrInvLy>(p, inst), &sb, &cb);
      rec[4 * npad + i] = ca;
      rec[5 * npad + i] = sa;
      rec[6 * npad + i] = cb;
      rec[7 * npad + i] = sb;
    }
    const int nvalid = min(32, p.N - r * 32);
    if (r < 2) EB_PHASE(2 + 2 * r);
    coeff_chunk<NB>(tabx, lane, valid, nvalid, ca, cb, acc);
    if (r < 2) EB_PHASE(3 + 2 * r);
  }

  // ---- c_k, S = lamda .* (c_k - phi_k) (:422), ergodic metric ---------------
  __syncwarp();
  {
    const int g = lane >> 2, q = lane & 3;
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
            // explicitly rounded (no FMA contraction): c_k as stored == c_k as used, whichever
            // way the compiler specialises the p.ck branch
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
  EB_PHASE(6);

  // ---- per round, last round first: gradient of the ergodic metric, one time
  //      step per lane (:419-436), then the backward co-state pass and the
  //      control update of the same 32 steps (:277, :439-451) -------------------
  double r0c = 0.0, r1c = 0.0, r2c = 0.0;  // rho(T) = 0 (:203)
  for (int r = rounds - 1; r >= 0; r--)
  {
    const int i = r * 32 + lane;
    const bool valid = i < p.N;
    const double ce = rec[0 * npad + i], se = rec[1 * npad + i];
    const double xf = rec[2 * npad + i], yf = rec[3 * npad + i];
    double u0 = 0.0, u1 = 0.0;  // issued ahead of the gradient: their L2 latency runs under it (C2: 22.55 -> 22.42 us)
    if (i + 1 < p.N)
    {
      u0 = ut_in[(i + 1) * 3 + 0];
      u1 = ut_in[(i + 1) * 3 + 1];
    }
    double ca, sa, cb, sb;
    if (Cfg::kRecompute)
    {
      fast_sincospi(xf * frame<PER_INST, kFrInvLx>(p, inst), &sa, &ca);
      fast_sincospi(yf * frame<PER_INST, kFrInvLy>(p, inst), &sb, &cb);
    }
    else
    {
      ca = rec[4 * npad + i];
      sa = rec[5 * npad + i];
      cb = rec[6 * npad + i];
      sb = rec[7 * npad + i];
    }
    double ex = 0.0, ey = 0.0;
    // (cos, sin)((k-1) a x), (cos, sin)(k a x) started at k = 0, carried across the kx blocks
    double xcm = ca, xck = 1.0, xsm = -sa, xsk = 0.0;
    const double xt2 = 2.0 * ca, yt2 = 2.0 * cb;
#pragma unroll
    for (int kb = 0; kb < NB; kb += KB)
    {
      double cx[KB], asx[KB];  // cos(kx a x), a_kx sin(kx a x) for kx = kb .. kb + KB - 1
#pragma unroll
      for (int j = 0; j < KB; j++)
      {
        cx[j] = xck;
        asx[j] = ((double)(kb + j) * frame<PER_INST, kFrAx>(p, inst)) * xsk;
        const double cn = xt2 * xck - xcm, sn = xt2 * xsk - xsm;
        xcm = xck;
        xck = cn;
        xsm = xsk;
        xsk = sn;
      }
      double cm = cb, ck = 1.0, sm = -sb, sk = 0.0;  // cos/sin(ky b y), advanced in the loop
#pragma unroll 2
      for (int ky = 0; ky < NB; ky++)
      {
        double rx0 = 0.0, rx1 = 0.0, ry0 = 0.0, ry1 = 0.0;
        const double* srow = Ssm + ky * Cfg::kSPitch + kb;
#pragma unroll
        for (int j = 0; j < KB; j += 2)
        {
          const double2 s2 = *reinterpret_cast<const double2*>(srow + j);
          rx0 = fma(s2.x, asx[j], rx0);
          rx1 = fma(s2.y, asx[j + 1], rx1);
          ry0 = fma(s2.x, cx[j], ry0);
          ry1 = fma(s2.y, cx[j + 1], ry1);
        }
        ex = fma(ck, rx0 + rx1, ex);
        ey = fma(((double)ky * frame<PER_INST, kFrBy>(p, inst)) * sk, ry0 + ry1, ey);
        const double cn = yt2 * ck - cm, sn = yt2 * sk - sm;
        cm = ck;
        ck = cn;
        sm = sk;
        sk = sn;
      }
    }
    // dF/dx = -a sin(a x) cos(b y), dF/dy = -b cos(a x) sin(b y); times expl_weight (:433)
    ex = -ex * p.w;
    ey = -ey * p.w;
    if (rounds - 1 - r < 2) EB_PHASE(7 + 2 * (rounds - 1 - r));
#ifdef EB_DEBUG_DUMP
    if (inst == 0 && i < 4096)
    {
      double* d = g_dbg + i * 16;
      d[0] = ex; d[1] = ey; d[2] = ca; d[3] = sa; d[4] = cb; d[5] = sb; d[6] = ce; d[7] = se; d[8] = xf; d[9] = yf;
      d[10] = Ssm[lane % (NB * NB)];
    }
#endif

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
    if (rounds - 1 - r < 2) EB_PHASE(8 + 2 * (rounds - 1 - r));
  }
  EB_PHASE(11);
#ifdef EB_PHASE_TIMING
  if (lane == 0 && inst < 65536)
  {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    g_phase[inst * kPhaseSlots + 15] = smid;
  }
#endif
}

// Fourier-frame cosines of stored states [first, first + n) x B: what the solve kernels need from the replay buffer
// (ergodic_control.hpp:243-244 + basis.cpp:85 at k = 1; the higher orders follow by recurrence).  Same arithmetic as the
// kernels' own path, so cached and uncached runs agree bit for bit.
__global__ void __launch_bounds__(256) hist_cos_kernel(const double* __restrict__ hist, double* __restrict__ out, long long n,
                                                       double xmin, double ymin, double inv_lx, double inv_ly)
{
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const double xf = hist[3 * e + 0] - xmin, yf = hist[3 * e + 1] - ymin;
  out[2 * e + 0] = fast_cospi(xf * inv_lx);
  out[2 * e + 1] = fast_cospi(yf * inv_ly);
}
// addStateMemory with the cache up to date: the new row and its cosines in one launch (instead of a copy + a launch).
// frames: per-instance targets, each row's cosines in its instance's frame (the scalar frame is ignored)
__global__ void __launch_bounds__(256) add_state_kernel(const double* __restrict__ x, double* __restrict__ hist_row,
                                                        double* __restrict__ cos_row, int B, double xmin, double ymin,
                                                        double inv_lx, double inv_ly, const double* __restrict__ frames)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const double a = x[3 * i + 0], b = x[3 * i + 1], c = x[3 * i + 2];
  hist_row[3 * i + 0] = a;
  hist_row[3 * i + 1] = b;
  hist_row[3 * i + 2] = c;
  if (frames)
  {
    const double* f = frames + (size_t)i * kFrDoubles;
    xmin = f[kFrXmin];
    ymin = f[kFrYmin];
    inv_lx = f[kFrInvLx];
    inv_ly = f[kFrInvLy];
  }
  const double xf = a - xmin, yf = b - ymin;
  cos_row[2 * i + 0] = fast_cospi(xf * inv_lx);
  cos_row[2 * i + 1] = fast_cospi(yf * inv_ly);
}

// optTraj() (ergodic_control.hpp:314-317): forward rollout of the CURRENT
// control signal from the last pose, map frame, heading wrapped per step.
template <int MODEL>
__global__ void __launch_bounds__(128) rollout_kernel(int B, int N, double dt, const double* __restrict__ pose,
                                                      const double* __restrict__ ut, double* __restrict__ xt,
                                                      int* fault)
{
  const int lane = threadIdx.x & 31;
  const int inst = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (inst >= B) return;
  const double* u = ut + (size_t)inst * N * 3;
  double* out = xt + (size_t)inst * N * 3;
  RolloutCarry cy;
  cy.x = pose[(size_t)inst * 3 + 0];
  cy.y = pose[(size_t)inst * 3 + 1];
  cy.th = pose[(size_t)inst * 3 + 2];
  fast_sincos(cy.th, &cy.sth, &cy.cth);
  for (int base = 0; base < N; base += 32)
  {
    const int i = base + lane;
    const bool valid = i < N;
    double u0 = 0.0, u1 = 0.0, u2 = 0.0;
    if (valid)
    {
      u0 = u[i * 3 + 0];
      u1 = u[i * 3 + 1];
      u2 = u[i * 3 + 2];
    }
    if (MODEL == kModelSimpleCart && !(fabs(u1 - 0.0) < 1.0e-12)) atomicOr(fault, 1);
    double xo, yo, tho, ce, se;
    rollout_round<MODEL>(dt, valid, lane, u0, u1, u2, cy, xo, yo, tho, ce, se);
    if (valid)
    {
      out[i * 3 + 0] = xo;
      out[i * 3 + 1] = yo;
      out[i * 3 + 2] = normalize_angle_pi(tho);
    }
  }
}
}  // namespace eb
