// phik_tma.cuh -- phi_raw = C_y^T Phi C_x with the density staged through shared memory by 2-D TMA tiles and
// contracted on the FP64 tensor cores (sm_100a).
//
// Replaces the hot loop of Basis::spatialCoeff (basis.cpp:122-133) for large dense densities (config C3: 8192 x 8192
// grid, 32 x 32 basis).  Algorithmic work: 8 nx ny bytes (Phi read once), 2 nx ny nb + 2 ny nb^2 flops.
// Round 1 streamed Phi through a register double buffer (LDG.256, 64 KB in flight per SM, 0.63 of the measured HBM
// bandwidth, spilling); here the copy engine does the streaming:
//  * a producer warp issues cp.async.bulk.tensor.2d (SASS UTMALDG) boxes of 64 rows x 16 doubles (128 bytes per
//    row, CU_TENSOR_MAP_SWIZZLE_128B) into a ring of kStages stages with full / empty mbarriers; a stage holds 64
//    rows x 32 column PAIRS with the mirror fold (two boxes from the left half of the rows, two from the mirrored
//    right half) or 64 rows x 64 columns without it -- 32 KB of Phi per stage, up to 128 KB in flight per SM --
//    plus the matching chunk of the C_x table (cp.async.bulk, UBLKCP) on the same barrier;
//  * 16 consumer warps: warp w owns 16 rows (two row groups) and a quarter of the stage's columns.  A fragments
//    come from the swizzled boxes with conflict-free LDS.128 (DMMA row g <-> box row rho(g) = (g >> 1) | ((g & 1) << 2),
//    so the two rows of a quarter-warp land in different 64-byte halves), B fragments from the C_x chunk (pitch
//    36, rows ordered so that the four contraction indices of a k-step are consecutive), each B fragment feeding
//    both row groups.  No Phi value ever sits in a register across iterations: nothing spills.
//  * band end: the column quarters' tiles are summed in shared memory in a fixed order and folded with C_y
//    (16 DMMAs per warp), exactly as in the round-1 kernel; per-CTA partials, deterministic final sum.
// Mirror fold (FOLD): as in phik_dmma.cuh -- on the configTarget grid cos(k pi x_{nx-1-j} / lx) = (-1)^k cos(k pi x_j / lx),
// so even orders see Phi[j] + Phi[nx-1-j] and odd orders the difference: half the DMMAs, HBM-bound at nb = 32.
#pragma once

#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "phik_dmma.cuh"

namespace eb
{
constexpr int kPtRows = 64;        // rows per band
constexpr int kPtBox = 16;         // doubles per box row: 128 bytes, the span of SWIZZLE_128B
constexpr int kPtWarps = 16;       // consumer warps: 4 row blocks of 16 rows x 4 column quarters
constexpr int kPtThreads = (kPtWarps + 1) * 32;
constexpr int kPtBoxBytes = kPtRows * kPtBox * 8;  // 8 KB
constexpr int kPtTPitch = 33;

// U8: the density is a byte -> double table lookup of an occupancy grid (map_target.cuh); the stage then holds the
// BYTES of the 64 x 32 left cells and of their 64 x 32 mirrors (two boxes of 2 KB, no swizzle) and the consumers look
// the values up in a 256-entry table in shared memory -- the 8 B / cell density never exists in HBM.
constexpr int kPtU8BoxBytes = kPtRows * 32;  // 64 rows x 32 one-byte cells

template <bool FOLD, bool U8 = false>
struct PtGeom
{
  static_assert(!U8 || FOLD, "the byte-source kernel is the folded one");
  static constexpr int kCols = FOLD ? 32 : 64;             // contraction columns (pairs with the fold) per stage
  static constexpr int kBoxes = 4;                         // FOLD: 2 left + 2 mirrored; else 4 consecutive
  static constexpr int kPhiBytes = U8 ? 2 * kPtU8BoxBytes : kBoxes * kPtBoxBytes;  // 4 KB | 32 KB
  static constexpr int kCxBytes = kCols * kPdPitch * 8;    // 9 / 18 KB
  static constexpr int kStageBytes = kPhiBytes + ((kCxBytes + 1023) / 1024) * 1024;
  static constexpr int kStages = U8 ? 6 : (FOLD ? 4 : 3);
  static constexpr int kKSteps = kCols / 16;               // k-steps per warp and stage (a quarter of the columns, 4 per step)
  static constexpr int kLutBytes = U8 ? 256 * 8 : 0;
  static constexpr int kSmemBytes =
      kStages * kStageBytes + kPtRows * kPtTPitch * 8 + 256 + kLutBytes + 1024;  // + barriers + table + alignment slack
};

inline bool phik_tma_supported(int nx, int ny) { return nx % 2 == 0 && nx >= 64 && ny >= 1; }

// C_x table re-laid for this kernel: rows padded to the stage width, pitch 36, and within every group of 8 contraction
// columns column (2 q + s) is stored at row (4 s + q): the four lanes q of k-step s read consecutive rows (72 words
// apart -> 8 banks apart, conflict-free with the 8 consecutive orders of a fragment).
// fold: only the left nx / 2 columns, orders re-ordered as [0, 2, .., 30 | 1, 3, .., 31].
__global__ void phik_tma_permute_cx(const double* __restrict__ cx, int ncols, int rows_padded, int fold,
                                    double* __restrict__ out)
{
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows_padded * kPdPitch) return;
  const int row = idx / kPdPitch, k = idx % kPdPitch;
  const int grp = row >> 3, w = row & 7, s = w >> 2, q = w & 3;
  const int j = 8 * grp + 2 * q + s;  // the contraction column stored at this row
  const int order = fold ? (k < 16 ? 2 * k : 2 * (k - 16) + 1) : k;
  out[idx] = (j < ncols && k < 32) ? cx[(size_t)j * 32 + order] : 0.0;
}

__device__ __forceinline__ void tma_tile_g2s(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar)
{
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
constexpr int kPtGroup = 13;       // CTAs per first-level group of the fused final sum
constexpr int kPtMaxGroups = 63;   // counters: 1 + kPtMaxGroups
__device__ __forceinline__ void pt_consumer_barrier()
{
  asm volatile("bar.sync 1, %0;" ::"n"(kPtWarps * 32) : "memory");
}

struct PhikTmaParams
{
  const double* cxp;   // permuted C_x, [nchunks * kCols][36]
  const double* cy;    // C_y, [ny][32]
  double* parts;       // [gridDim.x + groups][1024]: per-CTA blocks, then the per-group sums
  int nx, ny;
  int nchunks;         // stages per band
  long long total;     // bands * nchunks
  // fused final reduction: the last CTA to finish sums the per-CTA partials in index order (deterministic),
  // undoes the fold's order permutation and normalises by raw[0][0] = sum(Phi)
  unsigned int* done;  // arrival counters, zero between launches: [0] groups finished, [1 + g] CTAs of group g finished
  int nb, fold;
  double *phik, *phi_sum, *raw;  // any may be null
  // Row-sharded grids on several GPUs (SURVEY.md section 8e): the all-reduce of the ranks' raw 32 x 32 blocks is part
  // of THIS kernel.  The last CTA stores its block into every rank's receive buffer over NVLink peer memory (slot =
  // this rank), raises this rank's flag on every peer after a system-scope fence, waits for the other ranks' flags
  // and sums the slots in rank order -- identical bits on every rank, no NCCL call, no second launch.  Two receive
  // buffers alternate by step: a rank can start step s + 2 only after every peer has finished step s + 1, i.e. is
  // past its reads of step s.
  int n_peer;                                  // 0: single GPU
  double* peer_recv[8];                        // rank q's receive buffer of this step's parity, offset to this rank's slot
  unsigned long long* peer_flag[8];            // this rank's slot in rank q's arrival flags
  const unsigned long long* my_flags;          // [n_peer]
  const double* my_recv;                       // this rank's receive buffer of this step's parity, [n_peer][1024]
  unsigned long long step;                     // 1-based step number = flag value
  unsigned long long* trace;                   // EB_PT_TRACE builds: [gridDim.x][8] globaltimer stamps, else null
  const double* lut;                           // U8 kernels: density value of every byte, [256]
};

#ifdef EB_PT_TRACE
__device__ __forceinline__ void pt_stamp(const PhikTmaParams& p, int slot)
{
  if (threadIdx.x == 0 && p.trace)
  {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    p.trace[blockIdx.x * 8 + slot] = t;
  }
}
#define PT_STAMP(slot) pt_stamp(p, slot)
#else
#define PT_STAMP(slot)
#endif

template <bool FOLD, bool U8 = false>
__global__ void __launch_bounds__(kPtThreads, 1)
    phik_tma_kernel(const __grid_constant__ CUtensorMap tmap, const PhikTmaParams p)
{
  using G = PtGeom<FOLD, U8>;
  extern __shared__ unsigned char smem_dyn[];
  // SWIZZLE_128B destinations must be 1024-byte aligned
  unsigned char* const base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  double* const tstage = reinterpret_cast<double*>(base + G::kStages * G::kStageBytes);  // [64][33]
  uint64_t* const full = reinterpret_cast<uint64_t*>(base + G::kStages * G::kStageBytes + kPtRows * kPtTPitch * 8);
  uint64_t* const empty = full + G::kStages;
  double* const lut = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(full) + 256);  // U8 only

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  PT_STAMP(0);
  if (threadIdx.x == 0)
  {
    for (int s = 0; s < G::kStages; s++)
    {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], kPtWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // this CTA's contiguous range of (band, chunk) iterations, band-major
  const long long it_lo = p.total * (long long)blockIdx.x / (long long)gridDim.x;
  const long long it_hi = p.total * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
  const int total_it = (int)(it_hi - it_lo);

  if (warp == kPtWarps)
  {
    // ===== producer warp: one elected lane feeds the ring =====
    if (lane == 0)
    {
      int band = (int)(it_lo / p.nchunks), k = (int)(it_lo - (long long)band * p.nchunks);
      for (int it = 0; it < total_it; it++)
      {
        const int s = it % G::kStages;
        if (it >= G::kStages) mbar_wait(&empty[s], ((it / G::kStages) - 1) & 1);
        unsigned char* const st = base + s * G::kStageBytes;
        mbar_expect_tx(&full[s], G::kPhiBytes + G::kCxBytes);
        const int row0 = band * kPtRows, col0 = k * G::kCols;
        if (U8)
        {
          // cells col0 .. col0 + 31 and their mirrors nx - col0 - 32 .. nx - col0 - 1 (ascending: pair p <-> byte 31 - p)
          tma_tile_g2s(st, &tmap, col0, row0, &full[s]);
          tma_tile_g2s(st + kPtU8BoxBytes, &tmap, p.nx - col0 - 32, row0, &full[s]);
        }
        else if (FOLD)
        {
          // pairs col0 .. col0 + 31: left columns ascending, and their mirrors nx-1-c as two ascending boxes
          tma_tile_g2s(st + 0 * kPtBoxBytes, &tmap, col0, row0, &full[s]);
          tma_tile_g2s(st + 1 * kPtBoxBytes, &tmap, col0 + kPtBox, row0, &full[s]);
          tma_tile_g2s(st + 2 * kPtBoxBytes, &tmap, p.nx - col0 - kPtBox, row0, &full[s]);      // mirrors of box 0
          tma_tile_g2s(st + 3 * kPtBoxBytes, &tmap, p.nx - col0 - 2 * kPtBox, row0, &full[s]);  // mirrors of box 1
        }
        else
        {
#pragma unroll
          for (int b = 0; b < 4; b++) tma_tile_g2s(st + b * kPtBoxBytes, &tmap, col0 + b * kPtBox, row0, &full[s]);
        }
        tma_bulk_g2s(st + G::kPhiBytes, p.cxp + (size_t)k * G::kCols * kPdPitch, G::kCxBytes, &full[s]);
        if (++k == p.nchunks)
        {
          k = 0;
          band++;
        }
      }
    }
    return;
  }

  // ===== consumer warps =====
  const int g = lane >> 2, q = lane & 3;
  const int rb = warp & 3, cq = warp >> 2;  // 16-row block, column quarter
  const int rho = (g >> 1) | ((g & 1) << 2);  // box row (within a group of 8) that feeds DMMA row g

  if (U8)
  {
    if (threadIdx.x < 256) lut[threadIdx.x] = __ldg(p.lut + threadIdx.x);
    pt_consumer_barrier();
  }

  const bool hi_orders = p.nb > 16;  // orders 16 .. 31 (order tiles 1, 3 with the fold; 2, 3 without) are wanted
  double P[2] = { 0.0, 0.0 };  // this warp's 8x8 tile of the CTA's 32x32 partial
  double T[2][4][2];           // [row group][order tile][2]
#pragma unroll
  for (int r = 0; r < 2; r++)
#pragma unroll
    for (int t = 0; t < 4; t++) T[r][t][0] = T[r][t][1] = 0.0;

  int band = (int)(it_lo / p.nchunks), k = (int)(it_lo - (long long)band * p.nchunks);
  for (int it = 0; it < total_it; it++)
  {
    const int s = it % G::kStages;
    mbar_wait(&full[s], (it / G::kStages) & 1);
#ifdef EB_PT_TRACE
    if (it == 0) PT_STAMP(1);
    if (it + 1 == total_it) PT_STAMP(2);
#endif
    const unsigned char* const st = base + s * G::kStageBytes;
    const double* const cxs = reinterpret_cast<const double*>(st + G::kPhiBytes);
    if (FOLD)
    {
      // quarter cq = pairs 8 cq .. 8 cq + 7: box cq >> 1, 16-byte chunks 4 (cq & 1) + q (columns 2q, 2q + 1 of the
      // quarter); the mirrors sit in box 2 + (cq >> 1) at chunk 7 - 4 (cq & 1) - q with the two columns swapped
      const int bx = cq >> 1, ch = 4 * (cq & 1) + q;
      double ev[2][2], od[2][2];  // [row group][k-step]
#pragma unroll
      for (int r = 0; r < 2; r++)
      {
        const int row = 16 * rb + 8 * r + rho;
        double2 lo, hi;
        if (U8)
        {
          // pairs 8 cq + 2 q, + 1: two bytes of the left box; their mirrors are bytes 31 - p of the mirror box
          const int p0 = 8 * cq + 2 * q;
          const unsigned int wl = *reinterpret_cast<const unsigned short*>(st + row * 32 + p0);
          const unsigned int wh = *reinterpret_cast<const unsigned short*>(st + kPtU8BoxBytes + row * 32 + 30 - p0);
          lo = make_double2(lut[wl & 255u], lut[wl >> 8]);
          hi = make_double2(lut[wh & 255u], lut[wh >> 8]);
        }
        else
        {
          lo = *reinterpret_cast<const double2*>(st + bx * kPtBoxBytes + row * 128 + ((ch ^ rho) << 4));
          hi = *reinterpret_cast<const double2*>(st + (2 + bx) * kPtBoxBytes + row * 128 + (((7 - ch) ^ rho) << 4));
        }
        ev[r][0] = lo.x + hi.y;
        od[r][0] = lo.x - hi.y;
        ev[r][1] = lo.y + hi.x;
        od[r][1] = lo.y - hi.x;
      }
#pragma unroll
      for (int ks = 0; ks < 2; ks++)
      {
        const double* brow = cxs + (8 * cq + 4 * ks + q) * kPdPitch + g;
        const double b0 = brow[0], b2 = brow[16];
#pragma unroll
        for (int r = 0; r < 2; r++)
        {
          dmma884(T[r][0][0], T[r][0][1], ev[r][ks], b0);  // orders 0, 2, .., 14
          dmma884(T[r][2][0], T[r][2][1], od[r][ks], b2);  // orders 1, 3, .., 15
        }
        if (hi_orders)  // nb <= 16 never reads orders 16 .. 31: half the DMMAs
        {
          const double b1 = brow[8], b3 = brow[24];
#pragma unroll
          for (int r = 0; r < 2; r++)
          {
            dmma884(T[r][1][0], T[r][1][1], ev[r][ks], b1);  // orders 16, .., 30
            dmma884(T[r][3][0], T[r][3][1], od[r][ks], b3);  // orders 17, .., 31
          }
        }
      }
    }
    else
    {
      // quarter cq = columns 16 cq .. 16 cq + 15 = box cq; chunks q and 4 + q -> k-steps (0, 1) and (2, 3)
      double av[2][4];
#pragma unroll
      for (int r = 0; r < 2; r++)
      {
        const int row = 16 * rb + 8 * r + rho;
        const double2 v0 = *reinterpret_cast<const double2*>(st + cq * kPtBoxBytes + row * 128 + ((q ^ rho) << 4));
        const double2 v1 = *reinterpret_cast<const double2*>(st + cq * kPtBoxBytes + row * 128 + (((4 + q) ^ rho) << 4));
        av[r][0] = v0.x;
        av[r][1] = v0.y;
        av[r][2] = v1.x;
        av[r][3] = v1.y;
      }
#pragma unroll
      for (int ks = 0; ks < 4; ks++)
      {
        const double* brow = cxs + (16 * cq + 4 * ks + q) * kPdPitch + g;
        const double b0 = brow[0], b1 = brow[8];
#pragma unroll
        for (int r = 0; r < 2; r++)
        {
          dmma884(T[r][0][0], T[r][0][1], av[r][ks], b0);
          dmma884(T[r][1][0], T[r][1][1], av[r][ks], b1);
        }
        if (hi_orders)
        {
          const double b2 = brow[16], b3 = brow[24];
#pragma unroll
          for (int r = 0; r < 2; r++)
          {
            dmma884(T[r][2][0], T[r][2][1], av[r][ks], b2);
            dmma884(T[r][3][0], T[r][3][1], av[r][ks], b3);
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);  // this warp is done with the stage

    const bool last = it + 1 == total_it;
    if (++k == p.nchunks || last)
    {
      // End of the band (or of this CTA's range): sum the four column quarters' tiles in the stage, fixed order
      // (C layout: DMMA row g <-> band row 16 rb + 8 r + rho, cols 8 t + 2 q + e), then fold with C_y.
      k = 0;
      // warp w owns output tile (m, t) = (w / 4, w % 4) of the fold with C_y below; its C_y operands are fetched now so
      // that their L2 latency hides behind the four turns (the last band end of a CTA is on the kernel's critical path)
      const int m = warp >> 2, t = warp & 3;
      const int r0 = band * kPtRows;
      double cya[kPtRows / 4];
#pragma unroll
      for (int h = 0; h < kPtRows / 4; h++)
      {
        const int r = r0 + 4 * h + q;
        cya[h] = r < p.ny ? __ldg(p.cy + (size_t)r * 32 + 8 * m + g) : 0.0;
      }
#pragma unroll 1
      for (int turn = 0; turn < 4; turn++)
      {
        if (cq == turn)
        {
#pragma unroll
          for (int r = 0; r < 2; r++)
          {
            double* trow = tstage + (16 * rb + 8 * r + rho) * kPtTPitch + 2 * q;
#pragma unroll
            for (int t_ = 0; t_ < 4; t_++)
            {
              if (turn == 0)
              {
                trow[8 * t_ + 0] = T[r][t_][0];
                trow[8 * t_ + 1] = T[r][t_][1];
              }
              else
              {
                trow[8 * t_ + 0] += T[r][t_][0];
                trow[8 * t_ + 1] += T[r][t_][1];
              }
              T[r][t_][0] = T[r][t_][1] = 0.0;
            }
          }
        }
        pt_consumer_barrier();
      }
      // P[8m + g][8t + 2q + e] += sum_rows C_y[row][8m + g] T[row][8t + ..]
#pragma unroll
      for (int h = 0; h < kPtRows / 4; h++)
      {
        const double b = tstage[(4 * h + q) * kPtTPitch + 8 * t + g];
        dmma884(P[0], P[1], cya[h], b);
      }
      band++;
      pt_consumer_barrier();  // the T stage may be overwritten by the next band
    }
  }

  PT_STAMP(3);
  {
    // with the fold the partial's columns are in [even orders | odd orders] order; the final sum undoes it
    const int m = warp >> 2, t = warp & 3;
    double* out = p.parts + (size_t)blockIdx.x * 1024 + (8 * m + g) * 32 + 8 * t + 2 * q;
    out[0] = P[0];
    out[1] = P[1];
  }
  // ---- final sum over the partials, fused (what phik_finalize did as a second launch) ----
  // One SM summing every CTA's block is a serial tail of ~10 us (1.2 MB through one SM, 19 dependent rounds of L2
  // latency), so the sum has two levels: the last CTA to finish in each group of kPtGroup sums that group's blocks in
  // index order, and the last group to finish sums the group blocks in group order.  Who does the work depends on
  // timing, the ORDER of the additions does not: the result is deterministic.
  __shared__ unsigned int s_last;
  __shared__ double s_total;
  const int nparts = (int)gridDim.x;
  const int ngroups = (nparts + kPtGroup - 1) / kPtGroup;
  const int grp = (int)blockIdx.x / kPtGroup, g_lo = grp * kPtGroup, g_n = min(kPtGroup, nparts - g_lo);
  __threadfence();
  pt_consumer_barrier();
  if (threadIdx.x == 0) s_last = atomicAdd(p.done + 1 + grp, 1u) == (unsigned)(g_n - 1) ? 1u : 0u;
  pt_consumer_barrier();
  PT_STAMP(4);
  if (!s_last) return;
  __threadfence();  // the other CTAs' partials, released before their counter increments
  double sum2[2] = { 0.0, 0.0 };
  // 2 * kPtGroup loads per thread in flight (the partials sit in L2: the sum is latency-bound); 148 CTAs = 12 groups of
  // 13: one round of L2 latency per level
  auto sum_blocks = [&](const double* src, int n) {
    sum2[0] = sum2[1] = 0.0;
    for (int p0 = 0; p0 < n; p0 += kPtGroup)
    {
      double v[2][kPtGroup];
#pragma unroll
      for (int j = 0; j < kPtGroup; j++)
#pragma unroll
        for (int h = 0; h < 2; h++)
          v[h][j] = p0 + j < n ? __ldcg(src + (size_t)(p0 + j) * 1024 + threadIdx.x + h * (kPtWarps * 32)) : 0.0;
#pragma unroll
      for (int j = 0; j < kPtGroup; j++)
      {
        sum2[0] += v[0][j];
        sum2[1] += v[1][j];
      }
    }
  };
  sum_blocks(p.parts + (size_t)g_lo * 1024, g_n);
  if (ngroups > 1)
  {
    double* gout = p.parts + (size_t)(nparts + grp) * 1024;
    gout[threadIdx.x] = sum2[0];
    gout[threadIdx.x + kPtWarps * 32] = sum2[1];
    __threadfence();
    pt_consumer_barrier();
    if (threadIdx.x == 0) s_last = atomicAdd(p.done, 1u) == (unsigned)(ngroups - 1) ? 1u : 0u;
    pt_consumer_barrier();
    PT_STAMP(5);
    if (!s_last) return;
    __threadfence();
    sum_blocks(p.parts + (size_t)nparts * 1024, ngroups);
    PT_STAMP(6);
  }
  if (p.n_peer > 1)
  {
    // ---- fused all-reduce over NVLink peer memory ----
#pragma unroll
    for (int h = 0; h < 2; h++)
    {
      const int t = threadIdx.x + h * (kPtWarps * 32);
#pragma unroll
      for (int q_ = 0; q_ < 8; q_++)
        if (q_ < p.n_peer) p.peer_recv[q_][t] = sum2[h];  // slots keep the kernel's column order; every rank folds alike
    }
    __threadfence_system();
    pt_consumer_barrier();
    if (threadIdx.x < p.n_peer) *(volatile unsigned long long*)p.peer_flag[threadIdx.x] = p.step;
    if (threadIdx.x < p.n_peer)
      while (*(const volatile unsigned long long*)(p.my_flags + threadIdx.x) < p.step) __nanosleep(64);
    pt_consumer_barrier();
    __threadfence_system();
#pragma unroll
    for (int h = 0; h < 2; h++)
    {
      const int t = threadIdx.x + h * (kPtWarps * 32);
      double acc = 0.0;
      for (int r = 0; r < p.n_peer; r++) acc += *(const volatile double*)(p.my_recv + (size_t)r * 1024 + t);  // rank order
      sum2[h] = acc;
    }
  }
  if (threadIdx.x == 0) s_total = sum2[0];  // order (0, 0) sits at column 0 with or without the fold
  pt_consumer_barrier();
#pragma unroll
  for (int h = 0; h < 2; h++)
  {
    const int t = threadIdx.x + h * (kPtWarps * 32);
    const int ky = t >> 5, col = t & 31;
    const int kx = p.fold ? (col < 16 ? 2 * col : 2 * (col - 16) + 1) : col;
    if (p.raw) p.raw[ky * 32 + kx] = (ky < p.nb && kx < p.nb) ? sum2[h] : 0.0;
    if (p.phik && ky < p.nb && kx < p.nb) p.phik[ky * p.nb + kx] = sum2[h] / s_total;
  }
  if (threadIdx.x == 0 && p.phi_sum) *p.phi_sum = s_total;
  if (threadIdx.x <= ngroups) p.done[threadIdx.x] = 0u;  // every counter is complete by now: ready for the next launch
  PT_STAMP(7);
}

// ---- host side -------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_eb_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                       const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                       CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_eb_encodeTiled phik_tma_encoder()
{
  static PFN_eb_encodeTiled fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
    {
      cudaGetLastError();
      p = nullptr;
    }
    return reinterpret_cast<PFN_eb_encodeTiled>(p);
  }();
  return fn;
}

// tensor map of a dense row-major [ny][nx] f64 density: boxes of 64 rows x 16 columns, 128-byte swizzle, zero fill outside
inline bool phik_tma_make_map(const double* phi, int nx, int ny, CUtensorMap* map)
{
  PFN_eb_encodeTiled enc = phik_tma_encoder();
  if (!enc) return false;
  const cuuint64_t dims[2] = { (cuuint64_t)nx, (cuuint64_t)ny };
  const cuuint64_t strides[1] = { (cuuint64_t)nx * 8 };
  const cuuint32_t box[2] = { (cuuint32_t)kPtBox, (cuuint32_t)kPtRows };
  const cuuint32_t estr[2] = { 1, 1 };
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(phi), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// tensor map of a row-major [ny][nx] occupancy grid (one byte per cell): boxes of 64 rows x 32 cells, no swizzle, zero
// fill outside (rows past the grid carry zero C_y weight, columns past nx / 2 zero C_x rows: whatever the table holds
// for byte 0 never reaches the result)
inline bool phik_tma_u8_supported(int nx, int ny) { return nx % 16 == 0 && nx >= 64 && ny >= 1; }
inline bool phik_tma_make_map_u8(const signed char* cells, int nx, int ny, CUtensorMap* map)
{
  PFN_eb_encodeTiled enc = phik_tma_encoder();
  if (!enc) return false;
  const cuuint64_t dims[2] = { (cuuint64_t)nx, (cuuint64_t)ny };
  const cuuint64_t strides[1] = { (cuuint64_t)nx };
  const cuuint32_t box[2] = { 32u, (cuuint32_t)kPtRows };
  const cuuint32_t estr[2] = { 1, 1 };
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<signed char*>(cells), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Launches one persistent CTA per SM (fewer when there is less work than that); returns the number of partial
// blocks written (= grid size) or -1 on failure (no encoder, misaligned density, launch error).
struct PhikTmaPeer
{
  int n_peer = 0;
  double* peer_recv[8] = {};
  unsigned long long* peer_flag[8] = {};
  const unsigned long long* my_flags = nullptr;
  const double* my_recv = nullptr;
  unsigned long long step = 0;
};

struct PhikTmaOut
{
  unsigned int* done;
  int nb;
  double *phik, *phi_sum, *raw;
  const PhikTmaPeer* peer = nullptr;
};

template <bool FOLD, bool U8 = false>
inline int phik_tma_launch_t(const void* src, const double* lut, int nx, int ny, const double* cxp, const double* cy,
                             double* parts, int max_parts, const PhikTmaOut& out, cudaStream_t stream)
{
  using G = PtGeom<FOLD, U8>;
  if ((reinterpret_cast<uintptr_t>(src) & 15) != 0) return -1;
  CUtensorMap map;
  if (U8 ? !phik_tma_make_map_u8(static_cast<const signed char*>(src), nx, ny, &map) :
           !phik_tma_make_map(static_cast<const double*>(src), nx, ny, &map))
    return -1;
  PhikTmaParams p{};
  p.lut = lut;
  p.cxp = cxp;
  p.cy = cy;
  p.parts = parts;
  p.nx = nx;
  p.ny = ny;
  p.done = out.done;
  p.nb = out.nb;
  p.fold = FOLD ? 1 : 0;
  p.phik = out.phik;
  p.phi_sum = out.phi_sum;
  p.raw = out.raw;
  if (out.peer && out.peer->n_peer > 1)
  {
    p.n_peer = out.peer->n_peer;
    for (int q = 0; q < p.n_peer; q++)
    {
      p.peer_recv[q] = out.peer->peer_recv[q];
      p.peer_flag[q] = out.peer->peer_flag[q];
    }
    p.my_flags = out.peer->my_flags;
    p.my_recv = out.peer->my_recv;
    p.step = out.peer->step;
  }
  const int ncols = FOLD ? nx / 2 : nx;
  p.nchunks = (ncols + G::kCols - 1) / G::kCols;
  const int bands = (ny + kPtRows - 1) / kPtRows;
  p.total = (long long)bands * p.nchunks;
  const int grid = (int)std::min<long long>(p.total, max_parts);
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63])
  {
    if (cudaFuncSetAttribute(phik_tma_kernel<FOLD, U8>, cudaFuncAttributeMaxDynamicSharedMemorySize, G::kSmemBytes) !=
        cudaSuccess)
      return -1;
    configured[dev & 63] = true;
  }
#ifdef EB_PT_TRACE
  // debug build: per-CTA time line of every launch, summarised on stderr (synchronises; not for timing runs)
  static unsigned long long* d_trace = nullptr;
  if (!d_trace) cudaMalloc(&d_trace, sizeof(unsigned long long) * 8 * 1024);
  cudaMemsetAsync(d_trace, 0, sizeof(unsigned long long) * 8 * 1024, stream);
  p.trace = d_trace;
#endif
  phik_tma_kernel<FOLD, U8><<<grid, kPtThreads, G::kSmemBytes, stream>>>(map, p);
  if (cudaGetLastError() != cudaSuccess) return -1;
#ifdef EB_PT_TRACE
  {
    static unsigned long long h[8 * 1024];
    cudaStreamSynchronize(stream);
    cudaMemcpy(h, d_trace, sizeof(unsigned long long) * 8 * grid, cudaMemcpyDeviceToHost);
    unsigned long long t0 = ~0ull;
    for (int b = 0; b < grid; b++) t0 = std::min(t0, h[b * 8]);
    static const char* names[8] = { "entry", "first stage full", "last stage full", "loop done", "group counter", "top counter",
                                    "top sum done", "exit" };
    fprintf(stderr, "[phik trace] grid %d rows %d\n", grid, ny);
    for (int s = 0; s < 8; s++)
    {
      double lo = 1e30, hi = -1, sum = 0;
      int n = 0;
      for (int b = 0; b < grid; b++)
        if (h[b * 8 + s])
        {
          const double t = (double)(h[b * 8 + s] - t0) * 1e-3;
          lo = std::min(lo, t), hi = std::max(hi, t), sum += t, n++;
        }
      if (n) fprintf(stderr, "  %-18s n %3d  min %8.2f  mean %8.2f  max %8.2f us\n", names[s], n, lo, sum / n, hi);
    }
  }
#endif
  return grid;
}

inline int phik_tma_launch(const double* phi, int nx, int ny, const double* cxp, const double* cy, double* parts,
                           int max_parts, bool fold, const PhikTmaOut& out, cudaStream_t stream)
{
  return fold ? phik_tma_launch_t<true>(phi, nullptr, nx, ny, cxp, cy, parts, max_parts, out, stream) :
                phik_tma_launch_t<false>(phi, nullptr, nx, ny, cxp, cy, parts, max_parts, out, stream);
}

// the folded kernel over an occupancy grid: density = lut[cell byte], looked up in shared memory (map_target.cuh)
inline int phik_tma_launch_u8(const signed char* cells, const double* lut, int nx, int ny, const double* cxpf, const double* cy,
                              double* parts, int max_parts, const PhikTmaOut& out, cudaStream_t stream)
{
  return phik_tma_launch_t<true, true>(cells, lut, nx, ny, cxpf, cy, parts, max_parts, out, stream);
}

// rows of the permuted C_x table the kernel may touch (the last chunk is padded to the stage width)
inline int phik_tma_cx_rows(int ncols, bool fold)
{
  const int w = fold ? PtGeom<true>::kCols : PtGeom<false>::kCols;
  return ((ncols + w - 1) / w) * w;
}
}  // namespace eb
