// map_target_batch.cuh -- the map-derived (entropy) target of every instance of a per-instance controller, one launch
// (sm_100a, FP64 tensor cores).
//
// Instance i has its own occupancy map (ny_i x nx_i int8 cells, resolution res_i, origin o_i).  Its row of phi_k is
// what eb_map_target_create(nx_i, ny_i, res_i, nb) + eb_map_target_execute compute (map_target.cuh): the entropy
// density at the cell centres, contracted C_y^T Phi C_x and divided by raw[0] = sum(Phi).
//
// Work units = (instance, 64-row chunk of its map); how a map is cut depends only on its own geometry.  A persistent
// grid takes the units by static stride.  Per unit:
//  * every CTA tabulates the 256-entry entropy table in shared memory once (entropy_lut_kernel's expression, so the same
//    bits), which keeps the call at one launch;
//  * 64 x 64 cell tiles are converted through the table into a density tile in shared memory, and the cosine table of
//    the tile's columns is built with cos_table_kernel's expression on coordinates accumulated exactly as
//    accumulated_axis(n, res, res / 2) does (one thread carries the running sum) -- the single-map plan's bits;
//  * stage 1, T[64 rows][kx] += Phi C_x, and stage 2, raw[ky][kx] = C_y^T T, run as DMMA m8n8k4 tiles (dmma884);
//  * the unit's raw nb x nb block goes to a scratch slot of nb * nb doubles.
// The last unit of an instance to arrive (arrival counter, reset by it) sums the instance's slots in unit order (the
// result does not depend on which unit finished last, or on the other maps of the batch), divides by raw[0], writes
// the row and the frame record with target_batch_kernel's expressions, and re-derives the instance's replay cosines
// when its frame key moved.  num_basis > 32 loops over blocks of 32 orders, as elsewhere.
//
// KEPT (eb_set_map_targets_from_grid_batch): the slots are the controller's kept blocks, one region of consecutive
// units per instance that outlives the launch.  The work list holds only the units to recompute (MapKept: one non-empty
// run of consecutive units per listed map); the arrival count of an instance is the length of its run, and its last
// unit sums all of the instance's kept blocks in unit order.  A unit's block depends only on its cells and on nx, ny
// and res, so the row equals the one of a launch over every unit of the map, bit for bit.
#pragma once

#include "common.cuh"
#include "solve_kernel.cuh"

namespace eb
{
constexpr int kMbThreads = 256;          // 8 warps: warp w owns rows 8w..8w+7 of the unit in stage 1
constexpr int kMbRows = 64;              // map rows per work unit
constexpr int kMbCols = 64;              // columns per staged tile
constexpr int kMbPhiPitch = kMbCols + 4;  // density tile pitch: A-fragment loads hit distinct banks
constexpr int kMbTabPitch = 36;          // cosine-table / T pitch (as kPdPitch): B-fragment loads hit distinct banks
// dynamic shared memory: entropy table, density tile (aliased by T), C_x tile, C_y, coordinates
constexpr int kMbSmemDoubles = 256 + kMbRows * kMbPhiPitch + kMbCols * kMbTabPitch + kMbRows * kMbTabPitch + kMbCols + kMbRows;
constexpr size_t kMbSmemBytes = sizeof(double) * kMbSmemDoubles;

struct MapBatchDesc
{
  const signed char* cells;  // [ny][nx], GridMap layout
  int nx, ny;
  double res, ox, oy;        // resolution, origin (GridMap xmin / ymin)
  int inst;                  // controller instance
  int unit0;                 // first work unit of this map
};

// KEPT: map desc[j] recomputes units [first, first + count) of its map (work items [desc[j].unit0, + count)); its
// kept blocks are slots [slot0, slot0 + units of the map)
struct MapKept
{
  int first, count, slot0;
};

struct MapBatchParams
{
  const MapBatchDesc* desc;  // [n] maps to update, unit0 ascending
  int n, units, nb;
  double* slots;             // [units][nb * nb] raw blocks
  unsigned* arrive;          // [B] arrival counters, zero between launches
  double* frames;            // [B][kFrDoubles]
  double* phik;              // [B][nb * nb]
  const double* hist;        // [mem_count][B][3]
  double* hist_cos;          // [mem_count][B][2] or null
  long long mem_count;
  int B;
  const MapKept* kept;       // KEPT: [n] the recomputed units of each map and where its kept blocks live
};

__host__ __device__ inline int mb_units(int ny) { return (ny + kMbRows - 1) / kMbRows; }

// entropy_lut_kernel's expression (map_target.cuh) for byte pattern b
__device__ __forceinline__ double mb_entropy(int b)
{
  const int v = b < 128 ? b : b - 256;
  const double p = (double)v / 100.0;
  if (fabs(0.0 - p) < 1.0e-12 || fabs(1.0 - p) < 1.0e-12) return 1e-3;
  if (p < 0.0) return 0.7;
  return -p * log(p) - (1.0 - p) * log(1.0 - p);
}

template <bool KEPT>
__global__ void __launch_bounds__(kMbThreads, 3) map_target_batch_kernel(const MapBatchParams p)
{
  extern __shared__ __align__(16) double mb_smem[];
  double* const s_lut = mb_smem;
  double* const s_phi = s_lut + 256;                        // [64][kMbPhiPitch] density tile; T [64][36] after stage 1
  double* const s_cx = s_phi + kMbRows * kMbPhiPitch;       // [64 cols][36]
  double* const s_cy = s_cx + kMbCols * kMbTabPitch;        // [64 rows][36]
  double* const s_xs = s_cy + kMbRows * kMbTabPitch;        // [64] column coordinates of the tile
  double* const s_ys = s_xs + kMbCols;                      // [64] row coordinates of the unit
  double* const s_t = s_phi;
  __shared__ int s_last;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5, g = lane >> 2, q = lane & 3;
  const int nb = p.nb, K = nb * nb, nblk = (nb + 31) / 32;
  s_lut[t] = mb_entropy(t);

  for (int u = blockIdx.x; u < p.units; u += gridDim.x)
  {
    int lo = 0, hi = p.n - 1;  // the map whose units contain u
    while (lo < hi)
    {
      const int mid = (lo + hi + 1) >> 1;
      if (p.desc[mid].unit0 <= u) lo = mid;
      else hi = mid - 1;
    }
    const MapBatchDesc d = p.desc[lo];
    int mu = u - d.unit0, su = u;  // unit of the map, slot of the unit
    if constexpr (KEPT)
    {
      const MapKept k = p.kept[lo];
      mu += k.first;
      su = k.slot0 + mu;
    }
    const int r0 = mu * kMbRows, nrows = min(kMbRows, d.ny - r0), nx = d.nx;
    const double lx = (double)d.nx * d.res, ly = (double)d.ny * d.res;
    const double fx = kPi / lx, fy = kPi / ly;  // basis.cpp:85: cos(k * (PI / l) * x)
    double* const slot = p.slots + (size_t)su * K;
    __syncthreads();  // the previous unit's readers of s_ys / s_t are done
    if (t == 32)
    {
      double y = 0.5 * d.res;  // accumulated_axis(ny, res, res / 2) up to this unit's rows
      for (int r = 0; r < r0; r++) y += d.res;
      for (int r = 0; r < kMbRows; r++)
      {
        s_ys[r] = y;
        y += d.res;
      }
    }
    for (int bx = 0; bx < nblk; bx++)
    {
      const int ntx = min(4, (nb - 32 * bx + 7) >> 3);  // active 8-order tiles of this block
      double acc[4][2] = { { 0.0, 0.0 }, { 0.0, 0.0 }, { 0.0, 0.0 }, { 0.0, 0.0 } };  // T[8w + g][32 bx + 8 tt + 2q (+1)]
      double xc = 0.5 * d.res;  // thread 0: accumulated column coordinate
      for (int c0 = 0; c0 < nx; c0 += kMbCols)
      {
        __syncthreads();  // the previous tile's readers are done
        if (t == 0)
          for (int c = 0; c < kMbCols; c++)
          {
            s_xs[c] = xc;
            xc += d.res;
          }
        for (int e = t; e < kMbRows * kMbCols; e += kMbThreads)
        {
          const int r = e / kMbCols, c = e % kMbCols;
          double v = 0.0;
          if (r < nrows && c0 + c < nx)
            v = s_lut[(unsigned char)__ldg(d.cells + (size_t)(r0 + r) * nx + c0 + c)];
          s_phi[r * kMbPhiPitch + c] = v;
        }
        __syncthreads();
        for (int e = t; e < kMbCols * 32; e += kMbThreads)
        {
          const int c = e >> 5, k = 32 * bx + (e & 31);
          s_cx[c * kMbTabPitch + (e & 31)] = (k < nb && c0 + c < nx) ? cos((double)k * fx * s_xs[c]) : 0.0;
        }
        __syncthreads();
        if (8 * w < nrows)
        {
          const int jmax = min(kMbCols, (nx - c0 + 3) & ~3);
          const double* arow = s_phi + (8 * w + g) * kMbPhiPitch + q;
          for (int j0 = 0; j0 < jmax; j0 += 4)
          {
            const double a = arow[j0];
            const double* brow = s_cx + (j0 + q) * kMbTabPitch + g;
#pragma unroll
            for (int tt = 0; tt < 4; tt++)
              if (tt < ntx) dmma884(acc[tt][0], acc[tt][1], a, brow[8 * tt]);
          }
        }
      }
      __syncthreads();  // every warp is done with the density tile: T takes its place
#pragma unroll
      for (int tt = 0; tt < 4; tt++)
      {
        s_t[(8 * w + g) * kMbTabPitch + 8 * tt + 2 * q] = acc[tt][0];
        s_t[(8 * w + g) * kMbTabPitch + 8 * tt + 2 * q + 1] = acc[tt][1];
      }
      for (int by = 0; by < nblk; by++)
      {
        const int nty = min(4, (nb - 32 * by + 7) >> 3);
        __syncthreads();  // T is complete; the previous block's readers of s_cy are done
        for (int e = t; e < kMbRows * 32; e += kMbThreads)
        {
          const int r = e >> 5, k = 32 * by + (e & 31);
          s_cy[r * kMbTabPitch + (e & 31)] = (k < nb && r < nrows) ? cos((double)k * fy * s_ys[r]) : 0.0;
        }
        __syncthreads();
        const int imax = (nrows + 3) & ~3;
#pragma unroll
        for (int m = 0; m < 2; m++)
        {
          const int tile = w + 8 * m, ty = tile >> 2, tx = tile & 3;
          if (ty >= nty || tx >= ntx) continue;
          double d0 = 0.0, d1 = 0.0;  // raw[32 by + 8 ty + g][32 bx + 8 tx + 2q (+1)]
          for (int i0 = 0; i0 < imax; i0 += 4)
            dmma884(d0, d1, s_cy[(i0 + q) * kMbTabPitch + 8 * ty + g], s_t[(i0 + q) * kMbTabPitch + 8 * tx + g]);
          const int ky = 32 * by + 8 * ty + g, kx = 32 * bx + 8 * tx + 2 * q;
          if (ky < nb && kx < nb) slot[ky * nb + kx] = d0;
          if (ky < nb && kx + 1 < nb) slot[ky * nb + kx + 1] = d1;
        }
      }
    }

    // the last unit of this map to arrive finishes the instance
    const int nunits = mb_units(d.ny);
    int arrivals = nunits, s0 = d.unit0;
    if constexpr (KEPT)
    {
      arrivals = p.kept[lo].count;
      s0 = p.kept[lo].slot0;
    }
    __threadfence();
    __syncthreads();
    if (t == 0) s_last = atomicAdd(p.arrive + d.inst, 1u) == (unsigned)(arrivals - 1);
    __syncthreads();
    if (!s_last) continue;
    __threadfence();
    const double* base = p.slots + (size_t)s0 * K;
    double total = 0.0;  // raw[0] = sum(Phi), summed in unit order
    for (int v = 0; v < nunits; v++) total += __ldcg(base + (size_t)v * K);
    double* const row = p.phik + (size_t)d.inst * K;
    for (int e = t; e < K; e += kMbThreads)
    {
      double s = 0.0;
      for (int v = 0; v < nunits; v++) s += __ldcg(base + (size_t)v * K + e);
      row[e] = s / total;
    }
    double* const fr = p.frames + (size_t)d.inst * kFrDoubles;
    const double old_x = fr[kFrXmin], old_y = fr[kFrYmin], old_ilx = fr[kFrInvLx], old_ily = fr[kFrInvLy];
    const double ilx = 1.0 / lx, ily = 1.0 / ly;
    if (p.hist_cos && (__double_as_longlong(d.ox) != __double_as_longlong(old_x) ||
                       __double_as_longlong(d.oy) != __double_as_longlong(old_y) ||
                       __double_as_longlong(ilx) != __double_as_longlong(old_ilx) ||
                       __double_as_longlong(ily) != __double_as_longlong(old_ily)))
      for (long long r = t; r < p.mem_count; r += kMbThreads)
      {
        const size_t e = (size_t)r * p.B + d.inst;
        const double xf = p.hist[3 * e + 0] - d.ox, yf = p.hist[3 * e + 1] - d.oy;
        p.hist_cos[2 * e + 0] = fast_cospi(xf * ilx);
        p.hist_cos[2 * e + 1] = fast_cospi(yf * ily);
      }
    __syncthreads();  // every thread has read the old frame
    if (t == 0)
    {
      // target_batch_kernel's frame record
      fr[kFrXmin] = d.ox;
      fr[kFrYmin] = d.oy;
      fr[kFrLx] = lx;
      fr[kFrLy] = ly;
      fr[kFrInvLx] = ilx;
      fr[kFrInvLy] = ily;
      fr[kFrAx] = kPi / lx;
      fr[kFrBy] = kPi / ly;
      p.arrive[d.inst] = 0u;
    }
  }
}
}  // namespace eb
