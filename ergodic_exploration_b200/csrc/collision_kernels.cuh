// collision_kernels.cuh -- batched occupancy-grid collision checks (sm_100a).
//
// Replaces, for a batch of independent poses / candidate twists sharing one
// occupancy grid, Collision::collisionCheck (collision.cpp:126-143: search
// :150-167, bresenhamCircle :169-215, checkCell :217-244, GridMap::world2Grid
// grid.cpp:143-160, getCell :177-184) and validate_control (numerics.hpp:312-330:
// integrate_twist :273-298 + normalize_angle_PI :77-89 per step) -- the call the
// exploration loop makes right after control() on every tick (exploration.hpp:238).
//
// This is integer / byte gather work: one thread per instance walks the reference's
// Bresenham circles and probes int8 cells through the read-only path (the map is
// shared by the whole batch and stays L2-resident).  Two things differ from a
// transliteration, neither changes a result:
//  * Radius pruning.  checkCell reports a collision only for cells with
//    dx^2 + dy^2 <= r_col^2, and every cell this circle walk emits for radius r
//    lies farther than r - 1/2 from the centre (checked exhaustively for
//    r < kPruneVerified in tests/test_collision_cpu.py), so circles with
//    r > r_col can never hit: the search stops at min(r_max, r_col) instead of
//    r_max.  The closest-obstacle book-keeping of checkCell (cfg.sqrd_obs, dx, dy)
//    feeds minDistance / minDirection only and is not computed.
//  * world2Grid casts floor() to unsigned (undefined for poses left of / below
//    the map); the x86-64 behaviour -- wrap-around, i.e. the signed floor -- is
//    what the CPU checker under tests restates and what is implemented here.
// DynamicWindow::control (dynamic_window.cpp:93-287) runs on the same pieces (dwa_control_kernel).
// Per-instance maps (eb_grid_batch): the PER_MAP instantiations of the three check kernels read, per thread (DWA: per
// warp), the GridView record of their instance's map and derive its radii with collision_params' expressions; the
// circle walk, the pose chain and the objective are the same code.  They always walk the circles (no dilated map).
// The pose chain of validate_control / the window rollouts uses explicitly rounded multiplies / adds in
// the reference's association order; sin / cos come from the CUDA library, so a
// pose can differ from glibc's by an ulp or two (a cell index could differ only
// for a pose within ~1e-15 of a cell edge).
#pragma once

#include "common.cuh"

namespace eb
{
constexpr int kPruneVerified = 3000;  // radii for which the r - 1/2 bound has been checked exhaustively

// last radius worth walking: min(r_max, r_col) where the r - 1/2 bound has been verified and the
// collision radius is a plain non-negative one; otherwise the reference's full range
__host__ __device__ inline int prune_radius(int r_col, int r_max)
{
  return (r_col >= 0 && r_col + 1 < kPruneVerified) ? (r_max < r_col ? r_max : r_col) : r_max;
}

struct GridView
{
  const signed char* data;  // [ysize][xsize]
  unsigned int xsize, ysize;
  double resolution, xmin, ymin;
};

struct CollisionParams
{
  GridView g;
  int r_bnd, r_col, r_max;  // collision.cpp:130-133
  double occupied_threshold;
  int B;
  // validate_control
  int steps;
  double dt;
  const double* x0;  // [B][3] start poses (validate) or the poses themselves (check)
  const double* u;   // [B][3] twists (validate only)
  int* out;          // [B]: collision_check 1 = collision; validate_control 1 = collision free
  // optional pre-dilated map (inflate_kernel): one lookup answers collisionCheck for a centre cell
  const unsigned char* inflated;  // [ysize + 2 pad][xsize + 2 pad] or null
  int pad;
};

// the maps of an eb_grid_batch: pose / twist i of a PER_MAP call is checked against maps[i / per]
struct MapSet
{
  const GridView* maps;  // [B] records; data points into the handle's arena
  int per;
  double boundary, padded, search;  // boundary_radius, boundary_radius + obstacle_threshold, search_radius
};

// p with map `inst` of m and the radii of collision_params (collision.cpp:130-133) for that map's resolution
__device__ __forceinline__ CollisionParams on_map(const CollisionParams& p, const MapSet& m, int inst)
{
  CollisionParams q = p;
  q.g = m.maps[inst];
  q.r_bnd = (int)floor(__ddiv_rn(m.boundary, q.g.resolution));
  q.r_col = (int)floor(__ddiv_rn(m.padded, q.g.resolution));
  q.r_max = (int)floor(__ddiv_rn(m.search, q.g.resolution));
  return q;
}

// numerics.hpp:77-89 with every operation explicitly rounded (no FMA contraction)
__device__ __forceinline__ double normalize_angle_pi_rn(double rad)
{
  const double shifted = __dadd_rn(rad, kPi);
  const double q = floor(__ddiv_rn(shifted, __dmul_rn(2.0, kPi)));
  rad = __dsub_rn(shifted, __dmul_rn(__dmul_rn(q, 2.0), kPi));
  if (rad < 0.0) rad = __dadd_rn(rad, __dmul_rn(2.0, kPi));
  return __dsub_rn(rad, kPi);
}

// Collision::checkCell (:217-244) without the closest-obstacle book-keeping
__device__ __forceinline__ bool check_cell(const GridView& g, double thr, int cx, int cy, int r_col, unsigned int cj,
                                           unsigned int ci)
{
  if (!(ci <= g.ysize - 1u && cj <= g.xsize - 1u)) return false;  // GridMap::gridBounds grid.cpp:96-100
  const double cell = (double)__ldg(g.data + (size_t)ci * g.xsize + cj) / 100.0;  // getCell grid.cpp:177-184
  if (cell < thr) return false;
  const unsigned int dj = (unsigned int)cx - cj, di = (unsigned int)cy - ci;
  const int sqrd_obs = (int)(dj * dj + di * di);
  return sqrd_obs <= r_col * r_col;
}

// Collision::collisionCheck (:126-143) for one pose
__device__ __forceinline__ bool collision_check_pose(const CollisionParams& p, double px, double py)
{
  const GridView& g = p.g;
  // GridMap::world2Grid grid.cpp:143-160
  unsigned int j = (unsigned int)(long long)floor((px - g.xmin) / g.resolution);
  unsigned int i = (unsigned int)(long long)floor((py - g.ymin) / g.resolution);
  if (j == g.xsize) j--;
  if (i == g.ysize) i--;
  const int cx = (int)j, cy = (int)i;
  if (p.inflated)
  {
    // centres farther than `pad` outside the map cannot reach an in-bounds cell
    const long long px = (long long)cx + p.pad, py = (long long)cy + p.pad;
    const long long pw = (long long)g.xsize + 2 * p.pad, ph = (long long)g.ysize + 2 * p.pad;
    if (px < 0 || py < 0 || px >= pw || py >= ph) return false;
    return __ldg(p.inflated + (size_t)py * (size_t)pw + (size_t)px) != 0;
  }
  // Collision::search (:150-167), pruned to the radii that can satisfy sqrd_obs <= r_col^2
  const int r_last = prune_radius(p.r_col, p.r_max);
  for (int r0 = p.r_bnd; r0 <= r_last; r0++)
  {
    // Collision::bresenhamCircle (:169-215)
    int x = -r0, y = 0, err = 2 - 2 * r0;
    while (x < 0)
    {
      if (check_cell(g, p.occupied_threshold, cx, cy, p.r_col, (unsigned int)(cx - x), (unsigned int)(cy + y)) ||
          check_cell(g, p.occupied_threshold, cx, cy, p.r_col, (unsigned int)(cx - y), (unsigned int)(cy - x)) ||
          check_cell(g, p.occupied_threshold, cx, cy, p.r_col, (unsigned int)(cx + x), (unsigned int)(cy - y)) ||
          check_cell(g, p.occupied_threshold, cx, cy, p.r_col, (unsigned int)(cx + y), (unsigned int)(cy + x)))
        return true;
      const int r = err;
      if (r <= y)
      {
        y++;
        err += 2 * y + 1;
      }
      if (r > x || err > y)
      {
        x++;
        err += 2 * x + 1;
      }
    }
  }
  return false;
}

// Map dilation.  collisionCheck(pose) is the OR, over a FIXED set of cell offsets around the
// pose's cell (the cells of the circle walks r_bnd .. r_col that satisfy dx^2 + dy^2 <= r_col^2),
// of "in bounds and occupied" -- the early returns of the reference only shorten the walk.  For
// workloads that check far more poses than the map has cells (DynamicWindow: 120 rollouts x 20
// poses per robot) the OR is evaluated once per cell into a padded byte map and every pose
// check becomes a single lookup; the flags are identical by construction.  offsets: (dj, di).
__global__ void __launch_bounds__(256) inflate_kernel(const GridView g, double thr, const short2* __restrict__ offsets,
                                                      int noffsets, int pad, unsigned char* __restrict__ out)
{
  const long long pw = (long long)g.xsize + 2 * pad, ph = (long long)g.ysize + 2 * pad;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= pw * ph) return;
  const int cx = (int)(idx % pw) - pad, cy = (int)(idx / pw) - pad;
  unsigned char hit = 0;
  for (int o = 0; o < noffsets; o++)
  {
    const short2 d = __ldg(offsets + o);
    const unsigned int cj = (unsigned int)(cx + d.x), ci = (unsigned int)(cy + d.y);
    if (ci <= g.ysize - 1u && cj <= g.xsize - 1u &&
        !((double)__ldg(g.data + (size_t)ci * g.xsize + cj) / 100.0 < thr))
    {
      hit = 1;
      break;
    }
  }
  out[idx] = hit;
}

// The same map, built the other way round: every OCCUPIED in-bounds cell marks the centres
// that can see it (centre = cell - offset).  Occupied cells are a small fraction of a map, so
// this touches far fewer bytes than the per-centre gather above; `out` must be zeroed first.
// The stores race only with stores of the same value.
__global__ void __launch_bounds__(256) inflate_scatter_kernel(const GridView g, double thr,
                                                              const short2* __restrict__ offsets, int noffsets,
                                                              int pad, unsigned char* __restrict__ out)
{
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)g.xsize * g.ysize) return;
  if ((double)__ldg(g.data + idx) / 100.0 < thr) return;
  const int cj = (int)(idx % g.xsize), ci = (int)(idx / g.xsize);
  const long long pw = (long long)g.xsize + 2 * pad;
  for (int o = 0; o < noffsets; o++)
  {
    const short2 d = __ldg(offsets + o);
    // centre (cj - dx, ci - dy) always lies inside the padded map: |d| <= r_col = pad
    out[(size_t)(ci - d.y + pad) * (size_t)pw + (size_t)(cj - d.x + pad)] = 1;
  }
}

// The set call of an eb_grid_batch: one block per map that is written (a flagged instance's new cells) or moved (an
// unflagged instance's cells, when the arena is laid out again); the block also stores the instance's new record.
struct MapCopy
{
  const signed char* src;
  GridView view;  // the new record; view.data is the destination
  int inst;
};

__global__ void __launch_bounds__(256) map_copy_kernel(const MapCopy* __restrict__ copies, GridView* __restrict__ views)
{
  const MapCopy m = copies[blockIdx.x];
  const size_t bytes = (size_t)m.view.xsize * m.view.ysize;
  signed char* dst = const_cast<signed char*>(m.view.data);
  size_t k = threadIdx.x;
  if (((reinterpret_cast<uintptr_t>(m.src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0)
  {
    for (; k < bytes / 16; k += blockDim.x)
      reinterpret_cast<uint4*>(dst)[k] = __ldg(reinterpret_cast<const uint4*>(m.src) + k);
    k = bytes / 16 * 16 + threadIdx.x;
  }
  for (; k < bytes; k += blockDim.x) dst[k] = m.src[k];
  if (threadIdx.x == 0) views[m.inst] = m.view;
}

// eb_grid_batch_set_rows_*: one CTA per band of whole rows, a contiguous byte range of the map's slot; the map's
// record does not change
struct BandCopy
{
  const signed char* src;
  signed char* dst;
  size_t bytes;
};

__global__ void __launch_bounds__(256) band_copy_kernel(const BandCopy* __restrict__ bands)
{
  const BandCopy b = bands[blockIdx.x];
  size_t k = threadIdx.x;
  if (((reinterpret_cast<uintptr_t>(b.src) | reinterpret_cast<uintptr_t>(b.dst)) & 15) == 0)
  {
    for (; k < b.bytes / 16; k += blockDim.x)
      reinterpret_cast<uint4*>(b.dst)[k] = __ldg(reinterpret_cast<const uint4*>(b.src) + k);
    k = b.bytes / 16 * 16 + threadIdx.x;
  }
  for (; k < b.bytes; k += blockDim.x) b.dst[k] = b.src[k];
}

// fraction of occupied cells, to pick between the two builders
__global__ void __launch_bounds__(256) count_occupied_kernel(const GridView g, double thr, unsigned long long* count)
{
  const long long n = (long long)g.xsize * g.ysize;
  unsigned int local = 0;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x)
    local += !((double)__ldg(g.data + idx) / 100.0 < thr);
  local = __reduce_add_sync(kFull, local);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, (unsigned long long)local);
}

template <bool PER_MAP>
__global__ void __launch_bounds__(128) collision_check_kernel(const CollisionParams p, const MapSet m)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.B) return;
  if constexpr (PER_MAP)
    p.out[i] = collision_check_pose(on_map(p, m, i / m.per), p.x0[(size_t)i * 3 + 0], p.x0[(size_t)i * 3 + 1]) ? 1 : 0;
  else
    p.out[i] = collision_check_pose(p, p.x0[(size_t)i * 3 + 0], p.x0[(size_t)i * 3 + 1]) ? 1 : 0;
}

// integrate_twist (numerics.hpp:273-298): body-frame displacement of one step of a constant
// twist -- the same for every step -- with every operation explicitly rounded
struct TwistStep
{
  double d0, d1, d2;
  __device__ __forceinline__ TwistStep(double u0, double u1, double u2, double dt)
  {
    if (fabs(u2 - 0.0) < 1.0e-12)
    {
      d0 = __dmul_rn(u0, dt);
      d1 = __dmul_rn(u1, dt);
      d2 = 0.0;
    }
    else
    {
      const double vb0 = __dmul_rn(u0, dt), vb1 = __dmul_rn(u1, dt), vb2 = __dmul_rn(u2, dt);
      double s, c;
      sincos(vb2, &s, &c);
      d0 = __ddiv_rn(__dadd_rn(__dmul_rn(vb0, s), __dmul_rn(vb1, __dsub_rn(c, 1.0))), vb2);
      d1 = __ddiv_rn(__dadd_rn(__dmul_rn(vb1, s), __dmul_rn(vb0, __dsub_rn(1.0, c))), vb2);
      d2 = vb2;
    }
  }
  // x + transform2d(theta) * dqb, rows summed in column order (the third column is zero), then the wrap
  __device__ __forceinline__ void advance(double& x, double& y, double& th) const
  {
    double s, c;
    sincos(th, &s, &c);
    x = __dadd_rn(x, __dadd_rn(__dmul_rn(c, d0), __dmul_rn(-s, d1)));
    y = __dadd_rn(y, __dadd_rn(__dmul_rn(s, d0), __dmul_rn(c, d1)));
    th = normalize_angle_pi_rn(__dadd_rn(th, d2));
  }
};

// validate_control (numerics.hpp:312-330): constant twist integrated for `steps` steps,
// the pose checked after every step; 1 = collision free
__device__ __forceinline__ int validate_control_ok(const CollisionParams& p, int i)
{
  double x = p.x0[(size_t)i * 3 + 0], y = p.x0[(size_t)i * 3 + 1], th = p.x0[(size_t)i * 3 + 2];
  const TwistStep step(p.u[(size_t)i * 3 + 0], p.u[(size_t)i * 3 + 1], p.u[(size_t)i * 3 + 2], p.dt);
  int ok = 1;
  for (int k = 0; k < p.steps; k++)
  {
    step.advance(x, y, th);
    if (collision_check_pose(p, x, y))
    {
      ok = 0;
      break;
    }
  }
  return ok;
}

__device__ __forceinline__ void validate_control_one(const CollisionParams& p, int i) { p.out[i] = validate_control_ok(p, i); }

template <bool PER_MAP>
__global__ void __launch_bounds__(128) validate_control_kernel(const CollisionParams p, const MapSet m)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.B) return;
  if constexpr (PER_MAP)
    validate_control_one(on_map(p, m, i / m.per), i);
  else
    validate_control_one(p, i);
}

// integrate_twist + normalize_angle_PI for a batch of poses (numerics.hpp:273-298, 77-89): the
// constant-twist step the reference uses wherever a pose is propagated (validate_control,
// DynamicWindow, and the closed-loop harness of bench.py --workload c5loop).  In place is fine.
__global__ void __launch_bounds__(256) integrate_twist_kernel(const double* __restrict__ x, const double* __restrict__ u,
                                                              double dt, int count, double* __restrict__ out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double px = x[(size_t)i * 3 + 0], py = x[(size_t)i * 3 + 1], th = x[(size_t)i * 3 + 2];
  const TwistStep step(u[(size_t)i * 3 + 0], u[(size_t)i * 3 + 1], u[(size_t)i * 3 + 2], dt);
  step.advance(px, py, th);
  out[(size_t)i * 3 + 0] = px;
  out[(size_t)i * 3 + 1] = py;
  out[(size_t)i * 3 + 2] = th;
}

// ---- DynamicWindow::control (dynamic_window.cpp:93-187) ---------------------------------
// One warp per instance; the lanes stride over the vx * vy * vth candidate twists of the
// window (:189-235), each lane rolls its candidates out (objective :237-286: constant twist,
// collision check per step, tracking cost) and keeps its first strict minimum; a warp arg-min
// with ties to the lower candidate index reproduces the reference's loop order exactly.
// The candidate twists are the reference's accumulated sums (vx += dvx, ...).
struct DwaParams
{
  CollisionParams col;  // grid, radii, threshold, steps, dt (B, x0, u, out unused)
  int B;
  double acc_dt, acc_lim[3], vmin[3], vmax[3];
  unsigned int n[3];    // vx, vy, vth samples (>= 1)
  const double* x0;     // [B][3]
  const double* vb;     // [B][3] current body twist
  const double* vref;   // [B][3] reference twist, or null
  const double* xt_ref; // reference trajectory [ncols][3] (xt_stride = 0: shared) or [B][ncols][3]
  int ncols;
  long long xt_stride;
  double tf;            // ncols * dt_ref (:148)
  int* found;           // [B]
  double* u_opt;        // [B][3]
  double* min_cost;     // [B] or null
};

constexpr double kDblMax = 1.7976931348623157e308;

// col: p.col, or p.col on the instance's own map (PER_MAP)
__device__ __forceinline__ double dwa_objective(const DwaParams& p, const CollisionParams& col, const double* xt, double x,
                                                double y, double th, double u0, double u1, double u2, const double* vref)
{
  const TwistStep step(u0, u1, u2, p.col.dt);
  double t = 0.0, cost = 0.0;
  for (int k = 0; k < p.col.steps; k++)
  {
    step.advance(x, y, th);
    if (collision_check_pose(col, x, y)) return kDblMax;
    if (xt)
    {
      // index into the reference trajectory (:276)
      const unsigned int j = (unsigned int)round(__ddiv_rn(__dmul_rn((double)(p.ncols - 1), t), p.tf));
      const double dx = __dsub_rn(xt[3 * (size_t)j + 0], x), dy = __dsub_rn(xt[3 * (size_t)j + 1], y);
      cost = __dadd_rn(cost, __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))));
      cost = __dadd_rn(cost, fabs(normalize_angle_pi_rn(__dsub_rn(normalize_angle_pi_rn(xt[3 * (size_t)j + 2]), th))));
      t = __dadd_rn(t, p.col.dt);
    }
  }
  if (xt) return cost;
  const double e0 = __dsub_rn(vref[0], u0), e1 = __dsub_rn(vref[1], u1), e2 = __dsub_rn(vref[2], u2);
  return __dadd_rn(__dadd_rn(__dmul_rn(e0, e0), __dmul_rn(e1, e1)), __dmul_rn(e2, e2));
}

// DynamicWindow::window (:189-235) of robot inst: the first sample of each axis and the step between samples
__device__ __forceinline__ void dwa_window(const DwaParams& p, int inst, double (&lower)[3], double (&delta)[3])
{
#pragma unroll
  for (int a = 0; a < 3; a++)
  {
    const double v = p.vb[(size_t)inst * 3 + a], reach = __dmul_rn(p.acc_lim[a], p.acc_dt);
    lower[a] = fmax(__dsub_rn(v, reach), p.vmin[a]);
    const double upper = fmin(__dadd_rn(v, reach), p.vmax[a]);
    delta[a] = p.n[a] > 1 ? __ddiv_rn(__dsub_rn(upper, lower[a]), (double)(p.n[a] - 1)) : 0.0;
  }
}

// candidate c of the window in the reference's loop order (vx outer, vth inner), as its accumulated sums
__device__ __forceinline__ void dwa_twist(const DwaParams& p, const double (&lower)[3], const double (&delta)[3],
                                          unsigned int c, double& u0, double& u1, double& u2)
{
  const unsigned int k = c % p.n[2], j = (c / p.n[2]) % p.n[1], i = c / (p.n[2] * p.n[1]);
  u0 = lower[0];
  for (unsigned int s = 0; s < i; s++) u0 = __dadd_rn(u0, delta[0]);  // vx += dvx, i times
  u1 = lower[1];
  for (unsigned int s = 0; s < j; s++) u1 = __dadd_rn(u1, delta[1]);
  u2 = lower[2];
  for (unsigned int s = 0; s < k; s++) u2 = __dadd_rn(u2, delta[2]);
}

// warp arg-min of (cost, candidate) with ties to the lower candidate: the reference's first strict minimum in loop
// order, whichever lanes evaluated which candidates
__device__ __forceinline__ void dwa_argmin_warp(double& best, unsigned int& best_c)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
  {
    const double oc = __shfl_xor_sync(kFull, best, o);
    const unsigned int oi = __shfl_xor_sync(kFull, best_c, o);
    if (oc < best || (oc == best && oi < best_c))
    {
      best = oc;
      best_c = oi;
    }
  }
}

// almost_equal(min_cost, max) (:132): 0 when no candidate beat the initial min_cost (the window found nothing)
__device__ __forceinline__ int dwa_found(double best) { return (fabs(best - kDblMax) < 1.0e-12) ? 0 : 1; }

// PER_MAP: robot inst on map inst of m
template <bool PER_MAP>
__global__ void __launch_bounds__(128) dwa_control_kernel(const DwaParams p, const MapSet m)
{
  const int lane = threadIdx.x & 31;
  const int inst = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (inst >= p.B) return;
  const CollisionParams col = PER_MAP ? on_map(p.col, m, inst) : p.col;
  const double x = p.x0[(size_t)inst * 3 + 0], y = p.x0[(size_t)inst * 3 + 1], th = p.x0[(size_t)inst * 3 + 2];
  double lower[3], delta[3];
  dwa_window(p, inst, lower, delta);
  const double* xt = p.xt_ref ? p.xt_ref + (size_t)inst * (size_t)p.xt_stride : nullptr;
  const double* vref = p.vref ? p.vref + (size_t)inst * 3 : nullptr;
  const unsigned int total = p.n[0] * p.n[1] * p.n[2];
  // (the lambda and the inline arg-min below keep this kernel's instructions as they were before the helpers were
  // factored out for dwa_fallback_kernel; direct calls change its register allocation)
  auto twist = [&](unsigned int c, double& u0, double& u1, double& u2) { dwa_twist(p, lower, delta, c, u0, u1, u2); };
  double best = kDblMax;
  unsigned int best_c = 0xffffffffu;
  for (unsigned int c = lane; c < total; c += 32)
  {
    double u0, u1, u2;
    twist(c, u0, u1, u2);
    const double cost = dwa_objective(p, col, xt, x, y, th, u0, u1, u2, vref);
    if (cost < best)
    {
      best = cost;
      best_c = c;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
  {
    const double oc = __shfl_xor_sync(kFull, best, o);
    const unsigned int oi = __shfl_xor_sync(kFull, best_c, o);
    if (oc < best || (oc == best && oi < best_c))
    {
      best = oc;
      best_c = oi;
    }
  }
  if (lane == 0)
  {
    double u0 = 0.0, u1 = 0.0, u2 = 0.0;  // u_opt stays zero when nothing beats the initial min_cost (:99)
    if (best_c != 0xffffffffu) twist(best_c, u0, u1, u2);
    p.u_opt[(size_t)inst * 3 + 0] = u0;
    p.u_opt[(size_t)inst * 3 + 1] = u1;
    p.u_opt[(size_t)inst * 3 + 2] = u2;
    p.found[inst] = dwa_found(best);
    if (p.min_cost) p.min_cost[inst] = best;
  }
}
}  // namespace eb
