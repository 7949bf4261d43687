// target_batch.cuh -- configTarget (ergodic_control.hpp:363-416) for B instances that each own a target and a map
// frame, in one launch (sm_100a, FP64).
//
// One CTA per instance.  The origin of the frame is always recorded; phi_k is rebuilt only when the extent moved by
// 1e-12 or more (almost_equal), as the shared path (eb_config_target) does.  A rebuilding CTA evaluates the density
// on the fly from its Gaussians (gaussian_sum, the expression of target_fill_kernel) and contracts it with cosine
// tables built by the expression of cos_table_kernel, 32 x 32 grid tiles at a time, so any grid fits in shared memory
// and the density never reaches HBM.  Stage 1 sums the tile columns into T[row][kx], stage 2 folds T into the
// coefficients; every sum runs in a fixed order (deterministic).  The tables carry the same bits as the shared plan's,
// so the per-instance phi_k differs from the shared route only in summation order.  num_basis > 32 loops over blocks of
// 32 x 32 orders.
//
// The same launch keeps the replay buffer's cosine rows (hist_cos) valid: an instance whose frame key
// {xmin, ymin, 1 / lx, 1 / ly} moved gets every stored row re-derived (hist_cos_kernel's arithmetic).
#pragma once

#include "common.cuh"
#include "phik_kernels.cuh"
#include "solve_kernel.cuh"

namespace eb
{
constexpr int kTbThreads = 256;
constexpr int kTbTile = 32;        // grid rows / columns per tile, orders per block
constexpr int kTbMaxGauss = 256;   // Gaussians per instance (dynamic shared memory: 6 doubles each)
constexpr int kFaultTarget = 8;    // fault bit: an instance's extent moved without Gaussians, or is not positive

struct TargetBatchParams
{
  int B, nb, max_n;
  double res;
  const double* bounds;  // [B][4] xmin xmax ymin ymax (configure), or null: ...
  const double* extent;  // ... [B][2] lx ly given with the rows of phi_k (eb_set_phik_batch_dev), origin kept
  const int* counts;     // [B] Gaussians per instance
  const double* mu;      // [B][max_n][2]
  const double* sigma;   // [B][max_n][2]
  double* frames;        // [B][kFrDoubles], read and updated
  double* phik;          // [B][nb*nb]: rows of rebuilt instances are written
  int* rebuilt;          // [B] or null
  const double* hist;    // [mem_count][B][3]
  double* hist_cos;      // [mem_count][B][2] or null (no cosine cache)
  long long mem_count;
  int* fault;
};

__device__ __forceinline__ bool tb_almost_equal(double a, double b) { return fabs(a - b) < 1.0e-12; }  // numerics.hpp:67-70

__global__ void __launch_bounds__(kTbThreads) target_batch_kernel(const TargetBatchParams p)
{
  extern __shared__ double s_gauss[];  // [max_n][6], as target_fill_kernel's gauss
  __shared__ double s_d[kTbTile * kTbTile];   // density tile [row][col]
  __shared__ double s_cx[kTbTile * kTbTile];  // cos(kx a x_j) [col][kx]
  __shared__ double s_cy[kTbTile * kTbTile];  // cos(ky b y_i) [row][ky]
  __shared__ double s_t[kTbTile * kTbTile];   // stage 1 of the row tile [row][kx]
  __shared__ double s_xs[kTbTile], s_ys[kTbTile];
  __shared__ double s_total;
  const int inst = blockIdx.x, t = threadIdx.x;
  double* const fr = p.frames + (size_t)inst * kFrDoubles;
  const double old_x = fr[kFrXmin], old_y = fr[kFrYmin], lx = fr[kFrLx], ly = fr[kFrLy];
  const double old_ilx = fr[kFrInvLx], old_ily = fr[kFrInvLy];
  double xmin = old_x, ymin = old_y, nlx = lx, nly = ly;
  bool rebuild = false;
  if (p.bounds)
  {
    const double* b = p.bounds + (size_t)inst * 4;
    xmin = b[0];  // translation from map to fourier domain (:366-367)
    ymin = b[2];
    const double mx = b[1] - b[0], my = b[3] - b[2];
    if (!(tb_almost_equal(mx, lx) && tb_almost_equal(my, ly)))  // :374-377
    {
      if (!(mx > 0.0) || !(my > 0.0) || p.counts[inst] < 1)
      {
        if (t == 0) atomicOr(p.fault, kFaultTarget);
      }
      else
      {
        rebuild = true;
        nlx = mx;  // :382-383
        nly = my;
      }
    }
  }
  else
  {
    nlx = p.extent[2 * (size_t)inst + 0];
    nly = p.extent[2 * (size_t)inst + 1];
  }

  if (rebuild)
  {
    const int nx = (int)round(nlx / p.res) + 1, ny = (int)round(nly / p.res) + 1;  // :387-388
    const int ng = min(p.counts[inst], p.max_n);
    for (int g = t; g < ng; g += kTbThreads)
    {
      // Gaussian ctor (target.hpp:68-71): cov = diag(sigma^2), cov_inv by the 2x2 cofactor inverse; the mean is
      // translated by the origin at rebuild time (operator(), :91-102)
      const double* m = p.mu + ((size_t)inst * p.max_n + g) * 2;
      const double* s = p.sigma + ((size_t)inst * p.max_n + g) * 2;
      const double a = __dmul_rn(s[0], s[0]), d = __dmul_rn(s[1], s[1]);
      const double det = __dsub_rn(__dmul_rn(a, d), 0.0 * 0.0);
      double* G = s_gauss + 6 * g;
      G[0] = m[0] - xmin;
      G[1] = m[1] - ymin;
      G[2] = d / det;
      G[3] = -0.0 / det;
      G[4] = -0.0 / det;
      G[5] = a / det;
    }
    const double fx = kPi / nlx, fy = kPi / nly;  // basis.cpp:85: cos(k * (PI / l) * x)
    const int nblk = (p.nb + kTbTile - 1) / kTbTile;
    const int kxl = t & 31, r8 = t >> 5;  // this thread's column / order and first row of its four
    const int K = p.nb * p.nb;
    for (int by = 0; by < nblk; by++)
      for (int bx = 0; bx < nblk; bx++)
      {
        double acc[4] = { 0.0, 0.0, 0.0, 0.0 };  // raw[32 by + r8 + 8 m][32 bx + kxl]
        double yc = 0.0;                          // accumulated grid coordinates (:394-407), thread 0
        for (int r0 = 0; r0 < ny; r0 += kTbTile)
        {
          __syncthreads();  // the previous row tile's readers are done (and the Gaussians are staged)
          if (t == 0)
            for (int k = 0; k < kTbTile; k++)
            {
              s_ys[k] = yc;
              yc += p.res;
            }
          __syncthreads();
          for (int e = t; e < kTbTile * kTbTile; e += kTbThreads)
          {
            const int r = e >> 5, ky = kTbTile * by + (e & 31);
            s_cy[e] = (ky < p.nb && r0 + r < ny) ? cos((double)ky * fy * s_ys[r]) : 0.0;
          }
          double tacc[4] = { 0.0, 0.0, 0.0, 0.0 };  // T[r8 + 8 m][kxl]
          double xc = 0.0;
          for (int c0 = 0; c0 < nx; c0 += kTbTile)
          {
            __syncthreads();  // the previous column tile's readers are done
            if (t == 0)
              for (int k = 0; k < kTbTile; k++)
              {
                s_xs[k] = xc;
                xc += p.res;
              }
            __syncthreads();
            for (int e = t; e < kTbTile * kTbTile; e += kTbThreads)
            {
              const int r = e >> 5, j = e & 31;
              s_d[e] = (r0 + r < ny && c0 + j < nx) ? gaussian_sum(ng, s_gauss, s_xs[j], s_ys[r]) : 0.0;
              const int kx = kTbTile * bx + j;  // s_cx[e]: column r, order j
              s_cx[e] = (kx < p.nb && c0 + r < nx) ? cos((double)kx * fx * s_xs[r]) : 0.0;
            }
            __syncthreads();
#pragma unroll
            for (int m = 0; m < 4; m++)
            {
              const double* drow = s_d + (r8 + 8 * m) * kTbTile;
              double v = tacc[m];
              for (int j = 0; j < kTbTile; j++) v = fma(drow[j], s_cx[j * kTbTile + kxl], v);
              tacc[m] = v;
            }
          }
#pragma unroll
          for (int m = 0; m < 4; m++) s_t[(r8 + 8 * m) * kTbTile + kxl] = tacc[m];
          __syncthreads();
#pragma unroll
          for (int m = 0; m < 4; m++)
          {
            const int kyl = r8 + 8 * m;
            double v = acc[m];
            for (int r = 0; r < kTbTile; r++) v = fma(s_cy[r * kTbTile + kyl], s_t[r * kTbTile + kxl], v);
            acc[m] = v;
          }
        }
        if (by == 0 && bx == 0 && t == 0) s_total = acc[0];  // raw (0, 0) = sum of the density (target.cpp:87)
        __syncthreads();
        const double total = s_total;
#pragma unroll
        for (int m = 0; m < 4; m++)
        {
          const int ky = kTbTile * by + r8 + 8 * m, kx = kTbTile * bx + kxl;
          if (ky < p.nb && kx < p.nb) p.phik[(size_t)inst * K + ky * p.nb + kx] = acc[m] / total;
        }
      }
  }

  const double ilx = 1.0 / nlx, ily = 1.0 / nly;
  if (p.hist_cos && (__double_as_longlong(xmin) != __double_as_longlong(old_x) ||
                     __double_as_longlong(ymin) != __double_as_longlong(old_y) ||
                     __double_as_longlong(ilx) != __double_as_longlong(old_ilx) ||
                     __double_as_longlong(ily) != __double_as_longlong(old_ily)))
    for (long long r = t; r < p.mem_count; r += kTbThreads)
    {
      const size_t e = (size_t)r * p.B + inst;
      const double xf = p.hist[3 * e + 0] - xmin, yf = p.hist[3 * e + 1] - ymin;
      p.hist_cos[2 * e + 0] = fast_cospi(xf * ilx);
      p.hist_cos[2 * e + 1] = fast_cospi(yf * ily);
    }
  __syncthreads();  // every thread has read the old frame
  if (t == 0)
  {
    // the expressions of eb_control_dev's shared frame
    fr[kFrXmin] = xmin;
    fr[kFrYmin] = ymin;
    fr[kFrLx] = nlx;
    fr[kFrLy] = nly;
    fr[kFrInvLx] = ilx;
    fr[kFrInvLy] = ily;
    fr[kFrAx] = kPi / nlx;
    fr[kFrBy] = kPi / nly;
    if (p.rebuilt) p.rebuilt[inst] = rebuild ? 1 : 0;
  }
}
}  // namespace eb
