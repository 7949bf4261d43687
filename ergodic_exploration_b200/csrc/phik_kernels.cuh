// phik_kernels.cuh -- target density and phi_k target coefficients (sm_100a, FP64).
//
// Replaces Target::fill (target.cpp:78-89, Gaussian::operator() target.hpp:91-102)
// and Basis::spatialCoeff (basis.cpp:122-133).  The reference evaluates 2K
// cosines per grid cell into a K x G temporary; here the separable structure
// F_k(x, y) = cos(kx a x) cos(ky b y) turns the sum over cells into
//     phi_raw = C_y^T  Phi  C_x ,   C_x[j][kx] = cos(kx a x_j), C_y[i][ky] = cos(ky b y_i)
// and since F_0 == 1, sum(Phi) = phi_raw[0]: normalising the density
// (target.cpp:87) is one division after the contraction.
//
// This file holds the shape-agnostic kernels (any nx, ny, nb); the DMMA/TMA
// tile kernels for large grids (nb <= 32) are in phik_dmma.cuh / phik_tma.cuh.
// Tables and T have a leading dimension ld: 32 for nb <= 32 (what the tile
// kernels expect), nb rounded up to a multiple of 32 beyond that.
#pragma once

#include "common.cuh"

namespace eb
{
constexpr int kPhikLd = 32;  // leading dimension of the cosine tables / T for nb <= 32 (bases padded to 32)
__host__ __device__ inline int phik_ld(int nb) { return nb <= 32 ? kPhikLd : ((nb + 31) & ~31); }

// tab[j][k] = cos((k0 + k) * (PI / l) * coord[j]) for k0 + k < nb, else 0 (basis.cpp:85); k0: first order of the table
__global__ void cos_table_kernel(const double* __restrict__ coord, int n, double freq, int nb, int ld, int k0,
                                 double* __restrict__ tab)
{
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * ld) return;
  const int j = (int)(idx / ld), k = k0 + (int)(idx % ld);
  tab[idx] = k < nb ? cos((double)k * freq * coord[j]) : 0.0;
}

// Target::evaluate at one grid point (target.cpp:68-89, un-normalised).
// gauss: per Gaussian 6 doubles {mu_x - trans_x, mu_y - trans_y, ci00, ci10, ci01, ci11}
__device__ __forceinline__ double gaussian_sum(int ng, const double* __restrict__ gauss, double px, double py)
{
  double val = 0.0;
  for (int g = 0; g < ng; g++)
  {
    const double* G = gauss + 6 * g;
    const double d0 = px - G[0], d1 = py - G[1];
    const double r0 = d0 * G[2] + d1 * G[3];
    const double r1 = d0 * G[4] + d1 * G[5];
    val += exp(-0.5 * (r0 * d0 + r1 * d1));
  }
  return val;
}

// Target::evaluate over the configTarget grid
__global__ void target_fill_kernel(int ng, const double* __restrict__ gauss, const double* __restrict__ xs,
                                   const double* __restrict__ ys, int nx, int ny, double* __restrict__ phi)
{
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= (long long)nx * ny) return;
  const int i = (int)(c / nx), j = (int)(c % nx);
  phi[c] = gaussian_sum(ng, gauss, xs[j], ys[i]);
}

// stage 1: T[i][kx] = sum_j Phi[i][j] * Cx[j][kx]; one CTA (32 x 8 threads) per (row, block of 32 orders)
__global__ void __launch_bounds__(256) phik_stage1_simple(const double* __restrict__ phi, int nx,
                                                          const double* __restrict__ cx, int ld, double* __restrict__ T)
{
  __shared__ double red[8][32];
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5, kx = blockIdx.y * 32 + lane;
  const double* row = phi + (size_t)blockIdx.x * nx;
  double acc = 0.0;
  for (int j = part; j < nx; j += 8) acc = fma(row[j], cx[(size_t)j * ld + kx], acc);
  red[part][lane] = acc;
  __syncthreads();
  if (part == 0)
  {
    double s = red[0][lane];
#pragma unroll
    for (int pth = 1; pth < 8; pth++) s += red[pth][lane];
    T[(size_t)blockIdx.x * ld + kx] = s;
  }
}

// stage 2: raw[ky][kx] = sum_i Cy[i][ky] * T[i][kx]; one CTA per (ky, block of 32 orders kx)
__global__ void __launch_bounds__(256) phik_stage2_simple(const double* __restrict__ T, int ny,
                                                          const double* __restrict__ cyt, int ld, double* __restrict__ raw)
{
  __shared__ double red[8][32];
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5, ky = blockIdx.x, kx = blockIdx.y * 32 + lane;
  double acc = 0.0;
  for (int i = part; i < ny; i += 8) acc = fma(cyt[(size_t)i * ld + ky], T[(size_t)i * ld + kx], acc);
  red[part][lane] = acc;
  __syncthreads();
  if (part == 0)
  {
    double s = red[0][lane];
#pragma unroll
    for (int pth = 1; pth < 8; pth++) s += red[pth][lane];
    raw[(size_t)ky * ld + kx] = s;
  }
}

// nb > 32: normalisation of the ld x ld raw block of the simple pair; phik[ky*nb + kx] = raw[ky][kx] / raw[0][0]
__global__ void phik_finalize_wide(const double* __restrict__ parts, int nb, int ld, double* __restrict__ phik,
                                   double* __restrict__ phi_sum, double* __restrict__ raw)
{
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ld * ld) return;
  const double total = parts[0];
  const int ky = t / ld, kx = t % ld;
  const bool in = ky < nb && kx < nb;
  if (raw) raw[t] = in ? parts[t] : 0.0;
  if (phik && in) phik[ky * nb + kx] = parts[t] / total;
  if (t == 0 && phi_sum) *phi_sum = total;
}

// sums `nparts` partial 32x32 blocks in a fixed order (deterministic) and
// normalises: phik[ky*nb + kx] = raw[ky][kx] / raw[0][0].  fold: the partials'
// columns are in the tile kernel's [even orders | odd orders] order.
__global__ void __launch_bounds__(1024) phik_finalize(const double* __restrict__ parts, int nparts, int nb, int fold,
                                                      double* __restrict__ phik, double* __restrict__ phi_sum,
                                                      double* __restrict__ raw)
{
  __shared__ double total;
  const int t = threadIdx.x;
  double s = 0.0;
  for (int pth = 0; pth < nparts; pth++) s += parts[(size_t)pth * 1024 + t];
  if (t == 0) total = s;  // order (0, 0) sits at column 0 either way
  __syncthreads();
  const int ky = t >> 5, col = t & 31;
  const int kx = fold ? (col < 16 ? 2 * col : 2 * (col - 16) + 1) : col;
  if (raw) raw[ky * 32 + kx] = (ky < nb && kx < nb) ? s : 0.0;
  if (phik && ky < nb && kx < nb) phik[ky * nb + kx] = s / total;
  if (t == 0 && phi_sum) *phi_sum = total;
}

// nb > 32 through the 32-order tile kernels: blocks[by][bx][ky][kx] (1024 doubles each) -> phik / raw (ld x ld)
__global__ void phik_assemble_wide(const double* __restrict__ blocks, int nb, int nblk, int ld, double* __restrict__ phik,
                                   double* __restrict__ phi_sum, double* __restrict__ raw)
{
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ld * ld) return;
  const double total = blocks[0];
  const int ky = t / ld, kx = t % ld;
  const bool in = ky < nb && kx < nb;
  const double v = in ? blocks[((size_t)(ky >> 5) * nblk + (kx >> 5)) * 1024 + (ky & 31) * 32 + (kx & 31)] : 0.0;
  if (raw) raw[t] = v;
  if (phik && in) phik[ky * nb + kx] = v / total;
  if (t == 0 && phi_sum) *phi_sum = total;
}

// ---- point-wise Basis / Target entry points (arbitrary points, not a grid) ---
// One CTA per coefficient k = ky*nb + kx; threads stride over the points.
// mode 0: out[k] = scale * sum_c F_k(p_c) * w_c   (Basis::trajCoeff basis.cpp:109-120 with w = 1,
//                                                 Basis::spatialCoeff :122-133 with w = phi_vals)
__global__ void __launch_bounds__(256) basis_sum_kernel(double lx, double ly, int nb, const double* __restrict__ pts,
                                                        int ld, long long n, const double* __restrict__ w,
                                                        double scale, double* __restrict__ out)
{
  __shared__ double red[256];
  const int k = blockIdx.x, kx = k % nb, ky = k / nb;
  const double fx = (double)kx * (kPi / lx), fy = (double)ky * (kPi / ly);  // basis.cpp:85
  double acc = 0.0;
  for (long long c = threadIdx.x; c < n; c += blockDim.x)
  {
    const double f = cos(fx * pts[c * ld + 0]) * cos(fy * pts[c * ld + 1]);
    acc += w ? f * w[c] : f;
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1)
  {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[k] = scale * red[0];
}

// Basis::gradFourierBasis (basis.cpp:91-107): dfk is 2 x K column-major
__global__ void basis_grad_kernel(double lx, double ly, int nb, double x0, double x1, double* __restrict__ dfk)
{
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nb * nb) return;
  const double k1 = (double)(k % nb) * (kPi / lx), k2 = (double)(k / nb) * (kPi / ly);
  dfk[2 * k + 0] = -k1 * sin(k1 * x0) * cos(k2 * x1);
  dfk[2 * k + 1] = -k2 * cos(k1 * x0) * sin(k2 * x1);
}

// Target::fill over arbitrary points (target.cpp:78-89): un-normalised values,
// then a single-CTA sum; the division happens in target_scale_kernel.
__global__ void target_points_kernel(int ng, const double* __restrict__ gauss, const double* __restrict__ pts,
                                     long long n, double* __restrict__ vals)
{
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  const double px = pts[2 * c], py = pts[2 * c + 1];
  double val = 0.0;
  for (int g = 0; g < ng; g++)
  {
    const double* G = gauss + 6 * g;
    const double d0 = px - G[0], d1 = py - G[1];
    const double r0 = d0 * G[2] + d1 * G[3];
    const double r1 = d0 * G[4] + d1 * G[5];
    val += exp(-0.5 * (r0 * d0 + r1 * d1));
  }
  vals[c] = val;
}

__global__ void __launch_bounds__(1024) vector_sum_kernel(const double* __restrict__ v, long long n,
                                                          double* __restrict__ total)
{
  __shared__ double red[1024];
  double acc = 0.0;
  for (long long c = threadIdx.x; c < n; c += blockDim.x) acc += v[c];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1)
  {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = red[0];
}

__global__ void vector_div_kernel(double* __restrict__ v, long long n, const double* __restrict__ total)
{
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n) v[c] /= *total;
}

// ---- FP64 throughput probes (roofline denominator) -------------------------
__global__ void __launch_bounds__(256) dfma_probe(double* out, int iters, double seed)
{
  double a[8];
#pragma unroll
  for (int i = 0; i < 8; i++) a[i] = seed + i + threadIdx.x;
  const double m = 1.0000001, c = 1e-9;
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int r = 0; r < 8; r++)
#pragma unroll
      for (int i = 0; i < 8; i++) a[i] = fma(a[i], m, c);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += a[i];
  if (s == 123.456) out[0] = s;
}

__global__ void __launch_bounds__(256) dmma_probe(double* out, int iters, double seed)
{
  double d[8][2];
#pragma unroll
  for (int i = 0; i < 8; i++) d[i][0] = d[i][1] = seed;
  const double a = 1.0 + 1e-9 * threadIdx.x, b = 1e-9;
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
      for (int i = 0; i < 8; i++) dmma884(d[i][0], d[i][1], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += d[i][0] + d[i][1];
  if (s == 123.456) out[0] = s;
}
}  // namespace eb
