// common.cuh -- shared device helpers for the sm_100a ergodic-control kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace eb
{
constexpr double kPi = 3.14159265358979323846;  // numerics.hpp:58
constexpr unsigned kFull = 0xffffffffu;

// One FP64 tensor-core tile: D(8x8) += A(8x4, row) * B(4x8, col).
// Fragment ownership (PTX ISA, mma.m8n8k4 .f64): with g = lane >> 2 and
// q = lane & 3, a = A[g][q], b = B[q][g], {d0, d1} = D[g][2q], D[g][2q + 1].
// On sm_100a this assembles to DMMA.8x8x4.
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b)
{
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// inclusive prefix sum over the lanes of a warp (lane 0 first)
__device__ __forceinline__ double warp_scan_incl(double v, int lane)
{
#if defined(EB_ABL) && (EB_ABL & 64)
  return v + (double)lane;  // ablation timing only
#endif
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
  {
    const double n = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

// inclusive suffix sum over the lanes of a warp (lane 31 first)
__device__ __forceinline__ double warp_scan_incl_rev(double v, int lane)
{
#if defined(EB_ABL) && (EB_ABL & 64)
  return v - (double)lane;  // ablation timing only
#endif
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
  {
    const double n = __shfl_down_sync(kFull, v, o);
    if (lane + o < 32) v += n;
  }
  return v;
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// ---- sin/cos kernels -------------------------------------------------------
// Cody-Waite reduction to [-pi/4, pi/4] (two-term pi/2, exact to ~1e-33 * |q|)
// followed by the fdlibm minimax kernels (|error| < 1 ulp).  About a third of
// the instructions of the CUDA library sincos(), which carries a three-term
// reduction, a Payne-Hanek slow path and special-value handling that the
// bounded arguments of this kernel (headings, k*pi*x/l) never need; arguments
// beyond 2^30 take the (out-of-line) library path.  The polynomial
// coefficients live in constant memory so every DFMA reads them as a
// constant-bank operand instead of materialising 64-bit immediates.
__constant__ double kTrigS[6] = { -1.66666666666666324348e-01, 8.33333333332248946124e-03,
                                  -1.98412698298579493134e-04, 2.75573137070700676789e-06,
                                  -2.50507602534068634195e-08, 1.58969099521155010221e-10 };
__constant__ double kTrigC[6] = { 4.16666666666666019037e-02, -1.38888888888741095749e-03,
                                  2.48015872894767294178e-05, -2.75573143513906633035e-07,
                                  2.08757232129817482790e-09, -1.13596475577881948265e-11 };
__constant__ double kTrigR[5] = { 6.36619772367581382433e-01,   // 2/pi
                                  1.57079632679489655800e+00,   // pi/2 hi
                                  6.12323399573676603587e-17,   // pi/2 lo
                                  3.14159265358979311600e+00,   // pi hi
                                  1.22464679914735317723e-16 }; // pi lo

__device__ __forceinline__ void sincos_kernel(double r, int n, double* s, double* c)
{
#if defined(EB_ABL) && (EB_ABL & 8)
  *s = r * (double)(n + 1);  // ablation timing only: no polynomial (wrong values)
  *c = 1.0 - r;
  return;
#endif
  const double z = r * r;
  double ps = fma(z, kTrigS[5], kTrigS[4]);
  double pc = fma(z, kTrigC[5], kTrigC[4]);
  ps = fma(z, ps, kTrigS[3]);
  pc = fma(z, pc, kTrigC[3]);
  ps = fma(z, ps, kTrigS[2]);
  pc = fma(z, pc, kTrigC[2]);
  ps = fma(z, ps, kTrigS[1]);
  pc = fma(z, pc, kTrigC[1]);
  ps = fma(z, ps, kTrigS[0]);
  pc = fma(z, pc, kTrigC[0]);
  const double sn = fma(z * r, ps, r);                 // r + r^3 * P(r^2)
  const double cs = 1.0 - fma(0.5, z, -(z * z) * pc);  // 1 - (z/2 - z^2 * Q(r^2))
  // quadrant n: (sin, cos) = (sn, cs), (cs, -sn), (-sn, -cs), (-cs, sn); signs by
  // flipping the sign bit of the high word
  const bool swap = n & 1;
  const double a = swap ? cs : sn, b = swap ? sn : cs;
  const int sa = (n & 2) << 30, sb = ((n + 1) & 2) << 30;
  *s = __hiloint2double(__double2hiint(a) ^ sa, __double2loint(a));
  *c = __hiloint2double(__double2hiint(b) ^ sb, __double2loint(b));
}

// Out-of-line library path for arguments beyond 2^30.  Results come back BY
// VALUE: with pointer outputs the callers' sin / cos variables become
// address-taken stack objects, and the fused kernel built with nvcc 12.9 then
// produced wrong fast-path values (reproduced and bisected with
// tools/diag_dump.py: dropping the slow path, or returning by value as here,
// both give correct values).
__device__ __noinline__ double2 slow_sincos2(double x)
{
  double s, c;
  sincos(x, &s, &c);
  return make_double2(s, c);
}
__device__ __noinline__ double2 slow_sincospi2(double x)
{
  double s, c;
  sincospi(x, &s, &c);
  return make_double2(s, c);
}

__device__ __forceinline__ void fast_sincos(double x, double* s, double* c)
{
  double sv, cv;
  if (fabs(x) > 1073741824.0)
  {
    const double2 v = slow_sincos2(x);
    sv = v.x;
    cv = v.y;
  }
  else
  {
    const double q = rint(x * kTrigR[0]);
    double r = fma(-q, kTrigR[1], x);
    r = fma(-q, kTrigR[2], r);
    sincos_kernel(r, (int)q, &sv, &cv);
  }
  *s = sv;
  *c = cv;
}

// sin(pi t), cos(pi t): the reduction t - q/2 is exact
__device__ __forceinline__ void fast_sincospi(double t, double* s, double* c)
{
  double sv, cv;
  if (fabs(t) > 1073741824.0)
  {
    const double2 v = slow_sincospi2(t);
    sv = v.x;
    cv = v.y;
  }
  else
  {
    const double q = rint(t + t);
    const double f = fma(-0.5, q, t);  // exact, |f| <= 1/4
    const double r = fma(f, kTrigR[3], f * kTrigR[4]);
    sincos_kernel(r, (int)q, &sv, &cv);
  }
  *s = sv;
  *c = cv;
}

__device__ __forceinline__ double fast_cospi(double t)
{
  double s, c;
  fast_sincospi(t, &s, &c);
  return c;
}

// numerics.hpp:77-89
__device__ __forceinline__ double normalize_angle_pi(double rad)
{
  const double q = floor((rad + kPi) / (2.0 * kPi));
  rad = (rad + kPi) - q * 2.0 * kPi;
  if (rad < 0.0) rad += 2.0 * kPi;
  return rad - kPi;
}

// counter-based generator for the on-device replay sampler (splitmix64 finaliser)
__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

__device__ __forceinline__ double clampd(double v, double lo, double hi)
{
  // std::clamp(v, lo, hi): (v < lo) ? lo : (hi < v) ? hi : v
  return v < lo ? lo : (hi < v ? hi : v);
}
}  // namespace eb
