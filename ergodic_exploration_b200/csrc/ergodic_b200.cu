// ergodic_b200.cu -- C ABI (include/ergodic_b200.h) over the sm_100a kernels.
//
// Host-side state mirrors the private members of the reference's
// ErgodicControl (ergodic_control.hpp:165-184), batched over B instances and
// resident on the device: ut_ (ping-pong, 3 x N x B), pose_, phik_, the
// replay buffer (time-major [cap][B][3]) and the Basis tables.
// There is no CPU implementation behind this ABI: every entry point either
// launches CUDA work or fails.
#include "../../include/ergodic_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges show up under Nsight, cost ~nothing otherwise

#include "collision_kernels.cuh"
#include "map_target.cuh"
#include "map_target_batch.cuh"
#include "model_kernels.cuh"
#include "peer_gather.cuh"
#include "phik_dmma.cuh"
#include "phik_kernels.cuh"
#include "phik_tma.cuh"
#include "safe_control.cuh"
#include "solve_kernel.cuh"
#include "solve_kernel_v2.cuh"
#include "solve_kernel_big.cuh"
#include "target_batch.cuh"

namespace
{
thread_local std::string g_err;

eb_status fail(eb_status st, const std::string& msg)
{
  g_err = msg;
  return st;
}

#define EB_CUDA(expr)                                                                                   \
  do                                                                                                    \
  {                                                                                                     \
    cudaError_t e__ = (expr);                                                                           \
    if (e__ != cudaSuccess)                                                                             \
    {                                                                                                   \
      const eb_status st__ = (e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver ||         \
                              e__ == cudaErrorInvalidDevice) ?                                          \
                                 EB_ERR_NO_DEVICE :                                                     \
                                 EB_ERR_CUDA;                                                           \
      return fail(st__, std::string(#expr) + ": " + cudaGetErrorName(e__) + ": " + cudaGetErrorString(e__)); \
    }                                                                                                   \
  } while (0)

// NVTX range around a C-ABI call (SURVEY.md section 5: tracing hook)
struct NvtxRange
{
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
#define EB_TRACE(name) NvtxRange nvtx_range__(name)

// grid.hpp:61-64
unsigned axis_length(double lower, double upper, double resolution)
{
  return static_cast<unsigned>(std::round((upper - lower) / resolution));
}

// numerics.hpp:67-70
bool almost_equal(double a, double b) { return std::fabs(a - b) < 1.0e-12; }

// configTarget's accumulated grid coordinates (ergodic_control.hpp:394-407)
std::vector<double> accumulated_axis(int n, double resolution, double start = 0.0)
{
  std::vector<double> v(n);
  double x = start;
  for (int i = 0; i < n; i++)
  {
    v[i] = x;
    x += resolution;
  }
  return v;
}
}  // namespace

// ---------------------------------------------------------------------------
// phi_k plan
// ---------------------------------------------------------------------------
// The mirror fold of the tile kernel (phik_dmma.cuh) is taken when the cosine table of
// the plan's grid is symmetric to this tolerance; it bounds the fold's coefficient error.
constexpr double kFoldTol = 1.0e-10;

struct eb_phik_plan
{
  int device = 0, nx = 0, ny = 0, nb = 0, algo = 0;  // ny = rows held by this plan
  int ny_total = 0, row_begin = 0;
  int ld = 32;  // leading dimension of the cosine tables, T and the raw block: 32, or nb rounded up to 32 (nb > 32)
  double resolution = 0, lx = 0, ly = 0;
  cudaStream_t stream = nullptr;
  double *d_xs = nullptr, *d_ys = nullptr;  // grid coordinates
  double *d_cx = nullptr, *d_cy = nullptr;  // cosine tables [n][32]
  double* d_cxp = nullptr;                  // C_x re-laid for the DMMA tile kernel
  double* d_cxpf = nullptr;                 // ... for the mirror-folded tile kernel (left half, even | odd orders)
  double *d_cxt = nullptr, *d_cxtf = nullptr;  // C_x re-laid for the TMA tile kernel (phik_tma.cuh), unfolded / folded
  bool fold = false;                        // the grid's cosine tables are mirror-symmetric to <= kFoldTol
  double fold_dev = 0.0;                    // measured max |C_x[j][k] - (-1)^k C_x[nx-1-j][k]|
  double *d_T = nullptr;                    // stage-1 result [ny][32]
  double *d_parts = nullptr;                // partial 32x32 blocks
  double *d_phik = nullptr, *d_sum = nullptr;  // staging for the _host call
  double* d_phi_stage = nullptr;               // device copy of the density for the _host call (kept between calls)
  unsigned int* d_done = nullptr;              // arrival counter of the TMA kernel's fused final sum
  const eb::PhikTmaPeer* peer = nullptr;       // set for the duration of eb_phik_execute_allreduce_dev
  int max_parts = 0;
  long long launches = 0;
  // nb > 32 on large grids: the 32-order TMA tile kernel once per (by, bx) block of orders; per-block tables
  std::vector<double*> w_cxt, w_cxtf, w_cy;  // [nblk]: C_x re-laid (unfolded / folded), C_y [ny][32]
  double* d_wraw = nullptr;                  // [nblk][nblk][1024] raw blocks
};

extern "C" {

int eb_abi_version(void) { return EB_ABI_VERSION; }
const char* eb_last_error(void) { return g_err.c_str(); }

int eb_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess)
  {
    cudaGetLastError();
    return 0;
  }
  return n;
}

void eb_config_defaults(eb_config* cfg, int model)
{
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->model = model;
  cfg->batch = 1;
  cfg->device = 0;
  cfg->dt = 0.1;           // config/explore_*.yaml ec_dt
  cfg->horizon = 5.0;      // ec_horizon
  cfg->resolution = 0.1;   // target_resolution
  cfg->expl_weight = 1.0;  // expl_weight
  cfg->num_basis = 10;
  cfg->buffer_size = 1000000;
  cfg->batch_size = 100;
  // Rinv = diag(1 / control_weights) (exploration_omni_node.cpp:161-164,
  // exploration_cart_node.cpp:156-159)
  cfg->Rinv[0] = 1.0;
  cfg->Rinv[4] = model == EB_MODEL_OMNI ? 1.0 : 0.0;
  cfg->Rinv[8] = 2.0;
  cfg->umin[0] = -1.0;
  cfg->umax[0] = 1.0;
  cfg->umin[1] = model == EB_MODEL_OMNI ? -1.0 : 0.0;
  cfg->umax[1] = model == EB_MODEL_OMNI ? 1.0 : 0.0;
  cfg->umin[2] = -2.0;
  cfg->umax[2] = 2.0;
  cfg->barrier_weight = 25.0;  // ergodic_control.hpp:457
  cfg->barrier_eps = 0.05;     // ergodic_control.hpp:458
  cfg->seed = 0xE16C0D1Cull;
}

eb_status eb_phik_plan_create(int device, int nx, int ny, double resolution, double lx, double ly, int nb,
                              eb_phik_plan** out)
{
  return eb_phik_plan_create_rows(device, nx, ny, 0, ny, resolution, lx, ly, nb, out);
}

eb_status eb_phik_plan_create_rows(int device, int nx, int ny_total, int row_begin, int ny, double resolution,
                                   double lx, double ly, int nb, eb_phik_plan** out)
{
  return eb_phik_plan_create_ex(device, nx, ny_total, row_begin, ny, resolution, lx, ly, nb, 0.0, 0.0, out);
}

eb_status eb_phik_plan_create_ex(int device, int nx, int ny_total, int row_begin, int ny, double resolution, double lx,
                                 double ly, int nb, double x_first, double y_first, eb_phik_plan** out)
{
  EB_TRACE("eb_phik_plan_create");
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_plan_create: out is NULL");
  *out = nullptr;
  if (nx < 1 || ny < 1 || nb < 1 || nb > EB_MAX_NUM_BASIS)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_plan_create: need nx, ny >= 1 and 1 <= nb <= " + std::to_string(EB_MAX_NUM_BASIS));
  if (row_begin < 0 || row_begin + ny > ny_total)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_plan_create_rows: row range outside the grid");
  if (!(lx > 0.0) || !(ly > 0.0) || !(resolution > 0.0))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_plan_create: lx, ly, resolution must be positive");
  EB_CUDA(cudaSetDevice(device));
  eb_phik_plan* p = new (std::nothrow) eb_phik_plan();
  if (!p) return fail(EB_ERR_CUDA, "out of host memory");
  p->device = device;
  p->nx = nx;
  p->ny = ny;
  p->ny_total = ny_total;
  p->row_begin = row_begin;
  p->nb = nb;
  p->resolution = resolution;
  p->lx = lx;
  p->ly = ly;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  p->max_parts = std::min(std::max(1, sms), eb::kPtGroup * eb::kPtMaxGroups);
  const std::vector<double> xs = accumulated_axis(nx, resolution, x_first);
  const std::vector<double> ys_all = accumulated_axis(row_begin + ny, resolution, y_first);
  const std::vector<double> ys(ys_all.begin() + row_begin, ys_all.end());
  auto cleanup = [&](eb_status st) {
    eb_phik_plan_destroy(p);
    return st;
  };
#define EB_CUDA_P(expr)                                                                      \
  do                                                                                         \
  {                                                                                          \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return cleanup(fail(EB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__))); \
  } while (0)
  EB_CUDA_P(cudaMalloc(&p->d_xs, sizeof(double) * nx));
  EB_CUDA_P(cudaMalloc(&p->d_ys, sizeof(double) * ny));
  const int ld = eb::phik_ld(nb);  // 32, or nb rounded up to 32 for the wide (nb > 32) route
  const bool wide = nb > 32;       // simple pair only: the tile kernels are built around 32 x 32 coefficient blocks
  p->ld = ld;
  EB_CUDA_P(cudaMalloc(&p->d_cx, sizeof(double) * (size_t)nx * ld));
  EB_CUDA_P(cudaMalloc(&p->d_cy, sizeof(double) * (size_t)ny * ld));
  EB_CUDA_P(cudaMalloc(&p->d_T, sizeof(double) * (size_t)ny * ld));
  // per-CTA blocks + the per-group sums of the TMA kernel's two-level final sum (wide: the one ld x ld raw block)
  EB_CUDA_P(cudaMalloc(&p->d_parts, std::max(sizeof(double) * (size_t)ld * ld,
                                             sizeof(double) * 1024 * (size_t)(p->max_parts + eb::kPtMaxGroups))));
  EB_CUDA_P(cudaMalloc(&p->d_phik, sizeof(double) * (size_t)std::max(1024, nb * nb)));
  EB_CUDA_P(cudaMalloc(&p->d_sum, sizeof(double)));
  EB_CUDA_P(cudaMalloc(&p->d_done, sizeof(unsigned int) * (1 + eb::kPtMaxGroups)));
  EB_CUDA_P(cudaMemset(p->d_done, 0, sizeof(unsigned int) * (1 + eb::kPtMaxGroups)));
  EB_CUDA_P(cudaMemcpy(p->d_xs, xs.data(), sizeof(double) * nx, cudaMemcpyHostToDevice));
  EB_CUDA_P(cudaMemcpy(p->d_ys, ys.data(), sizeof(double) * ny, cudaMemcpyHostToDevice));
  // basis.cpp:85: cos(k * (PI / l) * x)
  eb::cos_table_kernel<<<(unsigned)(((size_t)nx * ld + 255) / 256), 256>>>(p->d_xs, nx, eb::kPi / lx, nb, ld, 0, p->d_cx);
  eb::cos_table_kernel<<<(unsigned)(((size_t)ny * ld + 255) / 256), 256>>>(p->d_ys, ny, eb::kPi / ly, nb, ld, 0, p->d_cy);
  p->launches += 2;
  if (wide && (long long)nx * ny >= (1 << 18) && eb::phik_tma_supported(nx, ny) && eb::phik_tma_encoder())
  {
    // large grid: the 32-order TMA tile kernel runs once per (by, bx) block of orders -- tables per block of 32 orders
    const int nblk = ld / 32;
    if (eb::phik_fold_shape_ok(nx))
    {
      double dev = 0.0;  // symmetry of the table on THIS grid over all nb orders (as below for nb <= 32)
      for (int j = 0; j < nx / 2; j++)
        for (int k = 0; k < nb; k++)
        {
          const double f = (double)k * (eb::kPi / lx);
          const double a = std::cos(f * xs[j]), b = std::cos(f * xs[nx - 1 - j]);
          dev = std::max(dev, std::fabs(a - ((k & 1) ? -b : b)));
        }
      p->fold_dev = dev;
      p->fold = dev <= kFoldTol;
    }
    double* d_tmp = nullptr;  // one block of C_x, [nx][32]
    EB_CUDA_P(cudaMalloc(&d_tmp, sizeof(double) * (size_t)nx * 32));
    EB_CUDA_P(cudaMalloc(&p->d_wraw, sizeof(double) * 1024 * (size_t)nblk * nblk));
    const int rows_u = eb::phik_tma_cx_rows(nx, false), rows_f = eb::phik_tma_cx_rows(nx / 2, true);
    cudaError_t we = cudaSuccess;
    for (int b = 0; b < nblk && we == cudaSuccess; b++)
    {
      double *cxt = nullptr, *cxtf = nullptr, *cyb = nullptr;
      eb::cos_table_kernel<<<(unsigned)(((size_t)nx * 32 + 255) / 256), 256>>>(p->d_xs, nx, eb::kPi / lx, nb, 32, 32 * b, d_tmp);
      we = cudaMalloc(&cxt, sizeof(double) * (size_t)rows_u * eb::kPdPitch);
      p->w_cxt.push_back(cxt);
      if (we == cudaSuccess)
        eb::phik_tma_permute_cx<<<(rows_u * eb::kPdPitch + 255) / 256, 256>>>(d_tmp, nx, rows_u, 0, cxt);
      if (we == cudaSuccess && p->fold)
      {
        we = cudaMalloc(&cxtf, sizeof(double) * (size_t)rows_f * eb::kPdPitch);
        if (we == cudaSuccess)
          eb::phik_tma_permute_cx<<<(rows_f * eb::kPdPitch + 255) / 256, 256>>>(d_tmp, nx / 2, rows_f, 1, cxtf);
      }
      p->w_cxtf.push_back(cxtf);
      if (we == cudaSuccess) we = cudaMalloc(&cyb, sizeof(double) * (size_t)ny * 32);
      p->w_cy.push_back(cyb);
      if (we == cudaSuccess)
        eb::cos_table_kernel<<<(unsigned)(((size_t)ny * 32 + 255) / 256), 256>>>(p->d_ys, ny, eb::kPi / ly, nb, 32, 32 * b, cyb);
      p->launches += 3 + (p->fold ? 1 : 0);
    }
    if (we == cudaSuccess) we = cudaDeviceSynchronize();
    cudaFree(d_tmp);
    EB_CUDA_P(we);
  }
  if (!wide && eb::phik_dmma_supported(nx, ny))
  {
    // room for the last column span's padding chunks (span <= nchunks)
    const int rows_padded = 2 * ((nx + eb::kPdChunk - 1) / eb::kPdChunk) * eb::kPdChunk;
    EB_CUDA_P(cudaMalloc(&p->d_cxp, sizeof(double) * (size_t)rows_padded * eb::kPdPitch));
    eb::phik_permute_cx<<<(rows_padded * eb::kPdPitch + 255) / 256, 256>>>(p->d_cx, nx, rows_padded, 0, p->d_cxp);
    p->launches += 1;
    if (eb::phik_fold_shape_ok(nx))
    {
      // symmetry of the table on THIS grid (accumulated coordinates, caller's lx), basis.cpp:85 arithmetic
      double dev = 0.0;
      for (int j = 0; j < nx / 2; j++)
        for (int k = 0; k < nb; k++)
        {
          const double f = (double)k * (eb::kPi / lx);
          const double a = std::cos(f * xs[j]), b = std::cos(f * xs[nx - 1 - j]);
          dev = std::max(dev, std::fabs(a - ((k & 1) ? -b : b)));
        }
      p->fold_dev = dev;
      p->fold = dev <= kFoldTol;
      if (p->fold)
      {
        const int chunk = eb::PdGeom<true>::kChunk;
        const int rows_f = 2 * ((nx / 2 + chunk - 1) / chunk) * chunk;
        EB_CUDA_P(cudaMalloc(&p->d_cxpf, sizeof(double) * (size_t)rows_f * eb::kPdPitch));
        eb::phik_permute_cx<<<(rows_f * eb::kPdPitch + 255) / 256, 256>>>(p->d_cx, nx / 2, rows_f, 1, p->d_cxpf);
        p->launches += 1;
      }
    }
  }
  if (!wide && eb::phik_tma_supported(nx, ny))
  {
    const int rows_u = eb::phik_tma_cx_rows(nx, false);
    EB_CUDA_P(cudaMalloc(&p->d_cxt, sizeof(double) * (size_t)rows_u * eb::kPdPitch));
    eb::phik_tma_permute_cx<<<(rows_u * eb::kPdPitch + 255) / 256, 256>>>(p->d_cx, nx, rows_u, 0, p->d_cxt);
    p->launches += 1;
    if (p->fold)
    {
      const int rows_f = eb::phik_tma_cx_rows(nx / 2, true);
      EB_CUDA_P(cudaMalloc(&p->d_cxtf, sizeof(double) * (size_t)rows_f * eb::kPdPitch));
      eb::phik_tma_permute_cx<<<(rows_f * eb::kPdPitch + 255) / 256, 256>>>(p->d_cx, nx / 2, rows_f, 1, p->d_cxtf);
      p->launches += 1;
    }
  }
  EB_CUDA_P(cudaGetLastError());
  EB_CUDA_P(cudaDeviceSynchronize());
#undef EB_CUDA_P
  *out = p;
  return EB_OK;
}

void eb_phik_plan_destroy(eb_phik_plan* p)
{
  if (!p) return;
  cudaSetDevice(p->device);
  cudaFree(p->d_xs);
  cudaFree(p->d_ys);
  cudaFree(p->d_cx);
  cudaFree(p->d_cy);
  cudaFree(p->d_cxp);
  cudaFree(p->d_cxpf);
  cudaFree(p->d_cxt);
  cudaFree(p->d_cxtf);
  cudaFree(p->d_T);
  cudaFree(p->d_parts);
  cudaFree(p->d_phik);
  cudaFree(p->d_sum);
  cudaFree(p->d_phi_stage);
  cudaFree(p->d_done);
  for (double* q : p->w_cxt) cudaFree(q);
  for (double* q : p->w_cxtf) cudaFree(q);
  for (double* q : p->w_cy) cudaFree(q);
  cudaFree(p->d_wraw);
  delete p;
}

eb_status eb_phik_plan_set_stream(eb_phik_plan* p, void* s)
{
  if (!p) return fail(EB_ERR_INVALID_ARGUMENT, "plan is NULL");
  p->stream = static_cast<cudaStream_t>(s);
  return EB_OK;
}

eb_status eb_phik_plan_set_algo(eb_phik_plan* p, int algo)
{
  if (!p) return fail(EB_ERR_INVALID_ARGUMENT, "plan is NULL");
  if (algo < 0 || algo > 5)
    return fail(EB_ERR_INVALID_ARGUMENT, "algo must be 0 (auto), 1 (simple), 2 / 3 (register-streamed DMMA tiles, with / without "
                                         "the mirror fold) or 4 / 5 (TMA-staged DMMA tiles, with / without the mirror fold)");
  if (algo >= 2 && p->nb > 32)
    return fail(EB_ERR_UNSUPPORTED, "num_basis > 32: algo 0 (auto: the TMA tile kernel per block of 32 x 32 orders on large grids, "
                                    "else the simple pair) or 1 (simple pair)");
  if ((algo == 2 || algo == 3) && !eb::phik_dmma_supported(p->nx, p->ny))
    return fail(EB_ERR_UNSUPPORTED, "the register-streamed DMMA phi_k kernel needs nx % 4 == 0 and nx >= 128");
  if (algo >= 4 && (!eb::phik_tma_supported(p->nx, p->ny) || !eb::phik_tma_encoder()))
    return fail(EB_ERR_UNSUPPORTED, "the TMA phi_k kernel needs an even nx >= 64 and a driver with cuTensorMapEncodeTiled");
  p->algo = algo;
  return EB_OK;
}

long long eb_phik_launch_count(const eb_phik_plan* p) { return p ? p->launches : 0; }

eb_status eb_phik_plan_fold(const eb_phik_plan* p, int* fold, double* deviation)
{
  if (!p) return fail(EB_ERR_INVALID_ARGUMENT, "plan is NULL");
  if (fold) *fold = p->fold ? 1 : 0;
  if (deviation) *deviation = p->fold_dev;
  return EB_OK;
}

static eb_status phik_execute(eb_phik_plan* p, const double* phi_dev, double* phik_dev, double* phi_sum_dev,
                              double* raw_dev);

eb_status eb_phik_execute_dev(eb_phik_plan* p, const double* phi_dev, double* phik_dev, double* phi_sum_dev)
{
  if (!p || !phi_dev || !phik_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_execute_dev: NULL argument");
  return phik_execute(p, phi_dev, phik_dev, phi_sum_dev, nullptr);
}

eb_status eb_phik_execute_raw_dev(eb_phik_plan* p, const double* phi_dev, double* raw_dev)
{
  if (!p || !phi_dev || !raw_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_execute_raw_dev: NULL argument");
  return phik_execute(p, phi_dev, nullptr, nullptr, raw_dev);
}

static eb_status phik_execute(eb_phik_plan* p, const double* phi_dev, double* phik_dev, double* phi_sum_dev,
                              double* raw_dev)
{
  EB_TRACE("eb_phik_execute");
  EB_CUDA(cudaSetDevice(p->device));
  int algo = p->algo;
  if (p->nb > 32 && p->d_wraw && algo != 1 && (reinterpret_cast<uintptr_t>(phi_dev) & 15) == 0)
  {
    // wide route on a large grid: the TMA tile kernel once per (by, bx) block of 32 x 32 orders (raw blocks), then
    // the assembly + normalisation
    const int ld = p->ld, nblk = ld / 32;
    for (int by = 0; by < nblk; by++)
      for (int bx = 0; bx < nblk; bx++)
      {
        const int nbm = std::min(32, p->nb - 32 * std::min(by, bx));  // orders present in the wider of the two blocks
        const eb::PhikTmaOut out{ p->d_done, nbm, nullptr, nullptr, p->d_wraw + 1024 * ((size_t)by * nblk + bx), nullptr };
        const int np = eb::phik_tma_launch(phi_dev, p->nx, p->ny, p->fold ? p->w_cxtf[bx] : p->w_cxt[bx], p->w_cy[by],
                                           p->d_parts, p->max_parts, p->fold, out, p->stream);
        if (np < 0) return fail(EB_ERR_CUDA, std::string("phik_tma_launch (wide): ") + cudaGetErrorString(cudaGetLastError()));
        p->launches += 1;
      }
    eb::phik_assemble_wide<<<(ld * ld + 255) / 256, 256, 0, p->stream>>>(p->d_wraw, p->nb, nblk, ld, phik_dev, phi_sum_dev, raw_dev);
    p->launches += 1;
    EB_CUDA(cudaGetLastError());
    return EB_OK;
  }
  if (p->nb > 32)
  {
    // wide route: the simple pair over blocks of 32 orders, then the normalisation
    const int ld = p->ld;
    eb::phik_stage1_simple<<<dim3(p->ny, ld / 32), 256, 0, p->stream>>>(phi_dev, p->nx, p->d_cx, ld, p->d_T);
    eb::phik_stage2_simple<<<dim3(p->nb, ld / 32), 256, 0, p->stream>>>(p->d_T, p->ny, p->d_cy, ld, p->d_parts);
    eb::phik_finalize_wide<<<(ld * ld + 255) / 256, 256, 0, p->stream>>>(p->d_parts, p->nb, ld, phik_dev, phi_sum_dev, raw_dev);
    p->launches += 3;
    EB_CUDA(cudaGetLastError());
    return EB_OK;
  }
  const bool big = (long long)p->nx * p->ny >= (1 << 18);
  if (algo == 0)
    algo = (big && eb::phik_tma_supported(p->nx, p->ny) && eb::phik_tma_encoder() && (reinterpret_cast<uintptr_t>(phi_dev) & 15) == 0) ? 4 :
           (big && eb::phik_dmma_supported(p->nx, p->ny))                                                                        ? 2 :
                                                                                                                                   1;
  int nparts = 1;
  const bool fold = (algo == 2 || algo == 4) && p->fold;
  if (algo >= 4)
  {
    // one launch: the last CTA to finish does the final sum (no separate phik_finalize)
    const eb::PhikTmaOut out{ p->d_done, p->nb, phik_dev, phi_sum_dev, raw_dev, p->peer };
    nparts = eb::phik_tma_launch(phi_dev, p->nx, p->ny, fold ? p->d_cxtf : p->d_cxt, p->d_cy, p->d_parts, p->max_parts, fold,
                                 out, p->stream);
    if (nparts < 0) return fail(EB_ERR_CUDA, std::string("phik_tma_launch: ") + cudaGetErrorString(cudaGetLastError()));
    p->launches += 1;
    return EB_OK;
  }
  else if (algo >= 2)
  {
    nparts = eb::phik_dmma_launch(phi_dev, p->nx, p->ny, fold ? p->d_cxpf : p->d_cxp, p->d_cy, p->d_parts, p->max_parts,
                                  fold, p->stream);
    if (nparts < 0) return fail(EB_ERR_CUDA, std::string("phik_dmma_launch: ") + cudaGetErrorString(cudaGetLastError()));
    p->launches += 1;
  }
  else
  {
    eb::phik_stage1_simple<<<p->ny, 256, 0, p->stream>>>(phi_dev, p->nx, p->d_cx, eb::kPhikLd, p->d_T);
    eb::phik_stage2_simple<<<32, 256, 0, p->stream>>>(p->d_T, p->ny, p->d_cy, eb::kPhikLd, p->d_parts);
    p->launches += 2;
  }
  eb::phik_finalize<<<1, 1024, 0, p->stream>>>(p->d_parts, nparts, p->nb, fold ? 1 : 0, phik_dev, phi_sum_dev, raw_dev);
  p->launches += 1;
  EB_CUDA(cudaGetLastError());
  return EB_OK;
}

eb_status eb_phik_execute_host(eb_phik_plan* p, const double* phi, double* phik, double* phi_sum)
{
  EB_TRACE("eb_phik_execute_host");
  if (!p || !phi || !phik) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_execute_host: NULL argument");
  EB_CUDA(cudaSetDevice(p->device));
  const size_t bytes = sizeof(double) * (size_t)p->nx * p->ny;
  if (!p->d_phi_stage) EB_CUDA(cudaMalloc(&p->d_phi_stage, bytes));  // once per plan: a map update reuses it
  double* const d_phi = p->d_phi_stage;
  cudaError_t e = cudaMemcpyAsync(d_phi, phi, bytes, cudaMemcpyHostToDevice, p->stream);
  eb_status st = EB_OK;
  if (e == cudaSuccess) st = eb_phik_execute_dev(p, d_phi, p->d_phik, p->d_sum);
  if (e == cudaSuccess && st == EB_OK)
    e = cudaMemcpyAsync(phik, p->d_phik, sizeof(double) * p->nb * p->nb, cudaMemcpyDeviceToHost, p->stream);
  if (e == cudaSuccess && st == EB_OK && phi_sum)
    e = cudaMemcpyAsync(phi_sum, p->d_sum, sizeof(double), cudaMemcpyDeviceToHost, p->stream);
  if (e == cudaSuccess && st == EB_OK) e = cudaStreamSynchronize(p->stream);
  if (st != EB_OK) return st;
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_phik_execute_host: ") + cudaGetErrorString(e));
  return EB_OK;
}

eb_status eb_phik_from_grid_host(int device, const double* phi, int nx, int ny, double resolution, double lx,
                                 double ly, int nb, double* phik, double* phi_sum)
{
  eb_phik_plan* p = nullptr;
  eb_status st = eb_phik_plan_create(device, nx, ny, resolution, lx, ly, nb, &p);
  if (st != EB_OK) return st;
  st = eb_phik_execute_host(p, phi, phik, phi_sum);
  eb_phik_plan_destroy(p);
  return st;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// controller
// ---------------------------------------------------------------------------
// arguments of one fused-gather launch (peer_gather.cuh)
struct PeerLaunch
{
  int n_peer = 0;
  double* u0_peer[eb::kMaxPeers] = {};
  unsigned long long* flag_peer[eb::kMaxPeers] = {};
  unsigned long long flag_value = 0;
  unsigned int* done_counter = nullptr;
  const unsigned long long* my_flags = nullptr;
  unsigned long long need = 0;
};

struct eb_controller
{
  eb_config cfg{};
  int N = 0, K = 0, nb = 0, B = 0;
  cudaStream_t stream = nullptr;
  double* d_ut[2] = { nullptr, nullptr };  // ping-pong control signal, [B][N][3]
  int cur = 0;                             // d_ut[cur] is ut_
  double* d_pose = nullptr;                // [B][3], pose_ of the last control()
  double* d_hist = nullptr;                // replay buffer [cap][B][3]
  // Fourier-frame cosines of the stored states [cap][B][2] (what the solve kernels need from the buffer): rows
  // [0, cos_count) are valid for the frame cos_key = {xmin, ymin, 1 / lx, 1 / ly}; brought up to date before a launch
  double* d_hist_cos = nullptr;
  long long cos_count = 0;
  double cos_key[4] = { 0.0, 0.0, 0.0, 0.0 };
  long long hist_cap = 0, mem_count = 0;
  double *d_phik = nullptr, *d_lamk = nullptr;
  double *d_u0 = nullptr, *d_metric = nullptr, *d_ck = nullptr, *d_x = nullptr;
  double* d_xt = nullptr;                  // [B][N][3] staging of eb_opt_traj_host (allocated on first use, kept)
  double* d_big_scratch = nullptr;         // num_basis > 32: [big_rows][K], one row per resident CTA of solve_kernel_big
  int big_rows = 0;
  int *d_mem_idx_in = nullptr, *d_mem_idx_out = nullptr;
  int *h_fault = nullptr, *d_fault = nullptr;  // pinned + mapped: the kernels set it, the host reads it after a sync
  int last_idx_count = 0;
  double lx = 0.0, ly = 0.0;  // basis_.lx_, basis_.ly_ (0, 0 at construction :208)
  double map_pos[2] = { 0.0, 0.0 };
  std::vector<double> gauss_mu, gauss_sigma;  // target_
  eb_phik_plan* plan = nullptr;               // cached for the current extent
  double* d_phi_grid = nullptr;
  size_t phi_grid_cells = 0;
  double* d_gauss = nullptr;
  int gauss_cap = 0;
  unsigned long long call = 0;
  long long launches = 0;
  bool have_pose = false;
  bool keep_ck = true;  // store the c_k by-product of every control() (eb_get_ck)
  const struct PeerLaunch* peer = nullptr;  // set for the duration of eb_control_dev_gather
  // per-instance targets (eb_*_batch calls): switched on by the first of them; the shared target calls refuse after it.
  // Every stored row's cosines (d_hist_cos) are then kept valid for its instance's current frame.
  bool per_inst = false;
  bool frames_set = false;          // a configure or eb_set_phik_batch_dev has given every instance a frame
  double* d_phik_b = nullptr;       // [B][K]
  double* d_frames = nullptr;       // [B][eb::kFrDoubles]
  double *d_gmu = nullptr, *d_gsig = nullptr;  // [B][gmax][2]
  int* d_gcount = nullptr;          // [B]
  int gmax = 0;
  double* d_bounds = nullptr;       // [B][4] staging of eb_control_batch_host
  // map-derived targets per instance (eb_set_map_targets_batch_*, map_target_batch.cuh)
  eb::MapBatchDesc* h_mb_desc = nullptr;  // [B] pinned: the maps of a call
  eb::MapBatchDesc* d_mb_desc = nullptr;  // [B]
  cudaEvent_t mb_staged = nullptr;        // recorded after the copies out of the pinned buffers
  double* d_mb_slots = nullptr;           // [units][K] raw blocks
  long long mb_slot_units = 0;
  unsigned* d_mb_arrive = nullptr;        // [B] arrival counters (zero between launches)
  signed char* h_mb_cells = nullptr;      // pinned staging of the _host call's maps
  signed char* d_mb_cells = nullptr;
  size_t mb_cells_bytes = 0;
  int mb_grid = 0;                        // resident CTAs of map_target_batch_kernel on the device
  // kept blocks of eb_set_map_targets_from_grid_batch: instance i's raw block of unit v of its map is slot
  // kb_slot0[i] + v of d_kb (kb_cap[i] slots reserved); kb_key[i] says which map the blocks belong to
  struct KeptKey
  {
    unsigned long long grid = 0, map = 0;  // grid batch serial (0: no kept blocks), map serial in it
    unsigned nx = 0, ny = 0;
    double res = 0.0;
  };
  double* d_kb = nullptr;
  std::vector<int> kb_slot0, kb_cap;
  std::vector<KeptKey> kb_key;
  eb::MapKept* h_mb_kept = nullptr;  // [B] pinned: the recomputed units of a call
  eb::MapKept* d_mb_kept = nullptr;
  // safe control tick (eb_control_safe_batch_*, safe_control.cuh)
  int* d_safe_list = nullptr;      // [1 + B]: the count of failing robots, then their indices
  int* d_safe_branch = nullptr;    // [B] staging of the _host call
  double* d_safe_vb = nullptr;     // [B][3] staging of the _host call
  int safe_grid = 0;               // resident CTAs of dwa_fallback_kernel with this horizon

  // device alias of a page-locked host buffer (nullptr for pageable memory);
  // looked up on every call -- a cached answer could outlive the allocation
  static double* mapped(const void* host)
  {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, host) != cudaSuccess)
    {
      cudaGetLastError();
      return nullptr;
    }
    return (a.type == cudaMemoryTypeHost && a.devicePointer) ? static_cast<double*>(a.devicePointer) : nullptr;
  }
};

// batches up to this size take the zero-copy host path (EB_ZEROCOPY_MAX_BATCH overrides; 0 disables)
inline int zero_copy_max_batch()
{
  static const int v = [] {
    const char* e = std::getenv("EB_ZEROCOPY_MAX_BATCH");
    return e ? std::atoi(e) : 16384;
  }();
  return v;
}

// EB_REPLAY_COS=0: the solve kernels derive the replay states' cosines themselves (no cached rows), for A/B runs
inline bool replay_cos_cache()
{
  static const bool v = [] {
    const char* e = std::getenv("EB_REPLAY_COS");
    return !e || std::atoi(e) != 0;
  }();
  return v;
}

namespace
{
// V2: solve_kernel2 (solve_kernel_v2.cuh), else solve_kernel (solve_kernel.cuh)
template <int MODEL, int NB, bool V2, bool PER_INST = false>
struct SolveLaunch
{
  static constexpr int kWide = []() constexpr {
    if constexpr (V2)
      return eb::Solve2Cfg<NB>::kWideWarps;
    else
      return eb::SolveCfg<NB>::kWideWarps;
  }();
  static size_t smem(int N, int warps = eb::kSolveWarps)
  {
    if constexpr (V2)
      return eb::solve2_smem_bytes<NB>(N, warps);
    else
      return eb::solve_smem_bytes(eb::SolveCfg<NB>::kTabDoubles, eb::SolveCfg<NB>::kFields, (N + 31) / 32, warps);
  }
  template <int WARPS>
  static cudaError_t launch_w(const eb::SolveParams& p, cudaStream_t s)
  {
    const size_t bytes = smem(p.N, WARPS);
    // the attribute is per device: remember what has been set, per instantiation and device
    static size_t configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    auto kernel = [] {
      if constexpr (V2)
        return eb::solve_kernel2<MODEL, NB, WARPS, PER_INST>;
      else
        return eb::solve_kernel<MODEL, NB, WARPS, PER_INST>;
    }();
    if (bytes > configured[dev & 63])
    {
      cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      if (e != cudaSuccess) return e;
      configured[dev & 63] = bytes;
    }
    const int grid = (p.B + WARPS - 1) / WARPS;
    // Programmatic dependent launch: consecutive control() steps on one stream are kernel -> kernel dependencies; the
    // next step's CTAs may be placed while this step's last ones drain (every global access of the kernel sits behind
    // its griddepcontrol.wait, so the data dependency is the stream's).
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)(WARPS * 32));
    cfg.dynamicSmemBytes = bytes;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, p);
  }
  static cudaError_t launch(const eb::SolveParams& p, cudaStream_t s)
  {
    // a batch that fits one wave of wide CTAs (one per SM) starts all of an SM's instances together
    static const int sms = [] {
      int dev = 0, n = 148;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
      return n;
    }();
    static const bool wide_ok = [] {
      const char* e = std::getenv("EB_SOLVE_WIDE");
      return !e || std::atoi(e) != 0;
    }();
    if (wide_ok && p.n_peer == 0 && p.B <= sms * kWide && p.B > sms * eb::kSolveWarps && smem(p.N, kWide) + 2048 <= wide_limit())
      return launch_w<kWide>(p, s);
    return launch_w<eb::kSolveWarps>(p, s);
  }
  static size_t wide_limit()
  {
    static const size_t lim = [] {
      int dev = 0, v = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
      return (size_t)v;
    }();
    return lim;
  }
};

// num_basis > 32: a CTA per instance (solve_kernel_big.cuh), persistent over the batch; one scratch row per CTA
template <int MODEL, bool PER_INST>
cudaError_t launch_solve_big(const eb::SolveParams& p, cudaStream_t s)
{
  const size_t bytes = eb::solve_big_smem_bytes(p.nb, p.N);
  static size_t configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (bytes > configured[dev & 63])
  {
    cudaError_t e = cudaFuncSetAttribute(eb::solve_kernel_big<MODEL, PER_INST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    configured[dev & 63] = bytes;
  }
  if (!p.big_scratch || p.big_rows < 1) return cudaErrorInvalidValue;
  const int grid = std::min(p.B, p.big_rows);
  eb::solve_kernel_big<MODEL, PER_INST><<<grid, eb::kBigThreads, bytes, s>>>(p, p.big_scratch);
  return cudaGetLastError();
}

// resident CTAs of solve_kernel_big on the current device (= scratch rows worth allocating)
int solve_big_resident(int nb, int N)
{
  const size_t bytes = eb::solve_big_smem_bytes(nb, N);
  int dev = 0, sms = 148, per_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaFuncSetAttribute(eb::solve_kernel_big<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eb::solve_kernel_big<0>, eb::kBigThreads, bytes) != cudaSuccess)
  {
    cudaGetLastError();
    per_sm = 1;
  }
  return sms * std::max(1, per_sm);
}

// The solve kernel that serves num_basis `nb` <= 32: f is called with a (stateless) value of its SolveLaunch type.
//   nb <= 8 | <= 10 | <= 12  -> solve_kernel<8 | 10 | 12>
//   13..16 | 17..20 | 21..24 -> solve_kernel2<16 | 20 | 24>
//   25..32                   -> solve_kernel<32>
// nb > 32 runs solve_kernel_big (launch_solve_big).
template <int MODEL, bool PER_INST, class F>
auto with_solve_launch(int nb, F&& f)
{
  if (nb <= 8) return f(SolveLaunch<MODEL, 8, false, PER_INST>{});
  if (nb <= 10) return f(SolveLaunch<MODEL, 10, false, PER_INST>{});
  if (nb <= 12) return f(SolveLaunch<MODEL, 12, false, PER_INST>{});
  if (nb <= 16) return f(SolveLaunch<MODEL, 16, true, PER_INST>{});
  if (nb <= 20) return f(SolveLaunch<MODEL, 20, true, PER_INST>{});
  if (nb <= 24) return f(SolveLaunch<MODEL, 24, true, PER_INST>{});
  return f(SolveLaunch<MODEL, 32, false, PER_INST>{});
}

template <int MODEL, bool PER_INST>
cudaError_t launch_solve_m(const eb::SolveParams& p, cudaStream_t s)
{
  if (p.nb > 32) return launch_solve_big<MODEL, PER_INST>(p, s);
  return with_solve_launch<MODEL, PER_INST>(p.nb, [&](auto L) { return decltype(L)::launch(p, s); });
}

// dynamic shared memory of the solve kernel that serves `nb` (the model does not change it)
size_t solve_smem_for(int nb, int N)
{
  if (nb > 32) return eb::solve_big_smem_bytes(nb, N);
  return with_solve_launch<0, false>(nb, [&](auto L) { return decltype(L)::smem(N); });
}

// per_inst: the kernels read each instance's frame and phi_k row (p.frames, p.phik [B][K])
cudaError_t launch_solve(const eb::SolveParams& p, int model, cudaStream_t s, bool per_inst)
{
  if (per_inst)
    return model == EB_MODEL_OMNI ? launch_solve_m<eb::kModelOmni, true>(p, s) :
                                    launch_solve_m<eb::kModelSimpleCart, true>(p, s);
  return model == EB_MODEL_OMNI ? launch_solve_m<eb::kModelOmni, false>(p, s) :
                                  launch_solve_m<eb::kModelSimpleCart, false>(p, s);
}

eb_status ensure_hist(eb_controller* c, long long need)
{
  if (need <= c->hist_cap) return EB_OK;
  long long cap = std::max<long long>(c->hist_cap ? 2 * c->hist_cap : 128, need);
  {
    // a replay buffer whose full size is a small part of the device memory is allocated once: growing it later
    // means cudaMalloc + copy + cudaFree in the middle of a control loop (and a re-mapping on every peer when the
    // context has peer access enabled)
    size_t free_b = 0, total_b = 0;
    const size_t full = sizeof(double) * (replay_cos_cache() ? 5 : 3) * (size_t)c->B * (size_t)c->cfg.buffer_size;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && full <= free_b / 8) cap = std::max<long long>(cap, c->cfg.buffer_size);
  }
  cap = std::min<long long>(cap, std::max<long long>((long long)c->cfg.buffer_size, need));
  double* nh = nullptr;
  EB_CUDA(cudaMalloc(&nh, sizeof(double) * 3 * (size_t)c->B * (size_t)cap));
  if (c->mem_count > 0)
    EB_CUDA(cudaMemcpyAsync(nh, c->d_hist, sizeof(double) * 3 * (size_t)c->B * (size_t)c->mem_count,
                            cudaMemcpyDeviceToDevice, c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));
  cudaFree(c->d_hist);
  c->d_hist = nh;
  c->hist_cap = cap;
  if (replay_cos_cache() && c->per_inst)
  {
    // per-instance frames: the rows are kept valid as they are written, so they move with the buffer
    double* nc = nullptr;
    EB_CUDA(cudaMalloc(&nc, sizeof(double) * 2 * (size_t)c->B * (size_t)cap));
    if (c->mem_count > 0 && c->d_hist_cos)
    {
      EB_CUDA(cudaMemcpyAsync(nc, c->d_hist_cos, sizeof(double) * 2 * (size_t)c->B * (size_t)c->mem_count,
                              cudaMemcpyDeviceToDevice, c->stream));
      EB_CUDA(cudaStreamSynchronize(c->stream));
    }
    cudaFree(c->d_hist_cos);
    c->d_hist_cos = nc;
  }
  else if (replay_cos_cache())
  {
    cudaFree(c->d_hist_cos);  // re-derived from the rows on the next control() (cos_count = 0)
    c->d_hist_cos = nullptr;
    c->cos_count = 0;
    EB_CUDA(cudaMalloc(&c->d_hist_cos, sizeof(double) * 2 * (size_t)c->B * (size_t)cap));
  }
  return EB_OK;
}

// the cosine rows of every stored state, valid for the current Fourier frame (map origin and extent)
eb_status ensure_hist_cos(eb_controller* c)
{
  if (!c->d_hist_cos || c->mem_count == 0) return EB_OK;
  const double key[4] = { c->map_pos[0], c->map_pos[1], 1.0 / c->lx, 1.0 / c->ly };
  if (std::memcmp(key, c->cos_key, sizeof(key)) != 0)
  {
    std::memcpy(c->cos_key, key, sizeof(key));
    c->cos_count = 0;  // the frame moved (map growth, new origin): every row is re-derived
  }
  if (c->cos_count < c->mem_count)
  {
    const long long n = (c->mem_count - c->cos_count) * (long long)c->B;
    const size_t off = (size_t)c->cos_count * (size_t)c->B;
    eb::hist_cos_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_hist + 3 * off, c->d_hist_cos + 2 * off, n,
                                                                            key[0], key[1], key[2], key[3]);
    EB_CUDA(cudaGetLastError());
    c->launches += 1;
    c->cos_count = c->mem_count;
  }
  return EB_OK;
}

eb_status check_fault(eb_controller* c)
{
  EB_CUDA(cudaStreamSynchronize(c->stream));
  const int f = *static_cast<volatile int*>(c->h_fault);
  if (f)
  {
    *c->h_fault = 0;
    if (f & 2)  // buffer.cpp:84,103: memory_.at(i) throws std::out_of_range
      return fail(EB_ERR_OUT_OF_RANGE, "replay-buffer sample index outside [0, stored states)");
    if (f & 4) return fail(EB_ERR_CUDA, "control(): non-finite state or control signal (NaN / Inf guard)");
    if (f & eb::kFaultTarget)
      return fail(EB_ERR_INVALID_ARGUMENT, "per-instance target: an instance's map extent changed but it has no "
                                           "Gaussians (eb_set_target_gaussians_batch), or its extent is not positive");
    return fail(EB_ERR_INVALID_ARGUMENT, "Invalid twist y-velocity must be 0.");  // cart.hpp:169
  }
  return EB_OK;
}

// the shared target calls on a controller that holds per-instance targets
eb_status refuse_per_inst(const char* call)
{
  return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the controller holds one target per instance (it has "
                                                           "taken an eb_*_batch target call); use the _batch calls");
}

// first per-instance call: phi_k rows and frames (all zero: lx = ly = 0, so the first configure rebuilds every instance)
eb_status ensure_per_inst(eb_controller* c)
{
  if (c->per_inst) return EB_OK;
  EB_CUDA(cudaSetDevice(c->cfg.device));
  const size_t pb = sizeof(double) * (size_t)c->K * c->B, fb = sizeof(double) * eb::kFrDoubles * (size_t)c->B;
  EB_CUDA(cudaMalloc(&c->d_phik_b, pb));
  EB_CUDA(cudaMalloc(&c->d_frames, fb));
  EB_CUDA(cudaMalloc(&c->d_gcount, sizeof(int) * (size_t)c->B));
  EB_CUDA(cudaMalloc(&c->d_bounds, sizeof(double) * 4 * (size_t)c->B));
  EB_CUDA(cudaMemsetAsync(c->d_phik_b, 0, pb, c->stream));
  EB_CUDA(cudaMemsetAsync(c->d_frames, 0, fb, c->stream));
  EB_CUDA(cudaMemsetAsync(c->d_gcount, 0, sizeof(int) * (size_t)c->B, c->stream));
  c->per_inst = true;
  return EB_OK;
}

// configTarget of every instance (bounds_dev [B][4]), or the frames of eb_set_phik_batch_dev (extent_dev [B][2])
eb_status target_batch(eb_controller* c, const double* bounds_dev, const double* extent_dev, int* rebuilt_dev)
{
  eb::TargetBatchParams tp{};
  tp.B = c->B;
  tp.nb = c->nb;
  tp.max_n = c->gmax;
  tp.res = c->cfg.resolution;
  tp.bounds = bounds_dev;
  tp.extent = extent_dev;
  tp.counts = c->d_gcount;
  tp.mu = c->d_gmu;
  tp.sigma = c->d_gsig;
  tp.frames = c->d_frames;
  tp.phik = c->d_phik_b;
  tp.rebuilt = rebuilt_dev;
  tp.hist = c->d_hist;
  tp.hist_cos = c->d_hist_cos;
  tp.mem_count = c->d_hist_cos ? c->mem_count : 0;
  tp.fault = c->d_fault;
  eb::target_batch_kernel<<<c->B, eb::kTbThreads, sizeof(double) * 6 * (size_t)c->gmax, c->stream>>>(tp);
  EB_CUDA(cudaGetLastError());
  c->launches += 1;
  c->frames_set = true;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_create(const eb_config* cfg, eb_controller** out)
{
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: out is NULL");
  *out = nullptr;
  if (!cfg) return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: cfg is NULL");
  if (cfg->model != EB_MODEL_SIMPLE_CART && cfg->model != EB_MODEL_OMNI)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: unknown model (only the 3-twist models SimpleCart and Omni "
                                         "can be driven by ErgodicControl)");
  if (cfg->batch < 1) return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: batch must be >= 1");
  if (cfg->num_basis < 1 || cfg->num_basis > EB_MAX_NUM_BASIS)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: num_basis must be in 1.." + std::to_string(EB_MAX_NUM_BASIS));
  if (!(cfg->dt != 0.0) || !std::isfinite(cfg->horizon / cfg->dt))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: dt must be non-zero and finite");
  const unsigned steps = static_cast<unsigned>(std::abs(cfg->horizon / cfg->dt));  // :199
  if (steps == 1)                                                                   // :212-216
    return fail(EB_ERR_INVALID_ARGUMENT,
                "Need at least two steps in forward simulation. Increase the horizon or decrease the time step.");
  if (steps == 0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_create: horizon / dt gives zero steps");
  if (steps > 4096) return fail(EB_ERR_UNSUPPORTED, "eb_create: more than 4096 horizon steps is not supported");
  if (eb_device_count() < 1) return fail(EB_ERR_NO_DEVICE, "no CUDA device is visible; there is no CPU fallback");
  EB_CUDA(cudaSetDevice(cfg->device));
  {
    // the fused kernel keeps per-step records of the whole horizon in shared memory: refuse horizons that cannot fit
    int optin = 0;
    EB_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device));
    const size_t need = solve_smem_for(static_cast<int>(cfg->num_basis), static_cast<int>(steps));
    if (need > static_cast<size_t>(optin))
      return fail(EB_ERR_UNSUPPORTED, "eb_create: a horizon of " + std::to_string(steps) + " steps with num_basis " +
                                          std::to_string(cfg->num_basis) + " needs " + std::to_string(need) +
                                          " bytes of shared memory per block; the device allows " + std::to_string(optin));
  }

  eb_controller* c = new (std::nothrow) eb_controller();
  if (!c) return fail(EB_ERR_CUDA, "out of host memory");
  c->cfg = *cfg;
  c->N = (int)steps;
  c->nb = (int)cfg->num_basis;
  c->K = c->nb * c->nb;
  c->B = cfg->batch;
  const size_t utb = sizeof(double) * 3 * (size_t)c->N * c->B;
  auto cleanup = [&](eb_status st) {
    eb_destroy(c);
    return st;
  };
#define EB_CUDA_C(expr)                                                                      \
  do                                                                                         \
  {                                                                                          \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return cleanup(fail(EB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__))); \
  } while (0)
  EB_CUDA_C(cudaMalloc(&c->d_ut[0], utb));
  EB_CUDA_C(cudaMalloc(&c->d_ut[1], utb));
  EB_CUDA_C(cudaMemset(c->d_ut[0], 0, utb));  // ut_ = zeros (:201)
  EB_CUDA_C(cudaMemset(c->d_ut[1], 0, utb));
  EB_CUDA_C(cudaMalloc(&c->d_pose, sizeof(double) * 3 * c->B));
  EB_CUDA_C(cudaMemset(c->d_pose, 0, sizeof(double) * 3 * c->B));
  EB_CUDA_C(cudaMalloc(&c->d_x, sizeof(double) * 3 * c->B));
  EB_CUDA_C(cudaMalloc(&c->d_u0, sizeof(double) * 3 * c->B));
  EB_CUDA_C(cudaMalloc(&c->d_metric, sizeof(double) * c->B));
  EB_CUDA_C(cudaMalloc(&c->d_ck, sizeof(double) * (size_t)c->K * c->B));
  EB_CUDA_C(cudaMemset(c->d_ck, 0, sizeof(double) * (size_t)c->K * c->B));
  EB_CUDA_C(cudaMalloc(&c->d_phik, sizeof(double) * c->K));
  EB_CUDA_C(cudaMemset(c->d_phik, 0, sizeof(double) * c->K));
  EB_CUDA_C(cudaMalloc(&c->d_lamk, sizeof(double) * c->K));
  EB_CUDA_C(cudaMalloc(&c->d_mem_idx_in, sizeof(int) * (size_t)std::max(1u, cfg->batch_size) * c->B));
  EB_CUDA_C(cudaMalloc(&c->d_mem_idx_out, sizeof(int) * (size_t)std::max(1u, cfg->batch_size) * c->B));
  EB_CUDA_C(cudaHostAlloc(&c->h_fault, sizeof(int), cudaHostAllocMapped));
  *c->h_fault = 0;
  EB_CUDA_C(cudaHostGetDevicePointer(&c->d_fault, c->h_fault, 0));
  // Basis::Basis (basis.cpp:48-77): index = ky*nb + kx, lamda_k = 1/(1+sqrt(kx^2+ky^2))^1.5
  std::vector<double> lam(c->K);
  for (int ky = 0; ky < c->nb; ky++)
    for (int kx = 0; kx < c->nb; kx++)
      lam[ky * c->nb + kx] = 1.0 / std::pow(1.0 + std::sqrt((double)((long long)kx * kx + (long long)ky * ky)), 1.5);
  EB_CUDA_C(cudaMemcpy(c->d_lamk, lam.data(), sizeof(double) * c->K, cudaMemcpyHostToDevice));
  if (c->nb > 32)
  {  // solve_kernel_big: S = lamda .* (c_k - phi_k) of every resident CTA
    c->big_rows = std::min(c->B, solve_big_resident(c->nb, c->N));
    if (const char* e = std::getenv("EB_BIG_ROWS"))  // tests: fewer CTAs than instances on a small batch
      c->big_rows = std::max(1, std::min(c->big_rows, std::atoi(e)));
    EB_CUDA_C(cudaMalloc(&c->d_big_scratch, sizeof(double) * (size_t)c->K * (size_t)c->big_rows));
  }
#undef EB_CUDA_C
  *out = c;
  return EB_OK;
}

void eb_destroy(eb_controller* c)
{
  if (!c) return;
  cudaSetDevice(c->cfg.device);
  cudaFree(c->d_ut[0]);
  cudaFree(c->d_ut[1]);
  cudaFree(c->d_pose);
  cudaFree(c->d_hist);
  cudaFree(c->d_hist_cos);
  cudaFree(c->d_phik);
  cudaFree(c->d_lamk);
  cudaFree(c->d_u0);
  cudaFree(c->d_xt);
  cudaFree(c->d_metric);
  cudaFree(c->d_ck);
  cudaFree(c->d_x);
  cudaFree(c->d_mem_idx_in);
  cudaFree(c->d_mem_idx_out);
  cudaFreeHost(c->h_fault);
  cudaFree(c->d_phi_grid);
  cudaFree(c->d_gauss);
  cudaFree(c->d_big_scratch);
  cudaFree(c->d_phik_b);
  cudaFree(c->d_frames);
  cudaFree(c->d_gmu);
  cudaFree(c->d_gsig);
  cudaFree(c->d_gcount);
  cudaFree(c->d_bounds);
  if (c->mb_staged) cudaEventSynchronize(c->mb_staged);
  cudaFreeHost(c->h_mb_desc);
  cudaFree(c->d_mb_desc);
  if (c->mb_staged) cudaEventDestroy(c->mb_staged);
  cudaFree(c->d_mb_slots);
  cudaFreeHost(c->h_mb_kept);
  cudaFree(c->d_mb_kept);
  cudaFree(c->d_kb);
  cudaFree(c->d_mb_arrive);
  cudaFreeHost(c->h_mb_cells);
  cudaFree(c->d_mb_cells);
  cudaFree(c->d_safe_list);
  cudaFree(c->d_safe_branch);
  cudaFree(c->d_safe_vb);
  eb_phik_plan_destroy(c->plan);
  delete c;
}

eb_status eb_clone(const eb_controller* src, eb_controller** out)
{
  if (!src || !out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_clone: NULL argument");
  eb_controller* c = nullptr;
  eb_status st = eb_create(&src->cfg, &c);
  if (st != EB_OK) return st;
  auto bail = [&](cudaError_t e) {
    eb_destroy(c);
    return fail(EB_ERR_CUDA, std::string("eb_clone: ") + cudaGetErrorString(e));
  };
  cudaError_t e = cudaStreamSynchronize(src->stream);
  if (e != cudaSuccess) return bail(e);
  const size_t utb = sizeof(double) * 3 * (size_t)src->N * src->B;
  c->cur = 0;
  if ((e = cudaMemcpy(c->d_ut[0], src->d_ut[src->cur], utb, cudaMemcpyDeviceToDevice)) != cudaSuccess) return bail(e);
  if ((e = cudaMemcpy(c->d_pose, src->d_pose, sizeof(double) * 3 * src->B, cudaMemcpyDeviceToDevice)) != cudaSuccess)
    return bail(e);
  if ((e = cudaMemcpy(c->d_phik, src->d_phik, sizeof(double) * src->K, cudaMemcpyDeviceToDevice)) != cudaSuccess)
    return bail(e);
  if ((e = cudaMemcpy(c->d_ck, src->d_ck, sizeof(double) * (size_t)src->K * src->B, cudaMemcpyDeviceToDevice)) !=
      cudaSuccess)
    return bail(e);
  if (src->mem_count > 0)
  {
    st = ensure_hist(c, src->mem_count);
    if (st != EB_OK)
    {
      eb_destroy(c);
      return st;
    }
    if ((e = cudaMemcpy(c->d_hist, src->d_hist, sizeof(double) * 3 * (size_t)src->B * (size_t)src->mem_count,
                        cudaMemcpyDeviceToDevice)) != cudaSuccess)
      return bail(e);
    c->mem_count = src->mem_count;
  }
  c->lx = src->lx;
  c->ly = src->ly;
  c->map_pos[0] = src->map_pos[0];
  c->map_pos[1] = src->map_pos[1];
  c->gauss_mu = src->gauss_mu;
  c->gauss_sigma = src->gauss_sigma;
  c->call = src->call;
  c->have_pose = src->have_pose;
  c->keep_ck = src->keep_ck;
  c->stream = src->stream;
  if (src->per_inst)
  {
    if ((st = ensure_per_inst(c)) != EB_OK)
    {
      eb_destroy(c);
      return st;
    }
    const size_t B = (size_t)src->B;
    if ((e = cudaMemcpy(c->d_phik_b, src->d_phik_b, sizeof(double) * src->K * B, cudaMemcpyDeviceToDevice)) != cudaSuccess ||
        (e = cudaMemcpy(c->d_frames, src->d_frames, sizeof(double) * eb::kFrDoubles * B, cudaMemcpyDeviceToDevice)) != cudaSuccess ||
        (e = cudaMemcpy(c->d_gcount, src->d_gcount, sizeof(int) * B, cudaMemcpyDeviceToDevice)) != cudaSuccess)
      return bail(e);
    if (src->gmax > 0)
    {
      const size_t gb = sizeof(double) * 2 * (size_t)src->gmax * B;
      if ((e = cudaMalloc(&c->d_gmu, gb)) != cudaSuccess || (e = cudaMalloc(&c->d_gsig, gb)) != cudaSuccess ||
          (e = cudaMemcpy(c->d_gmu, src->d_gmu, gb, cudaMemcpyDeviceToDevice)) != cudaSuccess ||
          (e = cudaMemcpy(c->d_gsig, src->d_gsig, gb, cudaMemcpyDeviceToDevice)) != cudaSuccess)
        return bail(e);
      c->gmax = src->gmax;
    }
    // the cosine rows (the shared path re-derives them; per-instance rows are only derived when a frame moves)
    if (src->mem_count > 0 && src->d_hist_cos && c->d_hist_cos &&
        (e = cudaMemcpy(c->d_hist_cos, src->d_hist_cos, sizeof(double) * 2 * B * (size_t)src->mem_count,
                        cudaMemcpyDeviceToDevice)) != cudaSuccess)
      return bail(e);
    c->frames_set = src->frames_set;
  }
  *out = c;
  return EB_OK;
}

eb_status eb_set_stream(eb_controller* c, void* s)
{
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  c->stream = static_cast<cudaStream_t>(s);
  if (c->plan) c->plan->stream = c->stream;
  return EB_OK;
}

int eb_steps(const eb_controller* c) { return c ? c->N : 0; }
int eb_num_coeff(const eb_controller* c) { return c ? c->K : 0; }
int eb_batch(const eb_controller* c) { return c ? c->B : 0; }
double eb_time_step(const eb_controller* c) { return c ? c->cfg.dt : 0.0; }
long long eb_memory_size(const eb_controller* c) { return c ? c->mem_count : 0; }
long long eb_launch_count(const eb_controller* c) { return c ? c->launches + (c->plan ? c->plan->launches : 0) : 0; }
double* eb_ut_dev(eb_controller* c) { return c ? c->d_ut[c->cur] : nullptr; }
double* eb_ck_dev(eb_controller* c) { return c ? c->d_ck : nullptr; }

eb_status eb_set_keep_ck(eb_controller* c, int keep)
{
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  c->keep_ck = keep != 0;
  return EB_OK;
}

eb_status eb_set_target_gaussians(eb_controller* c, int n, const double* mu, const double* sigma)
{
  if (!c || n < 0 || (n > 0 && (!mu || !sigma))) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_target_gaussians: bad argument");
  if (c->per_inst) return refuse_per_inst("eb_set_target_gaussians");
  c->gauss_mu.assign(mu, mu + 2 * (size_t)n);
  c->gauss_sigma.assign(sigma, sigma + 2 * (size_t)n);
  return EB_OK;
}

eb_status eb_config_target(eb_controller* c, double xmin, double xmax, double ymin, double ymax, int* rebuilt)
{
  EB_TRACE("eb_config_target");
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  if (c->per_inst) return refuse_per_inst("eb_config_target");
  if (rebuilt) *rebuilt = 0;
  // translation from map to fourier domain (:366-367)
  c->map_pos[0] = xmin;
  c->map_pos[1] = ymin;
  const double mx = xmax - xmin, my = ymax - ymin;
  if (almost_equal(mx, c->lx) && almost_equal(my, c->ly)) return EB_OK;  // :374-377
  if (!(mx > 0.0) || !(my > 0.0)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_config_target: empty map extent");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  const int nx = (int)axis_length(0.0, mx, c->cfg.resolution) + 1;  // :387-388
  const int ny = (int)axis_length(0.0, my, c->cfg.resolution) + 1;
  const int ng = (int)(c->gauss_mu.size() / 2);
  if (ng == 0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_config_target: no target set (call eb_set_target_gaussians)");
  eb_phik_plan* plan = nullptr;
  eb_status st = eb_phik_plan_create(c->cfg.device, nx, ny, c->cfg.resolution, mx, my, c->nb, &plan);
  if (st != EB_OK) return st;
  eb_phik_plan_destroy(c->plan);
  c->plan = plan;
  c->plan->stream = c->stream;
  const size_t cells = (size_t)nx * ny;
  if (cells > c->phi_grid_cells)
  {
    cudaFree(c->d_phi_grid);
    c->d_phi_grid = nullptr;
    c->phi_grid_cells = 0;
    EB_CUDA(cudaMalloc(&c->d_phi_grid, sizeof(double) * cells));
    c->phi_grid_cells = cells;
  }
  if (ng > c->gauss_cap)
  {
    cudaFree(c->d_gauss);
    c->d_gauss = nullptr;
    c->gauss_cap = 0;
    EB_CUDA(cudaMalloc(&c->d_gauss, sizeof(double) * 6 * (size_t)ng));
    c->gauss_cap = ng;
  }
  // Gaussian ctor (target.hpp:68-71): cov = diag(sigma^2), cov_inv = inv(cov)
  // (2x2 cofactor inverse); operator() (:91-102) translates the mean.
  std::vector<double> g(6 * (size_t)ng);
  for (int i = 0; i < ng; i++)
  {
    const double a = c->gauss_sigma[2 * i] * c->gauss_sigma[2 * i];
    const double d = c->gauss_sigma[2 * i + 1] * c->gauss_sigma[2 * i + 1];
    const double det = a * d - 0.0 * 0.0;
    g[6 * i + 0] = c->gauss_mu[2 * i] - xmin;
    g[6 * i + 1] = c->gauss_mu[2 * i + 1] - ymin;
    g[6 * i + 2] = d / det;     // ci(0,0)
    g[6 * i + 3] = -0.0 / det;  // ci(1,0)
    g[6 * i + 4] = -0.0 / det;  // ci(0,1)
    g[6 * i + 5] = a / det;     // ci(1,1)
  }
  EB_CUDA(cudaMemcpyAsync(c->d_gauss, g.data(), sizeof(double) * g.size(), cudaMemcpyHostToDevice, c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));  // g is a stack-lifetime buffer
  eb::target_fill_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, c->stream>>>(ng, c->d_gauss, c->plan->d_xs,
                                                                                 c->plan->d_ys, nx, ny, c->d_phi_grid);
  c->launches += 1;
  EB_CUDA(cudaGetLastError());
  st = eb_phik_execute_dev(c->plan, c->d_phi_grid, c->d_phik, nullptr);
  if (st != EB_OK) return st;
  c->lx = mx;  // :382-383
  c->ly = my;
  if (rebuilt) *rebuilt = 1;
  return EB_OK;
}

eb_status eb_set_phik(eb_controller* c, const double* phik, double lx, double ly)
{
  if (!c || !phik) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_phik: NULL argument");
  if (c->per_inst) return refuse_per_inst("eb_set_phik");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  EB_CUDA(cudaMemcpyAsync(c->d_phik, phik, sizeof(double) * c->K, cudaMemcpyHostToDevice, c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));
  c->lx = lx;
  c->ly = ly;
  return EB_OK;
}

eb_status eb_get_phik(const eb_controller* c, double* phik, double* lx, double* ly)
{
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  if (c->per_inst) return refuse_per_inst("eb_get_phik");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  if (phik)
  {
    EB_CUDA(cudaMemcpyAsync(phik, c->d_phik, sizeof(double) * c->K, cudaMemcpyDeviceToHost, c->stream));
    EB_CUDA(cudaStreamSynchronize(c->stream));
  }
  if (lx) *lx = c->lx;
  if (ly) *ly = c->ly;
  return EB_OK;
}

static eb_status add_state_memory(eb_controller* c, const double* x, cudaMemcpyKind kind)
{
  if (!c || !x) return fail(EB_ERR_INVALID_ARGUMENT, "eb_add_state_memory: NULL argument");
  if (c->mem_count >= (long long)c->cfg.buffer_size) return EB_OK;  // buffer.cpp:56-61: dropped when full
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_hist(c, c->mem_count + 1);
  if (st != EB_OK) return st;
  const size_t row = (size_t)c->B * (size_t)c->mem_count;
  if (c->per_inst && c->d_hist_cos)
  {
    // per-instance frames: the row and its cosines (each in its instance's frame) in one launch, always
    const double* xd = x;
    if (kind == cudaMemcpyHostToDevice)
    {
      EB_CUDA(cudaMemcpyAsync(c->d_x, x, sizeof(double) * 3 * c->B, kind, c->stream));
      xd = c->d_x;
    }
    eb::add_state_kernel<<<(c->B + 255) / 256, 256, 0, c->stream>>>(xd, c->d_hist + 3 * row, c->d_hist_cos + 2 * row, c->B,
                                                                    0.0, 0.0, 0.0, 0.0, c->d_frames);
    EB_CUDA(cudaGetLastError());
    if (kind == cudaMemcpyHostToDevice) EB_CUDA(cudaStreamSynchronize(c->stream));
    c->launches += 1;
    c->mem_count++;
    return EB_OK;
  }
  const double key[4] = { c->map_pos[0], c->map_pos[1], 1.0 / c->lx, 1.0 / c->ly };
  if (kind == cudaMemcpyDeviceToDevice && c->d_hist_cos && c->cos_count == c->mem_count && c->lx > 0.0 && c->ly > 0.0 &&
      std::memcmp(key, c->cos_key, sizeof(key)) == 0)
  {
    // the cosine rows are up to date for the current frame: the new row and its cosines in ONE launch
    eb::add_state_kernel<<<(c->B + 255) / 256, 256, 0, c->stream>>>(x, c->d_hist + 3 * row, c->d_hist_cos + 2 * row, c->B,
                                                                    key[0], key[1], key[2], key[3], nullptr);
    EB_CUDA(cudaGetLastError());
    c->launches += 1;
    c->cos_count++;
    c->mem_count++;
    return EB_OK;
  }
  EB_CUDA(cudaMemcpyAsync(c->d_hist + 3 * row, x, sizeof(double) * 3 * c->B, kind, c->stream));
  if (kind == cudaMemcpyHostToDevice) EB_CUDA(cudaStreamSynchronize(c->stream));
  c->mem_count++;
  return EB_OK;
}

// room for `count` stored states up front (at most buffer_size): no re-allocation inside the control loop
eb_status eb_reserve_state_memory(eb_controller* c, long long count)
{
  if (!c || count < 0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_reserve_state_memory: bad argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  return ensure_hist(c, std::min<long long>(count, (long long)c->cfg.buffer_size));
}

eb_status eb_add_state_memory_host(eb_controller* c, const double* x)
{
  EB_TRACE("eb_add_state_memory_host");
  return add_state_memory(c, x, cudaMemcpyHostToDevice);
}
eb_status eb_add_state_memory_dev(eb_controller* c, const double* x_dev)
{
  EB_TRACE("eb_add_state_memory_dev");
  return add_state_memory(c, x_dev, cudaMemcpyDeviceToDevice);
}

static eb_status solve_step(eb_controller* c, const double* x_dev, const int* mem_idx_dev, double* u0_dev,
                            double* metric_dev);

eb_status eb_control_dev(eb_controller* c, double xmin, double xmax, double ymin, double ymax, const double* x_dev,
                         const int* mem_idx_dev, double* u0_dev, double* metric_dev)
{
  EB_TRACE("eb_control_dev");
  if (!c || !x_dev || !u0_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_dev: NULL argument");
  if (c->per_inst) return refuse_per_inst("eb_control_dev");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = eb_config_target(c, xmin, xmax, ymin, ymax, nullptr);  // :230
  if (st != EB_OK) return st;
  return solve_step(c, x_dev, mem_idx_dev, u0_dev, metric_dev);
}

// one solve launch over the batch, after the target is configured (shared frame, or per-instance frames and rows)
static eb_status solve_step(eb_controller* c, const double* x_dev, const int* mem_idx_dev, double* u0_dev,
                            double* metric_dev)
{
  // pose_ = x (:227)
  c->have_pose = true;  // the kernel records x as pose_ (for optTraj)

  eb::SolveParams p{};
  p.B = c->B;
  p.N = c->N;
  p.nb = c->nb;
  p.mem_count = (int)std::min<long long>(c->mem_count, 0x7fffffff);
  p.batch_size = (int)c->cfg.batch_size;
  // ReplayBuffer::sampleMemory (buffer.cpp:64-111)
  if (c->mem_count == 0)
    p.M = 0;
  else if (c->mem_count <= (long long)c->cfg.batch_size)
  {
    p.M = (int)c->mem_count;
    p.idx_mode = 0;
  }
  else
  {
    p.M = (int)c->cfg.batch_size;
    p.idx_mode = mem_idx_dev ? 1 : 2;
  }
  c->last_idx_count = (p.M > 0 && p.idx_mode != 0) ? p.M : 0;
  p.dt = c->cfg.dt;
  p.lx = c->lx;
  p.ly = c->ly;
  p.inv_lx = 1.0 / c->lx;
  p.inv_ly = 1.0 / c->ly;
  p.ax = eb::kPi / c->lx;
  p.by = eb::kPi / c->ly;
  p.xmin = c->map_pos[0];
  p.ymin = c->map_pos[1];
  p.w = c->cfg.expl_weight;
  std::memcpy(p.Rinv, c->cfg.Rinv, sizeof(p.Rinv));
  std::memcpy(p.umin, c->cfg.umin, sizeof(p.umin));
  std::memcpy(p.umax, c->cfg.umax, sizeof(p.umax));
  p.bw = c->cfg.barrier_weight;
  p.beps = c->cfg.barrier_eps;
  p.seed = c->cfg.seed;
  p.call = c->call++;
  p.x = x_dev;
  p.pose_out = (x_dev != c->d_pose) ? c->d_pose : nullptr;
  p.ut_in = c->d_ut[c->cur];
  p.ut_out = c->d_ut[c->cur ^ 1];
  p.hist = c->d_hist;
  if (p.M > 0 && c->d_hist_cos && c->nb <= 32)
  {  // (the CTA-per-instance kernel starts its tables at arbitrary orders and needs the coordinates themselves)
    if (!c->per_inst)  // per-instance rows are kept valid as frames move and states are stored
    {
      const eb_status hs = ensure_hist_cos(c);
      if (hs != EB_OK) return hs;
    }
    p.hist_cos = c->d_hist_cos;
  }
  p.mem_idx = mem_idx_dev;
  p.mem_idx_out = c->d_mem_idx_out;
  p.phik = c->per_inst ? c->d_phik_b : c->d_phik;
  p.frames = c->d_frames;
  p.lamk = c->d_lamk;
  p.u0 = u0_dev;
  p.metric = metric_dev;
  p.ck = c->keep_ck ? c->d_ck : nullptr;
  p.fault = c->d_fault;
  p.big_scratch = c->d_big_scratch;
  p.big_rows = c->big_rows;
  if (c->peer)
  {
    p.n_peer = c->peer->n_peer;
    for (int q = 0; q < p.n_peer; q++)
    {
      p.u0_peer[q] = c->peer->u0_peer[q];
      p.flag_peer[q] = c->peer->flag_peer[q];
    }
    p.flag_value = c->peer->flag_value;
    p.done_counter = c->peer->done_counter;
    p.my_flags = c->peer->my_flags;
    p.need = c->peer->need;
  }
  cudaError_t e = launch_solve(p, c->cfg.model, c->stream, c->per_inst);
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("solve_kernel launch: ") + cudaGetErrorString(e));
  c->launches += 1;
  c->cur ^= 1;
  return EB_OK;
}

#ifdef EB_PHASE_TIMING
// debug build only (tools/phase_timing.py): copies the clock64() stamps of the last solve
extern "C" int eb_debug_phase_dump(long long* host, int n)
{
  return (int)cudaMemcpyFromSymbol(host, eb::g_phase, sizeof(long long) * eb::kPhaseSlots * (size_t)n);
}
#endif

#ifdef EB_DEBUG_DUMP
extern "C" int eb_debug_dump(double* host, int n)
{
  return (int)cudaMemcpyFromSymbol(host, eb::g_dbg, sizeof(double) * 16 * (size_t)n);
}
#endif

eb_status eb_check_status(eb_controller* c)
{
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  return check_fault(c);
}

eb_status eb_control_host(eb_controller* c, double xmin, double xmax, double ymin, double ymax, const double* x,
                          const int* mem_idx, double* u0, double* metric)
{
  EB_TRACE("eb_control_host");
  if (!c || !x || !u0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_host: NULL argument");
  if (c->per_inst) return refuse_per_inst("eb_control_host");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  const bool need_idx = mem_idx && c->mem_count > (long long)c->cfg.batch_size;
  if (need_idx)
    EB_CUDA(cudaMemcpyAsync(c->d_mem_idx_in, mem_idx, sizeof(int) * (size_t)c->cfg.batch_size * c->B,
                            cudaMemcpyHostToDevice, c->stream));
  // Small batches with page-locked caller buffers: the kernel reads x and writes
  // u0 / metric in place over PCIe (one launch + one sync, no copy-engine hops).
  double *xm = nullptr, *um = nullptr, *mm = nullptr;
  if (c->B <= zero_copy_max_batch())
  {
    xm = c->mapped(x);
    um = xm ? c->mapped(u0) : nullptr;
    mm = (um && metric) ? c->mapped(metric) : nullptr;
  }
  if (xm && um && (!metric || mm))
  {
    eb_status st = eb_control_dev(c, xmin, xmax, ymin, ymax, xm, need_idx ? c->d_mem_idx_in : nullptr, um, mm);
    if (st != EB_OK) return st;
    return check_fault(c);  // synchronises
  }
  EB_CUDA(cudaMemcpyAsync(c->d_pose, x, sizeof(double) * 3 * c->B, cudaMemcpyHostToDevice, c->stream));
  eb_status st = eb_control_dev(c, xmin, xmax, ymin, ymax, c->d_pose, need_idx ? c->d_mem_idx_in : nullptr, c->d_u0,
                                metric ? c->d_metric : nullptr);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(u0, c->d_u0, sizeof(double) * 3 * c->B, cudaMemcpyDeviceToHost, c->stream));
  if (metric) EB_CUDA(cudaMemcpyAsync(metric, c->d_metric, sizeof(double) * c->B, cudaMemcpyDeviceToHost, c->stream));
  return check_fault(c);  // synchronises
}

eb_status eb_opt_traj_dev(eb_controller* c, double* xt_dev)
{
  EB_TRACE("eb_opt_traj_dev");
  if (!c || !xt_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_opt_traj_dev: NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  const int threads = 128, wpb = threads / 32;
  const int grid = (c->B + wpb - 1) / wpb;
  if (c->cfg.model == EB_MODEL_OMNI)
    eb::rollout_kernel<eb::kModelOmni><<<grid, threads, 0, c->stream>>>(c->B, c->N, c->cfg.dt, c->d_pose,
                                                                        c->d_ut[c->cur], xt_dev, c->d_fault);
  else
    eb::rollout_kernel<eb::kModelSimpleCart><<<grid, threads, 0, c->stream>>>(c->B, c->N, c->cfg.dt, c->d_pose,
                                                                              c->d_ut[c->cur], xt_dev, c->d_fault);
  c->launches += 1;
  EB_CUDA(cudaGetLastError());
  return EB_OK;
}

eb_status eb_opt_traj_host(eb_controller* c, double* xt)
{
  if (!c || !xt) return fail(EB_ERR_INVALID_ARGUMENT, "eb_opt_traj_host: NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  const size_t bytes = sizeof(double) * 3 * (size_t)c->N * c->B;
  if (!c->d_xt) EB_CUDA(cudaMalloc(&c->d_xt, bytes));  // optTraj() runs every tick (exploration.hpp:234): keep it
  double* const d = c->d_xt;
  eb_status st = eb_opt_traj_dev(c, d);
  cudaError_t e = cudaSuccess;
  if (st == EB_OK) e = cudaMemcpyAsync(xt, d, bytes, cudaMemcpyDeviceToHost, c->stream);
  if (st == EB_OK && e == cudaSuccess) st = check_fault(c);
  cudaStreamSynchronize(c->stream);
  if (st != EB_OK) return st;
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_opt_traj_host: ") + cudaGetErrorString(e));
  return EB_OK;
}

eb_status eb_get_ut(const eb_controller* c, double* ut)
{
  if (!c || !ut) return fail(EB_ERR_INVALID_ARGUMENT, "eb_get_ut: NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  EB_CUDA(cudaMemcpyAsync(ut, c->d_ut[c->cur], sizeof(double) * 3 * (size_t)c->N * c->B, cudaMemcpyDeviceToHost,
                          c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));
  return EB_OK;
}

eb_status eb_set_ut(eb_controller* c, const double* ut)
{
  if (!c || !ut) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_ut: NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  EB_CUDA(cudaMemcpyAsync(c->d_ut[c->cur], ut, sizeof(double) * 3 * (size_t)c->N * c->B, cudaMemcpyHostToDevice,
                          c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));
  return EB_OK;
}

eb_status eb_get_ck(const eb_controller* c, double* ck)
{
  if (!c || !ck) return fail(EB_ERR_INVALID_ARGUMENT, "eb_get_ck: NULL argument");
  if (!c->keep_ck) return fail(EB_ERR_UNSUPPORTED, "eb_get_ck: the c_k by-product is switched off (eb_set_keep_ck)");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  EB_CUDA(cudaMemcpyAsync(ck, c->d_ck, sizeof(double) * (size_t)c->K * c->B, cudaMemcpyDeviceToHost, c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));
  return EB_OK;
}

eb_status eb_get_last_mem_idx(const eb_controller* c, int* mem_idx, int* count)
{
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  if (count) *count = c->last_idx_count;
  if (mem_idx && c->last_idx_count > 0)
  {
    EB_CUDA(cudaSetDevice(c->cfg.device));
    EB_CUDA(cudaMemcpyAsync(mem_idx, c->d_mem_idx_out, sizeof(int) * (size_t)c->cfg.batch_size * c->B,
                            cudaMemcpyDeviceToHost, c->stream));
    EB_CUDA(cudaStreamSynchronize(c->stream));
  }
  return EB_OK;
}

namespace
{
struct DevBuf
{
  double* p = nullptr;
  ~DevBuf() { cudaFree(p); }
  cudaError_t alloc(size_t n) { return cudaMalloc(&p, sizeof(double) * (n ? n : 1)); }
};

// Gaussian ctor (target.hpp:68-71) + mean translation (:100): 6 doubles per Gaussian
std::vector<double> pack_gaussians(int ng, const double* mu, const double* sigma, const double* trans)
{
  std::vector<double> g(6 * (size_t)ng);
  for (int i = 0; i < ng; i++)
  {
    const double a = sigma[2 * i] * sigma[2 * i], d = sigma[2 * i + 1] * sigma[2 * i + 1];
    const double det = a * d - 0.0 * 0.0;
    g[6 * i + 0] = mu[2 * i] - trans[0];
    g[6 * i + 1] = mu[2 * i + 1] - trans[1];
    g[6 * i + 2] = d / det;
    g[6 * i + 3] = -0.0 / det;
    g[6 * i + 4] = -0.0 / det;
    g[6 * i + 5] = a / det;
  }
  return g;
}
}  // namespace

static eb_status basis_sum(int device, double lx, double ly, int nb, const double* pts, int ld, long long n,
                           const double* w, double scale, double* out)
{
  if (nb < 1 || nb > EB_MAX_NUM_BASIS || n < 1 || !pts || !out || ld < 2)
    return fail(EB_ERR_INVALID_ARGUMENT, "Basis: need 1 <= num_basis <= " + std::to_string(EB_MAX_NUM_BASIS) + ", at least one point, ld >= 2");
  EB_CUDA(cudaSetDevice(device));
  DevBuf dp, dw, dout;
  EB_CUDA(dp.alloc((size_t)ld * n));
  EB_CUDA(dout.alloc((size_t)nb * nb));
  EB_CUDA(cudaMemcpy(dp.p, pts, sizeof(double) * ld * n, cudaMemcpyHostToDevice));
  if (w)
  {
    EB_CUDA(dw.alloc((size_t)n));
    EB_CUDA(cudaMemcpy(dw.p, w, sizeof(double) * n, cudaMemcpyHostToDevice));
  }
  eb::basis_sum_kernel<<<nb * nb, 256>>>(lx, ly, nb, dp.p, ld, n, w ? dw.p : nullptr, scale, dout.p);
  EB_CUDA(cudaGetLastError());
  EB_CUDA(cudaMemcpy(out, dout.p, sizeof(double) * nb * nb, cudaMemcpyDeviceToHost));
  return EB_OK;
}

eb_status eb_basis_traj_coeff_host(int device, double lx, double ly, int nb, const double* xt, int ld, int ncols,
                                   double* ck)
{
  return basis_sum(device, lx, ly, nb, xt, ld, ncols, nullptr, ncols > 0 ? 1.0 / (double)ncols : 0.0, ck);
}

eb_status eb_basis_spatial_coeff_host(int device, double lx, double ly, int nb, const double* phi_vals,
                                      const double* phi_grid, long long G, double* phik)
{
  if (!phi_vals) return fail(EB_ERR_INVALID_ARGUMENT, "Basis::spatialCoeff: phi_vals is NULL");
  return basis_sum(device, lx, ly, nb, phi_grid, 2, G, phi_vals, 1.0, phik);
}

eb_status eb_basis_grad_host(int device, double lx, double ly, int nb, const double* x, double* dfk)
{
  if (nb < 1 || nb > EB_MAX_NUM_BASIS || !x || !dfk) return fail(EB_ERR_INVALID_ARGUMENT, "Basis::gradFourierBasis: bad argument");
  EB_CUDA(cudaSetDevice(device));
  DevBuf d;
  EB_CUDA(d.alloc(2 * (size_t)nb * nb));
  eb::basis_grad_kernel<<<(nb * nb + 127) / 128, 128>>>(lx, ly, nb, x[0], x[1], d.p);
  EB_CUDA(cudaGetLastError());
  EB_CUDA(cudaMemcpy(dfk, d.p, sizeof(double) * 2 * nb * nb, cudaMemcpyDeviceToHost));
  return EB_OK;
}

eb_status eb_target_fill_host(int device, int ng, const double* mu, const double* sigma, const double* trans,
                              const double* phi_grid, long long G, double* phi_vals)
{
  if (ng < 1 || !mu || !sigma || !trans || !phi_grid || !phi_vals || G < 1)
    return fail(EB_ERR_INVALID_ARGUMENT, "Target::fill: bad argument");
  EB_CUDA(cudaSetDevice(device));
  const std::vector<double> g = pack_gaussians(ng, mu, sigma, trans);
  DevBuf dg, dp, dv, dt;
  EB_CUDA(dg.alloc(g.size()));
  EB_CUDA(dp.alloc(2 * (size_t)G));
  EB_CUDA(dv.alloc((size_t)G));
  EB_CUDA(dt.alloc(1));
  EB_CUDA(cudaMemcpy(dg.p, g.data(), sizeof(double) * g.size(), cudaMemcpyHostToDevice));
  EB_CUDA(cudaMemcpy(dp.p, phi_grid, sizeof(double) * 2 * G, cudaMemcpyHostToDevice));
  const unsigned blocks = (unsigned)((G + 255) / 256);
  eb::target_points_kernel<<<blocks, 256>>>(ng, dg.p, dp.p, G, dv.p);
  eb::vector_sum_kernel<<<1, 1024>>>(dv.p, G, dt.p);
  eb::vector_div_kernel<<<blocks, 256>>>(dv.p, G, dt.p);  // target.cpp:87
  EB_CUDA(cudaGetLastError());
  EB_CUDA(cudaMemcpy(phi_vals, dv.p, sizeof(double) * G, cudaMemcpyDeviceToHost));
  return EB_OK;
}

// ---------------------------------------------------------------------------
// fused multi-GPU gather over peer memory (peer_gather.cuh)
// ---------------------------------------------------------------------------
}  // extern "C"

// Batches of at least this many instances publish their first twists from inside the solve kernel; smaller
// (single-wave) batches from the group's side stream (peer_gather.cuh).  EB_GATHER_FUSE_MIN_BATCH overrides.
extern "C" int eb_gather_fuse_min_batch(void)
{
  const char* e = std::getenv("EB_GATHER_FUSE_MIN_BATCH");  // read at every group creation (tests switch it)
  return e ? std::atoi(e) : 8192;
}

struct eb_peer_group
{
  int device = 0, rank = 0, world = 1;
  long long elems = 0;                          // doubles per rank and step (3 * batch)
  double* gathered[eb::kPeerBuffers] = {};      // own copies, [world * elems], rotating by step
  unsigned long long* flags = nullptr;          // own arrival flags, [world]
  unsigned int* counter = nullptr;
  double* peer_gathered[eb::kMaxPeers][eb::kPeerBuffers] = {};  // every rank's buffers as seen from here (own: the local pointers)
  unsigned long long* peer_flags[eb::kMaxPeers] = {};
  bool connected = false;
  unsigned long long step = 0;                  // steps launched so far
  // side-stream publication (small batches): rotating local u0 blocks, the group's own stream and events
  double* local_u0[eb::kPeerBuffers] = {};
  cudaStream_t side = nullptr;
  cudaEvent_t solved[eb::kPeerBuffers] = {}, published[eb::kPeerBuffers] = {};
  unsigned int* side_counter = nullptr;
  bool side_used = false;                       // a side-stream publication has been enqueued at least once
  int fuse_min_batch = eb_gather_fuse_min_batch();  // batches at least this large publish from inside the solve kernel
};

extern "C" {

int eb_peer_blob_bytes(void) { return (eb::kPeerBuffers + 1) * (int)sizeof(cudaIpcMemHandle_t); }

eb_status eb_peer_group_create(int device, int rank, int world, long long elems_per_rank, eb_peer_group** out)
{
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_peer_group_create: out is NULL");
  *out = nullptr;
  if (world < 1 || world > eb::kMaxPeers || rank < 0 || rank >= world || elems_per_rank < 1)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_peer_group_create: need 1 <= world <= 8, 0 <= rank < world, elems >= 1");
  EB_CUDA(cudaSetDevice(device));
  eb_peer_group* g = new (std::nothrow) eb_peer_group();
  if (!g) return fail(EB_ERR_CUDA, "out of host memory");
  g->device = device;
  g->rank = rank;
  g->world = world;
  g->elems = elems_per_rank;
  const size_t bytes = sizeof(double) * (size_t)world * (size_t)elems_per_rank;
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < eb::kPeerBuffers && e == cudaSuccess; k++)
  {
    e = cudaMalloc(&g->gathered[k], bytes);
    if (e == cudaSuccess) e = cudaMemset(g->gathered[k], 0, bytes);
  }
  if (e == cudaSuccess) e = cudaMalloc(&g->flags, sizeof(unsigned long long) * eb::kMaxPeers);
  if (e == cudaSuccess) e = cudaMalloc(&g->counter, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMalloc(&g->side_counter, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMemset(g->side_counter, 0, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g->side, cudaStreamNonBlocking);
  for (int k = 0; k < eb::kPeerBuffers && e == cudaSuccess; k++)
  {
    e = cudaMalloc(&g->local_u0[k], sizeof(double) * (size_t)elems_per_rank);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->solved[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->published[k], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaMemset(g->flags, 0, sizeof(unsigned long long) * eb::kMaxPeers);
  if (e == cudaSuccess) e = cudaMemset(g->counter, 0, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess)
  {
    eb_peer_group_destroy(g);
    return fail(EB_ERR_CUDA, std::string("eb_peer_group_create: ") + cudaGetErrorString(e));
  }
  *out = g;
  return EB_OK;
}

// blob = IPC handles of {gathered[0..kPeerBuffers), flags}; all_gather the blobs of all ranks (rank order)
eb_status eb_peer_group_export(eb_peer_group* g, unsigned char* blob)
{
  if (!g || !blob) return fail(EB_ERR_INVALID_ARGUMENT, "eb_peer_group_export: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  cudaIpcMemHandle_t h[eb::kPeerBuffers + 1];
  for (int k = 0; k < eb::kPeerBuffers; k++) EB_CUDA(cudaIpcGetMemHandle(&h[k], g->gathered[k]));
  EB_CUDA(cudaIpcGetMemHandle(&h[eb::kPeerBuffers], g->flags));
  std::memcpy(blob, h, sizeof(h));
  return EB_OK;
}

eb_status eb_peer_group_connect(eb_peer_group* g, const unsigned char* blobs)
{
  if (!g || (g->world > 1 && !blobs)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_peer_group_connect: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  for (int r = 0; r < g->world; r++)
  {
    if (r == g->rank)
    {
      for (int k = 0; k < eb::kPeerBuffers; k++) g->peer_gathered[r][k] = g->gathered[k];
      g->peer_flags[r] = g->flags;
      continue;
    }
    cudaIpcMemHandle_t h[eb::kPeerBuffers + 1];
    std::memcpy(h, blobs + (size_t)r * sizeof(h), sizeof(h));
    void* ptr[eb::kPeerBuffers + 1] = {};
    for (int k = 0; k <= eb::kPeerBuffers; k++)
    {
      cudaError_t e = cudaIpcOpenMemHandle(&ptr[k], h[k], cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess)
        return fail(EB_ERR_CUDA, std::string("eb_peer_group_connect: cudaIpcOpenMemHandle (peer access over "
                                             "NVLink is required): ") + cudaGetErrorString(e));
    }
    for (int k = 0; k < eb::kPeerBuffers; k++) g->peer_gathered[r][k] = static_cast<double*>(ptr[k]);
    g->peer_flags[r] = static_cast<unsigned long long*>(ptr[eb::kPeerBuffers]);
  }
  g->connected = true;
  return EB_OK;
}

void eb_peer_group_destroy(eb_peer_group* g)
{
  if (!g) return;
  cudaSetDevice(g->device);
  cudaDeviceSynchronize();
  if (g->connected)
    for (int r = 0; r < g->world; r++)
      if (r != g->rank)
      {
        for (int k = 0; k < eb::kPeerBuffers; k++) cudaIpcCloseMemHandle(g->peer_gathered[r][k]);
        cudaIpcCloseMemHandle(g->peer_flags[r]);
      }
  if (g->side) cudaStreamSynchronize(g->side);
  for (int k = 0; k < eb::kPeerBuffers; k++)
  {
    cudaFree(g->gathered[k]);
    cudaFree(g->local_u0[k]);
    if (g->solved[k]) cudaEventDestroy(g->solved[k]);
    if (g->published[k]) cudaEventDestroy(g->published[k]);
  }
  if (g->side) cudaStreamDestroy(g->side);
  cudaFree(g->side_counter);
  cudaFree(g->flags);
  cudaFree(g->counter);
  delete g;
}

// device pointer of this rank's copy of the gathered first twists of step `step` (1-based count of
// eb_control_dev_gather calls): [world][batch][3]
double* eb_peer_gathered_dev(eb_peer_group* g, unsigned long long step)
{
  return (g && step >= 1) ? g->gathered[(step - 1) % eb::kPeerBuffers] : nullptr;
}

unsigned long long eb_peer_group_steps(const eb_peer_group* g) { return g ? g->step : 0; }

// 1: a batch of this size publishes from inside the solve kernel, 0: from the group's side stream
int eb_peer_group_fused(const eb_peer_group* g, int batch) { return (g && batch >= g->fuse_min_batch) ? 1 : 0; }

}  // extern "C"

namespace
{
// what every gathering call refuses about the group
eb_status peer_group_check(const eb_controller* c, const eb_peer_group* g, const std::string& call)
{
  if (!g->connected) return fail(EB_ERR_INVALID_ARGUMENT, call + ": peer group is not connected");
  if (g->elems != 3LL * c->B) return fail(EB_ERR_INVALID_ARGUMENT, call + ": peer group sized for another batch");
  return EB_OK;
}

// launching step n + 1 = g->step + 1 into the buffer of step n + 1 - kPeerBuffers: every rank must have finished step
// n + 2 - kPeerBuffers (its reads of the older step precede that launch)
unsigned long long peer_need(const eb_peer_group* g)
{
  return g->step + 2 > (unsigned long long)eb::kPeerBuffers ? g->step + 2 - eb::kPeerBuffers : 0;
}

// the publication of this rank's block of the next step, whose twists are in src
eb::PublishParams publish_params(const eb_peer_group* g, const double* src, unsigned int* counter)
{
  const int parity = (int)(g->step % eb::kPeerBuffers);
  eb::PublishParams pp{};
  pp.src = src;
  pp.elems = g->elems;
  pp.n_peer = g->world;
  for (int r = 0; r < g->world; r++)
  {
    pp.dst[r] = g->peer_gathered[r][parity] + (size_t)g->rank * (size_t)g->elems;
    pp.flag[r] = g->peer_flags[r] + g->rank;
  }
  pp.flag_value = g->step + 1;
  pp.my_flags = g->flags;
  pp.need = peer_need(g);
  pp.done_counter = counter;
  return pp;
}

// One gathered control() step, after the caller's checks.  solve(u0) makes the step's solve launch, writing the first
// twists to u0 (eb_control_dev or eb_control_batch_dev); while c->peer is set, the solve kernel also stores them into
// every rank's buffer.  wait = false: eb_control_dev_gather's contract, true: eb_control_dev_gather_wait's.
template <class Solve>
eb_status gather_step(eb_controller* c, eb_peer_group* g, const bool wait, const Solve& solve)
{
  if (c->B >= g->fuse_min_batch)
  {
    if (wait)
    {
      const eb_status st = gather_step(c, g, false, solve);
      if (st != EB_OK) return st;
      return eb_peer_group_wait(g, c, g->step);
    }
    const int parity = (int)(g->step % eb::kPeerBuffers);
    PeerLaunch pl;
    pl.n_peer = g->world;
    for (int r = 0; r < g->world; r++)
    {
      pl.u0_peer[r] = g->peer_gathered[r][parity] + (size_t)g->rank * (size_t)g->elems;
      pl.flag_peer[r] = g->peer_flags[r] + g->rank;
    }
    pl.flag_value = g->step + 1;
    pl.done_counter = g->counter;
    pl.my_flags = g->flags;
    pl.need = peer_need(g);
    c->peer = &pl;
    const eb_status st = solve(c->d_u0);
    c->peer = nullptr;
    if (st == EB_OK) g->step += 1;
    return st;
  }
  // single-wave batch: solve locally, then publish from the group's own stream under the next step (wait = false), or
  // publish and wait in one kernel right behind the solve kernel (wait = true)
  EB_CUDA(cudaSetDevice(g->device));
  const int parity = (int)(g->step % eb::kPeerBuffers);
  // a side-stream publication of an earlier step must have left this buffer
  if (g->step >= (unsigned long long)eb::kPeerBuffers && (!wait || g->side_used))
    EB_CUDA(cudaStreamWaitEvent(c->stream, g->published[parity], 0));
  const eb_status st = solve(g->local_u0[parity]);
  if (st != EB_OK) return st;
  if (!wait)
  {
    EB_CUDA(cudaEventRecord(g->solved[parity], c->stream));
    EB_CUDA(cudaStreamWaitEvent(g->side, g->solved[parity], 0));
    const eb::PublishParams pp = publish_params(g, g->local_u0[parity], g->side_counter);
    // Few blocks on purpose: a single-wave solve kernel needs nearly every resident-CTA slot of the
    // machine (1024 of 1036 at 4096 instances), and a publish block that is still running -- or
    // waiting in the reuse guard for a slower rank -- when the next solve kernel starts must fit
    // into the spare slots, or that kernel spills into a second wave.
    const int blocks = (int)std::max<long long>(1, std::min<long long>(4, (g->elems / 2 + 4095) / 4096));
    eb::peer_publish_kernel<<<blocks, 256, 0, g->side>>>(pp);
    g->side_used = true;
    EB_CUDA(cudaGetLastError());
    EB_CUDA(cudaEventRecord(g->published[parity], g->side));
  }
  else
  {
    const eb::PublishParams pp = publish_params(g, g->local_u0[parity], g->counter);
    const int blocks = (int)std::max<long long>(1, std::min<long long>(64, (g->elems / 2 + 255) / 256));
    // programmatic dependent launch behind the solve kernel (and ahead of the next step's): see SolveLaunch::launch_w
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(256);
    cfg.stream = c->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    EB_CUDA(cudaLaunchKernelEx(&cfg, eb::peer_publish_wait_kernel, pp));
  }
  c->launches += 1;
  g->step += 1;
  return EB_OK;
}

// the checks of eb_control_batch_dev_gather[_wait]: eb_control_batch_dev's and the group's
eb_status batch_gather_check(const eb_controller* c, const eb_peer_group* g, const double* bounds_dev,
                             const double* x_dev, const char* call)
{
  if (!c || !g || !x_dev) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  if (!bounds_dev && !c->frames_set)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": bounds NULL before any frame was configured");
  if (g->device != c->cfg.device)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the peer group and the controller are on different devices");
  return peer_group_check(c, g, call);
}
}  // namespace

extern "C" {

// control() whose first twists land in every rank's gathered buffer (no collective call)
eb_status eb_control_dev_gather(eb_controller* c, eb_peer_group* g, double xmin, double xmax, double ymin, double ymax,
                                const double* x_dev, const int* mem_idx_dev, double* metric_dev)
{
  EB_TRACE("eb_control_dev_gather");
  if (!c || !g) return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_dev_gather: NULL argument");
  if (c->per_inst) return fail(EB_ERR_UNSUPPORTED, "eb_control_dev_gather: not available with per-instance targets");
  const eb_status st = peer_group_check(c, g, "eb_control_dev_gather");
  if (st != EB_OK) return st;
  return gather_step(c, g, false, [&](double* u0) {
    return eb_control_dev(c, xmin, xmax, ymin, ymax, x_dev, mem_idx_dev, u0, metric_dev);
  });
}

// control() + gather + wait in one call, everything on the controller's stream: when it returns (stream order), the
// rows of EVERY rank for this step are in eb_peer_gathered_dev(g, step).  Single-wave batches publish and wait in one
// kernel behind the solve kernel (peer_publish_wait_kernel); larger ones publish from inside the solve kernel and
// enqueue the wait kernel.
eb_status eb_control_dev_gather_wait(eb_controller* c, eb_peer_group* g, double xmin, double xmax, double ymin, double ymax,
                                     const double* x_dev, const int* mem_idx_dev, double* metric_dev)
{
  EB_TRACE("eb_control_dev_gather_wait");
  if (!c || !g) return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_dev_gather_wait: NULL argument");
  if (c->per_inst) return fail(EB_ERR_UNSUPPORTED, "eb_control_dev_gather_wait: not available with per-instance targets");
  const eb_status st = peer_group_check(c, g, "eb_control_dev_gather_wait");
  if (st != EB_OK) return st;
  return gather_step(c, g, true, [&](double* u0) {
    return eb_control_dev(c, xmin, xmax, ymin, ymax, x_dev, mem_idx_dev, u0, metric_dev);
  });
}

// eb_control_batch_dev whose first twists land in every rank's gathered buffer: the same machinery as the shared calls
eb_status eb_control_batch_dev_gather(eb_controller* c, eb_peer_group* g, const double* bounds_dev, const double* x_dev,
                                      const int* mem_idx_dev, double* metric_dev)
{
  EB_TRACE("eb_control_batch_dev_gather");
  const eb_status st = batch_gather_check(c, g, bounds_dev, x_dev, "eb_control_batch_dev_gather");
  if (st != EB_OK) return st;
  return gather_step(c, g, false, [&](double* u0) {
    return eb_control_batch_dev(c, bounds_dev, x_dev, mem_idx_dev, u0, metric_dev);
  });
}

eb_status eb_control_batch_dev_gather_wait(eb_controller* c, eb_peer_group* g, const double* bounds_dev,
                                           const double* x_dev, const int* mem_idx_dev, double* metric_dev)
{
  EB_TRACE("eb_control_batch_dev_gather_wait");
  const eb_status st = batch_gather_check(c, g, bounds_dev, x_dev, "eb_control_batch_dev_gather_wait");
  if (st != EB_OK) return st;
  return gather_step(c, g, true, [&](double* u0) {
    return eb_control_batch_dev(c, bounds_dev, x_dev, mem_idx_dev, u0, metric_dev);
  });
}

// enqueues (on the controller's stream) a wait until every rank's rows of step `step` have arrived here
eb_status eb_peer_group_wait(eb_peer_group* g, eb_controller* c, unsigned long long step)
{
  if (!g || !c) return fail(EB_ERR_INVALID_ARGUMENT, "eb_peer_group_wait: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  eb::peer_wait_kernel<<<1, 32, 0, c->stream>>>(g->flags, g->world, step);
  EB_CUDA(cudaGetLastError());
  c->launches += 1;
  return EB_OK;
}

// ---------------------------------------------------------------------------
// occupancy-grid collision checks (collision_kernels.cuh)
// ---------------------------------------------------------------------------
}  // extern "C"

struct eb_grid
{
  int device = 0;
  eb::GridView view{};
  signed char* d_data = nullptr;
  cudaStream_t stream = nullptr;
  double* d_a = nullptr;  // staging for the _host calls: poses / x0
  double* d_b = nullptr;  // twists
  double* d_u = nullptr;  // DynamicWindow: optimal twists
  double* d_cost = nullptr;
  double* d_ref = nullptr;  // DynamicWindow: reference twists / trajectories
  size_t ref_cap = 0;
  int* d_out = nullptr;
  int cap = 0;
  long long launches = 0;
  // pre-dilated map for one set of collision radii / threshold (collision_kernels.cuh, inflate_kernel)
  unsigned char* d_inflated = nullptr;
  short2* d_offsets = nullptr;
  bool infl_valid = false;
  int infl_key[3] = { -1, -1, -1 };  // r_bnd, r_last, r_col
  double infl_thr = 0.0;
  int infl_pad = 0;
  int dilation_mode = 0;  // 0 auto (by pose count), 1 never, 2 always
  // pipelined host path of DynamicWindow::control (dwa_host): second stream, and the dilation decision of the
  // WHOLE batch while its chunks are launched one by one
  cudaStream_t side = nullptr;
  cudaEvent_t ev_ready = nullptr, ev_side = nullptr;
  long long batch_poses = -1;
};

namespace
{
// the checks of the Collision constructor (collision.cpp:46-64) and the radii of
// CollisionConfig (collision.cpp:130-133)
eb_status collision_check_config(const eb_collision* c)
{
  if (c->search_radius < c->boundary_radius)
    return fail(EB_ERR_INVALID_ARGUMENT, "Search radius must be at least the same size as the boundary radius");
  if (c->occupied_threshold > 100.0 || c->occupied_threshold < 0.0)
    return fail(EB_ERR_INVALID_ARGUMENT, "Occupied threshold must be between 0 and 100");
  return EB_OK;
}

eb_status collision_params(const eb_grid* g, const eb_collision* c, eb::CollisionParams* p)
{
  if (!g || !c) return fail(EB_ERR_INVALID_ARGUMENT, "grid / collision is NULL");
  const eb_status st = collision_check_config(c);
  if (st != EB_OK) return st;
  p->g = g->view;
  p->r_bnd = (int)std::floor(c->boundary_radius / g->view.resolution);
  p->r_col = (int)std::floor((c->boundary_radius + c->obstacle_threshold) / g->view.resolution);
  p->r_max = (int)std::floor(c->search_radius / g->view.resolution);
  p->occupied_threshold = c->occupied_threshold;
  return EB_OK;
}

// Points p at the dilated map of (g, radii, threshold), building it if `build`; with
// build = false it is used only when it already exists for exactly these parameters.
eb_status use_inflated(eb_grid* g, eb::CollisionParams* p, bool build)
{
  const int r_last = eb::prune_radius(p->r_col, p->r_max);
  const bool match = g->infl_valid && g->infl_key[0] == p->r_bnd && g->infl_key[1] == r_last &&
                     g->infl_key[2] == p->r_col && g->infl_thr == p->occupied_threshold;
  if (g->dilation_mode == 1) return EB_OK;
  if (g->dilation_mode == 2) build = true;
  if (!match)
  {
    if (!build) return EB_OK;
    if (p->r_col < 0 || p->r_col > 30000) return EB_OK;  // degenerate radii: keep the direct walk
    // the fixed offset set: cells of the reference's circle walks that can report a collision
    std::vector<short2> offs;
    {
      std::vector<long long> seen;
      for (int r0 = std::max(p->r_bnd, 0); r0 <= r_last; r0++)
      {
        int x = -r0, y = 0, err = 2 - 2 * r0;
        while (x < 0)
        {
          const int q[4][2] = { { -x, y }, { -y, -x }, { x, -y }, { y, x } };
          for (auto& d : q)
            if ((long long)d[0] * d[0] + (long long)d[1] * d[1] <= (long long)p->r_col * p->r_col)
              seen.push_back(((long long)(d[0] + 32768) << 20) | (long long)(d[1] + 32768));
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
      std::sort(seen.begin(), seen.end());
      seen.erase(std::unique(seen.begin(), seen.end()), seen.end());
      for (long long v : seen) offs.push_back(make_short2((short)((v >> 20) - 32768), (short)((v & 0xfffff) - 32768)));
    }
    const int pad = std::max(p->r_col, 0);
    const size_t pw = (size_t)g->view.xsize + 2 * (size_t)pad, ph = (size_t)g->view.ysize + 2 * (size_t)pad;
    cudaFree(g->d_inflated);
    cudaFree(g->d_offsets);
    g->d_inflated = nullptr;
    g->d_offsets = nullptr;
    g->infl_valid = false;
    EB_CUDA(cudaMalloc(&g->d_inflated, pw * ph));
    EB_CUDA(cudaMalloc(&g->d_offsets, sizeof(short2) * std::max<size_t>(offs.size(), 1)));
    EB_CUDA(cudaMemcpyAsync(g->d_offsets, offs.data(), sizeof(short2) * offs.size(), cudaMemcpyHostToDevice, g->stream));
    EB_CUDA(cudaStreamSynchronize(g->stream));  // offs is a stack-lifetime buffer
    const size_t total = pw * ph;
    // gather per centre, or scatter from the occupied cells when they are few (the usual case)
    unsigned long long* d_count = nullptr;
    unsigned long long occupied = 0;
    const size_t cells = (size_t)g->view.xsize * g->view.ysize;
    EB_CUDA(cudaMalloc(&d_count, sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), g->stream);
    if (e == cudaSuccess)
    {
      eb::count_occupied_kernel<<<(unsigned)std::min<size_t>((cells + 255) / 256, 4096), 256, 0, g->stream>>>(
          g->view, p->occupied_threshold, d_count);
      e = cudaMemcpyAsync(&occupied, d_count, sizeof(occupied), cudaMemcpyDeviceToHost, g->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->stream);
    cudaFree(d_count);
    if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("dilated map: ") + cudaGetErrorString(e));
    if (occupied * 4 <= cells)
    {
      EB_CUDA(cudaMemsetAsync(g->d_inflated, 0, total, g->stream));
      eb::inflate_scatter_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, g->stream>>>(
          g->view, p->occupied_threshold, g->d_offsets, (int)offs.size(), pad, g->d_inflated);
    }
    else
      eb::inflate_kernel<<<(unsigned)((total + 255) / 256), 256, 0, g->stream>>>(g->view, p->occupied_threshold,
                                                                                   g->d_offsets, (int)offs.size(), pad,
                                                                                   g->d_inflated);
    EB_CUDA(cudaGetLastError());
    g->launches += 2;
    g->infl_key[0] = p->r_bnd;
    g->infl_key[1] = r_last;
    g->infl_key[2] = p->r_col;
    g->infl_thr = p->occupied_threshold;
    g->infl_pad = pad;
    g->infl_valid = true;
  }
  p->inflated = g->d_inflated;
  p->pad = g->infl_pad;
  return EB_OK;
}

// staging of the _host calls (eb_grid, eb_grid_batch): grown on demand, so a control loop pays no allocation per tick
template <class G>
eb_status grid_reserve(G* g, int count)
{
  if (count <= g->cap) return EB_OK;
  cudaFree(g->d_a);
  cudaFree(g->d_b);
  cudaFree(g->d_u);
  cudaFree(g->d_cost);
  cudaFree(g->d_out);
  g->d_a = g->d_b = g->d_u = g->d_cost = nullptr;
  g->d_out = nullptr;
  g->cap = 0;
  EB_CUDA(cudaMalloc(&g->d_a, sizeof(double) * 3 * (size_t)count));
  EB_CUDA(cudaMalloc(&g->d_b, sizeof(double) * 3 * (size_t)count));
  EB_CUDA(cudaMalloc(&g->d_u, sizeof(double) * 3 * (size_t)count));
  EB_CUDA(cudaMalloc(&g->d_cost, sizeof(double) * (size_t)count));
  EB_CUDA(cudaMalloc(&g->d_out, sizeof(int) * (size_t)count));
  g->cap = count;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_grid_create(int device, const signed char* data, unsigned int xsize, unsigned int ysize,
                         double resolution, double xmin, double ymin, eb_grid** out)
{
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_create: out is NULL");
  *out = nullptr;
  if (!data || xsize == 0 || ysize == 0 || !(resolution > 0.0))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_create: need data, xsize, ysize >= 1 and resolution > 0");
  EB_CUDA(cudaSetDevice(device));
  eb_grid* g = new (std::nothrow) eb_grid();
  if (!g) return fail(EB_ERR_CUDA, "out of host memory");
  g->device = device;
  const size_t cells = (size_t)xsize * ysize;
  cudaError_t e = cudaMalloc(&g->d_data, cells);
  if (e == cudaSuccess) e = cudaMemcpy(g->d_data, data, cells, cudaMemcpyHostToDevice);
  if (e != cudaSuccess)
  {
    eb_grid_destroy(g);
    return fail(EB_ERR_CUDA, std::string("eb_grid_create: ") + cudaGetErrorString(e));
  }
  g->view = eb::GridView{ g->d_data, xsize, ysize, resolution, xmin, ymin };
  *out = g;
  return EB_OK;
}

eb_status eb_grid_update(eb_grid* g, const signed char* data)
{
  if (!g || !data) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_update: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  EB_CUDA(cudaMemcpyAsync(g->d_data, data, (size_t)g->view.xsize * g->view.ysize, cudaMemcpyHostToDevice, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  g->infl_valid = false;  // the dilated map belongs to the old cells
  return EB_OK;
}

void eb_grid_destroy(eb_grid* g)
{
  if (!g) return;
  cudaSetDevice(g->device);
  cudaFree(g->d_data);
  cudaFree(g->d_inflated);
  cudaFree(g->d_offsets);
  cudaFree(g->d_a);
  cudaFree(g->d_b);
  cudaFree(g->d_u);
  cudaFree(g->d_cost);
  cudaFree(g->d_ref);
  cudaFree(g->d_out);
  if (g->side) cudaStreamDestroy(g->side);
  if (g->ev_ready) cudaEventDestroy(g->ev_ready);
  if (g->ev_side) cudaEventDestroy(g->ev_side);
  delete g;
}

eb_status eb_grid_set_stream(eb_grid* g, void* s)
{
  if (!g) return fail(EB_ERR_INVALID_ARGUMENT, "grid is NULL");
  g->stream = static_cast<cudaStream_t>(s);
  return EB_OK;
}

long long eb_grid_launch_count(const eb_grid* g) { return g ? g->launches : 0; }

eb_status eb_grid_set_dilation(eb_grid* g, int mode)
{
  if (!g || mode < 0 || mode > 2) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_set_dilation: mode must be 0, 1 or 2");
  g->dilation_mode = mode;
  return EB_OK;
}

eb_status eb_collision_check_dev(eb_grid* g, const eb_collision* c, const double* poses_dev, int count, int* hit_dev)
{
  EB_TRACE("eb_collision_check_dev");
  eb::CollisionParams p{};
  eb_status st = collision_params(g, c, &p);
  if (st != EB_OK) return st;
  if (count < 0 || (count > 0 && (!poses_dev || !hit_dev)))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_collision_check: bad arguments");
  if (count == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(g->device));
  p.B = count;
  p.x0 = poses_dev;
  p.out = hit_dev;
  // a dilated map pays once the poses outnumber a fraction of the cells; an existing one is free
  st = use_inflated(g, &p, (long long)count * 4 >= (long long)g->view.xsize * g->view.ysize);
  if (st != EB_OK) return st;
  eb::collision_check_kernel<false><<<(count + 127) / 128, 128, 0, g->stream>>>(p, eb::MapSet{});
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}

eb_status eb_validate_control_dev(eb_grid* g, const eb_collision* c, const double* x0_dev, const double* u_dev,
                                  int count, double dt, double horizon, int* valid_dev)
{
  EB_TRACE("eb_validate_control_dev");
  eb::CollisionParams p{};
  eb_status st = collision_params(g, c, &p);
  if (st != EB_OK) return st;
  if (count < 0 || (count > 0 && (!x0_dev || !u_dev || !valid_dev)) || dt == 0.0)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_validate_control: bad arguments");
  if (count == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(g->device));
  p.B = count;
  p.x0 = x0_dev;
  p.u = u_dev;
  p.out = valid_dev;
  p.dt = dt;
  p.steps = (int)static_cast<unsigned int>(std::abs(horizon / dt));  // numerics.hpp:316
  st = use_inflated(g, &p, (long long)count * p.steps * 4 >= (long long)g->view.xsize * g->view.ysize);
  if (st != EB_OK) return st;
  eb::validate_control_kernel<false><<<(count + 127) / 128, 128, 0, g->stream>>>(p, eb::MapSet{});
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}

eb_status eb_collision_check_host(eb_grid* g, const eb_collision* c, const double* poses, int count, int* hit)
{
  if (!g) return fail(EB_ERR_INVALID_ARGUMENT, "grid is NULL");
  if (count > 0 && (!poses || !hit)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_collision_check_host: NULL argument");
  if (count <= 0) return count == 0 ? EB_OK : fail(EB_ERR_INVALID_ARGUMENT, "count < 0");
  EB_CUDA(cudaSetDevice(g->device));
  eb_status st = grid_reserve(g, count);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(g->d_a, poses, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice, g->stream));
  st = eb_collision_check_dev(g, c, g->d_a, count, g->d_out);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(hit, g->d_out, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

eb_status eb_validate_control_host(eb_grid* g, const eb_collision* c, const double* x0, const double* u, int count,
                                   double dt, double horizon, int* valid)
{
  if (!g) return fail(EB_ERR_INVALID_ARGUMENT, "grid is NULL");
  if (count > 0 && (!x0 || !u || !valid)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_validate_control_host: NULL argument");
  if (count <= 0) return count == 0 ? EB_OK : fail(EB_ERR_INVALID_ARGUMENT, "count < 0");
  EB_CUDA(cudaSetDevice(g->device));
  eb_status st = grid_reserve(g, count);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(g->d_a, x0, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice, g->stream));
  EB_CUDA(cudaMemcpyAsync(g->d_b, u, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice, g->stream));
  st = eb_validate_control_dev(g, c, g->d_a, g->d_b, count, dt, horizon, g->d_out);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(valid, g->d_out, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

// integrate_twist + normalize_angle_PI (numerics.hpp:273-298, 77-89), batched, on `stream`
eb_status eb_integrate_twist_dev(int device, const double* x_dev, const double* u_dev, double dt, int count,
                                 double* out_dev, void* cuda_stream)
{
  if (count < 0 || (count > 0 && (!x_dev || !u_dev || !out_dev)))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_integrate_twist_dev: bad arguments");
  if (count == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(device));
  eb::integrate_twist_kernel<<<(count + 255) / 256, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(x_dev, u_dev, dt,
                                                                                                      count, out_dev);
  EB_CUDA(cudaGetLastError());
  return EB_OK;
}

// ---- DynamicWindow::control (dynamic_window.cpp:93-187) -----------------------------
}  // extern "C"

namespace
{
// everything of DwaParams but the grid and the radii in p->col
eb_status dwa_window_params(const eb_dwa* d, int count, eb::DwaParams* p)
{
  if (count < 0 || d->dt == 0.0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control: bad arguments");
  p->col.dt = d->dt;
  p->col.steps = (int)static_cast<unsigned int>(std::abs(d->horizon / d->dt));  // dynamic_window.cpp:69
  p->B = count;
  p->acc_dt = d->acc_dt;
  const double acc[3] = { d->acc_lim_x, d->acc_lim_y, d->acc_lim_th };
  const double vmin[3] = { d->min_vel_x, d->min_vel_y, d->min_rot_vel };
  const double vmax[3] = { d->max_vel_x, d->max_vel_y, d->max_rot_vel };
  const unsigned int n[3] = { d->vx_samples, d->vy_samples, d->vth_samples };
  for (int a = 0; a < 3; a++)
  {
    p->acc_lim[a] = acc[a];
    p->vmin[a] = vmin[a];
    p->vmax[a] = vmax[a];
    p->n[a] = n[a] ? n[a] : 1u;  // dynamic_window.cpp:71-91: 0 samples -> 1
  }
  return EB_OK;
}

eb_status dwa_params(const eb_grid* g, const eb_collision* c, const eb_dwa* d, int count, eb::DwaParams* p)
{
  if (!d) return fail(EB_ERR_INVALID_ARGUMENT, "dwa is NULL");
  eb_status st = collision_params(g, c, &p->col);
  if (st != EB_OK) return st;
  return dwa_window_params(d, count, p);
}

// the reference trajectory of DynamicWindow::control (dynamic_window.cpp:141-187) in p
eb_status dwa_traj_params(const double* xt_ref_dev, int ncols, int per_instance, double dt_ref, eb::DwaParams* p)
{
  p->xt_ref = xt_ref_dev;
  p->ncols = ncols;
  p->xt_stride = per_instance ? 3LL * ncols : 0LL;
  p->tf = static_cast<double>(ncols) * dt_ref;  // dynamic_window.cpp:148
  // dynamic_window.cpp:276 indexes xt_ref with round((ncols - 1) * t / tf), t accumulated per rollout step; Armadillo's
  // bounds check throws when the rollout outlasts the reference trajectory -- refuse it here instead of reading past it
  double t = 0.0;
  for (int k = 0; k + 1 < p->col.steps; k++) t += p->col.dt;
  const double jmax = std::round((static_cast<double>(ncols - 1) * t) / p->tf);
  if (!(jmax <= static_cast<double>(ncols - 1)))
    return fail(EB_ERR_OUT_OF_RANGE, "eb_dwa_control_traj: the rollout horizon outlasts the reference trajectory "
                                     "(index past the last column; the reference's Armadillo access throws here)");
  return EB_OK;
}

eb_status dwa_launch(eb_grid* g, eb::DwaParams& p)
{
  if (p.B == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(g->device));
  {
    const long long poses =
        g->batch_poses >= 0 ? g->batch_poses : (long long)p.B * p.col.steps * p.n[0] * p.n[1] * p.n[2];
    const eb_status st = use_inflated(g, &p.col, poses * 4 >= (long long)g->view.xsize * g->view.ysize);
    if (st != EB_OK) return st;
  }
  const int threads = 128, warps_per_block = threads / 32;
  eb::dwa_control_kernel<false><<<(p.B + warps_per_block - 1) / warps_per_block, threads, 0, g->stream>>>(p, eb::MapSet{});
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_dwa_control_twist_dev(eb_grid* g, const eb_collision* c, const eb_dwa* d, const double* x0_dev,
                                   const double* vb_dev, const double* vref_dev, int count, int* found_dev,
                                   double* u_opt_dev, double* min_cost_dev)
{
  EB_TRACE("eb_dwa_control_twist_dev");
  eb::DwaParams p{};
  eb_status st = dwa_params(g, c, d, count, &p);
  if (st != EB_OK) return st;
  if (count > 0 && (!x0_dev || !vb_dev || !vref_dev || !found_dev || !u_opt_dev))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_twist: NULL argument");
  p.x0 = x0_dev;
  p.vb = vb_dev;
  p.vref = vref_dev;
  p.found = found_dev;
  p.u_opt = u_opt_dev;
  p.min_cost = min_cost_dev;
  return dwa_launch(g, p);
}

eb_status eb_dwa_control_traj_dev(eb_grid* g, const eb_collision* c, const eb_dwa* d, const double* x0_dev,
                                  const double* vb_dev, const double* xt_ref_dev, int ncols, int per_instance,
                                  double dt_ref, int count, int* found_dev, double* u_opt_dev, double* min_cost_dev)
{
  EB_TRACE("eb_dwa_control_traj_dev");
  eb::DwaParams p{};
  eb_status st = dwa_params(g, c, d, count, &p);
  if (st != EB_OK) return st;
  if (ncols < 1 || (count > 0 && (!x0_dev || !vb_dev || !xt_ref_dev || !found_dev || !u_opt_dev)))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_traj: bad arguments");
  p.x0 = x0_dev;
  p.vb = vb_dev;
  st = dwa_traj_params(xt_ref_dev, ncols, per_instance, dt_ref, &p);
  if (st != EB_OK) return st;
  p.found = found_dev;
  p.u_opt = u_opt_dev;
  p.min_cost = min_cost_dev;
  return dwa_launch(g, p);
}

static eb_status dwa_host(eb_grid* g, const eb_collision* c, const eb_dwa* d, const double* x0, const double* vb,
                          const double* ref, size_t ref_doubles, bool traj, int ncols, int per_instance, double dt_ref,
                          int count, int* found, double* u_opt, double* min_cost)
{
  if (!g) return fail(EB_ERR_INVALID_ARGUMENT, "grid is NULL");
  if (count < 0 || (count > 0 && (!x0 || !vb || !ref || !found || !u_opt)))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_host: bad arguments");
  if (count == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(g->device));
  // staging buffers live with the grid (grown on demand), so a control loop pays no allocation per tick
  eb_status st = grid_reserve(g, count);
  if (st != EB_OK) return st;
  if (ref_doubles > g->ref_cap)
  {
    cudaFree(g->d_ref);
    g->d_ref = nullptr;
    g->ref_cap = 0;
    EB_CUDA(cudaMalloc(&g->d_ref, sizeof(double) * ref_doubles));
    g->ref_cap = ref_doubles;
  }
  auto pinned = [](const void* ptr) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess)
    {
      cudaGetLastError();
      return false;
    }
    return a.type == cudaMemoryTypeHost;
  };
  auto run = [&](int lo, int n, bool copy_shared_ref) -> eb_status {
    // one slice [lo, lo + n) of the batch on the grid's CURRENT stream: H2D, kernel, D2H
    cudaStream_t s = g->stream;
    const size_t o3 = 3 * (size_t)lo;
    cudaError_t e = cudaMemcpyAsync(g->d_a + o3, x0 + o3, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(g->d_b + o3, vb + o3, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, s);
    const double* dref = g->d_ref;
    if (!traj || per_instance)
    {
      const size_t per = traj ? 3 * (size_t)ncols : 3;  // doubles of reference data per instance
      dref = g->d_ref + per * (size_t)lo;
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(g->d_ref + per * (size_t)lo, ref + per * (size_t)lo, sizeof(double) * per * (size_t)n, cudaMemcpyHostToDevice, s);
    }
    else if (copy_shared_ref && e == cudaSuccess)
      e = cudaMemcpyAsync(g->d_ref, ref, sizeof(double) * ref_doubles, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_dwa_control_host: ") + cudaGetErrorString(e));
    eb_status r = traj ? eb_dwa_control_traj_dev(g, c, d, g->d_a + o3, g->d_b + o3, dref, ncols, per_instance, dt_ref, n,
                                                 g->d_out + lo, g->d_u + o3, g->d_cost + lo) :
                         eb_dwa_control_twist_dev(g, c, d, g->d_a + o3, g->d_b + o3, dref, n, g->d_out + lo, g->d_u + o3,
                                                  g->d_cost + lo);
    if (r != EB_OK) return r;
    e = cudaMemcpyAsync(found + lo, g->d_out + lo, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(u_opt + o3, g->d_u + o3, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && min_cost)
      e = cudaMemcpyAsync(min_cost + lo, g->d_cost + lo, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_dwa_control_host: ") + cudaGetErrorString(e));
    return EB_OK;
  };
  // Large batches from page-locked caller buffers are cut into slices that alternate between two streams, so the
  // copies of one slice overlap the kernel of the other (the copy engines and the SMs work at the same time);
  // pageable buffers would serialise in the driver's staging path anyway.
  constexpr int kSlice = 32768;
  const bool pipelined = count >= 4 * kSlice && pinned(x0) && pinned(vb) && pinned(ref) && pinned(found) && pinned(u_opt) &&
                         (!min_cost || pinned(min_cost));
  if (!pipelined)
  {
    st = run(0, count, true);
    if (st != EB_OK) return st;
    cudaError_t e = cudaStreamSynchronize(g->stream);
    if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_dwa_control_host: ") + cudaGetErrorString(e));
    return EB_OK;
  }
  if (!g->side)
  {
    EB_CUDA(cudaStreamCreateWithFlags(&g->side, cudaStreamNonBlocking));
    EB_CUDA(cudaEventCreateWithFlags(&g->ev_ready, cudaEventDisableTiming));
    EB_CUDA(cudaEventCreateWithFlags(&g->ev_side, cudaEventDisableTiming));
  }
  cudaStream_t const main_stream = g->stream;
  {
    // the dilation decision belongs to the whole batch; what the first slice builds (on the main stream) the others reuse
    const unsigned int ns[3] = { d->vx_samples ? d->vx_samples : 1u, d->vy_samples ? d->vy_samples : 1u,
                                 d->vth_samples ? d->vth_samples : 1u };
    const long long steps = (long long)static_cast<unsigned int>(std::abs(d->horizon / d->dt));
    g->batch_poses = (long long)count * steps * ns[0] * ns[1] * ns[2];
  }
  st = EB_OK;
  int slice = 0;
  for (int lo = 0; lo < count && st == EB_OK; lo += kSlice, slice++)
  {
    const int n = std::min(kSlice, count - lo);
    g->stream = (slice & 1) ? g->side : main_stream;
    st = run(lo, n, slice == 0);
    if (slice == 0 && st == EB_OK)
    {
      // map (possibly rebuilt) and shared reference data are in place once the first slice's work is enqueued
      cudaEventRecord(g->ev_ready, main_stream);
      cudaStreamWaitEvent(g->side, g->ev_ready, 0);
    }
  }
  g->stream = main_stream;
  g->batch_poses = -1;
  cudaEventRecord(g->ev_side, g->side);
  cudaStreamWaitEvent(main_stream, g->ev_side, 0);
  cudaError_t e = cudaStreamSynchronize(main_stream);
  if (st != EB_OK) return st;
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_dwa_control_host: ") + cudaGetErrorString(e));
  return EB_OK;
}

eb_status eb_dwa_control_twist_host(eb_grid* g, const eb_collision* c, const eb_dwa* d, const double* x0,
                                    const double* vb, const double* vref, int count, int* found, double* u_opt,
                                    double* min_cost)
{
  return dwa_host(g, c, d, x0, vb, vref, 3 * (size_t)std::max(count, 0), false, 0, 0, 0.0, count, found, u_opt, min_cost);
}

eb_status eb_dwa_control_traj_host(eb_grid* g, const eb_collision* c, const eb_dwa* d, const double* x0,
                                   const double* vb, const double* xt_ref, int ncols, int per_instance, double dt_ref,
                                   int count, int* found, double* u_opt, double* min_cost)
{
  if (ncols < 1) return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_traj_host: ncols < 1");
  const size_t ref_doubles = 3 * (size_t)ncols * (per_instance ? (size_t)std::max(count, 0) : 1);
  return dwa_host(g, c, d, x0, vb, xt_ref, ref_doubles, true, ncols, per_instance, dt_ref, count, found, u_opt,
                  min_cost);
}

}  // extern "C"

// ---------------------------------------------------------------------------
// per-instance occupancy maps (eb_grid_batch): instance i's checks run against map i
// ---------------------------------------------------------------------------
struct eb_grid_batch
{
  int device = 0;
  int B = 0;
  cudaStream_t stream = nullptr;
  long long launches = 0;
  // host copy of the device records; data == nullptr: the instance has no map yet
  std::vector<eb::GridView> views;
  std::vector<size_t> slot;  // bytes of the arena reserved for each instance's map
  int unmapped = 0;
  eb::GridView* d_views = nullptr;
  signed char* d_arena = nullptr;
  signed char* d_retired = nullptr;  // the arena before the last relayout, read by that set call's copy kernel
  // set call: descriptors (pinned, one upload per call) and the _host call's packed cells
  eb::MapCopy* h_copies = nullptr;
  eb::MapCopy* d_copies = nullptr;
  cudaEvent_t staged = nullptr;  // the last upload out of h_copies has been made
  // eb_control_safe_batch_*: recorded on the grid batch's stream before a tick (maps_ready) and on the controller's
  // stream after it (ticked); the next set call waits for the last tick before it writes or frees an arena
  cudaEvent_t maps_ready = nullptr;
  cudaEvent_t ticked = nullptr;
  // eb_set_map_targets_from_grid_batch: this handle (unique per process) and, per map, how often a set call replaced it
  unsigned long long serial = 0;
  std::vector<unsigned long long> map_serial;
  eb::BandCopy* h_bands = nullptr;  // eb_grid_batch_set_rows_*: pinned band records, uploaded like h_copies
  eb::BandCopy* d_bands = nullptr;
  signed char* h_cells = nullptr;
  signed char* d_cells = nullptr;
  size_t cells_bytes = 0;
  // staging of the _host checks (grid_reserve)
  double* d_a = nullptr;
  double* d_b = nullptr;
  double* d_u = nullptr;
  double* d_cost = nullptr;
  double* d_ref = nullptr;
  size_t ref_cap = 0;
  int* d_out = nullptr;
  int cap = 0;
};

namespace
{
// arena slot of a map of `cells` bytes: a quarter of headroom, so a growing map does not relayout on every update
size_t grid_slot_bytes(size_t cells) { return (cells + cells / 4 + 255) & ~(size_t)255; }

// writes the flagged maps (device cell pointers) into their slots with one copy-kernel launch; when a flagged map
// outgrows its slot, every map moves to a new arena in the same launch
eb_status grid_batch_set(eb_grid_batch* g, const signed char* const* cells, const unsigned* xsize, const unsigned* ysize,
                         const double* resolution, const double* origin, const int* update, int n)
{
  if (n == 0) return EB_OK;
  const int B = g->B;
  EB_CUDA(cudaSetDevice(g->device));
  if (g->ticked) EB_CUDA(cudaStreamWaitEvent(g->stream, g->ticked, 0));  // a safe control tick may still read the maps
  if (!g->d_views)
  {
    EB_CUDA(cudaMalloc(&g->d_views, sizeof(eb::GridView) * (size_t)B));
    EB_CUDA(cudaHostAlloc(&g->h_copies, sizeof(eb::MapCopy) * (size_t)B, cudaHostAllocDefault));
    EB_CUDA(cudaMalloc(&g->d_copies, sizeof(eb::MapCopy) * (size_t)B));
    EB_CUDA(cudaEventCreateWithFlags(&g->staged, cudaEventDisableTiming));
  }
  bool relayout = false;
  for (int i = 0; i < B && !relayout; i++)
    relayout = !(update && !update[i]) && (size_t)xsize[i] * ysize[i] > g->slot[i];
  std::vector<size_t> slot = g->slot;
  signed char* arena = g->d_arena;
  if (relayout)
  {
    size_t total = 0;
    for (int i = 0; i < B; i++)
    {
      const bool flagged = !(update && !update[i]);
      const size_t cells_i = flagged ? (size_t)xsize[i] * ysize[i] :
                                       (g->views[i].data ? (size_t)g->views[i].xsize * g->views[i].ysize : 0);
      slot[i] = grid_slot_bytes(cells_i);
      total += slot[i];
    }
    if (g->d_retired)
    {
      EB_CUDA(cudaStreamSynchronize(g->stream));  // its copy kernel has run
      cudaFree(g->d_retired);
      g->d_retired = nullptr;
    }
    EB_CUDA(cudaMalloc(&arena, total));
  }
  cudaError_t e = cudaEventSynchronize(g->staged);  // the previous call's upload out of h_copies is done
  std::vector<eb::GridView> views = g->views;
  int k = 0;
  size_t off = 0;
  for (int i = 0; i < B; i++)
  {
    signed char* dst = arena + off;
    off += slot[i];
    if (!(update && !update[i]))
    {
      views[i] = eb::GridView{ dst, xsize[i], ysize[i], resolution[i], origin[2 * i + 0], origin[2 * i + 1] };
      g->h_copies[k++] = eb::MapCopy{ cells[i], views[i], i };
    }
    else if (relayout && views[i].data)
    {
      const signed char* src = views[i].data;
      views[i].data = dst;
      g->h_copies[k++] = eb::MapCopy{ src, views[i], i };
    }
  }
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(g->d_copies, g->h_copies, sizeof(eb::MapCopy) * (size_t)k, cudaMemcpyHostToDevice, g->stream);
  if (e == cudaSuccess) e = cudaEventRecord(g->staged, g->stream);
  if (e == cudaSuccess)
  {
    eb::map_copy_kernel<<<k, 256, 0, g->stream>>>(g->d_copies, g->d_views);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess)
  {
    if (relayout) cudaFree(arena);
    return fail(EB_ERR_CUDA, std::string("eb_grid_batch_set_maps: ") + cudaGetErrorString(e));
  }
  g->launches += 1;
  if (relayout)
  {
    g->d_retired = g->d_arena;
    g->d_arena = arena;
    g->slot = slot;
  }
  for (int i = 0; i < B; i++)
  {
    g->unmapped -= (!g->views[i].data && views[i].data) ? 1 : 0;
    g->map_serial[i] += (update && !update[i]) ? 0 : 1;  // kept target blocks of the old map are stale
  }
  g->views = views;
  return EB_OK;
}

// the argument rules of eb_set_map_targets_batch_* for the flagged maps; *n = flagged maps
eb_status grid_batch_check_maps(const eb_grid_batch* g, const signed char* const* cells, const unsigned* xsize,
                                const unsigned* ysize, const double* resolution, const double* origin, const int* update,
                                const char* call, int* n)
{
  *n = 0;
  if (!g || !cells || !xsize || !ysize || !resolution || !origin)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  for (int i = 0; i < g->B; i++)
  {
    if (update && !update[i]) continue;
    if (xsize[i] < 1 || ysize[i] < 1 || !(resolution[i] > 0.0) || !std::isfinite(resolution[i]))
      return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": map " + std::to_string(i) +
                                               " needs xsize, ysize >= 1 and a finite resolution > 0");
    if ((unsigned long long)xsize[i] * ysize[i] > 0x7fffffffull)
      return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": map " + std::to_string(i) + " has more than 2^31 - 1 cells");
    if (!cells[i]) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": cells of map " + std::to_string(i) + " is NULL");
    (*n)++;
  }
  return EB_OK;
}

// the collision part of a per-map check: Collision constructor checks, every instance has a map, per * B poses
eb_status grid_batch_params(const eb_grid_batch* g, const eb_collision* c, int per, eb::CollisionParams* p,
                            eb::MapSet* m)
{
  if (!g || !c) return fail(EB_ERR_INVALID_ARGUMENT, "grid batch / collision is NULL");
  const eb_status st = collision_check_config(c);
  if (st != EB_OK) return st;
  if (per < 1) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch: per must be >= 1");
  if ((long long)per * g->B > 0x7fffffffLL) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch: per * B overflows int");
  if (g->unmapped > 0)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch: " + std::to_string(g->unmapped) + " instance(s) have no map yet");
  p->occupied_threshold = c->occupied_threshold;
  p->B = per * g->B;
  *m = eb::MapSet{ g->d_views, per, c->boundary_radius, c->boundary_radius + c->obstacle_threshold, c->search_radius };
  return EB_OK;
}

eb_status grid_batch_dwa(eb_grid_batch* g, const eb_collision* c, const eb_dwa* d, eb::DwaParams* p, eb::MapSet* m)
{
  if (!d) return fail(EB_ERR_INVALID_ARGUMENT, "dwa is NULL");
  eb_status st = grid_batch_params(g, c, 1, &p->col, m);
  if (st != EB_OK) return st;
  return dwa_window_params(d, g->B, p);
}

eb_status grid_batch_dwa_launch(eb_grid_batch* g, const eb::DwaParams& p, const eb::MapSet& m)
{
  EB_CUDA(cudaSetDevice(g->device));
  const int threads = 128, warps_per_block = threads / 32;
  eb::dwa_control_kernel<true><<<(p.B + warps_per_block - 1) / warps_per_block, threads, 0, g->stream>>>(p, m);
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_grid_batch_create(int device, int batch, eb_grid_batch** out)
{
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch_create: out is NULL");
  *out = nullptr;
  if (batch < 1) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch_create: batch must be >= 1");
  EB_CUDA(cudaSetDevice(device));
  EB_CUDA(cudaFree(nullptr));  // a usable device, or EB_ERR_NO_DEVICE here rather than at the first set call
  eb_grid_batch* g = new (std::nothrow) eb_grid_batch();
  if (!g) return fail(EB_ERR_CUDA, "out of host memory");
  g->device = device;
  g->B = batch;
  g->views.assign((size_t)batch, eb::GridView{});
  g->slot.assign((size_t)batch, 0);
  g->map_serial.assign((size_t)batch, 0);
  static std::atomic<unsigned long long> next_serial{ 0 };
  g->serial = ++next_serial;
  g->unmapped = batch;
  *out = g;
  return EB_OK;
}

void eb_grid_batch_destroy(eb_grid_batch* g)
{
  if (!g) return;
  cudaSetDevice(g->device);
  if (g->staged) cudaEventSynchronize(g->staged);
  if (g->ticked) cudaEventSynchronize(g->ticked);
  cudaFree(g->d_views);
  cudaFree(g->d_arena);
  cudaFree(g->d_retired);
  cudaFreeHost(g->h_copies);
  cudaFree(g->d_copies);
  cudaFreeHost(g->h_bands);
  cudaFree(g->d_bands);
  cudaFreeHost(g->h_cells);
  cudaFree(g->d_cells);
  cudaFree(g->d_a);
  cudaFree(g->d_b);
  cudaFree(g->d_u);
  cudaFree(g->d_cost);
  cudaFree(g->d_ref);
  cudaFree(g->d_out);
  if (g->staged) cudaEventDestroy(g->staged);
  if (g->maps_ready) cudaEventDestroy(g->maps_ready);
  if (g->ticked) cudaEventDestroy(g->ticked);
  delete g;
}

eb_status eb_grid_batch_set_stream(eb_grid_batch* g, void* s)
{
  if (!g) return fail(EB_ERR_INVALID_ARGUMENT, "grid batch is NULL");
  g->stream = static_cast<cudaStream_t>(s);
  return EB_OK;
}

long long eb_grid_batch_launch_count(const eb_grid_batch* g) { return g ? g->launches : 0; }

eb_status eb_grid_batch_set_maps_dev(eb_grid_batch* g, const signed char* const* cells_dev, const unsigned* xsize,
                                     const unsigned* ysize, const double* resolution, const double* origin,
                                     const int* update)
{
  EB_TRACE("eb_grid_batch_set_maps_dev");
  int n = 0;
  const eb_status st =
      grid_batch_check_maps(g, cells_dev, xsize, ysize, resolution, origin, update, "eb_grid_batch_set_maps_dev", &n);
  if (st != EB_OK) return st;
  return grid_batch_set(g, cells_dev, xsize, ysize, resolution, origin, update, n);
}

eb_status eb_grid_batch_set_maps_host(eb_grid_batch* g, const signed char* const* cells, const unsigned* xsize,
                                      const unsigned* ysize, const double* resolution, const double* origin,
                                      const int* update)
{
  EB_TRACE("eb_grid_batch_set_maps_host");
  int n = 0;
  eb_status st = grid_batch_check_maps(g, cells, xsize, ysize, resolution, origin, update, "eb_grid_batch_set_maps_host", &n);
  if (st != EB_OK || n == 0) return st;
  // the flagged maps are packed into one pinned buffer (16-byte aligned offsets) and copied with one cudaMemcpyAsync
  std::vector<size_t> off((size_t)g->B, 0);
  size_t total = 0;
  for (int i = 0; i < g->B; i++)
  {
    if (update && !update[i]) continue;
    off[i] = total;
    total += ((size_t)xsize[i] * ysize[i] + 15) & ~(size_t)15;
  }
  EB_CUDA(cudaSetDevice(g->device));
  EB_CUDA(cudaStreamSynchronize(g->stream));  // no earlier copy still reads the staging buffers
  if (total > g->cells_bytes)
  {
    cudaFreeHost(g->h_cells);
    cudaFree(g->d_cells);
    g->h_cells = nullptr;
    g->d_cells = nullptr;
    g->cells_bytes = 0;
    EB_CUDA(cudaHostAlloc(&g->h_cells, total, cudaHostAllocDefault));
    EB_CUDA(cudaMalloc(&g->d_cells, total));
    g->cells_bytes = total;
  }
  std::vector<const signed char*> dptr((size_t)g->B, nullptr);
  for (int i = 0; i < g->B; i++)
    if (!(update && !update[i]))
    {
      std::memcpy(g->h_cells + off[i], cells[i], (size_t)xsize[i] * ysize[i]);
      dptr[i] = g->d_cells + off[i];
    }
  EB_CUDA(cudaMemcpyAsync(g->d_cells, g->h_cells, total, cudaMemcpyHostToDevice, g->stream));
  st = grid_batch_set(g, dptr.data(), xsize, ysize, resolution, origin, update, n);
  if (st != EB_OK) return st;
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

}  // extern "C"

namespace
{
// the rules of eb_grid_batch_set_rows_*; *n = bands with rows to write
eb_status grid_batch_check_rows(const eb_grid_batch* g, const signed char* const* rows, const unsigned* row_begin,
                                const unsigned* row_count, const int* update, const char* call, int* n)
{
  *n = 0;
  if (!g || !rows || !row_begin || !row_count) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  for (int i = 0; i < g->B; i++)
  {
    if (update && !update[i]) continue;
    const eb::GridView& v = g->views[i];
    if (!v.data) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": instance " + std::to_string(i) + " has no map");
    if ((unsigned long long)row_begin[i] + row_count[i] > v.ysize)
      return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": rows [" + std::to_string(row_begin[i]) + ", +" +
                                               std::to_string(row_count[i]) + ") of map " + std::to_string(i) +
                                               " pass its " + std::to_string(v.ysize) + " rows");
    if (row_count[i] == 0) continue;
    if (!rows[i]) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": rows of map " + std::to_string(i) + " is NULL");
    (*n)++;
  }
  return EB_OK;
}

// writes the bands (device pointers) into the arena with one band_copy_kernel launch
eb_status grid_batch_set_rows(eb_grid_batch* g, const signed char* const* rows, const unsigned* row_begin,
                              const unsigned* row_count, const int* update, int n)
{
  if (n == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(g->device));
  if (!g->h_bands)
  {
    EB_CUDA(cudaHostAlloc(&g->h_bands, sizeof(eb::BandCopy) * (size_t)g->B, cudaHostAllocDefault));
    EB_CUDA(cudaMalloc(&g->d_bands, sizeof(eb::BandCopy) * (size_t)g->B));
  }
  EB_CUDA(cudaEventSynchronize(g->staged));  // the previous upload out of the pinned records is done
  int k = 0;
  for (int i = 0; i < g->B; i++)
  {
    if ((update && !update[i]) || row_count[i] == 0) continue;
    const eb::GridView& v = g->views[i];
    signed char* dst = const_cast<signed char*>(v.data) + (size_t)row_begin[i] * v.xsize;
    g->h_bands[k++] = eb::BandCopy{ rows[i], dst, (size_t)row_count[i] * v.xsize };
  }
  // the records go up before the wait for the last tick, so the next call's wait on `staged` does not wait for it
  EB_CUDA(cudaMemcpyAsync(g->d_bands, g->h_bands, sizeof(eb::BandCopy) * (size_t)k, cudaMemcpyHostToDevice, g->stream));
  EB_CUDA(cudaEventRecord(g->staged, g->stream));
  if (g->ticked) EB_CUDA(cudaStreamWaitEvent(g->stream, g->ticked, 0));  // a tick or target call may still read the maps
  eb::band_copy_kernel<<<k, 256, 0, g->stream>>>(g->d_bands);
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_grid_batch_set_rows_dev(eb_grid_batch* g, const signed char* const* rows_dev, const unsigned* row_begin,
                                     const unsigned* row_count, const int* update)
{
  EB_TRACE("eb_grid_batch_set_rows_dev");
  int n = 0;
  const eb_status st = grid_batch_check_rows(g, rows_dev, row_begin, row_count, update, "eb_grid_batch_set_rows_dev", &n);
  if (st != EB_OK) return st;
  return grid_batch_set_rows(g, rows_dev, row_begin, row_count, update, n);
}

eb_status eb_grid_batch_set_rows_host(eb_grid_batch* g, const signed char* const* rows, const unsigned* row_begin,
                                      const unsigned* row_count, const int* update)
{
  EB_TRACE("eb_grid_batch_set_rows_host");
  int n = 0;
  eb_status st = grid_batch_check_rows(g, rows, row_begin, row_count, update, "eb_grid_batch_set_rows_host", &n);
  if (st != EB_OK || n == 0) return st;
  // the bands are packed into the set call's pinned buffer (16-byte aligned offsets) and copied with one
  // cudaMemcpyAsync
  std::vector<size_t> off((size_t)g->B, 0);
  size_t total = 0;
  for (int i = 0; i < g->B; i++)
  {
    if ((update && !update[i]) || row_count[i] == 0) continue;
    off[i] = total;
    total += ((size_t)row_count[i] * g->views[i].xsize + 15) & ~(size_t)15;
  }
  EB_CUDA(cudaSetDevice(g->device));
  EB_CUDA(cudaStreamSynchronize(g->stream));  // no earlier copy still reads the staging buffers
  if (total > g->cells_bytes)
  {
    cudaFreeHost(g->h_cells);
    cudaFree(g->d_cells);
    g->h_cells = nullptr;
    g->d_cells = nullptr;
    g->cells_bytes = 0;
    EB_CUDA(cudaHostAlloc(&g->h_cells, total, cudaHostAllocDefault));
    EB_CUDA(cudaMalloc(&g->d_cells, total));
    g->cells_bytes = total;
  }
  std::vector<const signed char*> dptr((size_t)g->B, nullptr);
  for (int i = 0; i < g->B; i++)
    if (!(update && !update[i]) && row_count[i] > 0)
    {
      std::memcpy(g->h_cells + off[i], rows[i], (size_t)row_count[i] * g->views[i].xsize);
      dptr[i] = g->d_cells + off[i];
    }
  EB_CUDA(cudaMemcpyAsync(g->d_cells, g->h_cells, total, cudaMemcpyHostToDevice, g->stream));
  st = grid_batch_set_rows(g, dptr.data(), row_begin, row_count, update, n);
  if (st != EB_OK) return st;
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

eb_status eb_grid_batch_get_map_host(const eb_grid_batch* g, int i, signed char* cells)
{
  if (!g || !cells) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch_get_map_host: NULL argument");
  if (i < 0 || i >= g->B)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch_get_map_host: instance " + std::to_string(i) + " is not in [0, " +
                                             std::to_string(g->B) + ")");
  const eb::GridView& v = g->views[(size_t)i];
  if (!v.data) return fail(EB_ERR_INVALID_ARGUMENT, "eb_grid_batch_get_map_host: instance " + std::to_string(i) + " has no map");
  EB_CUDA(cudaSetDevice(g->device));
  EB_CUDA(cudaMemcpyAsync(cells, v.data, (size_t)v.xsize * v.ysize, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

eb_status eb_collision_check_batch_dev(eb_grid_batch* g, const eb_collision* c, const double* poses_dev, int per,
                                       int* hit_dev)
{
  EB_TRACE("eb_collision_check_batch_dev");
  eb::CollisionParams p{};
  eb::MapSet m{};
  const eb_status st = grid_batch_params(g, c, per, &p, &m);
  if (st != EB_OK) return st;
  if (!poses_dev || !hit_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_collision_check_batch: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  p.x0 = poses_dev;
  p.out = hit_dev;
  eb::collision_check_kernel<true><<<(p.B + 127) / 128, 128, 0, g->stream>>>(p, m);
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}

eb_status eb_validate_control_batch_dev(eb_grid_batch* g, const eb_collision* c, const double* x0_dev,
                                        const double* u_dev, int per, double dt, double horizon, int* valid_dev)
{
  EB_TRACE("eb_validate_control_batch_dev");
  eb::CollisionParams p{};
  eb::MapSet m{};
  const eb_status st = grid_batch_params(g, c, per, &p, &m);
  if (st != EB_OK) return st;
  if (!x0_dev || !u_dev || !valid_dev || dt == 0.0)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_validate_control_batch: bad arguments");
  EB_CUDA(cudaSetDevice(g->device));
  p.x0 = x0_dev;
  p.u = u_dev;
  p.out = valid_dev;
  p.dt = dt;
  p.steps = (int)static_cast<unsigned int>(std::abs(horizon / dt));  // numerics.hpp:316
  eb::validate_control_kernel<true><<<(p.B + 127) / 128, 128, 0, g->stream>>>(p, m);
  EB_CUDA(cudaGetLastError());
  g->launches += 1;
  return EB_OK;
}

eb_status eb_collision_check_batch_host(eb_grid_batch* g, const eb_collision* c, const double* poses, int per, int* hit)
{
  eb::CollisionParams p{};
  eb::MapSet m{};
  eb_status st = grid_batch_params(g, c, per, &p, &m);
  if (st != EB_OK) return st;
  if (!poses || !hit) return fail(EB_ERR_INVALID_ARGUMENT, "eb_collision_check_batch_host: NULL argument");
  const int count = p.B;
  EB_CUDA(cudaSetDevice(g->device));
  st = grid_reserve(g, count);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(g->d_a, poses, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice, g->stream));
  st = eb_collision_check_batch_dev(g, c, g->d_a, per, g->d_out);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(hit, g->d_out, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

eb_status eb_validate_control_batch_host(eb_grid_batch* g, const eb_collision* c, const double* x0, const double* u,
                                         int per, double dt, double horizon, int* valid)
{
  eb::CollisionParams p{};
  eb::MapSet m{};
  eb_status st = grid_batch_params(g, c, per, &p, &m);
  if (st != EB_OK) return st;
  if (!x0 || !u || !valid || dt == 0.0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_validate_control_batch_host: bad arguments");
  const int count = p.B;
  EB_CUDA(cudaSetDevice(g->device));
  st = grid_reserve(g, count);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(g->d_a, x0, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice, g->stream));
  EB_CUDA(cudaMemcpyAsync(g->d_b, u, sizeof(double) * 3 * (size_t)count, cudaMemcpyHostToDevice, g->stream));
  st = eb_validate_control_batch_dev(g, c, g->d_a, g->d_b, per, dt, horizon, g->d_out);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(valid, g->d_out, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

eb_status eb_dwa_control_twist_batch_dev(eb_grid_batch* g, const eb_collision* c, const eb_dwa* d, const double* x0_dev,
                                         const double* vb_dev, const double* vref_dev, int* found_dev, double* u_opt_dev,
                                         double* min_cost_dev)
{
  EB_TRACE("eb_dwa_control_twist_batch_dev");
  eb::DwaParams p{};
  eb::MapSet m{};
  const eb_status st = grid_batch_dwa(g, c, d, &p, &m);
  if (st != EB_OK) return st;
  if (!x0_dev || !vb_dev || !vref_dev || !found_dev || !u_opt_dev)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_twist_batch: NULL argument");
  p.x0 = x0_dev;
  p.vb = vb_dev;
  p.vref = vref_dev;
  p.found = found_dev;
  p.u_opt = u_opt_dev;
  p.min_cost = min_cost_dev;
  return grid_batch_dwa_launch(g, p, m);
}

eb_status eb_dwa_control_traj_batch_dev(eb_grid_batch* g, const eb_collision* c, const eb_dwa* d, const double* x0_dev,
                                        const double* vb_dev, const double* xt_ref_dev, int ncols, int per_instance,
                                        double dt_ref, int* found_dev, double* u_opt_dev, double* min_cost_dev)
{
  EB_TRACE("eb_dwa_control_traj_batch_dev");
  eb::DwaParams p{};
  eb::MapSet m{};
  eb_status st = grid_batch_dwa(g, c, d, &p, &m);
  if (st != EB_OK) return st;
  if (ncols < 1 || !x0_dev || !vb_dev || !xt_ref_dev || !found_dev || !u_opt_dev)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_traj_batch: bad arguments");
  p.x0 = x0_dev;
  p.vb = vb_dev;
  st = dwa_traj_params(xt_ref_dev, ncols, per_instance, dt_ref, &p);
  if (st != EB_OK) return st;
  p.found = found_dev;
  p.u_opt = u_opt_dev;
  p.min_cost = min_cost_dev;
  return grid_batch_dwa_launch(g, p, m);
}

// H2D of x0 / vb / the reference, one launch, D2H of the results, synchronise
static eb_status dwa_batch_host(eb_grid_batch* g, const eb_collision* c, const eb_dwa* d, const double* x0,
                                const double* vb, const double* ref, bool traj, int ncols, int per_instance,
                                double dt_ref, int* found, double* u_opt, double* min_cost)
{
  if (!g) return fail(EB_ERR_INVALID_ARGUMENT, "grid batch is NULL");
  if (!x0 || !vb || !ref || !found || !u_opt) return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_batch_host: NULL argument");
  if (traj && ncols < 1) return fail(EB_ERR_INVALID_ARGUMENT, "eb_dwa_control_traj_batch_host: ncols < 1");
  const int B = g->B;
  const size_t ref_doubles = traj ? 3 * (size_t)ncols * (per_instance ? (size_t)B : 1) : 3 * (size_t)B;
  EB_CUDA(cudaSetDevice(g->device));
  eb_status st = grid_reserve(g, B);
  if (st != EB_OK) return st;
  if (ref_doubles > g->ref_cap)
  {
    cudaFree(g->d_ref);
    g->d_ref = nullptr;
    g->ref_cap = 0;
    EB_CUDA(cudaMalloc(&g->d_ref, sizeof(double) * ref_doubles));
    g->ref_cap = ref_doubles;
  }
  EB_CUDA(cudaMemcpyAsync(g->d_a, x0, sizeof(double) * 3 * (size_t)B, cudaMemcpyHostToDevice, g->stream));
  EB_CUDA(cudaMemcpyAsync(g->d_b, vb, sizeof(double) * 3 * (size_t)B, cudaMemcpyHostToDevice, g->stream));
  EB_CUDA(cudaMemcpyAsync(g->d_ref, ref, sizeof(double) * ref_doubles, cudaMemcpyHostToDevice, g->stream));
  st = traj ? eb_dwa_control_traj_batch_dev(g, c, d, g->d_a, g->d_b, g->d_ref, ncols, per_instance, dt_ref, g->d_out,
                                            g->d_u, g->d_cost) :
              eb_dwa_control_twist_batch_dev(g, c, d, g->d_a, g->d_b, g->d_ref, g->d_out, g->d_u, g->d_cost);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(found, g->d_out, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaMemcpyAsync(u_opt, g->d_u, sizeof(double) * 3 * (size_t)B, cudaMemcpyDeviceToHost, g->stream));
  if (min_cost) EB_CUDA(cudaMemcpyAsync(min_cost, g->d_cost, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, g->stream));
  EB_CUDA(cudaStreamSynchronize(g->stream));
  return EB_OK;
}

eb_status eb_dwa_control_twist_batch_host(eb_grid_batch* g, const eb_collision* c, const eb_dwa* d, const double* x0,
                                          const double* vb, const double* vref, int* found, double* u_opt,
                                          double* min_cost)
{
  return dwa_batch_host(g, c, d, x0, vb, vref, false, 0, 0, 0.0, found, u_opt, min_cost);
}

eb_status eb_dwa_control_traj_batch_host(eb_grid_batch* g, const eb_collision* c, const eb_dwa* d, const double* x0,
                                         const double* vb, const double* xt_ref, int ncols, int per_instance,
                                         double dt_ref, int* found, double* u_opt, double* min_cost)
{
  return dwa_batch_host(g, c, d, x0, vb, xt_ref, true, ncols, per_instance, dt_ref, found, u_opt, min_cost);
}

// ---------------------------------------------------------------------------
// row-sharded phi_k on several GPUs: all-reduce fused into the tile kernel (phik_tma.cuh)
// ---------------------------------------------------------------------------
}  // extern "C"

struct eb_phik_peer
{
  int device = 0, rank = 0, world = 1;
  double* recv[2] = {};                    // own receive buffers, [world][1024], alternating by step
  unsigned long long* flags = nullptr;     // own arrival flags, [8]
  double* peer_recv[8][2] = {};            // every rank's receive buffers as seen from here
  unsigned long long* peer_flags[8] = {};
  bool connected = false;
  unsigned long long step = 0;
};

extern "C" {

int eb_phik_peer_blob_bytes(void) { return 3 * (int)sizeof(cudaIpcMemHandle_t); }

eb_status eb_phik_peer_create(int device, int rank, int world, eb_phik_peer** out)
{
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_peer_create: out is NULL");
  *out = nullptr;
  if (world < 1 || world > 8 || rank < 0 || rank >= world)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_peer_create: need 1 <= world <= 8, 0 <= rank < world");
  EB_CUDA(cudaSetDevice(device));
  eb_phik_peer* g = new (std::nothrow) eb_phik_peer();
  if (!g) return fail(EB_ERR_CUDA, "out of host memory");
  g->device = device;
  g->rank = rank;
  g->world = world;
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < 2 && e == cudaSuccess; k++)
  {
    e = cudaMalloc(&g->recv[k], sizeof(double) * 1024 * (size_t)world);
    if (e == cudaSuccess) e = cudaMemset(g->recv[k], 0, sizeof(double) * 1024 * (size_t)world);
  }
  if (e == cudaSuccess) e = cudaMalloc(&g->flags, sizeof(unsigned long long) * 8);
  if (e == cudaSuccess) e = cudaMemset(g->flags, 0, sizeof(unsigned long long) * 8);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess)
  {
    eb_phik_peer_destroy(g);
    return fail(EB_ERR_CUDA, std::string("eb_phik_peer_create: ") + cudaGetErrorString(e));
  }
  *out = g;
  return EB_OK;
}

eb_status eb_phik_peer_export(eb_phik_peer* g, unsigned char* blob)
{
  if (!g || !blob) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_peer_export: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  cudaIpcMemHandle_t h[3];
  EB_CUDA(cudaIpcGetMemHandle(&h[0], g->recv[0]));
  EB_CUDA(cudaIpcGetMemHandle(&h[1], g->recv[1]));
  EB_CUDA(cudaIpcGetMemHandle(&h[2], g->flags));
  std::memcpy(blob, h, sizeof(h));
  return EB_OK;
}

eb_status eb_phik_peer_connect(eb_phik_peer* g, const unsigned char* blobs)
{
  if (!g || (g->world > 1 && !blobs)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_peer_connect: NULL argument");
  EB_CUDA(cudaSetDevice(g->device));
  for (int r = 0; r < g->world; r++)
  {
    if (r == g->rank)
    {
      g->peer_recv[r][0] = g->recv[0];
      g->peer_recv[r][1] = g->recv[1];
      g->peer_flags[r] = g->flags;
      continue;
    }
    cudaIpcMemHandle_t h[3];
    std::memcpy(h, blobs + (size_t)r * sizeof(h), sizeof(h));
    void* ptr[3] = {};
    for (int k = 0; k < 3; k++)
    {
      cudaError_t e = cudaIpcOpenMemHandle(&ptr[k], h[k], cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess)
        return fail(EB_ERR_CUDA, std::string("eb_phik_peer_connect: cudaIpcOpenMemHandle (peer access over NVLink is "
                                             "required): ") + cudaGetErrorString(e));
    }
    g->peer_recv[r][0] = static_cast<double*>(ptr[0]);
    g->peer_recv[r][1] = static_cast<double*>(ptr[1]);
    g->peer_flags[r] = static_cast<unsigned long long*>(ptr[2]);
  }
  g->connected = true;
  return EB_OK;
}

void eb_phik_peer_destroy(eb_phik_peer* g)
{
  if (!g) return;
  cudaSetDevice(g->device);
  cudaDeviceSynchronize();
  if (g->connected)
    for (int r = 0; r < g->world; r++)
      if (r != g->rank)
      {
        cudaIpcCloseMemHandle(g->peer_recv[r][0]);
        cudaIpcCloseMemHandle(g->peer_recv[r][1]);
        cudaIpcCloseMemHandle(g->peer_flags[r]);
      }
  cudaFree(g->recv[0]);
  cudaFree(g->recv[1]);
  cudaFree(g->flags);
  delete g;
}

// COLLECTIVE: every rank of the group calls this once per step with its own row block (a plan made by
// eb_phik_plan_create_rows).  One kernel per rank; the normalised coefficients of the WHOLE grid land in phik_dev on
// every rank, bit-identical.  Needs the TMA tile kernel (even nx >= 64, 16-byte aligned density).
eb_status eb_phik_execute_allreduce_dev(eb_phik_plan* p, eb_phik_peer* g, const double* phi_dev, double* phik_dev,
                                        double* phi_sum_dev)
{
  EB_TRACE("eb_phik_execute_allreduce_dev");
  if (!p || !g || !phi_dev || !phik_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_execute_allreduce_dev: NULL argument");
  if (!g->connected) return fail(EB_ERR_INVALID_ARGUMENT, "eb_phik_execute_allreduce_dev: peer group is not connected");
  if (p->nb > 32)
    return fail(EB_ERR_UNSUPPORTED, "eb_phik_execute_allreduce_dev: the fused all-reduce exchanges 32 x 32 blocks (num_basis <= 32); "
                                    "combine wider shards with eb_phik_execute_raw_dev + an all-reduce of the ld x ld block");
  if (!eb::phik_tma_supported(p->nx, p->ny) || !eb::phik_tma_encoder() || (reinterpret_cast<uintptr_t>(phi_dev) & 15) != 0)
    return fail(EB_ERR_UNSUPPORTED, "eb_phik_execute_allreduce_dev: needs the TMA tile kernel (even nx >= 64, aligned density)");
  const int par = (int)(g->step & 1);
  eb::PhikTmaPeer pp;
  pp.n_peer = g->world;
  for (int r = 0; r < g->world; r++)
  {
    pp.peer_recv[r] = g->peer_recv[r][par] + (size_t)g->rank * 1024;
    pp.peer_flag[r] = g->peer_flags[r] + g->rank;
  }
  pp.my_flags = g->flags;
  pp.my_recv = g->recv[par];
  pp.step = g->step + 1;
  const int saved = p->algo;
  p->algo = p->algo == 5 ? 5 : 4;
  p->peer = &pp;
  const eb_status st = phik_execute(p, phi_dev, phik_dev, phi_sum_dev, nullptr);
  p->peer = nullptr;
  p->algo = saved;
  if (st == EB_OK) g->step += 1;
  return st;
}

// ---------------------------------------------------------------------------
// map-derived target (map_target.cuh), SURVEY.md section 8f-4
// ---------------------------------------------------------------------------
}  // extern "C"

struct eb_map_target
{
  int device = 0, nb = 0;
  unsigned xsize = 0, ysize = 0;
  double resolution = 0.0;
  cudaStream_t stream = nullptr;
  eb_phik_plan* plan = nullptr;
  double* d_lut = nullptr;       // entropy of the 256 int8 patterns
  double* d_phi = nullptr;       // un-normalised density [ysize][xsize]: written by the two-kernel route or on demand
  const signed char* last_cells = nullptr;  // device cells of the last execute (must stay alive for a later density request)
  bool density_valid = false;    // d_phi holds the density of last_cells
  signed char* d_cells = nullptr;  // staging for the _host call
  double *d_phik = nullptr, *d_sum = nullptr;
  long long launches = 0;
};
extern "C" {
static eb_status map_density(eb_map_target* m);
}

extern "C" {

eb_status eb_map_target_create(int device, unsigned int xsize, unsigned int ysize, double resolution, int nb,
                               eb_map_target** out)
{
  if (!out) return fail(EB_ERR_INVALID_ARGUMENT, "eb_map_target_create: out is NULL");
  *out = nullptr;
  if (xsize < 1 || ysize < 1 || !(resolution > 0.0) || nb < 1 || nb > EB_MAX_NUM_BASIS)
    return fail(EB_ERR_INVALID_ARGUMENT,
                "eb_map_target_create: need xsize, ysize >= 1, resolution > 0, 1 <= nb <= " + std::to_string(EB_MAX_NUM_BASIS));
  if ((unsigned long long)xsize * ysize > 0x7fffffffull)
    return fail(EB_ERR_UNSUPPORTED, "eb_map_target_create: more than 2^31 - 1 cells");
  EB_CUDA(cudaSetDevice(device));
  eb_map_target* m = new (std::nothrow) eb_map_target();
  if (!m) return fail(EB_ERR_CUDA, "out of host memory");
  m->device = device;
  m->nb = nb;
  m->xsize = xsize;
  m->ysize = ysize;
  m->resolution = resolution;
  // sample points = cell centres, extent = the map's (grid.cpp:46-61: xmax = xmin + xsize * resolution)
  eb_status st = eb_phik_plan_create_ex(device, (int)xsize, (int)ysize, 0, (int)ysize, resolution, xsize * resolution,
                                        ysize * resolution, nb, 0.5 * resolution, 0.5 * resolution, &m->plan);
  if (st != EB_OK)
  {
    delete m;
    return st;
  }
  cudaError_t e = cudaMalloc(&m->d_lut, sizeof(double) * 256);
  if (e == cudaSuccess) e = cudaMalloc(&m->d_phik, sizeof(double) * (size_t)std::max(1024, nb * nb));
  if (e == cudaSuccess) e = cudaMalloc(&m->d_sum, sizeof(double));
  if (e == cudaSuccess)
  {
    eb::entropy_lut_kernel<<<1, 256>>>(m->d_lut);
    m->launches += 1;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess)
  {
    eb_map_target_destroy(m);
    return fail(EB_ERR_CUDA, std::string("eb_map_target_create: ") + cudaGetErrorString(e));
  }
  *out = m;
  return EB_OK;
}

void eb_map_target_destroy(eb_map_target* m)
{
  if (!m) return;
  cudaSetDevice(m->device);
  eb_phik_plan_destroy(m->plan);
  cudaFree(m->d_lut);
  cudaFree(m->d_phi);
  cudaFree(m->d_cells);
  cudaFree(m->d_phik);
  cudaFree(m->d_sum);
  delete m;
}

eb_status eb_map_target_set_stream(eb_map_target* m, void* s)
{
  if (!m) return fail(EB_ERR_INVALID_ARGUMENT, "map target is NULL");
  m->stream = static_cast<cudaStream_t>(s);
  m->plan->stream = m->stream;
  return EB_OK;
}

long long eb_map_target_launch_count(const eb_map_target* m) { return m ? m->launches + m->plan->launches : 0; }
double* eb_map_target_density_dev(eb_map_target* m)
{
  // the fused execute never writes the density: materialise it from the last execute's cells on demand
  if (!m || cudaSetDevice(m->device) != cudaSuccess || map_density(m) != EB_OK) return nullptr;
  return m->d_phi;
}

eb_status eb_map_target_extent(const eb_map_target* m, double* lx, double* ly)
{
  if (!m) return fail(EB_ERR_INVALID_ARGUMENT, "map target is NULL");
  if (lx) *lx = m->xsize * m->resolution;
  if (ly) *ly = m->ysize * m->resolution;
  return EB_OK;
}

// the density of the last execute's cells, materialised (allocated on first use)
static eb_status map_density(eb_map_target* m)
{
  if (m->density_valid) return EB_OK;
  if (!m->last_cells) return fail(EB_ERR_INVALID_ARGUMENT, "map target: no execute yet");
  const long long cells = (long long)m->xsize * m->ysize;
  if (!m->d_phi) EB_CUDA(cudaMalloc(&m->d_phi, sizeof(double) * (size_t)cells));
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device);
  const int grid = (int)std::min<long long>((cells / 512 + 7) / 8 + 1, (long long)sms * 8);  // 8 warps per CTA, 512 cells per warp iteration
  eb::entropy_density_kernel<<<grid, 256, 0, m->stream>>>(m->last_cells, cells, m->d_lut, m->d_phi);
  m->launches += 1;
  EB_CUDA(cudaGetLastError());
  m->density_valid = true;
  return EB_OK;
}

eb_status eb_map_target_execute_dev(eb_map_target* m, const signed char* cells_dev, double* phik_dev, double* phi_sum_dev)
{
  EB_TRACE("eb_map_target_execute_dev");
  if (!m || !cells_dev || !phik_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_map_target_execute_dev: NULL argument");
  EB_CUDA(cudaSetDevice(m->device));
  m->last_cells = cells_dev;
  m->density_valid = false;
  // ONE kernel when the folded TMA tile kernel applies: the bytes are staged by TMA and the entropy table is looked up in
  // shared memory -- the 8 B / cell density is never written.  Every other input takes the two-kernel route: the
  // density, then the plan's phi_k.
  eb_phik_plan* const pl = m->plan;
  const bool big = (long long)pl->nx * pl->ny >= (1 << 18);  // as phik_execute: small grids take the simple kernels
  if (pl->fold && pl->d_cxtf && (pl->algo == 4 || (pl->algo == 0 && big)) && !pl->peer &&
      eb::phik_tma_u8_supported(pl->nx, pl->ny) && eb::phik_tma_encoder() && (reinterpret_cast<uintptr_t>(cells_dev) & 15) == 0)
  {
    const eb::PhikTmaOut out{ pl->d_done, pl->nb, phik_dev, phi_sum_dev, nullptr, nullptr };
    const int nparts = eb::phik_tma_launch_u8(cells_dev, m->d_lut, pl->nx, pl->ny, pl->d_cxtf, pl->d_cy, pl->d_parts,
                                              pl->max_parts, out, m->stream);
    if (nparts < 0) return fail(EB_ERR_CUDA, std::string("phik_tma_launch_u8: ") + cudaGetErrorString(cudaGetLastError()));
    m->launches += 1;
    return EB_OK;
  }
  const eb_status st = map_density(m);
  if (st != EB_OK) return st;
  return eb_phik_execute_dev(m->plan, m->d_phi, phik_dev, phi_sum_dev);
}

eb_status eb_map_target_execute_host(eb_map_target* m, const signed char* cells, double* phik, double* phi_sum)
{
  EB_TRACE("eb_map_target_execute_host");
  if (!m || !cells || !phik) return fail(EB_ERR_INVALID_ARGUMENT, "eb_map_target_execute_host: NULL argument");
  EB_CUDA(cudaSetDevice(m->device));
  const size_t n = (size_t)m->xsize * m->ysize;
  if (!m->d_cells) EB_CUDA(cudaMalloc(&m->d_cells, n));
  EB_CUDA(cudaMemcpyAsync(m->d_cells, cells, n, cudaMemcpyHostToDevice, m->stream));
  eb_status st = eb_map_target_execute_dev(m, m->d_cells, m->d_phik, m->d_sum);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(phik, m->d_phik, sizeof(double) * m->nb * m->nb, cudaMemcpyDeviceToHost, m->stream));
  if (phi_sum) EB_CUDA(cudaMemcpyAsync(phi_sum, m->d_sum, sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  EB_CUDA(cudaStreamSynchronize(m->stream));
  return EB_OK;
}

// phi_k from a device buffer (e.g. the output of eb_map_target_execute_dev / eb_phik_execute_dev), no host round trip
eb_status eb_set_phik_dev(eb_controller* c, const double* phik_dev, double lx, double ly)
{
  if (!c || !phik_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_phik_dev: NULL argument");
  if (c->per_inst) return refuse_per_inst("eb_set_phik_dev");
  if (!(lx > 0.0) || !(ly > 0.0)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_phik_dev: lx, ly must be positive");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  EB_CUDA(cudaMemcpyAsync(c->d_phik, phik_dev, sizeof(double) * c->K, cudaMemcpyDeviceToDevice, c->stream));
  c->lx = lx;
  c->ly = ly;
  return EB_OK;
}

// ---------------------------------------------------------------------------
// per-instance targets: one target, phi_k row and Fourier frame per instance (target_batch.cuh)
// ---------------------------------------------------------------------------
eb_status eb_set_target_gaussians_batch(eb_controller* c, int max_n, const int* counts, const double* mu,
                                        const double* sigma)
{
  EB_TRACE("eb_set_target_gaussians_batch");
  if (!c || !counts || max_n < 0 || max_n > eb::kTbMaxGauss || (max_n > 0 && (!mu || !sigma)))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_target_gaussians_batch: bad argument (NULL, or max_n outside 0.." +
                                             std::to_string(eb::kTbMaxGauss) + ")");
  for (int i = 0; i < c->B; i++)
    if (counts[i] < 0 || counts[i] > max_n)
      return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_target_gaussians_batch: counts[" + std::to_string(i) +
                                               "] outside 0..max_n");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  if (max_n > c->gmax)
  {
    cudaFree(c->d_gmu);
    cudaFree(c->d_gsig);
    c->d_gmu = c->d_gsig = nullptr;
    c->gmax = 0;
    const size_t gb = sizeof(double) * 2 * (size_t)max_n * c->B;
    EB_CUDA(cudaMalloc(&c->d_gmu, gb));
    EB_CUDA(cudaMalloc(&c->d_gsig, gb));
  }
  c->gmax = std::max(c->gmax, max_n);
  // the caller's [B][max_n][2] rows into the [B][gmax][2] buffers
  const size_t row = sizeof(double) * 2 * (size_t)max_n, pitch = sizeof(double) * 2 * (size_t)c->gmax;
  if (max_n > 0)
  {
    EB_CUDA(cudaMemcpy2DAsync(c->d_gmu, pitch, mu, row, row, c->B, cudaMemcpyHostToDevice, c->stream));
    EB_CUDA(cudaMemcpy2DAsync(c->d_gsig, pitch, sigma, row, row, c->B, cudaMemcpyHostToDevice, c->stream));
  }
  EB_CUDA(cudaMemcpyAsync(c->d_gcount, counts, sizeof(int) * (size_t)c->B, cudaMemcpyHostToDevice, c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));  // the caller's buffers may go once this returns
  return EB_OK;
}

eb_status eb_config_target_batch_dev(eb_controller* c, const double* bounds_dev, int* rebuilt_dev)
{
  EB_TRACE("eb_config_target_batch_dev");
  if (!c || !bounds_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_config_target_batch_dev: NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  return target_batch(c, bounds_dev, nullptr, rebuilt_dev);
}

eb_status eb_set_phik_batch_dev(eb_controller* c, const double* phik_dev, const double* extent_dev)
{
  EB_TRACE("eb_set_phik_batch_dev");
  if (!c || !phik_dev || !extent_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_phik_batch_dev: NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(c->d_phik_b, phik_dev, sizeof(double) * (size_t)c->K * c->B, cudaMemcpyDeviceToDevice,
                          c->stream));
  return target_batch(c, nullptr, extent_dev, nullptr);
}

}  // extern "C"

namespace
{
// the geometry of every flagged map; *n = flagged maps, *units = their work units
eb_status map_targets_check(const eb_controller* c, const signed char* const* cells, const unsigned* xsize,
                            const unsigned* ysize, const double* resolution, const int* update, const char* call, int* n,
                            long long* units)
{
  *n = 0;
  *units = 0;
  for (int i = 0; i < c->B; i++)
  {
    if (update && !update[i]) continue;
    if (xsize[i] < 1 || ysize[i] < 1 || !(resolution[i] > 0.0) || !std::isfinite(resolution[i]))
      return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": map " + std::to_string(i) +
                                               " needs xsize, ysize >= 1 and a finite resolution > 0");
    if ((unsigned long long)xsize[i] * ysize[i] > 0x7fffffffull)
      return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": map " + std::to_string(i) + " has more than 2^31 - 1 cells");
    if (!cells[i]) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": cells of map " + std::to_string(i) + " is NULL");
    (*n)++;
    *units += eb::mb_units((int)ysize[i]);
  }
  return EB_OK;
}

// the descriptors, arrival counters and resident grid of map_target_batch_kernel, allocated at the first call
eb_status ensure_map_batch(eb_controller* c)
{
  if (c->h_mb_desc) return EB_OK;
  const int B = c->B;
  EB_CUDA(cudaHostAlloc(&c->h_mb_desc, sizeof(eb::MapBatchDesc) * (size_t)B, cudaHostAllocDefault));
  EB_CUDA(cudaMalloc(&c->d_mb_desc, sizeof(eb::MapBatchDesc) * (size_t)B));
  EB_CUDA(cudaMalloc(&c->d_mb_arrive, sizeof(unsigned) * (size_t)B));
  EB_CUDA(cudaMemset(c->d_mb_arrive, 0, sizeof(unsigned) * (size_t)B));
  EB_CUDA(cudaEventCreateWithFlags(&c->mb_staged, cudaEventDisableTiming));
  for (auto kernel : { eb::map_target_batch_kernel<false>, eb::map_target_batch_kernel<true> })
    EB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eb::kMbSmemBytes));
  int per_sm = 0, sms = 0;
  EB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eb::map_target_batch_kernel<false>, eb::kMbThreads,
                                                        eb::kMbSmemBytes));
  EB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->cfg.device));
  c->mb_grid = std::max(1, per_sm * sms);
  return EB_OK;
}

// map-derived targets of the flagged instances (map_target_batch.cuh); cells holds device pointers
eb_status map_targets_batch(eb_controller* c, const signed char* const* cells, const unsigned* xsize,
                            const unsigned* ysize, const double* resolution, const double* origin, const int* update,
                            const char* call)
{
  const int B = c->B;
  int n = 0;
  long long units = 0;
  eb_status st = map_targets_check(c, cells, xsize, ysize, resolution, update, call, &n, &units);
  if (st != EB_OK) return st;
  EB_CUDA(cudaSetDevice(c->cfg.device));
  st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  if (n == B) c->frames_set = true;
  if (n == 0) return EB_OK;
  if ((st = ensure_map_batch(c)) != EB_OK) return st;
  if (units > c->mb_slot_units)
  {
    cudaFree(c->d_mb_slots);  // synchronises with earlier launches that use it
    c->d_mb_slots = nullptr;
    c->mb_slot_units = 0;
    EB_CUDA(cudaMalloc(&c->d_mb_slots, sizeof(double) * (size_t)c->K * (size_t)units));
    c->mb_slot_units = units;
  }
  EB_CUDA(cudaEventSynchronize(c->mb_staged));  // the previous call's copy out of the pinned descriptors is done
  int k = 0, u0 = 0;
  for (int i = 0; i < B; i++)
  {
    if (update && !update[i]) continue;
    eb::MapBatchDesc& d = c->h_mb_desc[k++];
    d.cells = cells[i];
    d.nx = (int)xsize[i];
    d.ny = (int)ysize[i];
    d.res = resolution[i];
    d.ox = origin[2 * i + 0];
    d.oy = origin[2 * i + 1];
    d.inst = i;
    d.unit0 = u0;
    u0 += eb::mb_units(d.ny);
  }
  EB_CUDA(cudaMemcpyAsync(c->d_mb_desc, c->h_mb_desc, sizeof(eb::MapBatchDesc) * (size_t)n, cudaMemcpyHostToDevice,
                          c->stream));
  EB_CUDA(cudaEventRecord(c->mb_staged, c->stream));
  eb::MapBatchParams p{};
  p.desc = c->d_mb_desc;
  p.n = n;
  p.units = (int)units;
  p.nb = c->nb;
  p.slots = c->d_mb_slots;
  p.arrive = c->d_mb_arrive;
  p.frames = c->d_frames;
  p.phik = c->d_phik_b;
  p.hist = c->d_hist;
  p.hist_cos = c->d_hist_cos;
  p.mem_count = c->d_hist_cos ? c->mem_count : 0;
  p.B = B;
  const int grid = (int)std::min<long long>(units, c->mb_grid);
  eb::map_target_batch_kernel<false><<<grid, eb::kMbThreads, eb::kMbSmemBytes, c->stream>>>(p);
  EB_CUDA(cudaGetLastError());
  c->launches += 1;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_set_map_targets_batch_dev(eb_controller* c, const signed char* const* cells_dev, const unsigned* xsize,
                                       const unsigned* ysize, const double* resolution, const double* origin,
                                       const int* update)
{
  EB_TRACE("eb_set_map_targets_batch_dev");
  if (!c || !cells_dev || !xsize || !ysize || !resolution || !origin)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_map_targets_batch_dev: NULL argument");
  return map_targets_batch(c, cells_dev, xsize, ysize, resolution, origin, update, "eb_set_map_targets_batch_dev");
}

eb_status eb_set_map_targets_batch_host(eb_controller* c, const signed char* const* cells, const unsigned* xsize,
                                        const unsigned* ysize, const double* resolution, const double* origin,
                                        const int* update)
{
  EB_TRACE("eb_set_map_targets_batch_host");
  static const char* call = "eb_set_map_targets_batch_host";
  if (!c || !cells || !xsize || !ysize || !resolution || !origin) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  int n = 0;
  long long units = 0;
  eb_status st = map_targets_check(c, cells, xsize, ysize, resolution, update, call, &n, &units);
  if (st != EB_OK) return st;
  // the flagged maps are packed into one pinned buffer (16-byte aligned offsets) and copied with one cudaMemcpyAsync
  std::vector<size_t> off((size_t)c->B, 0);
  size_t total = 0;
  for (int i = 0; i < c->B; i++)
  {
    if (update && !update[i]) continue;
    off[i] = total;
    total += ((size_t)xsize[i] * ysize[i] + 15) & ~(size_t)15;
  }
  EB_CUDA(cudaSetDevice(c->cfg.device));
  EB_CUDA(cudaStreamSynchronize(c->stream));  // no earlier copy still reads the staging buffers
  if (total > c->mb_cells_bytes)
  {
    cudaFreeHost(c->h_mb_cells);
    cudaFree(c->d_mb_cells);
    c->h_mb_cells = nullptr;
    c->d_mb_cells = nullptr;
    c->mb_cells_bytes = 0;
    EB_CUDA(cudaHostAlloc(&c->h_mb_cells, total, cudaHostAllocDefault));
    EB_CUDA(cudaMalloc(&c->d_mb_cells, total));
    c->mb_cells_bytes = total;
  }
  std::vector<const signed char*> dptr((size_t)c->B, nullptr);
  for (int i = 0; i < c->B; i++)
    if (!(update && !update[i]))
    {
      std::memcpy(c->h_mb_cells + off[i], cells[i], (size_t)xsize[i] * ysize[i]);
      dptr[i] = c->d_mb_cells + off[i];
    }
  if (total > 0)
    EB_CUDA(cudaMemcpyAsync(c->d_mb_cells, c->h_mb_cells, total, cudaMemcpyHostToDevice, c->stream));
  st = map_targets_batch(c, dptr.data(), xsize, ysize, resolution, origin, update, call);
  if (st != EB_OK) return st;
  EB_CUDA(cudaStreamSynchronize(c->stream));
  return EB_OK;
}

}  // extern "C"

namespace
{
// moves the kept blocks to a new region in which instance i has cap[i] slots; the blocks of the instances whose slot
// keeps its size move with them (one copy per run of such instances), the others are recomputed whole by the caller
eb_status kept_relayout(eb_controller* c, const std::vector<int>& cap)
{
  const int B = c->B;
  const size_t K = (size_t)c->K;
  std::vector<int> slot0((size_t)B, 0);
  long long total = 0;
  for (int i = 0; i < B; i++)
  {
    slot0[i] = (int)total;
    total += cap[i];
  }
  if (total > 0x7fffffffLL) return fail(EB_ERR_INVALID_ARGUMENT, "eb_set_map_targets_from_grid_batch: more than 2^31 - 1 units");
  double* kb = nullptr;
  EB_CUDA(cudaMalloc(&kb, sizeof(double) * K * (size_t)total));
  cudaError_t e = cudaSuccess;
  bool copied = false;
  for (int i = 0; i < B && e == cudaSuccess;)
  {
    if (cap[i] != c->kb_cap[i] || c->kb_cap[i] == 0)
    {
      i++;
      continue;
    }
    int j = i, units = 0;
    for (; j < B && cap[j] == c->kb_cap[j]; j++) units += cap[j];
    e = cudaMemcpyAsync(kb + K * slot0[i], c->d_kb + K * c->kb_slot0[i], sizeof(double) * K * units,
                        cudaMemcpyDeviceToDevice, c->stream);
    copied = true;
    i = j;
  }
  if (e == cudaSuccess && copied) e = cudaStreamSynchronize(c->stream);  // the old region is read no more
  if (e != cudaSuccess)
  {
    cudaFree(kb);
    return fail(EB_ERR_CUDA, std::string("eb_set_map_targets_from_grid_batch: ") + cudaGetErrorString(e));
  }
  cudaFree(c->d_kb);
  c->d_kb = kb;
  for (int i = 0; i < B; i++)
    if (cap[i] != c->kb_cap[i]) c->kb_key[i] = eb_controller::KeptKey{};
  c->kb_cap = cap;
  c->kb_slot0 = slot0;
  return EB_OK;
}
}  // namespace

extern "C" {

eb_status eb_set_map_targets_from_grid_batch(eb_controller* c, eb_grid_batch* g, const unsigned* row_begin,
                                             const unsigned* row_count, const int* update)
{
  EB_TRACE("eb_set_map_targets_from_grid_batch");
  static const char* call = "eb_set_map_targets_from_grid_batch";
  if (!c || !g) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  if (!row_begin != !row_count)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": row_begin and row_count must both be given or both NULL");
  if (g->B != c->B)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the grid batch holds " + std::to_string(g->B) +
                                             " maps for " + std::to_string(c->B) + " instances");
  if (g->device != c->cfg.device)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the grid batch and the controller are on different devices");
  const int B = c->B;
  if (c->kb_key.empty())
  {
    c->kb_key.assign((size_t)B, eb_controller::KeptKey{});
    c->kb_cap.assign((size_t)B, 0);
    c->kb_slot0.assign((size_t)B, 0);
  }
  // the run of units each flagged instance recomputes: the units that meet its declared rows, or all of them
  std::vector<eb::MapKept> run((size_t)B, eb::MapKept{ 0, 0, 0 });
  std::vector<int> cap = c->kb_cap;
  int n = 0;
  long long work = 0;
  bool grown = false;
  for (int i = 0; i < B; i++)
  {
    if (update && !update[i]) continue;
    const eb::GridView& v = g->views[i];
    if (!v.data) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": instance " + std::to_string(i) + " has no map");
    if (row_begin && (unsigned long long)row_begin[i] + row_count[i] > v.ysize)
      return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": rows [" + std::to_string(row_begin[i]) + ", +" +
                                               std::to_string(row_count[i]) + ") of map " + std::to_string(i) +
                                               " pass its " + std::to_string(v.ysize) + " rows");
    n++;
    const int units = eb::mb_units((int)v.ysize);
    const eb_controller::KeptKey& k = c->kb_key[i];
    const bool whole = !row_begin || k.grid != g->serial || k.map != g->map_serial[i] || k.nx != v.xsize ||
                       k.ny != v.ysize || k.res != v.resolution || units > c->kb_cap[i];
    if (whole)
      run[i] = eb::MapKept{ 0, units, 0 };
    else if (row_count[i] > 0)
    {
      const int first = (int)(row_begin[i] / eb::kMbRows), last = (int)((row_begin[i] + row_count[i] - 1) / eb::kMbRows);
      run[i] = eb::MapKept{ first, last - first + 1, 0 };
    }
    work += run[i].count;
    if (units > cap[i])
    {
      cap[i] = units + units / 4;  // a quarter of headroom, as the grid batch's arena
      grown = true;
    }
  }
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  if (n == B) c->frames_set = true;
  if (work == 0) return EB_OK;
  if (work > 0x7fffffffLL) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": more than 2^31 - 1 units");
  if ((st = ensure_map_batch(c)) != EB_OK) return st;
  if (!c->h_mb_kept)
  {
    EB_CUDA(cudaHostAlloc(&c->h_mb_kept, sizeof(eb::MapKept) * (size_t)B, cudaHostAllocDefault));
    EB_CUDA(cudaMalloc(&c->d_mb_kept, sizeof(eb::MapKept) * (size_t)B));
  }
  if (grown && (st = kept_relayout(c, cap)) != EB_OK) return st;
  if (!g->maps_ready)
  {
    EB_CUDA(cudaEventCreateWithFlags(&g->maps_ready, cudaEventDisableTiming));
    EB_CUDA(cudaEventCreateWithFlags(&g->ticked, cudaEventDisableTiming));
  }
  EB_CUDA(cudaEventSynchronize(c->mb_staged));  // the previous call's copy out of the pinned descriptors is done
  int k = 0, u0 = 0;
  for (int i = 0; i < B; i++)
  {
    if (run[i].count == 0) continue;
    const eb::GridView& v = g->views[i];
    c->h_mb_desc[k] = eb::MapBatchDesc{ v.data, (int)v.xsize, (int)v.ysize, v.resolution, v.xmin, v.ymin, i, u0 };
    c->h_mb_kept[k++] = eb::MapKept{ run[i].first, run[i].count, c->kb_slot0[i] };
    u0 += run[i].count;
  }
  EB_CUDA(cudaMemcpyAsync(c->d_mb_desc, c->h_mb_desc, sizeof(eb::MapBatchDesc) * (size_t)k, cudaMemcpyHostToDevice,
                          c->stream));
  EB_CUDA(cudaMemcpyAsync(c->d_mb_kept, c->h_mb_kept, sizeof(eb::MapKept) * (size_t)k, cudaMemcpyHostToDevice,
                          c->stream));
  EB_CUDA(cudaEventRecord(c->mb_staged, c->stream));  // before the wait below: the next call's sync does not wait for it
  // after the set and rows calls already enqueued on the grid batch's stream, without a host synchronisation
  EB_CUDA(cudaEventRecord(g->maps_ready, g->stream));
  EB_CUDA(cudaStreamWaitEvent(c->stream, g->maps_ready, 0));
  eb::MapBatchParams p{};
  p.desc = c->d_mb_desc;
  p.n = k;
  p.units = (int)work;
  p.nb = c->nb;
  p.slots = c->d_kb;
  p.arrive = c->d_mb_arrive;
  p.frames = c->d_frames;
  p.phik = c->d_phik_b;
  p.hist = c->d_hist;
  p.hist_cos = c->d_hist_cos;
  p.mem_count = c->d_hist_cos ? c->mem_count : 0;
  p.B = B;
  p.kept = c->d_mb_kept;
  const int grid = (int)std::min<long long>(work, c->mb_grid);
  eb::map_target_batch_kernel<true><<<grid, eb::kMbThreads, eb::kMbSmemBytes, c->stream>>>(p);
  cudaError_t e = cudaGetLastError();
  const cudaError_t r = cudaEventRecord(g->ticked, c->stream);  // the grid batch's next set or rows call waits for this
  if (e == cudaSuccess) e = r;
  if (e != cudaSuccess)
  {
    for (int i = 0; i < B; i++)
      if (run[i].count > 0) c->kb_key[i] = eb_controller::KeptKey{};
    return fail(EB_ERR_CUDA, std::string(call) + ": " + cudaGetErrorString(e));
  }
  c->launches += 1;
  for (int i = 0; i < B; i++)
    if (run[i].count > 0)
      c->kb_key[i] = eb_controller::KeptKey{ g->serial, g->map_serial[i], g->views[i].xsize, g->views[i].ysize,
                                             g->views[i].resolution };
  return EB_OK;
}

eb_status eb_get_phik_batch(const eb_controller* c, double* phik, double* extent)
{
  if (!c) return fail(EB_ERR_INVALID_ARGUMENT, "controller is NULL");
  if (!c->per_inst) return fail(EB_ERR_INVALID_ARGUMENT, "eb_get_phik_batch: the controller holds a shared target (eb_get_phik)");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  if (phik)
    EB_CUDA(cudaMemcpyAsync(phik, c->d_phik_b, sizeof(double) * (size_t)c->K * c->B, cudaMemcpyDeviceToHost, c->stream));
  if (extent)
    EB_CUDA(cudaMemcpy2DAsync(extent, sizeof(double) * 2, c->d_frames + eb::kFrLx, sizeof(double) * eb::kFrDoubles,
                              sizeof(double) * 2, c->B, cudaMemcpyDeviceToHost, c->stream));
  EB_CUDA(cudaStreamSynchronize(c->stream));
  return EB_OK;
}

eb_status eb_control_batch_dev(eb_controller* c, const double* bounds_dev, const double* x_dev, const int* mem_idx_dev,
                               double* u0_dev, double* metric_dev)
{
  EB_TRACE("eb_control_batch_dev");
  if (!c || !x_dev || !u0_dev) return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_batch_dev: NULL argument");
  if (!bounds_dev && !c->frames_set)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_batch_dev: bounds NULL before any frame was configured");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  if (bounds_dev && (st = target_batch(c, bounds_dev, nullptr, nullptr)) != EB_OK) return st;  // :230
  return solve_step(c, x_dev, mem_idx_dev, u0_dev, metric_dev);
}

eb_status eb_control_batch_host(eb_controller* c, const double* bounds, const double* x, const int* mem_idx, double* u0,
                                double* metric)
{
  EB_TRACE("eb_control_batch_host");
  if (!c || !x || !u0) return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_batch_host: NULL argument");
  if (!bounds && !c->frames_set)
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_control_batch_host: bounds NULL before any frame was configured");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_per_inst(c);
  if (st != EB_OK) return st;
  if (bounds)
    EB_CUDA(cudaMemcpyAsync(c->d_bounds, bounds, sizeof(double) * 4 * (size_t)c->B, cudaMemcpyHostToDevice, c->stream));
  const double* bd = bounds ? c->d_bounds : nullptr;
  const bool need_idx = mem_idx && c->mem_count > (long long)c->cfg.batch_size;
  if (need_idx)
    EB_CUDA(cudaMemcpyAsync(c->d_mem_idx_in, mem_idx, sizeof(int) * (size_t)c->cfg.batch_size * c->B,
                            cudaMemcpyHostToDevice, c->stream));
  // as eb_control_host: page-locked caller buffers of a small batch are read / written in place
  double *xm = nullptr, *um = nullptr, *mm = nullptr;
  if (c->B <= zero_copy_max_batch())
  {
    xm = c->mapped(x);
    um = xm ? c->mapped(u0) : nullptr;
    mm = (um && metric) ? c->mapped(metric) : nullptr;
  }
  if (xm && um && (!metric || mm))
  {
    st = eb_control_batch_dev(c, bd, xm, need_idx ? c->d_mem_idx_in : nullptr, um, mm);
    if (st != EB_OK) return st;
    return check_fault(c);  // synchronises
  }
  EB_CUDA(cudaMemcpyAsync(c->d_pose, x, sizeof(double) * 3 * c->B, cudaMemcpyHostToDevice, c->stream));
  st = eb_control_batch_dev(c, bd, c->d_pose, need_idx ? c->d_mem_idx_in : nullptr, c->d_u0, metric ? c->d_metric : nullptr);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(u0, c->d_u0, sizeof(double) * 3 * c->B, cudaMemcpyDeviceToHost, c->stream));
  if (metric) EB_CUDA(cudaMemcpyAsync(metric, c->d_metric, sizeof(double) * c->B, cudaMemcpyDeviceToHost, c->stream));
  return check_fault(c);  // synchronises
}

}  // extern "C"

// ---------------------------------------------------------------------------
// safe control tick of B robots on B maps (safe_control.cuh)
// ---------------------------------------------------------------------------
namespace
{
// everything the tick refuses before it launches (or copies) anything, so an error leaves the controller as it was;
// fills the fallback's window and collision parameters
eb_status safe_batch_check(const eb_controller* c, eb_grid_batch* g, const eb_collision* col, const eb_dwa* d,
                           double val_dt, const double* bounds, const char* call, eb::DwaParams* p, eb::MapSet* m)
{
  if (!c || !g || !col || !d) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  if (!c->per_inst)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the controller holds a shared target; the safe tick "
                                                             "needs per-instance targets (the eb_*_batch calls)");
  if (!bounds && !c->frames_set)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": bounds NULL before any frame was configured");
  if (g->B != c->B)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the grid batch holds " + std::to_string(g->B) +
                                             " maps for " + std::to_string(c->B) + " instances");
  if (g->device != c->cfg.device)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the grid batch and the controller are on different devices");
  eb_status st = grid_batch_dwa(g, col, d, p, m);  // Collision constructor rules, every instance has a map, DWA dt
  if (st != EB_OK) return st;
  if (val_dt == 0.0) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": val_dt is 0");
  // the reference trajectory is each robot's optTraj(): N columns at the controller's time step
  return dwa_traj_params(nullptr, c->N, 1, c->cfg.dt, p);
}

// the failing-robot list and the _host staging, allocated at the first tick; the fallback's resident grid
eb_status ensure_safe(eb_controller* c)
{
  if (c->d_safe_list) return EB_OK;
  const size_t B = (size_t)c->B;
  EB_CUDA(cudaMalloc(&c->d_safe_branch, sizeof(int) * B));
  EB_CUDA(cudaMalloc(&c->d_safe_vb, sizeof(double) * 3 * B));
  const bool omni = c->cfg.model == EB_MODEL_OMNI;
  auto kernel = omni ? eb::dwa_fallback_kernel<eb::kModelOmni, false> : eb::dwa_fallback_kernel<eb::kModelSimpleCart, false>;
  auto publishing = omni ? eb::dwa_fallback_kernel<eb::kModelOmni, true> : eb::dwa_fallback_kernel<eb::kModelSimpleCart, true>;
  const size_t smem = sizeof(double) * 3 * (size_t)c->N;
  EB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * 3 * 4096)));
  EB_CUDA(cudaFuncSetAttribute(publishing, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * 3 * 4096)));
  int per_sm = 0, sms = 0;
  EB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, eb::kSafeThreads, smem));
  EB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->cfg.device));
  c->safe_grid = std::max(1, per_sm * sms);
  EB_CUDA(cudaMalloc(&c->d_safe_list, sizeof(int) * (1 + B)));  // last: it marks the scratch as complete
  return EB_OK;
}
}  // namespace

extern "C" {

}  // extern "C"

namespace
{
// The tick's launches after its checks: the solve writes u0 into u, validate_compact_kernel lists the failing robots
// and dwa_fallback_kernel overwrites their rows.  With pub (a peer group's step), both kernels also store the rows they
// decide into every rank's gathered buffer and the fallback raises the arrival flags (safe_control.cuh).
eb_status safe_tick(eb_controller* c, eb_grid_batch* g, eb::DwaParams& p, const eb::MapSet& m, double val_dt,
                    double val_horizon, const double* bounds_dev, const double* x_dev, const int* mem_idx_dev,
                    const double* vb_dev, double* u_dev, int* branch_dev, double* metric_dev,
                    const eb::SafePublishParams* pub, const char* call)
{
  EB_CUDA(cudaSetDevice(c->cfg.device));
  eb_status st = ensure_safe(c);
  if (st != EB_OK) return st;
  if (!g->maps_ready)
  {
    EB_CUDA(cudaEventCreateWithFlags(&g->maps_ready, cudaEventDisableTiming));
    EB_CUDA(cudaEventCreateWithFlags(&g->ticked, cudaEventDisableTiming));
  }
  // after the set calls already enqueued on the grid batch's stream, without a host synchronisation
  EB_CUDA(cudaEventRecord(g->maps_ready, g->stream));
  EB_CUDA(cudaStreamWaitEvent(c->stream, g->maps_ready, 0));
  EB_CUDA(cudaMemsetAsync(c->d_safe_list, 0, sizeof(int), c->stream));
  // 1. the solve writes u0 straight into u: the validate kernel reads it there and the fallback overwrites the rows
  //    of the robots whose twist collides
  if ((st = eb_control_batch_dev(c, bounds_dev, x_dev, mem_idx_dev, u_dev, metric_dev)) != EB_OK) return st;
  eb::SafePublishParams s{};
  if (pub) s = *pub;
  s.count = c->d_safe_list;
  s.list = c->d_safe_list + 1;
  s.ut = c->d_ut[c->cur];
  s.dt = c->cfg.dt;
  s.N = c->N;
  s.u = u_dev;
  s.branch = branch_dev;
  s.fault = c->d_fault;
  // 2. validate_control of every robot's twist on its map, failing robots listed
  eb::CollisionParams v = p.col;
  v.B = c->B;
  v.x0 = x_dev;
  v.u = u_dev;
  v.dt = val_dt;
  v.steps = (int)static_cast<unsigned int>(std::abs(val_horizon / val_dt));  // numerics.hpp:316
  const int vblocks = (c->B + 127) / 128, fblocks = std::min(c->B, c->safe_grid);
  if (pub)
  {
    s.arrivals = (unsigned int)(vblocks * (128 / 32) + fblocks);
    eb::validate_compact_kernel<true><<<vblocks, 128, 0, c->stream>>>(v, m, s);
  }
  else
    eb::validate_compact_kernel<false><<<vblocks, 128, 0, c->stream>>>(v, m, s);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess)
  {
    // 3. the dynamic window of the listed robots against their optTraj()
    c->launches += 1;
    p.x0 = x_dev;
    p.vb = vb_dev;
    const size_t smem = sizeof(double) * 3 * (size_t)c->N;
    const bool omni = c->cfg.model == EB_MODEL_OMNI;
    if (pub)
      (omni ? eb::dwa_fallback_kernel<eb::kModelOmni, true> : eb::dwa_fallback_kernel<eb::kModelSimpleCart, true>)
          <<<fblocks, eb::kSafeThreads, smem, c->stream>>>(p, m, s);
    else
      (omni ? eb::dwa_fallback_kernel<eb::kModelOmni, false> : eb::dwa_fallback_kernel<eb::kModelSimpleCart, false>)
          <<<fblocks, eb::kSafeThreads, smem, c->stream>>>(p, m, s);
    e = cudaGetLastError();
    if (e == cudaSuccess) c->launches += 1;
  }
  const cudaError_t r = cudaEventRecord(g->ticked, c->stream);  // the grid batch's next set call waits for this tick
  if (e == cudaSuccess) e = r;
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string(call) + ": " + cudaGetErrorString(e));
  return EB_OK;
}

// eb_control_safe_batch_dev_gather[_wait]: the tick whose final twists land in every rank's gathered buffer
eb_status safe_gather(eb_controller* c, eb_peer_group* pg, eb_grid_batch* g, const eb_collision* col, const eb_dwa* dwa,
                      double val_dt, double val_horizon, const double* bounds_dev, const double* x_dev,
                      const int* mem_idx_dev, const double* vb_dev, int* branch_dev, double* metric_dev, bool wait,
                      const char* call)
{
  eb::DwaParams p{};
  eb::MapSet m{};
  eb_status st = safe_batch_check(c, g, col, dwa, val_dt, bounds_dev, call, &p, &m);
  if (st != EB_OK) return st;
  if (!pg || !x_dev || !vb_dev || !branch_dev) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  if (pg->device != c->cfg.device)
    return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": the peer group and the controller are on different devices");
  if ((st = peer_group_check(c, pg, call)) != EB_OK) return st;
  EB_CUDA(cudaSetDevice(c->cfg.device));
  if (pg->side_used)
  {
    // side-stream publications of earlier steps (eb_control_*_gather on a single-wave batch): the one into this
    // step's buffer must have left it, and the last one must have raised its flags before this step raises higher ones
    const unsigned long long n = pg->step;
    if (n >= (unsigned long long)eb::kPeerBuffers) EB_CUDA(cudaStreamWaitEvent(c->stream, pg->published[n % eb::kPeerBuffers], 0));
    if (n >= 1) EB_CUDA(cudaStreamWaitEvent(c->stream, pg->published[(n - 1) % eb::kPeerBuffers], 0));
  }
  eb::SafePublishParams pub{};
  pub.peer = publish_params(pg, nullptr, pg->counter);
  pub.wait = wait ? 1 : 0;
  // the solve writes its twists into the controller's scratch, not to the peers: they are final only after the window
  st = safe_tick(c, g, p, m, val_dt, val_horizon, bounds_dev, x_dev, mem_idx_dev, vb_dev, c->d_u0, branch_dev,
                 metric_dev, &pub, call);
  if (st == EB_OK) pg->step += 1;
  return st;
}
}  // namespace

extern "C" {

eb_status eb_control_safe_batch_dev(eb_controller* c, eb_grid_batch* g, const eb_collision* col, const eb_dwa* dwa,
                                    double val_dt, double val_horizon, const double* bounds_dev, const double* x_dev,
                                    const int* mem_idx_dev, const double* vb_dev, double* u_dev, int* branch_dev,
                                    double* metric_dev)
{
  EB_TRACE("eb_control_safe_batch_dev");
  static const char* call = "eb_control_safe_batch_dev";
  eb::DwaParams p{};
  eb::MapSet m{};
  eb_status st = safe_batch_check(c, g, col, dwa, val_dt, bounds_dev, call, &p, &m);
  if (st != EB_OK) return st;
  if (!x_dev || !vb_dev || !u_dev || !branch_dev) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  return safe_tick(c, g, p, m, val_dt, val_horizon, bounds_dev, x_dev, mem_idx_dev, vb_dev, u_dev, branch_dev,
                   metric_dev, nullptr, call);
}

eb_status eb_control_safe_batch_dev_gather(eb_controller* c, eb_peer_group* pg, eb_grid_batch* g, const eb_collision* col,
                                           const eb_dwa* dwa, double val_dt, double val_horizon, const double* bounds_dev,
                                           const double* x_dev, const int* mem_idx_dev, const double* vb_dev,
                                           int* branch_dev, double* metric_dev)
{
  EB_TRACE("eb_control_safe_batch_dev_gather");
  return safe_gather(c, pg, g, col, dwa, val_dt, val_horizon, bounds_dev, x_dev, mem_idx_dev, vb_dev, branch_dev,
                     metric_dev, false, "eb_control_safe_batch_dev_gather");
}

eb_status eb_control_safe_batch_dev_gather_wait(eb_controller* c, eb_peer_group* pg, eb_grid_batch* g,
                                                const eb_collision* col, const eb_dwa* dwa, double val_dt,
                                                double val_horizon, const double* bounds_dev, const double* x_dev,
                                                const int* mem_idx_dev, const double* vb_dev, int* branch_dev,
                                                double* metric_dev)
{
  EB_TRACE("eb_control_safe_batch_dev_gather_wait");
  return safe_gather(c, pg, g, col, dwa, val_dt, val_horizon, bounds_dev, x_dev, mem_idx_dev, vb_dev, branch_dev,
                     metric_dev, true, "eb_control_safe_batch_dev_gather_wait");
}

eb_status eb_control_safe_batch_host(eb_controller* c, eb_grid_batch* g, const eb_collision* col, const eb_dwa* dwa,
                                     double val_dt, double val_horizon, const double* bounds, const double* x,
                                     const int* mem_idx, const double* vb, double* u, int* branch, double* metric)
{
  EB_TRACE("eb_control_safe_batch_host");
  static const char* call = "eb_control_safe_batch_host";
  eb::DwaParams p{};
  eb::MapSet m{};
  eb_status st = safe_batch_check(c, g, col, dwa, val_dt, bounds, call, &p, &m);
  if (st != EB_OK) return st;
  if (!x || !vb || !u || !branch) return fail(EB_ERR_INVALID_ARGUMENT, std::string(call) + ": NULL argument");
  EB_CUDA(cudaSetDevice(c->cfg.device));
  if ((st = ensure_safe(c)) != EB_OK) return st;
  const size_t B = (size_t)c->B;
  if (bounds) EB_CUDA(cudaMemcpyAsync(c->d_bounds, bounds, sizeof(double) * 4 * B, cudaMemcpyHostToDevice, c->stream));
  const bool need_idx = mem_idx && c->mem_count > (long long)c->cfg.batch_size;
  if (need_idx)
    EB_CUDA(cudaMemcpyAsync(c->d_mem_idx_in, mem_idx, sizeof(int) * (size_t)c->cfg.batch_size * B,
                            cudaMemcpyHostToDevice, c->stream));
  EB_CUDA(cudaMemcpyAsync(c->d_pose, x, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, c->stream));
  EB_CUDA(cudaMemcpyAsync(c->d_safe_vb, vb, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, c->stream));
  st = eb_control_safe_batch_dev(c, g, col, dwa, val_dt, val_horizon, bounds ? c->d_bounds : nullptr, c->d_pose,
                                 need_idx ? c->d_mem_idx_in : nullptr, c->d_safe_vb, c->d_u0, c->d_safe_branch,
                                 metric ? c->d_metric : nullptr);
  if (st != EB_OK) return st;
  EB_CUDA(cudaMemcpyAsync(u, c->d_u0, sizeof(double) * 3 * B, cudaMemcpyDeviceToHost, c->stream));
  EB_CUDA(cudaMemcpyAsync(branch, c->d_safe_branch, sizeof(int) * B, cudaMemcpyDeviceToHost, c->stream));
  if (metric) EB_CUDA(cudaMemcpyAsync(metric, c->d_metric, sizeof(double) * B, cudaMemcpyDeviceToHost, c->stream));
  return check_fault(c);  // synchronises
}

// ---------------------------------------------------------------------------
// kinematic models + forward RK4 (model_kernels.cuh), SURVEY.md section 8 row a8 / a9
// ---------------------------------------------------------------------------
static eb_status model_params(int model, const double* params, eb::ModelParams* m)
{
  if (model < 0 || model > 3) return fail(EB_ERR_INVALID_ARGUMENT, "unknown model (0 SimpleCart, 1 Omni, 2 Cart, 3 Mecanum)");
  m->model = model;
  m->a = m->b = m->c = 0.0;
  if (model == eb::kModelCart || model == eb::kModelMecanum)
  {
    if (!params) return fail(EB_ERR_INVALID_ARGUMENT, "Cart / Mecanum need their wheel parameters");
    m->a = params[0];
    m->b = params[1];
    m->c = model == eb::kModelMecanum ? params[2] : 0.0;
  }
  return EB_OK;
}

int eb_model_controls(int model) { return (model >= 0 && model <= 3) ? eb::model_controls(model) : 0; }

eb_status eb_rk4_solve_dev(int device, int model, const double* params, double dt, double horizon, const double* x0_dev,
                           const double* ut_dev, int per_instance, int count, double* xt_dev, int* fault_dev,
                           void* cuda_stream)
{
  EB_TRACE("eb_rk4_solve_dev");
  eb::ModelParams m{};
  eb_status st = model_params(model, params, &m);
  if (st != EB_OK) return st;
  if (count < 0 || (count > 0 && (!x0_dev || !ut_dev || !xt_dev || !fault_dev)))
    return fail(EB_ERR_INVALID_ARGUMENT, "eb_rk4_solve_dev: bad arguments");
  if (!(dt != 0.0) || !std::isfinite(horizon / dt)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_rk4_solve: dt must be non-zero");
  const unsigned steps = static_cast<unsigned>(std::abs(horizon / dt));  // integrator.hpp:140
  if (count == 0 || steps == 0) return EB_OK;
  EB_CUDA(cudaSetDevice(device));
  const long long stride = per_instance ? (long long)steps * eb::model_controls(model) : 0LL;
  eb::rk4_solve_kernel<<<(count + 127) / 128, 128, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
      m, count, (int)steps, dt, x0_dev, ut_dev, stride, xt_dev, fault_dev);
  EB_CUDA(cudaGetLastError());
  return EB_OK;
}

eb_status eb_rk4_solve_host(int device, int model, const double* params, double dt, double horizon, const double* x0,
                            const double* ut, int per_instance, int count, double* xt)
{
  if (count < 0 || (count > 0 && (!x0 || !ut || !xt))) return fail(EB_ERR_INVALID_ARGUMENT, "eb_rk4_solve_host: bad arguments");
  if (!(dt != 0.0) || !std::isfinite(horizon / dt)) return fail(EB_ERR_INVALID_ARGUMENT, "eb_rk4_solve: dt must be non-zero");
  const unsigned steps = static_cast<unsigned>(std::abs(horizon / dt));
  if (count == 0 || steps == 0) return EB_OK;
  if (model < 0 || model > 3) return fail(EB_ERR_INVALID_ARGUMENT, "unknown model (0 SimpleCart, 1 Omni, 2 Cart, 3 Mecanum)");
  EB_CUDA(cudaSetDevice(device));
  const int nu = eb::model_controls(model);
  const size_t nut = (size_t)steps * nu * (per_instance ? (size_t)count : 1);
  DevBuf dx, du, dxt;
  int* d_fault = nullptr;
  EB_CUDA(dx.alloc(3 * (size_t)count));
  EB_CUDA(du.alloc(nut));
  EB_CUDA(dxt.alloc(3 * (size_t)steps * count));
  EB_CUDA(cudaMalloc(&d_fault, sizeof(int)));
  cudaError_t e = cudaMemset(d_fault, 0, sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(dx.p, x0, sizeof(double) * 3 * count, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(du.p, ut, sizeof(double) * nut, cudaMemcpyHostToDevice);
  eb_status st = EB_OK;
  if (e == cudaSuccess) st = eb_rk4_solve_dev(device, model, params, dt, horizon, dx.p, du.p, per_instance, count, dxt.p, d_fault, nullptr);
  int fault = 0;
  if (e == cudaSuccess && st == EB_OK) e = cudaMemcpy(xt, dxt.p, sizeof(double) * 3 * (size_t)steps * count, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && st == EB_OK) e = cudaMemcpy(&fault, d_fault, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(d_fault);
  if (st != EB_OK) return st;
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_rk4_solve_host: ") + cudaGetErrorString(e));
  if (fault) return fail(EB_ERR_INVALID_ARGUMENT, "Invalid twist y-velocity must be 0.");  // cart.hpp:169
  return EB_OK;
}

eb_status eb_model_eval_host(int device, int model, const double* params, const double* x, const double* u, int count,
                             double* f, double* A, double* B, double* vb)
{
  eb::ModelParams m{};
  eb_status st = model_params(model, params, &m);
  if (st != EB_OK) return st;
  if (count < 1 || !x || !u) return fail(EB_ERR_INVALID_ARGUMENT, "eb_model_eval_host: bad arguments");
  EB_CUDA(cudaSetDevice(device));
  const int nu = eb::model_controls(model);
  DevBuf dx, du, df, dA, dB, dv;
  int* d_fault = nullptr;
  EB_CUDA(dx.alloc(3 * (size_t)count));
  EB_CUDA(du.alloc((size_t)nu * count));
  EB_CUDA(df.alloc(3 * (size_t)count));
  EB_CUDA(dA.alloc(9 * (size_t)count));
  EB_CUDA(dB.alloc(3 * (size_t)nu * count));
  EB_CUDA(dv.alloc(3 * (size_t)count));
  EB_CUDA(cudaMalloc(&d_fault, sizeof(int)));
  cudaError_t e = cudaMemset(d_fault, 0, sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(dx.p, x, sizeof(double) * 3 * count, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(du.p, u, sizeof(double) * nu * count, cudaMemcpyHostToDevice);
  if (e == cudaSuccess)
  {
    eb::model_eval_kernel<<<(count + 127) / 128, 128>>>(m, count, dx.p, du.p, f ? df.p : nullptr, A ? dA.p : nullptr,
                                                        B ? dB.p : nullptr, vb ? dv.p : nullptr, d_fault);
    e = cudaGetLastError();
  }
  int fault = 0;
  if (e == cudaSuccess && f) e = cudaMemcpy(f, df.p, sizeof(double) * 3 * count, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && A) e = cudaMemcpy(A, dA.p, sizeof(double) * 9 * count, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && B) e = cudaMemcpy(B, dB.p, sizeof(double) * 3 * nu * count, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && vb) e = cudaMemcpy(vb, dv.p, sizeof(double) * 3 * count, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(&fault, d_fault, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(d_fault);
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_model_eval_host: ") + cudaGetErrorString(e));
  if (fault) return fail(EB_ERR_INVALID_ARGUMENT, "Invalid twist y-velocity must be 0.");  // cart.hpp:169
  return EB_OK;
}

// measured rate of random 1-byte loads over a 16 MB (L2-resident) buffer, in G sectors/s: the roofline
// denominator of the collision / DynamicWindow kernels (every probe moves one 32-byte L2 sector)
eb_status eb_l2_gather_peak(int device, double* gsectors_per_s)
{
  if (!gsectors_per_s) return fail(EB_ERR_INVALID_ARGUMENT, "eb_l2_gather_peak: NULL argument");
  EB_CUDA(cudaSetDevice(device));
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const size_t bytes = 16u << 20;
  unsigned char* buf = nullptr;
  unsigned int* sink = nullptr;
  EB_CUDA(cudaMalloc(&buf, bytes));
  EB_CUDA(cudaMalloc(&sink, sizeof(unsigned int)));
  cudaMemset(buf, 1, bytes);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  const int grid = sms * 8, threads = 256, iters = 256;
  double best = 0.0;
  for (int rep = 0; rep < 4; rep++)
  {
    cudaEventRecord(a);
    eb::l2_gather_probe<<<grid, threads>>>(buf, (unsigned int)(bytes - 1), iters, sink);
    cudaEventRecord(b);
    if (cudaEventSynchronize(b) != cudaSuccess) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    if (rep > 0) best = std::max(best, (double)grid * threads * iters * 8.0 / (ms * 1e-3) / 1e9);
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(buf);
  cudaFree(sink);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(EB_ERR_CUDA, std::string("eb_l2_gather_peak: ") + cudaGetErrorString(e));
  *gsectors_per_s = best;
  return EB_OK;
}

eb_status eb_fp64_peak(int device, double* dfma_tflops, double* dmma_tflops)
{
  EB_CUDA(cudaSetDevice(device));
  int sms = 0;
  EB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  double* d = nullptr;
  EB_CUDA(cudaMalloc(&d, sizeof(double)));
  cudaEvent_t a, b;
  EB_CUDA(cudaEventCreate(&a));
  EB_CUDA(cudaEventCreate(&b));
  const int grid = sms * 8, threads = 256, iters = 4096;
  double best[2] = { 0.0, 0.0 };
  for (int which = 0; which < 2; which++)
    for (int rep = 0; rep < 5; rep++)
    {
      cudaEventRecord(a);
      if (which == 0)
        eb::dfma_probe<<<grid, threads>>>(d, iters, 1.0);
      else
        eb::dmma_probe<<<grid, threads>>>(d, iters, 1.0);
      cudaEventRecord(b);
      cudaError_t e = cudaEventSynchronize(b);
      if (e != cudaSuccess)
      {
        cudaFree(d);
        return fail(EB_ERR_CUDA, std::string("eb_fp64_peak: ") + cudaGetErrorString(e));
      }
      float ms = 0.f;
      cudaEventElapsedTime(&ms, a, b);
      // dfma: 64 FMA per thread-iteration; dmma: 32 tiles of 8x8x4 = 256 FMA per warp-iteration
      const double flops = which == 0 ? 2.0 * 64.0 * iters * (double)grid * threads :
                                        2.0 * 256.0 * 32.0 * iters * (double)grid * (threads / 32);
      if (rep > 0) best[which] = std::max(best[which], flops / (ms * 1e-3) / 1e12);
    }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(d);
  if (dfma_tflops) *dfma_tflops = best[0];
  if (dmma_tflops) *dmma_tflops = best[1];
  return EB_OK;
}

}  // extern "C"
