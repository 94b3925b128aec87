// pmg_blas.cu -- vector kernels of the hot path (SURVEY.md K8-K14): the subset of
// LinearAlgebra::distributed::Vector operations the V-cycle, Chebyshev and CG use
// (reference call sites include/multigrid/portable_v_cycle_multigrid.h:116-125,166 and
// deal.II SolverCG / PreconditionChebyshev).  All are single-pass, coalesced, grid-stride
// kernels sized to the SM count; reductions are deterministic (fixed-shape two-stage tree).
#include "pmg_cuda_common.h"
#include "pmg_kernels.h"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 148 * 8; // two-stage reduction width (work buffer size)

int g_sm_count = 0;

inline int blocks_for(int64_t n)
{
  int64_t b = (n + kThreads - 1) / kThreads;
  int cap = (g_sm_count > 0 ? g_sm_count : 148) * 8;
  if (cap > kMaxBlocks) cap = kMaxBlocks; // the reductions' work buffer holds kMaxBlocks partial sums
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

__global__ void k_set(double *x, double a, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] = a;
}

__global__ void k_copy(double *__restrict__ dst, const double *__restrict__ src, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

__global__ void k_axpby(double *out, double a, const double *x, double b, const double *y, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = a * x[i] + b * y[i];
}

__global__ void k_scale(double *x, double a, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= a;
}

__global__ void k_set_mod11(double *x, int64_t first, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    x[i] = (double)((first + i) % 11);
}

__device__ __forceinline__ double block_sum(double v)
{
  __shared__ double warp_part[kThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x < 32) {
    r = (threadIdx.x < kThreads / 32) ? warp_part[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
  }
  return r; // valid on thread 0
}

// stage 1: per-block partial sums (each thread walks a fixed, grid-size-independent-of-timing set)
__global__ void k_dot_partial(const double *__restrict__ x, const double *__restrict__ y, int64_t n, double *work)
{
  double s = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += x[i] * y[i];
  s = block_sum(s);
  if (threadIdx.x == 0) work[blockIdx.x] = s;
}

__global__ void k_sum_partial(const double *__restrict__ x, int64_t n, double *work)
{
  double s = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += x[i];
  s = block_sum(s);
  if (threadIdx.x == 0) work[blockIdx.x] = s;
}

// stage 2: one block folds the partials in a fixed order
__global__ void k_reduce_final(const double *work, int nparts, double *result)
{
  double s = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) s += work[i];
  s = block_sum(s);
  if (threadIdx.x == 0) result[0] = s;
}

__global__ void k_cg_update_xr(double *x, double *r, const double *__restrict__ p, const double *__restrict__ Ap,
                               const double *alpha_dev, int64_t n, double *work)
{
  const double alpha = alpha_dev[0];
  double s = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    x[i] += alpha * p[i];
    const double ri = r[i] - alpha * Ap[i];
    r[i] = ri;
    s += ri * ri;
  }
  s = block_sum(s);
  if (threadIdx.x == 0) work[blockIdx.x] = s;
}

__global__ void k_cg_update_p(double *p, const double *__restrict__ z, const double *beta_dev, int64_t n)
{
  const double beta = beta_dev[0];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = z[i] + beta * p[i];
}

__global__ void k_scalar_div(double *out, const double *num, const double *den) { out[0] = num[0] / den[0]; }

} // namespace

extern "C" int pmgk_device_sm_count(void)
{
  if (g_sm_count == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
    g_sm_count = n;
  }
  return g_sm_count;
}

#define LAUNCH_CHECK()                        \
  do {                                        \
    PMG_CUDA_CHECK(cudaGetLastError());       \
    pmg_count_launch(1);                      \
  } while (0)

extern "C" int pmgk_set(double *x, double a, int64_t n, void *stream)
{
  if (n <= 0) return 0;
  pmgk_device_sm_count();
  k_set<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(x, a, n);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_copy(double *dst, const double *src, int64_t n, void *stream)
{
  if (n <= 0 || dst == src) return 0;
  pmgk_device_sm_count();
  k_copy<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(dst, src, n);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_axpby(double *out, double a, const double *x, double b, const double *y, int64_t n, void *stream)
{
  if (n <= 0) return 0;
  pmgk_device_sm_count();
  k_axpby<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(out, a, x, b, y, n);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_scale(double *x, double a, int64_t n, void *stream)
{
  if (n <= 0) return 0;
  pmgk_device_sm_count();
  k_scale<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(x, a, n);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_set_mod11(double *x, int64_t first_global, int64_t n, void *stream)
{
  if (n <= 0) return 0;
  pmgk_device_sm_count();
  k_set_mod11<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(x, first_global, n);
  LAUNCH_CHECK();
  return 0;
}

namespace {
// out[(z * Ny + y) * Nx + x] = lx[x] * ly[y] * lz[z]: one CTA row per (z, y)
__global__ void k_outer3(double *out, const double *__restrict__ lx, const double *__restrict__ ly, const double *__restrict__ lz,
                         int Nx, int Ny, int nz)
{
  for (int row = blockIdx.x; row < Ny * nz; row += gridDim.x) {
    const double f = ly[row % Ny] * lz[row / Ny];
    double *o = out + (int64_t)row * Nx;
    for (int x = threadIdx.x; x < Nx; x += blockDim.x) o[x] = f * lx[x];
  }
}

// Dirichlet rows of a level (the face-bitmask test of the apply kernels): one CTA row per stored (z, y) line, threads along x.
// 2-D levels have one plane (Nz = 1) and faces bits 0..3 only, so the same test holds.
__device__ __forceinline__ bool pmg_row_constrained_yz(int gy, int gz, int Ny, int Nz, unsigned faces)
{
  return (gy == 0 && (faces >> 2 & 1u)) || (gy == Ny - 1 && (faces >> 3 & 1u)) || (gz == 0 && (faces >> 4 & 1u)) ||
         (gz == Nz - 1 && (faces >> 5 & 1u));
}

// out = 0 on constrained rows, a x + b y elsewhere (y NULL: a x)
__global__ void k_masked_axpby(double *out, double a, const double *x, double b, const double *y, int Nx, int Ny, int Nz, int z0,
                               int nzl, unsigned faces)
{
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    const bool dyz = pmg_row_constrained_yz(row % Ny, z0 + row / Ny, Ny, Nz, faces);
    const int64_t o = (int64_t)row * Nx;
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      const bool dir = dyz || (gx == 0 && (faces & 1u)) || (gx == Nx - 1 && (faces >> 1 & 1u));
      out[o + gx] = dir ? 0.0 : (y ? a * x[o + gx] + b * y[o + gx] : a * x[o + gx]);
    }
  }
}

// out = src on constrained rows; elsewhere 0 (zero_free) or untouched
__global__ void k_constrained_copy(double *out, const double *__restrict__ src, int zero_free, int Nx, int Ny, int Nz, int z0, int nzl,
                                   unsigned faces)
{
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    const bool dyz = pmg_row_constrained_yz(row % Ny, z0 + row / Ny, Ny, Nz, faces);
    const int64_t o = (int64_t)row * Nx;
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      const bool dir = dyz || (gx == 0 && (faces & 1u)) || (gx == Nx - 1 && (faces >> 1 & 1u));
      if (dir) out[o + gx] = src[o + gx];
      else if (zero_free) out[o + gx] = 0.0;
    }
  }
}

// threads per CTA of the kernels that walk one row of Nx dofs
inline int row_threads(int Nx) { return Nx >= 192 ? 256 : (Nx >= 96 ? 128 : (Nx >= 48 ? 64 : 32)); }
} // namespace

extern "C" int pmgk_masked_axpby(const pmgk_level *lv, double *out, double a, const double *x, double b, const double *y, void *stream)
{
  if (!lv || !out || !x) return PMG_ERR_ARG;
  if (lv->nzl <= 0) return 0;
  int64_t rows = (int64_t)lv->Ny * lv->nzl;
  const int cap = pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_masked_axpby<<<(unsigned)rows, row_threads(lv->Nx), 0, (cudaStream_t)stream>>>(out, a, x, b, y, lv->Nx, lv->Ny, lv->Nz, lv->z0,
                                                                                   lv->nzl, lv->faces);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_constrained_copy(const pmgk_level *lv, double *out, const double *src, int zero_free, void *stream)
{
  if (!lv || !out || !src) return PMG_ERR_ARG;
  if (lv->nzl <= 0) return 0;
  int64_t rows = (int64_t)lv->Ny * lv->nzl;
  const int cap = pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_constrained_copy<<<(unsigned)rows, row_threads(lv->Nx), 0, (cudaStream_t)stream>>>(out, src, zero_free, lv->Nx, lv->Ny, lv->Nz,
                                                                                       lv->z0, lv->nzl, lv->faces);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_outer3(double *out, const double *lx, const double *ly, const double *lz, int Nx, int Ny, int nz, void *stream)
{
  if (Nx <= 0 || Ny <= 0 || nz <= 0) return 0;
  int64_t rows = (int64_t)Ny * nz;
  const int cap = pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_outer3<<<(unsigned)rows, row_threads(Nx), 0, (cudaStream_t)stream>>>(out, lx, ly, lz, Nx, Ny, nz);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_dot_work_doubles(void) { return kMaxBlocks; }

extern "C" int pmgk_dot(const double *x, const double *y, int64_t n, double *result, double *work, void *stream)
{
  pmgk_device_sm_count();
  const int nb = (n > 0) ? blocks_for(n) : 1;
  k_dot_partial<<<nb, kThreads, 0, (cudaStream_t)stream>>>(x, y, n > 0 ? n : 0, work);
  LAUNCH_CHECK();
  k_reduce_final<<<1, kThreads, 0, (cudaStream_t)stream>>>(work, nb, result);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_sum(const double *x, int64_t n, double *result, double *work, void *stream)
{
  pmgk_device_sm_count();
  const int nb = (n > 0) ? blocks_for(n) : 1;
  k_sum_partial<<<nb, kThreads, 0, (cudaStream_t)stream>>>(x, n > 0 ? n : 0, work);
  LAUNCH_CHECK();
  k_reduce_final<<<1, kThreads, 0, (cudaStream_t)stream>>>(work, nb, result);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_cg_update_xr(double *x, double *r, const double *p, const double *Ap, const double *alpha_dev,
                                 int64_t n, double *result, double *work, void *stream)
{
  pmgk_device_sm_count();
  const int nb = (n > 0) ? blocks_for(n) : 1;
  k_cg_update_xr<<<nb, kThreads, 0, (cudaStream_t)stream>>>(x, r, p, Ap, alpha_dev, n > 0 ? n : 0, work);
  LAUNCH_CHECK();
  k_reduce_final<<<1, kThreads, 0, (cudaStream_t)stream>>>(work, nb, result);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_cg_update_p(double *p, const double *z, const double *beta_dev, int64_t n, void *stream)
{
  if (n <= 0) return 0;
  pmgk_device_sm_count();
  k_cg_update_p<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(p, z, beta_dev, n);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int pmgk_scalar_div(double *out, const double *num, const double *den, void *stream)
{
  k_scalar_div<<<1, 1, 0, (cudaStream_t)stream>>>(out, num, den);
  LAUNCH_CHECK();
  return 0;
}
