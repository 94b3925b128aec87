// pmg_apply_var.cu -- CUDA kernel + launcher of the variable-coefficient apply (csrc/pmg_apply_var.h) and its set-up
// kernels (coefficient at the quadrature points, inverse diagonal).  sm_100a only; there is no fallback path.
#include "pmg_apply_var.h"
#include "pmg_cuda_common.h"
#include "pmg_kernels.h"

namespace {

template <class Tile>
struct PmgVarDeviceExec {
  typename Tile::ThreadState st;
  template <class F> __device__ __forceinline__ void for_each_thread(F f) { f((int)threadIdx.x, st); }
  __device__ __forceinline__ void sync() { __syncthreads(); }
};

template <int P, int BX, int BY, int MINB>
__global__ void __launch_bounds__(PmgVarTile<P, BX, BY>::NT, MINB)
pmg_var_kernel(const __grid_constant__ PmgVarParams<P> p)
{
  using Tile = PmgVarTile<P, BX, BY>;
  extern __shared__ double pmg_var_smem[];
  PmgVarDeviceExec<Tile> ex;
  const int b = blockIdx.x;
  const int tile_x = b % p.tiles_x;
  const int tile_y = (b / p.tiles_x) % p.tiles_y;
  const int chunk = b / (p.tiles_x * p.tiles_y);
  Tile::run(p, ex, pmg_var_smem, tile_x, tile_y, chunk);
}

template <int P, int BX, int BY, int MINB>
int launch_var(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out,
               double f1, double f2, cudaStream_t stream, int *geom)
{
  using Tile = PmgVarTile<P, BX, BY>;
  constexpr int N1 = P + 1;
  PmgVarParams<P> p;
  p.nx = lv->nx; p.ny = lv->ny; p.nz = lv->nz;
  p.Nx = lv->Nx; p.Ny = lv->Ny; p.Nz = lv->Nz;
  p.faces = lv->faces;
  p.z0 = lv->z0; p.nzl = lv->nzl;
  p.cz_lo = lv->cz_lo; p.cz_hi = lv->cz_hi;
  p.z_own_lo = lv->z_own_lo; p.z_own_hi = lv->z_own_hi;
  p.tiles_x = (lv->nx + BX - 1) / BX;
  p.tiles_y = (lv->ny + BY - 1) / BY;
  const int smem_bytes = Tile::SMEM_DOUBLES * (int)sizeof(double);
  // per device: the shared-memory opt-in and the occupancy belong to the device the launch goes to
  enum { MAXDEV = 64 };
  static int ctas_per_sm_dev[MAXDEV];
  int dev = 0;
  PMG_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= MAXDEV) return PMG_ERR_UNSUPPORTED;
  int ctas_per_sm = __atomic_load_n(&ctas_per_sm_dev[dev], __ATOMIC_ACQUIRE);
  if (ctas_per_sm == 0) {
    PMG_CUDA_CHECK(cudaFuncSetAttribute(pmg_var_kernel<P, BX, BY, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    PMG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, pmg_var_kernel<P, BX, BY, MINB>, Tile::NT, smem_bytes));
    if (ctas_per_sm < 1) return PMG_ERR_CUDA;
    __atomic_store_n(&ctas_per_sm_dev[dev], ctas_per_sm, __ATOMIC_RELEASE);
  }
  const int slots = pmgk_device_sm_count() * ctas_per_sm;
  pmg_var_choose_chunks(p.tiles_x * p.tiles_y, lv->cz_hi - lv->cz_lo, slots, &p.n_chunks, &p.layers_per_chunk);
  for (int i = 0; i < N1 * N1; ++i) { p.S[i] = lv->Sq[i]; p.D[i] = lv->Dco[i]; }
  for (int i = 0; i < N1; ++i) p.lam[i] = 0.0;
  p.c[0] = lv->h[1] * lv->h[2] / lv->h[0];
  p.c[1] = lv->h[0] * lv->h[2] / lv->h[1];
  p.c[2] = lv->h[0] * lv->h[1] / lv->h[2];
  p.mode = mode; p.u = u; p.b = b; p.xold = xold; p.out = out; p.f1 = f1; p.f2 = f2;
  p.dinv_vec = lv->dinv_vec; p.dinv_tab = lv->dinv_tab;
  p.coef = lv->coef; p.coef_cz0 = lv->coef_cz0;
  const int grid = p.tiles_x * p.tiles_y * p.n_chunks;
  if (geom) { geom[0] = grid; geom[1] = Tile::NT; geom[2] = smem_bytes; geom[3] = p.n_chunks; return 0; }
  if (mode >= PMG_MODE_CHEB_FIRST && !lv->dinv_vec) {
    pmg_set_error("variable-coefficient smoother step before compute_diagonal()");
    return PMG_ERR_STATE;
  }
  pmg_var_kernel<P, BX, BY, MINB><<<grid, Tile::NT, smem_bytes, stream>>>(p);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

// ---- set-up kernels ------------------------------------------------------------------------------------
struct VarTables {
  double a[PMGK_MAX_N1 * PMGK_MAX_N1], b[PMGK_MAX_N1 * PMGK_MAX_N1]; // (gq, gw) or (S2, G2)
  double h[3], c[3];
};

// one CTA row per (q-plane, q-row): no integer division per element
template <int P>
__global__ void k_var_coef(const __grid_constant__ VarTables t, int Qx, int Qy, int qz0, int nqz, double *coef)
{
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, qz = qz0 + row / Qy;
    double *o = coef + (int64_t)row * Qx;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) o[qx] = pmg_var_coef_c5<P>(qx, qy, qz, t.a, t.b, t.h);
  }
}

template <int P>
__global__ void k_var_dinv(const __grid_constant__ VarTables t, int nx, int ny, int Nx, int Ny, int Nz, int z0, int nzl,
                           int cz_min, int cz_max, unsigned faces, const double *__restrict__ coef, int coef_cz0, double *dinv)
{
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    const int gy = row % Ny, gz = z0 + row / Ny;
    const bool dyz = (gy == 0 && (faces >> 2 & 1u)) || (gy == Ny - 1 && (faces >> 3 & 1u)) ||
                     (gz == 0 && (faces >> 4 & 1u)) || (gz == Nz - 1 && (faces >> 5 & 1u));
    double *o = dinv + (int64_t)row * Nx;
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      const bool dir = dyz || (gx == 0 && (faces & 1u)) || (gx == Nx - 1 && (faces >> 1 & 1u));
      double d = 1.0; // constrained entries are set to 1 before the inversion (:906)
      if (!dir) d = pmg_var_diag_entry<P>(gx, gy, gz, nx, ny, cz_min, cz_max, t.a, t.b, t.c, coef, coef_cz0);
      o[gx] = 1.0 / d;
    }
  }
}

template <int P>
int fill_coef(const pmgk_level *lv, const double *gq, const double *gw, double *coef, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  VarTables t;
  for (int i = 0; i < N1; ++i) { t.a[i] = gq[i]; t.b[i] = gw[i]; }
  for (int d = 0; d < 3; ++d) { t.h[d] = lv->h[d]; t.c[d] = 0.0; }
  const int Qx = lv->nx * N1, Qy = lv->ny * N1, nqz = (lv->cz_hi - lv->coef_cz0) * N1;
  if (nqz <= 0) return 0;
  int64_t rows = (int64_t)Qy * nqz;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_var_coef<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, Qx, Qy, lv->coef_cz0 * N1, nqz, coef);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

template <int P>
int fill_dinv(const pmgk_level *lv, const double *S2, const double *G2, double *dinv, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  VarTables t;
  for (int i = 0; i < N1 * N1; ++i) { t.a[i] = S2[i]; t.b[i] = G2[i]; }
  for (int d = 0; d < 3; ++d) t.h[d] = lv->h[d];
  t.c[0] = lv->h[1] * lv->h[2] / lv->h[0];
  t.c[1] = lv->h[0] * lv->h[2] / lv->h[1];
  t.c[2] = lv->h[0] * lv->h[1] / lv->h[2];
  if (lv->nzl <= 0) return 0;
  int64_t rows = (int64_t)lv->Ny * lv->nzl;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_var_dinv<P><<<(unsigned)rows, pmg_var_row_threads(lv->Nx), 0, s>>>(t, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->Nz, lv->z0, lv->nzl,
                                                               lv->coef_cz0, lv->cz_hi, lv->faces, lv->coef, lv->coef_cz0, dinv);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

// ---- coefficient from the caller (pmg_laplace_operator_set_coefficient) ------------------------------------------------
// err = the smallest index i with a[i] not finite or <= 0 (err is ~0 on entry)
__global__ void k_coef_check(const double *__restrict__ a, int64_t n, unsigned long long *err)
{
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (!(isfinite(a[i]) && a[i] > 0.0)) atomicMin(err, (unsigned long long)i);
}

// W = w_q a_q on the quadrature-point grid of the stored cell layers (a == NULL: a = 1); wz: 1 = the weight of the q-plane
// enters (3-D), 0 = one plane of the 2-D grid
template <int P>
__global__ void k_var_coef_caller(const __grid_constant__ VarTables t, int Qx, int Qy, int nqz, int wz, const double *__restrict__ a,
                                  double *coef)
{
  constexpr int N1 = P + 1;
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, qz = row / Qy;
    const double wyz = t.b[qy % N1] * (wz ? t.b[qz % N1] : 1.0);
    const int64_t o = (int64_t)row * Qx;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) coef[o + qx] = t.b[qx % N1] * wyz * (a ? a[o + qx] : 1.0);
  }
}

template <int P>
int set_coef(const pmgk_level *lv, const double *gw, const double *a, double *coef, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  VarTables t;
  for (int i = 0; i < N1; ++i) { t.a[i] = 0.0; t.b[i] = gw[i]; }
  const int Qx = lv->nx * N1, Qy = lv->ny * N1, nqz = lv->dim == 2 ? 1 : (lv->cz_hi - lv->coef_cz0) * N1;
  if (nqz <= 0) return 0;
  int64_t rows = (int64_t)Qy * nqz;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_var_coef_caller<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, Qx, Qy, nqz, lv->dim == 3, a, coef);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

} // namespace

// called by pmgk_apply (pmg_apply.cu) for levels that carry a coefficient
int pmg_var_dispatch(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out,
                     double f1, double f2, cudaStream_t s, int *geom)
{
  if (lv->nz < 1 || lv->cz_hi <= lv->cz_lo || !lv->coef) return PMG_ERR_ARG;
  switch (lv->degree) {
#define PMG_VAR_CASE(P, BX, BY, MINB) \
  case P: return launch_var<P, BX, BY, MINB>(lv, mode, u, b, xold, out, f1, f2, s, geom);
#include "pmg_apply_var_tiles.inc"
#undef PMG_VAR_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int64_t pmgk_var_coef_doubles(const pmgk_level *lv)
{
  if (!lv) return 0;
  const int64_t n1 = lv->degree + 1;
  const int64_t layers = lv->cz_hi - lv->coef_cz0;
  return layers > 0 ? layers * n1 * (lv->nx * n1) * (lv->ny * n1) : 0;
}

extern "C" int pmgk_var_fill_coef(const pmgk_level *lv, int kind, const double *gq, const double *gw, double *coef, void *stream)
{
  if (!lv || !gq || !gw || !coef) return PMG_ERR_ARG;
  if (kind != 1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
    case 1: return fill_coef<1>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 2: return fill_coef<2>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 3: return fill_coef<3>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 4: return fill_coef<4>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 5: return fill_coef<5>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 6: return fill_coef<6>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 7: return fill_coef<7>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 8: return fill_coef<8>(lv, gq, gw, coef, (cudaStream_t)stream);
    case 9: return fill_coef<9>(lv, gq, gw, coef, (cudaStream_t)stream);
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_var_fill_dinv(const pmgk_level *lv, const double *S2, const double *G2, double *dinv, void *stream)
{
  if (!lv || !S2 || !G2 || !dinv || !lv->coef) return PMG_ERR_ARG;
  switch (lv->degree) {
    case 1: return fill_dinv<1>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 2: return fill_dinv<2>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 3: return fill_dinv<3>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 4: return fill_dinv<4>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 5: return fill_dinv<5>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 6: return fill_dinv<6>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 7: return fill_dinv<7>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 8: return fill_dinv<8>(lv, S2, G2, dinv, (cudaStream_t)stream);
    case 9: return fill_dinv<9>(lv, S2, G2, dinv, (cudaStream_t)stream);
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_coef_check(const double *a, int64_t n, unsigned long long *err, void *stream)
{
  if (!a || !err || n < 0) return PMG_ERR_ARG;
  if (n == 0) return 0;
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  k_coef_check<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, n, err);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

extern "C" int pmgk_var_set_coef(const pmgk_level *lv, const double *gw, const double *a, double *coef, void *stream)
{
  if (!lv || !gw || !coef) return PMG_ERR_ARG;
  switch (lv->degree) {
    case 1: return set_coef<1>(lv, gw, a, coef, (cudaStream_t)stream);
    case 2: return set_coef<2>(lv, gw, a, coef, (cudaStream_t)stream);
    case 3: return set_coef<3>(lv, gw, a, coef, (cudaStream_t)stream);
    case 4: return set_coef<4>(lv, gw, a, coef, (cudaStream_t)stream);
    case 5: return set_coef<5>(lv, gw, a, coef, (cudaStream_t)stream);
    case 6: return set_coef<6>(lv, gw, a, coef, (cudaStream_t)stream);
    case 7: return set_coef<7>(lv, gw, a, coef, (cudaStream_t)stream);
    case 8: return set_coef<8>(lv, gw, a, coef, (cudaStream_t)stream);
    case 9: return set_coef<9>(lv, gw, a, coef, (cudaStream_t)stream);
    default: return PMG_ERR_UNSUPPORTED;
  }
}
