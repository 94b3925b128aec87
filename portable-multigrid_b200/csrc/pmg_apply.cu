// pmg_apply.cu -- CUDA kernels + thin C-ABI launcher for the fused Laplace apply (K1).
// Algorithm and citations: pmg_apply_sweep.h (line-marching kernel, the default; launched from pmg_apply_sweep_m<mode>.cu),
// pmg_apply_tile.h (cell-tile kernel: small levels) and pmg_apply_var.h (variable coefficient).  sm_100a only; there is no fallback path.
#include "pmg_apply_tile.h"
#include "pmg_cuda_common.h"
#include "pmg_kernels.h"

template <class Tile>
struct PmgDeviceExec {
  typename Tile::ThreadState st;
  template <class F> __device__ __forceinline__ void for_each_thread(F f) { f((int)threadIdx.x, st); }
  __device__ __forceinline__ void sync() { __syncthreads(); }
};

template <int P, int BX, int BY, int MINB>
__global__ void __launch_bounds__(PmgApplyTile<P, BX, BY>::NT, MINB)
pmg_apply_kernel(const __grid_constant__ PmgApplyParams<P> p)
{
  using Tile = PmgApplyTile<P, BX, BY>;
  extern __shared__ double pmg_smem[];
  PmgDeviceExec<Tile> ex;
  const int b = blockIdx.x;
  const int tile_x = b % p.tiles_x;
  const int tile_y = (b / p.tiles_x) % p.tiles_y;
  const int chunk = b / (p.tiles_x * p.tiles_y);
  Tile::run(p, ex, pmg_smem, tile_x, tile_y, chunk);
}

// choose the number of z-chunks: minimise waves * (layers + halo layer)
static void choose_chunks(int tiles, int layers, int slots, int *n_chunks, int *layers_per_chunk)
{
  long best_cost = -1;
  int best_c = 1;
  for (int c = 1; c <= layers; ++c) {
    const int lpc = (layers + c - 1) / c;
    const int used = (layers + lpc - 1) / lpc;
    if (used != c) continue;
    const long waves = ((long)tiles * c + slots - 1) / slots;
    const long cost = waves * (lpc + (c > 1 ? 1 : 0));
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_c = c; }
  }
  *n_chunks = best_c;
  *layers_per_chunk = (layers + best_c - 1) / best_c;
}

template <int P, int BX, int BY, int MINB>
static int launch(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                  double *out, double f1, double f2, cudaStream_t stream, int *geom)
{
  using Tile = PmgApplyTile<P, BX, BY>;
  constexpr int N1 = P + 1;
  PmgApplyParams<P> p;
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
    PMG_CUDA_CHECK(cudaFuncSetAttribute(pmg_apply_kernel<P, BX, BY, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    PMG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, pmg_apply_kernel<P, BX, BY, MINB>, Tile::NT, smem_bytes));
    if (ctas_per_sm < 1) return PMG_ERR_CUDA;
    __atomic_store_n(&ctas_per_sm_dev[dev], ctas_per_sm, __ATOMIC_RELEASE);
  }
  const int slots = pmgk_device_sm_count() * ctas_per_sm;
  choose_chunks(p.tiles_x * p.tiles_y, lv->cz_hi - lv->cz_lo, slots, &p.n_chunks, &p.layers_per_chunk);
  for (int i = 0; i < N1 * N1; ++i) p.S[i] = lv->S[i];
  for (int i = 0; i < N1; ++i) p.lam[i] = lv->lam[i];
  p.c[0] = lv->h[1] * lv->h[2] / lv->h[0];
  p.c[1] = lv->h[0] * lv->h[2] / lv->h[1];
  p.c[2] = lv->h[0] * lv->h[1] / lv->h[2];
  p.mode = mode; p.u = u; p.b = b; p.xold = xold; p.out = out; p.f1 = f1; p.f2 = f2;
  p.dinv_vec = lv->dinv_vec; p.dinv_tab = lv->dinv_tab;
  const int grid = p.tiles_x * p.tiles_y * p.n_chunks;
  if (geom) { geom[0] = grid; geom[1] = Tile::NT; geom[2] = smem_bytes; geom[3] = p.n_chunks; return 0; }
  pmg_apply_kernel<P, BX, BY, MINB><<<grid, Tile::NT, smem_bytes, stream>>>(p);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

// line-marching kernel, one translation unit per epilogue mode: csrc/pmg_apply_sweep_m<mode>.cu
#define PMG_SWEEP_DECL(m) \
  int pmg_sweep_dispatch_m##m(const pmgk_level *lv, const double *u, const double *b, const double *xold, double *out, double f1, \
                              double f2, cudaStream_t s, int *geom, int part);
PMG_SWEEP_DECL(0) PMG_SWEEP_DECL(1) PMG_SWEEP_DECL(2) PMG_SWEEP_DECL(3)
#undef PMG_SWEEP_DECL

// plane-per-step kernel, one translation unit per epilogue mode (4 = CHEB_STEP without x_old): csrc/pmg_apply_plane_m<mode>.cu
#define PMG_PLANE_DECL(m) \
  int pmg_plane_dispatch_m##m(const pmgk_level *lv, const double *u, const double *b, const double *xold, double *out, double f1, \
                              double f2, cudaStream_t s, int *geom, int part);
PMG_PLANE_DECL(0) PMG_PLANE_DECL(1) PMG_PLANE_DECL(2) PMG_PLANE_DECL(3) PMG_PLANE_DECL(4)
#undef PMG_PLANE_DECL
#define PMG_PLANE_MAX_DEGREE 6

// 2-D levels: csrc/pmg_dim2.cu
int pmg_dim2_apply(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out, double f1,
                   double f2, cudaStream_t s, int *geom);

// variable-coefficient levels: csrc/pmg_apply_var.cu
int pmg_var_dispatch(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out,
                     double f1, double f2, cudaStream_t s, int *geom);
// levels with mapped geometry: csrc/pmg_apply_geo.cu
int pmg_geo_dispatch(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out,
                     double f1, double f2, cudaStream_t s, int *geom);

/* Small coarse levels run the cell-tile kernel (direct loads, lowest launch-to-result latency on one GPU) -- unless the level is
   a slab with neighbours: there every apply of the cell-tile kernel costs a ghost exchange (~17-30 us), which the plane-per-step
   kernel delivers from its own epilogue (fused push), so distributed levels of degrees 1..6 with >= 2 cell layers take it. */
static bool small_level_of(const pmgk_level *lv)
{
  const int64_t n_local = (int64_t)lv->Nx * lv->Ny * lv->nzl;
  const bool small = n_local < (lv->degree == 1 ? 100000 : 300000) && lv->degree <= 5;
  const bool slab_with_neighbours = lv->z_own_lo > 0 || lv->z_own_hi < lv->Nz;
  return small && !(slab_with_neighbours && lv->cz_hi - lv->cz_lo >= 2);
}

static int dispatch(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                    double *out, double f1, double f2, cudaStream_t s, int *geom, int part = PMGK_PART_ALL)
{
  /* the plane-per-step and the line-marching kernel launch in parts (their launches are cut into z-chunks) */
  const bool chunked_kernel = lv->dim == 3 && !lv->coef &&
                              (lv->tile_variant == 1 || lv->tile_variant == 6 || (lv->tile_variant == 0 && !small_level_of(lv)));
  if (part != PMGK_PART_ALL && !chunked_kernel) return PMG_ERR_UNSUPPORTED;
  if (lv->dim == 2) return pmg_dim2_apply(lv, mode, u, b, xold, out, f1, f2, s, geom);
  if (lv->nz < 1 || lv->cz_hi <= lv->cz_lo) return PMG_ERR_ARG;
  if (lv->coef && lv->geo_stride) return pmg_geo_dispatch(lv, mode, u, b, xold, out, f1, f2, s, geom);
  if (lv->coef) return pmg_var_dispatch(lv, mode, u, b, xold, out, f1, f2, s, geom);
  /* tile_variant 0 (default): the line-marching kernel for levels large enough to fill its copy pipeline, the cell-tile
     kernel (direct loads, no staging prologue) for the small coarse levels, where launch-to-result latency is everything:
     measured on B200 (tools/small_levels.py) 5.6-7.2 us against 7.0-12.3 us per fused step for Q1 up to 32^3 cells and
     12.3 against 16.4 us for Q2 on 32^3; from 64^3 cells on the line-marching kernel wins (14.3 : 17.1, 38.9 : 55.3 us).
     1 = line-marching always; 2, 3 = cell-tile always (small / large tiles); 6 = plane-per-step kernel always. */
  const bool small_level = small_level_of(lv);
  /* round 2: the plane-per-step kernel (csrc/pmg_apply_plane.h) takes the large levels of degrees 1..6 (measured at 100 M DoFs,
     apply / fused step in GDoF/s against the line-marching kernel: Q2 170 / 123 : 112 / 80, Q4 140 / 98 : 122 / 87);
     tile_variant 6 forces it, 1 forces the line-marching kernel */
  if (lv->degree <= PMG_PLANE_MAX_DEGREE && (lv->tile_variant == 6 || (lv->tile_variant == 0 && !small_level))) {
    switch (mode) {
      case PMGK_APPLY: return pmg_plane_dispatch_m0(lv, u, b, xold, out, f1, f2, s, geom, part);
      case PMGK_RESIDUAL: return pmg_plane_dispatch_m1(lv, u, b, xold, out, f1, f2, s, geom, part);
      case PMGK_CHEB_FIRST: return pmg_plane_dispatch_m2(lv, u, b, xold, out, f1, f2, s, geom, part);
      case PMGK_CHEB_STEP: return xold ? pmg_plane_dispatch_m3(lv, u, b, xold, out, f1, f2, s, geom, part)
                                       : pmg_plane_dispatch_m4(lv, u, b, xold, out, f1, f2, s, geom, part);
      default: return PMG_ERR_ARG;
    }
  }
  if (lv->tile_variant == 1 || lv->tile_variant == 6 /* degrees 7, 8: the line-marching kernel */ || (lv->tile_variant == 0 && !small_level)) {
    switch (mode) { /* one kernel per epilogue mode: csrc/pmg_apply_sweep_m<mode>.cu */
      case PMGK_APPLY: return pmg_sweep_dispatch_m0(lv, u, b, xold, out, f1, f2, s, geom, part);
      case PMGK_RESIDUAL: return pmg_sweep_dispatch_m1(lv, u, b, xold, out, f1, f2, s, geom, part);
      case PMGK_CHEB_FIRST: return pmg_sweep_dispatch_m2(lv, u, b, xold, out, f1, f2, s, geom, part);
      case PMGK_CHEB_STEP: return pmg_sweep_dispatch_m3(lv, u, b, xold, out, f1, f2, s, geom, part);
      default: return PMG_ERR_ARG;
    }
  }
#define PMG_LAUNCH(P, BX, BY, MINB) return launch<P, BX, BY, MINB>(lv, mode, u, b, xold, out, f1, f2, s, geom)
  if (lv->tile_variant != 3) { /* default: smaller tiles, two CTAs per SM (variant 2 = one large CTA per SM) */
    switch (lv->degree) {
      case 1: PMG_LAUNCH(1, 10, 10, 2);
      case 2: PMG_LAUNCH(2, 8, 8, 2);
      case 3: PMG_LAUNCH(3, 7, 7, 2);
      case 4: PMG_LAUNCH(4, 6, 6, 2);
      case 5: PMG_LAUNCH(5, 5, 4, 2);
      default: break;
    }
  }
  switch (lv->degree) {
    case 1: PMG_LAUNCH(1, 16, 16, 1);
    case 2: PMG_LAUNCH(2, 12, 12, 1);
    case 3: PMG_LAUNCH(3, 10, 10, 1);
    case 4: PMG_LAUNCH(4, 8, 8, 1);
    case 5: PMG_LAUNCH(5, 7, 7, 1);
    case 6: PMG_LAUNCH(6, 5, 5, 1);
    case 7: PMG_LAUNCH(7, 4, 5, 1);
    case 8: PMG_LAUNCH(8, 4, 4, 1);
    case 9: PMG_LAUNCH(9, 3, 3, 1);
    default: return PMG_ERR_UNSUPPORTED;
  }
#undef PMG_LAUNCH
}

extern "C" int pmgk_apply(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                          double *out, double f1, double f2, void *stream)
{
  if (!lv || !u || !out) return PMG_ERR_ARG;
  if (mode != PMGK_APPLY && !b) return PMG_ERR_ARG;
  if (u == out) return PMG_ERR_ARG; /* the halo of u is read by neighbouring tiles */
  return dispatch(lv, mode, u, b, xold, out, f1, f2, (cudaStream_t)stream, nullptr);
}

extern "C" int pmgk_apply_part(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                               double *out, double f1, double f2, int part, void *stream)
{
  if (!lv || !u || !out) return PMG_ERR_ARG;
  if (mode != PMGK_APPLY && !b) return PMG_ERR_ARG;
  if (u == out) return PMG_ERR_ARG;
  return dispatch(lv, mode, u, b, xold, out, f1, f2, (cudaStream_t)stream, nullptr, part);
}

thread_local const pmgk_push *pmg_tl_push = nullptr;

static bool plane_kernel_level(const pmgk_level *lv)
{
  const bool small_level = small_level_of(lv);
  return lv->dim == 3 && !lv->coef && lv->degree <= PMG_PLANE_MAX_DEGREE && (lv->tile_variant == 6 || (lv->tile_variant == 0 && !small_level));
}

extern "C" int pmgk_apply_can_push(const pmgk_level *lv, int mode)
{
  return lv && (mode == PMGK_RESIDUAL || mode == PMGK_CHEB_FIRST || mode == PMGK_CHEB_STEP) && plane_kernel_level(lv) && lv->cz_hi - lv->cz_lo >= 2;
}

extern "C" int pmgk_apply_push(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                               double *out, double f1, double f2, const pmgk_push *push, void *stream)
{
  if (!lv || !u || !out || !push) return PMG_ERR_ARG;
  if (mode != PMGK_APPLY && !b) return PMG_ERR_ARG;
  if (u == out) return PMG_ERR_ARG;
  if (!pmgk_apply_can_push(lv, mode)) return PMG_ERR_UNSUPPORTED;
  pmg_tl_push = push;
  const int rc = dispatch(lv, mode, u, b, xold, out, f1, f2, (cudaStream_t)stream, nullptr);
  pmg_tl_push = nullptr;
  return rc;
}

extern "C" int pmgk_apply_splits(const pmgk_level *lv, int mode)
{
  int g[4] = {0, 0, 0, 0};
  if (!lv) return 0;
  return dispatch(lv, mode, (const double *)16, (const double *)16, nullptr, (double *)32, 0, 0, 0, g, PMGK_PART_INTERIOR) == 0;
}

extern "C" int pmgk_apply_geometry(const pmgk_level *lv, int *grid, int *block, int *smem_bytes, int *n_chunks)
{
  int g[4] = {0, 0, 0, 0};
  const int rc = dispatch(lv, 0, (const double *)8, nullptr, nullptr, (double *)16, 0, 0, 0, g);
  if (grid) *grid = g[0];
  if (block) *block = g[1];
  if (smem_bytes) *smem_bytes = g[2];
  if (n_chunks) *n_chunks = g[3];
  return rc;
}
