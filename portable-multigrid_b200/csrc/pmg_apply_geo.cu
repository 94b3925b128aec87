// pmg_apply_geo.cu -- the Laplace operator on mapped hexahedral meshes: CUDA kernel + launcher of the tensor variant of the
// variable-coefficient tile program (PmgVarTile<P, BX, BY, true>, csrc/pmg_apply_var.h) and its set-up kernels (the
// per-point tensor G_q from the cells' trilinear maps or, for curved cells, from their degree-k Lagrange maps through
// (k+1)^3 nodes, with the validity check; inverse diagonal; load vector; solution norm).  sm_100a only; there is no
// fallback path.
//
// The reference's quadrature-point operation is  g <- JxW J^-1 J^-T g  with inv_jacobian(q,cell,d,e) and JxW(q,cell)
// stored per point (include/operators/portable_laplace_operator.h:301-325).  Here the symmetric product is merged into
// six doubles per point (48 B instead of the reference's 10 geometry doubles), so an apply streams
// 16 + 48 (p+1)^3 / p^3 B/DoF.
#include "pmg_apply_var.h"
#include "pmg_cuda_common.h"
#include "pmg_kernels.h"

extern "C" void pmg_fe_gll(int n, double *x);
extern "C" void pmg_fe_lagrange(int n, const double *nodes, double x, double *val, double *der);

namespace {

template <class Tile>
struct PmgGeoDeviceExec {
  typename Tile::ThreadState st;
  template <class F> __device__ __forceinline__ void for_each_thread(F f) { f((int)threadIdx.x, st); }
  __device__ __forceinline__ void sync() { __syncthreads(); }
};

template <int P, int BX, int BY, int MINB>
__global__ void __launch_bounds__(PmgVarTile<P, BX, BY, true>::NT, MINB)
pmg_geo_kernel(const __grid_constant__ PmgGeoParams<P> p)
{
  using Tile = PmgVarTile<P, BX, BY, true>;
  extern __shared__ double pmg_geo_smem[];
  PmgGeoDeviceExec<Tile> ex;
  const int b = blockIdx.x;
  const int tile_x = b % p.tiles_x;
  const int tile_y = (b / p.tiles_x) % p.tiles_y;
  const int chunk = b / (p.tiles_x * p.tiles_y);
  Tile::run(p, ex, pmg_geo_smem, tile_x, tile_y, chunk);
}

template <int P, int BX, int BY, int MINB>
int launch_geo(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out,
               double f1, double f2, cudaStream_t stream, int *geom)
{
  using Tile = PmgVarTile<P, BX, BY, true>;
  constexpr int N1 = P + 1;
  PmgGeoParams<P> p;
  p.nx = lv->nx; p.ny = lv->ny; p.nz = lv->nz;
  p.Nx = lv->Nx; p.Ny = lv->Ny; p.Nz = lv->Nz;
  p.faces = lv->faces;
  p.z0 = lv->z0; p.nzl = lv->nzl;
  p.cz_lo = lv->cz_lo; p.cz_hi = lv->cz_hi;
  p.z_own_lo = lv->z_own_lo; p.z_own_hi = lv->z_own_hi;
  p.tiles_x = (lv->nx + BX - 1) / BX;
  p.tiles_y = (lv->ny + BY - 1) / BY;
  const int smem_bytes = Tile::SMEM_DOUBLES * (int)sizeof(double);
  enum { MAXDEV = 64 };
  static int ctas_per_sm_dev[MAXDEV];
  int dev = 0;
  PMG_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= MAXDEV) return PMG_ERR_UNSUPPORTED;
  int ctas_per_sm = __atomic_load_n(&ctas_per_sm_dev[dev], __ATOMIC_ACQUIRE);
  if (ctas_per_sm == 0) {
    PMG_CUDA_CHECK(cudaFuncSetAttribute(pmg_geo_kernel<P, BX, BY, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    PMG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, pmg_geo_kernel<P, BX, BY, MINB>, Tile::NT, smem_bytes));
    if (ctas_per_sm < 1) return PMG_ERR_CUDA;
    __atomic_store_n(&ctas_per_sm_dev[dev], ctas_per_sm, __ATOMIC_RELEASE);
  }
  const int slots = pmgk_device_sm_count() * ctas_per_sm;
  pmg_var_choose_chunks(p.tiles_x * p.tiles_y, lv->cz_hi - lv->cz_lo, slots, &p.n_chunks, &p.layers_per_chunk);
  for (int i = 0; i < N1 * N1; ++i) { p.S[i] = lv->Sq[i]; p.D[i] = lv->Dco[i]; }
  for (int i = 0; i < N1; ++i) p.lam[i] = 0.0;
  for (int d = 0; d < 3; ++d) p.c[d] = 0.0; // folded into G
  p.mode = mode; p.u = u; p.b = b; p.xold = xold; p.out = out; p.f1 = f1; p.f2 = f2;
  p.dinv_vec = lv->dinv_vec; p.dinv_tab = lv->dinv_tab;
  p.coef = lv->coef; p.coef_cz0 = lv->coef_cz0;
  p.gstride = lv->geo_stride;
  const int grid = p.tiles_x * p.tiles_y * p.n_chunks;
  if (geom) { geom[0] = grid; geom[1] = Tile::NT; geom[2] = smem_bytes; geom[3] = p.n_chunks; return 0; }
  if (mode >= PMG_MODE_CHEB_FIRST && !lv->dinv_vec) {
    pmg_set_error("mapped-geometry smoother step before compute_diagonal()");
    return PMG_ERR_STATE;
  }
  pmg_geo_kernel<P, BX, BY, MINB><<<grid, Tile::NT, smem_bytes, stream>>>(p);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

// ---- set-up kernels ------------------------------------------------------------------------------------
struct GeoTables {
  // (gq, gw, -), (S2, G2, SG), (S, -, -) or (E, gq, gw) of QGauss(p+2): E is (p+2) x (p+1)
  double a[(PMGK_MAX_N1 + 1) * PMGK_MAX_N1], b[PMGK_MAX_N1 * PMGK_MAX_N1], c[PMGK_MAX_N1 * PMGK_MAX_N1];
};

// curved cells (degree-k geometry): L / dL[q * (k+1) + i] = value / derivative of the degree-k Gauss-Lobatto basis function i
// at quadrature point q, w the quadrature weights, E (norm only) the (p+2) x (p+1) FE_Q(p) values at the points
struct CurvedTables {
  double L[(PMGK_MAX_N1 + 1) * PMGK_MAX_N1], dL[(PMGK_MAX_N1 + 1) * PMGK_MAX_N1], E[(PMGK_MAX_N1 + 1) * PMGK_MAX_N1];
  double w[PMGK_MAX_N1 + 1];
};

void curved_tables(int k, int nq, const double *xq, const double *wq, CurvedTables &t)
{
  double s[PMGK_MAX_N1];
  pmg_fe_gll(k + 1, s);
  for (int q = 0; q < nq; ++q) {
    pmg_fe_lagrange(k + 1, s, xq[q], t.L + q * (k + 1), t.dL + q * (k + 1));
    t.w[q] = wq[q];
  }
}

// first node of cell (cx, cy) of local cell layer lcz in the node planes of a level (k nodes per cell and direction)
__device__ const double *curved_cell_node(const double *nodes, int nx, int ny, int k, int cx, int cy, int lcz)
{
  const int64_t mx = (int64_t)nx * k + 1, my = (int64_t)ny * k + 1;
  return nodes + 3 * ((int64_t)lcz * k * mx * my + (int64_t)cy * k * mx + (int64_t)cx * k);
}

__device__ void geo_load_cell(const double *vert, int nx, int ny, int cx, int cy, int lcz, double (*v)[3])
{
  const int64_t vplane = (int64_t)(nx + 1) * (ny + 1);
  for (int c = 0; c < 8; ++c) {
    const double *pv = vert + 3 * ((int64_t)(lcz + (c >> 2)) * vplane + (int64_t)(cy + (c >> 1 & 1)) * (nx + 1) + cx + (c & 1));
    for (int d = 0; d < 3; ++d) v[c][d] = pv[d];
  }
}

// one CTA row per (q-plane, q-row) of the quadrature-point grid, threads along x
template <int P>
__global__ void k_geo_fill(const __grid_constant__ GeoTables t, int nx, int ny, int cz0, int nqz, int c5,
                           const double *__restrict__ vert, int64_t gstride, double *geo, unsigned long long *err)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1, Qy = ny * N1;
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, lqz = row / Qy;
    const int cy = qy / N1, b = qy % N1, lcz = lqz / N1, m = lqz % N1;
    double *o = geo + (int64_t)row * Qx;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) {
      const int cx = qx / N1, a = qx % N1;
      double v[8][3];
      geo_load_cell(vert, nx, ny, cx, cy, lcz, v);
      bool finite = true;
      for (int c = 0; c < 8; ++c)
        for (int d = 0; d < 3; ++d) finite = finite && isfinite(v[c][d]);
      double G[6];
      const double det = pmg_geo_point(v, t.a[a], t.a[b], t.a[m], t.b[a] * t.b[b] * t.b[m], c5, G);
      for (int k = 0; k < 6; ++k) o[qx + k * gstride] = G[k];
      if (!finite || !(det > 0.0))
        atomicMin(err, (unsigned long long)(cx + (int64_t)nx * (cy + (int64_t)ny * (cz0 + lcz))));
    }
  }
}

// as k_geo_fill for curved cells: x and J from the cell's (k+1)^3 nodes (pmg_curved_point)
template <int P>
__global__ void k_curved_fill(const __grid_constant__ CurvedTables t, int k, int nx, int ny, int cz0, int nqz, int c5,
                              const double *__restrict__ nodes, int64_t gstride, double *geo, unsigned long long *err)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1, Qy = ny * N1, k1 = k + 1;
  const int64_t sy = (int64_t)nx * k + 1, sz = sy * ((int64_t)ny * k + 1);
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, lqz = row / Qy;
    const int cy = qy / N1, b = qy % N1, lcz = lqz / N1, m = lqz % N1;
    double *o = geo + (int64_t)row * Qx;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) {
      const int cx = qx / N1, a = qx % N1;
      double G[6];
      const double det = pmg_curved_point(curved_cell_node(nodes, nx, ny, k, cx, cy, lcz), sy, sz, k, t.L + a * k1, t.dL + a * k1,
                                          t.L + b * k1, t.dL + b * k1, t.L + m * k1, t.dL + m * k1, t.w[a] * t.w[b] * t.w[m], c5, G);
      for (int e = 0; e < 6; ++e) o[qx + e * gstride] = G[e];
      if (!(det > 0.0)) atomicMin(err, (unsigned long long)(cx + (int64_t)nx * (cy + (int64_t)ny * (cz0 + lcz))));
    }
  }
}

template <int P>
__global__ void k_geo_dinv(const __grid_constant__ GeoTables t, int nx, int ny, int Nx, int Ny, int Nz, int z0, int nzl,
                           int cz_min, int cz_max, unsigned faces, const double *__restrict__ geo, int64_t gstride, double *dinv)
{
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    const int gy = row % Ny, gz = z0 + row / Ny;
    const bool dyz = (gy == 0 && (faces >> 2 & 1u)) || (gy == Ny - 1 && (faces >> 3 & 1u)) ||
                     (gz == 0 && (faces >> 4 & 1u)) || (gz == Nz - 1 && (faces >> 5 & 1u));
    double *o = dinv + (int64_t)row * Nx;
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      const bool dir = dyz || (gx == 0 && (faces & 1u)) || (gx == Nx - 1 && (faces >> 1 & 1u));
      double d = 1.0; // constrained entries are set to 1 before the inversion (:906)
      if (!dir) d = pmg_geo_diag_entry<P>(gx, gy, gz, nx, ny, cz_min, cz_max, t.a, t.b, t.c, geo, gstride, cz_min);
      o[gx] = 1.0 / d;
    }
  }
}

// ---- right-hand side and solution norm on the mapped mesh (not separable any more) --------------------------------------
// det J of the trilinear map with vertices v at the reference point (x, y, z)
__device__ double geo_det(const double (*v)[3], double x, double y, double z)
{
  double G[6];
  return pmg_geo_point(v, x, y, z, 1.0, 0, G);
}


// w_q |det J_q| on the quadrature-point grid of the stored cell layers (layout of one G grid)
template <int P>
__global__ void k_geo_jxw(const __grid_constant__ GeoTables t, int nx, int ny, int nqz, const double *__restrict__ vert, double *W)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1, Qy = ny * N1;
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, lqz = row / Qy;
    const int cy = qy / N1, b = qy % N1, lcz = lqz / N1, m = lqz % N1;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) {
      const int cx = qx / N1, a = qx % N1;
      double v[8][3];
      geo_load_cell(vert, nx, ny, cx, cy, lcz, v);
      W[(int64_t)row * Qx + qx] = t.b[a] * t.b[b] * t.b[m] * fabs(geo_det(v, t.a[a], t.a[b], t.a[m]));
    }
  }
}

// as k_geo_jxw for curved cells
template <int P>
__global__ void k_curved_jxw(const __grid_constant__ CurvedTables t, int k, int nx, int ny, int nqz, const double *__restrict__ nodes,
                             double *W)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1, Qy = ny * N1, k1 = k + 1;
  const int64_t sy = (int64_t)nx * k + 1, sz = sy * ((int64_t)ny * k + 1);
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, lqz = row / Qy;
    const int cy = qy / N1, b = qy % N1, lcz = lqz / N1, m = lqz % N1;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) {
      const int cx = qx / N1, a = qx % N1;
      double G[6];
      const double det = pmg_curved_point(curved_cell_node(nodes, nx, ny, k, cx, cy, lcz), sy, sz, k, t.L + a * k1, t.dL + a * k1,
                                          t.L + b * k1, t.dL + b * k1, t.L + m * k1, t.dL + m * k1, 1.0, 0, G);
      W[(int64_t)row * Qx + qx] = t.w[a] * t.w[b] * t.w[m] * fabs(det);
    }
  }
}

// load vector of f = 1: b_i = sum over the <= 8 cells of dof i of sum_q phi_i(xi_q) w_q |det J_q|, constrained rows 0;
// one thread per dof of the stored planes, cells [cz_min, cz_max) (ghost planes get the stored cells' part only)
template <int P>
__global__ void k_geo_rhs(const __grid_constant__ GeoTables t, int nx, int ny, int Nx, int Ny, int Nz, int z0, int nzl, int cz_min,
                          int cz_max, unsigned faces, const double *__restrict__ W, double *rhs)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1;
  const int64_t Qplane = (int64_t)Qx * (ny * N1);
  const double *S = t.a;
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    const int gy = row % Ny, gz = z0 + row / Ny;
    const bool dyz = (gy == 0 && (faces >> 2 & 1u)) || (gy == Ny - 1 && (faces >> 3 & 1u)) ||
                     (gz == 0 && (faces >> 4 & 1u)) || (gz == Nz - 1 && (faces >> 5 & 1u));
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      const bool dir = dyz || (gx == 0 && (faces & 1u)) || (gx == Nx - 1 && (faces >> 1 & 1u));
      double sum = 0.0;
      for (int ez = 0; ez < 2 && !dir; ++ez) {
        const int cz = gz / P - ez, iz = gz - cz * P;
        if (cz < cz_min || cz >= cz_max || iz > P) continue;
        for (int ey = 0; ey < 2; ++ey) {
          const int cy = gy / P - ey, iy = gy - cy * P;
          if (cy < 0 || cy >= ny || iy > P) continue;
          for (int ex = 0; ex < 2; ++ex) {
            const int cx = gx / P - ex, ix = gx - cx * P;
            if (cx < 0 || cx >= nx || ix > P) continue;
            const double *cw = W + (int64_t)(cz - cz_min) * N1 * Qplane + (int64_t)(cy * N1) * Qx + cx * N1;
            for (int m = 0; m < N1; ++m)
              for (int b = 0; b < N1; ++b) {
                const double *r = cw + m * Qplane + (int64_t)b * Qx;
                double s = 0.0;
                for (int a = 0; a < N1; ++a) s += S[a * N1 + ix] * r[a];
                sum += S[m * N1 + iz] * S[b * N1 + iy] * s;
              }
          }
        }
      }
      rhs[(int64_t)row * Nx + gx] = sum;
    }
  }
}

// integral of u_h^2 over one cell with QGauss(p+2) (integrate_difference, program.cc:382-395): u interpolated to the
// (p+2)^3 points with E[q][i] = phi_i(x_q), weighted with gw_x gw_y gw_z jac(qx, qy, qz), jac = |det J| at the point;
// x-interpolated values in t1
template <int P, class Jac>
__device__ __forceinline__ double geo_cell_u2(const double *E, const double *gw, int Nx, int Ny, int z0, int cx, int cy, int cz,
                                              const double *__restrict__ u, Jac jac)
{
  constexpr int N1 = P + 1, M = P + 2;
  double t1[N1][N1][M]; // [k][j][qx]
  for (int k = 0; k < N1; ++k)
    for (int j = 0; j < N1; ++j) {
      const double *row = u + ((int64_t)(cz * P + k - z0) * Ny + cy * P + j) * Nx + cx * P;
      for (int qx = 0; qx < M; ++qx) {
        double s = 0.0;
        for (int i = 0; i < N1; ++i) s += E[qx * N1 + i] * row[i];
        t1[k][j][qx] = s;
      }
    }
  double total = 0.0;
  for (int qz = 0; qz < M; ++qz)
    for (int qy = 0; qy < M; ++qy)
      for (int qx = 0; qx < M; ++qx) {
        double val = 0.0;
        for (int k = 0; k < N1; ++k) {
          double s = 0.0;
          for (int j = 0; j < N1; ++j) s += E[qy * N1 + j] * t1[k][j][qx];
          val += E[qz * N1 + k] * s;
        }
        total += val * val * gw[qx] * gw[qy] * gw[qz] * jac(qx, qy, qz);
      }
  return total;
}

// per owned cell of the mapped mesh: geo_cell_u2 with the trilinear map's det J; one thread per cell
template <int P>
__global__ void k_geo_norm_cells(const __grid_constant__ GeoTables t, int nx, int ny, int Nx, int Ny, int z0, int cz_lo, int cz_hi,
                                 int vert_cz0, const double *__restrict__ vert, const double *__restrict__ u, double *cell_sums)
{
  const double *E = t.a, *gq = t.b, *gw = t.c;
  const int64_t ncells = (int64_t)nx * ny * (cz_hi - cz_lo);
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x) {
    const int cx = (int)(c % nx), cy = (int)(c / nx % ny), cz = cz_lo + (int)(c / ((int64_t)nx * ny));
    double v[8][3];
    geo_load_cell(vert, nx, ny, cx, cy, cz - vert_cz0, v);
    cell_sums[c] = geo_cell_u2<P>(E, gw, Nx, Ny, z0, cx, cy, cz, u,
                                  [&](int qx, int qy, int qz) { return fabs(geo_det(v, gq[qx], gq[qy], gq[qz])); });
  }
}

// as k_geo_norm_cells for curved cells: det J of the degree-k map at the (p+2)^3 points
template <int P>
__global__ void k_curved_norm_cells(const __grid_constant__ CurvedTables t, int k, int nx, int ny, int Nx, int Ny, int z0,
                                    int cz_lo, int cz_hi, int node_cz0, const double *__restrict__ nodes, const double *__restrict__ u,
                                    double *cell_sums)
{
  const int k1 = k + 1;
  const int64_t sy = (int64_t)nx * k + 1, sz = sy * ((int64_t)ny * k + 1);
  const int64_t ncells = (int64_t)nx * ny * (cz_hi - cz_lo);
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x) {
    const int cx = (int)(c % nx), cy = (int)(c / nx % ny), cz = cz_lo + (int)(c / ((int64_t)nx * ny));
    const double *node = curved_cell_node(nodes, nx, ny, k, cx, cy, cz - node_cz0);
    cell_sums[c] = geo_cell_u2<P>(t.E, t.w, Nx, Ny, z0, cx, cy, cz, u, [&](int qx, int qy, int qz) {
      double G[6];
      return fabs(pmg_curved_point(node, sy, sz, k, t.L + qx * k1, t.dL + qx * k1, t.L + qy * k1, t.dL + qy * k1, t.L + qz * k1,
                                   t.dL + qz * k1, 1.0, 0, G));
    });
  }
}

// ---- problem data from the caller: load vector of a nodal f, support points ------------------------------------------
// W *= f_h at the quadrature points of the stored cell layers [cz_min, cz_max): f_h = sum_j f_j phi_j interpolated from the
// cell's (p+1)^3 dofs to its (p+1)^3 Gauss points by sum factorisation with S[q][i] = phi_i(x_q) (x, then y, then z); one
// thread per cell, W in the layout of one G grid, f a local vector with current ghosts
template <int P>
__global__ void k_geo_mul_f(const __grid_constant__ GeoTables t, int nx, int ny, int Nx, int Ny, int z0, int cz_min, int cz_max,
                            const double *__restrict__ f, double *W)
{
  constexpr int N1 = P + 1;
  const double *S = t.a;
  const int Qx = nx * N1;
  const int64_t Qplane = (int64_t)Qx * (ny * N1);
  const int64_t ncells = (int64_t)nx * ny * (cz_max - cz_min);
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x) {
    const int cx = (int)(c % nx), cy = (int)(c / nx % ny), lcz = (int)(c / ((int64_t)nx * ny)), cz = cz_min + lcz;
    double t1[N1][N1][N1]; // [k][j][qx]
    for (int k = 0; k < N1; ++k)
      for (int j = 0; j < N1; ++j) {
        const double *row = f + ((int64_t)(cz * P + k - z0) * Ny + cy * P + j) * Nx + cx * P;
        for (int a = 0; a < N1; ++a) {
          double s = 0.0;
          for (int i = 0; i < N1; ++i) s += S[a * N1 + i] * row[i];
          t1[k][j][a] = s;
        }
      }
    double *cw = W + (int64_t)lcz * N1 * Qplane + (int64_t)(cy * N1) * Qx + cx * N1;
    for (int b = 0; b < N1; ++b) {
      double t2[N1][N1]; // [k][qx] at qy = b
      for (int k = 0; k < N1; ++k)
        for (int a = 0; a < N1; ++a) {
          double s = 0.0;
          for (int j = 0; j < N1; ++j) s += S[b * N1 + j] * t1[k][j][a];
          t2[k][a] = s;
        }
      for (int m = 0; m < N1; ++m)
        for (int a = 0; a < N1; ++a) {
          double s = 0.0;
          for (int k = 0; k < N1; ++k) s += S[m * N1 + k] * t2[k][a];
          cw[m * Qplane + (int64_t)b * Qx + a] *= s;
        }
    }
  }
}

// The cell a dof of the stored planes is evaluated in: the lower one at a cell boundary (the last cell at the upper end), in z
// the stored cell layers [cz_min, cz_max).  At a cell boundary the 1-D weights are exactly 0 and 1, so every cell that holds
// the dof gives the same bits, on every rank.
__device__ __forceinline__ void support_cell(int g, int P, int c_max, int *c, int *i)
{
  int cc = g / P;
  if (cc > c_max - 1) cc = c_max - 1;
  *c = cc;
  *i = g - cc * P;
}

// support points of the trilinear cells: the map x(xi) = sum_c L_c(xi) v_c (the weights of pmg_geo_point) at the degree-P
// Gauss-Lobatto points s = t.a; one CTA row per stored (z, y) dof line, threads along x
template <int P>
__global__ void k_geo_support(const __grid_constant__ GeoTables t, int nx, int ny, int Nx, int Ny, int z0, int nzl, int cz_min,
                              int cz_max, const double *__restrict__ vert, double *X, double *Y, double *Z)
{
  const double *s = t.a;
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    int cy, iy, cz, iz;
    support_cell(row % Ny, P, ny, &cy, &iy);
    support_cell(z0 + row / Ny, P, cz_max, &cz, &iz);
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      int cx, ix;
      support_cell(gx, P, nx, &cx, &ix);
      double v[8][3];
      geo_load_cell(vert, nx, ny, cx, cy, cz - cz_min, v);
      const double L[2][3] = {{1.0 - s[ix], 1.0 - s[iy], 1.0 - s[iz]}, {s[ix], s[iy], s[iz]}};
      double x[3] = {0.0, 0.0, 0.0};
      for (int c = 0; c < 8; ++c) {
        const double w = L[c & 1][0] * L[c >> 1 & 1][1] * L[c >> 2][2];
        for (int d = 0; d < 3; ++d) x[d] += w * v[c][d];
      }
      const int64_t o = (int64_t)row * Nx + gx;
      X[o] = x[0];
      Y[o] = x[1];
      Z[o] = x[2];
    }
  }
}

// as k_geo_support for curved cells: the degree-k map (pmg_curved_map) with the tables t at the degree-P Gauss-Lobatto points
template <int P>
__global__ void k_curved_support(const __grid_constant__ CurvedTables t, int k, int nx, int ny, int Nx, int Ny, int z0, int nzl,
                                 int cz_min, int cz_max, const double *__restrict__ nodes, double *X, double *Y, double *Z)
{
  const int k1 = k + 1;
  const int64_t sy = (int64_t)nx * k + 1, sz = sy * ((int64_t)ny * k + 1);
  for (int row = blockIdx.x; row < Ny * nzl; row += gridDim.x) {
    int cy, iy, cz, iz;
    support_cell(row % Ny, P, ny, &cy, &iy);
    support_cell(z0 + row / Ny, P, cz_max, &cz, &iz);
    for (int gx = threadIdx.x; gx < Nx; gx += blockDim.x) {
      int cx, ix;
      support_cell(gx, P, nx, &cx, &ix);
      double x[3], J[3][3];
      pmg_curved_map(curved_cell_node(nodes, nx, ny, k, cx, cy, cz - cz_min), sy, sz, k, t.L + ix * k1, t.dL + ix * k1,
                     t.L + iy * k1, t.dL + iy * k1, t.L + iz * k1, t.dL + iz * k1, x, J);
      const int64_t o = (int64_t)row * Nx + gx;
      X[o] = x[0];
      Y[o] = x[1];
      Z[o] = x[2];
    }
  }
}

template <int P>
int geo_support_points(const pmgk_level *lv, int k, const double *vert, double *x, double *y, double *z, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  if (lv->nzl <= 0) return 0;
  double gll[N1];
  pmg_fe_gll(N1, gll);
  int64_t rows = (int64_t)lv->Ny * lv->nzl;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  if (k == 1) {
    GeoTables t;
    for (int i = 0; i < N1; ++i) t.a[i] = gll[i];
    k_geo_support<P><<<(unsigned)rows, pmg_var_row_threads(lv->Nx), 0, s>>>(t, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->z0, lv->nzl,
                                                                          lv->coef_cz0, lv->cz_hi, vert, x, y, z);
  } else {
    CurvedTables t;
    double unused_w[N1] = {};
    curved_tables(k, N1, gll, unused_w, t);
    k_curved_support<P><<<(unsigned)rows, pmg_var_row_threads(lv->Nx), 0, s>>>(t, k, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->z0, lv->nzl,
                                                                             lv->coef_cz0, lv->cz_hi, vert, x, y, z);
  }
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

// ---- coefficient from the caller: quadrature points, G_q scaled by a_q ------------------------------------------------
// the mapped Gauss points of the trilinear cells (the weights of pmg_geo_point), on the quadrature-point grid of the stored
// cell layers; one CTA row per (q-plane, q-row), threads along x.  Each point is computed from its own cell only, so a
// point of the layer two ranks store has the same bits on both.
template <int P>
__global__ void k_geo_qpoints(const __grid_constant__ GeoTables t, int nx, int ny, int nqz, const double *__restrict__ vert, double *X,
                              double *Y, double *Z)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1, Qy = ny * N1;
  const double *s = t.a;
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, lqz = row / Qy;
    const int cy = qy / N1, b = qy % N1, lcz = lqz / N1, m = lqz % N1;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) {
      const int cx = qx / N1, a = qx % N1;
      double v[8][3];
      geo_load_cell(vert, nx, ny, cx, cy, lcz, v);
      const double L[2][3] = {{1.0 - s[a], 1.0 - s[b], 1.0 - s[m]}, {s[a], s[b], s[m]}};
      double x[3] = {0.0, 0.0, 0.0};
      for (int c = 0; c < 8; ++c) {
        const double w = L[c & 1][0] * L[c >> 1 & 1][1] * L[c >> 2][2];
        for (int d = 0; d < 3; ++d) x[d] += w * v[c][d];
      }
      const int64_t o = (int64_t)row * Qx + qx;
      X[o] = x[0];
      Y[o] = x[1];
      Z[o] = x[2];
    }
  }
}

// as k_geo_qpoints for curved cells: the degree-k map (pmg_curved_map) with the tables t at the Gauss points
template <int P>
__global__ void k_curved_qpoints(const __grid_constant__ CurvedTables t, int k, int nx, int ny, int nqz, const double *__restrict__ nodes,
                                 double *X, double *Y, double *Z)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1, Qy = ny * N1, k1 = k + 1;
  const int64_t sy = (int64_t)nx * k + 1, sz = sy * ((int64_t)ny * k + 1);
  for (int row = blockIdx.x; row < Qy * nqz; row += gridDim.x) {
    const int qy = row % Qy, lqz = row / Qy;
    const int cy = qy / N1, b = qy % N1, lcz = lqz / N1, m = lqz % N1;
    for (int qx = threadIdx.x; qx < Qx; qx += blockDim.x) {
      const int cx = qx / N1, a = qx % N1;
      double x[3], J[3][3];
      pmg_curved_map(curved_cell_node(nodes, nx, ny, k, cx, cy, lcz), sy, sz, k, t.L + a * k1, t.dL + a * k1, t.L + b * k1,
                     t.dL + b * k1, t.L + m * k1, t.dL + m * k1, x, J);
      const int64_t o = (int64_t)row * Qx + qx;
      X[o] = x[0];
      Y[o] = x[1];
      Z[o] = x[2];
    }
  }
}

// G_q *= a_q, the six grids of the stored cell layers (a: one grid of that layout)
__global__ void k_geo_scale_coef(const double *__restrict__ a, int64_t n, int64_t gstride, double *geo)
{
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double ai = a[i];
    for (int e = 0; e < 6; ++e) geo[i + e * gstride] *= ai;
  }
}

template <int P>
int geo_quadrature_points(const pmgk_level *lv, int k, const double *vert, const double *gq, double *x, double *y, double *z,
                          cudaStream_t s)
{
  constexpr int N1 = P + 1;
  const int Qx = lv->nx * N1, Qy = lv->ny * N1, nqz = (lv->cz_hi - lv->coef_cz0) * N1;
  if (nqz <= 0) return 0;
  int64_t rows = (int64_t)Qy * nqz;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  if (k == 1) {
    GeoTables t;
    for (int i = 0; i < N1; ++i) t.a[i] = gq[i];
    k_geo_qpoints<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, lv->nx, lv->ny, nqz, vert, x, y, z);
  } else {
    CurvedTables t;
    double unused_w[N1] = {};
    curved_tables(k, N1, gq, unused_w, t);
    k_curved_qpoints<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, k, lv->nx, lv->ny, nqz, vert, x, y, z);
  }
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

template <int P>
int fill_geo(const pmgk_level *lv, int k, int c5, const double *vert, const double *gq, const double *gw, double *geo,
             unsigned long long *err, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  const int Qx = lv->nx * N1, Qy = lv->ny * N1, nqz = (lv->cz_hi - lv->coef_cz0) * N1;
  if (nqz <= 0) return 0;
  int64_t rows = (int64_t)Qy * nqz;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  if (k == 1) {
    GeoTables t;
    for (int i = 0; i < N1; ++i) { t.a[i] = gq[i]; t.b[i] = gw[i]; }
    k_geo_fill<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, lv->nx, lv->ny, lv->coef_cz0, nqz, c5, vert, lv->geo_stride, geo, err);
  } else {
    CurvedTables t;
    curved_tables(k, N1, gq, gw, t);
    k_curved_fill<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, k, lv->nx, lv->ny, lv->coef_cz0, nqz, c5, vert,
                                                                       lv->geo_stride, geo, err);
  }
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

template <int P>
int fill_geo_dinv(const pmgk_level *lv, const double *S2, const double *G2, const double *SG, double *dinv, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  GeoTables t;
  for (int i = 0; i < N1 * N1; ++i) { t.a[i] = S2[i]; t.b[i] = G2[i]; t.c[i] = SG[i]; }
  if (lv->nzl <= 0) return 0;
  int64_t rows = (int64_t)lv->Ny * lv->nzl;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  if (rows > cap) rows = cap;
  k_geo_dinv<P><<<(unsigned)rows, pmg_var_row_threads(lv->Nx), 0, s>>>(t, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->Nz, lv->z0, lv->nzl,
                                                                  lv->coef_cz0, lv->cz_hi, lv->faces, lv->coef, lv->geo_stride, dinv);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

// f: NULL = the load vector of f = 1; else the dof values of f_h (k_geo_mul_f between the w |det J| grid and the gather)
template <int P>
int geo_rhs(const pmgk_level *lv, int k, const double *vert, const double *S, const double *gq, const double *gw, const double *f,
            double *W, double *rhs, cudaStream_t s)
{
  constexpr int N1 = P + 1;
  GeoTables t;
  for (int i = 0; i < N1; ++i) { t.a[i] = gq[i]; t.b[i] = gw[i]; }
  const int Qx = lv->nx * N1, Qy = lv->ny * N1, nqz = (lv->cz_hi - lv->coef_cz0) * N1;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 32;
  int64_t rows = (int64_t)Qy * nqz;
  if (rows > cap) rows = cap;
  if (rows > 0) {
    if (k == 1) {
      k_geo_jxw<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(t, lv->nx, lv->ny, nqz, vert, W);
    } else {
      CurvedTables ct;
      curved_tables(k, N1, gq, gw, ct);
      k_curved_jxw<P><<<(unsigned)rows, pmg_var_row_threads(Qx), 0, s>>>(ct, k, lv->nx, lv->ny, nqz, vert, W);
    }
    PMG_CUDA_CHECK(cudaGetLastError());
    pmg_count_launch(1);
  }
  for (int i = 0; i < N1 * N1; ++i) t.a[i] = S[i];
  const int64_t ncells = (int64_t)lv->nx * lv->ny * (lv->cz_hi - lv->coef_cz0);
  if (f && ncells > 0) {
    int64_t blocks = (ncells + 127) / 128;
    const int64_t bcap = (int64_t)pmgk_device_sm_count() * 16;
    if (blocks > bcap) blocks = bcap;
    k_geo_mul_f<P><<<(unsigned)blocks, 128, 0, s>>>(t, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->z0, lv->coef_cz0, lv->cz_hi, f, W);
    PMG_CUDA_CHECK(cudaGetLastError());
    pmg_count_launch(1);
  }
  rows = (int64_t)lv->Ny * lv->nzl;
  if (rows > cap) rows = cap;
  if (rows <= 0) return 0;
  k_geo_rhs<P><<<(unsigned)rows, pmg_var_row_threads(lv->Nx), 0, s>>>(t, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->Nz, lv->z0, lv->nzl,
                                                                 lv->coef_cz0, lv->cz_hi, lv->faces, W, rhs);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

template <int P>
int geo_norm_cells(const pmgk_level *lv, int k, const double *vert, const double *E, const double *gq, const double *gw,
                   const double *u, double *cell_sums, cudaStream_t s)
{
  constexpr int N1 = P + 1, M = P + 2;
  const int64_t ncells = (int64_t)lv->nx * lv->ny * (lv->cz_hi - lv->cz_lo);
  if (ncells <= 0) return 0;
  int64_t blocks = (ncells + 127) / 128;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (k == 1) {
    GeoTables t;
    for (int i = 0; i < M * N1; ++i) t.a[i] = E[i];
    for (int i = 0; i < M; ++i) { t.b[i] = gq[i]; t.c[i] = gw[i]; }
    k_geo_norm_cells<P><<<(unsigned)blocks, 128, 0, s>>>(t, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->z0, lv->cz_lo, lv->cz_hi,
                                                         lv->coef_cz0, vert, u, cell_sums);
  } else {
    CurvedTables t;
    curved_tables(k, M, gq, gw, t);
    for (int i = 0; i < M * N1; ++i) t.E[i] = E[i];
    k_curved_norm_cells<P><<<(unsigned)blocks, 128, 0, s>>>(t, k, lv->nx, lv->ny, lv->Nx, lv->Ny, lv->z0, lv->cz_lo, lv->cz_hi,
                                                            lv->coef_cz0, vert, u, cell_sums);
  }
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

} // namespace

extern "C" int pmgk_geo_rhs(const pmgk_level *lv, int k, const double *vert, const double *S, const double *gq, const double *gw,
                            double *W, double *rhs, void *stream)
{
  if (!lv || !vert || !S || !gq || !gw || !W || !rhs) return PMG_ERR_ARG;
  if (k < 1 || k >= PMGK_MAX_N1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return geo_rhs<P>(lv, k, vert, S, gq, gw, NULL, W, rhs, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_rhs_f(const pmgk_level *lv, int k, const double *vert, const double *S, const double *gq, const double *gw,
                              const double *f, double *W, double *rhs, void *stream)
{
  if (!lv || !vert || !S || !gq || !gw || !f || !W || !rhs) return PMG_ERR_ARG;
  if (k < 1 || k >= PMGK_MAX_N1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return geo_rhs<P>(lv, k, vert, S, gq, gw, f, W, rhs, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_support_points(const pmgk_level *lv, int k, const double *vert, double *x, double *y, double *z, void *stream)
{
  if (!lv || !vert || !x || !y || !z) return PMG_ERR_ARG;
  if (k < 1 || k >= PMGK_MAX_N1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return geo_support_points<P>(lv, k, vert, x, y, z, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_norm_cells(const pmgk_level *lv, int k, const double *vert, const double *E, const double *gq,
                                   const double *gw, const double *u, double *cell_sums, void *stream)
{
  if (!lv || !vert || !E || !gq || !gw || !u || !cell_sums) return PMG_ERR_ARG;
  if (k < 1 || k >= PMGK_MAX_N1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return geo_norm_cells<P>(lv, k, vert, E, gq, gw, u, cell_sums, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

// called by pmgk_apply (pmg_apply.cu) for levels with mapped geometry
int pmg_geo_dispatch(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out,
                     double f1, double f2, cudaStream_t s, int *geom)
{
  if (lv->nz < 1 || lv->cz_hi <= lv->cz_lo || !lv->coef || lv->geo_stride <= 0) return PMG_ERR_ARG;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return launch_geo<P, BX, BY, MINB>(lv, mode, u, b, xold, out, f1, f2, s, geom);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_fill(const pmgk_level *lv, int k, int kind, const double *vert, const double *gq, const double *gw,
                             double *geo, unsigned long long *err, void *stream)
{
  if (!lv || !vert || !gq || !gw || !geo || !err || lv->geo_stride != pmgk_var_coef_doubles(lv)) return PMG_ERR_ARG;
  if ((kind != 0 && kind != 1) || k < 1 || k >= PMGK_MAX_N1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return fill_geo<P>(lv, k, kind, vert, gq, gw, geo, err, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_fill_dinv(const pmgk_level *lv, const double *S2, const double *G2, const double *SG, double *dinv, void *stream)
{
  if (!lv || !S2 || !G2 || !SG || !dinv || !lv->coef || lv->geo_stride <= 0) return PMG_ERR_ARG;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return fill_geo_dinv<P>(lv, S2, G2, SG, dinv, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_quadrature_points(const pmgk_level *lv, int k, const double *vert, const double *gq, double *x, double *y,
                                          double *z, void *stream)
{
  if (!lv || !vert || !gq || !x || !y || !z) return PMG_ERR_ARG;
  if (k < 1 || k >= PMGK_MAX_N1) return PMG_ERR_UNSUPPORTED;
  switch (lv->degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) \
  case P: return geo_quadrature_points<P>(lv, k, vert, gq, x, y, z, (cudaStream_t)stream);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_geo_scale_coef(const pmgk_level *lv, const double *a, double *geo, void *stream)
{
  if (!lv || !a || !geo || lv->geo_stride != pmgk_var_coef_doubles(lv)) return PMG_ERR_ARG;
  const int64_t n = lv->geo_stride;
  if (n == 0) return 0;
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)pmgk_device_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  k_geo_scale_coef<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, n, lv->geo_stride, geo);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}
