// pmg_apply_var.h -- variable-coefficient cell-loop apply  -div(a grad u), fused with the smoother update.
//
// BASELINE.json configs[4] ("3D variable-coefficient Poisson Q5").  The reference has no coefficient: its
// quadrature-point operation is  g <- JxW J^-1 J^-T g  (include/operators/portable_laplace_operator.h:301-325);
// the extension multiplies a(x_q) into JxW (SURVEY.md 8d), which is what the oracle does (oracle/mesh.c).
// With a coefficient the cell matrix no longer factorises, so this kernel keeps the reference's
// quadrature-point formulation (:267-357): interpolate nodal -> Gauss points (3 sweeps with the shape values S),
// collocation derivative per direction (D = co_shape_gradients), scale by  c_d w_q a(x_q),  transposed derivative,
// transposed interpolation -- 12 one-dimensional sweeps per cell.
//
// It is the cell-tile program of pmg_apply_tile.h (owner-computes tile of BX x BY cell columns marching in z, low-side
// halo cells recomputed, no atomics, no zeroing pass, fused epilogue) with another middle part; the load / x- and
// z-interpolation phase, the back-transformation, the carried z-plane and the epilogue ARE that file's functions, called
// with S = shape values instead of the pencil's eigenvectors.  Per cell layer:
//   F   thread (cell, j):  load the y-row's (x, z) slab, interpolate along x and z              -> T1
//   Y1  thread (cell, a):  per m: interpolate along y: U(a, ., m) (in place in T1);  Gy = D U   -> T2
//   XZ  thread (cell, b):  U(., b, .) and the coefficient row in registers:
//                          R = Dx^T (cx w a) Dx U + Dz^T (cz w a) Dz U  (in place in T1);  T2 *= cy w a
//   Y2  thread (cell, a):  per m: R += Dy^T T2; transposed interpolation along y (in place in T1)
//   B   thread (cell, j):  transposed interpolation along z and x -> cell-local output planes O (aliasing T2)
//   E   owned dof columns: sum of the <= 4 cell contributions per plane + epilogue + coalesced store
// The coefficient is streamed from HBM: one double  w_q a(x_q)  per quadrature point, stored as the lexicographic grid of
// all quadrature points ((nx N1) x (ny N1) x (layers N1), x fastest) so that the lanes of a warp -- consecutive cells in
// x -- read consecutive words: 8 (p+1)^3 / p^3 B/DoF on top of the 16 B/DoF of the vectors (SURVEY.md 8d).
//
// Written against the same executor as the other tile programs: runs under tests/emu on the CPU test-suite.
#pragma once
#include <math.h>
#include <type_traits>
#include "pmg_apply_tile.h"

template <int P>
struct PmgVarParams : PmgApplyParams<P> {
  // PmgApplyParams::S holds the shape values S[q][i] = phi_i(x_q) (row = Gauss point, column = nodal index)
  double D[(P + 1) * (P + 1)]; // co_shape_gradients D[q][r]: derivative of the Gauss-point Lagrange basis r at Gauss point q
  const double *coef;          // w_q a(x_q) on the lexicographic quadrature-point grid, cell layers from coef_cz0 on
  int coef_cz0;                // first cell layer stored in coef
};

// mapped geometry (PmgVarTile<.., GEO = true>): coef holds six quadrature-point grids, one per entry of the symmetric
// G_q = w_q a(x(xi_q)) |det J_q| J_q^-1 J_q^-T  in the order xx, xy, xz, yy, yz, zz, grid k at coef + k * gstride
template <int P>
struct PmgGeoParams : PmgVarParams<P> {
  int64_t gstride;
};

// the C5 coefficient a(x) = 1 / (0.05 + 2 |x|^2) (oracle/mesh.c: orc_coef_c5) times the quadrature weight, at
// quadrature point (qx, qy, qz) of the global quadrature-point grid (N1 points per cell and direction)
template <int P>
PMG_HD double pmg_var_coef_c5(int qx, int qy, int qz, const double *gq, const double *gw, const double *h)
{
  constexpr int N1 = P + 1;
  const double x = ((qx / N1) + gq[qx % N1]) * h[0], y = ((qy / N1) + gq[qy % N1]) * h[1], z = ((qz / N1) + gq[qz % N1]) * h[2];
  return gw[qx % N1] * gw[qy % N1] * gw[qz % N1] * (1.0 / (0.05 + 2.0 * (x * x + y * y + z * z)));
}

// diagonal entry of dof (gx, gy, gz): sum over the <= 8 cells that contain it of
//   sum_q w_q a_q [ cx G(qx,ix)^2 S(qy,iy)^2 S(qz,iz)^2 + cy S^2 G^2 S^2 + cz S^2 S^2 G^2 ]
// (= e_i^T A e_i of the unmasked cell operator, which is what LaplaceDiagonalOperator :104-209 computes);
// S2 / G2: squared shape values / nodal shape gradients at the Gauss points, [q][i]; cell layers [cz_min, cz_max).
template <int P>
PMG_HD double pmg_var_diag_entry(int gx, int gy, int gz, int nx, int ny, int cz_min, int cz_max, const double *S2,
                                 const double *G2, const double *c, const double *coef, int coef_cz0)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1;
  const int64_t Qplane = (int64_t)Qx * (ny * N1);
  double diag = 0.0;
  // cells along each direction: dof g = cell * P + i; a vertex dof belongs to two cells
  for (int ez = 0; ez < 2; ++ez) {
    const int cz = gz / P - ez, iz = gz - cz * P;
    if (cz < cz_min || cz >= cz_max || iz > P) continue;
    for (int ey = 0; ey < 2; ++ey) {
      const int cy = gy / P - ey, iy = gy - cy * P;
      if (cy < 0 || cy >= ny || iy > P) continue;
      for (int ex = 0; ex < 2; ++ex) {
        const int cx = gx / P - ex, ix = gx - cx * P;
        if (cx < 0 || cx >= nx || ix > P) continue;
        const double *cw = coef + (int64_t)(cz - coef_cz0) * N1 * Qplane + (int64_t)(cy * N1) * Qx + cx * N1;
        for (int m = 0; m < N1; ++m) {
          const double sz = S2[m * N1 + iz], dz = G2[m * N1 + iz];
          for (int b = 0; b < N1; ++b) {
            const double sy = S2[b * N1 + iy], dy = G2[b * N1 + iy];
            const double *row = cw + m * Qplane + (int64_t)b * Qx;
            const double f0 = c[0] * sy * sz, f12 = c[1] * dy * sz + c[2] * sy * dz;
            double s = 0.0;
            for (int a = 0; a < N1; ++a) s += row[a] * (G2[a * N1 + ix] * f0 + S2[a * N1 + ix] * f12);
            diag += s;
          }
        }
      }
    }
  }
  return diag;
}

// diagonal entry of the mapped operator: sum over the <= 8 cells that contain dof (gx, gy, gz) of
//   sum_q sum_{d,e} G_de(q) d_d phi_i(q) d_e phi_i(q),   d_x phi_i = G(qx,ix) S(qy,iy) S(qz,iz) etc.;
// S2 / G2 as above, SG[q][i] = S(q,i) G(q,i) for the cross terms; geo: the six grids of PmgGeoParams, gstride apart
template <int P>
PMG_HD double pmg_geo_diag_entry(int gx, int gy, int gz, int nx, int ny, int cz_min, int cz_max, const double *S2,
                                 const double *G2, const double *SG, const double *geo, int64_t gstride, int coef_cz0)
{
  constexpr int N1 = P + 1;
  const int Qx = nx * N1;
  const int64_t Qplane = (int64_t)Qx * (ny * N1);
  double diag = 0.0;
  for (int ez = 0; ez < 2; ++ez) {
    const int cz = gz / P - ez, iz = gz - cz * P;
    if (cz < cz_min || cz >= cz_max || iz > P) continue;
    for (int ey = 0; ey < 2; ++ey) {
      const int cy = gy / P - ey, iy = gy - cy * P;
      if (cy < 0 || cy >= ny || iy > P) continue;
      for (int ex = 0; ex < 2; ++ex) {
        const int cx = gx / P - ex, ix = gx - cx * P;
        if (cx < 0 || cx >= nx || ix > P) continue;
        const double *cw = geo + (int64_t)(cz - coef_cz0) * N1 * Qplane + (int64_t)(cy * N1) * Qx + cx * N1;
        for (int m = 0; m < N1; ++m) {
          const double sz = S2[m * N1 + iz], dz = G2[m * N1 + iz], xz = SG[m * N1 + iz];
          for (int b = 0; b < N1; ++b) {
            const double sy = S2[b * N1 + iy], dy = G2[b * N1 + iy], xy = SG[b * N1 + iy];
            const double *row = cw + m * Qplane + (int64_t)b * Qx;
            double s = 0.0;
            for (int a = 0; a < N1; ++a) {
              const double sx = S2[a * N1 + ix], dx = G2[a * N1 + ix], xx = SG[a * N1 + ix];
              s += row[a] * dx * sy * sz + row[3 * gstride + a] * sx * dy * sz + row[5 * gstride + a] * sx * sy * dz +
                   2.0 * (row[gstride + a] * xx * xy * sz + row[2 * gstride + a] * xx * sy * xz + row[4 * gstride + a] * sx * xy * xz);
            }
            diag += s;
          }
        }
      }
    }
  }
  return diag;
}

// G_q of one quadrature point from the map's Jacobian J (J[d][e] = d x_d / d xi_e) and the mapped point x; wq = quadrature
// weight.  Writes the six entries (xx, xy, xz, yy, yz, zz) of  wq a(x) |det J| J^-1 J^-T  (a = C5 coefficient at x when
// c5 != 0, else 1) and returns det J (<= 0 or NaN: the cell is inverted or degenerate).  The one copy of this arithmetic:
// the trilinear (pmg_geo_point) and the curved (pmg_curved_point) set-up both end here.
PMG_HD double pmg_geo_tensor(const double (*J)[3], const double *x, double wq, int c5, double *G)
{
  // adjugate: J^-1 = adj(J) / det
  const double A00 = J[1][1] * J[2][2] - J[1][2] * J[2][1], A01 = J[0][2] * J[2][1] - J[0][1] * J[2][2], A02 = J[0][1] * J[1][2] - J[0][2] * J[1][1];
  const double A10 = J[1][2] * J[2][0] - J[1][0] * J[2][2], A11 = J[0][0] * J[2][2] - J[0][2] * J[2][0], A12 = J[0][2] * J[1][0] - J[0][0] * J[1][2];
  const double A20 = J[1][0] * J[2][1] - J[1][1] * J[2][0], A21 = J[0][1] * J[2][0] - J[0][0] * J[2][1], A22 = J[0][0] * J[1][1] - J[0][1] * J[1][0];
  const double det = J[0][0] * A00 + J[0][1] * A10 + J[0][2] * A20;
  double f = wq / det; // w |det J| (adj/det)(adj/det)^T = w / det * adj adj^T for det > 0
  if (c5) f *= 1.0 / (0.05 + 2.0 * (x[0] * x[0] + x[1] * x[1] + x[2] * x[2]));
  G[0] = f * (A00 * A00 + A01 * A01 + A02 * A02);
  G[1] = f * (A00 * A10 + A01 * A11 + A02 * A12);
  G[2] = f * (A00 * A20 + A01 * A21 + A02 * A22);
  G[3] = f * (A10 * A10 + A11 * A11 + A12 * A12);
  G[4] = f * (A10 * A20 + A11 * A21 + A12 * A22);
  G[5] = f * (A20 * A20 + A21 * A21 + A22 * A22);
  return det;
}

// G_q of one quadrature point of the trilinear map of a cell (pmg_geo_tensor): v[c][d] = coordinate d of the cell's
// vertex c = ix + 2 iy + 4 iz; (xq, yq, zq) = the point on the reference cell [0,1]^3; wq = quadrature weight
PMG_HD double pmg_geo_point(const double (*v)[3], double xq, double yq, double zq, double wq, int c5, double *G)
{
  const double L[2][3] = {{1.0 - xq, 1.0 - yq, 1.0 - zq}, {xq, yq, zq}};
  double J[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, x[3] = {0, 0, 0}; // J[d][e] = d x_d / d xi_e
  for (int c = 0; c < 8; ++c) {
    const int i = c & 1, j = c >> 1 & 1, k = c >> 2;
    const double w = L[i][0] * L[j][1] * L[k][2];
    const double d0 = (i ? 1.0 : -1.0) * L[j][1] * L[k][2], d1 = L[i][0] * (j ? 1.0 : -1.0) * L[k][2], d2 = L[i][0] * L[j][1] * (k ? 1.0 : -1.0);
    for (int d = 0; d < 3; ++d) { x[d] += w * v[c][d]; J[d][0] += d0 * v[c][d]; J[d][1] += d1 * v[c][d]; J[d][2] += d2 * v[c][d]; }
  }
  return pmg_geo_tensor(J, x, wq, c5, G);
}

// x(xi) and J(xi) (J[d][e] = d x_d / d xi_e) of a curved cell at one reference point: the tensor-product Lagrange
// interpolant of degree k through the cell's (k+1)^3 nodes at the Gauss-Lobatto points of FE_Q(k) (MappingQ(k)), by sum
// factorisation -- contract x (values and derivatives), then y, then z.  Node (i, j, l) of the cell is at
// node + 3 (i + j sy + l sz), (x, y, z) interleaved; Lx[i] / dLx[i] = value / derivative of the 1-D basis function i at the
// point's xi_x, likewise for y and z.
PMG_HD void pmg_curved_map(const double *node, int64_t sy, int64_t sz, int k, const double *Lx, const double *dLx,
                           const double *Ly, const double *dLy, const double *Lz, const double *dLz, double *x, double (*J)[3])
{
  for (int d = 0; d < 3; ++d) { x[d] = 0.0; J[d][0] = 0.0; J[d][1] = 0.0; J[d][2] = 0.0; }
  for (int l = 0; l <= k; ++l) {
    double v[3] = {0, 0, 0}, vx[3] = {0, 0, 0}, vy[3] = {0, 0, 0}; // plane l contracted over x and y: value, d/dxi_x, d/dxi_y
    for (int j = 0; j <= k; ++j) {
      const double *row = node + 3 * (j * sy + l * sz);
      double s[3] = {0, 0, 0}, sx[3] = {0, 0, 0};
      for (int i = 0; i <= k; ++i)
        for (int d = 0; d < 3; ++d) { s[d] += Lx[i] * row[3 * i + d]; sx[d] += dLx[i] * row[3 * i + d]; }
      for (int d = 0; d < 3; ++d) { v[d] += Ly[j] * s[d]; vx[d] += Ly[j] * sx[d]; vy[d] += dLy[j] * s[d]; }
    }
    for (int d = 0; d < 3; ++d) { x[d] += Lz[l] * v[d]; J[d][0] += Lz[l] * vx[d]; J[d][1] += Lz[l] * vy[d]; J[d][2] += dLz[l] * v[d]; }
  }
}

// G_q of one quadrature point of a curved cell (pmg_curved_map, then pmg_geo_tensor); the arguments as there.  Returns
// det J, or -1 when a node of the cell is not finite (every node enters x(xi), so a non-finite node shows there).
PMG_HD double pmg_curved_point(const double *node, int64_t sy, int64_t sz, int k, const double *Lx, const double *dLx,
                               const double *Ly, const double *dLy, const double *Lz, const double *dLz, double wq, int c5,
                               double *G)
{
  double x[3], J[3][3];
  pmg_curved_map(node, sy, sz, k, Lx, dLx, Ly, dLy, Lz, dLz, x, J);
  const double det = pmg_geo_tensor(J, x, wq, c5, G);
  return isfinite(x[0] + x[1] + x[2]) && isfinite(det) ? det : -1.0;
}

// host side of the launchers (pmg_apply_var.cu, pmg_apply_geo.cu): number of z-chunks that minimises
// waves * (layers + recomputed layer below the chunk)
inline void pmg_var_choose_chunks(int tiles, int layers, int slots, int *n_chunks, int *layers_per_chunk)
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

// threads per CTA of the set-up kernels that walk one row of n points
inline int pmg_var_row_threads(int n) { return n >= 192 ? 256 : (n >= 96 ? 128 : (n >= 48 ? 64 : 32)); }

// hint: bring the line at `ptr` closer (L2, or L1 with PMG_VAR_PREFETCH_L1); the kernel's global loads are consumed right
// where they are issued, two to three barriers after the place where their addresses are known
PMG_HD void pmg_var_prefetch(const double *ptr)
{
#if defined(__CUDA_ARCH__)
#ifdef PMG_VAR_PREFETCH_L1
  asm volatile("prefetch.global.L1 [%0];\n" ::"l"(ptr));
#else
  asm volatile("prefetch.global.L2 [%0];\n" ::"l"(ptr));
#endif
#else
  (void)ptr;
#endif
}

template <int P, int BX, int BY, bool GEO = false>
struct PmgVarTile {
  using Base = PmgApplyTile<P, BX, BY>;
  using Params = std::conditional_t<GEO, PmgGeoParams<P>, PmgVarParams<P>>;
  using ThreadState = typename Base::ThreadState;
  static constexpr int N1 = Base::N1, CXC = Base::CXC, NITEM = Base::NITEM, NT = Base::NT, AP = Base::AP;
  static constexpr int T1_SIZE = Base::T1_SIZE, O_SIZE = Base::O_SIZE;
  static_assert(!Base::ALIAS, "the output planes must sit behind T1 (they share the space of T2)");
  static_assert(Base::O_OFFSET == T1_SIZE, "O aliases T2");
  static constexpr int T2_OFFSET = T1_SIZE;
  static constexpr int SMEM_DOUBLES = T1_SIZE + (T1_SIZE > O_SIZE ? T1_SIZE : O_SIZE);
  static_assert(SMEM_DOUBLES * 8 <= 227 * 1024, "tile does not fit the 227 KB of shared memory of a CTA");
  static constexpr int JSTRIDE = CXC * AP;   // distance between consecutive j (or b) of one cell in T1 / T2
  static constexpr int MSTRIDE = NITEM * AP; // distance between consecutive m

  // decode of the (cell, a) items of the y phases (as PmgApplyTile::phase_y): false = nothing to do
  static PMG_HD bool decode_y(const Params &p, int tid, int cx0, int cy0, int &a, int &tcx, int &tcy)
  {
    if (tid >= NITEM) return false;
    if (Base::Y_A_FASTEST) { a = tid % N1; tcx = (tid / N1) % CXC; tcy = tid / (N1 * CXC); }
    else { tcx = tid % CXC; a = (tid / CXC) % N1; tcy = tid / (CXC * N1); }
    const int cx = cx0 - 1 + tcx, cy = cy0 - 1 + tcy;
    return !(cx < 0 || cx >= p.nx || cy < 0 || cy >= p.ny);
  }

  // Y1: values at the quadrature points (in place) and their y derivative (-> T2)
  static PMG_HD void phase_y1(const Params &p, int tid, int cx0, int cy0, double *smem)
  {
    int a, tcx, tcy;
    if (!decode_y(p, tid, cx0, cy0, a, tcx, tcy)) return;
    double *col = smem + Base::t1_index(Base::item_index(tcx, 0, tcy), 0, a);
    double *col2 = col + T2_OFFSET;
#pragma unroll
    for (int m = 0; m < N1; ++m) {
      double T[N1], U[N1];
#pragma unroll
      for (int j = 0; j < N1; ++j) T[j] = col[j * JSTRIDE + m * MSTRIDE];
#pragma unroll
      for (int b = 0; b < N1; ++b) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < N1; ++j) s += p.S[b * N1 + j] * T[j];
        U[b] = s;
        col[b * JSTRIDE + m * MSTRIDE] = s;
      }
#pragma unroll
      for (int b = 0; b < N1; ++b) {
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < N1; ++r) s += p.D[b * N1 + r] * U[r];
        col2[b * JSTRIDE + m * MSTRIDE] = s;
      }
    }
  }

  // XZ: x and z derivative parts in registers, in place; the y derivative in T2 is scaled with its coefficient
  static PMG_HD void phase_xz(const Params &p, const ThreadState &st, double *smem, int cz)
  {
    if (!st.valid) return;
    double *t1 = smem + Base::t1_index(Base::item_index(st.tcx, st.j, st.tcy), 0, 0);
    double *t2 = t1 + T2_OFFSET;
    const int Qx = p.nx * N1;
    const int64_t Qplane = (int64_t)Qx * (p.ny * N1);
    const double *cw = p.coef + (int64_t)(cz - p.coef_cz0) * N1 * Qplane + (int64_t)(st.cy * N1 + st.j) * Qx + st.cx * N1;
#ifdef PMG_VAR_XZ_REGS
    double U[N1][N1], R[N1][N1];
#pragma unroll
    for (int m = 0; m < N1; ++m)
#pragma unroll
      for (int a = 0; a < N1; ++a) { U[m][a] = t1[m * MSTRIDE + a]; R[m][a] = 0.0; }
#pragma unroll
    for (int m = 0; m < N1; ++m) {
      double w[N1], gx[N1], gz[N1];
#pragma unroll
      for (int a = 0; a < N1; ++a) w[a] = cw[m * Qplane + a];
#pragma unroll
      for (int a = 0; a < N1; ++a) t2[m * MSTRIDE + a] *= p.c[1] * w[a];
      // derivatives at the quadrature points (a, b, m), a = 0..P
#pragma unroll
      for (int a = 0; a < N1; ++a) {
        double sx = 0.0, sz = 0.0;
#pragma unroll
        for (int r = 0; r < N1; ++r) { sx += p.D[a * N1 + r] * U[m][r]; sz += p.D[m * N1 + r] * U[r][a]; }
        gx[a] = sx * (p.c[0] * w[a]);
        gz[a] = sz * (p.c[2] * w[a]);
      }
      // transposed derivatives
#pragma unroll
      for (int r = 0; r < N1; ++r) {
        double s = R[m][r];
#pragma unroll
        for (int a = 0; a < N1; ++a) s += p.D[a * N1 + r] * gx[a];
        R[m][r] = s;
      }
#pragma unroll
      for (int r = 0; r < N1; ++r)
#pragma unroll
        for (int a = 0; a < N1; ++a) R[r][a] += p.D[m * N1 + r] * gz[a];
    }
#else
    // R stays in registers; U is read from T1 where it is needed (row m for the x derivative, all rows for the z
    // derivative): (P+1)^3 shared-memory loads per thread against 4 (P+1)^3 FMAs, and half the registers of holding both
    double R[N1][N1];
#pragma unroll
    for (int m = 0; m < N1; ++m)
#pragma unroll
      for (int a = 0; a < N1; ++a) R[m][a] = 0.0;
#pragma unroll
    for (int m = 0; m < N1; ++m) {
      double w[N1], gx[N1], gz[N1], Um[N1];
#pragma unroll
      for (int a = 0; a < N1; ++a) { w[a] = cw[m * Qplane + a]; Um[a] = t1[m * MSTRIDE + a]; gz[a] = 0.0; }
#pragma unroll
      for (int a = 0; a < N1; ++a) t2[m * MSTRIDE + a] *= p.c[1] * w[a];
      // derivatives at the quadrature points (a, b, m), a = 0..P
#pragma unroll
      for (int r = 0; r < N1; ++r) {
#pragma unroll
        for (int a = 0; a < N1; ++a) gz[a] += p.D[m * N1 + r] * t1[r * MSTRIDE + a];
      }
#pragma unroll
      for (int a = 0; a < N1; ++a) {
        double sx = 0.0;
#pragma unroll
        for (int r = 0; r < N1; ++r) sx += p.D[a * N1 + r] * Um[r];
        gx[a] = sx * (p.c[0] * w[a]);
        gz[a] *= p.c[2] * w[a];
      }
      // transposed derivatives
#pragma unroll
      for (int r = 0; r < N1; ++r) {
        double s = R[m][r];
#pragma unroll
        for (int a = 0; a < N1; ++a) s += p.D[a * N1 + r] * gx[a];
        R[m][r] = s;
      }
#pragma unroll
      for (int r = 0; r < N1; ++r)
#pragma unroll
        for (int a = 0; a < N1; ++a) R[r][a] += p.D[m * N1 + r] * gz[a];
    }
#endif
#pragma unroll
    for (int m = 0; m < N1; ++m)
#pragma unroll
      for (int a = 0; a < N1; ++a) t1[m * MSTRIDE + a] = R[m][a];
  }

  // XZ of the mapped operator: all three reference derivatives of the points (a, b, m) meet in this thread -- x and z in
  // registers, y in T2 -- so  (Gx, Gy, Gz) = G_q (gx, gy, gz)  is formed here; Gy goes back to T2 for Y2
  static PMG_HD void phase_xz_geo(const Params &p, const ThreadState &st, double *smem, int cz)
  {
    if (!st.valid) return;
    double *t1 = smem + Base::t1_index(Base::item_index(st.tcx, st.j, st.tcy), 0, 0);
    double *t2 = t1 + T2_OFFSET;
    const int Qx = p.nx * N1;
    const int64_t Qplane = (int64_t)Qx * (p.ny * N1);
    const double *cw = p.coef + (int64_t)(cz - p.coef_cz0) * N1 * Qplane + (int64_t)(st.cy * N1 + st.j) * Qx + st.cx * N1;
    double R[N1][N1];
#pragma unroll
    for (int m = 0; m < N1; ++m)
#pragma unroll
      for (int a = 0; a < N1; ++a) R[m][a] = 0.0;
#pragma unroll
    for (int m = 0; m < N1; ++m) {
      double gx[N1], gz[N1], Um[N1];
#pragma unroll
      for (int a = 0; a < N1; ++a) { Um[a] = t1[m * MSTRIDE + a]; gz[a] = 0.0; }
#pragma unroll
      for (int r = 0; r < N1; ++r) {
#pragma unroll
        for (int a = 0; a < N1; ++a) gz[a] += p.D[m * N1 + r] * t1[r * MSTRIDE + a];
      }
#pragma unroll
      for (int a = 0; a < N1; ++a) {
        double sx = 0.0;
#pragma unroll
        for (int r = 0; r < N1; ++r) sx += p.D[a * N1 + r] * Um[r];
        const double *g = cw + m * Qplane + a;
        const double gy = t2[m * MSTRIDE + a];
        const double gxx = g[0], gxy = g[p.gstride], gxz = g[2 * p.gstride];
        const double gyy = g[3 * p.gstride], gyz = g[4 * p.gstride], gzz = g[5 * p.gstride];
        const double sz = gz[a];
        gx[a] = gxx * sx + gxy * gy + gxz * sz;
        t2[m * MSTRIDE + a] = gxy * sx + gyy * gy + gyz * sz;
        gz[a] = gxz * sx + gyz * gy + gzz * sz;
      }
      // transposed derivatives
#pragma unroll
      for (int r = 0; r < N1; ++r) {
        double s = R[m][r];
#pragma unroll
        for (int a = 0; a < N1; ++a) s += p.D[a * N1 + r] * gx[a];
        R[m][r] = s;
      }
#pragma unroll
      for (int r = 0; r < N1; ++r)
#pragma unroll
        for (int a = 0; a < N1; ++a) R[r][a] += p.D[m * N1 + r] * gz[a];
    }
#pragma unroll
    for (int m = 0; m < N1; ++m)
#pragma unroll
      for (int a = 0; a < N1; ++a) t1[m * MSTRIDE + a] = R[m][a];
  }

  // Y2: add the y derivative part, then the transposed interpolation along y, in place in T1
  static PMG_HD void phase_y2(const Params &p, int tid, int cx0, int cy0, double *smem)
  {
    int a, tcx, tcy;
    if (!decode_y(p, tid, cx0, cy0, a, tcx, tcy)) return;
    double *col = smem + Base::t1_index(Base::item_index(tcx, 0, tcy), 0, a);
    const double *col2 = col + T2_OFFSET;
#pragma unroll
    for (int m = 0; m < N1; ++m) {
      double G[N1], R[N1];
#pragma unroll
      for (int b = 0; b < N1; ++b) { G[b] = col2[b * JSTRIDE + m * MSTRIDE]; R[b] = col[b * JSTRIDE + m * MSTRIDE]; }
#pragma unroll
      for (int r = 0; r < N1; ++r) {
        double s = R[r];
#pragma unroll
        for (int b = 0; b < N1; ++b) s += p.D[b * N1 + r] * G[b];
        R[r] = s;
      }
#pragma unroll
      for (int j = 0; j < N1; ++j) {
        double s = 0.0;
#pragma unroll
        for (int b = 0; b < N1; ++b) s += p.S[b * N1 + j] * R[b];
        col[j * JSTRIDE + m * MSTRIDE] = s;
      }
    }
  }

  // thread (cell, j): prefetch the coefficient rows phase XZ of layer cz will read and the u rows phase F of layer
  // cz + 1 will read (a row = P+1 consecutive doubles: one or two 32-byte sectors)
  static PMG_HD void prefetch_layer(const Params &p, const ThreadState &st, int cz, bool next_u)
  {
    if (!st.valid) return;
    const int Qx = p.nx * N1;
    const int64_t Qplane = (int64_t)Qx * (p.ny * N1);
    const double *cw = p.coef + (int64_t)(cz - p.coef_cz0) * N1 * Qplane + (int64_t)(st.cy * N1 + st.j) * Qx + st.cx * N1;
    if constexpr (GEO) {
#pragma unroll
      for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int m = 0; m < N1; ++m) {
          pmg_var_prefetch(cw + k * p.gstride + m * Qplane);
          if (N1 > 4) pmg_var_prefetch(cw + k * p.gstride + m * Qplane + P);
        }
    } else {
#pragma unroll
      for (int m = 0; m < N1; ++m) {
        pmg_var_prefetch(cw + m * Qplane);
        if (N1 > 4) pmg_var_prefetch(cw + m * Qplane + P);
      }
    }
    if (next_u) {
      const int64_t plane = (int64_t)p.Nx * p.Ny;
      const double *row = p.u + (int64_t)((cz + 1) * P - p.z0) * plane + (int64_t)(st.cy * P + st.j) * p.Nx + st.cx * P;
#pragma unroll
      for (int k = 1; k < N1; ++k) {
        pmg_var_prefetch(row + k * plane);
        if (N1 > 4) pmg_var_prefetch(row + k * plane + P);
      }
    }
  }

  template <class Exec>
  static PMG_HD void run(const Params &p, Exec &ex, double *smem, int tile_x, int tile_y, int chunk)
  {
    const int cx0 = tile_x * BX, cy0 = tile_y * BY;
    const int cz_begin = p.cz_lo + chunk * p.layers_per_chunk;
    int cz_end = cz_begin + p.layers_per_chunk;
    if (cz_end > p.cz_hi) cz_end = p.cz_hi;
    if (cz_begin >= cz_end) return;
    const bool halo = (cz_begin > 0) && ((cz_begin - 1) * P >= p.z0);
    const int cz_first = halo ? cz_begin - 1 : cz_begin;

    ex.for_each_thread([&](int tid, ThreadState &st) { Base::decode(tid, cx0, cy0, p, st); });

    for (int cz = cz_first; cz < cz_end; ++cz) {
      const bool first = (cz == cz_first);
      const bool write_out = (cz >= cz_begin);
      // T1 was last read by the previous layer's B phase, O (= T2) by its epilogue: F writes T1 only, and the barrier
      // after F orders the epilogue's reads of O before Y1's writes to T2
      ex.for_each_thread([&](int, ThreadState &st) {
#ifndef PMG_VAR_NO_PREFETCH
        prefetch_layer(p, st, cz, cz + 1 < cz_end);
#endif
        Base::phase_forward(p, st, smem, cz, first);
      });
      ex.sync();
      ex.for_each_thread([&](int tid, ThreadState &) { phase_y1(p, tid, cx0, cy0, smem); });
      ex.sync();
      if constexpr (GEO) ex.for_each_thread([&](int, ThreadState &st) { phase_xz_geo(p, st, smem, cz); });
      else ex.for_each_thread([&](int, ThreadState &st) { phase_xz(p, st, smem, cz); });
      ex.sync();
      ex.for_each_thread([&](int tid, ThreadState &) { phase_y2(p, tid, cx0, cy0, smem); });
      ex.sync();
      // T2 is dead after Y2: B reads its slab from T1 and writes the output planes O over T2
      ex.for_each_thread([&](int, ThreadState &st) { Base::phase_back_write(p, st, smem, first, write_out); });
      ex.sync();
      if (write_out)
        ex.for_each_thread([&](int tid, ThreadState &) { Base::template phase_epilogue<P>(p, tid, smem, cx0, cy0, cz * P); });
    }
    if (cz_end == p.cz_hi && cz_end * P < p.z_own_hi) {
      ex.sync();
      ex.for_each_thread([&](int, ThreadState &st) { Base::phase_flush(p, st, smem); });
      ex.sync();
      ex.for_each_thread([&](int tid, ThreadState &) { Base::template phase_epilogue<1>(p, tid, smem, cx0, cy0, cz_end * P); });
    }
  }
};
