// pmg_dim2_var.h -- the 2-D operator with a coefficient, -div(a grad u) on the box square, a given at the QGauss(p+1)
// points of every cell (pmg_laplace_operator_set_coefficient).  With a coefficient the cell matrix no longer factorises
// into cx K (x) M + cy M (x) K (csrc/pmg_dim2.h), so the apply runs the quadrature-point form of the 3-D
// variable-coefficient kernel (csrc/pmg_apply_var.h) in two passes, sized for levels that live in L2 and are bound by
// launch latency (the polynomial driver's <= (7 * 64 + 1)^2 DoFs):
//   pass 1, one thread per (cell, Gauss row b):  Ub_i = sum_j S(b,j) u_ij,  Vb_i = sum_j G(b,j) u_ij  (Dirichlet u read
//           as 0);  at the row's points  fx_a = cx W_ab sum_i G(a,i) Ub_i,  fy_a = cy W_ab sum_i S(a,i) Vb_i  (W = w_q a_q);
//           then the transposed x-contraction  Rx(ix, b) = sum_a G(a,ix) fx_a,  Ry(ix, b) = sum_a S(a,ix) fy_a,  stored on
//           the quadrature-point grid layout (cell-local column ix instead of Gauss point a);
//   pass 2, one thread per DoF:  (A u)_i = sum over the <= 2 x 2 cells of  sum_b S(b,iy) Rx(ix,b) + G(b,iy) Ry(ix,b),
//           Dirichlet rows identity, then the fused epilogue of pmg2_apply_dof.
// Every output is written by one thread: deterministic, no atomics.  S(q,i) = phi_i(x_q), G(q,i) = phi_i'(x_q) on [0,1]
// (host/pmg_fe.c pmg_fe_shape_tables), cx = hy / hx, cy = hx / hy.
// PMG_HD functions: the kernels of csrc/pmg_dim2_var.cu call them per thread, tests/emu calls them in a loop.
#pragma once
#include "pmg_dim2.h"

struct Pmg2VarLevel {
  int p, nx, ny, Nx, Ny;
  unsigned faces;                                                 // Dirichlet faces bitmask, bits 0..3
  double S[PMG2_MAX_N1 * PMG2_MAX_N1], G[PMG2_MAX_N1 * PMG2_MAX_N1]; // [q][i], (p+1)^2
  double cx, cy;                                                  // hy / hx, hx / hy
};

// host: the level's tables from the quadrature-point tables of host/pmg_fe.c (Sq, Dco, [q][i], n1 x n1): S = Sq and
// G = Dco Sq, the gradient of the nodal basis at the Gauss points as the 3-D kernel forms it (collocation derivative)
inline void pmg2v_level_init(Pmg2VarLevel &l, int p, int nx, int ny, unsigned faces, const double *h, const double *Sq, const double *Dco)
{
  const int n1 = p + 1;
  l.p = p; l.nx = nx; l.ny = ny; l.Nx = nx * p + 1; l.Ny = ny * p + 1; l.faces = faces & 0xFu;
  for (int q = 0; q < n1; ++q)
    for (int i = 0; i < n1; ++i) {
      double g = 0.0;
      for (int r = 0; r < n1; ++r) g += Dco[q * n1 + r] * Sq[r * n1 + i];
      l.S[q * n1 + i] = Sq[q * n1 + i];
      l.G[q * n1 + i] = g;
    }
  l.cx = h[1] / h[0]; l.cy = h[0] / h[1];
}

// pass 1 for cell (cx, cy), Gauss row b: W = w_q a_q on the (nx (p+1)) x (ny (p+1)) quadrature-point grid, x fastest;
// Rx / Ry: grids of the same layout
template <int P>
PMG_HD void pmg2v_row(const Pmg2VarLevel &l, const double *u, const double *W, double *Rx, double *Ry, int cx, int cy, int b)
{
  constexpr int N1 = P + 1;
  double U[N1], V[N1];
  for (int i = 0; i < N1; ++i) { U[i] = 0.0; V[i] = 0.0; }
  for (int j = 0; j < N1; ++j) {
    const int y = cy * P + j;
    if ((y == 0 && (l.faces >> 2 & 1u)) || (y == l.Ny - 1 && (l.faces >> 3 & 1u))) continue;
    const double s = l.S[b * N1 + j], g = l.G[b * N1 + j];
    const double *row = u + (int64_t)y * l.Nx + cx * P;
    for (int i = 0; i < N1; ++i) {
      const int x = cx * P + i;
      const double v = ((x == 0 && (l.faces & 1u)) || (x == l.Nx - 1 && (l.faces >> 1 & 1u))) ? 0.0 : row[i];
      U[i] += s * v;
      V[i] += g * v;
    }
  }
  const int64_t Qx = (int64_t)l.nx * N1, o = (int64_t)(cy * N1 + b) * Qx + cx * N1;
  double fx[N1], fy[N1];
  for (int a = 0; a < N1; ++a) {
    double gx = 0.0, gy = 0.0;
    for (int i = 0; i < N1; ++i) { gx += l.G[a * N1 + i] * U[i]; gy += l.S[a * N1 + i] * V[i]; }
    const double w = W[o + a];
    fx[a] = l.cx * w * gx;
    fy[a] = l.cy * w * gy;
  }
  for (int i = 0; i < N1; ++i) {
    double rx = 0.0, ry = 0.0;
    for (int a = 0; a < N1; ++a) { rx += l.G[a * N1 + i] * fx[a]; ry += l.S[a * N1 + i] * fy[a]; }
    Rx[o + i] = rx;
    Ry[o + i] = ry;
  }
}

// pass 2: (A u)(gx, gy) without the Dirichlet identity, from the grids of pass 1
template <int P>
PMG_HD double pmg2v_gather(const Pmg2VarLevel &l, const double *Rx, const double *Ry, int gx, int gy)
{
  constexpr int N1 = P + 1;
  const int64_t Qx = (int64_t)l.nx * N1;
  double acc = 0.0;
  for (int ey = 0; ey < 2; ++ey) {
    const int cy = gy / P - ey, iy = gy - cy * P;
    if (cy < 0 || cy >= l.ny || iy > P) continue;
    for (int ex = 0; ex < 2; ++ex) {
      const int cx = gx / P - ex, ix = gx - cx * P;
      if (cx < 0 || cx >= l.nx || ix > P) continue;
      const int64_t o = (int64_t)(cy * N1) * Qx + cx * N1 + ix;
      double s = 0.0;
      for (int b = 0; b < N1; ++b) s += l.S[b * N1 + iy] * Rx[o + b * Qx] + l.G[b * N1 + iy] * Ry[o + b * Qx];
      acc += s;
    }
  }
  return acc;
}

// pass 2 with the fused epilogue, the modes of pmg2_apply_dof; the inverse diagonal is the explicit vector dinv_vec
template <int P>
PMG_HD double pmg2v_apply_dof(const Pmg2VarLevel &l, int mode, const double *u, const double *Rx, const double *Ry, const double *b,
                              const double *xold, double f1, double f2, const double *dinv_vec, int gx, int gy)
{
  const int64_t g = (int64_t)gy * l.Nx + gx;
  const bool dir = pmg2_dirichlet(gx, gy, l.Nx, l.Ny, l.faces);
  const double uc = u[g];
  const double Au = dir ? uc : pmg2v_gather<P>(l, Rx, Ry, gx, gy);
  if (mode == 0) return Au;
  const double r = b[g] - Au;
  if (mode == 1) return r;
  const double corr = f2 * (dir ? 1.0 : dinv_vec[g]) * r;
  if (mode == 2) return uc + corr;
  return uc + f1 * (uc - (xold ? xold[g] : 0.0)) + corr;
}

// diagonal entry of DoF (gx, gy) (constrained DoFs are the caller's): sum over the <= 2 x 2 cells of
//   sum_q W_q [cx G(a,ix)^2 S(b,iy)^2 + cy S(a,ix)^2 G(b,iy)^2]
template <int P>
PMG_HD double pmg2v_diag_entry(const Pmg2VarLevel &l, const double *W, int gx, int gy)
{
  constexpr int N1 = P + 1;
  const int64_t Qx = (int64_t)l.nx * N1;
  double diag = 0.0;
  for (int ey = 0; ey < 2; ++ey) {
    const int cy = gy / P - ey, iy = gy - cy * P;
    if (cy < 0 || cy >= l.ny || iy > P) continue;
    for (int ex = 0; ex < 2; ++ex) {
      const int cx = gx / P - ex, ix = gx - cx * P;
      if (cx < 0 || cx >= l.nx || ix > P) continue;
      for (int b = 0; b < N1; ++b) {
        const double sy = l.S[b * N1 + iy] * l.S[b * N1 + iy], dy = l.G[b * N1 + iy] * l.G[b * N1 + iy];
        const double *row = W + (int64_t)(cy * N1 + b) * Qx + cx * N1;
        double s = 0.0;
        for (int a = 0; a < N1; ++a) {
          const double sx = l.S[a * N1 + ix] * l.S[a * N1 + ix], dx = l.G[a * N1 + ix] * l.G[a * N1 + ix];
          s += row[a] * (l.cx * dx * sy + l.cy * sx * dy);
        }
        diag += s;
      }
    }
  }
  return diag;
}
