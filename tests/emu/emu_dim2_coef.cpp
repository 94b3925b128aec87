// tests/emu/emu_dim2_coef.cpp -- host emulation of the 2-D kernels with a coefficient (TEST INFRASTRUCTURE): the PMG_HD
// functions of csrc/pmg_dim2_var.h, which the kernels of csrc/pmg_dim2_var.cu call per thread, run here in loops over the
// (cell, Gauss row) pairs and the DoFs with the tables of host/pmg_fe.c.  Built only by tests/; the product has no CPU path.
#include <cstring>
#include <vector>
#include "pmg_dim2_var.h"

extern "C" {
void pmg_fe_shape_tables(int p, double *Sq, double *Dco, double *G, double *gq, double *gw);
}

namespace {

// the level and W = w_q a_q as the set-up kernel forms it (csrc/pmg_apply_var.cu k_var_coef_caller, 2-D)
void make_level(int p, int nx, int ny, unsigned faces, const double *a, Pmg2VarLevel &l, std::vector<double> &W)
{
  const int n1 = p + 1;
  double Sq[PMG2_MAX_N1 * PMG2_MAX_N1], Dco[PMG2_MAX_N1 * PMG2_MAX_N1], gq[PMG2_MAX_N1], gw[PMG2_MAX_N1];
  pmg_fe_shape_tables(p, Sq, Dco, nullptr, gq, gw);
  const double h[3] = {1.0 / nx, 1.0 / ny, 1.0};
  pmg2v_level_init(l, p, nx, ny, faces, h, Sq, Dco);
  const int Qx = nx * n1, Qy = ny * n1;
  W.resize((size_t)Qx * Qy);
  for (int qy = 0; qy < Qy; ++qy)
    for (int qx = 0; qx < Qx; ++qx) W[(size_t)qy * Qx + qx] = gw[qx % n1] * (gw[qy % n1] * 1.0) * a[(size_t)qy * Qx + qx];
}

template <int P>
void apply(const Pmg2VarLevel &l, const std::vector<double> &W, int mode, const double *u, const double *b, const double *xold,
           double *out, double f1, double f2, const double *dinv_vec)
{
  std::vector<double> Rx(W.size()), Ry(W.size());
  for (int cy = 0; cy < l.ny; ++cy)
    for (int cx = 0; cx < l.nx; ++cx)
      for (int r = 0; r <= P; ++r) pmg2v_row<P>(l, u, W.data(), Rx.data(), Ry.data(), cx, cy, r);
  std::vector<double> res((size_t)l.Nx * l.Ny); // out may alias xold: every "thread" reads before any writes, as on the device
  for (int gy = 0; gy < l.Ny; ++gy)
    for (int gx = 0; gx < l.Nx; ++gx)
      res[(size_t)gy * l.Nx + gx] = pmg2v_apply_dof<P>(l, mode, u, Rx.data(), Ry.data(), b, xold, f1, f2, dinv_vec, gx, gy);
  std::memcpy(out, res.data(), res.size() * sizeof(double));
}

template <int P>
void dinv(const Pmg2VarLevel &l, const std::vector<double> &W, double *out)
{
  for (int gy = 0; gy < l.Ny; ++gy)
    for (int gx = 0; gx < l.Nx; ++gx)
      out[(size_t)gy * l.Nx + gx] = 1.0 / (pmg2_dirichlet(gx, gy, l.Nx, l.Ny, l.faces) ? 1.0 : pmg2v_diag_entry<P>(l, W.data(), gx, gy));
}

} // namespace

#define EMU2V_DEGREES(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9)

extern "C" {
// a: the coefficient at the (nx (p+1)) x (ny (p+1)) Gauss points, x fastest (pmg_laplace_operator_quadrature_points)
int emu2v_apply(int p, int nx, int ny, unsigned faces, const double *a, int mode, const double *u, const double *b, const double *xold,
                double *out, double f1, double f2, const double *dinv_vec)
{
  Pmg2VarLevel l;
  std::vector<double> W;
  if (p < 1 || p + 1 > PMG2_MAX_N1) return -3;
  make_level(p, nx, ny, faces, a, l, W);
  switch (p) {
#define EMU2V_CASE(P) case P: apply<P>(l, W, mode, u, b, xold, out, f1, f2, dinv_vec); return 0;
    EMU2V_DEGREES(EMU2V_CASE)
#undef EMU2V_CASE
  }
  return -3;
}

int emu2v_dinv(int p, int nx, int ny, unsigned faces, const double *a, double *out)
{
  Pmg2VarLevel l;
  std::vector<double> W;
  if (p < 1 || p + 1 > PMG2_MAX_N1) return -3;
  make_level(p, nx, ny, faces, a, l, W);
  switch (p) {
#define EMU2V_CASE(P) case P: dinv<P>(l, W, out); return 0;
    EMU2V_DEGREES(EMU2V_CASE)
#undef EMU2V_CASE
  }
  return -3;
}
}
