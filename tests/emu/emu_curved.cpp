// tests/emu/emu_curved.cpp -- host emulator of the mapped-geometry tile program on curved cells (TEST INFRASTRUCTURE).
//
// As emu_geo.cpp, with the six G grids built from the cells' degree-k nodes by pmg_curved_point, the PMG_HD routine the
// curved fill kernel of csrc/pmg_apply_geo.cu calls per quadrature point; the tile program (PmgVarTile<.., GEO = true>)
// is the unchanged K1g.  Built only by tests/; the product has no CPU path.
#include <cstring>
#include <vector>
#include "pmg_apply_var.h"
#include "pmg_kernels.h"

extern "C" void pmg_fe_shape_tables(int p, double *Sq, double *Dco, double *G, double *gq, double *gw);
extern "C" void pmg_fe_gll(int n, double *x);
extern "C" void pmg_fe_lagrange(int n, const double *nodes, double x, double *val, double *der);

namespace {

template <class Tile>
struct HostExecC {
  std::vector<typename Tile::ThreadState> st;
  template <class F> void for_each_thread(F f) { for (int t = 0; t < Tile::NT; ++t) f(t, st[t]); }
  void sync() {}
};

struct CurvedArgs {
  int nx, ny, nz; unsigned faces; int z0, nzl, cz_lo, cz_hi, z_own_lo, z_own_hi, n_chunks, c5, k;
  const double *nodes; int mode; const double *u, *b, *xold; double *out; double f1, f2; const double *dinv_vec; double *dinv_out;
};

template <int P, int BX, int BY>
int go(const CurvedArgs &a)
{
  using Tile = PmgVarTile<P, BX, BY, true>;
  constexpr int N1 = P + 1;
  PmgGeoParams<P> p;
  std::memset(&p, 0, sizeof(p));
  p.nx = a.nx; p.ny = a.ny; p.nz = a.nz;
  p.Nx = a.nx * P + 1; p.Ny = a.ny * P + 1; p.Nz = a.nz * P + 1;
  p.faces = a.faces; p.z0 = a.z0; p.nzl = a.nzl; p.cz_lo = a.cz_lo; p.cz_hi = a.cz_hi;
  p.z_own_lo = a.z_own_lo; p.z_own_hi = a.z_own_hi;
  double G[N1 * N1], gq[N1], gw[N1], S2[N1 * N1], G2[N1 * N1], SG[N1 * N1];
  pmg_fe_shape_tables(P, p.S, p.D, G, gq, gw);
  for (int i = 0; i < N1 * N1; ++i) { S2[i] = p.S[i] * p.S[i]; G2[i] = G[i] * G[i]; SG[i] = p.S[i] * G[i]; }
  // the six G grids of the locally stored cell layers, as k_curved_fill computes them (from the node planes k coef_cz0 ..)
  const int k = a.k, k1 = a.k + 1;
  double s[PMGK_MAX_N1], L[PMGK_MAX_N1 * PMGK_MAX_N1], dL[PMGK_MAX_N1 * PMGK_MAX_N1];
  pmg_fe_gll(k1, s);
  for (int q = 0; q < N1; ++q) pmg_fe_lagrange(k1, s, gq[q], L + q * k1, dL + q * k1);
  const int coef_cz0 = a.z0 / P;
  const int Qx = a.nx * N1, Qy = a.ny * N1, nqz = (a.cz_hi - coef_cz0) * N1;
  const int64_t n = (int64_t)Qx * Qy * nqz;
  const int64_t sy = (int64_t)a.nx * k + 1, sz = sy * ((int64_t)a.ny * k + 1);
  const double *planes = a.nodes + 3 * sz * k * coef_cz0; // the rank's node planes only
  std::vector<double> geo(6 * (size_t)n);
  int bad = 0;
  for (int qz = 0; qz < nqz; ++qz)
    for (int qy = 0; qy < Qy; ++qy)
      for (int qx = 0; qx < Qx; ++qx) {
        const int cx = qx / N1, cy = qy / N1, lcz = qz / N1;
        const int ia = qx % N1, ib = qy % N1, im = qz % N1;
        const double *node = planes + 3 * ((int64_t)lcz * k * sz + (int64_t)cy * k * sy + (int64_t)cx * k);
        double g[6];
        const double det = pmg_curved_point(node, sy, sz, k, L + ia * k1, dL + ia * k1, L + ib * k1, dL + ib * k1, L + im * k1,
                                            dL + im * k1, gw[ia] * gw[ib] * gw[im], a.c5, g);
        if (!(det > 0.0)) bad = 1;
        for (int e = 0; e < 6; ++e) geo[(size_t)e * n + ((size_t)qz * Qy + qy) * Qx + qx] = g[e];
      }
  if (bad) return -1;
  p.coef = geo.data(); p.coef_cz0 = coef_cz0; p.gstride = n;
  // inverse diagonal on all stored planes, as k_geo_dinv computes it
  std::vector<double> dinv;
  if (a.dinv_out || (a.mode >= 2 && !a.dinv_vec)) {
    dinv.resize((size_t)p.Nx * p.Ny * a.nzl);
    for (int l = 0; l < a.nzl; ++l)
      for (int gy = 0; gy < p.Ny; ++gy)
        for (int gx = 0; gx < p.Nx; ++gx) {
          const int gz = a.z0 + l;
          const bool dir = (gx == 0 && (a.faces & 1u)) || (gx == p.Nx - 1 && (a.faces >> 1 & 1u)) ||
                           (gy == 0 && (a.faces >> 2 & 1u)) || (gy == p.Ny - 1 && (a.faces >> 3 & 1u)) ||
                           (gz == 0 && (a.faces >> 4 & 1u)) || (gz == p.Nz - 1 && (a.faces >> 5 & 1u));
          const double d = dir ? 1.0 : pmg_geo_diag_entry<P>(gx, gy, gz, a.nx, a.ny, coef_cz0, a.cz_hi, S2, G2, SG, geo.data(), n, coef_cz0);
          dinv[((size_t)l * p.Ny + gy) * p.Nx + gx] = 1.0 / d;
        }
    if (a.dinv_out) std::memcpy(a.dinv_out, dinv.data(), dinv.size() * sizeof(double));
  }
  if (!a.out) return 0;
  p.mode = a.mode; p.u = a.u; p.b = a.b; p.xold = a.xold; p.out = a.out; p.f1 = a.f1; p.f2 = a.f2;
  p.dinv_vec = a.dinv_vec ? a.dinv_vec : (dinv.empty() ? nullptr : dinv.data());
  p.dinv_tab = nullptr;
  p.tiles_x = (p.nx + BX - 1) / BX;
  p.tiles_y = (p.ny + BY - 1) / BY;
  const int layers = p.cz_hi - p.cz_lo;
  int n_chunks = a.n_chunks < 1 ? 1 : a.n_chunks;
  if (n_chunks > layers) n_chunks = layers;
  p.layers_per_chunk = (layers + n_chunks - 1) / n_chunks;
  p.n_chunks = (layers + p.layers_per_chunk - 1) / p.layers_per_chunk;
  std::vector<double> smem(Tile::SMEM_DOUBLES);
  for (int chunk = 0; chunk < p.n_chunks; ++chunk)
    for (int ty = 0; ty < p.tiles_y; ++ty)
      for (int tx = 0; tx < p.tiles_x; ++tx) {
        HostExecC<Tile> ex;
        ex.st.resize(Tile::NT);
        for (auto &v : smem) v = 1e300; // poison shared memory so stale reads show up
        Tile::run(p, ex, smem.data(), tx, ty, chunk);
      }
  return 0;
}

} // namespace

// As emu_geo, with the mesh given by its geometry support points of degree k (the full global array,
// (nx k+1)(ny k+1)(nz k+1) points, xyz interleaved, x fastest).  Returns -1 for a cell with det J <= 0 at a Gauss point
// or a non-finite node.
extern "C" int emu_curved(int degree, int k, int small_tiles, int nx, int ny, int nz, unsigned faces, int z0, int nzl,
                          int cz_lo, int cz_hi, int z_own_lo, int z_own_hi, int n_chunks, int c5, const double *nodes, int mode,
                          const double *u, const double *b, const double *xold, double *out, double f1, double f2,
                          const double *dinv_vec, double *dinv_out)
{
  if (k < 1 || k >= PMGK_MAX_N1) return -3;
  const CurvedArgs a = {nx, ny, nz, faces, z0, nzl, cz_lo, cz_hi, z_own_lo, z_own_hi, n_chunks, c5, k, nodes, mode, u, b, xold, out, f1, f2, dinv_vec, dinv_out};
  if (small_tiles) {
    switch (degree) {
      case 1: return go<1, 3, 2>(a);
      case 2: return go<2, 2, 3>(a);
      case 3: return go<3, 2, 2>(a);
      case 4: return go<4, 3, 2>(a);
      case 5: return go<5, 2, 2>(a);
      case 6: return go<6, 2, 1>(a);
      case 7: return go<7, 1, 2>(a);
      case 8: return go<8, 2, 2>(a);
      case 9: return go<9, 1, 2>(a);
    }
    return -3;
  }
  switch (degree) {
#define PMG_GEO_CASE(P, BX, BY, MINB) case P: return go<P, BX, BY>(a);
#include "pmg_apply_geo_tiles.inc"
#undef PMG_GEO_CASE
  }
  return -3;
}

// x(xi) and J(xi) of cell (cx, cy, cz) of a curved mesh (nodes as emu_curved) at the reference points xi[npts][3], by
// pmg_curved_map: x[npts][3], J[npts][3][3] with J[d][e] = d x_d / d xi_e
extern "C" int emu_curved_map(int k, int nx, int ny, const double *nodes, int cx, int cy, int cz, int npts, const double *xi,
                              double *x, double *J)
{
  if (k < 1 || k >= PMGK_MAX_N1) return -3;
  const int k1 = k + 1;
  double s[PMGK_MAX_N1], L[3][PMGK_MAX_N1], dL[3][PMGK_MAX_N1];
  pmg_fe_gll(k1, s);
  const int64_t sy = (int64_t)nx * k + 1, sz = sy * ((int64_t)ny * k + 1);
  const double *node = nodes + 3 * ((int64_t)cz * k * sz + (int64_t)cy * k * sy + (int64_t)cx * k);
  for (int q = 0; q < npts; ++q) {
    for (int d = 0; d < 3; ++d) pmg_fe_lagrange(k1, s, xi[3 * q + d], L[d], dL[d]);
    pmg_curved_map(node, sy, sz, k, L[0], dL[0], L[1], dL[1], L[2], dL[2], x + 3 * q, (double (*)[3])(J + 9 * q));
  }
  return 0;
}
