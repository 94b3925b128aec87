/*
 * polynomial_multigrid.c -- C re-creation of the reference driver source/polynomial_multigrid/program.cc
 * on top of the C-ABI: p-multigrid with levels p = fe_degree-(mg_levels-1) .. fe_degree on one mesh
 * (program.cc:144-158, p -> p-1 transfers :241-242), V(2,2), Chebyshev(5)-Jacobi, coarsest level smoothed to
 * 1e-3 with eig_cg_n_iterations = m() (:320-336), CG to 1e-12 ||b|| (:346-353).
 * Defaults = the reference program (:439-441, :399): dim = 2, fe_degree = 7, mg_levels = 7, seven refinement cycles
 * (1 .. 64^2 cells).  --dim 3 runs the same hierarchy on the unit cube (then think of --degree 4 --cycles 5).
 * --hp 1 selects BASELINE config 2 instead: p = 4 -> 2 -> 1 followed by geometric levels.
 * --coefficient 1 | 2, --tol T, --profile 1, --distort EPS, --shell 1, --mapping-degree K: see driver_common.h (BASELINE config 5: --hp 1 --degree 5
 * --coefficient 1 --tol 1e-10).
 */
#include "driver_common.h"

int main(int argc, char **argv)
{
  const int fe_degree = arg_int(argc, argv, "--degree", 7);
  int mg_levels = arg_int(argc, argv, "--levels", fe_degree);
  const int cycles = arg_int(argc, argv, "--cycles", 7);
  const int cheb = arg_int(argc, argv, "--cheb-degree", 5);
  const int hp = arg_int(argc, argv, "--hp", 0);
  const int pre = arg_int(argc, argv, "--pre", 2), post = arg_int(argc, argv, "--post", 2);
  if (mg_levels > fe_degree) mg_levels = fe_degree; /* Assert(mg_levels <= fe_degree) (:140-142) */
  common_options(argc, argv);
  g_dim = arg_int(argc, argv, "--dim", 2);
  /* --cells N: one run on an N^dim mesh instead of the reference's cycles over 2^cycle cells (BASELINE config 5: N = 160) */
  const int cells_arg = arg_int(argc, argv, "--cells", 0);
  pmg_context *ctx;
  CK(driver_make_context(&ctx, arg_int(argc, argv, "--device", 0)));
  for (int cycle = 0; cycle < (cells_arg > 0 ? 1 : cycles); ++cycle) {
    RPRINT("\n\nCycle %d\n", cycle);
    const int n = cells_arg > 0 ? cells_arg : 1 << cycle;
    level_t lv[MAXL];
    int L = 0;
    if (hp) {
      int cells[MAXL], nc = 0;
      for (int m = n; ; m /= 2) { cells[nc++] = m; if (m % 2 || m == 1) break; }
      for (int i = nc - 1; i >= 1; --i) { lv[L].degree = 1; lv[L].n = cells[i]; ++L; }
      int degs[8], nd = 0;
      for (int d = fe_degree; ; d = d / 2) { degs[nd++] = d; if (d == 1) break; }
      for (int i = nd - 1; i >= 0; --i) { lv[L].degree = degs[i]; lv[L].n = n; ++L; }
    } else {
      for (int l = 0; l < mg_levels; ++l) { lv[L].degree = fe_degree - (mg_levels - 1 - l); lv[L].n = n; ++L; }
    }
    for (int l = 0; l < L; ++l)
      RPRINT("level %d: p = %d, DoFs = %lld\n", l, lv[l].degree, n_dofs_of(lv[l].degree, lv[l].n));
    if (solve_hierarchy(ctx, lv, L, pre, post, cheb)) return 1;
    RPRINT("\n");
  }
  pmg_context_destroy(ctx);
  return 0;
}
