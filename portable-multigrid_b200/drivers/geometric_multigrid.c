/*
 * geometric_multigrid.c -- C re-creation of the reference driver source/geometric_multigrid/program.cc
 * on top of the C-ABI (include/pmg.h): 3-D unit cube, degrees 1..7, six refinement cycles
 * (1, 8, ..., 32768 cells; program.cc:404-417), h-multigrid V(2,2) with Chebyshev(5)-Jacobi smoothing
 * (:267-285, :342-343), CG to 1e-12 ||b|| (:345-352).  Prints the reference's lines (:189-199, :354-355, :395).
 * Flags: --degree D (only that degree), --max-degree M (default 7), --cycles C (default 6),
 *        --cheb-degree K (default 5; BASELINE config 1 uses 3), --pre/--post (default 2).
 *        --cells N (one run on N^dim cells, e.g. BASELINE config 4), --coefficient 1, --tol T, --profile 1, --distort EPS,
 *        --shell 1, --mapping-degree K: see driver_common.h; --dim 2 runs the unit square (reference: dim = 3, :470).
 */
#include "driver_common.h"

static int g_cells = 0; /* --cells N: one run on an N^dim mesh, coarsened by halving while N stays even (BASELINE config 4: N = 160 per GPU) */

static int run_degree(pmg_context *ctx, int degree, int cycles, int pre, int post, int cheb)
{
  RPRINT("============== fe_degree = %d ============== \n\n", degree);
  for (int cycle = 0; cycle < (g_cells > 0 ? 1 : cycles); ++cycle) {
    RPRINT("\n\nCycle %d\n", cycle);
    level_t lv[MAXL];
    int L = cycle + 1; /* create_geometric_coarsening_sequence: 1, 2, 4, ... cells per direction */
    for (int l = 0; l < L; ++l) { lv[l].degree = degree; lv[l].n = 1 << l; }
    if (g_cells > 0) {
      int cells[MAXL], nc = 0;
      for (int m = g_cells; ; m /= 2) { cells[nc++] = m; if (m % 2 || m == 1) break; }
      L = nc;
      for (int l = 0; l < L; ++l) { lv[l].degree = degree; lv[l].n = cells[nc - 1 - l]; }
    }
    RPRINT(" Number of degrees of freedom: %lld (by level: ", n_dofs_of(degree, lv[L - 1].n));
    for (int l = 0; l < L; ++l) RPRINT("%lld%s", n_dofs_of(degree, lv[l].n), l == L - 1 ? ")" : ", ");
    RPRINT("\n");
    if (solve_hierarchy(ctx, lv, L, pre, post, cheb)) return 1;
    RPRINT("\n");
  }
  return 0;
}

int main(int argc, char **argv)
{
  const int only = arg_int(argc, argv, "--degree", 0);
  const int max_degree = arg_int(argc, argv, "--max-degree", 7);
  const int cycles = arg_int(argc, argv, "--cycles", 6);
  const int cheb = arg_int(argc, argv, "--cheb-degree", 5);
  const int pre = arg_int(argc, argv, "--pre", 2), post = arg_int(argc, argv, "--post", 2);
  common_options(argc, argv);
  g_dim = arg_int(argc, argv, "--dim", 3);
  g_cells = arg_int(argc, argv, "--cells", 0);
  pmg_context *ctx;
  CK(driver_make_context(&ctx, arg_int(argc, argv, "--device", 0)));
  for (int d = (only ? only : 1); d <= (only ? only : max_degree); ++d)
    if (run_degree(ctx, d, cycles, pre, post, cheb)) return 1;
  pmg_context_destroy(ctx);
  return 0;
}
