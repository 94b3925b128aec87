/* driver_common.h -- shared pieces of the C drivers (re-creations of the reference's program.cc files). */
#ifndef DRIVER_COMMON_H
#define DRIVER_COMMON_H
#include <pmg.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define CK(call)                                                                      \
  do {                                                                                \
    int rc_ = (call);                                                                 \
    if (rc_ != PMG_OK) {                                                              \
      fprintf(stderr, "\n----------------------------------------------------\n"      \
                      "Exception on processing:\n%s -> %d: %s\nAborting!\n"           \
                      "----------------------------------------------------\n",       \
              #call, rc_, pmg_last_error());                                          \
      return 1;                                                                       \
    }                                                                                 \
  } while (0)

#define MAXL 32

#include <unistd.h>

/* One process per GPU.  Launched alone the driver takes --device; launched under torchrun / mpirun-like launchers that export
   RANK, WORLD_SIZE and LOCAL_RANK (e.g. `python -m torch.distributed.run --no-python --nproc-per-node 8 ... bin/driver ...`)
   the ranks form one slab-distributed context: rank 0 creates the ncclUniqueId and hands it to the others through a file
   (PMG_NCCL_ID_FILE, default /tmp/pmg_nccl_id.<MASTER_PORT>; one node: a shared /tmp).  g_rank != 0 prints nothing. */
static int g_rank = 0, g_world = 1;
static int driver_make_context(pmg_context **ctx, int device_arg)
{
  const char *er = getenv("RANK"), *ew = getenv("WORLD_SIZE"), *el = getenv("LOCAL_RANK");
  g_rank = er ? atoi(er) : 0;
  g_world = ew ? atoi(ew) : 1;
  if (g_world <= 1) return pmg_context_create(ctx, device_arg);
  char path[512];
  const char *pf = getenv("PMG_NCCL_ID_FILE"), *port = getenv("MASTER_PORT");
  if (pf) snprintf(path, sizeof(path), "%s", pf);
  else snprintf(path, sizeof(path), "/tmp/pmg_nccl_id.%s", port ? port : "0");
  unsigned char id[128];
  if (g_rank == 0) {
    char tmp[600];
    snprintf(tmp, sizeof(tmp), "%s.tmp.%d", path, (int)getpid());
    int rc = pmg_nccl_unique_id(id);
    if (rc != PMG_OK) return rc;
    FILE *f = fopen(tmp, "wb");
    if (!f || fwrite(id, 1, sizeof(id), f) != sizeof(id)) { if (f) fclose(f); return PMG_ERR_ARG; }
    fclose(f);
    if (rename(tmp, path) != 0) return PMG_ERR_ARG; /* atomic: readers see the whole id or nothing */
  } else {
    size_t got = 0;
    for (int tries = 0; tries < 6000 && got != sizeof(id); ++tries) { /* up to 60 s */
      FILE *f = fopen(path, "rb");
      if (f) { got = fread(id, 1, sizeof(id), f); fclose(f); }
      if (got != sizeof(id)) usleep(10000);
    }
    if (got != sizeof(id)) { fprintf(stderr, "rank %d: no ncclUniqueId in %s\n", g_rank, path); return PMG_ERR_ARG; }
  }
  const int rc = pmg_context_create_distributed(ctx, el ? atoi(el) : g_rank, g_rank, g_world, id);
  if (g_rank == 0 && rc == PMG_OK) { /* everyone has joined the communicator: the file has served */
    unlink(path);
  }
  return rc;
}
/* printf on rank 0 only */
#define RPRINT(...) do { if (g_rank == 0) printf(__VA_ARGS__); } while (0)

typedef struct { int degree, n; } level_t;

static double now_s(void)
{
  struct timespec t;
  clock_gettime(CLOCK_MONOTONIC, &t);
  return t.tv_sec + 1e-9 * t.tv_nsec;
}

static int arg_int(int argc, char **argv, const char *name, int def)
{
  for (int i = 1; i + 1 < argc; ++i)
    if (!strcmp(argv[i], name)) return atoi(argv[i + 1]);
  return def;
}

static double arg_double(int argc, char **argv, const char *name, double def)
{
  for (int i = 1; i + 1 < argc; ++i)
    if (!strcmp(argv[i], name)) return atof(argv[i + 1]);
  return def;
}

/* options shared by both drivers: --coefficient 1 solves -div(a grad u) = 1, a = 1/(0.05 + 2|x|^2) (BASELINE config 5),
   --tol T the relative CG tolerance (reference 1e-12, config 5: 1e-10), --profile 1 prints the per-level device time of one
   V-cycle (smoother / transfer / halo / other), --distort EPS solves on the mesh moved by the smooth map
   x -> x + EPS sin(pi x) sin(pi y) sin(pi z) (1, 1, 1) (3-D; it fixes the boundary, so the domain stays the unit cube),
   --shell 1 solves on the quarter cylindrical shell 1 <= r <= 2, 0 <= theta <= pi/2, 0 <= z <= 1 with Dirichlet conditions
   on r = 1 and r = 2 and natural ones on the other faces (exact solution u = (1 - r^2)/4 + 3 ln r / (4 ln 2),
   ||u||_L2 = 0.14143644722133), --mapping-degree K the geometry degree of the cells of --distort / --shell: 1 (default)
   trilinear cells, 0 the level's FE degree (MappingQ(p) on every level), K >= 2 curved cells of degree K */
static int g_coefficient = 0, g_profile = 0, g_dim = 3, g_shell = 0, g_mapping_degree = 1;
static double g_tol = 1e-12, g_distort = 0.0;
static void common_options(int argc, char **argv)
{
  g_coefficient = arg_int(argc, argv, "--coefficient", 0);
  g_profile = arg_int(argc, argv, "--profile", 0);
  g_tol = arg_double(argc, argv, "--tol", 1e-12);
  g_distort = arg_double(argc, argv, "--distort", 0.0);
  g_shell = arg_int(argc, argv, "--shell", 0);
  g_mapping_degree = arg_int(argc, argv, "--mapping-degree", 1);
}

/* the level's operator: on the unit cube, or with --distort / --shell on the image of the unit cube's mesh of n^3 cells
   under the map, with cells of geometry degree k: the map evaluated at the degree-k Gauss-Lobatto grid of every cell
   (pmg_laplace_operator_create_curved; k = 1 gives the vertices of the trilinear cells, nested on the h-levels) */
static int create_level_operator(pmg_context *ctx, const level_t *lv, pmg_operator **op)
{
  if (g_distort == 0.0 && !g_shell)
    return pmg_laplace_operator_create(ctx, g_dim, lv->degree, lv->n, lv->n, lv->n, PMG_ALL_FACES, g_coefficient, op);
  if (g_dim != 3) {
    fprintf(stderr, "--distort / --shell: the mapped operator is 3-D only\n");
    return PMG_ERR_UNSUPPORTED;
  }
  const int k = g_mapping_degree == 0 ? lv->degree : g_mapping_degree;
  double s1[PMG_MAX_DEGREE + 1];
  if (k < 1 || k > PMG_MAX_DEGREE) {
    fprintf(stderr, "--mapping-degree %d outside 0..%d\n", g_mapping_degree, PMG_MAX_DEGREE);
    return PMG_ERR_UNSUPPORTED;
  }
  pmg_host_support_points(k, s1);
  const int n = lv->n, nv = n * k + 1;
  double *v = (double *)malloc(sizeof(double) * 3 * nv * nv * nv), *t = (double *)malloc(sizeof(double) * nv);
  if (!v || !t) { free(v); free(t); return PMG_ERR_NOMEM; }
  for (int c = 0; c < n; ++c)
    for (int i = 0; i < k; ++i) t[c * k + i] = (c + s1[i]) / n;
  t[n * k] = 1.0;
  const double pi = 3.14159265358979323846;
  for (int kz = 0; kz < nv; ++kz)
    for (int j = 0; j < nv; ++j)
      for (int i = 0; i < nv; ++i) {
        const double x = t[i], y = t[j], z = t[kz];
        double *p = v + 3 * ((size_t)i + (size_t)nv * (j + (size_t)nv * kz));
        if (g_shell) {
          const double r = 1.0 + x, th = 0.5 * pi * y;
          p[0] = r * cos(th); p[1] = r * sin(th); p[2] = z;
        } else {
          const double s = g_distort * sin(pi * x) * sin(pi * y) * sin(pi * z);
          p[0] = x + s; p[1] = y + s; p[2] = z + s;
        }
      }
  const unsigned faces = g_shell ? 0x3u : PMG_ALL_FACES;
  const int rc = pmg_laplace_operator_create_curved(ctx, lv->degree, k, n, n, n, faces, g_coefficient, v, op);
  free(v);
  free(t);
  return rc;
}

static long long n_dofs_of(int degree, int n)
{
  long long r = 1;
  for (int d = 0; d < g_dim; ++d) r *= (long long)n * degree + 1;
  return r;
}

/* builds operators, transfers, smoothers (program.cc:203-287) and solves (:336-364); prints the reference's lines */
static int solve_hierarchy(pmg_context *ctx, const level_t *lv, int L, int pre, int post, int cheb_degree)
{
  pmg_operator *ops[MAXL];
  pmg_transfer *tr[MAXL];
  pmg_chebyshev *sm[MAXL];
  memset(tr, 0, sizeof(tr));
  if (g_shell) RPRINT("  curved mesh: quarter cylindrical shell 1 <= r <= 2, 0 <= theta <= pi/2, 0 <= z <= 1\n");
  else if (g_distort != 0.0) RPRINT("  mapped mesh: x + %g sin(pi x) sin(pi y) sin(pi z) (1, 1, 1)\n", g_distort);
  if ((g_shell || g_distort != 0.0) && g_mapping_degree != 1) {
    if (g_mapping_degree == 0) RPRINT("  geometry: MappingQ(p) cells, p the level's FE degree\n");
    else RPRINT("  geometry: MappingQ(%d) cells\n", g_mapping_degree);
  }
  for (int l = 0; l < L; ++l) CK(create_level_operator(ctx, &lv[l], &ops[l]));
  for (int l = 1; l < L; ++l) {
    if (lv[l].degree == lv[l - 1].degree) CK(pmg_transfer_create_geometric(ops[l - 1], ops[l], &tr[l]));
    else CK(pmg_transfer_create_polynomial(ops[l - 1], ops[l], &tr[l]));
  }
  for (int l = 0; l < L; ++l) {
    int64_t m = 0;
    CK(pmg_laplace_operator_m(ops[l], &m));
    CK(pmg_laplace_operator_compute_diagonal(ops[l]));
    if (l > 0) CK(pmg_chebyshev_create(ops[l], 15.0, cheb_degree, 10, &sm[l]));
    else CK(pmg_chebyshev_create(ops[l], 1e-3, PMG_INVALID_DEGREE, (int)(m > 2000000000 ? 2000000000 : m), &sm[l]));
  }
  pmg_vcycle *mg;
  CK(pmg_vcycle_create(ops, tr, sm, L, pre, post, &mg));
  pmg_operator *A = ops[L - 1];
  pmg_vector *rhs, *x;
  CK(pmg_laplace_operator_initialize_dof_vector(A, &rhs));
  CK(pmg_laplace_operator_initialize_dof_vector(A, &x));
  CK(pmg_laplace_operator_assemble_rhs(A, rhs));
  double bnorm = 0.0;
  CK(pmg_vector_l2_norm(rhs, &bnorm));
  int64_t n_dofs = 0;
  CK(pmg_laplace_operator_m(A, &n_dofs));
  /* set-up (eigenvalue estimates) outside the timed solve, like the lazy first vmult of the reference */
  for (int l = 0; l < L; ++l) CK(pmg_chebyshev_info(sm[l], NULL, NULL, NULL, NULL));
  int last_step = 0;
  CK(pmg_sync(ctx));
  const double t0 = now_s();
  CK(pmg_cg_solve(A, x, rhs, mg, (int)(n_dofs > 100000 ? 100000 : n_dofs), g_tol * bnorm, &last_step, NULL, 0));
  CK(pmg_sync(ctx));
  const double dt = now_s() - t0;
  RPRINT("  Solver converged in %d iterations.\n", last_step);
  double norm = 0.0;
  CK(pmg_laplace_operator_solution_norm(A, x, &norm));
  RPRINT("  solution norm: %.10g\n", norm);
  RPRINT("  [b200] solve time %.3f ms on %d GPU(s), %.3f GDoF/s (DoFs x iterations / time)\n", dt * 1e3, g_world, (double)n_dofs * last_step / dt / 1e9);
  if (g_profile) {
    double ms[MAXL * 4];
    pmg_vector *z;
    CK(pmg_laplace_operator_initialize_dof_vector(A, &z));
    CK(pmg_vcycle_profile(mg, z, rhs, ms, MAXL));
    RPRINT("  [b200] one V-cycle, device ms on rank 0 per level (smoother / transfer / halo / other):\n");
    for (int l = L - 1; l >= 0; --l)
      RPRINT("    level %2d  Q%d %4d^d cells: %9.4f %9.4f %9.4f %9.4f\n", l, lv[l].degree, lv[l].n, ms[l * 4], ms[l * 4 + 1], ms[l * 4 + 2], ms[l * 4 + 3]);
    pmg_vector_destroy(z);
  }
  pmg_vector_destroy(rhs); pmg_vector_destroy(x);
  pmg_vcycle_destroy(mg);
  for (int l = 0; l < L; ++l) { pmg_chebyshev_destroy(sm[l]); if (tr[l]) pmg_transfer_destroy(tr[l]); }
  for (int l = 0; l < L; ++l) pmg_laplace_operator_destroy(ops[l]);
  return 0;
}
#endif
