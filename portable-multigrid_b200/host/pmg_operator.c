/*
 * pmg_operator.c -- LaplaceOperator of the C-ABI (host C).
 *
 * Mirrors Portable::LaplaceOperator<dim,fe_degree,number>
 * (reference include/operators/portable_laplace_operator.h:383-461) method by method; the
 * cell loop itself is csrc/pmg_apply_sweep.h.  The constructor replaces MatrixFree::reinit +
 * setup_dirichlet_boundary_dofs_masks (:463-555): on the structured box nothing needs to be
 * stored per cell, only the 1-D tables.
 */
#include "pmg_internal.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* Variable coefficient (BASELINE config 5; no reference equivalent, SURVEY.md 8d): w_q a(x_q) of every quadrature point of
   the locally stored cell layers is evaluated once on the device and streamed by the apply kernel
   (csrc/pmg_apply_var.h); the inverse diagonal of such an operator is an explicit vector. */
static int var_diagonal(pmg_operator *op)
{
  const int n1 = op->degree + 1;
  double Sq[PMGK_MAX_N1 * PMGK_MAX_N1], G[PMGK_MAX_N1 * PMGK_MAX_N1];
  pmg_fe_shape_tables(op->degree, Sq, NULL, G, NULL, NULL);
  for (int i = 0; i < n1 * n1; ++i) { Sq[i] *= Sq[i]; G[i] *= G[i]; }
  return pmgk_var_fill_dinv(&op->lv, Sq, G, op->dinv->d, op->ctx->stream);
}

static int setup_coefficient(pmg_operator *op)
{
  pmgk_level *lv = &op->lv;
  double gq[PMGK_MAX_N1], gw[PMGK_MAX_N1];
  pmg_fe_shape_tables(op->degree, lv->Sq, lv->Dco, NULL, gq, gw);
  lv->coef_cz0 = lv->z0 / op->degree;
  PMG_CHECK(pmg_vector_create_layout(op->ctx, &op->lay, &op->dinv));
  if (!op->lay.active) return PMG_OK;
  const int64_t n = pmgk_var_coef_doubles(lv);
  if (cudaMalloc((void **)&op->d_coef, sizeof(double) * (size_t)n) != cudaSuccess) {
    pmg_set_error("cudaMalloc of %lld coefficient values failed", (long long)n);
    return PMG_ERR_NOMEM;
  }
  PMG_CHECK(pmgk_var_fill_coef(lv, op->coefficient, gq, gw, op->d_coef, op->ctx->stream));
  lv->coef = op->d_coef;
  PMG_CHECK(var_diagonal(op));
  lv->dinv_vec = op->dinv->d;
  return PMG_OK;
}

/* Mapped geometry (SURVEY.md row f4): the six entries of G_q = w_q a(x_q) |det J_q| J_q^-1 J_q^-T of every quadrature point
   of the locally stored cell layers, computed on the device from the cells' maps (csrc/pmg_apply_geo.cu) -- trilinear
   (geometry degree 1) or the degree-k Lagrange interpolant through (k+1)^3 nodes (curved cells, MappingQ(k)) -- and
   streamed by the tensor variant of the variable-coefficient kernel.  Only the node planes of the stored layers are
   uploaded; a cell with det J <= 0 at a Gauss point or a non-finite node rejects the mesh. */
static int geo_diagonal(pmg_operator *op)
{
  const int n1 = op->degree + 1;
  double Sq[PMGK_MAX_N1 * PMGK_MAX_N1], G[PMGK_MAX_N1 * PMGK_MAX_N1], SG[PMGK_MAX_N1 * PMGK_MAX_N1];
  pmg_fe_shape_tables(op->degree, Sq, NULL, G, NULL, NULL);
  for (int i = 0; i < n1 * n1; ++i) { SG[i] = Sq[i] * G[i]; Sq[i] *= Sq[i]; G[i] *= G[i]; }
  return pmgk_geo_fill_dinv(&op->lv, Sq, G, SG, op->dinv->d, op->ctx->stream);
}

static int setup_geometry(pmg_operator *op, const double *nodes)
{
  const int k = op->geo_degree;
  pmgk_level *lv = &op->lv;
  double gq[PMGK_MAX_N1], gw[PMGK_MAX_N1];
  pmg_fe_shape_tables(op->degree, lv->Sq, lv->Dco, NULL, gq, gw);
  lv->coef_cz0 = lv->z0 / op->degree;
  PMG_CHECK(pmg_vector_create_layout(op->ctx, &op->lay, &op->dinv));
  if (!op->lay.active) return PMG_OK;
  const int64_t n = pmgk_var_coef_doubles(lv);
  lv->geo_stride = n;
  if (cudaMalloc((void **)&op->d_coef, sizeof(double) * 6 * (size_t)n) != cudaSuccess) {
    pmg_set_error("cudaMalloc of %lld geometry values failed", (long long)(6 * n));
    return PMG_ERR_NOMEM;
  }
  lv->coef = op->d_coef;
  /* node planes k coef_cz0 .. k cz_hi of the stored cell layers, and one error word */
  const size_t vplane = (size_t)(lv->nx * (size_t)k + 1) * (lv->ny * (size_t)k + 1) * 3;
  const size_t nv = vplane * ((size_t)(lv->cz_hi - lv->coef_cz0) * k + 1);
  cudaStream_t st = op->ctx->stream;
  unsigned long long *d_err = NULL, h_err = 0;
  int rc = PMG_OK;
  if (cudaMalloc((void **)&op->d_vert, sizeof(double) * nv + sizeof(unsigned long long)) != cudaSuccess) {
    pmg_set_error("cudaMalloc of %lld node coordinates failed", (long long)nv);
    return PMG_ERR_NOMEM;
  }
  d_err = (unsigned long long *)(op->d_vert + nv);
  if (cudaMemcpyAsync(op->d_vert, nodes + vplane * k * lv->coef_cz0, sizeof(double) * nv, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemsetAsync(d_err, 0xFF, sizeof(unsigned long long), st) != cudaSuccess) rc = PMG_ERR_CUDA;
  if (rc == PMG_OK) rc = pmgk_geo_fill(lv, k, op->coefficient, op->d_vert, gq, gw, op->d_coef, d_err, st);
  if (rc == PMG_OK && cudaMemcpyAsync(&h_err, d_err, sizeof(h_err), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = PMG_ERR_CUDA;
  if (cudaStreamSynchronize(st) != cudaSuccess && rc == PMG_OK) rc = PMG_ERR_CUDA; /* nodes and h_err are pageable */
  if (rc != PMG_OK) return rc;
  if (h_err != ~0ull) {
    const long long c = (long long)h_err, cx = c % lv->nx, cy = c / lv->nx % lv->ny, cz = c / ((long long)lv->nx * lv->ny);
    pmg_set_error("mapped mesh: cell %lld = (%lld, %lld, %lld) has det J <= 0 at a Gauss point or a non-finite %s", c, cx, cy, cz,
                  k == 1 ? "vertex" : "node");
    return PMG_ERR_ARG;
  }
  PMG_CHECK(geo_diagonal(op));
  lv->dinv_vec = op->dinv->d;
  return PMG_OK;
}

/* nodes: NULL (the box), or the mesh's geometry support points of geometry degree k (k = 1: the vertices) */
static int operator_create(pmg_context *ctx, int dim, int degree, int nx, int ny, int nz, unsigned faces, int coefficient,
                           const double *nodes, int k, pmg_operator **out)
{
  if (!ctx || !out || nx < 1 || ny < 1 || nz < 1) { pmg_set_error("operator_create: bad arguments"); return PMG_ERR_ARG; }
  if (dim != 2 && dim != 3) { pmg_set_error("dim = %d: the reference instantiates dim = 2 and dim = 3", dim); return PMG_ERR_UNSUPPORTED; }
  if (dim == 2) { nz = 1; faces &= 0xFu; }
  if (dim == 2 && coefficient != 0) { pmg_set_error("the variable-coefficient operator is 3-D only"); return PMG_ERR_UNSUPPORTED; }
  if (degree < 1 || degree > PMG_MAX_DEGREE) { pmg_set_error("degree %d outside 1..%d", degree, PMG_MAX_DEGREE); return PMG_ERR_UNSUPPORTED; }
  if (coefficient != 0 && coefficient != 1) { pmg_set_error("coefficient %d: 0 = constant, 1 = 1/(0.05 + 2|x|^2)", coefficient); return PMG_ERR_UNSUPPORTED; }
  if ((int64_t)(nx * (int64_t)degree + 1) * (ny * (int64_t)degree + 1) >= (int64_t)1 << 31) return PMG_ERR_ARG;
  pmg_operator *op = (pmg_operator *)calloc(1, sizeof(*op));
  if (!op) return PMG_ERR_NOMEM;
  op->ctx = ctx; op->dim = dim; op->degree = degree; op->coefficient = coefficient; op->faces = faces & PMG_ALL_FACES;
  op->mapped = nodes != NULL;
  op->geo_degree = nodes ? k : 0;
  PMG_CHECK(pmg_layout_make(ctx, dim, degree, nx, ny, nz, &op->lay));
  pmgk_level *lv = &op->lv;
  lv->dim = dim;
  lv->degree = degree;
  lv->nx = nx; lv->ny = ny; lv->nz = nz;
  lv->Nx = op->lay.Nx; lv->Ny = op->lay.Ny; lv->Nz = op->lay.Nz;
  lv->faces = op->faces;
  lv->z0 = op->lay.z0; lv->nzl = op->lay.nzl;
  lv->cz_lo = op->lay.cz_lo; lv->cz_hi = op->lay.cz_hi;
  lv->z_own_lo = op->lay.z_own_lo; lv->z_own_hi = op->lay.z_own_hi;
  lv->h[0] = 1.0 / nx; lv->h[1] = 1.0 / ny; lv->h[2] = (dim == 2) ? 1.0 : 1.0 / nz;
  pmg_fe_fastdiag(degree, lv->S, lv->lam);
  pmg_fe_pencil(degree, lv->Mref, lv->Kref);
  const int T = degree + 2;
  double *tab = (double *)malloc(sizeof(double) * T * T * T);
  if (!tab) { free(op); return PMG_ERR_NOMEM; }
  pmg_fe_dinv_table(degree, lv->h, dim, tab);
  PMG_CUDA(cudaSetDevice(ctx->device));
  PMG_CUDA(cudaMalloc((void **)&op->d_dinv_tab, sizeof(double) * T * T * T));
  PMG_CUDA(cudaMemcpyAsync(op->d_dinv_tab, tab, sizeof(double) * T * T * T, cudaMemcpyHostToDevice, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  free(tab);
  lv->dinv_tab = op->d_dinv_tab;
  lv->dinv_vec = NULL;
  const char *tv = getenv("PMG_TILE_VARIANT");
  lv->tile_variant = tv ? atoi(tv) : 0;
  if (nodes) {
    const int rc = setup_geometry(op, nodes);
    if (rc != PMG_OK) { pmg_laplace_operator_destroy(op); return rc; }
  } else if (coefficient != 0) {
    const int rc = setup_coefficient(op);
    if (rc != PMG_OK) { pmg_laplace_operator_destroy(op); return rc; }
  }
  *out = op;
  return PMG_OK;
}

int pmg_laplace_operator_create(pmg_context *ctx, int dim, int degree, int nx, int ny, int nz,
                                unsigned faces, int coefficient, pmg_operator **out)
{
  return operator_create(ctx, dim, degree, nx, ny, nz, faces, coefficient, NULL, 0, out);
}

int pmg_laplace_operator_create_mapped(pmg_context *ctx, int degree, int nx, int ny, int nz, unsigned faces, int coefficient,
                                       const double *vertices, pmg_operator **out)
{
  if (!vertices) { pmg_set_error("operator_create_mapped: no vertices"); return PMG_ERR_ARG; }
  return operator_create(ctx, 3, degree, nx, ny, nz, faces, coefficient, vertices, 1, out);
}

int pmg_laplace_operator_create_curved(pmg_context *ctx, int degree, int geometry_degree, int nx, int ny, int nz, unsigned faces,
                                       int coefficient, const double *nodes, pmg_operator **out)
{
  if (geometry_degree < 1 || geometry_degree > PMG_MAX_DEGREE) {
    pmg_set_error("geometry degree %d outside 1..%d", geometry_degree, PMG_MAX_DEGREE);
    return PMG_ERR_UNSUPPORTED;
  }
  if (!nodes) { pmg_set_error("operator_create_curved: no nodes"); return PMG_ERR_ARG; }
  return operator_create(ctx, 3, degree, nx, ny, nz, faces, coefficient, nodes, geometry_degree, out);
}

int pmg_laplace_operator_destroy(pmg_operator *op)
{
  if (!op) return PMG_OK;
  cudaStreamSynchronize(op->ctx->stream);
  if (op->dinv) pmg_vector_destroy(op->dinv);
  for (int i = 0; i < 4; ++i) if (op->cg_ws[i]) pmg_vector_destroy(op->cg_ws[i]);
  cudaFree(op->d_dinv_tab);
  cudaFree(op->d_coef);
  cudaFree(op->d_vert);
  free(op);
  return PMG_OK;
}

static int check_vec(const pmg_operator *op, const pmg_vector *v, const char *what)
{
  if (!v || v->ctx != op->ctx || !pmg_layout_same(&v->lay, &op->lay)) {
    pmg_set_error("%s: vector is not initialised for this operator (initialize_dof_vector)", what);
    return PMG_ERR_ARG;
  }
  return PMG_OK;
}

/* chunk launch order of fused launches (bit 1 of pmgk_push.consume): natural (bottom chunk first), the default -- measured
   6.34 : 6.52 ms per C2 cycle on 2 GPUs and 7.67 : 7.92 ms on 8 against "top chunk first, bottom chunk last"
   (PMG_FUSED_ORDER=1), which gives the flags more slack but changes the order of the memory streams */
static int fused_order_bit(void)
{
  static int natural_order = -1;
  if (natural_order < 0) { const char *e = getenv("PMG_FUSED_ORDER"); natural_order = (e && atoi(e) == 1) ? 0 : 1; }
  return natural_order ? 2 : 0;
}

/* ghost update of u followed by the fused apply (every operator application of the path goes through here) */
int pmg_apply_with_halo(const pmg_operator *op, int mode, double *u, const double *b, const double *xold, double *out, double f1, double f2)
{
  if (op) PMG_CHECK(pmg_enter(op->ctx));
  pmg_context *ctx = op->ctx;
  if (!op->lay.active) return PMG_OK;
  /* src.update_ghost_values() (:661); there is no compress(add): the kernel owns complete rows */
  const int slab = ctx->has_comm && !op->lay.gathered;
  if (slab && ctx->overlap && pmgk_apply_splits(&op->lv, mode)) {
    /* the reference's overlap of communication and computation (:635-657: ghost_start, interior cells, ghost_finish,
       boundary cells), here for the z-chunks of the launch: the chunks that read no ghost plane run while the ghost planes
       travel on the halo stream / communicator; the first and the last chunk follow.  Event fork / join, capturable. */
    PMG_CUDA(cudaEventRecord(ctx->ev_ready, ctx->stream));
    PMG_CUDA(cudaStreamWaitEvent(ctx->halo_stream, ctx->ev_ready, 0));
    PMG_CHECK(pmg_halo_update_on(ctx, &op->lay, u, ctx->halo_comm, ctx->halo_stream));
    PMG_CUDA(cudaEventRecord(ctx->ev_halo, ctx->halo_stream));
    PMG_CHECK(pmgk_apply_part(&op->lv, mode, u, b, xold, out, f1, f2, PMGK_PART_INTERIOR, ctx->stream));
    PMG_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_halo, 0));
    return pmgk_apply_part(&op->lv, mode, u, b, xold, out, f1, f2, PMGK_PART_BOUNDARY, ctx->stream);
  }
  PMG_CHECK(pmg_halo_update(ctx, &op->lay, u));
  {
    /* PMG_FUSED_SELFTEST=1 (experiments, one GPU): run the kernel instance that carries the fused ghost exchange -- flag words,
       tickets, push code -- without neighbours, to time what that machinery costs by itself */
    static int selftest = -1;
    if (selftest < 0) { const char *e = getenv("PMG_FUSED_SELFTEST"); selftest = (e && atoi(e) != 0) ? 1 : 0; }
    if (selftest && !ctx->has_comm && pmgk_apply_can_push(&op->lv, mode)) {
      if (!ctx->p2p.mailbox) {
        PMG_CUDA(cudaMalloc((void **)&ctx->p2p.mailbox, 16 * sizeof(uint64_t)));
        PMG_CUDA(cudaMemset(ctx->p2p.mailbox, 0, 16 * sizeof(uint64_t)));
      }
      pmgk_push d;
      memset(&d, 0, sizeof(d));
      d.mailbox = ctx->p2p.mailbox; d.consume = 1 | fused_order_bit();
      { const char *e = getenv("PMG_FUSED_SELFTEST_BITS"); if (e) d.consume |= atoi(e); }
      return pmgk_apply_push(&op->lv, mode, u, b, xold, out, f1, f2, &d, ctx->stream);
    }
  }
  return pmgk_apply(&op->lv, mode, u, b, xold, out, f1, f2, ctx->stream);
}

/* Can a chain of applies on this operator exchange its ghost planes by fused pushes?  (slab with neighbours, the level's
   kernel supports it, both ping-pong vectors mapped on the neighbours; identical answer on every rank: slabs are equal and
   vectors are created collectively) */
int pmg_apply_chain_ok(const pmg_operator *op, int mode, double *v0, double *v1)
{
  pmg_context *ctx = op->ctx;
  pmgk_push d;
  if (!op->lay.active || !ctx->has_comm || op->lay.gathered || ctx->overlap) return 0;
  if (!pmgk_apply_can_push(&op->lv, mode)) return 0;
  return pmg_p2p_push_desc(ctx, &op->lay, v0, &d) && pmg_p2p_push_desc(ctx, &op->lay, v1, &d);
}

/* One apply of a chain (pmg_apply_chain_ok): consume = u was written by the previous apply of the chain, which pushed its
   boundary planes into the neighbours' ghost planes, so no exchange happens here; push = the next apply of the chain reads
   `out`.  Reference: src.update_ghost_values() before every cell loop (:661) -- here the cell loop of the previous step
   has already delivered them. */
int pmg_apply_chained(const pmg_operator *op, int mode, double *u, const double *b, const double *xold, double *out, double f1,
                      double f2, int consume, int push)
{
  PMG_CHECK(pmg_enter(op->ctx));
  pmg_context *ctx = op->ctx;
  if (!op->lay.active) return PMG_OK;
  pmgk_push d;
  if (push) { if (!pmg_p2p_push_desc(ctx, &op->lay, out, &d)) return PMG_ERR_ARG; }
  else if (!pmg_p2p_push_desc(ctx, &op->lay, u, &d)) return PMG_ERR_ARG; /* consume only: the flag words, no target */
  d.push = push; d.consume = (consume ? 1 : 0) | fused_order_bit();
  if (!consume) PMG_CHECK(pmg_halo_update(ctx, &op->lay, u));
  else ++ctx->p2p.n_fused;
  return pmgk_apply_push(&op->lv, mode, u, b, xold, out, f1, f2, &d, ctx->stream);
}

static int apply_mode(const pmg_operator *op, int mode, pmg_vector *dst, const pmg_vector *src, const pmg_vector *b,
                      const pmg_vector *xold, double f1, double f2)
{
  return pmg_apply_with_halo(op, mode, src->d, b ? b->d : NULL, xold ? xold->d : NULL, dst->d, f1, f2);
}

int pmg_laplace_operator_vmult(const pmg_operator *op, pmg_vector *dst, const pmg_vector *src)
{
  if (!op) return PMG_ERR_ARG;
  PMG_CHECK(check_vec(op, dst, "vmult(dst)"));
  PMG_CHECK(check_vec(op, src, "vmult(src)"));
  if (dst == src) { pmg_set_error("vmult: dst and src must differ"); return PMG_ERR_ARG; }
  return apply_mode(op, PMGK_APPLY, dst, src, NULL, NULL, 0.0, 0.0);
}

int pmg_laplace_operator_Tvmult(const pmg_operator *op, pmg_vector *dst, const pmg_vector *src)
{
  return pmg_laplace_operator_vmult(op, dst, src); /* symmetric (:721-735) */
}

int pmg_laplace_operator_residual(const pmg_operator *op, pmg_vector *dst, const pmg_vector *b, const pmg_vector *src)
{
  if (!op) return PMG_ERR_ARG;
  PMG_CHECK(check_vec(op, dst, "residual(dst)"));
  PMG_CHECK(check_vec(op, src, "residual(src)"));
  PMG_CHECK(check_vec(op, b, "residual(b)"));
  if (dst == src) { pmg_set_error("residual: dst and src must differ"); return PMG_ERR_ARG; }
  return apply_mode(op, PMGK_RESIDUAL, dst, src, b, NULL, 0.0, 0.0);
}

int pmg_laplace_operator_chebyshev_step(const pmg_operator *op, pmg_vector *dst, const pmg_vector *src,
                                        const pmg_vector *xold, const pmg_vector *b, double f1, double f2)
{
  if (!op) return PMG_ERR_ARG;
  PMG_CHECK(check_vec(op, dst, "chebyshev_step(dst)"));
  PMG_CHECK(check_vec(op, src, "chebyshev_step(src)"));
  PMG_CHECK(check_vec(op, b, "chebyshev_step(b)"));
  if (xold) PMG_CHECK(check_vec(op, xold, "chebyshev_step(xold)"));
  if (dst == src) { pmg_set_error("chebyshev_step: dst and src must differ"); return PMG_ERR_ARG; }
  return apply_mode(op, PMGK_CHEB_STEP, dst, src, b, xold, f1, f2);
}

int pmg_laplace_operator_initialize_dof_vector(const pmg_operator *op, pmg_vector **vec)
{
  if (!op || !vec) return PMG_ERR_ARG;
  return pmg_vector_create_layout(op->ctx, &op->lay, vec);
}

int pmg_laplace_operator_compute_diagonal(pmg_operator *op)
{
  if (!op) return PMG_ERR_ARG;
  if (!op->dinv) PMG_CHECK(pmg_vector_create_layout(op->ctx, &op->lay, &op->dinv));
  if (!op->lay.active) return PMG_OK;
  if (op->lv.geo_stride) return geo_diagonal(op);
  if (op->coefficient != 0) return var_diagonal(op);
  /* diagonal of the tensor-product cell matrices summed at shared dofs, 1 on constrained dofs,
     inverted (:752-917).  The fused smoother keeps using the (p+2)^3 table: same numbers,
     no 8 B/DoF stream. */
  return pmgk_fill_dinv(&op->lv, op->dinv->d, op->ctx->stream);
}

int pmg_laplace_operator_get_matrix_diagonal_inverse(const pmg_operator *op, const pmg_vector **dinv)
{
  if (!op || !dinv) return PMG_ERR_ARG;
  if (!op->dinv) { pmg_set_error("compute_diagonal() has not been called"); return PMG_ERR_STATE; }
  *dinv = op->dinv;
  return PMG_OK;
}

int pmg_laplace_operator_m(const pmg_operator *op, int64_t *m) { if (!op || !m) return PMG_ERR_ARG; *m = op->lay.n_global; return PMG_OK; }
int pmg_laplace_operator_n(const pmg_operator *op, int64_t *n) { return pmg_laplace_operator_m(op, n); }

int pmg_laplace_operator_el(const pmg_operator *op, int64_t row, int64_t col, double *value)
{
  if (!op || !value || row < 0 || row >= op->lay.n_global) return PMG_ERR_ARG;
  if (row != col) { pmg_set_error("el(): only diagonal entries are available (reference: ExcNotImplemented)"); return PMG_ERR_UNSUPPORTED; }
  if (!op->dinv) { pmg_set_error("el(): compute_diagonal() has not been called"); return PMG_ERR_STATE; }
  /* 1 / inverse_diagonal(row,row) (:953); the owner of the row reads it, the others get it by allreduce */
  pmg_context *ctx = op->ctx;
  const pmg_layout *l = &op->lay;
  const int gz = (int)(row / l->plane);
  double v = 0.0;
  PMG_CUDA(cudaMemsetAsync(ctx->scalars + 1, 0, sizeof(double), ctx->stream));
  if (l->active && gz >= l->z_own_lo && gz < l->z_own_hi)
    PMG_CUDA(cudaMemcpyAsync(ctx->scalars + 1, op->dinv->d + (row - l->plane * l->z0), sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  PMG_CHECK(pmg_allreduce_sum(ctx, ctx->scalars + 1, 1));
  PMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 1, ctx->scalars + 1, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  v = ctx->h_scalars[1];
  *value = 1.0 / v;
  return PMG_OK;
}

int pmg_laplace_operator_degree(const pmg_operator *op, int *degree) { if (!op || !degree) return PMG_ERR_ARG; *degree = op->degree; return PMG_OK; }

int pmg_laplace_operator_cells(const pmg_operator *op, int *nx, int *ny, int *nz)
{
  if (!op) return PMG_ERR_ARG;
  if (nx) *nx = op->lay.nx;
  if (ny) *ny = op->lay.ny;
  if (nz) *nz = op->lay.nz;
  return PMG_OK;
}

int pmg_laplace_operator_vmult_host(const pmg_operator *op, double *dst_host, const double *src_host)
{
  if (!op || !dst_host || !src_host) return PMG_ERR_ARG;
  pmg_vector *s = NULL, *d = NULL;
  PMG_CHECK(pmg_laplace_operator_initialize_dof_vector(op, &s));
  PMG_CHECK(pmg_laplace_operator_initialize_dof_vector(op, &d));
  int rc = pmg_vector_import_host(s, src_host);
  if (!rc) rc = pmg_laplace_operator_vmult(op, d, s);
  if (!rc) rc = pmg_vector_export_host(d, dst_host);
  pmg_vector_destroy(s);
  pmg_vector_destroy(d);
  return rc;
}

/* ---- driver helpers: right-hand side and solution norm ---------------------------------- */
/* Mapped mesh: neither the load vector nor the norm factorises.  b_i = sum_cells sum_q phi_i(x_q) w_q |det J_q| (QGauss(p+1),
   constrained rows dropped) as a deterministic per-dof gather over the <= 8 cells of each dof; the ghost planes are then
   refreshed from their owners. */
static int mapped_rhs(const pmg_operator *op, pmg_vector *rhs)
{
  const pmgk_level *lv = &op->lv;
  if (!op->lay.active) return PMG_OK;
  double S[PMGK_MAX_N1 * PMGK_MAX_N1], gq[PMGK_MAX_N1], gw[PMGK_MAX_N1];
  pmg_fe_shape_tables(op->degree, S, NULL, NULL, gq, gw);
  cudaStream_t st = op->ctx->stream;
  double *W = NULL;
  const int64_t n = pmgk_var_coef_doubles(lv);
  if (cudaMallocAsync((void **)&W, sizeof(double) * (size_t)(n > 0 ? n : 1), st) != cudaSuccess) return PMG_ERR_NOMEM;
  int rc = pmgk_geo_rhs(lv, op->geo_degree, op->d_vert, S, gq, gw, W, rhs->d, st);
  cudaFreeAsync(W, st);
  if (rc != PMG_OK) return rc;
  return pmg_halo_update(op->ctx, &op->lay, rhs->d);
}

/* ||u_h||_L2 with QGauss(p+2) as integrate_difference (program.cc:382-395): per owned cell u_h interpolated to the (p+2)^3
   points, weighted with w |det J|; the cell sums are reduced deterministically (two-stage) and over the ranks */
static int mapped_norm(const pmg_operator *op, const pmg_vector *u, double *norm)
{
  pmg_context *ctx = op->ctx;
  const pmgk_level *lv = &op->lv;
  const int p = op->degree, n1 = p + 1, m = p + 2;
  double gll[PMG_MAX_DEGREE + 2], g[PMG_MAX_DEGREE + 2], w[PMG_MAX_DEGREE + 2], E[(PMG_MAX_DEGREE + 2) * (PMG_MAX_DEGREE + 1)];
  pmg_fe_gll(n1, gll);
  pmg_fe_gauss(m, g, w);
  for (int q = 0; q < m; ++q) pmg_fe_lagrange(n1, gll, g[q], E + q * n1, NULL);
  PMG_CUDA(cudaMemsetAsync(ctx->scalars, 0, sizeof(double), ctx->stream));
  if (op->lay.active) {
    const int64_t ncells = (int64_t)lv->nx * lv->ny * (lv->cz_hi - lv->cz_lo);
    double *sums = NULL;
    PMG_CHECK(pmg_halo_update(ctx, &u->lay, u->d));
    if (cudaMallocAsync((void **)&sums, sizeof(double) * (size_t)(ncells > 0 ? ncells : 1), ctx->stream) != cudaSuccess) return PMG_ERR_NOMEM;
    int rc = pmgk_geo_norm_cells(lv, op->geo_degree, op->d_vert, E, g, w, u->d, sums, ctx->stream);
    if (rc == PMG_OK) rc = pmgk_sum(sums, ncells, ctx->scalars, ctx->work, ctx->stream);
    cudaFreeAsync(sums, ctx->stream);
    if (rc != PMG_OK) return rc;
  }
  PMG_CHECK(pmg_allreduce_sum(ctx, ctx->scalars, 1));
  PMG_CUDA(cudaMemcpyAsync(ctx->h_scalars, ctx->scalars, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  *norm = sqrt(fabs(ctx->h_scalars[0]));
  return PMG_OK;
}

/* Load vector of f = 1 (reference source/geometric_multigrid/program.cc:289-334).  On the box mesh
   the cell vector is the tensor product of the 1-D load b1[i] = sum_q w_q phi_i(x_q) h, so the global
   vector is separable too: rhs(x,y,z) = bx(x) by(y) bz(z), constrained rows dropped.  Assembled on
   the host once (setup path, SURVEY.md row f3). */
int pmg_laplace_operator_assemble_rhs(const pmg_operator *op, pmg_vector *rhs)
{
  if (!op) return PMG_ERR_ARG;
  PMG_CHECK(check_vec(op, rhs, "assemble_rhs"));
  if (op->mapped) return mapped_rhs(op, rhs);
  const pmg_layout *l = &op->lay;
  if (!l->active) return PMG_OK;
  const int p = op->degree, n1 = p + 1;
  double gll[PMG_MAX_DEGREE + 2], g[PMG_MAX_DEGREE + 2], w[PMG_MAX_DEGREE + 2], v[PMG_MAX_DEGREE + 2], b1[PMG_MAX_DEGREE + 2];
  pmg_fe_gll(n1, gll);
  pmg_fe_gauss(n1, g, w);
  memset(b1, 0, sizeof(b1));
  for (int q = 0; q < n1; ++q) {
    pmg_fe_lagrange(n1, gll, g[q], v, NULL);
    for (int i = 0; i < n1; ++i) b1[i] += w[q] * v[i];
  }
  const int N[3] = {l->Nx, l->Ny, l->Nz}, nc[3] = {l->nx, l->ny, l->nz};
  double *line[3];
  for (int d = 0; d < 3; ++d) {
    line[d] = (double *)calloc((size_t)N[d], sizeof(double));
    if (!line[d]) return PMG_ERR_NOMEM;
    if (d == 2 && op->dim == 2) { line[d][0] = 1.0; continue; } /* 2-D: the single plane */
    for (int c = 0; c < nc[d]; ++c)
      for (int i = 0; i < n1; ++i) line[d][c * p + i] += b1[i] * op->lv.h[d];
    if (op->faces >> (2 * d) & 1u) line[d][0] = 0.0;
    if (op->faces >> (2 * d + 1) & 1u) line[d][N[d] - 1] = 0.0;
  }
  /* the load vector of f = 1 is the tensor product of the three 1-D lines: formed on the device (no O(N) host work) */
  const size_t nl = (size_t)N[0] + N[1] + N[2];
  double *d_lines = NULL, *h_lines = (double *)malloc(sizeof(double) * nl);
  if (!h_lines) { for (int d = 0; d < 3; ++d) free(line[d]); return PMG_ERR_NOMEM; }
  memcpy(h_lines, line[0], sizeof(double) * N[0]);
  memcpy(h_lines + N[0], line[1], sizeof(double) * N[1]);
  memcpy(h_lines + N[0] + N[1], line[2], sizeof(double) * N[2]);
  for (int d = 0; d < 3; ++d) free(line[d]);
  cudaStream_t st = op->ctx->stream;
  int rc = PMG_OK;
  if (cudaMallocAsync((void **)&d_lines, sizeof(double) * nl, st) != cudaSuccess ||
      cudaMemcpyAsync(d_lines, h_lines, sizeof(double) * nl, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = PMG_ERR_CUDA;
  if (rc == PMG_OK) rc = pmgk_outer3(rhs->d, d_lines, d_lines + N[0], d_lines + N[0] + N[1] + l->z0, l->Nx, l->Ny, l->nzl, st);
  if (d_lines) cudaFreeAsync(d_lines, st);
  if (cudaStreamSynchronize(st) != cudaSuccess && rc == PMG_OK) rc = PMG_ERR_CUDA; /* h_lines is pageable */
  free(h_lines);
  return rc;
}

/* ||u_h||_L2 (program.cc:382-395; QGauss(p+2) there, exact for the degree-2p integrand like the (p+1)-point rule of the
   cell mass matrix): ||u_h||^2 = u^T (Mx (x) My (x) Mz) u.  The apply kernel with the 1-D stiffness matrix replaced by
   the mass matrix computes (cx + cy + cz) (M (x) M (x) M) u for the reference-cell M (csrc/pmg_apply_sweep.h), so the norm
   costs one apply and one dot on the device; boundary values of u are part of the norm, hence no Dirichlet faces. */
int pmg_laplace_operator_solution_norm(const pmg_operator *op, const pmg_vector *u, double *norm)
{
  if (!op || !norm) return PMG_ERR_ARG;
  PMG_CHECK(check_vec(op, u, "solution_norm"));
  if (op->mapped) return mapped_norm(op, u, norm);
  pmg_context *ctx = op->ctx;
  pmg_vector *t = NULL;
  PMG_CHECK(pmg_vector_create_layout(ctx, &op->lay, &t));
  pmgk_level lv = op->lv;
  memcpy(lv.Kref, lv.Mref, sizeof(lv.Kref));
  lv.faces = 0;
  lv.coef = NULL; /* the mass matrix has no coefficient */
  lv.tile_variant = 1; /* the line-marching kernel: the cell-tile kernel works in the eigenbasis of the (M, K) pencil */
  int rc = PMG_OK;
  double uMu = 0.0;
  if (op->lay.active) {
    rc = pmg_halo_update(ctx, &u->lay, u->d);
    if (rc == PMG_OK) rc = pmgk_apply(&lv, PMGK_APPLY, u->d, NULL, NULL, t->d, 0.0, 0.0, ctx->stream);
  }
  if (rc == PMG_OK) rc = pmg_vector_dot(u, t, &uMu);
  pmg_vector_destroy(t);
  if (rc != PMG_OK) return rc;
  const double *h = op->lv.h;
  if (op->dim == 2) { /* the 2-D apply computes (hy/hx + hx/hy) (M (x) M) u */
    *norm = sqrt(fabs(uMu) * (h[0] * h[1]) / (h[1] / h[0] + h[0] / h[1]));
    return PMG_OK;
  }
  const double cx = h[1] * h[2] / h[0], cy = h[0] * h[2] / h[1], cz = h[0] * h[1] / h[2];
  *norm = sqrt(fabs(uMu) * (h[0] * h[1] * h[2]) / (cx + cy + cz));
  return PMG_OK;
}
