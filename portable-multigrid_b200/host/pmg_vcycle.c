/*
 * pmg_vcycle.c -- VCycleMultigrid and the outer CG of the C-ABI (host C).
 *
 * Mirrors Portable::VCycleMultigrid (reference include/multigrid/portable_v_cycle_multigrid.h:
 * ctor :66-77, vmult :79-94, smooth :96-126, v_cycle :128-190) and deal.II's SolverCG as the
 * drivers call it (source/geometric_multigrid/program.cc:342-355).
 *
 * B200-first differences: all level vectors are allocated once (the reference allocates 2 device
 * vectors per smooth() and 3 per level per cycle, :116-118,:163-176); smoothing steps are fused
 * passes (pmg_smoother.c); the first pre-smoothing step of every level starts from a zero guess and
 * skips A*0; after a warm-up call the whole cycle is replayed from one CUDA graph, which removes the
 * launch latency that dominates the coarse levels (1..512 cells).
 */
#include "pmg_internal.h"
#include <nvtx3/nvToolsExt.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define PMG_MAX_LEVELS 32

struct pmg_vcycle {
  pmg_context *ctx;
  int n_levels, pre, post;
  pmg_operator *op[PMG_MAX_LEVELS];
  pmg_transfer *tr[PMG_MAX_LEVELS];
  pmg_chebyshev *sm[PMG_MAX_LEVELS];
  pmg_vector *sol[PMG_MAX_LEVELS], *rhs[PMG_MAX_LEVELS], *tmp[PMG_MAX_LEVELS], *res[PMG_MAX_LEVELS];
  int coarse_top;   /* levels 0 .. coarse_top run as one single-CTA kernel (csrc/pmg_coarse_cycle.h); -1 = none, -2 = undecided */
  int graph_enabled, calls;
  int nvtx_open;
  /* captured cycles, keyed by the (dst, src) pair they were captured for: the CG work vectors and a caller's own vectors
     alternate without re-capturing; when the cache is full the oldest entry goes (round robin) */
#define PMG_GRAPH_CACHE 4
  cudaGraphExec_t graph_exec[PMG_GRAPH_CACHE];
  const double *graph_dst[PMG_GRAPH_CACHE], *graph_src[PMG_GRAPH_CACHE];
  int graph_next;
  pmg_vector *host_dst, *host_src;
  double *pinned_in, *pinned_out;
  /* profiling */
  int profiling;
  int cur_level, cur_cat; /* the phase the last mark() opened */
  int n_marks;
  cudaEvent_t ev[4096];
  int mark_level[4096], mark_cat[4096];
};

enum { CAT_SMOOTH = 0, CAT_TRANSFER = 1, CAT_HALO = 2, CAT_OTHER = 3 };

/* NVTX ranges (visible to Nsight tools; a no-op without one): one per phase of a level while the cycle is enqueued kernel by
   kernel -- "pmg L<level> smooth | transfer | residual" -- and one around a replayed graph; CG iterations get their own. */
static void nvtx_phase(pmg_vcycle *v, int level, int cat)
{
  static const char *const names[] = {"smooth", "transfer", "halo", "residual+copy"};
  char buf[64];
  if (v->nvtx_open) nvtxRangePop();
  v->nvtx_open = 0;
  if (level < 0) return;
  snprintf(buf, sizeof(buf), "pmg L%d Q%d %s", level, v->op[level]->degree, names[cat < 0 || cat > 3 ? 3 : cat]);
  nvtxRangePushA(buf);
  v->nvtx_open = 1;
}

static int mark(pmg_vcycle *v, int level, int cat)
{
  nvtx_phase(v, level, cat);
  if (!v->profiling) return PMG_OK;
  if (cat != CAT_HALO) { v->cur_level = level; v->cur_cat = cat; }
  if (v->n_marks >= 4096) return PMG_OK;
  const int i = v->n_marks++;
  PMG_CUDA(cudaEventCreate(&v->ev[i]));
  PMG_CUDA(cudaEventRecord(v->ev[i], v->ctx->stream));
  v->mark_level[i] = level; v->mark_cat[i] = cat;
  return PMG_OK;
}

int pmg_vcycle_create(pmg_operator *const *ops, pmg_transfer *const *transfers, pmg_chebyshev *const *smoothers,
                      int n_levels, int pre, int post, pmg_vcycle **out)
{
  if (!ops || !smoothers || !out || n_levels < 1 || n_levels > PMG_MAX_LEVELS || pre < 0 || post < 0 || (n_levels > 1 && !transfers)) {
    pmg_set_error("vcycle_create: bad arguments");
    return PMG_ERR_ARG;
  }
  pmg_vcycle *v = (pmg_vcycle *)calloc(1, sizeof(*v));
  if (!v) return PMG_ERR_NOMEM;
  v->ctx = ops[0]->ctx; v->n_levels = n_levels; v->pre = pre; v->post = post;
  v->graph_enabled = 1;
  v->coarse_top = -2;
  for (int l = 0; l < n_levels; ++l) {
    if (!ops[l] || !smoothers[l] || smoothers[l]->op != ops[l] || (l > 0 && !transfers[l])) {
      pmg_set_error("vcycle_create: level %d is incomplete or its smoother belongs to another operator", l);
      free(v);
      return PMG_ERR_ARG;
    }
    if (l > 0 && (transfers[l]->coarse != ops[l - 1] || transfers[l]->fine != ops[l])) {
      pmg_set_error("vcycle_create: transfer %d does not connect levels %d and %d", l, l - 1, l);
      free(v);
      return PMG_ERR_ARG;
    }
    v->op[l] = ops[l]; v->tr[l] = (l > 0) ? transfers[l] : NULL; v->sm[l] = smoothers[l];
  }
  for (int l = 0; l < n_levels; ++l) {
    PMG_CHECK(pmg_vector_create_layout(v->ctx, &ops[l]->lay, &v->tmp[l]));
    PMG_CHECK(pmg_vector_create_layout(v->ctx, &ops[l]->lay, &v->res[l]));
    if (l < n_levels - 1) {
      PMG_CHECK(pmg_vector_create_layout(v->ctx, &ops[l]->lay, &v->sol[l]));
      PMG_CHECK(pmg_vector_create_layout(v->ctx, &ops[l]->lay, &v->rhs[l]));
    }
  }
  *out = v;
  return PMG_OK;
}

int pmg_vcycle_destroy(pmg_vcycle *v)
{
  if (!v) return PMG_OK;
  cudaStreamSynchronize(v->ctx->stream);
  for (int i = 0; i < PMG_GRAPH_CACHE; ++i)
    if (v->graph_exec[i]) cudaGraphExecDestroy(v->graph_exec[i]);
  for (int l = 0; l < v->n_levels; ++l) {
    pmg_vector_destroy(v->tmp[l]); pmg_vector_destroy(v->res[l]);
    pmg_vector_destroy(v->sol[l]); pmg_vector_destroy(v->rhs[l]);
  }
  pmg_vector_destroy(v->host_dst); pmg_vector_destroy(v->host_src);
  if (v->pinned_in) cudaFreeHost(v->pinned_in);
  if (v->pinned_out) cudaFreeHost(v->pinned_out);
  free(v);
  return PMG_OK;
}

int pmg_vcycle_set_graph(pmg_vcycle *v, int enable)
{
  if (!v) return PMG_ERR_ARG;
  v->graph_enabled = enable ? 1 : 0;
  return PMG_OK;
}

/* Which levels run inside the single-CTA coarse kernel (csrc/pmg_coarse_cycle.h): the longest prefix 0 .. L of levels of one
   degree, connected by geometric transfers, each wholly on this GPU, with DoFs x row length <= PMG_COARSE_MAX_WORK
   multiply-adds per apply.  OFF by default: measured on B200 (tools/coarse_sweep.py, profiles/r01_coarse_cycle_kernel_sweep.txt)
   the per-level kernels inside the CUDA graph (5.4 us per operation on the small levels) beat the single CTA at every bound
   -- C2 cycle 6.62 ms without it, 6.81 / 7.04 / 8.75 ms with levels up to 5^3 / 9^3 / 17^3 DoFs inside; one SM's gather loops
   with a block barrier and an L2 round trip per operation cost 8 us and more.  PMG_COARSE_KERNEL=1 enables it (kept for the
   next round: vectors in shared memory, a thread-block cluster instead of one CTA). */
#define PMG_COARSE_MAX_WORK 1.0e5
static void choose_coarse_top(pmg_vcycle *v)
{
  v->coarse_top = -1;
  const char *e = getenv("PMG_COARSE_KERNEL");
  if (!e || atoi(e) == 0) return;
  for (int l = 0; l < v->n_levels && l < 8; ++l) {
    const pmg_operator *op = v->op[l];
    if (!pmgk_coarse_cycle_supported(&op->lv) && op->lay.active) break;
    if (op->ctx->n_ranks > 1 && !op->lay.gathered) break;
    if (op->degree != v->op[0]->degree || op->coefficient != 0 || op->mapped || op->dim != 3) break;
    if (l > 0 && v->tr[l]->kind != 0) break;
    const double n1 = op->degree + 1;
    const char *w = getenv("PMG_COARSE_MAX_WORK");
    if ((double)op->lay.n_global * 8.0 * n1 * n1 * n1 > (w ? atof(w) : PMG_COARSE_MAX_WORK)) break;
    v->coarse_top = l;
  }
}

static int coarse_cycle(pmg_vcycle *v, int top, pmg_vector *u, const pmg_vector *rhs)
{
  if (!v->op[top]->lay.active) return PMG_OK; /* gathered levels live on rank 0 */
  pmgk_coarse_level cl[8];
  for (int l = 0; l <= top; ++l) {
    cl[l].lv = &v->op[l]->lv;
    cl[l].cheb_degree = v->sm[l]->degree; cl[l].theta = v->sm[l]->theta; cl[l].delta = v->sm[l]->delta;
    cl[l].sol = (l == top) ? u->d : v->sol[l]->d;
    cl[l].rhs = (l == top) ? rhs->d : v->rhs[l]->d;
    cl[l].tmp = v->tmp[l]->d; cl[l].res = v->res[l]->d;
  }
  double P[(PMG_MAX_DEGREE + 1) * (2 * PMG_MAX_DEGREE + 1)];
  pmg_fe_prolongation_h(v->op[0]->degree, P);
  return pmgk_coarse_cycle(cl, top + 1, v->pre, v->post, P, v->ctx->stream);
}

/* v_cycle (:128-190).  u holds the iterate on entry unless zero_guess; on return u holds the result. */
static int v_cycle(pmg_vcycle *v, int level, pmg_vector *u, const pmg_vector *rhs, int zero_guess)
{
  pmg_vector *cur = u, *other = v->tmp[level], *r = NULL;
  if (level == v->coarse_top && zero_guess) {
    PMG_CHECK(mark(v, level, CAT_SMOOTH));
    return coarse_cycle(v, level, u, rhs);
  }
  if (level == 0) {
    /* coarsest level: one smooth() (:148-154) */
    PMG_CHECK(mark(v, level, CAT_SMOOTH));
    PMG_CHECK(pmg_chebyshev_smooth(v->sm[0], cur, rhs, other, zero_guess, &r));
    if (r != u) PMG_CHECK(pmg_vector_copy(u, r));
    return PMG_OK;
  }
  /* pre-smoothing (:157-160) */
  PMG_CHECK(mark(v, level, CAT_SMOOTH));
  int zg = zero_guess;
  /* Slabs with neighbours: smooth, smooth, residual are one chain of applies, each reading what the one before wrote; every
     apply pushes its boundary planes into the neighbours' ghost planes itself (fused compute + exchange), so the chain needs
     ONE ghost exchange, before its first apply (pmg_smoother.c, pmg_operator.c: pmg_apply_chained) */
  int pushed = 0;
  for (int s = 0; s < v->pre; ++s) {
    PMG_CHECK(pmg_chebyshev_smooth_chain(v->sm[level], cur, rhs, other, zg, &r, pushed, 1, &pushed));
    if (r != cur) { other = cur; cur = r; }
    zg = 0;
  }
  /* residual = src - A dst (:163-166), restricted to the next coarser level (:169-172) */
  PMG_CHECK(mark(v, level, CAT_OTHER));
  if (zg) PMG_CHECK(pmg_vector_copy(v->res[level], rhs)); /* no pre-smoothing and u = 0: residual = rhs */
  else if (pushed) PMG_CHECK(pmg_apply_chained(v->op[level], PMGK_RESIDUAL, cur->d, rhs->d, NULL, v->res[level]->d, 0.0, 0.0, 1, 0));
  else PMG_CHECK(pmg_laplace_operator_residual(v->op[level], v->res[level], rhs, cur));
  PMG_CHECK(mark(v, level, CAT_TRANSFER));
  PMG_CHECK(pmg_vector_set(v->rhs[level - 1], 0.0));
  PMG_CHECK(pmg_transfer_restrict_and_add(v->tr[level], v->rhs[level - 1], v->res[level]));
  /* coarse correction from a zero guess (:175-179) */
  PMG_CHECK(v_cycle(v, level - 1, v->sol[level - 1], v->rhs[level - 1], 1));
  /* prolongate and add (:182) */
  PMG_CHECK(mark(v, level, CAT_TRANSFER));
  if (zg) { PMG_CHECK(pmg_vector_set(cur, 0.0)); zg = 0; }
  PMG_CHECK(pmg_transfer_prolongate_and_add(v->tr[level], cur, v->sol[level - 1]));
  /* post-smoothing (:185-188) */
  PMG_CHECK(mark(v, level, CAT_SMOOTH));
  pushed = 0;
  for (int s = 0; s < v->post; ++s) {
    PMG_CHECK(pmg_chebyshev_smooth_chain(v->sm[level], cur, rhs, other, 0, &r, pushed, s + 1 < v->post, &pushed));
    if (r != cur) { other = cur; cur = r; }
  }
  PMG_CHECK(mark(v, level, CAT_OTHER));
  if (cur != u) PMG_CHECK(pmg_vector_copy(u, cur));
  return PMG_OK;
}

static int ensure_initialized(pmg_vcycle *v)
{
  for (int l = 0; l < v->n_levels; ++l)
    if (!v->sm[l]->initialized) PMG_CHECK(pmg_chebyshev_estimate(v->sm[l]));
  if (v->coarse_top == -2) choose_coarse_top(v);
  return PMG_OK;
}

int pmg_vcycle_vmult(pmg_vcycle *v, pmg_vector *dst, const pmg_vector *src)
{
  if (v) PMG_CHECK(pmg_enter(v->ctx));
  if (!v || !dst || !src || dst == src) { pmg_set_error("vcycle_vmult: bad arguments"); return PMG_ERR_ARG; }
  const int top = v->n_levels - 1;
  if (!pmg_layout_same(&dst->lay, &v->op[top]->lay) || !pmg_layout_same(&src->lay, &v->op[top]->lay)) {
    pmg_set_error("vcycle_vmult: vectors are not initialised for the finest level");
    return PMG_ERR_ARG;
  }
  PMG_CHECK(ensure_initialized(v));
  pmg_context *ctx = v->ctx;
  pmg_p2p_forget(ctx); /* a captured cycle's first exchange must not rely on what preceded the capture */
  /* dst = 0 (:92) is implied: the cycle starts from a zero guess */
  if (!v->graph_enabled || v->profiling) {
    const int rc = v_cycle(v, top, dst, src, 1);
    nvtx_phase(v, -1, 0);
    return rc;
  }
  for (int i = 0; i < PMG_GRAPH_CACHE; ++i)
    if (v->graph_exec[i] && v->graph_dst[i] == dst->d && v->graph_src[i] == src->d) {
      nvtxRangePushA("pmg V-cycle (graph replay)");
      const cudaError_t ge = cudaGraphLaunch(v->graph_exec[i], ctx->stream);
      nvtxRangePop();
      pmg_p2p_forget(ctx);
      PMG_CUDA(ge);
      pmg_count_launch(1);
      return PMG_OK;
    }
  if (v->calls++ == 0) { /* warm-up: sets kernel attributes outside capture */
    const int rc0 = v_cycle(v, top, dst, src, 1);
    nvtx_phase(v, -1, 0);
    return rc0;
  }
  const int slot = v->graph_next;
  v->graph_next = (slot + 1) % PMG_GRAPH_CACHE;
  if (v->graph_exec[slot]) { cudaGraphExecDestroy(v->graph_exec[slot]); v->graph_exec[slot] = NULL; }
  cudaGraph_t graph = NULL;
  PMG_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  const int rc = v_cycle(v, top, dst, src, 1);
  nvtx_phase(v, -1, 0);
  cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
  if (rc != PMG_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    v->graph_enabled = 0; /* fall back to plain stream launches of the same kernels */
    return v_cycle(v, top, dst, src, 1);
  }
  ce = cudaGraphInstantiate(&v->graph_exec[slot], graph, 0);
  cudaGraphDestroy(graph);
  if (ce != cudaSuccess) { cudaGetLastError(); v->graph_exec[slot] = NULL; v->graph_enabled = 0; return v_cycle(v, top, dst, src, 1); }
  v->graph_dst[slot] = dst->d; v->graph_src[slot] = src->d;
  pmg_p2p_forget(ctx);
  PMG_CUDA(cudaGraphLaunch(v->graph_exec[slot], ctx->stream));
  pmg_count_launch(1);
  return PMG_OK;
}

int pmg_vcycle_vmult_host(pmg_vcycle *v, double *dst_host, const double *src_host)
{
  if (!v || !dst_host || !src_host) return PMG_ERR_ARG;
  const int top = v->n_levels - 1;
  if (!v->host_dst) {
    PMG_CHECK(pmg_vector_create_layout(v->ctx, &v->op[top]->lay, &v->host_dst));
    PMG_CHECK(pmg_vector_create_layout(v->ctx, &v->op[top]->lay, &v->host_src));
  }
  PMG_CHECK(pmg_vector_import_host(v->host_src, src_host));
  PMG_CHECK(pmg_vcycle_vmult(v, v->host_dst, v->host_src));
  return pmg_vector_export_host(v->host_dst, dst_host);
}

int pmg_vcycle_vmult_host_owned(pmg_vcycle *v, double *dst_host_owned, const double *src_host_owned)
{
  if (!v || !dst_host_owned || !src_host_owned) return PMG_ERR_ARG;
  const int top = v->n_levels - 1;
  if (!v->host_dst) {
    PMG_CHECK(pmg_vector_create_layout(v->ctx, &v->op[top]->lay, &v->host_dst));
    PMG_CHECK(pmg_vector_create_layout(v->ctx, &v->op[top]->lay, &v->host_src));
  }
  PMG_CHECK(pmg_vector_import_owned(v->host_src, src_host_owned));
  PMG_CHECK(pmg_vcycle_vmult(v, v->host_dst, v->host_src));
  return pmg_vector_export_owned(v->host_dst, dst_host_owned);
}

/* ghost exchanges inside a phase are booked to the level's halo column: device time between the exchange's enqueue points on
   the compute stream, so it includes waiting for the neighbour ranks to arrive */
static void profile_halo_hook(void *user, int begin)
{
  pmg_vcycle *v = (pmg_vcycle *)user;
  if (!v->profiling || v->cur_cat < 0) return;
  if (begin) (void)mark(v, v->cur_level, CAT_HALO);
  else (void)mark(v, v->cur_level, v->cur_cat);
}

int pmg_vcycle_profile(pmg_vcycle *v, pmg_vector *dst, const pmg_vector *src, double *out_ms, int cap_levels)
{
  if (!v || !out_ms || cap_levels < v->n_levels) return PMG_ERR_ARG;
  PMG_CHECK(ensure_initialized(v));
  memset(out_ms, 0, sizeof(double) * 4 * cap_levels);
  v->profiling = 1; v->n_marks = 0; v->cur_cat = -1;
  v->ctx->halo_hook = profile_halo_hook; v->ctx->halo_hook_user = v;
  int rc = pmg_vcycle_vmult(v, dst, src);
  v->ctx->halo_hook = NULL; v->ctx->halo_hook_user = NULL;
  if (!rc) rc = mark(v, 0, -1);
  v->profiling = 0;
  if (rc) return rc;
  PMG_CUDA(cudaStreamSynchronize(v->ctx->stream));
  for (int i = 0; i + 1 < v->n_marks; ++i) {
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, v->ev[i], v->ev[i + 1]));
    out_ms[v->mark_level[i] * 4 + v->mark_cat[i]] += ms;
  }
  for (int i = 0; i < v->n_marks; ++i) cudaEventDestroy(v->ev[i]);
  v->n_marks = 0;
  return PMG_OK;
}

/* ---- SolverCG ----------------------------------------------------------------------------- */
int pmg_cg_solve(const pmg_operator *A, pmg_vector *x, const pmg_vector *b, pmg_vcycle *precond,
                 int max_it, double tol, int *last_step, double *history, int history_cap)
{
  if (A) PMG_CHECK(pmg_enter(A->ctx));
  if (!A || !x || !b || max_it < 0) { pmg_set_error("cg_solve: bad arguments"); return PMG_ERR_ARG; }
  if (!pmg_layout_same(&x->lay, &A->lay) || !pmg_layout_same(&b->lay, &A->lay)) {
    pmg_set_error("cg_solve: vectors are not initialised for the operator");
    return PMG_ERR_ARG;
  }
  pmg_context *ctx = A->ctx;
  const pmg_layout *l = &A->lay;
  /* work vectors live with the operator (the reference's SolverCG keeps them in a GrowingVectorMemory pool): a
     cudaMalloc / cudaFree pair of four fine-level vectors per solve costs more than the iterations at C2 */
  pmg_operator *Aw = (pmg_operator *)A;
  for (int i = 0; i < 4; ++i)
    if (!Aw->cg_ws[i]) PMG_CHECK(pmg_vector_create_layout(ctx, l, &Aw->cg_ws[i]));
  pmg_vector *r = Aw->cg_ws[0], *z = Aw->cg_ws[1], *p = Aw->cg_ws[2], *Ap = Aw->cg_ws[3];
  int it = 0, converged = 0, rc = PMG_OK;
  double res = 0.0;
  /* device scalars of the iteration (slots of ctx->scalars): the host reads back ONE number per iteration, ||r||^2 */
  enum { S_RR = 0, S_ALPHA = 8, S_RZ = 16, S_PAP = 17, S_RZNEW = 18, S_BETA = 19 };
  double *S = ctx->scalars;
#define CG(call) do { rc = (call); if (rc != PMG_OK) goto done; } while (0)
#define CGC(call) do { if ((call) != cudaSuccess) { rc = PMG_ERR_CUDA; goto done; } } while (0)
  /* r = b - A x; convergence check before the first iteration */
  CG(pmg_laplace_operator_residual(A, r, b, x));
  CG(pmg_vector_l2_norm(r, &res));
  if (history && history_cap > 0) history[0] = res;
  if (res <= tol) converged = 1;
  if (!converged) {
    if (precond) CG(pmg_vcycle_vmult(precond, z, r)); else CG(pmg_vector_copy(z, r));
    CG(pmg_vector_copy(p, z));
    CG(pmg_vector_dot_device(r, z, S_RZ));
  }
  while (!converged && it < max_it) {
    ++it;
    CG(pmg_laplace_operator_vmult(A, Ap, p));
    CG(pmg_vector_dot_device(p, Ap, S_PAP));
    CG(pmgk_scalar_div(S + S_ALPHA, S + S_RZ, S + S_PAP, ctx->stream)); /* alpha = r.z / p.Ap */
    /* x += alpha p; r -= alpha Ap; ||r||^2 in one pass over the owned planes (ghost planes are refreshed before they are read) */
    if (l->active) {
      const int64_t lo = l->plane * (l->z_own_lo - l->z0), n_own = l->plane * (l->z_own_hi - l->z_own_lo);
      CG(pmgk_cg_update_xr(x->d + lo, r->d + lo, p->d + lo, Ap->d + lo, S + S_ALPHA, n_own, S + S_RR, ctx->work, ctx->stream));
    } else {
      CGC(cudaMemsetAsync(S + S_RR, 0, sizeof(double), ctx->stream));
    }
    CG(pmg_allreduce_sum(ctx, S + S_RR, 1));
    /* the one host round trip of the iteration: SolverCG compares ||r|| with the tolerance before it preconditions again */
    CGC(cudaMemcpyAsync(ctx->h_scalars + S_RR, S + S_RR, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CGC(cudaStreamSynchronize(ctx->stream));
    res = sqrt(ctx->h_scalars[S_RR]);
    if (history && it < history_cap) history[it] = res;
    if (res <= tol) { converged = 1; break; }
    if (precond) CG(pmg_vcycle_vmult(precond, z, r)); else CG(pmg_vector_copy(z, r));
    CG(pmg_vector_dot_device(r, z, S_RZNEW));
    CG(pmgk_scalar_div(S + S_BETA, S + S_RZNEW, S + S_RZ, ctx->stream)); /* beta = r.z (new) / r.z (old) */
    if (l->active) CG(pmgk_cg_update_p(p->d, z->d, S + S_BETA, l->n_local, ctx->stream)); /* p = z + beta p */
    CGC(cudaMemcpyAsync(S + S_RZ, S + S_RZNEW, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  }
#undef CGC
#undef CG
done:
  if (last_step) *last_step = it;
  if (rc != PMG_OK) return rc;
  if (!converged) { pmg_set_error("CG did not converge in %d iterations (residual %g, tolerance %g)", it, res, tol); return PMG_ERR_NOT_CONVERGED; }
  return PMG_OK;
}

int pmg_microbench(pmg_context *ctx, double *fma, double *dmma, double *hbm)
{
  if (!ctx) return PMG_ERR_ARG;
  PMG_CUDA(cudaSetDevice(ctx->device));
  if (fma) PMG_CHECK(pmgk_bench_fp64_fma(fma, ctx->stream));
  if (dmma) PMG_CHECK(pmgk_bench_fp64_dmma(dmma, ctx->stream));
  if (hbm) PMG_CHECK(pmgk_bench_hbm_copy(hbm, ctx->stream));
  return PMG_OK;
}

/* ---- host-only helpers ------------------------------------------------------------------------ */
int pmg_host_fastdiag_tables(int degree, double *S, double *lam)
{
  if (degree < 1 || degree > PMG_MAX_DEGREE || !S || !lam) return PMG_ERR_ARG;
  pmg_fe_fastdiag(degree, S, lam);
  return PMG_OK;
}

int pmg_host_pencil(int degree, double *M, double *K)
{
  if (degree < 1 || degree > PMG_MAX_DEGREE || !M || !K) return PMG_ERR_ARG;
  pmg_fe_pencil(degree, M, K);
  return PMG_OK;
}

int pmg_host_support_points(int degree, double *x)
{
  if (degree < 1 || degree > PMG_MAX_DEGREE || !x) return PMG_ERR_ARG;
  pmg_fe_gll(degree + 1, x);
  return PMG_OK;
}

int pmg_host_prolongation_1d(int kind, int degree_coarse, int degree_fine, double *P)
{
  if (!P || degree_coarse < 1 || degree_coarse > PMG_MAX_DEGREE) return PMG_ERR_ARG;
  if (kind == 0) { pmg_fe_prolongation_h(degree_coarse, P); return PMG_OK; }
  if (degree_fine <= degree_coarse || degree_fine > PMG_MAX_DEGREE) return PMG_ERR_ARG;
  pmg_fe_prolongation_p(degree_coarse, degree_fine, P);
  return PMG_OK;
}
