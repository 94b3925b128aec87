/*
 * pmg_kernels.h -- thin C-ABI between the C host layer (portable-multigrid_b200/host)
 * and the hand-written sm_100a CUDA kernels (portable-multigrid_b200/csrc).
 *
 * Plain pointers and sizes only; every function enqueues work on `stream`
 * (a cudaStream_t passed as void*) and returns 0 or a negative pmg error code.
 * Device pointers unless stated otherwise.  No CPU fallback exists behind any entry.
 */
#ifndef PMG_KERNELS_H
#define PMG_KERNELS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMGK_MAX_N1 10

/* One multigrid level as the kernels see it (structured box, lexicographic dofs). */
typedef struct pmgk_level {
  int dim;               /* 3, or 2: one dof plane (Nz = 1, nz = 1 as a placeholder), faces bits 0..3, kernels of csrc/pmg_dim2.cu */
  int degree;
  int nx, ny, nz;        /* global cells */
  int Nx, Ny, Nz;        /* global dofs per direction */
  unsigned faces;        /* Dirichlet faces bitmask */
  int z0, nzl;           /* local plane l holds global plane z0 + l */
  int cz_lo, cz_hi;      /* owned cell layers */
  int z_own_lo, z_own_hi;/* owned dof planes */
  double h[3];
  double S[PMGK_MAX_N1 * PMGK_MAX_N1]; /* nodal -> pencil eigenbasis, row a, column i (n1 x n1) */
  double lam[PMGK_MAX_N1];
  double Mref[PMGK_MAX_N1 * PMGK_MAX_N1]; /* 1-D cell mass matrix of FE_Q(p) on [0,1] with QGauss(p+1) (n1 x n1) */
  double Kref[PMGK_MAX_N1 * PMGK_MAX_N1]; /* 1-D cell stiffness matrix */
  const double *dinv_tab;  /* device, (p+2)^3 */
  const double *dinv_vec;  /* device, local vector or NULL */
  int tile_variant;        /* tuning knob: 0 = default choice per level; 1 = line-marching kernel; 2, 3 = cell-tile kernel, small/large tiles; 4, 5 = pipelined line-marching kernel (experimental; 5: fused modes without shared-memory boxes for b / x_old) */
  /* variable coefficient -div(a grad u) (BASELINE config 5; NULL = the reference's constant-coefficient operator):
     w_q a(x_q) on the lexicographic grid of all quadrature points, (nx n1) x (ny n1) x ((cz_hi - coef_cz0) n1), x fastest */
  const double *coef;
  int coef_cz0;            /* first cell layer stored in coef (= z0 / degree) */
  double Sq[PMGK_MAX_N1 * PMGK_MAX_N1];  /* shape values phi_i(x_q), row q (Gauss point), column i (n1 x n1) */
  double Dco[PMGK_MAX_N1 * PMGK_MAX_N1]; /* co_shape_gradients: derivative of Gauss-point Lagrange basis r at Gauss point q */
  /* mapped geometry (0 = the box's affine cells): coef then holds six grids of the layout above, geo_stride doubles apart --
     the entries xx, xy, xz, yy, yz, zz of  G_q = w_q a(x_q) |det J_q| J_q^-1 J_q^-T  of the cells' trilinear or curved maps */
  int64_t geo_stride;
} pmgk_level;

enum { PMGK_APPLY = 0, PMGK_RESIDUAL = 1, PMGK_CHEB_FIRST = 2, PMGK_CHEB_STEP = 3 };

/* K1 fused: out = epilogue(A u); replaces LaplaceOperator::vmult (+ smoother update)
   (reference include/operators/portable_laplace_operator.h:557-719) */
int pmgk_apply(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
               double *out, double f1, double f2, void *stream);
/* The same launch in two parts, for slabs with neighbours: PMGK_PART_INTERIOR = the z-chunks that read no ghost plane,
   PMGK_PART_BOUNDARY = the first and the last chunk.  INTERIOR + BOUNDARY write exactly what PMGK_PART_ALL writes.
   pmgk_apply_splits: 1 if the level's launch can be split (line-marching kernel, >= 3 chunks). */
enum { PMGK_PART_ALL = 0, PMGK_PART_INTERIOR = 1, PMGK_PART_BOUNDARY = 2 };
int pmgk_apply_part(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                    double *out, double f1, double f2, int part, void *stream);
int pmgk_apply_splits(const pmgk_level *lv, int mode);
/* Fused compute + ghost exchange (plane-per-step kernel, slabs with neighbours): the launch stores its boundary planes of
   `out` straight into the neighbours' ghost planes over NVLink (push != 0) and, with consume != 0, takes u's ghost planes as
   already pushed by the neighbours' previous fused launch (its boundary chunks wait for their flag; no exchange of u before
   the launch).  out_lower / out_upper: the neighbours' copies of `out` as mapped here (NULL: no neighbour), lower_z0 /
   upper_z0: their first stored planes; mailbox*: 16 flag words per rank, zero-initialised (words 8..11 are used here).
   Every rank must issue the same sequence of fused launches.  Replaces update_ghost_values() + vmult of the reference
   (include/operators/portable_laplace_operator.h:635-661) inside the smoother.
   pmgk_apply_can_push: 1 if the level's launch supports it. */
typedef struct pmgk_push {
  double *out_lower, *out_upper;
  int lower_z0, upper_z0;
  void *mailbox, *mailbox_lower, *mailbox_upper;
  int push, consume;
} pmgk_push;
int pmgk_apply_push(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold,
                    double *out, double f1, double f2, const pmgk_push *push, void *stream);
int pmgk_apply_can_push(const pmgk_level *lv, int mode);
/* number of kernel launches pmgk_apply issues (1) and the launch geometry it would use */
int pmgk_apply_geometry(const pmgk_level *lv, int *grid, int *block, int *smem_bytes, int *n_chunks);

/* variable-coefficient set-up (csrc/pmg_apply_var.cu).  kind 1: a(x) = 1 / (0.05 + 2 |x|^2); gq / gw: HOST arrays, the
   n1 Gauss points / weights on [0,1].  coef: device, pmgk_var_coef_doubles(lv) doubles. */
int64_t pmgk_var_coef_doubles(const pmgk_level *lv);
int pmgk_var_fill_coef(const pmgk_level *lv, int kind, const double *gq, const double *gw, double *coef, void *stream);
/* inverse diagonal of the variable-coefficient operator on all stored planes (1 on constrained dofs);
   S2 / G2: HOST n1 x n1 tables, squared shape values / squared nodal shape gradients at the Gauss points, row q */
int pmgk_var_fill_dinv(const pmgk_level *lv, const double *S2, const double *G2, double *dinv, void *stream);

/* mapped-geometry set-up (csrc/pmg_apply_geo.cu).  k: the geometry degree, 1 = trilinear cells, 2 .. PMGK_MAX_N1-1 = curved
   cells, each the Lagrange interpolant of degree k through (k+1)^3 nodes at the Gauss-Lobatto points (MappingQ(k)).  vert:
   device, the node planes k coef_cz0 .. k cz_hi of the level, (nx k+1) x (ny k+1) points per plane, x fastest, (x, y, z)
   interleaved (k = 1: the vertex planes); kind 0: a = 1, 1: the C5 coefficient at the mapped point; gq / gw: HOST Gauss
   points / weights on [0,1]; geo: device, 6 pmgk_var_coef_doubles(lv) doubles (lv->geo_stride must be
   pmgk_var_coef_doubles(lv)).  err: device word, ~0 on entry; on return (when the stream has run) it holds the smallest
   global index cx + nx (cy + ny cz) of a cell with det J <= 0 at a Gauss point or a non-finite node, else ~0. */
int pmgk_geo_fill(const pmgk_level *lv, int k, int kind, const double *vert, const double *gq, const double *gw, double *geo,
                  unsigned long long *err, void *stream);
/* inverse diagonal of the mapped operator; S2 / G2 as pmgk_var_fill_dinv, SG: HOST table S(q,i) G(q,i) */
int pmgk_geo_fill_dinv(const pmgk_level *lv, const double *S2, const double *G2, const double *SG, double *dinv, void *stream);

/* load vector of f = 1 on the mapped mesh on all stored planes (constrained rows 0; a ghost plane holds the part of the
   stored cells only): k, vert as pmgk_geo_fill; S: HOST n1 x n1 shape values [q][i], gq / gw: HOST Gauss points / weights;
   W: device scratch of pmgk_var_coef_doubles(lv) doubles */
int pmgk_geo_rhs(const pmgk_level *lv, int k, const double *vert, const double *S, const double *gq, const double *gw, double *W,
                 double *rhs, void *stream);
/* integral of u^2 over each owned cell of the mapped mesh with QGauss(p+2): cell_sums[c], c = cx + nx (cy + ny (cz - cz_lo));
   k, vert as pmgk_geo_fill; E: HOST (p+2) x (p+1) values phi_i(x_q), gq / gw: HOST the p+2 Gauss points / weights; u: local
   vector, ghosts current */
int pmgk_geo_norm_cells(const pmgk_level *lv, int k, const double *vert, const double *E, const double *gq, const double *gw,
                        const double *u, double *cell_sums, void *stream);

/* inverse diagonal as an explicit vector (LaplaceOperator::compute_diagonal, :752-917) */
int pmgk_fill_dinv(const pmgk_level *lv, double *dinv, void *stream);
/* out = f * Dinv * b (first Chebyshev step from a zero guess) */
int pmgk_scale_dinv(const pmgk_level *lv, double f, const double *b, double *out, void *stream);

/* BLAS-1 on local vectors (LinearAlgebra::distributed::Vector ops used on the path, SURVEY a11) */
int pmgk_set(double *x, double a, int64_t n, void *stream);
int pmgk_copy(double *dst, const double *src, int64_t n, void *stream);
int pmgk_axpby(double *out, double a, const double *x, double b, const double *y, int64_t n, void *stream); /* out = a x + b y */
int pmgk_scale(double *x, double a, int64_t n, void *stream);
/* result[0] = sum x_i y_i over [0,n): deterministic two-stage reduction; work >= pmgk_dot_work_doubles() */
int pmgk_dot(const double *x, const double *y, int64_t n, double *result, double *work, void *stream);
int pmgk_sum(const double *x, int64_t n, double *result, double *work, void *stream);
int pmgk_dot_work_doubles(void);
/* CG fused updates: x += alpha p, r -= alpha Ap, result[0] = r.r  (alpha read from device) */
int pmgk_cg_update_xr(double *x, double *r, const double *p, const double *Ap, const double *alpha_dev,
                      int64_t n, double *result, double *work, void *stream);
/* p = z + beta p (beta read from device) */
int pmgk_cg_update_p(double *p, const double *z, const double *beta_dev, int64_t n, void *stream);
/* tiny device-scalar helper: out[0] = num[0] / den[0] */
int pmgk_scalar_div(double *out, const double *num, const double *den, void *stream);
/* out[(z * Ny + y) * Nx + x] = lx[x] * ly[y] * lz[z] over nz local planes (lx, ly, lz device arrays): tensor-product
   load vector of the drivers' right-hand side (program.cc:289-334) */
int pmgk_outer3(double *out, const double *lx, const double *ly, const double *lz, int Nx, int Ny, int nz, void *stream);
/* x_i = ((first_global + i) mod 11), Chebyshev eigenvalue-estimate start vector */
int pmgk_set_mod11(double *x, int64_t first_global, int64_t n, void *stream);

/* The coarse part of the V-cycle -- levels[0 .. n_levels) coarse -> fine, one degree, geometric transfers, each wholly on this
   GPU -- as one single-CTA kernel (csrc/pmg_coarse_cycle.h): v_cycle(levels[n_levels-1]) from a zero guess, sol <- cycle(rhs),
   with the operations of VCycleMultigrid::v_cycle / smooth (include/multigrid/portable_v_cycle_multigrid.h:96-190).
   P1d_host: HOST (p+1) x (2p+1) h-prolongation matrix. */
typedef struct pmgk_coarse_level {
  const pmgk_level *lv;
  int cheb_degree;       /* smoother degree and parameters of the level */
  double theta, delta;
  double *sol, *rhs, *tmp, *res; /* device vectors of the level */
} pmgk_coarse_level;
int pmgk_coarse_cycle_supported(const pmgk_level *lv);
int pmgk_coarse_cycle(const pmgk_coarse_level *levels, int n_levels, int pre, int post, const double *P1d_host, void *stream);

/* transfers (K4-K7).  kind 0 = geometric (fine mesh = coarse refined once, same degree),
   kind 1 = polynomial (same mesh, degree pc < pf).  P1d: device, (pc+1) x nf1 row-major,
   nf1 = 2p+1 (h) or pf+1 (p).  scratch: device doubles, >= pmgk_restrict_scratch_doubles(). */
int pmgk_prolongate_and_add(int kind, const pmgk_level *coarse, const pmgk_level *fine, const double *P1d,
                            double *dst_fine, const double *src_coarse, void *stream);
int pmgk_restrict_and_add(int kind, const pmgk_level *coarse, const pmgk_level *fine, const double *P1d,
                          double *dst_coarse, const double *src_fine, double *scratch, void *stream);
int64_t pmgk_restrict_scratch_doubles(int kind, const pmgk_level *coarse, const pmgk_level *fine);

/* ghost planes of a z-slab over NVLink peer memory (csrc/pmg_halo.cu): this rank's boundary planes are stored into the
   neighbours' ghost planes -- peer_lower[dst_in_lower + i] = mine[src_to_lower + i], i < n_to_lower (NULL peer: no neighbour),
   likewise upper -- ordered by flags; mailbox: this rank's six 64-bit flag words (device, zero-initialised),
   mailbox_lower / _upper: the neighbours' mailboxes as mapped here; need_ready: first wait until the neighbours no longer read the
   ghost planes that are about to be overwritten (required when the previous exchange was on the same vector).  When the kernel
   ends this rank's ghost planes are current. */
int pmgk_halo_push(const double *mine, double *peer_lower, double *peer_upper, int64_t n_to_lower, int64_t src_to_lower,
                   int64_t dst_in_lower, int64_t n_to_upper, int64_t src_to_upper, int64_t dst_in_upper, void *mailbox,
                   void *mailbox_lower, void *mailbox_upper, int need_ready, void *stream);

/* device properties the host layer needs */
int pmgk_device_sm_count(void);
/* FP64 microbenchmarks (roofline denominators): returns TFLOP/s */
int pmgk_bench_fp64_fma(double *tflops, void *stream);
int pmgk_bench_fp64_dmma(double *tflops, void *stream);
int pmgk_bench_hbm_copy(double *gbs, void *stream);

#ifdef __cplusplus
}
#endif
#endif
