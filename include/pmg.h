/*
 * pmg.h -- C-ABI of the B200-native matrix-free multigrid hot path.
 *
 * Drop-in boundary for dealii-X/portable-multigrid's operator / transfer / V-cycle
 * interfaces.  The reference has no C API: its boundary is three C++ abstract classes.
 * Each entry point below mirrors one virtual (or the constructor) of those classes and
 * cites it; INTEGRATION.md shows the adapter a reference maintainer would write.
 *
 *   LaplaceOperatorBase<dim,number>   include/base/portable_laplace_operator_base.h:16-60
 *   MGTransferBase<dim,number>        include/base/portable_mg_transfer_base.h:15-38
 *   VCycleMultigrid<dim,number,T>     include/multigrid/portable_v_cycle_multigrid.h:26-63
 *   PreconditionChebyshev / SolverCG / LinearAlgebra::distributed::Vector (deal.II, un-vendored):
 *     call sites source/geometric_multigrid/program.cc:267-285, 342-355
 *
 * Conventions: opaque handles; every call returns 0 (PMG_OK) or a negative error code and
 * never throws; pmg_last_error() gives a message for the calling thread's last failure;
 * one host thread per context (the reference runs one thread per rank, program.cc:452);
 * all device work is stream-ordered on the context's stream and asynchronous to the host
 * unless a value is returned to the host; pmg_sync() waits for it.  Vectors are
 * caller-owned; operators, transfers, smoothers and V-cycles hold non-owning references to
 * the objects they were created from (as the reference's ObserverPointers do).
 * There is no CPU fallback: without a CUDA device every compute entry returns PMG_ERR_CUDA.
 *
 * Mesh: the reference takes a deal.II DoFHandler + AffineConstraints; its drivers only ever
 * build the unit hyper-cube, uniformly refined, homogeneous Dirichlet on boundary id 0.
 * This library generates exactly that family itself: a structured box of nx*ny*nz cells of
 * FE_Q(degree), DoFs numbered lexicographically (x fastest), Dirichlet faces chosen by a
 * bitmask.  Host import/export use that global lexicographic order on every rank.
 */
#ifndef PMG_H
#define PMG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMG_OK 0
#define PMG_ERR_ARG (-1)          /* invalid argument / incompatible objects (reference: Assert) */
#define PMG_ERR_CUDA (-2)         /* CUDA runtime failure or no device */
#define PMG_ERR_UNSUPPORTED (-3)  /* degree/dimension outside the compiled range (reference: dispatch() == false) */
#define PMG_ERR_NOMEM (-4)
#define PMG_ERR_NCCL (-5)
#define PMG_ERR_NOT_CONVERGED (-6)/* SolverControl::NoConvergence */
#define PMG_ERR_STATE (-7)        /* e.g. diagonal requested before compute_diagonal (reference: ExcNotInitialized) */

#define PMG_MAX_DEGREE 9          /* = the reference dispatcher's max_degree (portable_laplace_operator_base.h:65) */
#define PMG_ALL_FACES 0x3Fu
#define PMG_INVALID_DEGREE (-1)   /* numbers::invalid_unsigned_int for the Chebyshev degree */

typedef struct pmg_context pmg_context;
typedef struct pmg_vector pmg_vector;
typedef struct pmg_operator pmg_operator;
typedef struct pmg_transfer pmg_transfer;
typedef struct pmg_chebyshev pmg_chebyshev;
typedef struct pmg_vcycle pmg_vcycle;

const char *pmg_last_error(void);
const char *pmg_version(void);

/* ---- context (MPI_InitFinalize + Kokkos execution space of the reference, program.cc:452) ---- */
/* Single-GPU context on CUDA device `device`. */
int pmg_context_create(pmg_context **ctx, int device);
/* One rank of an n_ranks job (one process per GPU).  nccl_id: the 128-byte ncclUniqueId obtained
   from pmg_nccl_unique_id() on rank 0 and broadcast by the launcher (torch.distributed / MPI / file). */
int pmg_context_create_distributed(pmg_context **ctx, int device, int rank, int n_ranks, const void *nccl_id);
int pmg_nccl_unique_id(void *out128);
int pmg_context_destroy(pmg_context *ctx);
int pmg_sync(pmg_context *ctx);
int pmg_context_rank(const pmg_context *ctx, int *rank, int *n_ranks);
/* levels with fewer global DoFs than this are kept on rank 0 only (replaces the commented-out
   MinimalGranularityPolicy, program.cc:139-142); default 262144 */
int pmg_context_set_coarse_threshold(pmg_context *ctx, int64_t n_dofs);
void *pmg_context_stream(pmg_context *ctx); /* cudaStream_t */
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t pmg_context_launch_count(const pmg_context *ctx);
/* applies launched so far that exchanged ghost planes by the fused push (no exchange of their own), see pmg_chebyshev_vmult */
int64_t pmg_context_fused_halo_count(const pmg_context *ctx);

/* ---- LaplaceOperator (include/operators/portable_laplace_operator.h:383-461) ---- */
/* ctor (DoFHandler, AffineConstraints, overlap) :463-485.  coefficient: 0 = constant (reference),
   1 = a(x) = 1/(0.05 + 2|x|^2) at the quadrature points (BASELINE config 5 extension; 3-D only),
   PMG_COEFFICIENT_CALLER = -div(a grad u) with a given by the caller at the quadrature points
   (pmg_laplace_operator_set_coefficient; a = 1 until then).  dim 2 and 3, and _create_mapped / _create_curved. */
#define PMG_COEFFICIENT_CALLER 2
int pmg_laplace_operator_create(pmg_context *ctx, int dim, int degree, int nx, int ny, int nz,
                                unsigned dirichlet_faces, int coefficient, pmg_operator **op);
/* The Laplace operator (with coefficient 0 or 1 as above) on a deformed structured hexahedral mesh of nx x ny x nz cells, 3-D
   only.  vertices: HOST array of the (nx+1)(ny+1)(nz+1) mesh vertices, (x, y, z) interleaved, in global lexicographic order
   (x fastest), the same full array on every rank; it is read during the call only.  Cell (cx, cy, cz) is the trilinear map
   of its 8 vertices (cx+i, cy+j, cz+k), i, j, k in {0, 1} -- the geometry MappingQ(p) gives such a mesh with deal.II's
   FlatManifold.  DoF numbering and Dirichlet faces are those of pmg_laplace_operator_create; the coefficient is evaluated
   at the mapped quadrature points.  Every other operator, transfer, smoother, V-cycle and CG entry takes the result;
   assemble_rhs and solution_norm integrate over the mapped cells (QGauss(p+1) and QGauss(p+2)).  For the h-transfer the
   coarse mesh's vertex (i, j, k) must be the fine mesh's vertex (2i, 2j, 2k) (nested meshes; not checked).
   Errors: PMG_ERR_ARG with the first offending cell in pmg_last_error() if a cell has det J <= 0 at one of its Gauss points
   (inverted or degenerate) or a vertex that is not finite; PMG_ERR_UNSUPPORTED for degrees outside 1..PMG_MAX_DEGREE. */
int pmg_laplace_operator_create_mapped(pmg_context *ctx, int degree, int nx, int ny, int nz, unsigned dirichlet_faces,
                                       int coefficient, const double *vertices, pmg_operator **op);
/* The Laplace operator (coefficient 0 or 1 as above) on a structured mesh of nx x ny x nz curved hexahedra, 3-D only: the
   geometry MappingQ(k) gives the cells of a mesh on a curved manifold (a cylinder, a shell, a pipe bend).  nodes: HOST array
   of the (nx k + 1)(ny k + 1)(nz k + 1) geometry support points, (x, y, z) interleaved, in global lexicographic order
   (x fastest), the same full array on every rank; it is read during the call only.  Cell (cx, cy, cz) is the
   tensor-product Lagrange interpolant of degree k = geometry_degree through the nodes (cx k + i, cy k + j, cz k + l),
   0 <= i, j, l <= k, placed at the Gauss-Lobatto points of FE_Q(k) (pmg_host_support_points).  k = degree: the nodes are
   the DoF support points, the MappingQ(degree) the reference's operator builds; k = 1: the array is the vertex array of
   pmg_laplace_operator_create_mapped, with the same result.  Everything else as pmg_laplace_operator_create_mapped; the
   h-transfer and p-transfer are reference-cell contractions, so the meshes of an h-hierarchy need not be nested: each
   level interpolates the manifold itself, as MappingQ on every level does.
   Errors: PMG_ERR_ARG with the first offending cell in pmg_last_error() if a cell has det J <= 0 at one of its Gauss points
   or a node that is not finite; PMG_ERR_UNSUPPORTED for degree or geometry_degree outside 1..PMG_MAX_DEGREE. */
int pmg_laplace_operator_create_curved(pmg_context *ctx, int degree, int geometry_degree, int nx, int ny, int nz,
                                       unsigned dirichlet_faces, int coefficient, const double *nodes, pmg_operator **op);
int pmg_laplace_operator_destroy(pmg_operator *op);
int pmg_laplace_operator_vmult(const pmg_operator *op, pmg_vector *dst, const pmg_vector *src);  /* :557-719 */
int pmg_laplace_operator_Tvmult(const pmg_operator *op, pmg_vector *dst, const pmg_vector *src); /* :721-735 */
int pmg_laplace_operator_initialize_dof_vector(const pmg_operator *op, pmg_vector **vec);          /* :737-743 */
int pmg_laplace_operator_compute_diagonal(pmg_operator *op);                                       /* :752-917 */
int pmg_laplace_operator_get_matrix_diagonal_inverse(const pmg_operator *op, const pmg_vector **dinv); /* :919-925 */
int pmg_laplace_operator_m(const pmg_operator *op, int64_t *m);                                    /* :927-932 */
int pmg_laplace_operator_n(const pmg_operator *op, int64_t *n);                                    /* :934-939 */
int pmg_laplace_operator_el(const pmg_operator *op, int64_t row, int64_t col, double *value);      /* :941-954 (diagonal only) */
int pmg_laplace_operator_degree(const pmg_operator *op, int *degree);
int pmg_laplace_operator_cells(const pmg_operator *op, int *nx, int *ny, int *nz);
/* fused variants used by the smoother (one pass over HBM each; no reference equivalent):
   dst = b - A src */
int pmg_laplace_operator_residual(const pmg_operator *op, pmg_vector *dst, const pmg_vector *b, const pmg_vector *src);
/* one fused Chebyshev step: dst = src + f1 (src - xold) + f2 Dinv (b - A src); xold may be NULL (= 0)
   or alias dst.  This is the kernel every smoothing step of the V-cycle launches. */
int pmg_laplace_operator_chebyshev_step(const pmg_operator *op, pmg_vector *dst, const pmg_vector *src,
                                        const pmg_vector *xold, const pmg_vector *b, double f1, double f2);
/* same as vmult with HOST buffers of m() doubles in global lexicographic order (H2D + apply + D2H) */
int pmg_laplace_operator_vmult_host(const pmg_operator *op, double *dst_host, const double *src_host);
/* driver helpers: assemble_rhs (program.cc:289-334, f = 1) and the printed solution norm (:382-395) */
int pmg_laplace_operator_assemble_rhs(const pmg_operator *op, pmg_vector *rhs);
int pmg_laplace_operator_solution_norm(const pmg_operator *op, const pmg_vector *u, double *norm);

/* ---- problem data from the caller: f and g as dof vectors of the operator's layout (values at the dof support points) ----
   The workflow of the reference's matrix-free drivers with inhomogeneous data: fill f and g (e.g. with the coordinates from
   support_points, pmg_vector_import_host / _import_owned), assemble_rhs_data, solve A u0 = rhs with pmg_cg_solve and the
   V-cycle (rhs has zero constrained rows, like assemble_rhs), then distribute(u0, g); solution_norm then includes the
   boundary values.  Every call below returns PMG_ERR_ARG for a vector of another layout. */
/* Coordinates of the dof support points (FE_Q(degree) Gauss-Lobatto points mapped by the cell's geometry) on all stored
   planes, ghosts included; z must be NULL for dim = 2 (else PMG_ERR_UNSUPPORTED).  Box: the Gauss-Lobatto grid of the unit
   cube; mapped: the trilinear map; curved: the degree-k map evaluated at the degree-p Gauss-Lobatto points (k = degree:
   the nodes themselves). */
int pmg_laplace_operator_support_points(const pmg_operator *op, pmg_vector *x, pmg_vector *y, pmg_vector *z);
/* rhs = M f_h - A_free g_D on unconstrained rows, 0 on constrained rows (VectorTools::create_right_hand_side of the nodal
   interpolant f_h = sum_j f_j phi_j, interpolate_boundary_values + AffineConstraints, program.cc:163-187, 289-334).
   M: the mass matrix with QGauss(p+1) over the (mapped) cells.  A_free: the operator (with its coefficient and geometry)
   without Dirichlet masking.  g_D: g on constrained dofs, 0 elsewhere; only the constrained entries of g are read.
   f == NULL: no volume term; g == NULL: homogeneous.  rhs must differ from f and g.  The ghost planes of rhs are current
   on return. */
int pmg_laplace_operator_assemble_rhs_data(const pmg_operator *op, pmg_vector *rhs, const pmg_vector *f, const pmg_vector *g);
/* u_c = g_c on every constrained dof of the stored planes, other entries untouched (AffineConstraints::distribute, :361) */
int pmg_laplace_operator_distribute(const pmg_operator *op, pmg_vector *u, const pmg_vector *g);

/* ---- coefficient from the caller: a at the QGauss(degree+1) points of the operator's cells (step-37's coefficient table,
   FEEvaluation::quadrature_point) ----
   The rank's quadrature-point grid: Qx = nx (degree+1) by Qy = ny (degree+1) points per q-plane, lexicographic (x fastest),
   nqz q-planes from the global q-plane qz0 on -- the stored cell layers, the halo layer below the owned ones included.  2-D:
   qz0 = 0, nqz = 1; a rank that holds no part of the level: nqz = 0.  Cell (cx, cy, cz), local point (a, b, m) is grid point
   (cx (degree+1) + a, cy (degree+1) + b, cz (degree+1) + m). */
int pmg_laplace_operator_quadrature_grid(const pmg_operator *op, int64_t *qx, int64_t *qy, int64_t *qz0, int64_t *nqz);
/* The points of that grid: the Gauss points mapped by the cell's geometry (box, trilinear or degree-k map).  x, y, z: HOST
   arrays of Qx Qy nqz doubles; z must be NULL in 2-D (else PMG_ERR_UNSUPPORTED).  A point two ranks store has the same
   bits on both.  Works on every operator. */
int pmg_laplace_operator_quadrature_points(const pmg_operator *op, double *x, double *y, double *z);
/* Sets a at the points of pmg_laplace_operator_quadrature_points (a: HOST, Qx Qy nqz values in that order, each finite
   and > 0; read during the call only) and recomputes the operator's per-point data and its inverse diagonal.  A second
   call replaces the coefficient: the result equals a fresh operator given the second a.  Chebyshev smoothers keep the
   eigenvalue estimates of the operator they were created on: create them after the coefficient is set.
   Errors: PMG_ERR_STATE if the operator was not created with PMG_COEFFICIENT_CALLER; PMG_ERR_ARG for a == NULL or a value
   that is not finite or <= 0, with the first offending cell and local point in pmg_last_error() (the operator is then
   unchanged). */
int pmg_laplace_operator_set_coefficient(pmg_operator *op, const double *a);

/* ---- LinearAlgebra::distributed::Vector subset used on the path (SURVEY.md a11) ---- */
int pmg_vector_destroy(pmg_vector *v);
int pmg_vector_size(const pmg_vector *v, int64_t *global_size);
int pmg_vector_locally_owned_size(const pmg_vector *v, int64_t *n);
int pmg_vector_set(pmg_vector *v, double value);                                  /* operator=(s) */
int pmg_vector_copy(pmg_vector *dst, const pmg_vector *src);                      /* operator=(v) */
int pmg_vector_scale(pmg_vector *v, double a);                                    /* operator*= */
int pmg_vector_add(pmg_vector *v, double a, const pmg_vector *x);                 /* add(a,x): v += a x */
int pmg_vector_sadd(pmg_vector *v, double s, double a, const pmg_vector *x);      /* sadd(s,a,x): v = s v + a x */
int pmg_vector_dot(const pmg_vector *x, const pmg_vector *y, double *result);     /* operator* (allreduce) */
int pmg_vector_l2_norm(const pmg_vector *x, double *result);
int pmg_vector_mean_value(const pmg_vector *x, double *result);
int pmg_vector_update_ghost_values(pmg_vector *v);
int pmg_vector_compress_add(pmg_vector *v);
int pmg_vector_zero_out_ghost_values(pmg_vector *v);
int pmg_vector_import_host(pmg_vector *v, const double *host_global);             /* ReadWriteVector import, H2D */
int pmg_vector_export_host(const pmg_vector *v, double *host_global);             /* D2H; every rank receives the full vector */
double *pmg_vector_device_ptr(pmg_vector *v);                                     /* get_values() */
/* the rank's part (get_vector_partitioner analogue, include/base/portable_laplace_operator_base.h:58-59): stored dof planes
   [z0, z0 + n_planes) of plane_size dofs, of which [z_own_lo, z_own_hi) are owned; lexicographic inside a plane */
int pmg_vector_local_range(const pmg_vector *v, int64_t *plane_size, int *z0, int *n_planes, int *z_own_lo, int *z_own_hi);
/* owned planes only <-> host (no collective; ghosts untouched).  import is stream-ordered: keep the buffer until pmg_context_sync */
int pmg_vector_import_owned(pmg_vector *v, const double *host_owned);
int pmg_vector_export_owned(const pmg_vector *v, double *host_owned);
/* all stored planes, ghosts included <-> host (blocking) */
int pmg_vector_import_local(pmg_vector *v, const double *host_local);
int pmg_vector_export_local(const pmg_vector *v, double *host_local);
/* a vector over caller-owned device memory laid out like `like` (all stored planes): the adapter wraps the storage of a
   LinearAlgebra::distributed::Vector<double, MemorySpace::Default> instead of copying it per vmult; destroy frees the handle only */
int pmg_vector_wrap(const pmg_vector *like, double *device_values, pmg_vector **out);

/* ---- MGTransferBase (include/base/portable_mg_transfer_base.h:21-37) ---- */
/* GeometricTransfer::reinit  include/multigrid/portable_geometric_transfer.h:892-1327 */
int pmg_transfer_create_geometric(const pmg_operator *coarse, const pmg_operator *fine, pmg_transfer **t);
/* PolynomialTransfer::reinit include/multigrid/portable_polynomial_tranfer.h:903-1031 */
int pmg_transfer_create_polynomial(const pmg_operator *coarse, const pmg_operator *fine, pmg_transfer **t);
int pmg_transfer_destroy(pmg_transfer *t);
int pmg_transfer_prolongate_and_add(const pmg_transfer *t, pmg_vector *dst_fine, const pmg_vector *src_coarse);
int pmg_transfer_restrict_and_add(const pmg_transfer *t, pmg_vector *dst_coarse, const pmg_vector *src_fine);

/* ---- PreconditionChebyshev<LaplaceOperatorBase, Vector> with the Jacobi (inverse diagonal) inner
        preconditioner (configured at source/geometric_multigrid/program.cc:267-285) ---- */
int pmg_chebyshev_create(pmg_operator *op, double smoothing_range, int degree, int eig_cg_n_iterations,
                         pmg_chebyshev **s);
int pmg_chebyshev_destroy(pmg_chebyshev *s);
int pmg_chebyshev_vmult(pmg_chebyshev *s, pmg_vector *dst, const pmg_vector *src); /* zero initial guess */
int pmg_chebyshev_info(pmg_chebyshev *s, double *lambda_min, double *lambda_max, int *degree, int *cg_iterations);

/* ---- VCycleMultigrid (include/multigrid/portable_v_cycle_multigrid.h:35-43) ---- */
/* ops[0..n_levels) coarse -> fine; transfers[l] maps level l-1 <-> l (transfers[0] ignored);
   ctor :66-77 */
int pmg_vcycle_create(pmg_operator *const *ops, pmg_transfer *const *transfers, pmg_chebyshev *const *smoothers,
                      int n_levels, int pre_smoothing_steps, int post_smoothing_steps, pmg_vcycle **v);
int pmg_vcycle_destroy(pmg_vcycle *v);
int pmg_vcycle_vmult(pmg_vcycle *v, pmg_vector *dst, const pmg_vector *src);      /* :79-94 */
/* HOST-buffer variant (fine-level m() doubles each): H2D src, V-cycle, D2H dst */
/* the same with every rank's OWNED part of the vectors in host memory (plane_size * (z_own_hi - z_own_lo) doubles each) */
int pmg_vcycle_vmult_host_owned(pmg_vcycle *v, double *dst_host_owned, const double *src_host_owned);
int pmg_vcycle_vmult_host(pmg_vcycle *v, double *dst_host, const double *src_host);
/* 1 = replay the cycle from a CUDA graph (default), 0 = launch kernel by kernel */
int pmg_vcycle_set_graph(pmg_vcycle *v, int enable);
/* per-level device time of the last profiled cycle, ms: out[level*4 + {0 smoother,1 transfer,2 halo,3 other}] */
int pmg_vcycle_profile(pmg_vcycle *v, pmg_vector *dst, const pmg_vector *src, double *out_ms, int cap_levels);

/* ---- SolverCG + SolverControl (source/geometric_multigrid/program.cc:345-355) ---- */
/* precond may be NULL.  history (host, optional) receives residual norms 0..last_step. */
int pmg_cg_solve(const pmg_operator *A, pmg_vector *x, const pmg_vector *b, pmg_vcycle *precond,
                 int max_iterations, double tolerance, int *last_step, double *history, int history_cap);

/* ---- host-only helpers (no GPU needed; exercised by the CPU test-suite) ---- */
/* 1-D tables for FE_Q(degree): S (n1*n1, M = S^T S, K = S^T diag(lam) S), lam (n1) */
int pmg_host_fastdiag_tables(int degree, double *S, double *lam);
int pmg_host_pencil(int degree, double *M, double *K);
/* the degree + 1 Gauss-Lobatto points of [0, 1] (support points of FE_Q(degree)): where the nodes of a curved cell sit on the
   reference cell, i.e. where a caller evaluates its manifold for pmg_laplace_operator_create_curved */
int pmg_host_support_points(int degree, double *x);
int pmg_host_prolongation_1d(int kind, int degree_coarse, int degree_fine, double *P);
/* z-slab decomposition: owned cell layers of `rank` on a level with nz layers */
int pmg_host_partition(int nz, int n_ranks, int rank, int *cz_lo, int *cz_hi);
/* Chebyshev parameters from eigenvalue estimates (PreconditionChebyshev::estimate_eigenvalues) */
int pmg_host_chebyshev_parameters(double lambda_min_est, double lambda_max_est, double smoothing_range,
                                  int degree_in, double *theta, double *delta, int *degree_out);
/* extreme eigenvalues of a symmetric tridiagonal matrix */
int pmg_host_tridiag_extreme_eigenvalues(int n, const double *diag, const double *offdiag, double *lmin, double *lmax);

/* FP64 / HBM microbenchmarks for the roofline denominators */
int pmg_microbench(pmg_context *ctx, double *fp64_fma_tflops, double *fp64_dmma_tflops, double *hbm_copy_gbs);

#ifdef __cplusplus
}
#endif
#endif
