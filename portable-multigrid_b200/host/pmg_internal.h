/* pmg_internal.h -- internal declarations of the C host layer. */
#ifndef PMG_INTERNAL_H
#define PMG_INTERNAL_H

#include <cuda_runtime_api.h>
#include <nccl.h>
#include <stdint.h>
#include "pmg.h"
#include "pmg_kernels.h"

#ifdef __cplusplus
extern "C" {
#endif

void pmg_set_error(const char *fmt, ...);
void pmg_count_launch(int n);
/* every public entry point that enqueues work makes the context's device current first (a caller thread may have switched
   devices, or hold contexts on several GPUs) */
int pmg_enter(const pmg_context *ctx);

#define PMG_CHECK(call)                        \
  do {                                         \
    int pmg_rc_ = (call);                      \
    if (pmg_rc_ != PMG_OK) return pmg_rc_;     \
  } while (0)

#define PMG_CUDA(call)                                                                            \
  do {                                                                                            \
    cudaError_t pmg_e_ = (call);                                                                  \
    if (pmg_e_ != cudaSuccess) {                                                                  \
      pmg_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(pmg_e_)); \
      return PMG_ERR_CUDA;                                                                        \
    }                                                                                             \
  } while (0)

/* inside ncclGroupStart() .. ncclGroupEnd(): a failing call closes the group before the function returns */
#define PMG_NCCL_IN_GROUP(call)                                                                   \
  do {                                                                                            \
    ncclResult_t pmg_n_ = (call);                                                                 \
    if (pmg_n_ != ncclSuccess) {                                                                  \
      pmg_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, ncclGetErrorString(pmg_n_)); \
      ncclGroupEnd();                                                                             \
      return PMG_ERR_NCCL;                                                                        \
    }                                                                                             \
  } while (0)

#define PMG_NCCL(call)                                                                            \
  do {                                                                                            \
    ncclResult_t pmg_n_ = (call);                                                                 \
    if (pmg_n_ != ncclSuccess) {                                                                  \
      pmg_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, ncclGetErrorString(pmg_n_)); \
      return PMG_ERR_NCCL;                                                                        \
    }                                                                                             \
  } while (0)

/* pmg_fe.c */
void pmg_fe_gauss(int n, double *x, double *w);
void pmg_fe_gll(int n, double *x);
void pmg_fe_lagrange(int n, const double *nodes, double x, double *val, double *der);
void pmg_fe_pencil(int p, double *M, double *K);
void pmg_fe_fastdiag(int p, double *S, double *lam);
void pmg_fe_prolongation_h(int p, double *P);
void pmg_fe_prolongation_p(int pc, int pf, double *P);
void pmg_fe_diag_1d(int p, double *Md, double *Kd);
void pmg_fe_dinv_table(int p, const double h[3], int dim, double *tab);
void pmg_fe_shape_tables(int p, double *Sq, double *Dco, double *G, double *gq, double *gw);

/* peer mapping of the slab neighbours' vectors (pmg_p2p.c) */
#define PMG_P2P_MAX_REG 512
typedef struct pmg_p2p_reg {
  double *base;                       /* this rank's array */
  const double *peer_lower, *peer_upper; /* the neighbours' arrays of the same vector, mapped here */
  int lower_z0, upper_z0;             /* their first stored dof plane */
  int key[4];                         /* the level the array was made for: Nx, Ny, Nz, degree (identical on every rank) */
  int in_use;                         /* 0: released by its vector, kept (mapped on the neighbours) for the next vector of that level */
} pmg_p2p_reg;
typedef struct pmg_p2p {
  int enabled;                        /* the neighbours' mailboxes (and, per vector, arrays) are mapped */
  int explicit_push;                  /* stand-alone exchanges use the push kernel instead of the NCCL group (PMG_P2P_HALO=1) */
  int fused;                          /* the smoother's applies push their boundary planes themselves (PMG_FUSED_HALO, default on) */
  int64_t push_min_bytes;             /* stand-alone exchanges of at least this many bytes per neighbour pair use the push kernel (PMG_P2P_MIN_BYTES) */
  void *msg_dev;                      /* device scratch of the handle exchange */
  uint64_t *mailbox, *mb_lower, *mb_upper;
  pmg_p2p_reg reg[PMG_P2P_MAX_REG];
  int n_reg;
  const double *last_base;            /* the array of the previous exchange (NULL: unknown) */
  int64_t n_fused;                    /* applies that consumed pushed ghost planes (statistics) */
} pmg_p2p;

struct pmg_context {
  int device;
  int rank, n_ranks;
  cudaStream_t stream;
  ncclComm_t comm;
  int has_comm;
  /* halo exchange overlapped with the interior chunks of the apply (pmg_operator.c): its own stream and communicator */
  cudaStream_t halo_stream;
  ncclComm_t halo_comm;
  cudaEvent_t ev_ready, ev_halo;
  int overlap;
  /* profiling hook (pmg_vcycle_profile): called with 1 before and 0 after every ghost exchange enqueued on ctx->stream */
  void (*halo_hook)(void *user, int begin);
  void *halo_hook_user;
  int64_t coarse_threshold;
  double *work;      /* device: reduction workspace */
  double *scalars;   /* device: small scalar slots */
  double *h_scalars; /* pinned host mirror */
  int sm_count;
  pmg_p2p p2p;
};


/* one level's decomposition: z-slabs of cell layers, or everything on rank 0 */
typedef struct pmg_layout {
  int nx, ny, nz, degree;
  int Nx, Ny, Nz;
  int active;            /* this rank holds part of the level */
  int gathered;          /* 1 = whole level on rank 0 */
  int cz_lo, cz_hi;      /* owned cell layers */
  int z0, nzl;           /* stored planes */
  int z_own_lo, z_own_hi;/* owned planes */
  int lower, upper;      /* neighbour ranks or -1 */
  int64_t plane;         /* Nx*Ny */
  int64_t n_local;       /* nzl*plane */
  int64_t n_global;
} pmg_layout;

/* pmg_p2p.c */
int pmg_p2p_init(pmg_context *ctx);
void pmg_p2p_shutdown(pmg_context *ctx);
int pmg_p2p_register(pmg_context *ctx, const pmg_layout *lay, double *d);
double *pmg_p2p_acquire(pmg_context *ctx, const pmg_layout *lay);
int pmg_p2p_release(pmg_context *ctx, double *d);
int pmg_p2p_halo(pmg_context *ctx, const pmg_layout *lay, double *d, cudaStream_t stream, int *done);
void pmg_p2p_forget(pmg_context *ctx);
/* 1 and *desc filled (push / consume left 0) if `out` is a mapped vector of a slab with neighbours and fused pushes are on */
int pmg_p2p_push_desc(pmg_context *ctx, const pmg_layout *lay, double *out, pmgk_push *desc);

struct pmg_vector {
  pmg_context *ctx;
  pmg_layout lay;
  double *d;
  int borrowed; /* d belongs to the caller (pmg_vector_wrap): never freed here */
};

struct pmg_operator {
  pmg_context *ctx;
  int dim, degree, coefficient;
  unsigned faces;
  pmg_layout lay;
  pmgk_level lv;
  double *d_dinv_tab;
  double *d_coef;        /* variable coefficient at the quadrature points (coefficient != 0), or the six grids of the
                            mapped geometry's G_q (mapped) */
  int mapped;            /* created by pmg_laplace_operator_create_mapped / _curved: lv.geo_stride != 0 where the level is stored */
  int geo_degree;        /* mapped: the cells' geometry degree k (1 = trilinear) */
  double *d_vert;        /* mapped: node planes k lv.coef_cz0 .. k lv.cz_hi of the stored cell layers (rhs, solution norm) */
  pmg_vector *dinv;      /* explicit inverse diagonal once compute_diagonal() ran */
  pmg_vector *cg_ws[4];  /* CG work vectors r, z, p, Ap: created by the first pmg_cg_solve, kept until destroy */
};

struct pmg_transfer {
  pmg_context *ctx;
  int kind;
  const pmg_operator *coarse, *fine;
  double *d_P;
  double *d_scratch;
  pmg_vector *gather_buf; /* coarse-level vector in the fine level's layout when layouts differ */
};

struct pmg_chebyshev {
  pmg_operator *op;
  double smoothing_range;
  int degree, eig_cg_n_iterations;
  int initialized;
  double lambda_min, lambda_max, theta, delta;
  int cg_iterations;
  pmg_vector *t0, *t1;   /* ping-pong work vectors */
};

int pmg_layout_make(pmg_context *ctx, int dim, int degree, int nx, int ny, int nz, pmg_layout *lay);
int pmg_layout_same(const pmg_layout *a, const pmg_layout *b);
int pmg_vector_create_layout(pmg_context *ctx, const pmg_layout *lay, pmg_vector **v);
int pmg_halo_update(pmg_context *ctx, const pmg_layout *lay, double *d);
int pmg_halo_update_on(pmg_context *ctx, const pmg_layout *lay, double *d, ncclComm_t comm, cudaStream_t stream);
int pmg_allreduce_sum(pmg_context *ctx, double *dev_scalar, int count);
int pmg_vector_dot_device(const pmg_vector *x, const pmg_vector *y, int slot);
/* ghost update of u + fused apply; the exchange overlaps the interior z-chunks when the launch splits (pmg_operator.c) */
int pmg_apply_with_halo(const pmg_operator *op, int mode, double *u, const double *b, const double *xold, double *out, double f1, double f2);
int pmg_apply_chain_ok(const pmg_operator *op, int mode, double *v0, double *v1);
int pmg_apply_chained(const pmg_operator *op, int mode, double *u, const double *b, const double *xold, double *out, double f1,
                      double f2, int consume, int push);
int pmg_chebyshev_estimate(pmg_chebyshev *s);
/* fused smoother: u <- smooth(u, rhs); zero_guess => u is taken as 0 on entry.  tmp: work vector.
   On return *result points at the vector that holds the smoothed iterate (u or tmp). */
int pmg_chebyshev_smooth(pmg_chebyshev *s, pmg_vector *u, const pmg_vector *rhs, pmg_vector *tmp,
                         int zero_guess, pmg_vector **result);
int pmg_chebyshev_smooth_chain(pmg_chebyshev *s, pmg_vector *u, const pmg_vector *rhs, pmg_vector *tmp, int zero_guess,
                               pmg_vector **result, int chain_in, int want_out, int *pushed_out);

#ifdef __cplusplus
}
#endif
#endif
