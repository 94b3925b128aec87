// pmg_dim2_var.cu -- kernels of the 2-D operator with a coefficient (csrc/pmg_dim2_var.h): pass 1 one thread per
// (cell, Gauss row), pass 2 one thread per DoF, and the inverse diagonal.  sm_100a only.
#include "pmg_dim2_var.h"
#include "pmg_cuda_common.h"
#include "pmg_kernels.h"

namespace {

// threads along (b, cx) fastest, then cy: neighbouring lanes read neighbouring words of u, W and R
template <int P>
__global__ void __launch_bounds__(128) k2v_row(const __grid_constant__ Pmg2VarLevel l, const double *__restrict__ u,
                                               const double *__restrict__ W, double *__restrict__ Rx, double *__restrict__ Ry)
{
  constexpr int N1 = P + 1;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= l.nx * N1 * l.ny) return;
  const int b = t % N1, c = t / N1;
  pmg2v_row<P>(l, u, W, Rx, Ry, c % l.nx, c / l.nx, b);
}

template <int P>
__global__ void __launch_bounds__(128) k2v_apply(const __grid_constant__ Pmg2VarLevel l, int mode, const double *__restrict__ u,
                                                 const double *__restrict__ Rx, const double *__restrict__ Ry,
                                                 const double *__restrict__ b, const double *xold, double *out, double f1, double f2,
                                                 const double *__restrict__ dinv_vec)
{
  const int gx = blockIdx.x * blockDim.x + threadIdx.x, gy = blockIdx.y;
  if (gx >= l.Nx) return;
  out[(int64_t)gy * l.Nx + gx] = pmg2v_apply_dof<P>(l, mode, u, Rx, Ry, b, xold, f1, f2, dinv_vec, gx, gy);
}

template <int P>
__global__ void __launch_bounds__(128) k2v_dinv(const __grid_constant__ Pmg2VarLevel l, const double *__restrict__ W, double *dinv)
{
  const int gx = blockIdx.x * blockDim.x + threadIdx.x, gy = blockIdx.y;
  if (gx >= l.Nx) return;
  // constrained entries are set to 1 before the inversion (reference :906)
  const double d = pmg2_dirichlet(gx, gy, l.Nx, l.Ny, l.faces) ? 1.0 : pmg2v_diag_entry<P>(l, W, gx, gy);
  dinv[(int64_t)gy * l.Nx + gx] = 1.0 / d;
}

void level_of(const pmgk_level *lv, Pmg2VarLevel &l)
{
  pmg2v_level_init(l, lv->degree, lv->nx, lv->ny, lv->faces, lv->h, lv->Sq, lv->Dco);
}

template <int P>
int apply_var2(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out, double f1, double f2,
               cudaStream_t s, int *geom)
{
  constexpr int N1 = P + 1;
  Pmg2VarLevel l;
  level_of(lv, l);
  const int64_t rows = (int64_t)lv->nx * N1 * lv->ny, nq = rows * N1;
  const dim3 grid((unsigned)((lv->Nx + 127) / 128), (unsigned)lv->Ny);
  if (geom) { geom[0] = (int)((rows + 127) / 128 + grid.x * grid.y); geom[1] = 128; geom[2] = 0; geom[3] = 1; return 0; }
  if (mode >= PMGK_CHEB_FIRST && !lv->dinv_vec) {
    pmg_set_error("variable-coefficient smoother step before compute_diagonal()");
    return PMG_ERR_STATE;
  }
  // the operator's allocation holds W and, right behind it, the two grids of pass 1 (host/pmg_operator.c)
  double *Rx = const_cast<double *>(lv->coef) + nq, *Ry = Rx + nq;
  k2v_row<P><<<(unsigned)((rows + 127) / 128), 128, 0, s>>>(l, u, lv->coef, Rx, Ry);
  PMG_CUDA_CHECK(cudaGetLastError());
  k2v_apply<P><<<grid, 128, 0, s>>>(l, mode, u, Rx, Ry, b, xold, out, f1, f2, lv->dinv_vec);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(2);
  return 0;
}

template <int P>
int fill_dinv2(const pmgk_level *lv, double *dinv, cudaStream_t s)
{
  Pmg2VarLevel l;
  level_of(lv, l);
  k2v_dinv<P><<<dim3((unsigned)((lv->Nx + 127) / 128), (unsigned)lv->Ny), 128, 0, s>>>(l, lv->coef, dinv);
  PMG_CUDA_CHECK(cudaGetLastError());
  pmg_count_launch(1);
  return 0;
}

} // namespace

#define PMG2V_DEGREES(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9)

// called by pmgk_apply (pmg_apply.cu) for levels with dim == 2 that carry a coefficient
int pmg_dim2_var_apply(const pmgk_level *lv, int mode, const double *u, const double *b, const double *xold, double *out, double f1,
                       double f2, cudaStream_t s, int *geom)
{
  switch (lv->degree) {
#define PMG2V_CASE(P) case P: return apply_var2<P>(lv, mode, u, b, xold, out, f1, f2, s, geom);
    PMG2V_DEGREES(PMG2V_CASE)
#undef PMG2V_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}

extern "C" int pmgk_dim2_var_fill_dinv(const pmgk_level *lv, double *dinv, void *stream)
{
  if (!lv || !dinv || !lv->coef || lv->dim != 2) return PMG_ERR_ARG;
  switch (lv->degree) {
#define PMG2V_CASE(P) case P: return fill_dinv2<P>(lv, dinv, (cudaStream_t)stream);
    PMG2V_DEGREES(PMG2V_CASE)
#undef PMG2V_CASE
    default: return PMG_ERR_UNSUPPORTED;
  }
}
