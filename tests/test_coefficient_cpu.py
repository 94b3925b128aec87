"""The caller-coefficient references (tests/coefficient_ref.py) and the 2-D kernel with a coefficient (no GPU).

- The oracle built with a ctypes a(x, y, z) callback equals the oracle whose JxW is multiplied by a at the reference's
  quadrature points, in 2-D and 3-D, Q1-Q5; the trilinear and curved point references agree with the box grid and with
  each other.
- The PMG_HD functions of csrc/pmg_dim2_var.h, run by the host emulator, equal the oracle with a jump coefficient: every
  epilogue mode and the inverse diagonal, Q1-Q9, faces 0xF, 0x5 and 0x0.
- Convergence of the oracle for a manufactured solution with a smooth coefficient a = 1 + |x|^2: the right-hand side of
  u* = cos(pi x) cos(pi y) [cos(pi z)] with f = -div(a grad u*) in closed form, error against the interpolant.
"""
import ctypes as C

import numpy as np
import pytest

from coefficient_ref import (cells_to_grid, grid_to_cells, jump, quadrature_points_box, quadrature_points_curved,
                             quadrature_points_trilinear, with_coefficient)
from curved_mesh import nodes_of, shell_map, trilinear_nodes
from helpers import rel_l2, splitmix_src
from mapped_mesh import random_vertices
from problem_data_ref import box_jxw, box_support_points, rhs_reference

_CB = C.CFUNCTYPE(C.c_double, C.c_double, C.c_double, C.c_double)
_dp = C.POINTER(C.c_double)


def _smooth(x, y, z):
    return 1.0 + x * x + 2.0 * y * y + 0.5 * z * z + 0.3 * np.sin(3.0 * x + y)


def callback_matrix_free(oracle, dim, p, n, fn, faces=None):
    """oracle.MatrixFree built by orc_mf_create with a ctypes a(x, y, z) callback (nothing under oracle/ changes)"""
    cb = _CB(lambda x, y, z: float(fn(x, y, z)))
    mf = oracle.MatrixFree.__new__(oracle.MatrixFree)
    n3 = tuple(n) + (1,) * (3 - len(n))
    if faces is None:
        faces = oracle.ALL_FACES_3D if dim == 3 else oracle.ALL_FACES_2D
    mf.h = oracle.lib().orc_mf_create(dim, p, n3[0], n3[1], n3[2], faces, C.cast(cb, C.c_void_p))
    mf.s = oracle._MFStruct.from_address(mf.h)
    mf.dim, mf.p = dim, p
    mf.n_dofs, mf.n_cells = int(mf.s.n_dofs), int(mf.s.n_cells)
    mf.nd, mf.ncell = tuple(mf.s.nd)[:dim], tuple(n)
    mf._cb = cb
    return mf


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("dim", [2, 3])
def test_callback_oracle_equals_jxw_times_a(dim, p, oracle):
    n = (3, 2, 2)[:dim] if dim == 3 else (3, 4)
    mf_cb = callback_matrix_free(oracle, dim, p, n, _smooth)
    P = quadrature_points_box(p, n)
    a = _smooth(*[P[:, d] for d in range(dim)], *([0.0] if dim == 2 else []))
    mf = with_coefficient(oracle.MatrixFree(dim, p, n), a)
    src = splitmix_src(mf.n_dofs)
    assert rel_l2(mf.vmult(src), mf_cb.vmult(src)) <= 1e-14
    assert rel_l2(mf.compute_diagonal(), mf_cb.compute_diagonal()) <= 1e-14


def test_grid_layout_round_trip():
    for p, n in ((2, (3, 4)), (3, (2, 3, 4))):
        v = np.arange(int(np.prod(n)) * (p + 1) ** len(n), dtype=float)
        assert np.array_equal(cells_to_grid(grid_to_cells(v, p, n), p, n), v)
    # cell (1, 0), point (a, b) = (2, 1) of a Q2 mesh of 3 x 4 cells: grid (1 * 3 + 2, 0 * 3 + 1)
    g = grid_to_cells(np.arange(9 * 12 * 1.0), 2, (3, 4))
    assert g[1, 2 + 3 * 1] == 1 * 9 + 5


@pytest.mark.parametrize("p", [1, 2, 4, 7])
def test_quadrature_point_references_agree(p):
    n = (3, 2, 4)
    box = quadrature_points_box(p, n)
    assert np.abs(quadrature_points_trilinear(p, n, random_vertices(n, 0.0)) - box).max() <= 1e-15
    v = random_vertices(n, 0.2, seed=p)
    tri = quadrature_points_trilinear(p, n, v)
    assert np.abs(quadrature_points_curved(p, n, trilinear_nodes(v, n, 1), 1) - tri).max() <= 1e-15
    assert np.abs(quadrature_points_curved(p, n, trilinear_nodes(v, n, 3), 3) - tri).max() <= 1e-14
    # the points lie inside their cells: the shell's points have 1 <= r <= 2
    sh = quadrature_points_curved(p, n, nodes_of(shell_map, n, 2), 2)
    r = np.hypot(sh[:, 0], sh[:, 1])
    assert r.min() > 1.0 and r.max() < 2.0


# ---- the 2-D kernel with a coefficient, on the host emulator -------------------------------------------------------------
def _emu2v(emu, p, n, faces, a, mode, u, b=None, xold=None, f1=0.0, f2=0.0, dinv=None):
    out = np.empty_like(u)
    P = lambda v: None if v is None else np.ascontiguousarray(v).ctypes.data_as(_dp)  # noqa: E731
    rc = emu.emu2v_apply(C.c_int(p), C.c_int(n[0]), C.c_int(n[1]), C.c_uint(faces), P(a), C.c_int(mode), P(u), P(b), P(xold),
                         out.ctypes.data_as(_dp), C.c_double(f1), C.c_double(f2), P(dinv))
    assert rc == 0
    return out


@pytest.mark.parametrize("faces", [0xF, 0x5, 0x0])
@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8, 9])
def test_emulated_dim2_coefficient_kernel_matches_oracle(p, faces, emu, oracle):
    n = (3, 4)
    a = jump(quadrature_points_box(p, n))
    mf = with_coefficient(oracle.MatrixFree(2, p, n, faces=faces), a)
    m = mf.n_dofs
    u, b, xo = splitmix_src(m), splitmix_src(m, salt=1), splitmix_src(m, salt=2)
    Au = mf.vmult(u)
    dinv_ref = mf.compute_diagonal()
    dinv = np.empty(m)
    assert emu.emu2v_dinv(C.c_int(p), C.c_int(n[0]), C.c_int(n[1]), C.c_uint(faces), a.ctypes.data_as(_dp), dinv.ctypes.data_as(_dp)) == 0
    assert rel_l2(dinv, dinv_ref) <= 1e-13
    assert rel_l2(_emu2v(emu, p, n, faces, a, 0, u), Au) <= 1e-13
    assert rel_l2(_emu2v(emu, p, n, faces, a, 1, u, b), b - Au) <= 1e-13
    f1, f2 = 0.3, 0.7
    assert rel_l2(_emu2v(emu, p, n, faces, a, 2, u, b, f2=f2, dinv=dinv), u + f2 * dinv_ref * (b - Au)) <= 1e-13
    step = u + f1 * (u - xo) + f2 * dinv_ref * (b - Au)
    assert rel_l2(_emu2v(emu, p, n, faces, a, 3, u, b, xo, f1, f2, dinv), step) <= 1e-13
    assert rel_l2(_emu2v(emu, p, n, faces, a, 3, u, b, None, f1, f2, dinv), u + f1 * u + f2 * dinv_ref * (b - Au)) <= 1e-13
    # x_old aliasing the output: every entry is read before it is written
    alias = xo.copy()
    out = _emu2v(emu, p, n, faces, a, 3, u, b, alias, f1, f2, dinv)
    assert rel_l2(out, step) <= 1e-13


# ---- manufactured solution with a smooth coefficient --------------------------------------------------------------------
def manufactured(P):
    """u* = cos(pi x) cos(pi y) [cos(pi z)], a = 1 + |x|^2, f = -div(a grad u*) = -grad a . grad u* - a laplace u*"""
    P = np.asarray(P)
    dim = P.shape[1]
    c, s = np.cos(np.pi * P), np.sin(np.pi * P)
    u = np.prod(c, axis=1)
    a = 1.0 + np.sum(P * P, axis=1)
    grad = [-np.pi * s[:, d] * np.prod(np.delete(c, d, axis=1), axis=1) for d in range(dim)]
    f = -sum(2.0 * P[:, d] * grad[d] for d in range(dim)) + a * dim * np.pi ** 2 * u
    return u, f


def manufactured_error(oracle, dim, p, nc):
    """||u_h - I_h u*||_L2 of the oracle's solution on nc^dim cells"""
    n = (nc,) * dim
    a = 1.0 + np.sum(quadrature_points_box(p, n) ** 2, axis=1)
    mf = with_coefficient(oracle.MatrixFree(dim, p, n), a)
    mf_free = with_coefficient(oracle.MatrixFree(dim, p, n, faces=0), a)
    u, f = manufactured(box_support_points(p, n))
    c = mf.constrained()
    b = rhs_reference(p, n, box_jxw(p, n), c, f=f, g=u, mf_free=mf_free)
    x, _, _, rc = oracle.cg_solve(mf, b, rel_tol=1e-13, max_it=5000)
    assert rc == 0
    x[c] = u[c]
    return mf.l2_norm_solution(x - u)


# rates computed with this oracle: 2-D Q3 on 2, 4, 8, 16 cells 4.95, 4.92, 4.96; 3-D Q2 on 2, 4, 8 cells 3.81, 3.80 -- the
# interpolant is superclose to u_h (order p + 2 on these uniform meshes), pinned with a margin
@pytest.mark.parametrize("dim, p, cells, rate", [(2, 3, (2, 4, 8), 4.6), (3, 2, (2, 4, 8), 3.5)])
def test_manufactured_convergence_with_coefficient(dim, p, cells, rate, oracle):
    errs = [manufactured_error(oracle, dim, p, nc) for nc in cells]
    rates = [np.log2(errs[i] / errs[i + 1]) for i in range(len(errs) - 1)]
    assert min(rates) >= rate, (errs, rates)
