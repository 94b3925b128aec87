"""The numpy reference of the problem-data entries (tests/problem_data_ref.py) against the oracle (no GPU).

- With f = 1 the reference load vector reproduces the oracle's assemble_rhs on box, trilinear and curved meshes.
- Galerkin exactness: a polynomial u* the FE space contains, with f = -laplace(u*) interpolated and g = u* on the Dirichlet
  faces, is reproduced by the oracle's CG on the reference right-hand side plus the lifting.  Only affine cells qualify:
  on curved or non-affine trilinear cells the QGauss(p+1) stiffness integrand is not a polynomial the rule integrates
  exactly, so not even a linear u* comes back to round-off.
"""
import numpy as np
import pytest

from curved_mesh import SHELL_FACES, nodes_of, shell_map
from curved_oracle import curved_matrix_free
from helpers import rel_l2, splitmix_src
from mapped_mesh import random_vertices, sheared_box_vertices
from mapped_oracle import geometry, mapped_matrix_free
from problem_data_ref import (box_jxw, box_support_points, cell_dof_table, curved_support_points, load_vector,
                              rhs_reference, trilinear_support_points)


def _box_u(P):
    x, y, z = P.T
    return x * x * y + y * y * z + z * z * x, -2.0 * (x + y + z)


def _sheared_u(P):
    x, y, z = P.T
    return x * x + 2.0 * y * y - z * z + 0.5 * x * y - 0.3 * y * z + x - 1.0, np.full(len(P), -4.0)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("kind", ["box", "mapped", "curved"])
def test_load_vector_of_one_matches_oracle(kind, p, oracle):
    n = (3, 2, 4)
    if kind == "box":
        mf = oracle.MatrixFree(3, p, n, faces=0x15)
    elif kind == "mapped":
        mf = mapped_matrix_free(oracle, p, n, random_vertices(n, 0.2, seed=p), faces=0x15)
    else:
        mf = curved_matrix_free(oracle, p, n, nodes_of(shell_map, n, p), p, faces=SHELL_FACES)
    jxw = geometry(mf)[1]
    if kind == "box":
        assert np.abs(jxw - box_jxw(p, n)).max() <= 1e-15
    b = load_vector(p, n, jxw, np.ones(mf.n_dofs), mf.constrained())
    assert rel_l2(b, mf.assemble_rhs()) <= 1e-13


def test_dof_table_matches_oracle(oracle):
    import ctypes as C

    for p, n in ((1, (3, 2, 4)), (3, (2, 3, 2))):
        mf = oracle.MatrixFree(3, p, n)
        nl, nc = int(mf.s.n_loc), mf.n_cells
        l2g = np.ctypeslib.as_array(C.cast(mf.s.local_to_global, C.POINTER(C.c_uint32)), shape=(nc * nl,)).reshape(nc, nl)
        assert np.array_equal(cell_dof_table(p, n), l2g)


def test_support_point_references_agree():
    """trilinear and curved references at k = 1 on the same mesh, and both on the uniform mesh against the box grid"""
    n = (3, 2, 4)
    v = random_vertices(n, 0.2, seed=3)
    for p in (1, 2, 4):
        assert np.abs(trilinear_support_points(p, n, v) - curved_support_points(p, n, v, 1)).max() <= 1e-15
        uni = random_vertices(n, 0.0)
        assert np.abs(trilinear_support_points(p, n, uni) - box_support_points(p, n)).max() <= 1e-15
    nodes = nodes_of(shell_map, n, 3)
    assert np.abs(curved_support_points(3, n, nodes, 3) - nodes.reshape(-1, 3)).max() == 0.0


def _galerkin(oracle, mf, mf_free, jxw, P, u_fn):
    u, f = u_fn(P)
    c = mf.constrained()
    b = rhs_reference(mf.p, mf.ncell, jxw, c, f=f, g=u, mf_free=mf_free)
    x, it, _, rc = oracle.cg_solve(mf, b, rel_tol=1e-14, max_it=2000)
    x[c] = u[c]
    return x, u, rc


@pytest.mark.parametrize("p", [2, 3, 4])
def test_galerkin_exactness_box(p, oracle):
    n = (3, 3, 2)
    mf, mf_free = oracle.MatrixFree(3, p, n), oracle.MatrixFree(3, p, n, faces=0)
    x, u, rc = _galerkin(oracle, mf, mf_free, box_jxw(p, n), box_support_points(p, n), _box_u)
    assert np.abs(x - u).max() <= 1e-10


@pytest.mark.parametrize("p", [2, 3])
def test_galerkin_exactness_sheared(p, oracle):
    n = (3, 2, 2)
    v = sheared_box_vertices(n)
    mf = mapped_matrix_free(oracle, p, n, v)  # every face Dirichlet: u* has no zero normal derivative anywhere
    mf_free = mapped_matrix_free(oracle, p, n, v, faces=0)
    x, u, rc = _galerkin(oracle, mf, mf_free, geometry(mf)[1], trilinear_support_points(p, n, v), _sheared_u)
    assert np.abs(x - u).max() <= 1e-10


def test_lifting_is_linear_and_reads_constrained_entries_only(oracle):
    p, n = 2, (3, 2, 3)
    mf, mf_free = oracle.MatrixFree(3, p, n, faces=0x15), oracle.MatrixFree(3, p, n, faces=0)
    c = mf.constrained()
    g = splitmix_src(mf.n_dofs, salt=5)
    g2 = np.where(c, g, splitmix_src(mf.n_dofs, salt=6))
    b1 = rhs_reference(p, n, box_jxw(p, n), c, g=g, mf_free=mf_free)
    b2 = rhs_reference(p, n, box_jxw(p, n), c, g=g2, mf_free=mf_free)
    assert np.array_equal(b1, b2)
    assert np.all(b1[c] == 0.0)
