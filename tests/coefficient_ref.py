"""numpy reference of the caller-coefficient entries (test infrastructure, pinned by tests/test_coefficient_cpu.py).

The operator takes a at the QGauss(p+1) points of its cells, on the lexicographic grid of all quadrature points
(pmg_laplace_operator_quadrature_grid: Qx = nx (p+1), Qy = ny (p+1), then the q-planes, x fastest).  The oracle stores the
same points per cell (JxW(q, cell), q and cells lexicographic): grid_to_cells / cells_to_grid convert between the two.
quadrature_points_* give the Gauss points mapped by the cell's geometry: the box, the trilinear map, the degree-k map.
with_coefficient multiplies an oracle's JxW by a, which is what the oracle's a(x,y,z) callback does at construction.
"""
import ctypes as C

import numpy as np

from curved_oracle import curved_cells
from mapped_oracle import ref_points, trilinear_cells
from test_oracle_dense import gauss

_dp = C.POINTER(C.c_double)


def grid_to_cells(v, p, n):
    """values on the quadrature-point grid -> (nc, nq), cells and points lexicographic (x fastest); trailing axes kept"""
    n1, dim = p + 1, len(n)
    v = np.asarray(v)
    tail = v.shape[1:]
    if dim == 2:
        g = v.reshape((n[1], n1, n[0], n1) + tail)
        return np.moveaxis(g, (0, 2, 1, 3), (0, 1, 2, 3)).reshape((n[0] * n[1], n1 * n1) + tail)
    g = v.reshape((n[2], n1, n[1], n1, n[0], n1) + tail)
    return np.moveaxis(g, (0, 2, 4, 1, 3, 5), (0, 1, 2, 3, 4, 5)).reshape((n[0] * n[1] * n[2], n1 ** 3) + tail)


def cells_to_grid(v, p, n):
    """inverse of grid_to_cells"""
    n1, dim = p + 1, len(n)
    v = np.asarray(v)
    tail = v.shape[2:]
    if dim == 2:
        g = v.reshape((n[1], n[0], n1, n1) + tail)
        return np.moveaxis(g, (0, 1, 2, 3), (0, 2, 1, 3)).reshape((-1,) + tail)
    g = v.reshape((n[2], n[1], n[0], n1, n1, n1) + tail)
    return np.moveaxis(g, (0, 1, 2, 3, 4, 5), (0, 2, 4, 1, 3, 5)).reshape((-1,) + tail)


def quadrature_points_box(p, n):
    """(Q, dim) Gauss points of the unit cube's (square's) equal cells, grid order: (c + g_a) / n per direction"""
    g = gauss(p + 1)[0]
    lines = [np.concatenate([(c + g) / nd for c in range(nd)]) for nd in n]
    mesh = np.meshgrid(*lines[::-1], indexing="ij")[::-1]
    return np.stack([m.ravel() for m in mesh], axis=1)


def quadrature_points_trilinear(p, n, vertices):
    """(Q, 3) the trilinear maps of the cells at their Gauss points, grid order"""
    x, _ = trilinear_cells(vertices, n, ref_points(p + 1)[0])
    return cells_to_grid(x, p, n)


def quadrature_points_curved(p, n, nodes, k):
    """(Q, 3) the degree-k maps of the cells at their Gauss points, grid order"""
    x, _ = curved_cells(nodes, n, k, p + 1)
    return cells_to_grid(x, p, n)


def jxw_array(mf):
    """the oracle's JxW(q, cell) as a writable (nc, nq) view"""
    nq, nc = int(mf.s.n_q), mf.n_cells
    return np.ctypeslib.as_array(C.cast(mf.s.JxW, _dp), shape=(nc * nq,)).reshape(nc, nq)


def with_coefficient(mf, a_grid):
    """JxW *= a at every quadrature point (a on the grid of the oracle's mesh); returns mf"""
    jxw_array(mf)[:] *= grid_to_cells(a_grid, mf.p, mf.ncell)
    return mf


def jump(P, inside=100.0):
    """the jump coefficient of the drivers' --coefficient 2 on the cube / square: 100 in [1/4, 3/4]^dim, 1 elsewhere"""
    P = np.asarray(P)
    m = np.all((P >= 0.25) & (P <= 0.75), axis=1)
    return np.where(m, inside, 1.0)


def c5(P):
    """a = 1/(0.05 + 2|x|^2), the operator's coefficient 1"""
    P = np.asarray(P)
    return 1.0 / (0.05 + 2.0 * np.sum(P * P, axis=1))
