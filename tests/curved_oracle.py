"""The CPU oracle on a curved hexahedral mesh (test infrastructure).

As tests/mapped_oracle.py, with every cell the tensor-product Lagrange interpolant of degree k through its (k+1)^3 nodes
(tests/curved_mesh.py), i.e. what MappingQ(k) computes: curved_matrix_free() overwrites the oracle's per-point
inv_jacobian / JxW with the values of those maps at the Gauss points, and l2_norm_curved() integrates the QGauss(p+2) norm
over the curved cells.  Nothing under oracle/ changes.
"""
import ctypes as C

import numpy as np

from mapped_oracle import ref_points
from test_oracle_dense import gauss, gll_nodes, kron_xyz

_dp = C.POINTER(C.c_double)


def _array(ptr, n):
    return np.ctypeslib.as_array(C.cast(ptr, _dp), shape=(n,))


def basis_1d(k, x):
    """values and derivatives (len(x), k+1) of the degree-k Lagrange basis on the Gauss-Lobatto points at x (FE_Q(k)), in
    barycentric form: the monomial form of test_oracle_dense.shape_1d loses digits from k ~ 6 on (3e-11 at k = 9)"""
    s = gll_nodes(k)
    wb = np.array([1.0 / np.prod([s[i] - s[j] for j in range(k + 1) if j != i]) for i in range(k + 1)])
    S, D = np.zeros((len(x), k + 1)), np.zeros((len(x), k + 1))
    for q, xq in enumerate(x):
        hit = np.flatnonzero(s == xq)
        if hit.size == 0:
            d = xq - s
            S[q] = np.prod(d) * wb / d
            D[q] = S[q] * (np.sum(1.0 / d) - 1.0 / d)
        else:  # x is node h: phi_i(x) = delta_ih, phi_i'(x_h) = (wb_i / wb_h) / (x_h - x_i), phi_h' = sum 1 / (x_h - x_j)
            h = hit[0]
            S[q, h] = 1.0
            o = np.arange(k + 1) != h
            D[q, o] = (wb[o] / wb[h]) / (s[h] - s[o])
            D[q, h] = np.sum(1.0 / (s[h] - s[o]))
    return S, D


def cell_blocks(nodes, n, k):
    """(nc, k+1, k+1, k+1, 3) [cell, l, j, i, d]: the nodes of every cell, cells lexicographic (x fastest)"""
    nx, ny, nz = n
    N = np.asarray(nodes, dtype=np.float64).reshape(nz * k + 1, ny * k + 1, nx * k + 1, 3)
    cz, cy, cx = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    r = np.arange(k + 1)
    iz = (k * cz.ravel())[:, None, None, None] + r[None, :, None, None]
    iy = (k * cy.ravel())[:, None, None, None] + r[None, None, :, None]
    ix = (k * cx.ravel())[:, None, None, None] + r[None, None, None, :]
    return N[iz, iy, ix]


def curved_cells(nodes, n, k, m):
    """x (nc, m^3, 3) and J (nc, m^3, 3, 3), J[..., d, e] = d x_d / d xi_e, of every cell's degree-k map at the m^3 Gauss
    points (x fastest), by contraction of the cell's nodes with the 1-D GLL basis of degree k"""
    S, D = basis_1d(k, gauss(m)[0])  # (m, k+1)
    B = cell_blocks(nodes, n, k)
    nc = B.shape[0]
    x = np.einsum("zl,yj,xi,cljid->czyxd", S, S, S, B).reshape(nc, m ** 3, 3)
    J = np.stack([np.einsum("zl,yj,xi,cljid->czyxd", S, S, D, B), np.einsum("zl,yj,xi,cljid->czyxd", S, D, S, B),
                  np.einsum("zl,yj,xi,cljid->czyxd", D, S, S, B)], axis=-1).reshape(nc, m ** 3, 3, 3)
    return x, J


def curved_matrix_free(oracle, p, n, nodes, k, faces=None, coef=None):
    """oracle.MatrixFree of the 3-D mesh of n cells of geometry degree k with these nodes; coef "c5": a(x) at the mapped
    quadrature points.  ValueError if a cell has det J <= 0 at a Gauss point."""
    n = (n,) * 3 if isinstance(n, int) else tuple(n)
    mf = oracle.MatrixFree(3, p, n, faces=faces)
    _, w = ref_points(p + 1)
    x, J = curved_cells(nodes, n, k, p + 1)
    det = np.linalg.det(J)
    if not (det > 0).all():
        raise ValueError("curved mesh has a cell with det J <= 0 at a Gauss point")
    inv = np.linalg.inv(J)
    jxw = w[None, :] * det
    if coef == "c5":
        jxw = jxw / (0.05 + 2.0 * np.sum(x * x, axis=2))
    nq, nc = int(mf.s.n_q), mf.n_cells
    _array(mf.s.inv_jacobian, 9 * nc * nq)[:] = inv.transpose(3, 2, 0, 1).ravel()
    _array(mf.s.JxW, nc * nq)[:] = jxw.ravel()
    mf.nodes, mf.ncells3, mf.geometry_degree = np.ascontiguousarray(nodes, dtype=np.float64), n, k
    return mf


def l2_norm_curved(mf, u):
    """||u_h||_L2 over the curved cells with QGauss(p+2) (integrate_difference, program.cc:382-395)"""
    p, n = mf.p, mf.ncells3
    _, w = ref_points(p + 2)
    _, J = curved_cells(mf.nodes, n, mf.geometry_degree, p + 2)
    E = kron_xyz([basis_1d(p, gauss(p + 2)[0])[0]] * 3)
    nl, nc = int(mf.s.n_loc), mf.n_cells
    l2g = np.ctypeslib.as_array(C.cast(mf.s.local_to_global, C.POINTER(C.c_uint32)), shape=(nc * nl,)).reshape(nc, nl)
    vals = np.asarray(u)[l2g] @ E.T
    return float(np.sqrt(np.sum(vals * vals * w[None, :] * np.abs(np.linalg.det(J)))))
