"""The CPU oracle on a deformed hexahedral mesh (test infrastructure).

The oracle (oracle/orc.h) stores the reference's per-quadrature-point geometry -- inv_jacobian(q,cell,d,e) and JxW(q,cell)
in Kokkos LayoutLeft -- and applies the full tensor  JxW J^-1 J^-T  in its operator and diagonal
(include/operators/portable_laplace_operator.h:301-325).  Its constructor fills them for the unit cube's equal boxes;
mapped_matrix_free() overwrites them with the values of the trilinear map of every cell at its Gauss points, as MappingQ(p)
computes them for such a mesh with a flat manifold.  Everything the oracle derives from them -- vmult, the inverse diagonal,
the load vector of f = 1, Chebyshev, V-cycle, CG -- then runs on the mapped mesh; the transfers are reference-cell
contractions and need no geometry.  The printed QGauss(p+2) norm is the one quantity the oracle computes from the box
widths; l2_norm_mapped() integrates it over the mapped cells.
"""
import ctypes as C

import numpy as np

from mapped_mesh import uniform_vertices  # noqa: F401  (re-exported for the test modules)
from test_oracle_dense import gauss, kron_xyz, shape_1d

_dp = C.POINTER(C.c_double)


def ref_points(m):
    """m^3 Gauss points of [0, 1]^3, lexicographic (x fastest), and their weights"""
    xq, wq = gauss(m)
    Z, Y, X = np.meshgrid(xq, xq, xq, indexing="ij")
    return np.stack([X.ravel(), Y.ravel(), Z.ravel()], axis=1), kron_xyz([wq[:, None]] * 3).ravel()


def trilinear_cells(vertices, n, xi):
    """x (nc, nq, 3) and J (nc, nq, 3, 3), J[..., d, e] = d x_d / d xi_e, of every cell's trilinear map at the reference
    points xi (nq, 3); cells in lexicographic order (x fastest)"""
    nx, ny, nz = n
    V = np.asarray(vertices, dtype=np.float64).reshape(nz + 1, ny + 1, nx + 1, 3)
    x = np.zeros((nx * ny * nz, len(xi), 3))
    J = np.zeros((nx * ny * nz, len(xi), 3, 3))
    for c in range(8):
        ijk = (c & 1, c >> 1 & 1, c >> 2)
        Vc = V[ijk[2]:ijk[2] + nz, ijk[1]:ijk[1] + ny, ijk[0]:ijk[0] + nx].reshape(-1, 3)
        L = np.stack([xi[:, d] if ijk[d] else 1.0 - xi[:, d] for d in range(3)], axis=1)  # (nq, 3)
        s = np.array([1.0 if ijk[d] else -1.0 for d in range(3)])
        x += np.prod(L, axis=1)[None, :, None] * Vc[:, None, :]
        for e in range(3):
            dL = np.prod(np.where(np.arange(3) == e, s[None, :], L), axis=1)  # d L_c / d xi_e
            J[:, :, :, e] += dL[None, :, None] * Vc[:, None, :]
    return x, J


def _array(ptr, n):
    return np.ctypeslib.as_array(C.cast(ptr, _dp), shape=(n,))


def geometry(mf):
    """(inv_jacobian indexed [e, d, cell, q], JxW indexed [cell, q]) as the oracle stores them"""
    nq, nc = int(mf.s.n_q), mf.n_cells
    return (_array(mf.s.inv_jacobian, 9 * nc * nq).reshape(3, 3, nc, nq).copy(),
            _array(mf.s.JxW, nc * nq).reshape(nc, nq).copy())


def mapped_matrix_free(oracle, p, n, vertices, faces=None, coef=None):
    """oracle.MatrixFree of the 3-D mesh of n cells whose vertices are `vertices` ((nz+1, ny+1, nx+1, 3), x fastest);
    coef "c5": a(x) at the mapped quadrature points.  ValueError if a cell has det J <= 0 at a Gauss point."""
    n = (n,) * 3 if isinstance(n, int) else tuple(n)
    mf = oracle.MatrixFree(3, p, n, faces=faces)
    xi, w = ref_points(p + 1)
    x, J = trilinear_cells(vertices, n, xi)
    det = np.linalg.det(J)
    if not (det > 0).all():
        raise ValueError("mapped mesh has a cell with det J <= 0 at a Gauss point")
    inv = np.linalg.inv(J)  # inv[c, q, d, e] = (J^-1)_de = inv_jacobian(q, c, d, e)
    jxw = w[None, :] * det
    if coef == "c5":
        jxw = jxw / (0.05 + 2.0 * np.sum(x * x, axis=2))
    nq, nc = int(mf.s.n_q), mf.n_cells
    _array(mf.s.inv_jacobian, 9 * nc * nq)[:] = inv.transpose(3, 2, 0, 1).ravel()
    _array(mf.s.JxW, nc * nq)[:] = jxw.ravel()
    mf.vertices, mf.ncells3 = np.ascontiguousarray(vertices, dtype=np.float64), n
    return mf


def l2_norm_mapped(mf, u):
    """||u_h||_L2 over the mapped cells with QGauss(p+2) (integrate_difference, program.cc:382-395)"""
    p, n = mf.p, mf.ncells3
    xi, w = ref_points(p + 2)
    _, J = trilinear_cells(mf.vertices, n, xi)
    E = kron_xyz([shape_1d(p, gauss(p + 2)[0])[0]] * 3)  # (q, i)
    nl, nc = int(mf.s.n_loc), mf.n_cells
    l2g = np.ctypeslib.as_array(C.cast(mf.s.local_to_global, C.POINTER(C.c_uint32)), shape=(nc * nl,)).reshape(nc, nl)
    vals = np.asarray(u)[l2g] @ E.T  # (nc, q)
    return float(np.sqrt(np.sum(vals * vals * w[None, :] * np.abs(np.linalg.det(J)))))
