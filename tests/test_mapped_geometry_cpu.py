"""The Laplace operator on deformed hexahedral meshes (trilinear cells), on the CPU.

1. The oracle on a mapped mesh (tests/mapped_oracle.py: its per-point inv_jacobian / JxW filled from the trilinear maps)
   against an independent numpy dense assembly with the physical gradients J^-T grad_xi phi: operator, inverse diagonal,
   load vector and the QGauss(p+2) norm.
2. The identity map gives exactly the data of the unit-cube constructor; affine (sheared box) cells match the assembly too.
3. The tensor variant of the variable-coefficient tile program (csrc/pmg_apply_var.h, GEO = true) under the host
   emulator against the oracle: all epilogues, z-chunks, tile sizes, slabs, faces, degrees 1..9.
"""
import ctypes as C

import numpy as np
import pytest

from helpers import rel_l2, splitmix_src
from mapped_mesh import cell_vertices, random_vertices, sheared_box_vertices, smooth_map_vertices, trilinear, uniform_vertices
from mapped_oracle import geometry, l2_norm_mapped, mapped_matrix_free, ref_points
from test_oracle_dense import constrained_mask, cell_dofs, gauss, kron_xyz, shape_1d

C5 = lambda x, y, z: 1.0 / (0.05 + 2.0 * (x * x + y * y + z * z))  # noqa: E731


def dense_mapped(p, n, faces, vertices, coef=None):
    """A_ij = sum_cells sum_q a(x(xi_q)) w_q |det J| (J^-T grad phi_i) . (J^-T grad phi_j), Dirichlet rows / columns
    replaced by the identity; the load vector of f = 1 with constrained rows dropped; the QGauss(p+2) mass matrix."""
    xq, _ = gauss(p + 1)
    S, D = shape_1d(p, xq)
    xi, w = ref_points(p + 1)
    Gref = [kron_xyz([D if e == d else S for e in range(3)]) for d in range(3)]  # (q, i)
    Sk = kron_xyz([S] * 3)
    xi2, w2 = ref_points(p + 2)
    E = kron_xyz([shape_1d(p, gauss(p + 2)[0])[0]] * 3)
    ndofs = int(np.prod([nd * p + 1 for nd in n]))
    A, b, M = np.zeros((ndofs, ndofs)), np.zeros(ndofs), np.zeros((ndofs, ndofs))
    for cell in np.ndindex(*n[::-1]):
        cell = cell[::-1]
        V = cell_vertices(vertices, cell)
        x, J = trilinear(V, xi)
        det = np.linalg.det(J)
        assert (det > 0).all()
        Jinv = np.linalg.inv(J)  # Jinv[q, d, e] = d xi_d / d x_e
        wq = w * det * (coef(*x.T) if coef is not None else 1.0)
        grad = [sum(Jinv[:, d, e][:, None] * Gref[d] for d in range(3)) for e in range(3)]  # d phi / d x_e
        idx = cell_dofs(p, n, cell)
        A[np.ix_(idx, idx)] += sum(g.T @ (wq[:, None] * g) for g in grad)
        b[idx] += Sk.T @ (w * det)
        _, J2 = trilinear(V, xi2)
        M[np.ix_(idx, idx)] += E.T @ ((w2 * np.abs(np.linalg.det(J2)))[:, None] * E)
    c = constrained_mask(p, n, faces)
    A[c, :] = 0
    A[:, c] = 0
    A[c, c] = 1.0
    b[c] = 0.0
    return A, b, M, c


@pytest.mark.parametrize("p,n,faces,coef", [(1, (3, 2, 2), 0x3F, None), (2, (2, 3, 2), 0x15, None), (3, (2, 2, 2), 0x3F, "c5"),
                                            (4, (2, 2, 2), 0x2A, None), (5, (2, 2, 2), 0x3F, "c5"), (2, (3, 2, 2), 0x00, "c5"),
                                            (1, (2, 2, 3), 0x0C, "c5")])
def test_mapped_oracle_matches_dense_assembly(p, n, faces, coef, oracle):
    v = random_vertices(n, 0.2, seed=p + 7 * faces)
    A, b, M, c = dense_mapped(p, n, faces, v, C5 if coef else None)
    mf = mapped_matrix_free(oracle, p, n, v, faces=faces, coef=coef)
    assert np.array_equal(mf.constrained(), c)
    rng = np.random.default_rng(p)
    for _ in range(2):
        u = rng.standard_normal(mf.n_dofs)
        assert rel_l2(mf.vmult(u), A @ u) < 1e-12
    assert rel_l2(mf.compute_diagonal(), 1.0 / np.diag(A)) < 1e-12
    if coef is None:  # the load vector of f = 1 carries no coefficient only when there is none (as for the cube)
        assert rel_l2(mf.assemble_rhs(), b) < 1e-12
    u = rng.standard_normal(mf.n_dofs)
    ref = np.sqrt(u @ M @ u)
    assert abs(l2_norm_mapped(mf, u) - ref) < 1e-12 * ref
    # the distortion matters: not the cube's operator
    u = rng.standard_normal(mf.n_dofs)
    assert rel_l2(mf.vmult(u), oracle.MatrixFree(3, p, n, faces=faces, coef=coef).vmult(u)) > 1e-3


@pytest.mark.parametrize("p,n", [(1, (3, 2, 2)), (2, (2, 2, 2)), (4, (2, 1, 2))])
def test_mapped_oracle_affine_sheared_box(p, n, oracle):
    v = sheared_box_vertices(n)
    A, b, M, c = dense_mapped(p, n, 0x3F, v)
    mf = mapped_matrix_free(oracle, p, n, v)
    u = np.random.default_rng(5).standard_normal(mf.n_dofs)
    assert rel_l2(mf.vmult(u), A @ u) < 1e-12
    assert rel_l2(mf.compute_diagonal(), 1.0 / np.diag(A)) < 1e-12
    assert rel_l2(mf.assemble_rhs(), b) < 1e-12
    assert abs(l2_norm_mapped(mf, u) - np.sqrt(u @ M @ u)) < 1e-12 * np.sqrt(u @ M @ u)


@pytest.mark.parametrize("p,n,coef", [(1, (3, 2, 2), None), (2, (2, 3, 2), "c5"), (4, (2, 2, 1), None), (5, (1, 2, 2), "c5")])
def test_identity_map_equals_cube_oracle(p, n, coef, oracle):
    """uniform vertices: the mapped geometry equals the unit-cube constructor's to 1e-14 in every array"""
    cube = oracle.MatrixFree(3, p, n, coef=coef)
    mapped = mapped_matrix_free(oracle, p, n, uniform_vertices(n), coef=coef)
    (ij0, jxw0), (ij1, jxw1) = geometry(cube), geometry(mapped)
    assert np.abs(ij1 - ij0).max() <= 1e-14 * np.abs(ij0).max()
    assert np.abs(jxw1 - jxw0).max() <= 1e-14 * np.abs(jxw0).max()
    u = splitmix_src(cube.n_dofs, salt=p)
    assert rel_l2(mapped.vmult(u), cube.vmult(u)) < 1e-14
    assert rel_l2(mapped.compute_diagonal(), cube.compute_diagonal()) < 1e-14
    assert rel_l2(mapped.assemble_rhs(), cube.assemble_rhs()) < 1e-14
    # the mapped norm is a numpy sum over all cells, the cube's the oracle's per-cell loop: another summation order
    assert abs(l2_norm_mapped(mapped, u) - cube.l2_norm_solution(u)) < 1e-13 * cube.l2_norm_solution(u)


def test_mapped_oracle_rejects_inverted_cell(oracle):
    n = (2, 2, 2)
    v = uniform_vertices(n)
    v[1, 1, 1] = (0.9, 0.9, 0.9)  # the centre vertex pushed almost to the far corner: the cells around it fold
    with pytest.raises(ValueError):
        mapped_matrix_free(oracle, 2, n, v)


# ---- the tensor tile program under the host emulator -------------------------------------------------------------
def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def emu_geo(emu, p, n, vertices, u, mode=0, b=None, xold=None, f1=0.0, f2=0.0, small=1, chunks=1, faces=0x3F, c5=0,
            slab=None, want_dinv=False):
    nx, ny, nz = n
    Nz = nz * p + 1
    z0, nzl, czlo, czhi, zol, zoh = (0, Nz, 0, nz, 0, Nz) if slab is None else slab
    out = np.full(u.shape, np.nan)
    dv = np.empty(u.shape) if want_dinv else None
    v = np.ascontiguousarray(vertices, dtype=np.float64)
    rc = emu.emu_geo(p, small, nx, ny, nz, C.c_uint(faces), z0, nzl, czlo, czhi, zol, zoh, chunks, c5, _dp(v), mode, _dp(u),
                     _dp(b), _dp(xold), _dp(out), C.c_double(f1), C.c_double(f2), None, _dp(dv))
    assert rc == 0
    return (out, dv) if want_dinv else out


def _slab_of(p, n, cz_lo, cz_hi):
    Nz = n[2] * p + 1
    z0 = 0 if cz_lo == 0 else cz_lo * p - p
    z_end = Nz if cz_hi == n[2] else cz_hi * p + 1
    return z0, z_end - z0, cz_lo, cz_hi, cz_lo * p, (Nz if cz_hi == n[2] else cz_hi * p)


@pytest.mark.parametrize("p", range(1, 10))
@pytest.mark.parametrize("small,chunks", [(1, 1), (1, 2), (0, 2)])
def test_emulated_mapped_apply_matches_oracle(p, small, chunks, emu, oracle):
    n = (4, 3, 3) if p < 5 else (3, 2, 2)
    v = random_vertices(n, 0.2, seed=p)
    mf = mapped_matrix_free(oracle, p, n, v)
    u = splitmix_src(mf.n_dofs, salt=p)
    out = emu_geo(emu, p, n, v, u, small=small, chunks=chunks)
    assert not np.isnan(out).any()
    assert rel_l2(out, mf.vmult(u)) < 1e-13


@pytest.mark.parametrize("p", range(1, 10))
def test_emulated_mapped_epilogues_diagonal_faces(p, emu, oracle):
    n = (3, 2, 3) if p < 5 else (2, 2, 2)
    v = random_vertices(n, 0.2, seed=30 + p)
    for faces, coef in ((0x3F, None), (0x2A, "c5"), (0x00, None)):
        mf = mapped_matrix_free(oracle, p, n, v, faces=faces, coef=coef)
        c5 = 1 if coef else 0
        u, b, xo = (splitmix_src(mf.n_dofs, salt=s) for s in (21, 22, 23))
        Au, dinv = mf.vmult(u), mf.compute_diagonal()
        out, dv = emu_geo(emu, p, n, v, u, mode=2, b=b, f2=0.8, faces=faces, c5=c5, want_dinv=True)
        assert rel_l2(dv, dinv) < 1e-13
        assert rel_l2(out, u + 0.8 * dinv * (b - Au)) < 1e-13
        assert rel_l2(emu_geo(emu, p, n, v, u, faces=faces, c5=c5), Au) < 1e-13
        assert rel_l2(emu_geo(emu, p, n, v, u, mode=1, b=b, faces=faces, c5=c5), b - Au) < 1e-13
        ref = u + 0.3 * (u - xo) + 0.8 * dinv * (b - Au)
        assert rel_l2(emu_geo(emu, p, n, v, u, mode=3, b=b, xold=xo, f1=0.3, f2=0.8, faces=faces, c5=c5, chunks=2), ref) < 1e-13


@pytest.mark.parametrize("p,splits", [(1, [(0, 2), (2, 4)]), (3, [(0, 1), (1, 3), (3, 4)])])
def test_emulated_mapped_slabs(p, splits, emu, oracle):
    """z-slabs: each rank stores G of its own cell layers plus the ghost layer below, from its vertex planes only."""
    n = (3, 3, 4)
    v = smooth_map_vertices(n, 0.1)
    mf = mapped_matrix_free(oracle, p, n, v)
    u, b = splitmix_src(mf.n_dofs, salt=7), splitmix_src(mf.n_dofs, salt=8)
    ref = u + 0.6 * mf.compute_diagonal() * (b - mf.vmult(u))
    plane = mf.nd[0] * mf.nd[1]
    got = np.full(mf.n_dofs, np.nan)
    for lo, hi in splits:
        z0, nzl, _, _, zol, zoh = sl = _slab_of(p, n, lo, hi)
        ul, bl = u[z0 * plane:(z0 + nzl) * plane].copy(), b[z0 * plane:(z0 + nzl) * plane].copy()
        ol = emu_geo(emu, p, n, v, ul, mode=2, b=bl, f2=0.6, slab=sl, chunks=2)
        owned = np.zeros(nzl * plane, bool)
        owned[(zol - z0) * plane:(zoh - z0) * plane] = True
        assert np.isnan(ol[~owned]).all() and not np.isnan(ol[owned]).any()
        got[zol * plane:zoh * plane] = ol[owned]
    assert rel_l2(got, ref) < 1e-13
