"""The Laplace operator on curved hexahedral meshes (cells of geometry degree k, MappingQ(k)), on the CPU.

1. The oracle on a curved mesh (tests/curved_oracle.py: its per-point inv_jacobian / JxW filled from the degree-k maps)
   against an independent numpy dense assembly: operator, inverse diagonal, load vector and the QGauss(p+2) norm.
2. Nodes of geometry degree 2 that sample trilinear cells give the trilinear oracle; nodes of a polynomial map of degree
   <= k reproduce its analytic Jacobian, in the oracle and in the product's per-point routine (pmg_curved_map).
3. The quarter cylindrical shell: MappingQ(p) cells converge at order ~2p to the exact norm, trilinear cells stay at O(h^2).
4. The unchanged tensor tile program (PmgVarTile<.., GEO = true>) under the host emulator with G built by
   pmg_curved_point, against the curved oracle: all epilogues, z-chunks, tile sizes, slabs, faces, degrees 1..9.
"""
import ctypes as C

import numpy as np
import pytest

from curved_mesh import SHELL_FACES, SHELL_NORM, nodes_of, perturbed_map, shell_map, smooth_map, support_grid, trilinear_nodes
from curved_oracle import curved_cells, curved_matrix_free, l2_norm_curved
from helpers import hierarchy_levels, rel_l2, splitmix_src
from mapped_mesh import random_vertices
from mapped_oracle import geometry, mapped_matrix_free, ref_points
from test_oracle_dense import cell_dofs, constrained_mask, gauss, gll_nodes, kron_xyz, shape_1d

C5 = lambda x, y, z: 1.0 / (0.05 + 2.0 * (x * x + y * y + z * z))  # noqa: E731


def cell_map(nodes, n, k, cell, m):
    """x (m^3, 3) and J (m^3, 3, 3) of one cell at the m^3 Gauss points from the full 3-D Lagrange basis (kron of the 1-D
    tables: no sum factorisation), independent of tests/curved_oracle.py"""
    S, D = shape_1d(k, gauss(m)[0])
    cx, cy, cz = cell
    N = np.asarray(nodes).reshape(n[2] * k + 1, n[1] * k + 1, n[0] * k + 1, 3)
    X = N[cz * k:cz * k + k + 1, cy * k:cy * k + k + 1, cx * k:cx * k + k + 1].reshape(-1, 3)  # (node, d), x fastest
    x = kron_xyz([S, S, S]) @ X
    J = np.stack([kron_xyz([D, S, S]) @ X, kron_xyz([S, D, S]) @ X, kron_xyz([S, S, D]) @ X], axis=-1)
    return x, J


def dense_curved(p, n, faces, nodes, k, coef=None):
    """A_ij = sum_cells sum_q a(x_q) w_q |det J| (J^-T grad phi_i) . (J^-T grad phi_j), Dirichlet rows / columns replaced by
    the identity; the load vector of f = 1 with constrained rows dropped; the QGauss(p+2) mass matrix"""
    S, D = shape_1d(p, gauss(p + 1)[0])
    _, w = ref_points(p + 1)
    _, w2 = ref_points(p + 2)
    Gref = [kron_xyz([D if e == d else S for e in range(3)]) for d in range(3)]
    Sk = kron_xyz([S] * 3)
    E = kron_xyz([shape_1d(p, gauss(p + 2)[0])[0]] * 3)
    ndofs = int(np.prod([nd * p + 1 for nd in n]))
    A, b, M = np.zeros((ndofs, ndofs)), np.zeros(ndofs), np.zeros((ndofs, ndofs))
    for cell in np.ndindex(*n[::-1]):
        cell = cell[::-1]
        x, J = cell_map(nodes, n, k, cell, p + 1)
        det = np.linalg.det(J)
        assert (det > 0).all()
        Jinv = np.linalg.inv(J)
        wq = w * det * (coef(*x.T) if coef is not None else 1.0)
        grad = [sum(Jinv[:, d, e][:, None] * Gref[d] for d in range(3)) for e in range(3)]
        idx = cell_dofs(p, n, cell)
        A[np.ix_(idx, idx)] += sum(g.T @ (wq[:, None] * g) for g in grad)
        b[idx] += Sk.T @ (w * det)
        _, J2 = cell_map(nodes, n, k, cell, p + 2)
        M[np.ix_(idx, idx)] += E.T @ ((w2 * np.abs(np.linalg.det(J2)))[:, None] * E)
    c = constrained_mask(p, n, faces)
    A[c, :] = 0
    A[:, c] = 0
    A[c, c] = 1.0
    b[c] = 0.0
    return A, b, M, c


@pytest.mark.parametrize("p,k,n,faces,coef", [(1, 1, (3, 2, 2), 0x3F, None), (1, 2, (2, 2, 3), 0x0C, "c5"), (1, 3, (2, 2, 2), 0x3F, None),
                                              (2, 1, (2, 2, 2), 0x3F, "c5"), (2, 2, (2, 3, 2), 0x15, None), (2, 3, (3, 2, 2), 0x00, "c5"),
                                              (3, 1, (2, 2, 2), 0x2A, None), (3, 2, (2, 2, 2), 0x3F, "c5"), (3, 3, (2, 2, 2), 0x03, None),
                                              (4, 1, (2, 2, 1), 0x3F, "c5"), (4, 2, (2, 1, 2), 0x2A, None), (4, 3, (2, 2, 2), 0x3F, "c5")])
def test_curved_oracle_matches_dense_assembly(p, k, n, faces, coef, oracle):
    nodes = nodes_of(perturbed_map(0.03, seed=p + 10 * k), n, k)
    A, b, M, c = dense_curved(p, n, faces, nodes, k, C5 if coef else None)
    mf = curved_matrix_free(oracle, p, n, nodes, k, faces=faces, coef=coef)
    assert np.array_equal(mf.constrained(), c)
    rng = np.random.default_rng(p + k)
    for _ in range(2):
        u = rng.standard_normal(mf.n_dofs)
        assert rel_l2(mf.vmult(u), A @ u) < 1e-12
    assert rel_l2(mf.compute_diagonal(), 1.0 / np.diag(A)) < 1e-12
    if coef is None:
        assert rel_l2(mf.assemble_rhs(), b) < 1e-12
    u = rng.standard_normal(mf.n_dofs)
    ref = np.sqrt(u @ M @ u)
    assert abs(l2_norm_curved(mf, u) - ref) < 1e-12 * ref


@pytest.mark.parametrize("p,n,coef", [(1, (3, 2, 2), None), (2, (2, 3, 2), "c5"), (3, (2, 2, 3), None), (4, (2, 2, 2), "c5")])
def test_trilinear_sampled_nodes_give_trilinear_oracle(p, n, coef, oracle):
    v = random_vertices(n, 0.2, seed=40 + p)
    tri = mapped_matrix_free(oracle, p, n, v, coef=coef)
    cur = curved_matrix_free(oracle, p, n, trilinear_nodes(v, n, 2), 2, coef=coef)
    (ij0, jxw0), (ij1, jxw1) = geometry(tri), geometry(cur)
    assert np.abs(ij1 - ij0).max() <= 1e-13 * np.abs(ij0).max()
    assert np.abs(jxw1 - jxw0).max() <= 1e-13 * np.abs(jxw0).max()
    u = splitmix_src(tri.n_dofs, salt=p)
    assert rel_l2(cur.vmult(u), tri.vmult(u)) < 1e-13
    # k = 1 nodes are the vertices themselves
    assert np.array_equal(trilinear_nodes(v, n, 1), v)


def _poly_map(k):
    """a map of degree <= k in each reference variable, and its analytic Jacobian"""
    a = 0.3 / k

    def f(X, Y, Z):
        return np.stack([X + a * Y ** k * Z, Y + a * X ** k - 0.5 * a * Z ** k * X, Z + a * X * Y ** (k - 1)], axis=-1)

    def jac(X, Y, Z):
        J = np.zeros(X.shape + (3, 3))
        J[..., 0, 0], J[..., 0, 1], J[..., 0, 2] = 1.0, a * k * Y ** (k - 1) * Z, a * Y ** k
        J[..., 1, 0], J[..., 1, 1], J[..., 1, 2] = a * k * X ** (k - 1) - 0.5 * a * Z ** k, 1.0, -0.5 * a * k * Z ** (k - 1) * X
        J[..., 2, 0], J[..., 2, 1], J[..., 2, 2] = a * Y ** (k - 1), a * (k - 1) * X * Y ** max(k - 2, 0), 1.0
        return J
    return f, jac


@pytest.mark.parametrize("k", [1, 2, 3, 5])
def test_polynomial_map_reproduces_analytic_jacobian(k, emu):
    n = (2, 3, 2)
    f, jac = _poly_map(k)
    nodes = nodes_of(f, n, k)
    m = 4
    xi, _ = ref_points(m)
    xo, Jo = curved_cells(nodes, n, k, m)  # the oracle's contraction
    emu.emu_curved_map.argtypes = [C.c_int] * 3 + [C.c_void_p] + [C.c_int] * 4 + [C.c_void_p] * 3
    for ci, cell in enumerate(np.ndindex(*n[::-1])):
        cz, cy, cx = cell
        X = np.stack([(cx + xi[:, 0]) / n[0], (cy + xi[:, 1]) / n[1], (cz + xi[:, 2]) / n[2]], axis=1)
        J_ref = jac(*X.T) / np.array(n)[None, None, :]  # d x / d xi = d x / d X * dX / dxi
        x_ref = f(*X.T)
        assert np.abs(Jo[ci] - J_ref).max() < 1e-12 and np.abs(xo[ci] - x_ref).max() < 1e-12
        x, J = np.zeros((m ** 3, 3)), np.zeros((m ** 3, 3, 3))
        assert emu.emu_curved_map(k, n[0], n[1], nodes.ctypes.data, cx, cy, cz, m ** 3, np.ascontiguousarray(xi).ctypes.data,
                                  x.ctypes.data, J.ctypes.data) == 0
        assert np.abs(J - J_ref).max() < 1e-12 and np.abs(x - x_ref).max() < 1e-12


def test_mesh_nodes_on_the_support_grid(pmg):
    for k in (1, 2, 4, 9):
        assert np.abs(pmg.host_support_points(k) - gll_nodes(k)).max() < 1e-15
    n = (3, 2, 4)
    for k in (1, 3):
        assert np.abs(pmg.mesh_nodes(shell_map, n, k) - nodes_of(shell_map, n, k)).max() < 1e-15
    assert np.array_equal(support_grid(4, 1), np.arange(5) / 4)


def shell_solve(oracle, p, n, k):
    """the oracle's solution of -Delta u = 1 on the shell (n^3 cells of geometry degree k; k = 0: the level's degree) with
    a V-cycle-preconditioned CG to 1e-13, and its relative QGauss(p+2) norm error"""
    levels = hierarchy_levels("h", p, n)
    mfs = [curved_matrix_free(oracle, q, m, nodes_of(shell_map, m, k or q), k or q, faces=SHELL_FACES) for (q, m) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h") for l in range(1, len(levels))]
    vc = oracle.VCycle(mfs, trs)
    vc.estimate()
    x, _, _, rc = oracle.cg_solve(mfs[-1], mfs[-1].assemble_rhs(), vc, rel_tol=1e-13)
    assert rc == 0
    return abs(l2_norm_curved(mfs[-1], x) - SHELL_NORM) / SHELL_NORM


# relative errors of the norm with MappingQ(p) cells (Q2 and Q3 at 2, 4, 8 cells per direction; Q4 at 2 and 4)
SHELL_TABLE = {(2, 2): 1.2e-3, (2, 4): 6.4e-5, (2, 8): 3.8e-6, (3, 2): 2.2e-5, (3, 4): 3.9e-7, (3, 8): 6.3e-9,
               (4, 2): 1.2e-7, (4, 4): 6.5e-10}


@pytest.mark.parametrize("p,n", sorted(SHELL_TABLE))
def test_shell_converges_with_mapping_q(p, n, oracle):
    err = shell_solve(oracle, p, n, 0)
    assert SHELL_TABLE[p, n] / 3 <= err <= 3 * SHELL_TABLE[p, n], err


@pytest.mark.parametrize("p", [2, 3])
def test_shell_trilinear_cells_stay_second_order(p, oracle):
    assert shell_solve(oracle, p, 8, 1) > 5e-3


# ---- the tensor tile program under the host emulator, G from pmg_curved_point -----------------------------------
def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def emu_curved(emu, p, k, n, nodes, u, mode=0, b=None, xold=None, f1=0.0, f2=0.0, small=1, chunks=1, faces=0x3F, c5=0,
               slab=None, want_dinv=False):
    nx, ny, nz = n
    Nz = nz * p + 1
    z0, nzl, czlo, czhi, zol, zoh = (0, Nz, 0, nz, 0, Nz) if slab is None else slab
    out = np.full(u.shape, np.nan)
    dv = np.empty(u.shape) if want_dinv else None
    v = np.ascontiguousarray(nodes, dtype=np.float64)
    rc = emu.emu_curved(p, k, small, nx, ny, nz, C.c_uint(faces), z0, nzl, czlo, czhi, zol, zoh, chunks, c5, _dp(v), mode, _dp(u),
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
def test_emulated_curved_apply_matches_oracle(p, small, chunks, emu, oracle):
    n = (4, 3, 3) if p < 5 else (3, 2, 2)
    nodes = nodes_of(perturbed_map(0.03, seed=p), n, p)
    mf = curved_matrix_free(oracle, p, n, nodes, p)
    u = splitmix_src(mf.n_dofs, salt=p)
    out = emu_curved(emu, p, p, n, nodes, u, small=small, chunks=chunks)
    assert not np.isnan(out).any()
    assert rel_l2(out, mf.vmult(u)) < 1e-13


@pytest.mark.parametrize("p", range(1, 10))
def test_emulated_curved_epilogues_diagonal_faces(p, emu, oracle):
    n = (3, 2, 3) if p < 5 else (2, 2, 2)
    nodes = nodes_of(shell_map, n, p)
    for faces, coef in ((0x3F, None), (0x2A, "c5"), (SHELL_FACES, None)):
        mf = curved_matrix_free(oracle, p, n, nodes, p, faces=faces, coef=coef)
        c5 = 1 if coef else 0
        u, b, xo = (splitmix_src(mf.n_dofs, salt=s) for s in (21, 22, 23))
        Au, dinv = mf.vmult(u), mf.compute_diagonal()
        out, dv = emu_curved(emu, p, p, n, nodes, u, mode=2, b=b, f2=0.8, faces=faces, c5=c5, want_dinv=True)
        assert rel_l2(dv, dinv) < 1e-13
        assert rel_l2(out, u + 0.8 * dinv * (b - Au)) < 1e-13
        assert rel_l2(emu_curved(emu, p, p, n, nodes, u, faces=faces, c5=c5), Au) < 1e-13
        assert rel_l2(emu_curved(emu, p, p, n, nodes, u, mode=1, b=b, faces=faces, c5=c5), b - Au) < 1e-13
        ref = u + 0.3 * (u - xo) + 0.8 * dinv * (b - Au)
        assert rel_l2(emu_curved(emu, p, p, n, nodes, u, mode=3, b=b, xold=xo, f1=0.3, f2=0.8, faces=faces, c5=c5, chunks=2), ref) < 1e-13


@pytest.mark.parametrize("p,k,splits", [(1, 3, [(0, 2), (2, 4)]), (3, 3, [(0, 1), (1, 3), (3, 4)]), (2, 4, [(0, 3), (3, 4)])])
def test_emulated_curved_slabs(p, k, splits, emu, oracle):
    """z-slabs: each rank builds G of its own cell layers plus the ghost layer below from its node planes only."""
    n = (3, 3, 4)
    nodes = nodes_of(smooth_map(0.1), n, k)
    mf = curved_matrix_free(oracle, p, n, nodes, k)
    u, b = splitmix_src(mf.n_dofs, salt=7), splitmix_src(mf.n_dofs, salt=8)
    ref = u + 0.6 * mf.compute_diagonal() * (b - mf.vmult(u))
    plane = mf.nd[0] * mf.nd[1]
    got = np.full(mf.n_dofs, np.nan)
    for lo, hi in splits:
        z0, nzl, _, _, zol, zoh = sl = _slab_of(p, n, lo, hi)
        ul, bl = u[z0 * plane:(z0 + nzl) * plane].copy(), b[z0 * plane:(z0 + nzl) * plane].copy()
        ol = emu_curved(emu, p, k, n, nodes, ul, mode=2, b=bl, f2=0.6, slab=sl, chunks=2)
        owned = np.zeros(nzl * plane, bool)
        owned[(zol - z0) * plane:(zoh - z0) * plane] = True
        assert np.isnan(ol[~owned]).all() and not np.isnan(ol[owned]).any()
        got[zol * plane:zoh * plane] = ol[owned]
    assert rel_l2(got, ref) < 1e-13
