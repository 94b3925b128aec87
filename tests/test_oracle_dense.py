"""The oracle against an INDEPENDENT dense assembly of the same discretisation (numpy only).

The reference ships no tests or golden vectors (SURVEY.md section 4), so the oracle -- a C restatement of the reference's
matrix-free algorithm: stored indices, masks, per-q-point Jacobians, 12 one-dimensional sweeps per cell, scatter-add -- is pinned
here against the textbook definition of what that algorithm computes, written a second time with nothing in common but the
published ingredients (SURVEY.md section 8c: FE_Q(p) = Lagrange basis on Gauss-Lobatto nodes, QGauss(p+1), Cartesian cells of the
unit cube, lexicographic numbering, Dirichlet rows / columns replaced by the identity):

    A_ij = sum_cells sum_q  a(x_q) w_q |J|  grad phi_i(x_q) . grad phi_j(x_q)

assembled as a dense matrix from numpy's Legendre routines (nodes, weights, polynomial arithmetic), cell by cell through an
explicit local-to-global map.  Same for the transfers (interpolation matrices of nested spaces) and the inverse diagonal.
"""
import numpy as np
import pytest
from numpy.polynomial import legendre as L
from numpy.polynomial import polynomial as Pn

from helpers import rel_l2


# ---- published ingredients, from numpy only ------------------------------------------------------------------------
def gll_nodes(p):
    """p + 1 Gauss-Lobatto points on [0, 1]: the end points and the roots of P_p'."""
    if p == 1:
        return np.array([0.0, 1.0])
    inner = L.legroots(L.legder([0] * p + [1]))
    return 0.5 * (np.concatenate([[-1.0], np.sort(inner.real), [1.0]]) + 1.0)


def gauss(nq):
    x, w = L.leggauss(nq)
    return 0.5 * (x + 1.0), 0.5 * w


def lagrange(nodes):
    """Monomial coefficients (ascending) of the Lagrange polynomials on `nodes`."""
    out = []
    for i, xi in enumerate(nodes):
        c = np.array([1.0])
        for j, xj in enumerate(nodes):
            if j != i:
                c = Pn.polymul(c, np.array([-xj, 1.0]) / (xi - xj))
        out.append(c)
    return out


def shape_1d(p, x):
    """values and derivatives of the FE_Q(p) basis of the unit interval at the points x: two (len(x), p + 1) arrays"""
    basis = lagrange(gll_nodes(p))
    S = np.stack([Pn.polyval(x, c) for c in basis], axis=1)
    D = np.stack([Pn.polyval(x, Pn.polyder(c)) for c in basis], axis=1)
    return S, D


def dof_grid(p, n):
    """dofs per direction and the coordinates of the 1-D dof lines of an n-cell mesh of the unit cube"""
    g = gll_nodes(p)
    return [np.concatenate([(c + g[:-1]) / nd for c in range(nd)] + [[1.0]]) for nd in n]


def cell_dofs(p, n, cell):
    """global lexicographic (x fastest) dof indices of a cell's local dofs, local numbering lexicographic as well"""
    dim = len(n)
    N = [nd * p + 1 for nd in n]
    idx = np.zeros([p + 1] * dim, dtype=np.int64)
    for loc in np.ndindex(*[p + 1] * dim):  # loc = (i_z, i_y, i_x) in 3-D
        g, stride = 0, 1
        for d in range(dim):  # d = 0 is x
            g += (cell[d] * p + loc[dim - 1 - d]) * stride
            stride *= N[d]
        idx[loc] = g
    return idx.ravel()


def constrained_mask(p, n, faces):
    dim = len(n)
    N = [nd * p + 1 for nd in n]
    grids = np.meshgrid(*[np.arange(N[d]) for d in range(dim)][::-1], indexing="ij")[::-1]  # grids[d] = index along d, x fastest
    m = np.zeros(grids[0].shape, bool)
    for d in range(dim):
        if faces >> (2 * d) & 1:
            m |= grids[d] == 0
        if faces >> (2 * d + 1) & 1:
            m |= grids[d] == N[d] - 1
    return m.ravel()


def dense_operator(p, n, faces, coef=None):
    """Dense A with Dirichlet rows / columns replaced by the identity, and the mask."""
    dim = len(n)
    nq = p + 1
    xq, wq = gauss(nq)
    S, D = shape_1d(p, xq)
    h = [1.0 / nd for nd in n]
    ndofs = int(np.prod([nd * p + 1 for nd in n]))
    A = np.zeros((ndofs, ndofs))
    for cell in np.ndindex(*n[::-1]):  # (c_z, c_y, c_x)
        cell = cell[::-1]
        # tensor-product tables at the cell's quadrature points, q and local index lexicographic with x fastest
        def kron_all(mats):  # mats[d] for d = x, y, z  ->  kron(z, kron(y, x))
            out = mats[0]
            for d in range(1, dim):
                out = np.kron(mats[d], out)
            return out
        w = kron_all([wq[:, None] * h[d] for d in range(dim)]).ravel()
        if coef is not None:
            X = [kron_all([((cell[d] + xq) * h[d])[:, None] if e == d else np.ones((nq, 1)) for e in range(dim)]).ravel() for d in range(dim)]
            w = w * coef(*X)
        Ac = np.zeros(((p + 1) ** dim,) * 2)
        for d in range(dim):
            G = kron_all([D / h[e] if e == d else S for e in range(dim)])  # d/dx_d of every local basis function at every q
            Ac += G.T @ (w[:, None] * G)
        idx = cell_dofs(p, n, cell)
        A[np.ix_(idx, idx)] += Ac
    c = constrained_mask(p, n, faces)
    A[c, :] = 0
    A[:, c] = 0
    A[c, c] = 1.0
    return A, c


def interpolation_1d(p_from, n_from, p_to, n_to):
    """(dofs_to, dofs_from): values at the `to` dof line of the FE functions of the `from` space (nested spaces of [0, 1])."""
    x_to = dof_grid(p_to, [n_to])[0]
    Nf = n_from * p_from + 1
    M = np.zeros((len(x_to), Nf))
    g = gll_nodes(p_from)
    for r, x in enumerate(x_to):
        c = min(int(np.floor(x * n_from + 1e-12)), n_from - 1)
        xi = x * n_from - c
        for i in range(p_from + 1):
            # product form of the Lagrange polynomial: monomial coefficients lose ~1e-11 to cancellation at degree 9
            v = np.prod([(xi - g[j]) / (g[i] - g[j]) for j in range(p_from + 1) if j != i])
            M[r, c * p_from + i] = v  # a vertex of the `from` mesh is found in one cell only: assigned, not summed
    return M


def kron_xyz(mats):
    out = mats[0]
    for m in mats[1:]:
        out = np.kron(m, out)
    return out


# ---- the tests -----------------------------------------------------------------------------------------------------
def test_ingredients(oracle):
    for p in range(1, 9):
        assert np.abs(gll_nodes(p) - oracle.gauss_lobatto(p + 1)).max() < 1e-14
        x, w = gauss(p + 1)
        xo, wo = oracle.gauss_legendre(p + 1)
        assert np.abs(x - xo).max() < 1e-14 and np.abs(w - wo).max() < 1e-14


@pytest.mark.parametrize("p,n,faces", [(1, (3, 2, 2), 0x3F), (2, (2, 3, 2), 0x3F), (3, (2, 2, 2), 0x15), (4, (2, 1, 2), 0x3F),
                                       (5, (1, 2, 1), 0x2A), (2, (3, 2, 2), 0x00), (3, (4, 3), 0x0F), (7, (2, 2), 0x0F), (4, (3, 2), 0x05)])
def test_operator_matches_dense_assembly(p, n, faces, oracle):
    A, c = dense_operator(p, n, faces)
    mf = oracle.MatrixFree(len(n), p, n, faces=faces)
    assert mf.n_dofs == A.shape[0] and np.array_equal(mf.constrained(), c)
    rng = np.random.default_rng(p)
    for _ in range(3):
        u = rng.standard_normal(mf.n_dofs)  # non-zero on constrained dofs: identity rows
        assert rel_l2(mf.vmult(u), A @ u) < 1e-12
    assert rel_l2(mf.compute_diagonal(), 1.0 / np.diag(A)) < 1e-12


@pytest.mark.parametrize("p,n", [(1, (3, 3, 2)), (2, (2, 2, 2)), (3, (2, 1, 2)), (5, (1, 1, 2))])
def test_variable_coefficient_operator_matches_dense_assembly(p, n, oracle):
    """BASELINE config 5's operator -div(a grad u), a = 1 / (0.05 + 2 |x|^2) at the quadrature points (SURVEY.md section 8d)."""
    A, c = dense_operator(p, n, 0x3F, coef=lambda x, y, z: 1.0 / (0.05 + 2.0 * (x * x + y * y + z * z)))
    mf = oracle.MatrixFree(3, p, n, coef="c5")
    rng = np.random.default_rng(10 + p)
    u = rng.standard_normal(mf.n_dofs)
    assert rel_l2(mf.vmult(u), A @ u) < 1e-12
    assert rel_l2(mf.compute_diagonal(), 1.0 / np.diag(A)) < 1e-12


_TRANSFER_CASES = [("h", 1, 1, (2, 2, 1)), ("h", 2, 2, (2, 1, 2)), ("h", 3, 3, (1, 2, 1)), ("h", 4, 4, (2, 2)),
                   ("p", 1, 2, (2, 3, 2)), ("p", 2, 4, (2, 2, 1)), ("p", 1, 3, (3, 2)), ("p", 3, 7, (2, 2)), ("p", 2, 5, (1, 2, 2))]
# natural faces (the oracle's transfers skip constrained dofs by face) and the degrees 5..9 of the GPU transfers' generic kernels:
# h Q5..Q9, and the p pairs of the halving hierarchies and of the largest degree gaps
_TRANSFER_CASES_FACES = [(kind, pc, pf, n, faces) for (kind, pc, pf, n) in
                         [("h", 1, 1, (2, 1, 2)), ("h", 2, 2, (1, 2, 2)), ("h", 5, 5, (1, 2, 1)), ("h", 6, 6, (2, 1, 1)),
                          ("h", 7, 7, (1, 1, 2)), ("h", 8, 8, (1, 2, 1)), ("h", 9, 9, (1, 1, 1)), ("p", 1, 2, (2, 1, 2)),
                          ("p", 1, 3, (1, 2, 1)), ("p", 2, 5, (2, 1, 1)), ("p", 3, 6, (1, 1, 2)), ("p", 3, 7, (1, 2, 1)),
                          ("p", 4, 8, (2, 1, 1)), ("p", 4, 9, (1, 1, 2)), ("p", 2, 9, (1, 2, 1)), ("p", 8, 9, (2, 1, 1))]
                         for faces in (0x00, 0x15, 0x2A, 0x03, 0x30, 0x09)]


@pytest.mark.parametrize("kind,pc,pf,n,faces",
                         [pytest.param(*c, 0x3F if len(c[3]) == 3 else 0x0F, id="%s-%d-%d-n%d" % (*c[:3], i)) for i, c in enumerate(_TRANSFER_CASES)] +
                         [pytest.param(*c, id="%s-%d-%d-%s-f%02x" % (*c[:3], "x".join(map(str, c[3])), c[4])) for c in _TRANSFER_CASES_FACES])
def test_transfers_match_dense_interpolation(kind, pc, pf, n, faces, oracle):
    """prolongate_and_add: x_f += Z_f P x_c; restrict_and_add: x_c += Z_c P^T Z_f x_f, P = interpolation between the nested spaces
    (the reference realises Z by zero weights and invalid coarse indices, SURVEY.md section 8a8)."""
    dim = len(n)
    nf = tuple(2 * c for c in n) if kind == "h" else n
    Pd = kron_xyz([interpolation_1d(pc, n[d], pf, nf[d]) for d in range(dim)])
    zc, zf = ~constrained_mask(pc, n, faces), ~constrained_mask(pf, nf, faces)
    mc, mf = oracle.MatrixFree(dim, pc, n, faces=faces), oracle.MatrixFree(dim, pf, nf, faces=faces)
    t = oracle.Transfer(mc, mf, kind)
    rng = np.random.default_rng(pc + 10 * pf)
    xc, xf = rng.standard_normal(mc.n_dofs), rng.standard_normal(mf.n_dofs)
    d0 = rng.standard_normal(mf.n_dofs)
    got = t.prolongate_and_add(d0.copy(), xc * zc)  # constrained coarse values are zero in every vector the V-cycle prolongates
    assert rel_l2(got, d0 + zf * (Pd @ (xc * zc))) < 1e-12
    c0 = rng.standard_normal(mc.n_dofs)
    got = t.restrict_and_add(c0.copy(), xf)
    assert rel_l2(got, c0 + zc * (Pd.T @ (zf * xf))) < 1e-12


@pytest.mark.parametrize("p,n", [(2, (2, 2, 2)), (3, (3, 2)), (4, (2, 1, 2))])
def test_load_vector_and_solution_norm_match_dense(p, n, oracle):
    """Right-hand side of f = 1 with constrained rows dropped (program.cc:289-334) and the printed L2 norm of a FE function."""
    dim = len(n)
    xq, wq = gauss(p + 1)
    S, _ = shape_1d(p, xq)
    h = [1.0 / nd for nd in n]
    faces = 0x3F if dim == 3 else 0x0F
    ndofs = int(np.prod([nd * p + 1 for nd in n]))
    b, Mass = np.zeros(ndofs), np.zeros((ndofs, ndofs))
    for cell in np.ndindex(*n[::-1]):
        cell = cell[::-1]
        Sk = kron_xyz([S] * dim)
        w = kron_xyz([wq[:, None] * h[d] for d in range(dim)]).ravel()
        idx = cell_dofs(p, n, cell)
        b[idx] += Sk.T @ w
        Mass[np.ix_(idx, idx)] += Sk.T @ (w[:, None] * Sk)
    c = constrained_mask(p, n, faces)
    b[c] = 0
    mf = oracle.MatrixFree(dim, p, n)
    assert rel_l2(mf.assemble_rhs(), b) < 1e-13
    u = np.random.default_rng(3).standard_normal(ndofs)
    assert abs(mf.l2_norm_solution(u) - np.sqrt(u @ Mass @ u)) < 1e-12 * np.sqrt(u @ Mass @ u)
