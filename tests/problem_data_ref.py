"""numpy reference of the problem-data entries (test infrastructure, pinned by tests/test_problem_data_cpu.py).

The load vector of the nodal interpolant f_h = sum_j f_j phi_j is  b = sum_cells S^T diag(JxW_c) S f_c  with S the FE_Q(p)
shape values at the QGauss(p+1) points (kron of the 1-D table) and JxW_c the cell's w_q |det J_q|, the same arrays the
oracle stores (tests/mapped_oracle.py geometry(), tests/curved_oracle.py).  The lifting of Dirichlet values g is
A_free g_D: the oracle's vmult on the same mesh without Dirichlet faces, applied to g masked to the constrained dofs.
Support points are the Gauss-Lobatto grid of every cell mapped by the cell's geometry.
"""
import numpy as np

from curved_oracle import basis_1d
from test_oracle_dense import gauss, gll_nodes


def cell_dof_table(p, n):
    """(nc, (p+1)^dim) global lexicographic dof indices of every cell's local dofs, cells and local dofs x fastest"""
    dim = len(n)
    N = [nd * p + 1 for nd in n]
    r = np.arange(p + 1)
    if dim == 2:
        cy, cx = np.meshgrid(np.arange(n[1]), np.arange(n[0]), indexing="ij")
        iy = (p * cy.ravel())[:, None, None] + r[None, :, None]
        ix = (p * cx.ravel())[:, None, None] + r[None, None, :]
        return (iy * N[0] + ix).reshape(-1, (p + 1) ** 2)
    cz, cy, cx = np.meshgrid(np.arange(n[2]), np.arange(n[1]), np.arange(n[0]), indexing="ij")
    iz = (p * cz.ravel())[:, None, None, None] + r[None, :, None, None]
    iy = (p * cy.ravel())[:, None, None, None] + r[None, None, :, None]
    ix = (p * cx.ravel())[:, None, None, None] + r[None, None, None, :]
    return ((iz * N[1] + iy) * N[0] + ix).reshape(-1, (p + 1) ** 3)


def shape_matrix(p, dim):
    """(nq, nloc) values of the cell's shape functions at its QGauss(p+1) points, both lexicographic (x fastest)"""
    S = basis_1d(p, gauss(p + 1)[0])[0]  # barycentric form: exact to round-off up to Q9
    out = S
    for _ in range(dim - 1):
        out = np.kron(S, out)
    return out


def box_jxw(p, n):
    """(nc, nq) w_q |det J| of the unit cube's (square's) equal cells"""
    w = gauss(p + 1)[1]
    out = w * (1.0 / n[0])
    for d in range(1, len(n)):
        out = np.kron(w * (1.0 / n[d]), out)
    return np.tile(out, (int(np.prod(n)), 1))


def load_vector(p, n, jxw, f, constrained):
    """sum_cells S^T diag(JxW_c) S f_c, constrained rows 0"""
    n = tuple(n)
    l2g = cell_dof_table(p, n)
    S = shape_matrix(p, len(n))
    fq = np.asarray(f)[l2g] @ S.T  # (nc, nq): f_h at the Gauss points
    cell = (jxw * fq) @ S  # (nc, nloc)
    b = np.zeros(int(np.prod([nd * p + 1 for nd in n])))
    np.add.at(b, l2g.ravel(), cell.ravel())
    b[constrained] = 0.0
    return b


def rhs_reference(p, n, jxw, constrained, f=None, g=None, mf_free=None):
    """M f_h - A_free g_D on unconstrained rows, 0 on constrained rows; mf_free: the oracle MatrixFree of the same mesh,
    coefficient and geometry with faces = 0 (needed when g is given)"""
    m = int(np.prod([nd * p + 1 for nd in n]))
    b = load_vector(p, n, jxw, f, constrained) if f is not None else np.zeros(m)
    if g is not None:
        gD = np.where(constrained, g, 0.0)
        b = b - mf_free.vmult(gD)
        b[constrained] = 0.0
    return b


def dof_cells_1d(p, nc):
    """cell index and Gauss-Lobatto point of every dof of an nc-cell direction: the lower cell at a cell boundary"""
    g = np.arange(nc * p + 1)
    c = np.minimum(g // p, nc - 1)
    return c, gll_nodes(p)[g - c * p]


def box_support_points(p, n):
    """(m, dim): the Gauss-Lobatto grid (c + s_i) / n_d, global lexicographic order"""
    lines = []
    for nd in n:
        c, s = dof_cells_1d(p, nd)
        lines.append((c + s) / nd)
    grids = np.meshgrid(*lines[::-1], indexing="ij")[::-1]
    return np.stack([gr.ravel() for gr in grids], axis=1)


def trilinear_support_points(p, n, vertices):
    """(m, 3): every dof's trilinear cell map at its Gauss-Lobatto point"""
    V = np.asarray(vertices, dtype=np.float64).reshape(n[2] + 1, n[1] + 1, n[0] + 1, 3)
    (cx, sx), (cy, sy), (cz, sz) = (dof_cells_1d(p, n[d]) for d in range(3))
    out = 0.0
    for c in range(8):
        i, j, k = c & 1, c >> 1 & 1, c >> 2
        w = ((sz if k else 1.0 - sz)[:, None, None] * (sy if j else 1.0 - sy)[None, :, None]
             * (sx if i else 1.0 - sx)[None, None, :])
        out = out + w[..., None] * V[(cz + k)[:, None, None], (cy + j)[None, :, None], (cx + i)[None, None, :]]
    return out.reshape(-1, 3)


def curved_support_points(p, n, nodes, k):
    """(m, 3): every dof's degree-k cell map (MappingQ(k)) at its degree-p Gauss-Lobatto point"""
    Nn = np.asarray(nodes, dtype=np.float64).reshape(n[2] * k + 1, n[1] * k + 1, n[0] * k + 1, 3)
    L, idx = [], []
    for d in range(3):
        c, s = dof_cells_1d(p, n[d])
        L.append(basis_1d(k, s)[0])  # (N_d, k+1)
        idx.append(c[:, None] * k + np.arange(k + 1)[None, :])  # (N_d, k+1) node index
    G = Nn[idx[2][:, :, None, None, None, None], idx[1][None, None, :, :, None, None], idx[0][None, None, None, None, :, :]]
    return np.einsum("zl,yj,xi,zlyjxid->zyxd", L[2], L[1], L[0], G).reshape(-1, 3)
