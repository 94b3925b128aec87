"""Curved structured hexahedral meshes for the curved-geometry tests (CPU and GPU modules).

A mesh of n = (nx, ny, nz) cells with geometry degree k is given by its (nx k+1)(ny k+1)(nz k+1) geometry support points,
shape (nz k+1, ny k+1, nx k+1, 3), x fastest: the layout of pmg_laplace_operator_create_curved and tests/curved_oracle.py.
Node (cx k + i, cy k + j, cz k + l) of cell (cx, cy, cz) sits at the Gauss-Lobatto point (i, j, l) of FE_Q(k) on the
reference cell.  Everything here is numpy only (the grid comes from tests/test_oracle_dense.py's Gauss-Lobatto points).
"""
import numpy as np

from test_oracle_dense import gll_nodes

SHELL_FACES = 0x3  # Dirichlet on r = 1 (reference face x-low) and r = 2 (x-high), natural conditions elsewhere
SHELL_NORM = 0.14143644722133  # ||u||_L2 of u = (1 - r^2)/4 + 3 ln r / (4 ln 2): (pi/2) int_1^2 u^2 r dr, scipy quad


def shell_map(X, Y, Z):
    """the unit cube onto the quarter cylindrical shell 1 <= r <= 2, 0 <= theta <= pi/2, 0 <= z <= 1"""
    r, th = 1.0 + X, 0.5 * np.pi * Y
    return np.stack([r * np.cos(th), r * np.sin(th), Z], axis=-1)


def smooth_map(eps):
    """x -> x + eps sin(pi x) sin(pi y) sin(pi z) (1, 1, 1): the drivers' --distort map; it keeps the unit cube"""
    def f(X, Y, Z):
        s = eps * np.sin(np.pi * X) * np.sin(np.pi * Y) * np.sin(np.pi * Z)
        return np.stack([X + s, Y + s, Z + s], axis=-1)
    return f


def perturbed_map(amount=0.03, seed=0):
    """a smooth, seeded, non-polynomial perturbation of the identity: component c moves by amount times two products of
    sines of random amplitude (|a| <= 1) and phase, of frequencies pi and 2 pi.  Each entry of the perturbation's gradient
    is at most 3 pi amount, so for amount <= 0.035 its Frobenius norm stays below 1 and det J > 0 everywhere."""
    rng = np.random.default_rng(seed)
    a = rng.uniform(-1.0, 1.0, size=(3, 2))
    ph = rng.uniform(0.0, 2.0 * np.pi, size=(3, 2, 3))

    def f(X, Y, Z):
        P = [X, Y, Z]
        out = []
        for c in range(3):
            d = sum(a[c, m] * np.sin((m + 1) * np.pi * X + ph[c, m, 0]) * np.sin((m + 1) * np.pi * Y + ph[c, m, 1])
                    * np.sin((m + 1) * np.pi * Z + ph[c, m, 2]) for m in range(2))
            out.append(P[c] + amount * d)
        return np.stack(out, axis=-1)
    return f


def support_grid(n, k):
    """the 1-D node coordinates of an n-cell direction at geometry degree k: (c + s_i) / n, s = the GLL points"""
    s = gll_nodes(k)
    return np.concatenate([(c + s[:-1]) / n for c in range(n)] + [[1.0]])


def nodes_of(mapping, n, k):
    """the geometry support points of the image of the unit cube's n-cell mesh under mapping (pmg_b200.mesh_nodes)"""
    n = (n,) * 3 if isinstance(n, int) else tuple(n)
    Z, Y, X = np.meshgrid(support_grid(n[2], k), support_grid(n[1], k), support_grid(n[0], k), indexing="ij")
    return np.ascontiguousarray(mapping(X, Y, Z), dtype=np.float64)


def trilinear_nodes(vertices, n, k):
    """nodes of geometry degree k that sample the trilinear cells of `vertices` ((nz+1, ny+1, nx+1, 3)): every cell's
    degree-k interpolant is then its trilinear map"""
    n = (n,) * 3 if isinstance(n, int) else tuple(n)
    V = np.asarray(vertices, dtype=np.float64)
    g = [support_grid(n[d], k) * n[d] for d in range(3)]  # in cell units
    out = np.zeros((len(g[2]), len(g[1]), len(g[0]), 3))
    for iz, tz in enumerate(g[2]):
        cz = min(int(tz), n[2] - 1)
        fz = tz - cz
        for iy, ty in enumerate(g[1]):
            cy = min(int(ty), n[1] - 1)
            fy = ty - cy
            cx = np.minimum(g[0].astype(int), n[0] - 1)
            fx = (g[0] - cx)[:, None]
            acc = 0.0
            for c in range(8):
                i, j, l = c & 1, c >> 1 & 1, c >> 2
                w = (fx if i else 1.0 - fx) * (fy if j else 1.0 - fy) * (fz if l else 1.0 - fz)
                acc = acc + w * V[cz + l, cy + j, cx + i]
            out[iz, iy] = acc
    return np.ascontiguousarray(out)
