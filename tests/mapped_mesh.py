"""Deformed structured hexahedral meshes for the mapped-geometry tests (CPU and GPU modules).

Vertices are arrays of shape (nz+1, ny+1, nx+1, 3): global lexicographic order, x fastest, xyz interleaved -- the layout
pmg_laplace_operator_create_mapped and tests/mapped_oracle.py take.
"""
import numpy as np


def uniform_vertices(n, box=(1.0, 1.0, 1.0)):
    z, y, x = np.meshgrid(*[np.arange(n[d] + 1) * (box[d] / n[d]) for d in (2, 1, 0)], indexing="ij")
    return np.ascontiguousarray(np.stack([x, y, z], axis=-1))


def random_vertices(n, amount=0.2, seed=0):
    """The unit cube's uniform grid with every interior vertex moved by up to amount * h per coordinate (seeded);
    boundary vertices stay, so the domain is the unit cube."""
    v = uniform_vertices(n)
    rng = np.random.default_rng(seed)
    h = np.array([1.0 / n[0], 1.0 / n[1], 1.0 / n[2]])
    d = rng.uniform(-amount, amount, size=v.shape) * h
    d[0, :, :] = d[-1, :, :] = 0.0
    d[:, 0, :] = d[:, -1, :] = 0.0
    d[:, :, 0] = d[:, :, -1] = 0.0
    return np.ascontiguousarray(v + d)


def smooth_map_vertices(n, eps):
    """x -> x + eps sin(pi x) sin(pi y) sin(pi z) (1, 1, 1) of the uniform grid: fixes the boundary of the unit cube."""
    v = uniform_vertices(n)
    s = eps * np.sin(np.pi * v[..., 0]) * np.sin(np.pi * v[..., 1]) * np.sin(np.pi * v[..., 2])
    return np.ascontiguousarray(v + s[..., None])


def sheared_box_vertices(n):
    """[0, 2] x [0, 1] x [0, 0.5], then the shear (x, y, z) -> (x + 0.3 y + 0.2 z, y + 0.1 z, z): every cell affine."""
    v = uniform_vertices(n, (2.0, 1.0, 0.5))
    x, y, z = v[..., 0], v[..., 1], v[..., 2]
    return np.ascontiguousarray(np.stack([x + 0.3 * y + 0.2 * z, y + 0.1 * z, z], axis=-1))


def cell_vertices(vertices, cell):
    """the 8 vertices of cell (cx, cy, cz), index c = i + 2 j + 4 k for vertex (cx+i, cy+j, cz+k)"""
    cx, cy, cz = cell
    return np.array([vertices[cz + k, cy + j, cx + i] for k in (0, 1) for j in (0, 1) for i in (0, 1)])


def trilinear(V, xi):
    """x(xi) and J (npts, 3, 3) with J[:, d, e] = d x_d / d xi_e of the trilinear map with vertices V (8, 3) at the
    reference points xi (npts, 3)"""
    x = np.zeros((len(xi), 3))
    J = np.zeros((len(xi), 3, 3))
    for c in range(8):
        ijk = (c & 1, c >> 1 & 1, c >> 2)
        L = np.stack([xi[:, d] if ijk[d] else 1.0 - xi[:, d] for d in range(3)], axis=1)
        dL = np.array([1.0 if ijk[d] else -1.0 for d in range(3)])
        x += np.prod(L, axis=1)[:, None] * V[c]
        for e in range(3):
            f = np.prod(np.where(np.arange(3) == e, dL[None, :], L), axis=1)
            J[:, :, e] += f[:, None] * V[c][None, :]
    return x, J
