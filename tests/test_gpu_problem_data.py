"""GPU tests of the problem-data entries: support_points, assemble_rhs_data (load vector of a nodal f, Dirichlet lifting)
and distribute, against the numpy reference of tests/problem_data_ref.py (pinned by tests/test_problem_data_cpu.py) and the
oracle, on box, coefficient-1, trilinear and curved operators, then the whole workflow and its convergence."""
import os
import subprocess
import sys

import numpy as np
import pytest

from curved_mesh import SHELL_FACES, nodes_of, perturbed_map, shell_map
from curved_oracle import curved_matrix_free
from helpers import hierarchy_levels, rel_l2, splitmix_src
from mapped_mesh import random_vertices, sheared_box_vertices
from mapped_oracle import geometry, mapped_matrix_free
from problem_data_ref import (box_jxw, box_support_points, curved_support_points, rhs_reference,
                              trilinear_support_points)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEGREES = [1, 2, 3, 4, 5, 6, 7, 8, 9]


def _cells(p, dim=3):
    n = {1: (5, 4, 6), 2: (4, 3, 5), 3: (3, 4, 3), 4: (3, 2, 3)}.get(p, (2, 2, 3))
    return n[:dim]


def _case(kind, p, faces, oracle, pmg, ctx, want_free=True):
    """(operator, oracle MatrixFree, oracle MatrixFree without Dirichlet faces, JxW of the mass matrix, support points)"""
    n = _cells(p, 2 if kind == "box2d" else 3)
    if kind == "box2d":
        faces &= 0xF
        op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces, dim=2)
        mf = oracle.MatrixFree(2, p, n, faces=faces)
        mff = oracle.MatrixFree(2, p, n, faces=0) if want_free else None
        return op, mf, mff, box_jxw(p, n), box_support_points(p, n)
    if kind in ("box", "coef"):
        coef = "c5" if kind == "coef" else None
        op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces, coefficient=1 if coef else 0)
        mf = oracle.MatrixFree(3, p, n, faces=faces, coef=coef)
        mff = oracle.MatrixFree(3, p, n, faces=0, coef=coef) if want_free else None
        return op, mf, mff, box_jxw(p, n), box_support_points(p, n)
    if kind == "mapped":
        v = random_vertices(n, 0.2, seed=10 + p)
        op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces, vertices=v)
        mf = mapped_matrix_free(oracle, p, n, v, faces=faces)
        mff = mapped_matrix_free(oracle, p, n, v, faces=0) if want_free else None
        return op, mf, mff, geometry(mf)[1], trilinear_support_points(p, n, v)
    nodes = nodes_of(shell_map, n, p)
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces, nodes=nodes)
    mf = curved_matrix_free(oracle, p, n, nodes, p, faces=faces)
    mff = curved_matrix_free(oracle, p, n, nodes, p, faces=0) if want_free else None
    return op, mf, mff, geometry(mf)[1], curved_support_points(p, n, nodes, p)


# ---- support points ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", DEGREES)
def test_support_points(p, pmg, ctx):
    n3, n2 = _cells(p), _cells(p, 2)
    box = pmg.LaplaceOperator(ctx, p, n3)
    assert np.abs(box.support_points() - box_support_points(p, n3)).max() <= 1e-15
    sq = pmg.LaplaceOperator(ctx, p, n2, dim=2)
    got = sq.support_points()
    assert got.shape == (sq.m(), 2) and np.abs(got - box_support_points(p, n2)).max() <= 1e-15
    v = random_vertices(n3, 0.2, seed=p)
    tri = pmg.LaplaceOperator(ctx, p, n3, vertices=v)
    assert np.abs(tri.support_points() - trilinear_support_points(p, n3, v)).max() <= 1e-14
    nodes = nodes_of(shell_map, n3, p)
    cur = pmg.LaplaceOperator(ctx, p, n3, dirichlet_faces=SHELL_FACES, nodes=nodes)
    assert np.abs(cur.support_points() - nodes.reshape(-1, 3)).max() <= 1e-15
    for k in {1, 2, 3, max(1, p - 2), min(9, p + 2)} - {p}:
        nk = nodes_of(perturbed_map(0.03, seed=p + k), n3, k)
        op = pmg.LaplaceOperator(ctx, p, n3, nodes=nk, geometry_degree=k)
        assert np.abs(op.support_points() - curved_support_points(p, n3, nk, k)).max() <= 1e-14, k


# ---- assemble_rhs_data ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", DEGREES)
@pytest.mark.parametrize("kind", ["box", "box2d", "coef", "mapped", "curved"])
def test_rhs_data_of_one_equals_assemble_rhs(kind, p, pmg, ctx, oracle):
    op = _case(kind, p, 0x3F if kind != "curved" else SHELL_FACES, oracle, pmg, ctx, want_free=False)[0]
    assert min(op.ncells[:op.dim]) >= 2
    ref, got = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(ref)
    op.assemble_rhs_data(got, f=op.interpolate(lambda *x: 1.0))
    assert rel_l2(got.export_host(), ref.export_host()) <= 1e-13


@pytest.mark.parametrize("faces", [0x3F, 0x15, 0x3])
@pytest.mark.parametrize("p", DEGREES)
@pytest.mark.parametrize("kind", ["box", "box2d", "coef", "mapped", "curved"])
def test_rhs_data_against_numpy_reference(kind, p, faces, pmg, ctx, oracle):
    op, mf, mff, jxw, _ = _case(kind, p, faces, oracle, pmg, ctx)
    c = mf.constrained()
    f, g = splitmix_src(mf.n_dofs, salt=11), splitmix_src(mf.n_dofs, salt=12)
    vf, vg = op.vector_from(f), op.vector_from(g)
    rhs = op.initialize_dof_vector()
    for use_f, use_g in ((True, False), (False, True), (True, True)):
        if not c.any() and use_g and not use_f:
            continue
        ref = rhs_reference(p, mf.ncell, jxw, c, f=f if use_f else None, g=g if use_g else None, mf_free=mff)
        rhs.set(np.nan)
        op.assemble_rhs_data(rhs, f=vf if use_f else None, g=vg if use_g else None)
        out = rhs.export_host()
        assert np.all(out[c] == 0.0), (use_f, use_g)
        assert rel_l2(out, ref) <= 1e-12, (use_f, use_g)
    # only the constrained entries of g are read
    g2 = np.where(c, g, splitmix_src(mf.n_dofs, salt=13))
    rhs2 = op.initialize_dof_vector()
    op.assemble_rhs_data(rhs2, f=vf, g=op.vector_from(g2))
    assert np.array_equal(rhs2.export_host(), out)


@pytest.mark.parametrize("kind", ["box", "box2d", "coef", "mapped", "curved"])
def test_distribute(kind, pmg, ctx, oracle):
    op, mf, _, _, _ = _case(kind, 3, 0x15, oracle, pmg, ctx, want_free=False)
    c = mf.constrained()
    u0, g = splitmix_src(mf.n_dofs, salt=21), splitmix_src(mf.n_dofs, salt=22)
    u = op.vector_from(u0)
    op.distribute(u, op.vector_from(g))
    out = u.export_host()
    assert np.array_equal(out[c], g[c]) and np.array_equal(out[~c], u0[~c])


# ---- the whole workflow ----------------------------------------------------------------------------------------------
def _solve(pmg, ctx, levels, u_fn, **kw):
    """interpolate, assemble_rhs_data, CG + V-cycle, distribute; returns (top operator, u_h, I_h u*, iterations)"""
    ops, _, _, mg = pmg.build_hierarchy(ctx, levels, **kw)
    top = ops[-1]
    P = top.support_points()
    u, f = u_fn(P)
    vg, vf = top.vector_from(u), top.vector_from(f)
    b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs_data(b, f=vf, g=vg)
    it, _, rc = pmg.cg_solve(top, x, b, mg)
    assert rc == 0
    top.distribute(x, vg)
    return top, x, vg, it


def _poly_box(P):
    x, y, z = P.T
    return x * x * y + y * y * z + z * z * x, -2.0 * (x + y + z)


def _poly_sheared(P):
    x, y, z = P.T
    return x * x + 2.0 * y * y - z * z + 0.5 * x * y - 0.3 * y * z + x - 1.0, np.full(len(P), -4.0)


def _cube(P):
    u = np.prod(np.cos(np.pi * P), axis=1)
    return u, P.shape[1] * np.pi ** 2 * u


def _radial(P):
    r = np.hypot(P[:, 0], P[:, 1])
    return r * r + np.sin(np.pi * r), -4.0 + np.pi ** 2 * np.sin(np.pi * r) - np.pi * np.cos(np.pi * r) / r


@pytest.mark.parametrize("p", [2, 3, 4])
def test_workflow_reproduces_polynomial_box(p, pmg, ctx):
    _, x, ustar, _ = _solve(pmg, ctx, hierarchy_levels("h", p, 4), _poly_box)
    assert np.abs(x.export_host() - ustar.export_host()).max() <= 1e-9


@pytest.mark.parametrize("p", [2, 3])
def test_workflow_reproduces_polynomial_sheared(p, pmg, ctx):
    n = 4
    _, x, ustar, _ = _solve(pmg, ctx, hierarchy_levels("h", p, n), _poly_sheared, vertices=sheared_box_vertices((n,) * 3))
    assert np.abs(x.export_host() - ustar.export_host()).max() <= 1e-9


def test_workflow_shell_matches_oracle(pmg, ctx, oracle):
    p, n = 3, 4
    levels = hierarchy_levels("h", p, n)
    top, x, _, it = _solve(pmg, ctx, levels, _radial, faces=SHELL_FACES, mapping=shell_map)
    mfs = [curved_matrix_free(oracle, q, m, nodes_of(shell_map, m, q), q, faces=SHELL_FACES) for (q, m) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h") for l in range(1, len(levels))]
    vc = oracle.VCycle(mfs, trs)
    vc.estimate()
    nodes = nodes_of(shell_map, n, p)
    mff = curved_matrix_free(oracle, p, n, nodes, p, faces=0)
    u, f = _radial(curved_support_points(p, (n,) * 3, nodes, p))
    c = mfs[-1].constrained()
    b = rhs_reference(p, (n,) * 3, geometry(mfs[-1])[1], c, f=f, g=u, mf_free=mff)
    x_ref, it_ref, _, rc = oracle.cg_solve(mfs[-1], b, vc)
    x_ref[c] = u[c]
    assert rc == 0 and it == it_ref
    assert np.abs(x.export_host() - x_ref).max() <= 1e-9


def _rates(pmg, ctx, p, ns, u_fn, **kw):
    errs = []
    for n in ns:
        top, x, ustar, _ = _solve(pmg, ctx, hierarchy_levels("h", p, n), u_fn, **kw)
        ustar.sadd(-1.0, 1.0, x)
        errs.append(top.solution_norm(ustar))
    return errs, [np.log2(errs[i] / errs[i + 1]) for i in range(len(errs) - 1)]


@pytest.mark.parametrize("p", [2, 4])
def test_convergence_cube(p, pmg, ctx):
    errs, rates = _rates(pmg, ctx, p, (4, 8), _cube)
    print("cube Q%d: errors %s, rates %s" % (p, errs, rates))
    assert min(rates) >= p + 1 - 0.3


@pytest.mark.parametrize("p", [2, 3])
def test_convergence_shell_mapping_qp(p, pmg, ctx):
    errs, rates = _rates(pmg, ctx, p, (4, 8), _radial, faces=SHELL_FACES, mapping=shell_map)
    print("shell MappingQ(%d): errors %s, rates %s" % (p, errs, rates))
    assert min(rates) >= p + 1 - 0.3


def test_convergence_shell_trilinear(pmg, ctx):
    """Trilinear shell cells at Q3.  The error against the interpolant does not stall at order 2 here: the radial u* solves
    the problem on the trilinear domain as well (its natural faces are planes through the axis, where du*/dn = 0, and g is
    u* at the support points on the faceted faces), so there is no geometry error to see.  The CPU oracle gives the same
    rates (about 5 from 2^3 to 8^3 cells)."""
    errs, rates = _rates(pmg, ctx, 3, (4, 8), _radial, faces=SHELL_FACES, mapping=shell_map, geometry_degree=1)
    print("shell trilinear Q3: errors %s, rates %s" % (errs, rates))
    assert min(rates) >= 3 + 1 - 0.3


# ---- errors ------------------------------------------------------------------------------------------------------------
def test_error_paths(pmg, ctx):
    a = pmg.LaplaceOperator(ctx, 2, 3)
    b = pmg.LaplaceOperator(ctx, 2, 4)
    va, vb = a.initialize_dof_vector(), b.initialize_dof_vector()
    for call in (lambda: a.assemble_rhs_data(vb, f=va), lambda: a.assemble_rhs_data(va, f=vb),
                 lambda: a.assemble_rhs_data(va, g=vb), lambda: a.assemble_rhs_data(va, f=va),
                 lambda: a.distribute(vb, va), lambda: a.distribute(va, vb)):
        with pytest.raises(pmg.PmgError) as e:
            call()
        assert e.value.code == -1
    lib = pmg.lib()
    for z in (None, vb):  # a vector of another layout
        rc = lib.pmg_laplace_operator_support_points(a.h, va.h, vb.h, z.h if z is not None else None)
        assert rc == -1
    sq = pmg.LaplaceOperator(ctx, 2, (3, 3), dim=2)
    x, y, z = (sq.initialize_dof_vector() for _ in range(3))
    assert lib.pmg_laplace_operator_support_points(sq.h, x.h, y.h, z.h) == -3
    assert lib.pmg_laplace_operator_support_points(sq.h, x.h, y.h, None) == 0


def test_two_gpu_problem_data():
    """support_points, assemble_rhs_data, distribute and a manufactured shell solve, slab-distributed on two GPUs
    (tools/dist_check_problem_data.py), against one GPU"""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", os.path.join(ROOT, "tools", "dist_check_problem_data.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert "DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
