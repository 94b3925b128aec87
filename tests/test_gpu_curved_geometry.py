"""GPU parity of the Laplace operator on curved hexahedral meshes (pmg_laplace_operator_create_curved: every cell the
degree-k Lagrange interpolant through its (k+1)^3 nodes, MappingQ(k)) against the CPU oracle on the same mesh
(tests/curved_oracle.py), which tests/test_curved_geometry_cpu.py pins against a dense numpy assembly.  Tolerances as in
test_gpu_mapped_geometry.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from curved_mesh import SHELL_FACES, SHELL_NORM, nodes_of, perturbed_map, shell_map, trilinear_nodes
from curved_oracle import curved_matrix_free, l2_norm_curved
from helpers import hierarchy_levels, rel_l2, splitmix_src
from mapped_mesh import random_vertices

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8, 9])
@pytest.mark.parametrize("coef", [0, 1])
def test_curved_vmult_diagonal_and_fused_steps(p, coef, pmg, ctx, oracle):
    n = {1: (9, 8, 10), 2: (7, 8, 6), 3: (6, 5, 7), 4: (5, 6, 4)}.get(p, (3, 4, 3))
    nodes = nodes_of(perturbed_map(0.03, seed=200 + p) if coef else shell_map, n, p)
    faces = 0x3F if coef else SHELL_FACES
    mf = curved_matrix_free(oracle, p, n, nodes, p, faces=faces, coef="c5" if coef else None)
    u, b, xo = (splitmix_src(mf.n_dofs, salt=s) for s in (41, 42, 43))
    Au = mf.vmult(u)
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces, coefficient=coef, nodes=nodes)
    assert op.geometry_degree == p
    s, d = op.vector_from(u), op.initialize_dof_vector()
    op.vmult(d, s)
    out = d.export_host()
    assert rel_l2(out, Au) <= 1e-12
    dinv = mf.compute_diagonal()
    op.compute_diagonal()
    assert rel_l2(op.get_matrix_diagonal_inverse().export_host(), dinv) <= 1e-12
    vb, vx = op.vector_from(b), op.vector_from(xo)
    op.residual(d, vb, s)
    assert rel_l2(d.export_host(), b - Au) <= 1e-12
    op.chebyshev_step(d, s, None, vb, 0.0, 0.7)
    assert rel_l2(d.export_host(), u + 0.7 * dinv * (b - Au)) <= 1e-12
    op.chebyshev_step(vx, s, vx, vb, 0.3, 0.7)
    assert rel_l2(vx.export_host(), u + 0.3 * (u - xo) + 0.7 * dinv * (b - Au)) <= 1e-12
    if not coef:  # the oracle's JxW carries a(x); its load vector matches only without a coefficient
        rhs = op.initialize_dof_vector()
        op.assemble_rhs(rhs)
        assert rel_l2(rhs.export_host(), mf.assemble_rhs()) <= 1e-13
    assert abs(op.solution_norm(s) - l2_norm_curved(mf, u)) <= 1e-12 * l2_norm_curved(mf, u)


@pytest.mark.parametrize("p,coef", [(2, 0), (3, 1), (5, 0)])
def test_trilinear_sampled_nodes_equal_create_mapped(p, coef, pmg, ctx):
    n = (6, 5, 7)
    v = random_vertices(n, 0.2, seed=50 + p)
    tri = pmg.LaplaceOperator(ctx, p, n, coefficient=coef, vertices=v)
    cur = pmg.LaplaceOperator(ctx, p, n, coefficient=coef, nodes=trilinear_nodes(v, n, 2))
    k1 = pmg.LaplaceOperator(ctx, p, n, coefficient=coef, nodes=v)  # k = 1: the vertex array, the trilinear set-up
    assert (cur.geometry_degree, k1.geometry_degree) == (2, 1)
    u = splitmix_src(tri.m(), salt=p)
    outs = []
    for op in (tri, cur, k1):
        s, d, b = op.vector_from(u), op.initialize_dof_vector(), op.initialize_dof_vector()
        op.vmult(d, s)
        op.compute_diagonal()
        op.assemble_rhs(b)
        outs.append((d.export_host(), op.get_matrix_diagonal_inverse().export_host(), b.export_host(), op.solution_norm(s)))
    for got in outs[1:]:
        for a, r in zip(got[:3], outs[0][:3]):
            assert rel_l2(a, r) <= 1e-12
        assert abs(got[3] - outs[0][3]) <= 1e-12 * outs[0][3]
    assert all(np.array_equal(a, r) for a, r in zip(outs[2][:3], outs[0][:3]))  # k = 1 is create_mapped


def test_curved_large_is_symmetric(pmg, ctx):
    """<A u, v> = <u, A v> at 1.5 M+ DoFs (Q4, 29^3 cells on the shell, MappingQ(4))."""
    n = (29, 29, 29)
    op = pmg.LaplaceOperator(ctx, 4, n, dirichlet_faces=SHELL_FACES, coefficient=1, nodes=pmg.mesh_nodes(shell_map, n, 4))
    m = op.m()
    assert m >= 1_500_000
    u, v = op.vector_from(splitmix_src(m, salt=45)), op.vector_from(splitmix_src(m, salt=46))
    Au, Av = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.vmult(Au, u)
    op.vmult(Av, v)
    a, b = Au.dot(v), Av.dot(u)
    assert abs(a - b) <= 1e-12 * max(abs(a), abs(b))


@pytest.mark.parametrize("kind,p,n,coef", [("h", 2, 8, 0), ("hp", 4, 8, 1), ("hp", 5, 4, 0)])
def test_curved_vcycle_and_cg(kind, p, n, coef, pmg, ctx, oracle):
    levels = hierarchy_levels(kind, p, n)
    mapping = perturbed_map(0.03, seed=7 + p)
    mfs = [curved_matrix_free(oracle, q, m, nodes_of(mapping, m, q), q, coef="c5" if coef else None) for (q, m) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h" if levels[l][0] == levels[l - 1][0] else "p") for l in range(1, len(levels))]
    vc_ref = oracle.VCycle(mfs, trs)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels, coefficient=coef, mapping=mapping)
    assert [op.geometry_degree for op in ops] == [q for (q, _) in levels]
    top = ops[-1]
    est = vc_ref.estimate()
    for l, sm in enumerate(smoothers):
        info = sm.info()
        assert info["degree"] == est[l][2], (l, info, est[l])
        assert info["cg_iterations"] == est[l][3]
        assert abs(info["lambda_max"] - est[l][1]) <= 1e-8 * est[l][1]
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=47)
    z_ref = vc_ref.vmult(r)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    for rep in range(3):  # eager warm-up, graph capture, graph replay
        mg.vmult(dz, dr)
        assert rel_l2(dz.export_host(), z_ref) <= 1e-10, rep
    b_ref = curved_matrix_free(oracle, *levels[-1], nodes_of(mapping, levels[-1][1], p), p).assemble_rhs()
    b = top.initialize_dof_vector()
    top.assemble_rhs(b)
    assert rel_l2(b.export_host(), b_ref) <= 1e-13
    x_ref, it_ref, hist_ref, rc_ref = oracle.cg_solve(mfs[-1], b_ref, vc_ref)
    x = top.initialize_dof_vector()
    it, hist, rc = pmg.cg_solve(top, x, b, mg)
    assert rc == 0 and rc_ref == 0
    assert it == it_ref
    assert np.all(np.abs(hist - hist_ref) <= 1e-10 * hist_ref[0])
    assert rel_l2(x.export_host(), x_ref) <= 1e-9
    assert abs(top.solution_norm(x) - l2_norm_curved(mfs[-1], x_ref)) <= 1e-10


def test_shell_solution_norm_against_oracle_and_exact(pmg, ctx, oracle):
    """Q3, 8^3 cells, MappingQ(3) on every level: the oracle's distance from the exact norm is 6.3e-9 (relative); the
    bound 2e-8 leaves a factor ~3."""
    p, n = 3, 8
    levels = hierarchy_levels("h", p, n)
    mfs = [curved_matrix_free(oracle, q, m, nodes_of(shell_map, m, q), q, faces=SHELL_FACES) for (q, m) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h") for l in range(1, len(levels))]
    vc_ref = oracle.VCycle(mfs, trs)
    vc_ref.estimate()
    x_ref, it_ref, _, rc_ref = oracle.cg_solve(mfs[-1], mfs[-1].assemble_rhs(), vc_ref)
    norm_ref = l2_norm_curved(mfs[-1], x_ref)
    ops, _, _, mg = pmg.build_hierarchy(ctx, levels, faces=SHELL_FACES, mapping=shell_map)
    top = ops[-1]
    b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    it, _, rc = pmg.cg_solve(top, x, b, mg)
    norm = top.solution_norm(x)
    print("shell Q3 8^3 MappingQ(3): CG %d iterations, ||u|| = %.12f, oracle %.12f, |norm - exact| / exact = %.3e"
          % (it, norm, norm_ref, abs(norm - SHELL_NORM) / SHELL_NORM))
    assert rc == 0 and rc_ref == 0 and it == it_ref
    assert abs(norm - norm_ref) <= 1e-10
    assert abs(norm - SHELL_NORM) <= 2e-8 * SHELL_NORM


def test_invalid_curved_meshes_are_rejected(pmg, ctx):
    n, k = (4, 3, 3), 2
    good = nodes_of(shell_map, n, k)
    v = good.copy()
    v[2, 2, 2] = v[2, 2, 6]  # an interior node dragged across its cell: the cell folds
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, n, nodes=v)
    assert e.value.code == -1 and "det J" in str(e.value) and "cell" in str(e.value)
    v = good.copy()
    v[3, 1, 5, 2] = np.nan
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 3, n, nodes=v)
    assert e.value.code == -1 and "non-finite" in str(e.value)
    for bad_k in (0, 10):
        with pytest.raises(pmg.PmgError) as e:
            pmg.LaplaceOperator(ctx, 2, n, nodes=good, geometry_degree=bad_k)
        assert e.value.code == -3 and "geometry degree" in str(e.value)
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, n, nodes=good[:-1])  # a size that fits no geometry degree
    assert e.value.code == -1
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, n, nodes=good, geometry_degree=3)  # the size of k = 2, not 3
    assert e.value.code == -1
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, n, nodes=good, vertices=good)
    assert e.value.code == -1
    # the context is still usable
    op = pmg.LaplaceOperator(ctx, 2, n, nodes=good)
    u = splitmix_src(op.m(), salt=2)
    s, d = op.vector_from(u), op.initialize_dof_vector()
    op.vmult(d, s)
    assert np.isfinite(d.export_host()).all()


def test_two_gpu_curved_hierarchy():
    """Slab-distributed curved hierarchy on two GPUs (tools/dist_check_curved.py) against the CPU oracle."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tools", "dist_check_curved.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert "DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
