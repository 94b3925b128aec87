"""GPU parity of the Laplace operator on deformed hexahedral meshes (pmg_laplace_operator_create_mapped: every cell the
trilinear map of its 8 vertices, G_q = w a |det J| J^-1 J^-T per quadrature point) against the CPU oracle on the same
mesh (tests/mapped_oracle.py), which tests/test_mapped_geometry_cpu.py pins against a dense numpy assembly.
Tolerances as in test_gpu_variable_coefficient.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import hierarchy_levels, rel_l2, splitmix_src
from mapped_mesh import random_vertices, smooth_map_vertices, uniform_vertices
from mapped_oracle import l2_norm_mapped, mapped_matrix_free

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ANCHOR = 0.0249871331  # ||u||_L2 of the continuous problem (tests/golden/anchors.json)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8, 9])
def test_mapped_vmult_diagonal_and_fused_steps(p, pmg, ctx, oracle):
    n = {1: (17, 16, 18), 2: (13, 14, 9), 3: (11, 10, 7), 4: (9, 8, 5)}.get(p, (5, 6, 4))
    coef = p % 2  # the C5 coefficient on odd degrees, a = 1 on even ones
    v = random_vertices(n, 0.2, seed=100 + p)
    mf = mapped_matrix_free(oracle, p, n, v, coef="c5" if coef else None)
    u, b, xo = (splitmix_src(mf.n_dofs, salt=s) for s in (31, 32, 33))
    Au = mf.vmult(u)
    op = pmg.LaplaceOperator(ctx, p, n, coefficient=coef, vertices=v)
    s, d = op.vector_from(u), op.initialize_dof_vector()
    op.vmult(d, s)
    out = d.export_host()
    assert rel_l2(out, Au) <= 1e-12
    c = mf.constrained()
    assert np.array_equal(out[c], u[c])
    dinv = mf.compute_diagonal()
    op.compute_diagonal()
    assert rel_l2(op.get_matrix_diagonal_inverse().export_host(), dinv) <= 1e-12
    vb, vx = op.vector_from(b), op.vector_from(xo)
    op.residual(d, vb, s)
    assert rel_l2(d.export_host(), b - Au) <= 1e-12
    op.chebyshev_step(d, s, None, vb, 0.0, 0.7)
    assert rel_l2(d.export_host(), u + 0.7 * dinv * (b - Au)) <= 1e-12
    op.chebyshev_step(vx, s, vx, vb, 0.3, 0.7)  # x_old overwritten in place
    assert rel_l2(vx.export_host(), u + 0.3 * (u - xo) + 0.7 * dinv * (b - Au)) <= 1e-12


@pytest.mark.parametrize("faces", [0x00, 0x15, 0x2A])
def test_mapped_mixed_boundary(faces, pmg, ctx, oracle):
    p, n = 3, (6, 5, 7)
    v = random_vertices(n, 0.2, seed=faces)
    mf = mapped_matrix_free(oracle, p, n, v, faces=faces)
    u = splitmix_src(mf.n_dofs, salt=34)
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces, vertices=v)
    s, d = op.vector_from(u), op.initialize_dof_vector()
    op.vmult(d, s)
    assert rel_l2(d.export_host(), mf.vmult(u)) <= 1e-12
    op.compute_diagonal()
    assert rel_l2(op.get_matrix_diagonal_inverse().export_host(), mf.compute_diagonal()) <= 1e-12


@pytest.mark.parametrize("p,coef", [(2, 0), (4, 1), (5, 0)])
def test_identity_map_gives_cube_operator(p, coef, pmg, ctx):
    n = (7, 6, 8)
    cube = pmg.LaplaceOperator(ctx, p, n, coefficient=coef)
    mapped = pmg.LaplaceOperator(ctx, p, n, coefficient=coef, vertices=uniform_vertices(n))
    u = splitmix_src(cube.m(), salt=p)
    outs = []
    for op in (cube, mapped):
        s, d = op.vector_from(u), op.initialize_dof_vector()
        op.vmult(d, s)
        op.compute_diagonal()
        outs.append((d.export_host(), op.get_matrix_diagonal_inverse().export_host()))
    assert rel_l2(outs[1][0], outs[0][0]) <= 1e-12
    assert rel_l2(outs[1][1], outs[0][1]) <= 1e-12


def test_mapped_large_is_symmetric(pmg, ctx):
    """<A u, v> = <u, A v> at a size the oracle would not finish (Q5, 24^3 cells, 1.8 M DoFs, random distortion)."""
    n = (24, 24, 24)
    op = pmg.LaplaceOperator(ctx, 5, n, coefficient=1, vertices=random_vertices(n, 0.2, seed=5))
    m = op.m()
    assert m >= 1_500_000
    u, v = op.vector_from(splitmix_src(m, salt=35)), op.vector_from(splitmix_src(m, salt=36))
    Au, Av = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.vmult(Au, u)
    op.vmult(Av, v)
    a, b = Au.dot(v), Av.dot(u)
    assert abs(a - b) <= 1e-12 * max(abs(a), abs(b))


def _coarsened(v, n_fine, n):
    f = n_fine // n
    return v[::f, ::f, ::f]


@pytest.mark.parametrize("kind,p,n,coef", [("h", 2, 8, 0), ("hp", 4, 8, 1), ("hp", 5, 4, 0)])
def test_mapped_vcycle_and_cg(kind, p, n, coef, pmg, ctx, oracle):
    levels = hierarchy_levels(kind, p, n)
    vf = random_vertices((n,) * 3, 0.2, seed=7 + p)
    mfs = [mapped_matrix_free(oracle, q, m, _coarsened(vf, n, m), coef="c5" if coef else None) for (q, m) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h" if levels[l][0] == levels[l - 1][0] else "p") for l in range(1, len(levels))]
    vc_ref = oracle.VCycle(mfs, trs)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels, coefficient=coef, vertices=vf)
    top = ops[-1]
    est = vc_ref.estimate()
    for l, sm in enumerate(smoothers):
        info = sm.info()
        assert info["degree"] == est[l][2], (l, info, est[l])
        assert info["cg_iterations"] == est[l][3]
        assert abs(info["lambda_max"] - est[l][1]) <= 1e-8 * est[l][1]
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=37)
    z_ref = vc_ref.vmult(r)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    for rep in range(3):  # eager warm-up, graph capture, graph replay
        mg.vmult(dz, dr)
        assert rel_l2(dz.export_host(), z_ref) <= 1e-10, rep
    # load vector of f = 1 on the mapped mesh: the oracle's JxW carries a(x), so it comes from the level without coefficient
    b_ref = mapped_matrix_free(oracle, *levels[-1], vf).assemble_rhs()
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
    assert abs(top.solution_norm(x) - l2_norm_mapped(mfs[-1], x_ref)) <= 1e-10


def test_smooth_map_solution_norm_against_oracle_and_anchor(pmg, ctx, oracle):
    """x -> x + 0.1 sin(pi x) sin(pi y) sin(pi z) (1, 1, 1) keeps the unit cube, so the analytic anchor still holds up to the
    discretisation error.  The oracle's distance from it was 1.27e-9 (relative) when this test was written (Q4, 16^3 cells);
    the bound leaves a factor ~80."""
    p, n = 4, 16
    levels = hierarchy_levels("h", p, n)
    vf = smooth_map_vertices((n,) * 3, 0.1)
    mfs = [mapped_matrix_free(oracle, q, m, _coarsened(vf, n, m)) for (q, m) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h") for l in range(1, len(levels))]
    vc_ref = oracle.VCycle(mfs, trs)
    vc_ref.estimate()
    x_ref, it_ref, _, rc_ref = oracle.cg_solve(mfs[-1], mfs[-1].assemble_rhs(), vc_ref)
    norm_ref = l2_norm_mapped(mfs[-1], x_ref)
    ops, _, _, mg = pmg.build_hierarchy(ctx, levels, vertices=vf)
    top = ops[-1]
    b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    it, _, rc = pmg.cg_solve(top, x, b, mg)
    norm = top.solution_norm(x)
    print("smooth map EPS = 0.1, Q4 16^3: CG %d iterations, ||u|| = %.12f, oracle %.12f, |oracle - anchor| / anchor = %.3e"
          % (it, norm, norm_ref, abs(norm_ref - ANCHOR) / ANCHOR))
    assert rc == 0 and rc_ref == 0 and it == it_ref
    assert abs(norm - norm_ref) <= 1e-10
    assert abs(norm_ref - ANCHOR) <= 1e-7 * ANCHOR


def test_invalid_meshes_are_rejected(pmg, ctx):
    n = (4, 3, 3)
    v = uniform_vertices(n)
    v[1, 1, 1] = (0.9, 0.9, 0.9)  # an interior vertex dragged across its neighbours: cells fold
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, n, vertices=v)
    assert e.value.code == -1 and "det J" in str(e.value) and "cell" in str(e.value)
    v = uniform_vertices(n)
    v[2, 1, 3, 1] = np.nan
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 3, n, vertices=v)
    assert e.value.code == -1 and "non-finite" in str(e.value)
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, (4, 3), dim=2, vertices=np.zeros((4, 5, 3)))
    assert e.value.code == -3 and "3-D" in str(e.value)
    # the context is still usable
    op = pmg.LaplaceOperator(ctx, 2, n, vertices=random_vertices(n, 0.2, seed=1))
    u = splitmix_src(op.m(), salt=2)
    s, d = op.vector_from(u), op.initialize_dof_vector()
    op.vmult(d, s)
    assert np.isfinite(d.export_host()).all()


def test_two_gpu_mapped_hierarchy():
    """Slab-distributed mapped hierarchy on two GPUs (tools/dist_check_mapped.py) against the CPU oracle."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(ROOT, "tools", "dist_check_mapped.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert "DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
