"""GPU parity of the coefficient from the caller (PMG_COEFFICIENT_CALLER, pmg_laplace_operator_quadrature_points /
set_coefficient) against the CPU oracle with the same a multiplied into its JxW (tests/coefficient_ref.py, pinned by
tests/test_coefficient_cpu.py): quadrature points, the operator and its fused steps, the diagonal, multigrid, the
manufactured workflow and the error paths, on box, trilinear, curved and 2-D operators."""
import os
import subprocess
import sys

import numpy as np
import pytest

from coefficient_ref import (c5, jump, quadrature_points_box, quadrature_points_curved, quadrature_points_trilinear,
                             with_coefficient)
from curved_mesh import SHELL_FACES, nodes_of, shell_map
from curved_oracle import curved_matrix_free
from helpers import hierarchy_levels, rel_l2, splitmix_src
from mapped_mesh import random_vertices
from mapped_oracle import mapped_matrix_free
from problem_data_ref import box_jxw, rhs_reference

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ["box", "trilinear", "curved", "2d"]


def _shell_jump(P):
    return np.where(np.hypot(P[:, 0], P[:, 1]) < 1.5, 100.0, 1.0)


def _mesh(kind, p):
    """(dim, n, vertices, nodes, k, faces pair) of the test mesh of each operator kind"""
    if kind == "2d":
        return 2, (5, 4) if p <= 4 else (3, 4), None, None, None, (0xF, 0x5)
    n = (4, 3, 5) if p <= 3 else (3, 2, 3)
    if kind == "box":
        return 3, n, None, None, None, (0x3F, 0x15)
    if kind == "trilinear":
        return 3, n, random_vertices(n, 0.2, seed=30 + p), None, 1, (0x3F, 0x2A)
    return 3, n, None, nodes_of(shell_map, n, 2), 2, (SHELL_FACES, 0x3F)


def make_pair(pmg, ctx, oracle, kind, p, faces, afn, coefficient=None):
    """(GPU operator with the caller coefficient a = afn(points), oracle with the same a, the points, a)"""
    dim, n, v, nodes, k, _ = _mesh(kind, p)
    coef = pmg.PMG_COEFFICIENT_CALLER if coefficient is None else coefficient
    op = pmg.LaplaceOperator(ctx, p, n, faces, dim=dim, coefficient=coef, vertices=v, nodes=nodes, geometry_degree=k)
    if kind in ("box", "2d"):
        P = quadrature_points_box(p, n)
        mf = oracle.MatrixFree(dim, p, n, faces=faces)
    elif kind == "trilinear":
        P = quadrature_points_trilinear(p, n, v)
        mf = mapped_matrix_free(oracle, p, n, v, faces=faces)
    else:
        P = quadrature_points_curved(p, n, nodes, k)
        mf = curved_matrix_free(oracle, p, n, nodes, k, faces=faces)
    a = afn(P) if afn is not None else None
    if a is not None:
        with_coefficient(mf, a)
        if coefficient is None:
            op.set_coefficient(a)
    return op, mf, P, a


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8, 9])
@pytest.mark.parametrize("kind", KINDS)
def test_quadrature_points_match_reference(kind, p, pmg, ctx, oracle):
    dim, n, v, nodes, k, faces = _mesh(kind, p)
    op, _, P, _ = make_pair(pmg, ctx, oracle, kind, p, faces[0], None)
    got = op.quadrature_points()
    assert got.shape == P.shape
    assert np.abs(got - P).max() <= (1e-15 if kind in ("box", "2d") else 1e-14)
    qx, qy, qz0, nqz = op.quadrature_grid()
    assert (qx, qy, qz0) == (n[0] * (p + 1), n[1] * (p + 1), 0) and nqz == (1 if dim == 2 else n[2] * (p + 1))
    # any operator has them, not only PMG_COEFFICIENT_CALLER ones
    op0 = pmg.LaplaceOperator(ctx, p, n, faces[0], dim=dim, vertices=v, nodes=nodes, geometry_degree=k)
    assert np.array_equal(op0.quadrature_points(), got)


def _vmult(op, u):
    s, d = op.vector_from(u), op.initialize_dof_vector()
    op.vmult(d, s)
    return d.export_host()


def _dinv(op):
    op.compute_diagonal()
    return op.get_matrix_diagonal_inverse().export_host()


@pytest.mark.parametrize("kind", KINDS)
def test_caller_operator_before_set_equals_constant(kind, pmg, ctx, oracle):
    for p in (1, 3, 6):
        _, _, _, _, _, faces = _mesh(kind, p)
        op, _, _, _ = make_pair(pmg, ctx, oracle, kind, p, faces[0], None)
        op0, _, _, _ = make_pair(pmg, ctx, oracle, kind, p, faces[0], None, coefficient=0)
        u = splitmix_src(op.m(), salt=3)
        assert rel_l2(_vmult(op, u), _vmult(op0, u)) <= 1e-13
        assert rel_l2(_dinv(op), _dinv(op0)) <= 1e-13


@pytest.mark.parametrize("kind", ["box", "trilinear", "curved"])
def test_c5_at_the_points_reproduces_coefficient_one(kind, pmg, ctx, oracle):
    for p in (1, 2, 4, 7):
        _, _, _, _, _, faces = _mesh(kind, p)
        op, _, _, _ = make_pair(pmg, ctx, oracle, kind, p, faces[0], c5)
        op1, _, _, _ = make_pair(pmg, ctx, oracle, kind, p, faces[0], None, coefficient=1)
        u = splitmix_src(op.m(), salt=4)
        assert rel_l2(_vmult(op, u), _vmult(op1, u)) <= 1e-14
        assert rel_l2(_dinv(op), _dinv(op1)) <= 1e-14


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8, 9])
@pytest.mark.parametrize("kind", KINDS)
def test_jump_coefficient_operator_matches_oracle(kind, p, pmg, ctx, oracle):
    afn = _shell_jump if kind == "curved" else jump
    for faces in _mesh(kind, p)[5]:
        op, mf, _, _ = make_pair(pmg, ctx, oracle, kind, p, faces, afn)
        m = mf.n_dofs
        u, b, xo = (splitmix_src(m, salt=s) for s in (11, 12, 13))
        Au = mf.vmult(u)
        dref = mf.compute_diagonal()
        assert rel_l2(_vmult(op, u), Au) <= 1e-12
        dinv = _dinv(op)
        assert rel_l2(dinv, dref) <= 1e-12
        i = int(np.argmax(~mf.constrained()))
        assert abs(op.el(i, i) - 1.0 / dref[i]) <= 1e-12 * abs(1.0 / dref[i])
        s, bb, d = op.vector_from(u), op.vector_from(b), op.initialize_dof_vector()
        op.residual(d, bb, s)
        assert rel_l2(d.export_host(), b - Au) <= 1e-12
        f1, f2 = 0.4, 0.6
        step = u + f1 * (u - xo) + f2 * dref * (b - Au)
        x = op.vector_from(xo)
        op.chebyshev_step(d, s, x, bb, f1, f2)
        assert rel_l2(d.export_host(), step) <= 1e-12
        d2 = op.vector_from(xo)
        op.chebyshev_step(d2, s, d2, bb, f1, f2)  # x_old aliases dst
        assert rel_l2(d2.export_host(), step) <= 1e-12
        op.chebyshev_step(d, s, None, bb, f1, f2)
        assert rel_l2(d.export_host(), u + f1 * u + f2 * dref * (b - Au)) <= 1e-12


@pytest.mark.parametrize("kind", KINDS)
def test_set_coefficient_twice_equals_fresh_operator(kind, pmg, ctx, oracle):
    p = 3
    faces = _mesh(kind, p)[5][0]
    op, _, P, _ = make_pair(pmg, ctx, oracle, kind, p, faces, c5)
    a2 = 1.0 + 3.0 * jump(P[:, :2])
    op.set_coefficient(a2)
    fresh, _, _, _ = make_pair(pmg, ctx, oracle, kind, p, faces, lambda _: a2)
    u = splitmix_src(op.m(), salt=5)
    assert np.array_equal(_vmult(op, u), _vmult(fresh, u))
    assert np.array_equal(_dinv(op), _dinv(fresh))


def _oracle_levels(oracle, kind, levels, ops, afn, faces, mapping=None):
    """the oracle's levels with a evaluated at the GPU levels' own points (test_quadrature_points_match_reference checks
    those): a jump evaluated at two roundings of a point on the jump could differ"""
    mfs = []
    for (q, m), op in zip(levels, ops):
        if kind == "curved":
            mf = curved_matrix_free(oracle, q, (m,) * 3, nodes_of(mapping, m, q), q, faces=faces)
        else:
            mf = oracle.MatrixFree(2 if kind == "2d" else 3, q, m, faces=faces)
        mfs.append(with_coefficient(mf, afn(op.quadrature_points())))
    return mfs


@pytest.mark.parametrize("kind,levels", [
    ("box", hierarchy_levels("h", 2, 8)), ("box", hierarchy_levels("hp", 4, 4)),
    ("curved", hierarchy_levels("h", 2, 4)), ("2d", [(1, 16), (2, 16), (3, 16), (4, 16), (5, 16), (6, 16), (7, 16)])])
def test_jump_coefficient_multigrid_matches_oracle(kind, levels, pmg, ctx, oracle):
    dim = 2 if kind == "2d" else 3
    faces = SHELL_FACES if kind == "curved" else (0xF if dim == 2 else 0x3F)
    afn = _shell_jump if kind == "curved" else jump
    mapping = shell_map if kind == "curved" else None
    fn = (lambda x, y, z: _shell_jump(np.stack([x, y, z], axis=1))) if kind == "curved" else \
        (lambda *X: jump(np.stack(X, axis=1)))
    ops, _, smoothers, mg = pmg.build_hierarchy(ctx, levels, faces=faces, dim=dim, coefficient=fn, mapping=mapping)
    mfs = _oracle_levels(oracle, kind, levels, ops, afn, faces, mapping)
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h" if levels[l][0] == levels[l - 1][0] else "p") for l in range(1, len(levels))]
    vc_ref = oracle.VCycle(mfs, trs)
    est = vc_ref.estimate()
    for l, sm in enumerate(smoothers):
        info = sm.info()
        assert info["degree"] == est[l][2] and info["cg_iterations"] == est[l][3], (l, info, est[l])
        assert abs(info["lambda_max"] - est[l][1]) <= 1e-8 * est[l][1]
    top = ops[-1]
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=7)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    z_ref = vc_ref.vmult(r)
    for rep in range(2):
        mg.vmult(dz, dr)
        assert rel_l2(dz.export_host(), z_ref) <= 1e-10, rep
    b_ref = mfs[-1].assemble_rhs()
    b = top.vector_from(b_ref)
    x_ref, it_ref, hist_ref, rc_ref = oracle.cg_solve(mfs[-1], b_ref, vc_ref)
    x = top.initialize_dof_vector()
    it, hist, rc = pmg.cg_solve(top, x, b, mg)
    print("%s jump coefficient: CG %d iterations (oracle %d)" % (kind, it, it_ref))
    assert rc == 0 and rc_ref == 0 and it == it_ref
    assert np.all(np.abs(hist - hist_ref) <= 1e-10 * hist_ref[0])


def _smooth_a(P):
    return 1.0 + np.sum(P * P, axis=1)


@pytest.mark.parametrize("dim,p,nc", [(3, 2, 8), (2, 3, 16)])
def test_manufactured_workflow_with_smooth_coefficient(dim, p, nc, pmg, ctx, oracle):
    from test_coefficient_cpu import manufactured

    n = (nc,) * dim
    levels = hierarchy_levels("h", p, nc)
    ops, _, _, mg = pmg.build_hierarchy(ctx, levels, dim=dim, faces=0x3F if dim == 3 else 0xF,
                                        coefficient=lambda *X: _smooth_a(np.stack(X, axis=1)))
    top = ops[-1]
    u_star, f = manufactured(top.support_points())
    g, fv, rhs, x = top.vector_from(u_star), top.vector_from(f), top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs_data(rhs, f=fv, g=g)
    a = _smooth_a(quadrature_points_box(p, n))
    mf = with_coefficient(oracle.MatrixFree(dim, p, n), a)
    mf_free = with_coefficient(oracle.MatrixFree(dim, p, n, faces=0), a)
    c = mf.constrained()
    b_ref = rhs_reference(p, n, box_jxw(p, n), c, f=f, g=u_star, mf_free=mf_free)
    assert rel_l2(rhs.export_host(), b_ref) <= 1e-12
    it, _, rc = pmg.cg_solve(top, x, rhs, mg)
    assert rc == 0
    top.distribute(x, g)
    x_ref, _, _, rc_ref = oracle.cg_solve(mf, b_ref, rel_tol=1e-13, max_it=5000)
    x_ref[c] = u_star[c]
    err, err_ref = top.solution_norm(top.vector_from(x.export_host() - u_star)), mf.l2_norm_solution(x_ref - u_star)
    print("manufactured, a = 1 + |x|^2, dim %d Q%d %d cells: ||u_h - I_h u*|| = %.6e (oracle %.6e), CG %d" % (dim, p, nc, err, err_ref, it))
    assert abs(err - err_ref) <= 1e-3 * err_ref


def test_error_paths(pmg, ctx):
    op0 = pmg.LaplaceOperator(ctx, 2, 3)
    op1 = pmg.LaplaceOperator(ctx, 2, 3, coefficient=1)
    for op in (op0, op1):
        with pytest.raises(pmg.PmgError) as e:
            op.set_coefficient(np.ones(op.quadrature_points().shape[0]))
        assert e.value.code == -7
    for dim in (2, 3):
        op = pmg.LaplaceOperator(ctx, 2, (3, 2, 2)[:dim], dim=dim, coefficient=pmg.PMG_COEFFICIENT_CALLER)
        P = op.quadrature_points()
        u = splitmix_src(op.m(), salt=9)
        ref = _vmult(op, u)
        for bad in (np.nan, 0.0, -1.0, np.inf):
            a = np.ones(len(P))
            a[4 * 9 + 4] = bad  # Qx = 9: grid point (4, 4, 0) = cell (1, 1[, 0]), local point (1, 1[, 0])
            with pytest.raises(pmg.PmgError) as e:
                op.set_coefficient(a)
            assert e.value.code == -1 and "cell (1, 1" in str(e.value) and "local point (1, 1" in str(e.value), str(e.value)
        assert np.array_equal(_vmult(op, u), ref)  # unchanged after the refusals
    op2 = pmg.LaplaceOperator(ctx, 2, (3, 2), dim=2, coefficient=pmg.PMG_COEFFICIENT_CALLER)
    x = np.empty(op2.quadrature_points().shape[0])
    rc = pmg.lib().pmg_laplace_operator_quadrature_points(op2.h, pmg._np_ptr(x), pmg._np_ptr(x.copy()), pmg._np_ptr(x.copy()))
    assert rc == -3
    assert pmg.lib().pmg_laplace_operator_set_coefficient(op2.h, None) == -1
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, (3, 2), dim=2, coefficient=1)
    assert e.value.code == -3
    with pytest.raises(pmg.PmgError) as e:
        pmg.LaplaceOperator(ctx, 2, 3, coefficient=3)
    assert e.value.code == -3


def _driver(name, *args):
    exe = os.path.join(ROOT, "portable-multigrid_b200", "bin", name)
    out = subprocess.run([exe, *args], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    return out.stdout


@pytest.mark.parametrize("name,args", [
    ("geometric_multigrid", ["--coefficient", "2", "--degree", "2", "--cycles", "4"]),
    ("polynomial_multigrid", ["--coefficient", "2", "--cycles", "5"]),
    ("geometric_multigrid", ["--coefficient", "2", "--shell", "1", "--degree", "3", "--cycles", "4", "--mapping-degree", "0"]),
    ("polynomial_multigrid", ["--coefficient", "2", "--dim", "3", "--degree", "4", "--cycles", "3"])])
def test_drivers_with_jump_coefficient(name, args):
    out = _driver(name, *args)
    print(out)
    assert "coefficient: a = 100" in out
    its = [int(l.split()[3]) for l in out.splitlines() if "Solver converged in" in l]
    assert its and max(its) < 100


def test_two_gpu_caller_coefficient():
    """each rank sets a on its own points, halo layer included; the z-slab apply, diagonal and CG equal one GPU
    (tools/dist_check_coefficient.py)"""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "tools", "dist_check_coefficient.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert "DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
