"""GPU parity tests: the CUDA path, called through the C-ABI (libpmg.so), against the CPU oracle.

Tolerances are the ones BASELINE.json's north_star states: operator apply <= 1e-12 relative in
l2, identical CG / V-cycle iteration counts, residual histories <= 1e-10 relative.
"""
import os

import numpy as np
import pytest

from helpers import hierarchy_levels, rel_l2, splitmix_src

pytestmark = pytest.mark.gpu

APPLY_TOL = 1e-12
HISTORY_TOL = 1e-10


_KERNELS = ["auto", "plane", "sweep", "celltile"]


@pytest.fixture(autouse=True, params=_KERNELS)
def apply_kernel(request, monkeypatch):
    """Every test runs with the library's default choice of apply kernel (plane-per-step kernel for large levels, cell-tile
    kernel for small ones) and with each kernel forced: the meshes here are small, so the default alone would never reach the
    large-level kernels ("plane": csrc/pmg_apply_plane.h, degrees 1..6, above that the line-marching kernel; "sweep": the
    line-marching kernel of round 1, still used for degrees 7, 8).  PMG_TILE_VARIANT is read when an operator is created."""
    if request.param == "auto":
        monkeypatch.delenv("PMG_TILE_VARIANT", raising=False)
    else:
        monkeypatch.setenv("PMG_TILE_VARIANT", {"sweep": "1", "celltile": "2", "plane": "6"}[request.param])
    return request.param


def _oracle_levels(oracle, levels, faces=0x3F):
    return [oracle.MatrixFree(3, p, n, faces=faces) for (p, n) in levels]


def _oracle_hierarchy(oracle, levels, **kw):
    mfs = _oracle_levels(oracle, levels)
    trs = []
    for l in range(1, len(levels)):
        kind = "h" if levels[l][0] == levels[l - 1][0] else "p"
        trs.append(oracle.Transfer(mfs[l - 1], mfs[l], kind))
    return mfs, trs, oracle.VCycle(mfs, trs, **kw)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8, 9])
def test_vmult_matches_oracle(p, pmg, ctx, oracle):
    n = {1: (17, 16, 18), 2: (13, 14, 9), 3: (11, 10, 7), 4: (9, 8, 5)}.get(p, (5, 6, 4))
    mf = oracle.MatrixFree(3, p, n)
    src = splitmix_src(mf.n_dofs)  # non-zero on Dirichlet dofs on purpose: dst[c] = src[c] there
    ref = mf.vmult(src)
    op = pmg.LaplaceOperator(ctx, p, n)
    assert op.m() == mf.n_dofs == op.n()
    s, d = op.vector_from(src), op.initialize_dof_vector()
    op.vmult(d, s)
    out = d.export_host()
    assert rel_l2(out, ref) <= APPLY_TOL
    c = mf.constrained()
    assert np.array_equal(out[c], src[c])  # identity on Dirichlet dofs, bit for bit
    op.Tvmult(d, s)
    assert np.array_equal(d.export_host(), out)  # Tvmult == vmult, deterministic


@pytest.mark.parametrize("faces", [0x00, 0x15, 0x2A, 0x03, 0x30])
def test_vmult_mixed_boundary(faces, pmg, ctx, oracle):
    p, n = 3, (6, 5, 7)
    mf = oracle.MatrixFree(3, p, n, faces=faces)
    src = splitmix_src(mf.n_dofs, salt=faces)
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces)
    s, d = op.vector_from(src), op.initialize_dof_vector()
    op.vmult(d, s)
    assert rel_l2(d.export_host(), mf.vmult(src)) <= APPLY_TOL


def test_vmult_large_properties(pmg, ctx):
    """Size-independent properties at a BASELINE-scale mesh (Q4, 48^3 cells, 7.2M DoFs)."""
    p, n = 4, 48
    op = pmg.LaplaceOperator(ctx, p, n)
    N = op.m()
    u, v = splitmix_src(N, salt=1), splitmix_src(N, salt=2)
    du, dv = op.vector_from(u), op.vector_from(v)
    Au, Av, Aw = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.vmult(Au, du)
    op.vmult(Av, dv)
    # symmetry (on vectors vanishing on the boundary) and linearity
    Nx = n * p + 1
    g = np.arange(N)
    x, y, z = g % Nx, (g // Nx) % Nx, g // (Nx * Nx)
    bnd = (x == 0) | (x == Nx - 1) | (y == 0) | (y == Nx - 1) | (z == 0) | (z == Nx - 1)
    u0, v0 = u.copy(), v.copy()
    u0[bnd] = 0
    v0[bnd] = 0
    du.import_host(u0)
    dv.import_host(v0)
    op.vmult(Au, du)
    op.vmult(Av, dv)
    a, b = dv.dot(Au), du.dot(Av)
    assert abs(a - b) <= 1e-12 * abs(a)
    w = 0.3 * u0 - 1.7 * v0
    dw = op.vector_from(w)
    op.vmult(Aw, dw)
    lin = 0.3 * Au.export_host() - 1.7 * Av.export_host()
    assert rel_l2(Aw.export_host(), lin) <= 1e-13
    # constants are in the kernel away from the boundary: (A 1)_i = 0 for interior rows not adjacent to it
    one = np.ones(N)
    one[bnd] = 0
    d1 = op.vector_from(one)
    op.vmult(Au, d1)
    r = Au.export_host()
    deep = (x > p) & (x < Nx - 1 - p) & (y > p) & (y < Nx - 1 - p) & (z > p) & (z < Nx - 1 - p)
    assert np.abs(r[deep]).max() <= 1e-12


@pytest.mark.parametrize("p", [1, 2, 3, 4, 6])
def test_diagonal_and_el(p, pmg, ctx, oracle):
    n = (4, 3, 5) if p < 6 else (2, 3, 2)
    mf = oracle.MatrixFree(3, p, n)
    ref = mf.compute_diagonal()
    op = pmg.LaplaceOperator(ctx, p, n)
    with pytest.raises(pmg.PmgError):
        op.get_matrix_diagonal_inverse()
    op.compute_diagonal()
    d = op.get_matrix_diagonal_inverse().export_host()
    assert rel_l2(d, ref) <= 1e-13
    row = mf.n_dofs // 2 + 3
    assert abs(op.el(row, row) - 1.0 / ref[row]) <= 1e-12 / ref[row]
    with pytest.raises(pmg.PmgError):
        op.el(row, row + 1)


def test_residual_and_vector_ops(pmg, ctx, oracle):
    p, n = 2, (5, 6, 4)
    mf = oracle.MatrixFree(3, p, n)
    N = mf.n_dofs
    u, b = splitmix_src(N, salt=3), splitmix_src(N, salt=4)
    op = pmg.LaplaceOperator(ctx, p, n)
    du, db, dr = op.vector_from(u), op.vector_from(b), op.initialize_dof_vector()
    op.residual(dr, db, du)
    assert rel_l2(dr.export_host(), b - mf.vmult(u)) <= APPLY_TOL
    assert abs(du.dot(db) - float(u @ b)) <= 1e-12 * np.linalg.norm(u) * np.linalg.norm(b)
    assert abs(du.l2_norm() - np.linalg.norm(u)) <= 1e-13 * np.linalg.norm(u)
    assert abs(du.mean_value() - u.mean()) <= 1e-14
    du.sadd(0.5, -2.0, db)
    assert rel_l2(du.export_host(), 0.5 * u - 2.0 * b) <= 1e-15
    du.add(3.0, db)
    assert rel_l2(du.export_host(), 0.5 * u + b) <= 1e-15
    du.scale(2.0)
    du.set(1.25)
    assert np.all(du.export_host() == 1.25)
    assert du.size() == N and du.locally_owned_size() == N


@pytest.mark.parametrize("p,nc", [(1, (3, 4, 2)), (2, (3, 2, 4)), (3, (2, 3, 2)), (4, (2, 2, 3)), (5, (2, 1, 2)),
                                  (6, (2, 1, 2)), (7, (1, 2, 1)), (8, (2, 1, 1)), (9, (1, 1, 2))])
def test_h_transfer_matches_oracle(p, nc, pmg, ctx, oracle):
    nf = tuple(2 * c for c in nc)
    mc, mf = oracle.MatrixFree(3, p, nc), oracle.MatrixFree(3, p, nf)
    t_ref = oracle.Transfer(mc, mf, "h")
    oc, of = pmg.LaplaceOperator(ctx, p, nc), pmg.LaplaceOperator(ctx, p, nf)
    t = pmg.GeometricTransfer(oc, of)
    xc, xf = splitmix_src(mc.n_dofs, salt=5), splitmix_src(mf.n_dofs, salt=6)
    dst0 = splitmix_src(mf.n_dofs, salt=7)
    ref = t_ref.prolongate_and_add(dst0.copy(), xc)
    dc, df = oc.vector_from(xc), of.vector_from(dst0)
    t.prolongate_and_add(df, dc)
    assert rel_l2(df.export_host(), ref) <= 1e-13
    dstc0 = splitmix_src(mc.n_dofs, salt=8)
    ref = t_ref.restrict_and_add(dstc0.copy(), xf)
    dc2, df2 = oc.vector_from(dstc0), of.vector_from(xf)
    t.restrict_and_add(dc2, df2)
    assert rel_l2(dc2.export_host(), ref) <= 1e-13


@pytest.mark.parametrize("pc,pf", [(1, 2), (2, 4), (1, 4), (3, 4), (2, 3), (4, 7), (6, 7), (4, 8), (4, 9), (3, 7), (3, 6), (2, 5), (1, 3)])
def test_p_transfer_matches_oracle(pc, pf, pmg, ctx, oracle):
    n = (3, 2, 3)
    mc, mf = oracle.MatrixFree(3, pc, n), oracle.MatrixFree(3, pf, n)
    t_ref = oracle.Transfer(mc, mf, "p")
    oc, of = pmg.LaplaceOperator(ctx, pc, n), pmg.LaplaceOperator(ctx, pf, n)
    t = pmg.PolynomialTransfer(oc, of)
    xc, xf = splitmix_src(mc.n_dofs, salt=9), splitmix_src(mf.n_dofs, salt=10)
    dst0 = splitmix_src(mf.n_dofs, salt=11)
    ref = t_ref.prolongate_and_add(dst0.copy(), xc)
    dc, df = oc.vector_from(xc), of.vector_from(dst0)
    t.prolongate_and_add(df, dc)
    assert rel_l2(df.export_host(), ref) <= 1e-13
    dstc0 = splitmix_src(mc.n_dofs, salt=12)
    ref = t_ref.restrict_and_add(dstc0.copy(), xf)
    dc2, df2 = oc.vector_from(dstc0), of.vector_from(xf)
    t.restrict_and_add(dc2, df2)
    assert rel_l2(dc2.export_host(), ref) <= 1e-13


def test_transfer_rejects_incompatible_levels(pmg, ctx):
    a, b = pmg.LaplaceOperator(ctx, 2, 4), pmg.LaplaceOperator(ctx, 2, 6)
    with pytest.raises(pmg.PmgError):
        pmg.GeometricTransfer(a, b)  # not one global refinement (reference AssertThrow)
    with pytest.raises(pmg.PmgError):
        pmg.PolynomialTransfer(a, a)
    with pytest.raises(pmg.PmgError):
        pmg.LaplaceOperator(ctx, 10, 4)  # outside the compiled degree range (1..9, the reference dispatcher's max_degree)


@pytest.mark.parametrize("p,n,deg", [(2, (6, 5, 4), 5), (3, (4, 4, 4), 3), (4, (3, 4, 3), 5), (1, (8, 8, 8), 1)])
def test_chebyshev_matches_oracle(p, n, deg, pmg, ctx, oracle):
    mf = oracle.MatrixFree(3, p, n)
    src = splitmix_src(mf.n_dofs, mf.constrained(), salt=13)
    ref, info = oracle.chebyshev_vmult(mf, src, degree=deg)
    op = pmg.LaplaceOperator(ctx, p, n)
    op.compute_diagonal()
    sm = pmg.Chebyshev(op, 15.0, deg, 10)
    s, d = op.vector_from(src), op.initialize_dof_vector()
    sm.vmult(d, s)
    got = sm.info()
    assert got["cg_iterations"] == info["cg_iterations"]
    assert abs(got["lambda_max"] - info["lambda_max"]) <= 1e-9 * info["lambda_max"]
    assert abs(got["lambda_min"] - info["lambda_min"]) <= 1e-7 * max(info["lambda_min"], 1e-3)
    assert rel_l2(d.export_host(), ref) <= 1e-11


@pytest.mark.parametrize("kind,p,n", [("h", 2, 8), ("h", 3, 8), ("h", 1, 16), ("hp", 4, 8), ("hp", 3, 4)])
def test_vcycle_and_cg_match_oracle(kind, p, n, pmg, ctx, oracle):
    levels = hierarchy_levels(kind, p, n)
    mfs, trs, vc_ref = _oracle_hierarchy(oracle, levels)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels)
    top = ops[-1]
    # smoother set-up parity (eigenvalue estimates, auto degree on the coarsest level)
    est = vc_ref.estimate()
    for l, sm in enumerate(smoothers):
        info = sm.info()
        assert info["degree"] == est[l][2], (l, info, est[l])
        assert info["cg_iterations"] == est[l][3]
        assert abs(info["lambda_max"] - est[l][1]) <= 1e-8 * est[l][1]
    # one V-cycle on a synthetic residual
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=14)
    z_ref = vc_ref.vmult(r)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    for rep in range(3):  # eager warm-up, graph capture, graph replay must agree
        mg.vmult(dz, dr)
        assert rel_l2(dz.export_host(), z_ref) <= 1e-10, rep
    # full solve: same iteration count, residual history within 1e-10 relative
    b_ref = mfs[-1].assemble_rhs()
    b = top.initialize_dof_vector()
    top.assemble_rhs(b)
    assert rel_l2(b.export_host(), b_ref) <= 1e-14
    x_ref, it_ref, hist_ref, rc_ref = oracle.cg_solve(mfs[-1], b_ref, vc_ref)
    x = top.initialize_dof_vector()
    it, hist, rc = pmg.cg_solve(top, x, b, mg)
    assert rc == 0 and rc_ref == 0
    assert it == it_ref
    assert np.all(np.abs(hist - hist_ref) <= HISTORY_TOL * hist_ref[0])
    assert rel_l2(x.export_host(), x_ref) <= 1e-9
    norm = top.solution_norm(x)
    assert abs(norm - mfs[-1].l2_norm_solution(x_ref)) <= 1e-10
    assert abs(norm - 0.0249871331) < 2e-4  # analytic ||u||_L2 for -Laplace u = 1 on the unit cube


# ---- the BASELINE.json configurations at their own size (VERDICT r01: "no oracle comparison at any BASELINE size").
# These run once, with the library's own kernel choice (the large-level kernels, chunked multi-wave launches included).
def _only_default_kernel(apply_kernel):
    if apply_kernel != "auto":
        pytest.skip("BASELINE-size comparison runs once, with the library's own kernel choice")


def test_baseline_config1_full_size(pmg, ctx, oracle, apply_kernel):
    """configs[0]: Q2, 64^3 cells (2 146 689 DoFs), geometric multigrid 64 -> 1 cells, V(2,2) Chebyshev(3)-Jacobi, CG to 1e-12:
    operator apply <= 1e-12, V-cycle <= 1e-10, same CG iteration count, residual history within 1e-10."""
    _only_default_kernel(apply_kernel)
    levels = hierarchy_levels("h", 2, 64)
    mfs, trs, vc_ref = _oracle_hierarchy(oracle, levels, degree=3)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels, degree=3)
    top = ops[-1]
    assert top.m() == mfs[-1].n_dofs == 2146689
    src = splitmix_src(mfs[-1].n_dofs, salt=21)
    s, d = top.vector_from(src), top.initialize_dof_vector()
    top.vmult(d, s)
    assert rel_l2(d.export_host(), mfs[-1].vmult(src)) <= APPLY_TOL
    est = vc_ref.estimate()
    for l, sm in enumerate(smoothers):
        info = sm.info()
        assert info["degree"] == est[l][2] and info["cg_iterations"] == est[l][3], (l, info, est[l])
        assert abs(info["lambda_max"] - est[l][1]) <= 1e-8 * est[l][1]
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=22)
    z_ref = vc_ref.vmult(r)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    for rep in range(3):  # eager, capture, replay
        mg.vmult(dz, dr)
        assert rel_l2(dz.export_host(), z_ref) <= HISTORY_TOL, rep
    b_ref = mfs[-1].assemble_rhs()
    b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    x_ref, it_ref, hist_ref, rc_ref = oracle.cg_solve(mfs[-1], b_ref, vc_ref)
    it, hist, rc = pmg.cg_solve(top, x, b, mg)
    assert rc == 0 and rc_ref == 0 and it == it_ref, (rc, rc_ref, it, it_ref)
    assert np.all(np.abs(hist - hist_ref) <= HISTORY_TOL * hist_ref[0])
    assert rel_l2(x.export_host(), x_ref) <= 1e-9


def test_baseline_config2_hierarchy_32_cells(pmg, ctx, oracle, apply_kernel):
    """configs[1]'s hierarchy (Q4 -> Q2 -> Q1 + geometric levels, Chebyshev(5)) at 32^3 cells (2 146 689 DoFs): apply, V-cycle
    and the CG solve against the oracle."""
    _only_default_kernel(apply_kernel)
    levels = hierarchy_levels("hp", 4, 32)
    mfs, trs, vc_ref = _oracle_hierarchy(oracle, levels)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels)
    top = ops[-1]
    for l in (len(levels) - 1, len(levels) - 2):  # the Q4 and the Q2 level: large-level kernels
        src = splitmix_src(mfs[l].n_dofs, salt=30 + l)
        s, d = ops[l].vector_from(src), ops[l].initialize_dof_vector()
        ops[l].vmult(d, s)
        assert rel_l2(d.export_host(), mfs[l].vmult(src)) <= APPLY_TOL
    vc_ref.estimate()
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=23)
    z_ref = vc_ref.vmult(r)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    for rep in range(3):
        mg.vmult(dz, dr)
        assert rel_l2(dz.export_host(), z_ref) <= HISTORY_TOL, rep
    b_ref = mfs[-1].assemble_rhs()
    b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    x_ref, it_ref, hist_ref, rc_ref = oracle.cg_solve(mfs[-1], b_ref, vc_ref)
    it, hist, rc = pmg.cg_solve(top, x, b, mg)
    assert rc == 0 and rc_ref == 0 and it == it_ref, (rc, rc_ref, it, it_ref)
    assert np.all(np.abs(hist - hist_ref) <= HISTORY_TOL * hist_ref[0])


def test_baseline_config2_apply_and_step_full_size(pmg, ctx, oracle, apply_kernel):
    """configs[1] at its own size: Q4, 64^3 cells (16 974 593 DoFs).  The operator apply and one fused Chebyshev step of the
    finest level against the oracle (the oracle's cell loop in the reference layout: 3.7 GB, ~1 s per apply)."""
    _only_default_kernel(apply_kernel)
    mf = oracle.MatrixFree(3, 4, 64)
    op = pmg.LaplaceOperator(ctx, 4, 64)
    assert op.m() == mf.n_dofs == 16974593
    src = splitmix_src(mf.n_dofs, salt=24)
    Au = mf.vmult(src)
    s, d = op.vector_from(src), op.initialize_dof_vector()
    op.vmult(d, s)
    assert rel_l2(d.export_host(), Au) <= APPLY_TOL
    bb, xo = splitmix_src(mf.n_dofs, salt=25), splitmix_src(mf.n_dofs, salt=26)
    db, dx = op.vector_from(bb), op.vector_from(xo)
    op.chebyshev_step(dx, s, dx, db, 0.37, 0.81)  # x_old overwritten in place, as the smoother calls it
    ref = src + 0.37 * (src - xo) + 0.81 * mf.compute_diagonal() * (bb - Au)
    assert rel_l2(dx.export_host(), ref) <= APPLY_TOL


def test_vector_local_part_wrap_and_ghost_operations_one_rank(pmg, ctx, oracle):
    """The partitioner-style vector API on one rank: the local range is the whole vector, owned import / export round-trips,
    a wrapped caller-owned array is used in place (no copy) and the ghost operations are no-ops (no ghosts exist)."""
    p, n = 2, (5, 4, 6)
    mf = oracle.MatrixFree(3, p, n)
    op = pmg.LaplaceOperator(ctx, p, n)
    src = splitmix_src(mf.n_dofs, salt=31)
    v = op.initialize_dof_vector()
    plane, z0, nz, lo, hi = v.local_range()
    assert (plane, z0, nz, lo, hi) == (mf.nd[0] * mf.nd[1], 0, mf.nd[2], 0, mf.nd[2])
    v.import_owned(src)
    assert np.array_equal(v.export_owned(), src) and np.array_equal(v.export_local(), src) and np.array_equal(v.export_host(), src)
    for f in (v.update_ghost_values, v.zero_out_ghost_values, v.compress_add):
        f()
        assert np.array_equal(v.export_host(), src)
    # wrap: the operator reads and writes the caller's arrays (here: two library vectors' storage seen through new handles)
    a, b = op.vector_from(src), op.initialize_dof_vector()
    wa, wb = a.wrap(a.device_ptr()), b.wrap(b.device_ptr())
    op.vmult(wb, wa)
    assert rel_l2(b.export_host(), mf.vmult(src)) <= APPLY_TOL
    del wa, wb  # frees the handles only
    assert np.array_equal(a.export_host(), src)
    # V-cycle through host buffers holding the owned part == through the global host buffers
    levels = hierarchy_levels("h", 2, 8)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels)
    r = splitmix_src(ops[-1].m(), salt=32)
    z1, z2 = np.empty_like(r), np.empty_like(r)
    mg.vmult_host(z1, r)
    mg.vmult_host_owned(z2, r)
    assert np.array_equal(z1, z2)


def test_vcycle_graph_vs_eager_bitwise(pmg, ctx):
    levels = hierarchy_levels("h", 2, 16)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels)
    top = ops[-1]
    r = splitmix_src(top.m(), salt=15)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    mg.set_graph(False)
    mg.vmult(dz, dr)
    eager = dz.export_host()
    mg.set_graph(True)
    for _ in range(3):
        mg.vmult(dz, dr)
    assert np.array_equal(dz.export_host(), eager)  # deterministic kernels: bit-identical
    prof = mg.profile(dz, dr)
    assert prof.shape == (len(levels), 4) and prof.sum() > 0


@pytest.mark.parametrize("kind,p,n", [("h", 1, 32), ("h", 2, 16), ("hp", 4, 8)])
def test_coarse_cycle_kernel_matches_per_level_kernels(kind, p, n, pmg, ctx, monkeypatch):
    """PMG_COARSE_KERNEL=1 runs the small levels inside one single-CTA kernel (csrc/pmg_coarse_cycle.h; off by default, it
    measured slower than the per-level kernels): the two cycles agree to round-off (the gather order inside a row differs)."""
    levels = hierarchy_levels(kind, p, n)
    r = None
    results = []
    for flag in ("0", "1"):
        monkeypatch.setenv("PMG_COARSE_KERNEL", flag)  # read at the cycle's first vmult
        monkeypatch.setenv("PMG_COARSE_MAX_WORK", "4e5")
        ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels)
        top = ops[-1]
        if r is None:
            r = splitmix_src(top.m(), salt=17)
        dr, dz = top.vector_from(r), top.initialize_dof_vector()
        launches = []
        for rep in range(3):
            before = ctx.launch_count()
            mg.vmult(dz, dr)
            launches.append(ctx.launch_count() - before)
        results.append((dz.export_host(), launches[0]))
    assert rel_l2(results[1][0], results[0][0]) <= 1e-12
    assert results[1][1] < results[0][1]  # fewer launches: the coarse levels are one kernel


def test_host_buffer_entry_points(pmg, ctx, oracle):
    p, n = 2, (6, 6, 6)
    mf = oracle.MatrixFree(3, p, n)
    src = splitmix_src(mf.n_dofs, salt=16)
    op = pmg.LaplaceOperator(ctx, p, n)
    out = np.empty(mf.n_dofs)
    op.vmult_host(out, src)
    assert rel_l2(out, mf.vmult(src)) <= APPLY_TOL


def test_error_paths(pmg, ctx):
    a, b = pmg.LaplaceOperator(ctx, 2, 4), pmg.LaplaceOperator(ctx, 3, 4)
    va, vb = a.initialize_dof_vector(), b.initialize_dof_vector()
    with pytest.raises(pmg.PmgError):
        a.vmult(va, vb)  # vector of another level
    with pytest.raises(pmg.PmgError):
        a.vmult(va, va)  # aliasing
    with pytest.raises(pmg.PmgError):
        va.add(1.0, vb)
    with pytest.raises(pmg.PmgError):
        pmg.LaplaceOperator(ctx, 2, 4, dim=4)
    with pytest.raises(pmg.PmgError):
        pmg.LaplaceOperator(ctx, 2, 4, dim=2, coefficient=1)  # the coefficient extension is 3-D only
