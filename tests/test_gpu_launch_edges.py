"""The constant-coefficient box operator's kernels at their launch edges, against the oracle.

The parity module compares every kernel along one diagonal: plain apply at every degree on one mesh each, all faces
Dirichlet.  Here the meshes come from the kernels' own tile tables (csrc/pmg_apply_plane_tiles.inc,
csrc/pmg_apply_sweep_tiles.inc and the cell-tile table of csrc/pmg_apply.cu), parsed at collection time, so that a retuned
table gets its own edges tested: one tile and one tile plus a cell in x, one and almost two tiles in y, one, two and an odd
number of cell layers, under faces that switch the high faces' virtual-cell tiles on and off.  Every epilogue is compared
(apply, residual, the Chebyshev step with a separate, an aliased and no x_old).  Larger meshes, picked on the device at hand
through pmgk_apply_geometry, reach multi-wave launches with multi-layer z-chunks and a short last chunk.  Transfers, the
inverse diagonal, the load vector, the norm, V-cycles and CG run on non-cubic meshes with natural faces.

Tolerances as in the parity module: apply 1e-12 relative in l2, transfers and the diagonal 1e-13, V-cycle 1e-10.
"""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

from helpers import rel_l2, splitmix_src

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "portable-multigrid_b200", "csrc")
APPLY_TOL = 1e-12
XFER_TOL = 1e-13
HISTORY_TOL = 1e-10
CASE_CAP = 500_000  # DoFs of one case of the apply matrix
FACES = [0x3F, 0x15, 0x2A, 0x09]  # all Dirichlet; high faces natural (virtual-cell tiles); low faces natural; x low + y high
VARIANT = {"default": None, "sweep": "1", "celltile_small": "2", "celltile_large": "3", "plane": "6"}


# ---- the tile tables ----------------------------------------------------------------------------------------------------
def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _plane_tables():
    """{(degree, 'apply' | 'fused'): (BX, BY)} from the PMG_PLANE_CASE / PMG_PLANE_CASE_F lines"""
    out = {}
    for kind, p, bx, by in re.findall(r"^PMG_PLANE_CASE(_F)?\((\d+),\s*(\d+),\s*(\d+),", _read("pmg_apply_plane_tiles.inc"), re.M):
        out[(int(p), "fused" if kind else "apply")] = (int(bx), int(by))
    return out


def _sweep_table():
    """{degree: (BX, BY, LZ)} from the PMG_SWEEP_CASE lines"""
    return {int(p): (int(bx), int(by), int(lz)) for p, bx, by, lz in
            re.findall(r"^PMG_SWEEP_CASE\((\d+),\s*(\d+),\s*(\d+),\s*(\d+),", _read("pmg_apply_sweep_tiles.inc"), re.M)}


def _celltile_tables():
    """({degree: (BX, BY)} small tiles, the same for large tiles): the cell-tile launcher's first switch (tile_variant != 3)
    holds the small tiles of the degrees it lists, the second switch the large tiles of every degree, which the degrees the
    first one omits also take under tile_variant 2."""
    src = _read("pmg_apply.cu")
    body = src[src.index("#define PMG_LAUNCH"):src.index("#undef PMG_LAUNCH")]
    switches = body.split("switch (lv->degree)")[1:]
    assert len(switches) == 2, "the cell-tile launcher no longer has a small- and a large-tile switch"
    small, large = ({int(p): (int(bx), int(by)) for p, bx, by in re.findall(r"case (\d+): PMG_LAUNCH\(\d+,\s*(\d+),\s*(\d+),", s)}
                    for s in switches)
    for p, t in large.items():
        small.setdefault(p, t)
    return small, large


PLANE = _plane_tables()
SWEEP = _sweep_table()
CELL_SMALL, CELL_LARGE = _celltile_tables()
PLANE_DEGREES = sorted({p for p, _ in PLANE})


def _n_dofs(p, n):
    return (n[0] * p + 1) * (n[1] * p + 1) * (n[2] * p + 1)


def _edge_meshes(p, bx, by, lz=1):
    """nx in {BX, BX + 1}, ny in {BY, 2 BY - 1}, nz in {1, 2, odd}; the odd layer count is 1 mod LZ (one partial step)"""
    odd = 2 * lz + 1 if lz > 1 else 5
    out = []
    for nx in (bx, bx + 1):
        for ny in sorted({by, 2 * by - 1}):
            for nz in (1, 2, odd):
                if _n_dofs(p, (nx, ny, nz)) <= CASE_CAP and (nx, ny, nz) not in out:
                    out.append((nx, ny, nz))
    return out


def _apply_cases():
    cases = []  # (kernel, degree, table, mesh)

    def add(kernel, p, table, tiles, lz=1):
        for n in _edge_meshes(p, *tiles, lz=lz):
            if not any(c[0] == kernel and c[1] == p and c[3] == n for c in cases):
                cases.append((kernel, p, table, n))

    for (p, table), tiles in sorted(PLANE.items()):
        add("plane", p, table, tiles)
    for p, (bx, by, lz) in sorted(SWEEP.items()):
        add("sweep", p, "sweep", (bx, by), lz)
    for p, tiles in sorted(CELL_SMALL.items()):
        add("celltile_small", p, "cell", tiles)
    for p, tiles in sorted(CELL_LARGE.items()):
        if CELL_SMALL.get(p) != tiles:  # degrees where variant 3 differs from variant 2
            add("celltile_large", p, "cell", tiles)
    # the library's own choice on these small meshes: the cell-tile kernel where it takes small levels, the plane kernel
    # for the other degrees it covers, the line-marching kernel above
    for p in range(1, 10):
        if p in CELL_SMALL and p <= 5:
            add("default", p, "cell", CELL_SMALL[p])
        elif p in PLANE_DEGREES:
            for table in ("apply", "fused"):
                add("default", p, table, PLANE[(p, table)])
        else:
            bx, by, lz = SWEEP[p]
            add("default", p, "sweep", (bx, by), lz)
    return cases


APPLY_CASES = _apply_cases()


def _set_variant(monkeypatch, kernel):
    v = VARIANT[kernel]
    if v is None:
        monkeypatch.delenv("PMG_TILE_VARIANT", raising=False)
    else:
        monkeypatch.setenv("PMG_TILE_VARIANT", v)  # read when an operator is created


@pytest.fixture
def kernel_variant(monkeypatch):
    """set_variant(kernel): PMG_TILE_VARIANT for the operators created next (none for 'default')"""
    return lambda kernel: _set_variant(monkeypatch, kernel)


# ---- the launch geometry, as the device computes it ---------------------------------------------------------------------
class PmgkLevel(C.Structure):
    """ctypes mirror of pmgk_level (include/pmg_kernels.h); its layout is checked against the header by
    test_level_mirror_matches_header"""
    _fields_ = [
        ("dim", C.c_int), ("degree", C.c_int), ("nx", C.c_int), ("ny", C.c_int), ("nz", C.c_int),
        ("Nx", C.c_int), ("Ny", C.c_int), ("Nz", C.c_int), ("faces", C.c_uint),
        ("z0", C.c_int), ("nzl", C.c_int), ("cz_lo", C.c_int), ("cz_hi", C.c_int), ("z_own_lo", C.c_int), ("z_own_hi", C.c_int),
        ("h", C.c_double * 3), ("S", C.c_double * 100), ("lam", C.c_double * 10), ("Mref", C.c_double * 100),
        ("Kref", C.c_double * 100), ("dinv_tab", C.c_void_p), ("dinv_vec", C.c_void_p), ("tile_variant", C.c_int),
        ("coef", C.c_void_p), ("coef_cz0", C.c_int), ("Sq", C.c_double * 100), ("Dco", C.c_double * 100),
        ("geo_stride", C.c_int64),
    ]


_LAYOUT_PROGRAM = r"""
#include <stddef.h>
#include <stdio.h>
#include "pmg_kernels.h"
#define F(m) printf("%s %zu\n", #m, offsetof(pmgk_level, m));
int main(void)
{
  printf("sizeof %zu\n", sizeof(pmgk_level));
  FIELDS
  return 0;
}
"""


def test_level_mirror_matches_header(tmp_path):
    """The mirror's size and every field offset against a C program compiled against include/pmg_kernels.h.  A mismatch
    fails: the geometry checks below would read another level than the one they describe."""
    src = tmp_path / "layout.c"
    src.write_text(_LAYOUT_PROGRAM.replace("FIELDS", " ".join("F(%s)" % f for f, _ in PmgkLevel._fields_)))
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got.pop("sizeof")) == C.sizeof(PmgkLevel)
    assert {f: int(v) for f, v in got.items()} == {f: getattr(PmgkLevel, f).offset for f, _ in PmgkLevel._fields_}


def _geometry(pmg, kernel, p, n, faces):
    """(grid, block, smem_bytes, n_chunks) of the apply launch the library issues for this box level on this device"""
    lib = pmg.lib()
    lv = PmgkLevel()
    lv.dim, lv.degree, (lv.nx, lv.ny, lv.nz) = 3, p, n
    lv.Nx, lv.Ny, lv.Nz = (c * p + 1 for c in n)
    lv.faces = faces
    lv.z0, lv.nzl, lv.cz_lo, lv.cz_hi, lv.z_own_lo, lv.z_own_hi = 0, lv.Nz, 0, n[2], 0, lv.Nz
    for d in range(3):
        lv.h[d] = 1.0 / n[d]
    v = VARIANT[kernel]
    lv.tile_variant = 0 if v is None else int(v)
    out = [C.c_int() for _ in range(4)]
    rc = lib.pmgk_apply_geometry(C.byref(lv), *[C.byref(o) for o in out])
    assert rc == 0, rc
    return tuple(o.value for o in out)


def _chunks(layers, n_chunks):
    """(layers per chunk, layers of the last chunk): both launchers cut ceil(layers / n_chunks) layers per chunk"""
    lpc = -(-layers // n_chunks)
    return lpc, layers - (n_chunks - 1) * lpc


def _sm_count(pmg):
    return int(pmg.lib().pmgk_device_sm_count())


# ---- apply matrix -------------------------------------------------------------------------------------------------------
F1, F2 = 0.37, 0.81


def _check_all_epilogues(pmg, ctx, oracle, p, n, faces, salt):
    mf = oracle.MatrixFree(3, p, n, faces=faces)
    N = mf.n_dofs
    u = splitmix_src(N, salt=salt)  # non-zero on constrained dofs: they must come out as src, bit for bit
    b = splitmix_src(N, salt=salt + 1)
    xo = splitmix_src(N, salt=salt + 2)
    Au = mf.vmult(u)
    dinv = mf.compute_diagonal()
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces)
    assert op.m() == N
    nan = np.full(N, np.nan)
    du, db = op.vector_from(u), op.vector_from(b)

    d = op.vector_from(nan)
    op.vmult(d, du)
    out = d.export_host()
    assert np.all(np.isfinite(out)), "vmult left entries unwritten"
    assert rel_l2(out, Au) <= APPLY_TOL, "vmult"
    c = mf.constrained()
    assert np.array_equal(out[c], u[c])
    op.vmult(d, du)
    assert np.array_equal(d.export_host(), out), "vmult not deterministic"

    r = op.vector_from(nan)
    op.residual(r, db, du)
    got = r.export_host()
    assert np.all(np.isfinite(got)) and rel_l2(got, b - Au) <= APPLY_TOL, "residual"

    def step_ref(x_old):
        return u + F1 * (u - x_old) + F2 * dinv * (b - Au)

    dst, dxo = op.vector_from(nan), op.vector_from(xo)
    op.chebyshev_step(dst, du, dxo, db, F1, F2)
    got = dst.export_host()
    assert np.all(np.isfinite(got)) and rel_l2(got, step_ref(xo)) <= APPLY_TOL, "chebyshev_step, separate x_old"
    assert np.array_equal(dxo.export_host(), xo), "chebyshev_step wrote x_old"
    op.chebyshev_step(dxo, du, dxo, db, F1, F2)  # x_old overwritten in place, as the smoother calls it
    assert rel_l2(dxo.export_host(), step_ref(xo)) <= APPLY_TOL, "chebyshev_step, x_old aliasing dst"
    dst = op.vector_from(nan)
    op.chebyshev_step(dst, du, None, db, F1, F2)
    got = dst.export_host()
    assert np.all(np.isfinite(got)) and rel_l2(got, step_ref(np.zeros(N))) <= APPLY_TOL, "chebyshev_step, no x_old"
    return op, mf


@pytest.mark.parametrize("faces", FACES, ids=lambda f: "f%02x" % f)
@pytest.mark.parametrize("kernel,p,table,n", APPLY_CASES,
                         ids=["%s-Q%d-%s-%dx%dx%d" % (k, p, t, *n) for k, p, t, n in APPLY_CASES])
def test_apply_epilogues_at_tile_edges(kernel, p, table, n, faces, pmg, ctx, oracle, kernel_variant):
    kernel_variant(kernel)
    _check_all_epilogues(pmg, ctx, oracle, p, n, faces, salt=p + 16 * faces)


@pytest.mark.parametrize("p", PLANE_DEGREES)
def test_plane_virtual_cell_tile_reached(p, pmg):
    """nx = BX with a natural high x face: the plane kernel's second x tile holds the virtual cell and nothing else (likewise
    y).  The launch on the device has that tile: grid = tiles_x tiles_y n_chunks with the extra tile counted."""
    bx, by = PLANE[(p, "apply")]
    for n, faces, tiles in (((bx, by, 2), 0x15, 4), ((bx, by, 2), 0x3F, 1), ((bx, by, 2), 0x2A, 1), ((bx, by, 2), 0x09, 2)):
        grid, _, _, n_chunks = _geometry(pmg, "plane", p, n, faces)
        assert grid == tiles * n_chunks, (n, hex(faces), grid, n_chunks)


# ---- large launches: multi-wave, multi-layer z-chunks with a short last chunk ---------------------------------------------
# every degree's large-level kernel (plane-per-step at the degrees of its table, line-marching above) and the line-marching
# kernel forced at the plane kernel's degrees
LARGE_CASES = [("plane", p) for p in PLANE_DEGREES] + [("sweep", p) for p in sorted(SWEEP)]


def _large_candidates(kernel, p):
    bx, by = PLANE[(p, "apply")] if kernel == "plane" else SWEEP[p][:2]
    cap = 3_500_000 if p >= 7 else 1_600_000
    out = []
    for a in range(1, 25):
        for b in range(1, 25):
            for nz in range(3, 400, 2):
                n = (a * bx + 1, max(b * by - 1, 1), nz)
                N = _n_dofs(p, n)
                if N > cap:
                    break
                out.append((N, n))
    return [n for _, n in sorted(out)]


def _large_mesh(pmg, kernel, p, faces):
    """The smallest candidate mesh whose launch on this device reaches every edge: >= 2 z-chunks and a last chunk shorter
    than the others; for the library's default large-level kernels a grid above twice the SM count; for the line-marching
    kernel with LZ > 1 layers per step, chunks of more than one step of which one ends in a partial step."""
    default_kernel = kernel == "plane" or p not in PLANE_DEGREES
    lz = SWEEP[p][2] if kernel == "sweep" else 1
    sms = _sm_count(pmg)
    for n in _large_candidates(kernel, p):
        grid, _, _, n_chunks = _geometry(pmg, kernel, p, n, faces)
        if n_chunks < 2:
            continue
        lpc, last = _chunks(n[2], n_chunks)
        if last >= lpc or (default_kernel and grid <= 2 * sms):
            continue
        if lz > 1 and not (lpc > lz and (lpc % lz or last % lz)):
            continue
        return n, grid, n_chunks
    pytest.fail("no mesh of at most %d DoFs reaches the launch edges of the %s kernel at Q%d" % (_n_dofs(p, n), kernel, p))


@pytest.mark.parametrize("kernel,p", LARGE_CASES, ids=["%s-Q%d" % c for c in LARGE_CASES])
def test_large_launch_chunks(kernel, p, pmg, ctx, oracle, kernel_variant):
    kernel_variant(kernel)
    faces = 0x15
    n, grid, n_chunks = _large_mesh(pmg, kernel, p, faces)
    mf = oracle.MatrixFree(3, p, n, faces=faces)
    N = mf.n_dofs
    u, b, xo = (splitmix_src(N, salt=40 + p + s) for s in range(3))
    Au = mf.vmult(u)
    dinv = mf.compute_diagonal()
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces)
    du, db, d = op.vector_from(u), op.vector_from(b), op.vector_from(np.full(N, np.nan))
    op.vmult(d, du)
    assert rel_l2(d.export_host(), Au) <= APPLY_TOL, (n, grid, n_chunks)
    op.residual(d, db, du)
    assert rel_l2(d.export_host(), b - Au) <= APPLY_TOL, (n, grid, n_chunks)
    dx = op.vector_from(xo)
    op.chebyshev_step(dx, du, dx, db, F1, F2)
    assert rel_l2(dx.export_host(), u + F1 * (u - xo) + F2 * dinv * (b - Au)) <= APPLY_TOL, (n, grid, n_chunks)
    op.chebyshev_step(d, du, None, db, F1, F2)
    assert rel_l2(d.export_host(), u + F1 * u + F2 * dinv * (b - Au)) <= APPLY_TOL, (n, grid, n_chunks)


# ---- transfers ----------------------------------------------------------------------------------------------------------
XFER_FACES = [0x3F, 0x15, 0x2A, 0x30, 0x00]
H_CASES = [(p, (3, 1, 2) if p % 2 else (1, 2, 3)) for p in range(1, 10)]  # one coarse cell in one direction
P_CASES = [(pc, pf) for pf in range(2, 10) for pc in range(1, pf)]


def _check_transfer(pmg, ctx, oracle, kind, pc, pf, nc, nf, faces):
    mc, mf = oracle.MatrixFree(3, pc, nc, faces=faces), oracle.MatrixFree(3, pf, nf, faces=faces)
    t_ref = oracle.Transfer(mc, mf, kind)
    oc, of = pmg.LaplaceOperator(ctx, pc, nc, dirichlet_faces=faces), pmg.LaplaceOperator(ctx, pf, nf, dirichlet_faces=faces)
    t = pmg.GeometricTransfer(oc, of) if kind == "h" else pmg.PolynomialTransfer(oc, of)
    salt = 100 * pc + pf + 1000 * faces
    xc, xf = splitmix_src(mc.n_dofs, mc.constrained(), salt=salt), splitmix_src(mf.n_dofs, salt=salt + 1)
    dst0, dstc0 = splitmix_src(mf.n_dofs, salt=salt + 2), splitmix_src(mc.n_dofs, salt=salt + 3)
    ref = t_ref.prolongate_and_add(dst0.copy(), xc)
    df = of.vector_from(dst0)
    t.prolongate_and_add(df, oc.vector_from(xc))
    assert rel_l2(df.export_host(), ref) <= XFER_TOL, "prolongate_and_add"
    ref = t_ref.restrict_and_add(dstc0.copy(), xf)
    dc = oc.vector_from(dstc0)
    t.restrict_and_add(dc, of.vector_from(xf))
    assert rel_l2(dc.export_host(), ref) <= XFER_TOL, "restrict_and_add"


@pytest.mark.parametrize("faces", XFER_FACES, ids=lambda f: "f%02x" % f)
@pytest.mark.parametrize("p,nc", H_CASES)
def test_h_transfer_all_degrees_and_faces(p, nc, faces, pmg, ctx, oracle):
    _check_transfer(pmg, ctx, oracle, "h", p, p, nc, tuple(2 * c for c in nc), faces)


@pytest.mark.parametrize("faces", XFER_FACES, ids=lambda f: "f%02x" % f)
@pytest.mark.parametrize("pc,pf", P_CASES)
def test_p_transfer_all_pairs_and_faces(pc, pf, faces, pmg, ctx, oracle):
    n = (2, 1, 3)
    _check_transfer(pmg, ctx, oracle, "p", pc, pf, n, n, faces)


def _interp_1d_sparse(p, n_from):
    """(dofs of the refined line, dofs of the coarse line): the coarse FE_Q(p) functions at the dofs of the mesh refined
    once, assembled as in the dense check (tests/test_oracle_dense.py interpolation_1d), sparse"""
    import scipy.sparse as sp
    from test_oracle_dense import interpolation_1d

    M1 = interpolation_1d(p, 1, p, 2)  # one coarse cell: (2p + 1) x (p + 1)
    rows, cols, vals = [], [], []
    for c in range(n_from):
        r0 = 0 if c == 0 else 1  # a coarse vertex lies in one cell only: its row is assigned once
        for r in range(r0, 2 * p + 1):
            for i in range(p + 1):
                if M1[r, i] != 0.0:
                    rows.append(c * 2 * p + r)
                    cols.append(c * p + i)
                    vals.append(M1[r, i])
    return sp.csr_matrix((vals, (rows, cols)), shape=(2 * n_from * p + 1, n_from * p + 1))


def _kron_apply(mats, x, shape_from):
    """(Mz kron My kron Mx) x, x lexicographic with x fastest, one factor at a time"""
    X = x.reshape(shape_from)  # (z, y, x)
    X = (mats[0] @ X.reshape(-1, shape_from[2]).T).T.reshape(shape_from[0], shape_from[1], -1)
    X = np.stack([mats[1] @ X[k] for k in range(X.shape[0])])
    X = (mats[2] @ X.reshape(X.shape[0], -1)).reshape(-1, X.shape[1], X.shape[2])
    return X.ravel()


@pytest.mark.parametrize("p", [1, 2])
def test_h_transfer_generic_instances_long_mesh(p, pmg, ctx):
    """65536 coarse cells in y: above the column kernels' 65535 grid rows, so the transfers run the generic kernels'
    compile-time instances (<8,2,3> at Q1, <8,3,5> at Q2).  Checked against the interpolation of the nested spaces as a
    Kronecker product of the 1-D interpolations with the constraint masks."""
    from test_oracle_dense import constrained_mask

    faces = 0x15
    nc, nf = (1, 65536, 1), (2, 131072, 2)
    oc, of = pmg.LaplaceOperator(ctx, p, nc, dirichlet_faces=faces), pmg.LaplaceOperator(ctx, p, nf, dirichlet_faces=faces)
    t = pmg.GeometricTransfer(oc, of)
    Pm = [_interp_1d_sparse(p, c) for c in nc]  # x, y, z
    zc, zf = ~constrained_mask(p, nc, faces), ~constrained_mask(p, nf, faces)
    sc = tuple(c * p + 1 for c in nc)[::-1]
    sf = tuple(c * p + 1 for c in nf)[::-1]
    xc = splitmix_src(oc.m(), salt=50) * zc
    xf, d0, c0 = splitmix_src(of.m(), salt=51), splitmix_src(of.m(), salt=52), splitmix_src(oc.m(), salt=53)
    df = of.vector_from(d0)
    t.prolongate_and_add(df, oc.vector_from(xc))
    assert rel_l2(df.export_host(), d0 + zf * _kron_apply(Pm, xc, sc)) <= XFER_TOL
    dc = oc.vector_from(c0)
    t.restrict_and_add(dc, of.vector_from(xf))
    ref = c0 + zc * _kron_apply([m.T.tocsr() for m in Pm], zf * xf, sf)
    assert rel_l2(dc.export_host(), ref) <= XFER_TOL


# ---- inverse diagonal, el, load vector, norm ------------------------------------------------------------------------------
DIAG_CASES = [(p, (5, 3, 2) if p % 2 else (2, 4, 3)) for p in range(1, 10)]
# Nx >= 48, 96, 192: the 64-, 128- and 256-thread blocks of k_dinv; the last one has more (plane, row) pairs than 32 per SM
# (checked in the test), so its blocks stride over rows
DIAG_WIDE = [(1, (50, 3, 4)), (2, (50, 5, 3)), (1, (200, 6, 5)), (2, (100, 60, 40))]


def _check_diag_rhs_norm(pmg, ctx, oracle, p, n, faces):
    mf = oracle.MatrixFree(3, p, n, faces=faces)
    ref = mf.compute_diagonal()
    op = pmg.LaplaceOperator(ctx, p, n, dirichlet_faces=faces)
    op.compute_diagonal()
    assert rel_l2(op.get_matrix_diagonal_inverse().export_host(), ref) <= XFER_TOL
    b = op.initialize_dof_vector()
    op.assemble_rhs(b)
    assert rel_l2(b.export_host(), mf.assemble_rhs()) <= XFER_TOL
    u = splitmix_src(mf.n_dofs, salt=60 + p)
    norm, norm_ref = op.solution_norm(op.vector_from(u)), mf.l2_norm_solution(u)
    assert abs(norm - norm_ref) <= XFER_TOL * norm_ref
    return mf, op, ref


@pytest.mark.parametrize("faces", FACES, ids=lambda f: "f%02x" % f)
@pytest.mark.parametrize("p,n", DIAG_CASES)
def test_diagonal_rhs_norm_mixed_faces(p, n, faces, pmg, ctx, oracle):
    mf, op, ref = _check_diag_rhs_norm(pmg, ctx, oracle, p, n, faces)
    Nx, Ny, Nz = mf.nd
    c = mf.constrained()
    # a row on a natural face (x = 0 or x = Nx - 1, whichever is natural), interior in y and z
    for gx in (0, Nx - 1):
        row = ((Nz // 2) * Ny + Ny // 2) * Nx + gx
        if not c[row]:
            assert abs(op.el(row, row) - 1.0 / ref[row]) <= 1e-12 / ref[row]
    row = int(np.flatnonzero(c)[0]) if c.any() else 0
    assert abs(op.el(row, row) - 1.0 / ref[row]) <= 1e-12 / ref[row]  # 1 on a constrained row


@pytest.mark.parametrize("p,n", DIAG_WIDE)
def test_diagonal_wide_rows(p, n, pmg, ctx, oracle):
    if n == DIAG_WIDE[-1][1]:
        assert (n[1] * p + 1) * (n[2] * p + 1) > 32 * _sm_count(pmg), "the mesh no longer reaches k_dinv's row loop"
    _check_diag_rhs_norm(pmg, ctx, oracle, p, n, 0x15)


# ---- multigrid on mixed faces -----------------------------------------------------------------------------------------------
# Natural faces everywhere but two (0x09) or three (0x15, 0x2A).  One Dirichlet face alone (0x01) is not compared: the coarse
# level's eigenvalue estimate then runs CG until its residual falls below 1e-10, 17 iterations for 16 free dofs at Q1 and 101 at
# Q5, where round-off decides the count -- two runs of the multi-threaded oracle on the same Q5 level return lambda_max 2.7286
# and 2.7438.
MG_FACES = [0x15, 0x2A, 0x09]
MG_KERNELS = ["default", "plane", "sweep"]
H2_LEVELS = {p: [(p, (2, 3, 1)), (p, (4, 6, 2))] for p in range(1, 10)}
HP_LEVELS = {"9-4-2-1": [9, 4, 2, 1], "7-3-1": [7, 3, 1], "6-3-1": [6, 3, 1], "5-2-1": [5, 2, 1]}
MG_CASES = [("h%d" % p, lv) for p, lv in H2_LEVELS.items()] + \
           [("hp" + k, [(d, (2, 3, 2)) for d in reversed(v)]) for k, v in HP_LEVELS.items()]


def _check_vcycle_and_cg(pmg, ctx, oracle, levels, faces, launches=None):
    mfs = [oracle.MatrixFree(3, p, n, faces=faces) for (p, n) in levels]
    trs = [oracle.Transfer(mfs[l - 1], mfs[l], "h" if levels[l][0] == levels[l - 1][0] else "p") for l in range(1, len(levels))]
    vc_ref = oracle.VCycle(mfs, trs)
    ops, transfers, smoothers, mg = pmg.build_hierarchy(ctx, levels, faces=faces)
    top = ops[-1]
    est = vc_ref.estimate()
    for l, sm in enumerate(smoothers):
        info = sm.info()
        assert info["degree"] == est[l][2] and info["cg_iterations"] == est[l][3], (l, info, est[l])
        assert abs(info["lambda_max"] - est[l][1]) <= 1e-8 * est[l][1], (l, info, est[l])
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=70)
    z_ref = vc_ref.vmult(r)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    for rep in range(3):  # eager, graph capture, graph replay
        before = ctx.launch_count()
        mg.vmult(dz, dr)
        if launches is not None:
            launches.append(ctx.launch_count() - before)
        assert rel_l2(dz.export_host(), z_ref) <= HISTORY_TOL, rep
    b_ref = mfs[-1].assemble_rhs()
    b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    x_ref, it_ref, hist_ref, rc_ref = oracle.cg_solve(mfs[-1], b_ref, vc_ref)
    it, hist, rc = pmg.cg_solve(top, x, b, mg)
    assert rc == 0 and rc_ref == 0 and it == it_ref, (rc, rc_ref, it, it_ref)
    assert np.all(np.abs(hist - hist_ref) <= HISTORY_TOL * hist_ref[0])
    assert rel_l2(x.export_host(), x_ref) <= 1e-9


@pytest.mark.parametrize("kernel", MG_KERNELS)
@pytest.mark.parametrize("faces", MG_FACES, ids=lambda f: "f%02x" % f)
@pytest.mark.parametrize("name,levels", MG_CASES, ids=[c[0] for c in MG_CASES])
def test_vcycle_and_cg_mixed_faces(name, levels, faces, kernel, pmg, ctx, oracle, kernel_variant):
    """Every smoother step of the V-cycle runs a fused epilogue (the first Chebyshev step included, which no operator call
    reaches), on every level's kernel."""
    kernel_variant(kernel)
    _check_vcycle_and_cg(pmg, ctx, oracle, levels, faces)


@pytest.mark.parametrize("faces", MG_FACES, ids=lambda f: "f%02x" % f)
@pytest.mark.parametrize("p", [1, 2, 3, 4])  # the degrees the single-CTA coarse-cycle kernel is compiled for
def test_coarse_cycle_kernel_mixed_faces(p, faces, pmg, ctx, oracle, monkeypatch):
    """PMG_COARSE_KERNEL=1 runs both levels inside the single-CTA kernel; compared with the oracle itself."""
    monkeypatch.setenv("PMG_COARSE_KERNEL", "1")  # read at the cycle's first vmult
    monkeypatch.setenv("PMG_COARSE_MAX_WORK", "4e6")
    launches = []
    _check_vcycle_and_cg(pmg, ctx, oracle, H2_LEVELS[p], faces, launches)
    assert launches[0] <= 2, launches  # the whole cycle is the coarse kernel (and at most one copy)


# ---- reductions ---------------------------------------------------------------------------------------------------------------
def test_reductions_large_odd_level(pmg, ctx):
    p, n = 2, (63, 61, 67)  # 2 096 953 DoFs (odd): more blocks than the reductions' cap
    op = pmg.LaplaceOperator(ctx, p, n)
    N = op.m()
    assert N % 2 == 1 and N > 2_000_000
    x, y = splitmix_src(N, salt=80), splitmix_src(N, salt=81) + 0.25
    dx, dy = op.vector_from(x), op.vector_from(y)
    terms = x * y
    dot = dx.dot(dy)
    assert abs(dot - math.fsum(terms)) <= 1e-14 * np.abs(terms).sum()
    nrm = dx.l2_norm()
    sq = x * x
    assert abs(nrm * nrm - math.fsum(sq)) <= 1e-14 * sq.sum()
    mean = dy.mean_value()
    assert abs(mean - math.fsum(y) / N) <= 1e-14 * np.abs(y).sum() / N
    for _ in range(3):
        assert dx.dot(dy) == dot and dx.l2_norm() == nrm and dy.mean_value() == mean
