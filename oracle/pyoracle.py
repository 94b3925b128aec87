"""ctypes binding of the CPU oracle (oracle/orc.h).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Never imported by the product package.
Parity unpinned (see orc.h): the reference has no golden vectors and cannot be built here.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)


def build(native=False, out_dir=None):
    """Compile the oracle (make) into oracle/_build, or into out_dir (the source tree may be read-only).
    native=True builds -march=native into a second .so."""
    out = os.path.join(out_dir or os.path.join(_HERE, "_build"), "liborc_native.so" if native else "liborc.so")
    args = ["make", "-C", _HERE, "OUT=" + out] + (["MARCH=native"] if native else [])
    subprocess.run(args, check=True, stdout=subprocess.DEVNULL)
    return out


def _load(native=False, path=None):
    if path is None:
        path = os.path.join(_HERE, "_build", "liborc_native.so" if native else "liborc.so")
        if not os.path.exists(path):
            path = build(native)
    lib = C.CDLL(path)
    vp = C.c_void_p
    lib.orc_mf_create.restype = vp
    lib.orc_mf_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint, vp]
    lib.orc_mf_destroy.argtypes = [vp]
    lib.orc_vmult.argtypes = [vp, _dp, _dp]
    lib.orc_compute_diagonal.argtypes = [vp]
    lib.orc_transfer_create_h.restype = vp
    lib.orc_transfer_create_h.argtypes = [vp, vp]
    lib.orc_transfer_create_p.restype = vp
    lib.orc_transfer_create_p.argtypes = [vp, vp]
    lib.orc_transfer_destroy.argtypes = [vp]
    lib.orc_prolongate_and_add.argtypes = [vp, _dp, _dp]
    lib.orc_restrict_and_add.argtypes = [vp, _dp, _dp]
    lib.orc_assemble_rhs.argtypes = [vp, _dp]
    lib.orc_l2_norm_solution.restype = C.c_double
    lib.orc_l2_norm_solution.argtypes = [vp, _dp]
    lib.orc_tridiag_eigenvalues.argtypes = [C.c_int, _dp, _dp, _dp]
    lib.orc_shape_tables.argtypes = [C.c_int, _dp, _dp, _dp]
    lib.orc_h_prolongation_1d.argtypes = [C.c_int, _dp]
    lib.orc_p_prolongation_1d.argtypes = [C.c_int, C.c_int, _dp]
    lib.orc_gauss_legendre.argtypes = [C.c_int, _dp, _dp]
    lib.orc_gauss_lobatto.argtypes = [C.c_int, _dp]
    lib.orc_num_threads.restype = C.c_int
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load(os.environ.get("ORC_NATIVE", "0") == "1")
    return _lib


def use_library(path):
    """Switch to the oracle library at `path`, as returned by build(native, out_dir) (bench.py's CPU legs)."""
    global _lib
    _lib = _load(path=path)


def _p(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


class _MFStruct(C.Structure):
    _fields_ = [
        ("dim", C.c_int), ("p", C.c_int), ("n", C.c_int * 3), ("nd", C.c_int * 3),
        ("h", C.c_double * 3), ("faces", C.c_uint), ("n_cells", C.c_int64), ("n_dofs", C.c_int64),
        ("n_loc", C.c_int), ("n_q", C.c_int),
        ("local_to_global", C.c_void_p), ("mask", C.c_void_p), ("inv_jacobian", C.c_void_p),
        ("JxW", C.c_void_p), ("constrained", C.c_void_p),
        ("shape_values", C.c_double * 100), ("co_shape_gradients", C.c_double * 100),
        ("gauss_w", C.c_double * 10),
        ("n_colors", C.c_int), ("color_start", C.c_void_p), ("color_cells", C.c_void_p),
        ("inv_diag", C.c_void_p),
    ]


class _ChebStruct(C.Structure):
    _fields_ = [
        ("mf", C.c_void_p), ("smoothing_range", C.c_double), ("degree", C.c_int),
        ("eig_cg_n_iterations", C.c_int), ("initialized", C.c_int),
        ("lambda_min", C.c_double), ("lambda_max", C.c_double), ("theta", C.c_double),
        ("delta", C.c_double), ("cg_iterations", C.c_int),
    ]


class _VCycleStruct(C.Structure):
    _fields_ = [
        ("n_levels", C.c_int), ("mf", C.POINTER(C.c_void_p)), ("transfer", C.POINTER(C.c_void_p)),
        ("smoother", C.POINTER(_ChebStruct)), ("pre", C.c_int), ("post", C.c_int),
    ]


ALL_FACES_3D = 0x3F
ALL_FACES_2D = 0x0F


class MatrixFree:
    """One level: reference-layout matrix-free data + LaplaceOperator."""

    def __init__(self, dim, p, n, faces=None, coef=None):
        if isinstance(n, int):
            n = (n,) * dim
        n = tuple(n) + (1,) * (3 - len(n))
        if faces is None:
            faces = ALL_FACES_3D if dim == 3 else ALL_FACES_2D
        cf = None
        if coef == "c5":
            cf = C.cast(lib().orc_coef_c5, C.c_void_p)
        self.h = lib().orc_mf_create(dim, p, n[0], n[1], n[2], faces, cf)
        self.s = _MFStruct.from_address(self.h)
        self.dim, self.p = dim, p
        self.n_dofs = int(self.s.n_dofs)
        self.n_cells = int(self.s.n_cells)
        self.nd = tuple(self.s.nd)[:dim]
        self.ncell = n[:dim]

    def __del__(self):
        try:
            lib().orc_mf_destroy(self.h)
        except Exception:
            pass

    def vmult(self, src):
        dst = np.empty(self.n_dofs)
        lib().orc_vmult(self.h, _p(dst), _p(np.ascontiguousarray(src, dtype=np.float64)))
        return dst

    def compute_diagonal(self):
        lib().orc_compute_diagonal(self.h)
        return self.inv_diag()

    def inv_diag(self):
        return np.ctypeslib.as_array(C.cast(self.s.inv_diag, _dp), shape=(self.n_dofs,)).copy()

    def constrained(self):
        return np.ctypeslib.as_array(C.cast(self.s.constrained, C.POINTER(C.c_uint8)), shape=(self.n_dofs,)).astype(bool)

    def assemble_rhs(self):
        b = np.empty(self.n_dofs)
        lib().orc_assemble_rhs(self.h, _p(b))
        return b

    def l2_norm_solution(self, u):
        return float(lib().orc_l2_norm_solution(self.h, _p(np.ascontiguousarray(u))))


class Transfer:
    def __init__(self, coarse, fine, kind):
        self.coarse, self.fine, self.kind = coarse, fine, kind
        f = lib().orc_transfer_create_h if kind == "h" else lib().orc_transfer_create_p
        self.h = f(coarse.h, fine.h)
        if not self.h:
            raise ValueError("incompatible levels for %s-transfer" % kind)

    def __del__(self):
        try:
            lib().orc_transfer_destroy(self.h)
        except Exception:
            pass

    def prolongate_and_add(self, dst_fine, src_coarse):
        lib().orc_prolongate_and_add(self.h, _p(dst_fine), _p(np.ascontiguousarray(src_coarse)))
        return dst_fine

    def restrict_and_add(self, dst_coarse, src_fine):
        lib().orc_restrict_and_add(self.h, _p(dst_coarse), _p(np.ascontiguousarray(src_fine)))
        return dst_coarse


class VCycle:
    """VCycleMultigrid with PreconditionChebyshev smoothers configured like the drivers
    (source/geometric_multigrid/program.cc:267-279)."""

    def __init__(self, levels, transfers, pre=2, post=2, degree=5, smoothing_range=15.0,
                 eig_cg_n_iterations=10, coarse_range=1e-3):
        L = len(levels)
        assert len(transfers) == L - 1
        self.levels, self.transfers = levels, transfers
        self._mf = (C.c_void_p * L)(*[m.h for m in levels])
        self._tr = (C.c_void_p * L)(*([None] + [t.h for t in transfers]))
        self._sm = (_ChebStruct * L)()
        for l, m in enumerate(levels):
            if m.s.inv_diag is None:
                m.compute_diagonal()
            if l > 0:
                lib().orc_chebyshev_init(C.byref(self._sm[l]), C.c_void_p(m.h), C.c_double(smoothing_range),
                                         degree, eig_cg_n_iterations)
            else:
                lib().orc_chebyshev_init(C.byref(self._sm[l]), C.c_void_p(m.h), C.c_double(coarse_range),
                                         -1, int(m.n_dofs))
        self.s = _VCycleStruct(L, C.cast(self._mf, C.POINTER(C.c_void_p)), C.cast(self._tr, C.POINTER(C.c_void_p)),
                               C.cast(self._sm, C.POINTER(_ChebStruct)), pre, post)

    def estimate(self):
        for l in range(len(self.levels)):
            lib().orc_chebyshev_estimate(C.byref(self._sm[l]))
        return [(s.lambda_min, s.lambda_max, s.degree, s.cg_iterations, s.theta, s.delta) for s in self._sm]

    def vmult(self, src):
        dst = np.empty(self.levels[-1].n_dofs)
        lib().orc_vcycle_vmult(C.byref(self.s), _p(dst), _p(np.ascontiguousarray(src)))
        return dst


def chebyshev_vmult(mf, src, degree=5, smoothing_range=15.0, eig_cg_n_iterations=10):
    c = _ChebStruct()
    if mf.s.inv_diag is None:
        mf.compute_diagonal()
    lib().orc_chebyshev_init(C.byref(c), C.c_void_p(mf.h), C.c_double(smoothing_range), degree, eig_cg_n_iterations)
    dst = np.empty(mf.n_dofs)
    lib().orc_chebyshev_vmult(C.byref(c), _p(dst), _p(np.ascontiguousarray(src)))
    return dst, dict(lambda_min=c.lambda_min, lambda_max=c.lambda_max, degree=c.degree,
                     cg_iterations=c.cg_iterations, theta=c.theta, delta=c.delta)


def cg_solve(A, b, precond=None, max_it=None, rel_tol=1e-12, x0=None):
    n = A.n_dofs
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)
    max_it = n if max_it is None else max_it
    hist = np.zeros(max_it + 2)
    last = C.c_int(0)
    tol = rel_tol * float(np.linalg.norm(b))
    lib().orc_cg_solve.argtypes = [C.c_void_p, _dp, _dp, C.c_void_p, C.c_int, C.c_double,
                                   C.POINTER(C.c_int), _dp, C.c_int]
    rc = lib().orc_cg_solve(A.h, _p(x), _p(np.ascontiguousarray(b)), C.byref(precond.s) if precond else None,
                            max_it, tol, C.byref(last), _p(hist), len(hist))
    return x, last.value, hist[: last.value + 1].copy(), rc


def shape_tables(p):
    n = p + 1
    S, D, w = np.zeros(n * n), np.zeros(n * n), np.zeros(n)
    lib().orc_shape_tables(p, _p(S), _p(D), _p(w))
    return S.reshape(n, n), D.reshape(n, n), w


def gauss_lobatto(n):
    x = np.zeros(n)
    lib().orc_gauss_lobatto(n, _p(x))
    return x


def gauss_legendre(n):
    x, w = np.zeros(n), np.zeros(n)
    lib().orc_gauss_legendre(n, _p(x), _p(w))
    return x, w


def h_prolongation_1d(p):
    P = np.zeros((p + 1) * (2 * p + 1))
    lib().orc_h_prolongation_1d(p, _p(P))
    return P.reshape(p + 1, 2 * p + 1)


def p_prolongation_1d(pc, pf):
    P = np.zeros((pc + 1) * (pf + 1))
    lib().orc_p_prolongation_1d(pc, pf, _p(P))
    return P.reshape(pc + 1, pf + 1)


def tridiag_eigenvalues(diag, off):
    n = len(diag)
    e = np.zeros(n)
    lib().orc_tridiag_eigenvalues(n, _p(np.ascontiguousarray(diag, dtype=np.float64)),
                                  _p(np.ascontiguousarray(np.append(off, 0.0), dtype=np.float64)), _p(e))
    return e


def num_threads():
    return int(lib().orc_num_threads())


def synthetic_src(n_dofs, constrained=None):
    """src_i = 2*u01(splitmix64(i ^ 0x9E3779B97F4A7C15)) - 1, zero on Dirichlet dofs (SURVEY.md 8d)."""
    i = np.arange(n_dofs, dtype=np.uint64) ^ np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        z = i + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    u = (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    v = 2.0 * u - 1.0
    if constrained is not None:
        v[constrained] = 0.0
    return v
