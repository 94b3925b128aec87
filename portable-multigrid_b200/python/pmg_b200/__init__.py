"""ctypes binding of libpmg.so (include/pmg.h) for the test-suite, bench.py and smoke().

Thin, one class per handle type, method names = the reference's method names
(LaplaceOperatorBase, MGTransferBase, VCycleMultigrid; reference include/base/*.h).
This module contains no numerics of its own and no CPU fallback: if the CUDA library is missing or
no GPU is present, the calls raise PmgError.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.normpath(os.path.join(_HERE, "..", "..", "lib", "libpmg.so"))

PMG_ALL_FACES = 0x3F
PMG_INVALID_DEGREE = -1
PMG_MAX_DEGREE = 9
_dp = C.POINTER(C.c_double)
_vp = C.c_void_p


class PmgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("pmg error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    """Load libpmg.so (built by `make -C portable-multigrid_b200` / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PmgError(-2, "libpmg.so not built at %s (run __graft_entry__.build()); there is no fallback" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _lib.pmg_last_error.restype = C.c_char_p
        _lib.pmg_version.restype = C.c_char_p
        _lib.pmg_vector_device_ptr.restype = C.c_void_p
        _lib.pmg_vector_device_ptr.argtypes = [_vp]
        _lib.pmg_context_stream.restype = C.c_void_p
        _lib.pmg_context_stream.argtypes = [_vp]
        _lib.pmg_context_launch_count.restype = C.c_int64
        _lib.pmg_context_launch_count.argtypes = [_vp]
        _lib.pmg_context_fused_halo_count.restype = C.c_int64
        _lib.pmg_context_fused_halo_count.argtypes = [_vp]
    return _lib


def _ck(rc):
    if rc != 0:
        raise PmgError(rc, lib().pmg_last_error().decode(errors="replace"))


def _np_ptr(a):
    assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


def _host_ptr(a):
    """numpy array or an int address (e.g. a pinned torch tensor's data_ptr())."""
    if isinstance(a, np.ndarray):
        return _np_ptr(a)
    return C.cast(C.c_void_p(int(a)), _dp)


class Context:
    def __init__(self, device=0, rank=0, n_ranks=1, nccl_id=None):
        self.h = _vp()
        if n_ranks == 1:
            _ck(lib().pmg_context_create(C.byref(self.h), C.c_int(device)))
        else:
            buf = C.create_string_buffer(bytes(nccl_id), 128)
            _ck(lib().pmg_context_create_distributed(C.byref(self.h), C.c_int(device), C.c_int(rank), C.c_int(n_ranks), buf))
        self.rank, self.n_ranks, self.device = rank, n_ranks, device

    @staticmethod
    def nccl_unique_id():
        buf = C.create_string_buffer(128)
        _ck(lib().pmg_nccl_unique_id(buf))
        return bytes(buf.raw)

    def sync(self):
        _ck(lib().pmg_sync(self.h))

    def set_coarse_threshold(self, n):
        _ck(lib().pmg_context_set_coarse_threshold(self.h, C.c_int64(n)))

    def stream(self):
        return lib().pmg_context_stream(self.h)

    def launch_count(self):
        return int(lib().pmg_context_launch_count(self.h))

    def fused_halo_count(self):
        """Applies whose ghost planes came from the previous apply's fused push (no exchange of their own)."""
        return int(lib().pmg_context_fused_halo_count(self.h))

    def microbench(self):
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        _ck(lib().pmg_microbench(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return dict(fp64_fma_tflops=a.value, fp64_dmma_tflops=b.value, hbm_copy_gbs=c.value)

    def close(self):
        if self.h:
            lib().pmg_context_destroy(self.h)
            self.h = _vp()


class Vector:
    def __init__(self, handle, ctx, owned=True):
        self.h, self.ctx, self._owned = handle, ctx, owned

    def __del__(self):
        try:
            if self._owned and self.h and self.ctx.h:
                lib().pmg_vector_destroy(self.h)
        except Exception:
            pass

    def size(self):
        n = C.c_int64()
        _ck(lib().pmg_vector_size(self.h, C.byref(n)))
        return n.value

    def locally_owned_size(self):
        n = C.c_int64()
        _ck(lib().pmg_vector_locally_owned_size(self.h, C.byref(n)))
        return n.value

    def set(self, value):
        _ck(lib().pmg_vector_set(self.h, C.c_double(value)))

    def copy_from(self, other):
        _ck(lib().pmg_vector_copy(self.h, other.h))

    def scale(self, a):
        _ck(lib().pmg_vector_scale(self.h, C.c_double(a)))

    def add(self, a, x):
        _ck(lib().pmg_vector_add(self.h, C.c_double(a), x.h))

    def sadd(self, s, a, x):
        _ck(lib().pmg_vector_sadd(self.h, C.c_double(s), C.c_double(a), x.h))

    def dot(self, other):
        r = C.c_double()
        _ck(lib().pmg_vector_dot(self.h, other.h, C.byref(r)))
        return r.value

    def l2_norm(self):
        r = C.c_double()
        _ck(lib().pmg_vector_l2_norm(self.h, C.byref(r)))
        return r.value

    def mean_value(self):
        r = C.c_double()
        _ck(lib().pmg_vector_mean_value(self.h, C.byref(r)))
        return r.value

    def update_ghost_values(self):
        _ck(lib().pmg_vector_update_ghost_values(self.h))

    def compress_add(self):
        _ck(lib().pmg_vector_compress_add(self.h))

    def zero_out_ghost_values(self):
        _ck(lib().pmg_vector_zero_out_ghost_values(self.h))

    def import_host(self, a):
        _ck(lib().pmg_vector_import_host(self.h, _host_ptr(a)))
        self.ctx.sync()

    def export_host(self, out=None):
        if out is None:
            out = np.empty(self.size())
        _ck(lib().pmg_vector_export_host(self.h, _host_ptr(out)))
        return out

    def device_ptr(self):
        return lib().pmg_vector_device_ptr(self.h)

    def local_range(self):
        """(plane_size, z0, n_planes, z_own_lo, z_own_hi): the rank's stored / owned dof planes."""
        pl = C.c_int64()
        z0, nz, lo, hi = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _ck(lib().pmg_vector_local_range(self.h, C.byref(pl), C.byref(z0), C.byref(nz), C.byref(lo), C.byref(hi)))
        return pl.value, z0.value, nz.value, lo.value, hi.value

    def import_owned(self, a):
        _ck(lib().pmg_vector_import_owned(self.h, _host_ptr(a)))
        self.ctx.sync()

    def export_owned(self, out=None):
        pl, _, _, lo, hi = self.local_range()
        if out is None:
            out = np.empty(pl * (hi - lo))
        _ck(lib().pmg_vector_export_owned(self.h, _host_ptr(out)))
        return out

    def import_local(self, a):
        _ck(lib().pmg_vector_import_local(self.h, _host_ptr(a)))

    def export_local(self, out=None):
        pl, _, nz, _, _ = self.local_range()
        if out is None:
            out = np.empty(pl * nz)
        _ck(lib().pmg_vector_export_local(self.h, _host_ptr(out)))
        return out

    def wrap(self, device_ptr):
        """A non-owning vector with this vector's layout over caller-owned device memory (pmg_vector_wrap)."""
        v = _vp()
        _ck(lib().pmg_vector_wrap(self.h, C.c_void_p(device_ptr), C.byref(v)))
        return Vector(v, self.ctx)


class LaplaceOperator:
    """Portable::LaplaceOperator (reference include/operators/portable_laplace_operator.h:383-461)."""

    def __init__(self, ctx, degree, n, dirichlet_faces=PMG_ALL_FACES, dim=3, coefficient=0, vertices=None, nodes=None,
                 geometry_degree=None):
        """vertices: None (the unit cube cut into equal boxes) or the (nx+1)(ny+1)(nz+1) mesh vertices of a deformed
        structured mesh, shape (nz+1, ny+1, nx+1, 3) or flat in that order (pmg_laplace_operator_create_mapped); 3-D only.
        nodes: instead of vertices, the (nx k+1)(ny k+1)(nz k+1) geometry support points of curved cells of degree
        k = geometry_degree (mesh_nodes; pmg_laplace_operator_create_curved), shape (nz k+1, ny k+1, nx k+1, 3) or flat;
        geometry_degree None: the k the array's size implies."""
        if isinstance(n, int):
            n = (n,) * dim
        n = tuple(n) + (1,) * (3 - len(n))  # dim = 2: (nx, ny); the C-ABI ignores nz
        self.ctx, self.degree, self.ncells, self.dim = ctx, degree, tuple(n), dim
        self.h = _vp()
        self.vertices = None
        self.nodes, self.geometry_degree = None, None
        if vertices is None and nodes is None:
            _ck(lib().pmg_laplace_operator_create(ctx.h, C.c_int(dim), C.c_int(degree), C.c_int(n[0]), C.c_int(n[1]),
                                                  C.c_int(n[2]), C.c_uint(dirichlet_faces), C.c_int(coefficient), C.byref(self.h)))
            return
        if vertices is not None and nodes is not None:
            raise PmgError(-1, "vertices= and nodes= are mutually exclusive")
        if dim != 3:
            raise PmgError(-3, "the mapped operator is 3-D only (dim = %d)" % dim)
        if nodes is not None:
            v = np.ascontiguousarray(nodes, dtype=np.float64).reshape(-1)
            k = geometry_degree if geometry_degree is not None else _geometry_degree_of(v.size, n)
            if 1 <= k <= PMG_MAX_DEGREE and v.size != 3 * _n_nodes(n, k):
                raise PmgError(-1, "nodes: %d values for %d x %d x %d cells of geometry degree %d, need 3 (nx k+1)(ny k+1)(nz k+1)"
                               % (v.size, *n, k))
            _ck(lib().pmg_laplace_operator_create_curved(ctx.h, C.c_int(degree), C.c_int(k), C.c_int(n[0]), C.c_int(n[1]),
                                                         C.c_int(n[2]), C.c_uint(dirichlet_faces), C.c_int(coefficient),
                                                         _np_ptr(v), C.byref(self.h)))
            self.nodes, self.geometry_degree = v.reshape(n[2] * k + 1, n[1] * k + 1, n[0] * k + 1, 3), k
            return
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1)
        if v.size != 3 * (n[0] + 1) * (n[1] + 1) * (n[2] + 1):
            raise PmgError(-1, "vertices: %d values for %d x %d x %d cells, need 3 (nx+1)(ny+1)(nz+1)" % (v.size, *n))
        self.vertices = v.reshape(n[2] + 1, n[1] + 1, n[0] + 1, 3)
        _ck(lib().pmg_laplace_operator_create_mapped(ctx.h, C.c_int(degree), C.c_int(n[0]), C.c_int(n[1]), C.c_int(n[2]),
                                                     C.c_uint(dirichlet_faces), C.c_int(coefficient), _np_ptr(v),
                                                     C.byref(self.h)))

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                lib().pmg_laplace_operator_destroy(self.h)
        except Exception:
            pass

    def initialize_dof_vector(self):
        v = _vp()
        _ck(lib().pmg_laplace_operator_initialize_dof_vector(self.h, C.byref(v)))
        return Vector(v, self.ctx)

    def vector_from(self, host):
        v = self.initialize_dof_vector()
        v.import_host(np.ascontiguousarray(host, dtype=np.float64))
        return v

    def vmult(self, dst, src):
        _ck(lib().pmg_laplace_operator_vmult(self.h, dst.h, src.h))

    def Tvmult(self, dst, src):
        _ck(lib().pmg_laplace_operator_Tvmult(self.h, dst.h, src.h))

    def residual(self, dst, b, src):
        _ck(lib().pmg_laplace_operator_residual(self.h, dst.h, b.h, src.h))

    def chebyshev_step(self, dst, src, xold, b, f1, f2):
        _ck(lib().pmg_laplace_operator_chebyshev_step(self.h, dst.h, src.h, xold.h if xold is not None else None, b.h,
                                                      C.c_double(f1), C.c_double(f2)))

    def vmult_host(self, dst, src):
        _ck(lib().pmg_laplace_operator_vmult_host(self.h, _host_ptr(dst), _host_ptr(src)))

    def compute_diagonal(self):
        _ck(lib().pmg_laplace_operator_compute_diagonal(self.h))

    def get_matrix_diagonal_inverse(self):
        v = _vp()
        _ck(lib().pmg_laplace_operator_get_matrix_diagonal_inverse(self.h, C.byref(v)))
        return Vector(v, self.ctx, owned=False)

    def m(self):
        n = C.c_int64()
        _ck(lib().pmg_laplace_operator_m(self.h, C.byref(n)))
        return n.value

    def n(self):
        n = C.c_int64()
        _ck(lib().pmg_laplace_operator_n(self.h, C.byref(n)))
        return n.value

    def el(self, row, col):
        r = C.c_double()
        _ck(lib().pmg_laplace_operator_el(self.h, C.c_int64(row), C.c_int64(col), C.byref(r)))
        return r.value

    def assemble_rhs(self, rhs):
        _ck(lib().pmg_laplace_operator_assemble_rhs(self.h, rhs.h))

    def solution_norm(self, u):
        r = C.c_double()
        _ck(lib().pmg_laplace_operator_solution_norm(self.h, u.h, C.byref(r)))
        return r.value


class _Transfer:
    def __del__(self):
        try:
            if self.h and self.ctx.h:
                lib().pmg_transfer_destroy(self.h)
        except Exception:
            pass

    def prolongate_and_add(self, dst_fine, src_coarse):
        _ck(lib().pmg_transfer_prolongate_and_add(self.h, dst_fine.h, src_coarse.h))

    def restrict_and_add(self, dst_coarse, src_fine):
        _ck(lib().pmg_transfer_restrict_and_add(self.h, dst_coarse.h, src_fine.h))


class GeometricTransfer(_Transfer):
    """Portable::GeometricTransfer (reference include/multigrid/portable_geometric_transfer.h:687-753)."""

    def __init__(self, coarse, fine):
        self.ctx, self.coarse, self.fine = coarse.ctx, coarse, fine
        self.h = _vp()
        _ck(lib().pmg_transfer_create_geometric(coarse.h, fine.h, C.byref(self.h)))


class PolynomialTransfer(_Transfer):
    """Portable::PolynomialTransfer (reference include/multigrid/portable_polynomial_tranfer.h:618-668)."""

    def __init__(self, coarse, fine):
        self.ctx, self.coarse, self.fine = coarse.ctx, coarse, fine
        self.h = _vp()
        _ck(lib().pmg_transfer_create_polynomial(coarse.h, fine.h, C.byref(self.h)))


class Chebyshev:
    """PreconditionChebyshev with the Jacobi inner preconditioner (program.cc:267-285)."""

    def __init__(self, op, smoothing_range=15.0, degree=5, eig_cg_n_iterations=10):
        self.ctx, self.op = op.ctx, op
        self.h = _vp()
        _ck(lib().pmg_chebyshev_create(op.h, C.c_double(smoothing_range), C.c_int(degree), C.c_int(eig_cg_n_iterations), C.byref(self.h)))

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                lib().pmg_chebyshev_destroy(self.h)
        except Exception:
            pass

    def vmult(self, dst, src):
        _ck(lib().pmg_chebyshev_vmult(self.h, dst.h, src.h))

    def info(self):
        a, b, d, i = C.c_double(), C.c_double(), C.c_int(), C.c_int()
        _ck(lib().pmg_chebyshev_info(self.h, C.byref(a), C.byref(b), C.byref(d), C.byref(i)))
        return dict(lambda_min=a.value, lambda_max=b.value, degree=d.value, cg_iterations=i.value)


class VCycleMultigrid:
    """Portable::VCycleMultigrid (reference include/multigrid/portable_v_cycle_multigrid.h:26-63)."""

    def __init__(self, ops, transfers, smoothers, pre=2, post=2):
        L = len(ops)
        assert len(smoothers) == L and len(transfers) == L - 1
        self.ctx, self.ops, self.transfers, self.smoothers = ops[0].ctx, ops, transfers, smoothers
        o = (_vp * L)(*[x.h for x in ops])
        t = (_vp * L)(*([None] + [x.h for x in transfers]))
        s = (_vp * L)(*[x.h for x in smoothers])
        self.h = _vp()
        _ck(lib().pmg_vcycle_create(o, t, s, C.c_int(L), C.c_int(pre), C.c_int(post), C.byref(self.h)))

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                lib().pmg_vcycle_destroy(self.h)
        except Exception:
            pass

    def vmult(self, dst, src):
        _ck(lib().pmg_vcycle_vmult(self.h, dst.h, src.h))

    def vmult_host(self, dst, src):
        _ck(lib().pmg_vcycle_vmult_host(self.h, _host_ptr(dst), _host_ptr(src)))

    def vmult_host_owned(self, dst, src):
        """Every rank passes its OWNED part of the vectors (host memory)."""
        _ck(lib().pmg_vcycle_vmult_host_owned(self.h, _host_ptr(dst), _host_ptr(src)))

    def set_graph(self, enable):
        _ck(lib().pmg_vcycle_set_graph(self.h, C.c_int(1 if enable else 0)))

    def profile(self, dst, src):
        L = len(self.ops)
        out = np.zeros(4 * L)
        _ck(lib().pmg_vcycle_profile(self.h, dst.h, src.h, _np_ptr(out), C.c_int(L)))
        return out.reshape(L, 4)


def cg_solve(A, x, b, precond=None, max_iterations=None, tolerance=None, rel_tol=1e-12):
    """SolverCG(SolverControl(max_it, tol)).solve(A, x, b, precond) (program.cc:345-352)."""
    if max_iterations is None:
        max_iterations = min(A.m(), 10000)
    if tolerance is None:
        tolerance = rel_tol * b.l2_norm()
    hist = np.zeros(max_iterations + 2)
    last = C.c_int()
    rc = lib().pmg_cg_solve(A.h, x.h, b.h, precond.h if precond is not None else None, C.c_int(max_iterations),
                            C.c_double(tolerance), C.byref(last), _np_ptr(hist), C.c_int(len(hist)))
    if rc not in (0, -6):
        _ck(rc)
    return last.value, hist[: last.value + 1].copy(), rc


def build_hierarchy(ctx, levels, pre=2, post=2, degree=5, smoothing_range=15.0, eig_cg_n_iterations=10,
                    coarse_range=1e-3, faces=PMG_ALL_FACES, coefficient=0, dim=3, vertices=None, mapping=None,
                    geometry_degree=None):
    """levels: list of (degree, n_cells) coarse -> fine; consecutive levels must be related by one
    global refinement (h) or a degree change on the same mesh (p).  Smoother parameters as in the
    reference drivers (program.cc:267-279).  coefficient = 1: every level discretises -div(a grad u) with
    a = 1/(0.05 + 2|x|^2) at its own quadrature points (BASELINE config 5).  vertices: the finest mesh's vertices
    (LaplaceOperator); a coarser mesh takes every 2^k-th vertex in each direction (nested meshes), p-levels share them.
    mapping: instead of vertices, a map of the unit cube (mesh_nodes); every level gets curved cells interpolating it,
    of the level's FE degree (MappingQ(p) on every level) or of geometry_degree when that is given."""
    if vertices is not None and mapping is not None:
        raise PmgError(-1, "vertices= and mapping= are mutually exclusive")

    def level_op(p, n):
        if mapping is not None:
            k = p if geometry_degree is None else geometry_degree
            return LaplaceOperator(ctx, p, n, faces, dim=dim, coefficient=coefficient, nodes=mesh_nodes(mapping, n, k),
                                   geometry_degree=k)
        return LaplaceOperator(ctx, p, n, faces, dim=dim, coefficient=coefficient,
                               vertices=None if vertices is None else mesh_vertices_coarsened(vertices, levels[-1][1], n))

    ops = [level_op(p, n) for (p, n) in levels]
    transfers = []
    for l in range(1, len(levels)):
        if levels[l][0] == levels[l - 1][0]:
            transfers.append(GeometricTransfer(ops[l - 1], ops[l]))
        else:
            transfers.append(PolynomialTransfer(ops[l - 1], ops[l]))
    smoothers = []
    for l, op in enumerate(ops):
        op.compute_diagonal()
        if l > 0:
            smoothers.append(Chebyshev(op, smoothing_range, degree, eig_cg_n_iterations))
        else:
            smoothers.append(Chebyshev(op, coarse_range, PMG_INVALID_DEGREE, min(op.m(), 2 ** 31 - 1)))
    mg = VCycleMultigrid(ops, transfers, smoothers, pre, post)
    return ops, transfers, smoothers, mg


# ---- host-only helpers (no GPU needed) -------------------------------------------------------
def mesh_vertices_coarsened(vertices, n_fine, n_coarse):
    """The vertices of the coarse mesh of a nested pair: vertex (i, j, k) of the coarse mesh is vertex (f i, f j, f k)
    of the fine one, f = n_fine / n_coarse per direction (a power of two)."""
    nf = (n_fine,) * 3 if isinstance(n_fine, int) else tuple(n_fine)
    nc = (n_coarse,) * 3 if isinstance(n_coarse, int) else tuple(n_coarse)
    v = np.asarray(vertices, dtype=np.float64).reshape(nf[2] + 1, nf[1] + 1, nf[0] + 1, 3)
    f = []
    for a, b in zip(nf, nc):
        if b < 1 or a % b or (a // b) & (a // b - 1):
            raise PmgError(-1, "mesh of %s cells is not a refinement of %s cells" % (nf, nc))
        f.append(a // b)
    return np.ascontiguousarray(v[:: f[2], :: f[1], :: f[0]])


def mesh_vertices_uniform(n, box=(1.0, 1.0, 1.0)):
    """Vertices of the box [0, box] cut into n equal cells per direction, shape (nz+1, ny+1, nx+1, 3)."""
    n = (n,) * 3 if isinstance(n, int) else tuple(n)
    z, y, x = np.meshgrid(*[np.arange(n[d] + 1) * (box[d] / n[d]) for d in (2, 1, 0)], indexing="ij")
    return np.ascontiguousarray(np.stack([x, y, z], axis=-1))


def _n_nodes(n, k):
    return (n[0] * k + 1) * (n[1] * k + 1) * (n[2] * k + 1)


def _geometry_degree_of(size, n):
    """the geometry degree k >= 1 with 3 (nx k+1)(ny k+1)(nz k+1) = size; PmgError(-1) when there is none"""
    k = 1
    while 3 * _n_nodes(n, k) < size:
        k += 1
    if 3 * _n_nodes(n, k) != size:
        raise PmgError(-1, "nodes: %d values fit no geometry degree for %d x %d x %d cells" % (size, *n))
    return k


def host_support_points(k):
    """the k + 1 Gauss-Lobatto points of [0, 1] the nodes of a curved cell of geometry degree k sit at"""
    x = np.zeros(k + 1)
    _ck(lib().pmg_host_support_points(C.c_int(k), _np_ptr(x)))
    return x


def mesh_nodes(mapping, n, k):
    """Geometry support points of a structured mesh of n cells (int or (nx, ny, nz)) on the image of the unit cube under
    mapping(X, Y, Z) -> array (..., 3): the map evaluated at the degree-k Gauss-Lobatto grid of every cell
    (host_support_points), shape (nz k+1, ny k+1, nx k+1, 3) -- the nodes= array of LaplaceOperator."""
    n = (n,) * 3 if isinstance(n, int) else tuple(n)
    s = host_support_points(k)
    t = [np.concatenate([(c + s[:-1]) / nd for c in range(nd)] + [[1.0]]) for nd in n]
    Z, Y, X = np.meshgrid(t[2], t[1], t[0], indexing="ij")
    out = np.ascontiguousarray(np.asarray(mapping(X, Y, Z), dtype=np.float64))
    if out.shape != X.shape + (3,):
        raise PmgError(-1, "mapping returned shape %s for points of shape %s, need (..., 3)" % (out.shape, X.shape))
    return out


def host_fastdiag_tables(p):
    n = p + 1
    S, lam = np.zeros(n * n), np.zeros(n)
    _ck(lib().pmg_host_fastdiag_tables(C.c_int(p), _np_ptr(S), _np_ptr(lam)))
    return S.reshape(n, n), lam


def host_pencil(p):
    n = p + 1
    M, K = np.zeros(n * n), np.zeros(n * n)
    _ck(lib().pmg_host_pencil(C.c_int(p), _np_ptr(M), _np_ptr(K)))
    return M.reshape(n, n), K.reshape(n, n)


def host_prolongation_1d(kind, pc, pf=None):
    nf = 2 * pc + 1 if kind == 0 else pf + 1
    P = np.zeros((pc + 1) * nf)
    _ck(lib().pmg_host_prolongation_1d(C.c_int(kind), C.c_int(pc), C.c_int(pf if pf else pc), _np_ptr(P)))
    return P.reshape(pc + 1, nf)


def host_partition(nz, n_ranks, rank):
    lo, hi = C.c_int(), C.c_int()
    rc = lib().pmg_host_partition(C.c_int(nz), C.c_int(n_ranks), C.c_int(rank), C.byref(lo), C.byref(hi))
    if rc < 0:
        _ck(rc)
    return lo.value, hi.value, rc == 0


def host_chebyshev_parameters(lmin, lmax_est, smoothing_range, degree):
    t, d, k = C.c_double(), C.c_double(), C.c_int()
    _ck(lib().pmg_host_chebyshev_parameters(C.c_double(lmin), C.c_double(lmax_est), C.c_double(smoothing_range),
                                            C.c_int(degree), C.byref(t), C.byref(d), C.byref(k)))
    return t.value, d.value, k.value


def host_tridiag_extreme_eigenvalues(diag, off):
    a, b = C.c_double(), C.c_double()
    diag = np.ascontiguousarray(diag, dtype=np.float64)
    off = np.ascontiguousarray(np.append(off, 0.0), dtype=np.float64)
    _ck(lib().pmg_host_tridiag_extreme_eigenvalues(C.c_int(len(diag)), _np_ptr(diag), _np_ptr(off), C.byref(a), C.byref(b)))
    return a.value, b.value
