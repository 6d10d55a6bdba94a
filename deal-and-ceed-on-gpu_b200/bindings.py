"""ctypes binding of the C ABI (include/bp5_b200.h) plus a thin Python mirror of the
reference's host classes for this path, so tests and bench.py read like the
reference driver (bp5/step-64.cu:341-561):

    PoissonOperator(dof_handler, constraints)   bp5/step-64.cu:199-224
        .vmult(dst, src) / .initialize_dof_vector(vec) / .do_zero_out
    LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>   [UPSTREAM]
    SolverCGFullMerge(control).solve(A, x, b, preconditioner)       bp5/solver.h:15-31
    SolverCG(control).solve(...)                                    bp5/step-64.cu:446-453
    IterationNumberControl / SolverControl                          bp5/step-64.cu:443 ; step-64/step-64.cu:513

No torch types cross the ABI.  There is no CPU fallback: if libbp5b200.so is
missing or no B200 is present every compute call raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BP5_LIB", os.path.join(_HERE, "libbp5b200.so"))   # BP5_LIB: tuning builds only

QUAD_GAUSS, QUAD_GLL = 0, 1
OP_POISSON, OP_HELMHOLTZ = 0, 1
GEOM_STORED, GEOM_ON_THE_FLY = 0, 1
CELL_ORDER_DEFAULT, CELL_ORDER_COLORED = 0, 1
CONTROL_ITERATION_NUMBER, CONTROL_SOLVER = 0, 1
CG_STANDARD, CG_MERGED = 0, 1
OK, ERR_INVALID, ERR_CUDA, ERR_NO_CONVERGENCE, ERR_DIVIDE_BY_ZERO, ERR_UNSUPPORTED = range(6)


class Problem(C.Structure):
    _fields_ = [
        ("degree", C.c_int32), ("quadrature", C.c_int32), ("operator_kind", C.c_int32), ("geometry_mode", C.c_int32),
        ("cells", C.c_int32 * 3), ("lower", C.c_double * 3), ("upper", C.c_double * 3),
        ("deformation", C.c_int32), ("deformation_eps", C.c_double),
        ("part_grid", C.c_int32 * 3), ("part_coord", C.c_int32 * 3), ("cell_order", C.c_int32), ("refine_lo", C.c_int32 * 3), ("refine_hi", C.c_int32 * 3),
        ("reserved", C.c_int32 * 1),
    ]


class PeerInfo(C.Structure):
    """bp5_peer_info_t: what a rank publishes for the peer-memory transport."""
    _fields_ = [("buf_handle", C.c_ubyte * 64), ("dvec_handle", C.c_ubyte * 64),
                ("n_owned", C.c_int64), ("n_ghost", C.c_int64), ("n_send", C.c_int64),
                ("ghost_offset", C.c_int64 * 8), ("send_offset", C.c_int64 * 8),
                ("rank", C.c_int32), ("device", C.c_int32)]


class MgParams(C.Structure):
    """bp5_mg_params_t: zero selects the default."""
    _fields_ = [("max_levels", C.c_int32), ("smoothing_degree", C.c_int32), ("smoothing_range", C.c_double),
                ("eig_iterations", C.c_int32), ("coarse_max_its", C.c_int32), ("coarse_tol", C.c_double),
                ("reserved", C.c_int32 * 4)]


class Bp5Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bp5 error {code}: {msg}")
        self.code = code


class NoConvergence(Bp5Error):
    """SolverControl::NoConvergence (bp5/solver.h:540)."""


_dp = C.POINTER(C.c_double)
_vp = C.c_void_p
_lib = None

# every symbol include/bp5_b200.h declares: (name, restype, argtypes)
ABI = [
    ("bp5_context_create", C.c_int, [C.c_int, C.POINTER(_vp)]),
    ("bp5_context_destroy", C.c_int, [_vp]),
    ("bp5_context_synchronize", C.c_int, [_vp]),
    ("bp5_context_stream", _vp, [_vp]),
    ("bp5_last_error", C.c_char_p, []),
    ("bp5_version", C.c_char_p, []),
    ("bp5_operator_create", C.c_int, [_vp, C.POINTER(Problem), C.POINTER(_vp)]),
    ("bp5_operator_destroy", C.c_int, [_vp]),
    ("bp5_operator_sizes", C.c_int, [_vp] + [C.POINTER(C.c_int64)] * 4),
    ("bp5_operator_initialize_dof_vector", C.c_int, [_vp, C.POINTER(_vp)]),
    ("bp5_operator_set_zero_out", C.c_int, [_vp, C.c_int]),
    ("bp5_operator_vmult", C.c_int, [_vp, _vp, _vp]),
    ("bp5_operator_cell_loop", C.c_int, [_vp, _vp, _vp]),
    ("bp5_operator_copy_constrained_values", C.c_int, [_vp, _vp, _vp]),
    ("bp5_operator_vmult_ptr", C.c_int, [_vp, _vp, _vp, C.c_int]),
    ("bp5_operator_assemble_rhs", C.c_int, [_vp, _vp]),
    ("bp5_operator_export_coefficients", C.c_int, [_vp, _dp]),
    ("bp5_operator_export_dof_coordinates", C.c_int, [_vp, _dp]),
    ("bp5_operator_export_global_indices", C.c_int, [_vp, C.POINTER(C.c_int64)]),
    ("bp5_operator_l2_norm_sqr", C.c_int, [_vp, _vp, _dp]),
    ("bp5_operator_compute_diagonal", C.c_int, [_vp, _vp, C.c_int]),
    ("bp5_operator_algorithmic_bytes", C.c_int, [_vp, _dp, _dp]),
    ("bp5_operator_profile", C.c_int, [_vp, C.c_int]),
    ("bp5_operator_profile_result", C.c_int, [_vp, C.POINTER(C.c_int64), _dp]),
    ("bp5_operator_kernel_name", C.c_char_p, [_vp]),
    ("bp5_context_launch_count", C.c_int64, [_vp]),
    ("bp5_vector_create", C.c_int, [_vp, C.c_int64, C.c_int64, C.POINTER(_vp)]),
    ("bp5_vector_create_like", C.c_int, [_vp, C.POINTER(_vp)]),
    ("bp5_vector_owner", _vp, [_vp]),
    ("bp5_vector_destroy", C.c_int, [_vp]),
    ("bp5_vector_local_size", C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("bp5_vector_get_values", _vp, [_vp]),
    ("bp5_vector_set", C.c_int, [_vp, C.c_double]),
    ("bp5_vector_import_host", C.c_int, [_vp, _vp, C.c_int64]),
    ("bp5_vector_export_host", C.c_int, [_vp, _vp, C.c_int64]),
    ("bp5_vector_copy", C.c_int, [_vp, _vp]),
    ("bp5_vector_add", C.c_int, [_vp, C.c_double, _vp]),
    ("bp5_vector_equ", C.c_int, [_vp, C.c_double, _vp]),
    ("bp5_vector_sadd", C.c_int, [_vp, C.c_double, C.c_double, _vp]),
    ("bp5_vector_scale", C.c_int, [_vp, _vp]),
    ("bp5_vector_dot_local", C.c_int, [_vp, _vp, _dp]),
    ("bp5_vector_norm_sqr_local", C.c_int, [_vp, _dp]),
    ("bp5_vector_all_zero_local", C.c_int, [_vp, C.POINTER(C.c_int)]),
    ("bp5_vector_zero_out_ghosts", C.c_int, [_vp]),
    ("bp5_cg_solve", C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_int), _dp,
                               _dp, C.c_int]),
    ("bp5_cg_solve_host", C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int,
                                    C.POINTER(C.c_int), _dp]),
    ("bp5_operator_matrix_free_data", C.c_int, [_vp, _vp]),
    ("bp5_operator_matrix_free_data_colored", C.c_int, [_vp, C.c_int, _vp]),
    ("bp5_operator_halo_info", C.c_int, [_vp] + [C.POINTER(C.c_int64)] * 4),
    ("bp5_operator_halo_pack", C.c_int, [_vp, _vp, _vp]),
    ("bp5_operator_halo_unpack_add", C.c_int, [_vp, _vp, _vp]),
    ("bp5_cg_step_begin", C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int]),
    ("bp5_cg_step_vectors", C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    ("bp5_cg_step_update", C.c_int, [_vp, C.c_int]),
    ("bp5_cg_step_apply_local", C.c_int, [_vp]),
    ("bp5_cg_step_constrained", C.c_int, [_vp]),
    ("bp5_cg_step_local_dots", C.c_int, [_vp, _vp]),
    ("bp5_cg_step_scalars", C.c_int, [_vp, _vp]),
    ("bp5_cg_step_poll", C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), _dp]),
    ("bp5_cg_step_finish", C.c_int, [_vp, _dp]),
    ("bp5_peer_export", C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(PeerInfo)]),
    ("bp5_peer_connect", C.c_int, [_vp, C.POINTER(PeerInfo), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("bp5_peer_vmult", C.c_int, [_vp, _vp, _vp]),
    ("bp5_peer_cg_solve", C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_int), _dp, _dp,
                                    C.c_int]),
    ("bp5_peer_allreduce", C.c_int, [_vp, _dp, C.c_int]),
    ("bp5_peer_world_size", C.c_int, [_vp]),
    ("bp5_vector_update_ghost_values", C.c_int, [_vp, _vp]),
    ("bp5_vector_compress_add", C.c_int, [_vp, _vp]),
    ("bp5_peer_cg_solve_host", C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int,
                                         C.POINTER(C.c_int), _dp]),
    ("bp5_mg_create", C.c_int, [_vp, C.POINTER(MgParams), C.POINTER(_vp)]),
    ("bp5_mg_destroy", C.c_int, [_vp]),
    ("bp5_mg_n_levels", C.c_int, [_vp, C.POINTER(C.c_int)]),
    ("bp5_mg_level_operator", C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
    ("bp5_mg_get_lambda_max", C.c_int, [_vp, C.c_int, _dp]),
    ("bp5_mg_set_lambda_max", C.c_int, [_vp, C.c_int, C.c_double]),
    ("bp5_mg_prolongate", C.c_int, [_vp, C.c_int, _vp, _vp]),
    ("bp5_mg_restrict", C.c_int, [_vp, C.c_int, _vp, _vp]),
    ("bp5_mg_smooth", C.c_int, [_vp, C.c_int, _vp, _vp]),
    ("bp5_mg_vcycle", C.c_int, [_vp, _vp, _vp]),
    ("bp5_mg_cg_solve", C.c_int, [_vp, _vp, _vp, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_int), _dp, _dp,
                                  C.c_int]),
    ("bp5_mg_profile", C.c_int, [_vp, C.c_int]),
    ("bp5_mg_profile_result", C.c_int, [_vp, _dp, C.POINTER(C.c_int64)]),
]


def lib():
    """Load libbp5b200.so.  Fails loudly when the CUDA extension is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, res, args in ABI:
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def _check(rc):
    if rc == OK:
        return
    msg = lib().bp5_last_error().decode()
    if rc == ERR_NO_CONVERGENCE:
        raise NoConvergence(rc, msg)
    raise Bp5Error(rc, msg)


class Context:
    def __init__(self, device=0):
        self.h = _vp()
        _check(lib().bp5_context_create(int(device), C.byref(self.h)))
        self.device = device

    def synchronize(self):
        _check(lib().bp5_context_synchronize(self.h))

    @property
    def stream(self):
        return lib().bp5_context_stream(self.h)

    @property
    def launch_count(self):
        return lib().bp5_context_launch_count(self.h)

    def close(self):
        if self.h:
            lib().bp5_context_destroy(self.h)
            self.h = _vp()


class Vector:
    """LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>: [owned | ghost] on the device."""

    def __init__(self, ctx, n_owned=None, n_ghost=0, handle=None):
        self.ctx = ctx
        self.h = _vp()
        if handle is not None:
            self.h = handle
        else:
            _check(lib().bp5_vector_create(ctx.h, int(n_owned), int(n_ghost), C.byref(self.h)))
        a, b = C.c_int64(), C.c_int64()
        _check(lib().bp5_vector_local_size(self.h, C.byref(a), C.byref(b)))
        self.n_owned, self.n_ghost = a.value, b.value

    def reinit_like(self):
        h = _vp()
        _check(lib().bp5_vector_create_like(self.h, C.byref(h)))
        return Vector(self.ctx, handle=h)

    def local_size(self):
        return self.n_owned

    def get_values(self):
        return lib().bp5_vector_get_values(self.h)

    def set(self, value):
        _check(lib().bp5_vector_set(self.h, float(value)))

    def import_host(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float64)
        _check(lib().bp5_vector_import_host(self.h, arr.ctypes.data, arr.size))

    def to_host(self, with_ghosts=False):
        n = self.n_owned + (self.n_ghost if with_ghosts else 0)
        out = np.empty(n)
        _check(lib().bp5_vector_export_host(self.h, out.ctypes.data, n))
        return out

    def add(self, a, x):
        _check(lib().bp5_vector_add(self.h, float(a), x.h))

    def equ(self, a, x):
        _check(lib().bp5_vector_equ(self.h, float(a), x.h))

    def sadd(self, s, a, x):
        _check(lib().bp5_vector_sadd(self.h, float(s), float(a), x.h))

    def dot_local(self, other):
        out = C.c_double()
        _check(lib().bp5_vector_dot_local(self.h, other.h, C.byref(out)))
        return out.value

    def l2_norm(self):
        out = C.c_double()
        _check(lib().bp5_vector_norm_sqr_local(self.h, C.byref(out)))
        return float(np.sqrt(out.value))

    def all_zero(self):
        out = C.c_int()
        _check(lib().bp5_vector_all_zero_local(self.h, C.byref(out)))
        return bool(out.value)

    def zero_out_ghosts(self):
        _check(lib().bp5_vector_zero_out_ghosts(self.h))

    def close(self):
        if self.h:
            lib().bp5_vector_destroy(self.h)
            self.h = _vp()


def make_problem(degree, cells, quadrature=QUAD_GAUSS, operator_kind=OP_POISSON, lower=(0., 0., 0.), upper=None,
                 deformation=0, eps=0.0, part_grid=(1, 1, 1), part_coord=(0, 0, 0), geometry_mode=GEOM_STORED,
                 cell_order=CELL_ORDER_DEFAULT, refine_lo=(0, 0, 0), refine_hi=(0, 0, 0)):
    """refine_lo / refine_hi: the coarse cells with indices in [lo, hi) are replaced by their eight children (hanging
    nodes on the box's faces); all zero: conforming mesh"""
    p = Problem()
    p.degree, p.quadrature, p.operator_kind, p.geometry_mode = degree, quadrature, operator_kind, geometry_mode
    if upper is None:
        upper = tuple(float(c) for c in cells)   # unit cells
    for d in range(3):
        p.cells[d] = int(cells[d]); p.lower[d] = float(lower[d]); p.upper[d] = float(upper[d])
        p.part_grid[d] = int(part_grid[d]); p.part_coord[d] = int(part_coord[d])
    p.deformation, p.deformation_eps = int(deformation), float(eps)
    p.cell_order = int(cell_order)
    for d in range(3):
        p.refine_lo[d] = int(refine_lo[d]); p.refine_hi[d] = int(refine_hi[d])
    return p


class PoissonOperator:
    """BP5::PoissonOperator / Step64::HelmholtzOperator over the C ABI."""

    def __init__(self, ctx, problem):
        self.ctx = ctx
        self.problem = problem
        self.h = _vp()
        _check(lib().bp5_operator_create(ctx.h, C.byref(problem), C.byref(self.h)))
        s = [C.c_int64() for _ in range(4)]
        _check(lib().bp5_operator_sizes(self.h, *[C.byref(v) for v in s]))
        self.n_owned, self.n_ghost, self.n_global, self.n_cells = [v.value for v in s]
        self._zero = True

    @property
    def do_zero_out(self):
        return self._zero

    @do_zero_out.setter
    def do_zero_out(self, v):
        self._zero = bool(v)
        _check(lib().bp5_operator_set_zero_out(self.h, int(self._zero)))

    def initialize_dof_vector(self):
        h = _vp()
        _check(lib().bp5_operator_initialize_dof_vector(self.h, C.byref(h)))
        return Vector(self.ctx, handle=h)

    def vmult(self, dst, src):
        _check(lib().bp5_operator_vmult(self.h, dst.h, src.h))

    def cell_loop(self, dst, src):
        _check(lib().bp5_operator_cell_loop(self.h, dst.h, src.h))

    def copy_constrained_values(self, dst, src):
        _check(lib().bp5_operator_copy_constrained_values(self.h, dst.h, src.h))

    def vmult_ptr(self, dst_ptr, src_ptr, zero_dst=True):
        _check(lib().bp5_operator_vmult_ptr(self.h, dst_ptr, src_ptr, int(zero_dst)))

    def assemble_rhs(self, b):
        _check(lib().bp5_operator_assemble_rhs(self.h, b.h))

    def compute_diagonal(self, diag, invert=False):
        """diagonal of the operator (or its reciprocal): Jacobi preconditioner for the DiagonalMatrix slot"""
        _check(lib().bp5_operator_compute_diagonal(self.h, diag.h, int(invert)))

    def l2_norm(self, u):
        """||u||_L2 of the finite element function with QGauss(p+2) (output_results, bp5/step-64.cu:604-615)."""
        out = C.c_double()
        _check(lib().bp5_operator_l2_norm_sqr(self.h, u.h, C.byref(out)))
        return float(np.sqrt(out.value))

    def coefficients(self):
        n3 = (self.problem.degree + 1) ** 3
        out = np.empty((6, self.n_cells, n3))
        _check(lib().bp5_operator_export_coefficients(self.h, out.ctypes.data_as(_dp)))
        return out

    def dof_coordinates(self):
        out = np.empty((self.n_owned + self.n_ghost, 3))
        _check(lib().bp5_operator_export_dof_coordinates(self.h, out.ctypes.data_as(_dp)))
        return out

    def global_indices(self):
        out = np.empty(self.n_owned + self.n_ghost, dtype=np.int64)
        _check(lib().bp5_operator_export_global_indices(self.h, out.ctypes.data_as(C.POINTER(C.c_int64))))
        return out

    def algorithmic_bytes(self):
        a, b = C.c_double(), C.c_double()
        _check(lib().bp5_operator_algorithmic_bytes(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def profile(self, enable=True):
        _check(lib().bp5_operator_profile(self.h, int(enable)))

    def profile_result(self):
        n, ms = C.c_int64(), C.c_double()
        _check(lib().bp5_operator_profile_result(self.h, C.byref(n), C.byref(ms)))
        return n.value, ms.value

    @property
    def kernel_name(self):
        return lib().bp5_operator_kernel_name(self.h).decode()

    def close(self):
        if self.h:
            lib().bp5_operator_destroy(self.h)
            self.h = _vp()


class _LevelOperator(PoissonOperator):
    """A multigrid level's operator: owned by the Multigrid object (close() does not destroy it)."""

    def __init__(self, ctx, handle, problem):
        self.ctx, self.problem, self.h = ctx, problem, handle
        s = [C.c_int64() for _ in range(4)]
        _check(lib().bp5_operator_sizes(self.h, *[C.byref(v) for v in s]))
        self.n_owned, self.n_ghost, self.n_global, self.n_cells = [v.value for v in s]
        self._zero = True

    def close(self):
        self.h = _vp()


class Multigrid:
    """Geometric multigrid V-cycle (Chebyshev-Jacobi smoothing, CG on the coarsest level) on the levels of `op`'s
    mesh: PreconditionMG with MGTransferMatrixFree, PreconditionChebyshev and MGCoarseGridIterativeSolver.
    One block, conforming mesh, stored geometry, default cell order.  `op` must outlive this object.

    params (0 or None: default): max_levels, smoothing_degree (5), smoothing_range (15), eig_iterations (12),
    coarse_tol (1e-6, relative), coarse_max_its (1000)."""

    _INT = ("max_levels", "smoothing_degree", "eig_iterations", "coarse_max_its")
    _FLOAT = ("smoothing_range", "coarse_tol")

    def __init__(self, op, **params):
        unknown = set(params) - set(self._INT) - set(self._FLOAT)
        if unknown:
            raise TypeError(f"unknown multigrid parameter(s): {sorted(unknown)}")
        prm = MgParams()
        for k, v in params.items():
            if v is None:
                continue
            if k in self._INT:
                if int(v) != v or v < 0:
                    raise ValueError(f"{k} must be a non-negative integer (0: default), got {v!r}")
                setattr(prm, k, int(v))
            else:
                if not np.isfinite(v) or v < 0:
                    raise ValueError(f"{k} must be a non-negative number (0: default), got {v!r}")
                setattr(prm, k, float(v))
        if prm.smoothing_range != 0.0 and prm.smoothing_range <= 1.0:
            raise ValueError("smoothing_range must exceed 1")
        if not isinstance(op, PoissonOperator):
            raise TypeError("Multigrid needs a PoissonOperator")
        self.op, self.ctx = op, op.ctx
        self.h = _vp()
        _check(lib().bp5_mg_create(op.h, C.byref(prm), C.byref(self.h)))
        n = C.c_int()
        _check(lib().bp5_mg_n_levels(self.h, C.byref(n)))
        self.n_levels = n.value
        self._levels = {}

    def level_operator(self, level):
        """the operator of `level` (n_levels - 1 is the caller's)"""
        if level == self.n_levels - 1:
            return self.op
        if level not in self._levels:
            h = _vp()
            _check(lib().bp5_mg_level_operator(self.h, int(level), C.byref(h)))
            prob = Problem.from_buffer_copy(self.op.problem)
            c = self.op.problem.cells
            f = 2 ** (self.n_levels - 1 - level)
            for d in range(3):
                prob.cells[d] = c[d] // f
            self._levels[level] = _LevelOperator(self.ctx, h, prob)
        return self._levels[level]

    def lambda_max(self, level):
        """estimate of the largest eigenvalue of D^-1 A on `level` >= 1 (the smoother uses 1.2 times it)"""
        out = C.c_double()
        _check(lib().bp5_mg_get_lambda_max(self.h, int(level), C.byref(out)))
        return out.value

    def set_lambda_max(self, level, value):
        _check(lib().bp5_mg_set_lambda_max(self.h, int(level), float(value)))

    def prolongate(self, fine_level, dst, src):
        """dst (level fine_level) = P src (level fine_level - 1)"""
        _check(lib().bp5_mg_prolongate(self.h, int(fine_level), dst.h, src.h))

    def restrict(self, fine_level, dst, src):
        """dst (level fine_level - 1) = P^T src, Dirichlet rows zero"""
        _check(lib().bp5_mg_restrict(self.h, int(fine_level), dst.h, src.h))

    def smooth(self, level, x, b):
        """Chebyshev smoothing of A x = b on `level` >= 1 from the x given"""
        _check(lib().bp5_mg_smooth(self.h, int(level), x.h, b.h))

    def vmult(self, dst, src):
        """dst = V-cycle(src)"""
        _check(lib().bp5_mg_vcycle(self.h, dst.h, src.h))

    def profile(self, enable=True):
        _check(lib().bp5_mg_profile(self.h, int(enable)))

    def profile_result(self):
        """({level: {"operator", "transfer", "vector", "coarse"} ms}, V-cycles) since the last call"""
        ms = np.zeros(4 * self.n_levels)
        n = C.c_int64()
        _check(lib().bp5_mg_profile_result(self.h, ms.ctypes.data_as(_dp), C.byref(n)))
        keys = ("operator", "transfer", "vector", "coarse")
        return {l: dict(zip(keys, ms[4 * l: 4 * l + 4].tolist())) for l in range(self.n_levels)}, n.value

    def close(self):
        for L in self._levels.values():
            L.close()
        self._levels = {}
        if self.h:
            lib().bp5_mg_destroy(self.h)
            self.h = _vp()


class SolverControl:
    """SolverControl(max_its, tol): failure at max_its (step-64/step-64.cu:513)."""
    kind = CONTROL_SOLVER

    def __init__(self, max_its, tol):
        self.max_its, self.tol = int(max_its), float(tol)
        self._last_step, self._last_value = 0, float("nan")
        self.history = None

    def last_step(self):
        return self._last_step

    def last_value(self):
        return self._last_value


class IterationNumberControl(SolverControl):
    """IterationNumberControl(max_its, tol): success at tol OR at max_its (bp5/step-64.cu:443)."""
    kind = CONTROL_ITERATION_NUMBER


class _SolverBase:
    variant = CG_MERGED

    def __init__(self, control):
        self.control = control

    def solve(self, A, x, b, preconditioner=None, history=True):
        c = self.control
        its, val = C.c_int(0), C.c_double(0.0)
        hist = np.full(c.max_its + 2, np.nan) if history else None
        if isinstance(preconditioner, Multigrid):
            if self.variant != CG_STANDARD:
                raise Bp5Error(ERR_UNSUPPORTED, "a multigrid preconditioner needs the standard CG (SolverCG); "
                                                "the merged variant takes a diagonal only")
            if A is not preconditioner.op:
                raise ValueError("the multigrid preconditioner was built on a different operator")
            rc = lib().bp5_mg_cg_solve(preconditioner.h, x.h, b.h, c.kind, c.tol, c.max_its, C.byref(its),
                                       C.byref(val), hist.ctypes.data_as(_dp) if hist is not None else None,
                                       len(hist) if hist is not None else 0)
            c._last_step, c._last_value = its.value, val.value
            c.history = hist[: its.value + 1] if hist is not None else None
            _check(rc)
            return
        rc = lib().bp5_cg_solve(A.h, x.h, b.h, preconditioner.h if preconditioner is not None else None,
                                self.variant, c.kind, c.tol, c.max_its, C.byref(its), C.byref(val),
                                hist.ctypes.data_as(_dp) if hist is not None else None,
                                len(hist) if hist is not None else 0)
        c._last_step, c._last_value = its.value, val.value
        c.history = hist[: its.value + 1] if hist is not None else None
        _check(rc)


class SolverCGFullMerge(_SolverBase):
    """SolverCGFullMerge<VectorType> (bp5/solver.h:15-31)."""
    variant = CG_MERGED


class SolverCG(_SolverBase):
    """dealii::SolverCG as used for "pcg-standard" (bp5/step-64.cu:446-453)."""
    variant = CG_STANDARD


def cg_solve_host(A, x_host, b_host, control, variant=CG_MERGED, x0_is_zero=False):
    """End-to-end entry point with HOST buffers (copies inside).  x0_is_zero: zero initial guess, x_host output only."""
    its, val = C.c_int(0), C.c_double(0.0)
    rc = lib().bp5_cg_solve_host(A.h, x_host.ctypes.data, b_host.ctypes.data, x_host.size, int(x0_is_zero), variant,
                                 control.kind,
                                 control.tol, control.max_its, C.byref(its), C.byref(val))
    control._last_step, control._last_value = its.value, val.value
    _check(rc)
