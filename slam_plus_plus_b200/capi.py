"""ctypes binding of libspp_b200.so (include/spp_b200.h). Plumbing only: every numeric step runs in the library.

The library is built in-tree by ``__graft_entry__.build()`` (``make -C slam_plus_plus_b200/csrc``). There is no
CPU fallback: loading fails loudly when the shared object is missing, and ``Context()`` raises when no sm_100
device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libspp_b200.so")

SPP_OK, SPP_NOT_POSDEF = 0, 1
SPP_ERR_INVALID, SPP_ERR_CUDA, SPP_ERR_NOMEM, SPP_ERR_COMM = -1, -2, -3, -4
JAC_FD_REFERENCE, JAC_ANALYTIC = 0, 1
LOSS_NONE, LOSS_HUBER, LOSS_CAUCHY = 0, 1, 2
RCS_AUTO, RCS_DENSE, RCS_SPARSE = 0, 1, 2
MAX_TRACE = 64

# every symbol include/spp_b200.h declares (tests check that the library exports all of them)
EXPORTED_SYMBOLS = [
    "spp_create", "spp_destroy", "spp_last_error", "spp_describe", "spp_kernel_launches", "spp_stream",
    "spp_synchronize", "spp_set_allreduce", "spp_partition_landmarks", "spp_rcs_block_pattern", "spp_ba_get_partition", "spp_ba_set_graph", "spp_ba_append_graph", "spp_ba_set_states", "spp_ba_get_states", "spp_ba_gather_states",
    "spp_ba_restore_initial", "spp_ba_set_jacobian_mode", "spp_ba_set_robust_loss", "spp_ba_get_observation_errors", "spp_ba_linearise", "spp_ba_get_lambda", "spp_ba_get_blocks", "spp_ba_chi2", "spp_ba_solve_step",
    "spp_ba_optimize", "spp_ba_marginals", "spp_schur_symbolic", "spp_schur_solve", "spp_schur_marginals",
    "spp_ba_marginals_sparse", "spp_schur_marginals_sparse", "spp_ba_covariance_blocks", "spp_schur_covariance_pattern", "spp_ba_joint_marginals", "spp_schur_joint_marginals",
    "spp_schur_get_reduced_system",
    "spp_schur_set_rcs_solver", "spp_schur_set_rcs_ordering", "spp_schur_get_rcs_info", "spp_schur_get_rcs_owners", "spp_schur_get_rcs_residual", "spp_block_ordering",
    "spp_block_symbolic_stats", "spp_block_subtree_owners", "spp_dense_posdef_solve", "spp_dense_panel_factor", "spp_nccl_get_unique_id", "spp_set_nccl",
    "spp_chol_symbolic", "spp_chol_solve", "spp_chol_get_factor",
    "spp_pose_set_graph", "spp_pose_set_ordering", "spp_pose_set_states", "spp_pose_get_states", "spp_pose_restore_initial",
    "spp_pose_linearise", "spp_pose_get_lambda", "spp_pose_chi2", "spp_pose_solve_step", "spp_pose_optimize",
    "spp_pose_marginals",
]


class Report(C.Structure):
    _fields_ = [
        ("n_iterations", C.c_int32), ("n_accepted", C.c_int32), ("n_rejected", C.c_int32), ("status", C.c_int32),
        ("chi2_initial", C.c_double), ("chi2_final", C.c_double), ("alpha_initial", C.c_double),
        ("alpha_final", C.c_double), ("last_dx_norm", C.c_double),
        ("trace_alpha", C.c_double * MAX_TRACE), ("trace_chi2", C.c_double * MAX_TRACE),
        ("trace_dx_norm", C.c_double * MAX_TRACE), ("trace_accepted", C.c_uint8 * MAX_TRACE),
        ("ms_linearise", C.c_double), ("ms_schur", C.c_double), ("ms_factor", C.c_double),
        ("ms_backsubst", C.c_double), ("ms_update", C.c_double), ("ms_chi2", C.c_double), ("ms_total", C.c_double),
        ("ms_factor_kernel", C.c_double),
    ]

    def as_dict(self) -> dict:
        n = min(self.n_iterations, MAX_TRACE)
        return dict(
            n_iterations=self.n_iterations, n_accepted=self.n_accepted, n_rejected=self.n_rejected,
            status=self.status, chi2_initial=self.chi2_initial, chi2_final=self.chi2_final,
            alpha_initial=self.alpha_initial, alpha_final=self.alpha_final, last_dx_norm=self.last_dx_norm,
            trace_alpha=list(self.trace_alpha[:n]), trace_chi2=list(self.trace_chi2[:n]),
            trace_dx_norm=list(self.trace_dx_norm[:n]), trace_accepted=[int(x) for x in self.trace_accepted[:n]],
            ms=dict(linearise=self.ms_linearise, schur=self.ms_schur, factor=self.ms_factor,
                    backsubst=self.ms_backsubst, update=self.ms_update, chi2=self.ms_chi2, total=self.ms_total,
                    factor_kernel=self.ms_factor_kernel))


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)

_lib = None


def load_library() -> C.CDLL:
    """Loads libspp_b200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() (make -C slam_plus_plus_b200/csrc). "
                           "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, dp, u64p, u8p = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)
    lib.spp_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.spp_destroy.argtypes = [vp]
    lib.spp_destroy.restype = None
    lib.spp_last_error.argtypes = [vp]
    lib.spp_last_error.restype = C.c_char_p
    lib.spp_describe.argtypes = [vp, C.c_char_p, C.c_size_t]
    lib.spp_kernel_launches.argtypes = [vp]
    lib.spp_kernel_launches.restype = C.c_uint64
    lib.spp_stream.argtypes = [vp]
    lib.spp_stream.restype = vp
    lib.spp_synchronize.argtypes = [vp]
    lib.spp_set_allreduce.argtypes = [vp, ALLREDUCE_FN, vp, C.c_int, C.c_int]
    lib.spp_partition_landmarks.argtypes = [C.c_size_t, C.POINTER(C.c_uint32), C.c_int, u64p]
    lib.spp_rcs_block_pattern.argtypes = [C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), u64p,
                                          C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.spp_ba_get_partition.argtypes = [vp, u64p, u64p]
    lib.spp_ba_set_graph.argtypes = [vp, C.c_size_t, u8p, dp, dp, C.c_size_t, u64p, u64p, dp, dp]
    lib.spp_ba_gather_states.argtypes = [vp, dp, dp]
    lib.spp_ba_append_graph.argtypes = [vp, C.c_size_t, u8p, dp, dp, C.c_size_t, u64p, u64p, dp, dp]
    lib.spp_ba_set_states.argtypes = [vp, dp, dp]
    lib.spp_ba_get_states.argtypes = [vp, dp, dp]
    lib.spp_ba_restore_initial.argtypes = [vp]
    lib.spp_ba_set_jacobian_mode.argtypes = [vp, C.c_int]
    lib.spp_ba_set_robust_loss.argtypes = [vp, C.c_int, C.c_double]
    lib.spp_ba_get_observation_errors.argtypes = [vp, dp, dp]
    lib.spp_ba_linearise.argtypes = [vp]
    lib.spp_ba_get_lambda.argtypes = [vp, u64p, u64p, u64p, u64p, u64p, u64p, dp, dp]
    lib.spp_ba_get_blocks.argtypes = [vp, dp, dp, dp, dp, dp]
    lib.spp_ba_chi2.argtypes = [vp, dp]
    lib.spp_ba_solve_step.argtypes = [vp, C.c_double, dp]
    lib.spp_ba_optimize.argtypes = [vp, C.c_size_t, C.c_double, C.POINTER(Report)]
    lib.spp_schur_symbolic.argtypes = [vp, C.c_size_t, u64p, u64p, u64p, u64p, u64p]
    lib.spp_schur_solve.argtypes = [vp, dp, dp]
    lib.spp_ba_marginals.argtypes = [vp, C.c_double, dp, dp]
    lib.spp_schur_marginals.argtypes = [vp, C.c_double, dp, dp]
    lib.spp_ba_marginals_sparse.argtypes = [vp, C.c_double, dp, dp]
    lib.spp_schur_marginals_sparse.argtypes = [vp, C.c_double, dp, dp]
    lib.spp_ba_covariance_blocks.argtypes = [vp, C.c_double, C.c_size_t, u64p, u64p, dp, C.c_size_t, u64p, dp, dp, dp]
    lib.spp_schur_covariance_pattern.argtypes = [vp, C.c_double, dp]
    lib.spp_ba_joint_marginals.argtypes = [vp, C.c_double, C.c_size_t, u64p, u64p, dp]
    lib.spp_schur_joint_marginals.argtypes = [vp, C.c_double, C.c_size_t, u64p, u64p, dp]
    lib.spp_schur_get_reduced_system.argtypes = [vp, u64p, dp, dp, u8p]
    lib.spp_dense_posdef_solve.argtypes = [vp, C.c_size_t, dp, dp]
    lib.spp_dense_panel_factor.argtypes = [vp, C.c_size_t, C.c_size_t, dp]
    lib.spp_nccl_get_unique_id.argtypes = [C.c_void_p]
    lib.spp_set_nccl.argtypes = [vp, C.c_void_p, C.c_int, C.c_int]
    lib.spp_schur_set_rcs_solver.argtypes = [vp, C.c_int]
    lib.spp_schur_get_rcs_owners.argtypes = [vp, C.POINTER(C.c_int32)]
    lib.spp_block_subtree_owners.argtypes = [C.c_size_t, u64p, u64p, u64p, C.c_int, C.c_double, C.POINTER(C.c_int32), dp]
    lib.spp_schur_set_rcs_ordering.argtypes = [vp, C.c_size_t, u64p]
    lib.spp_schur_get_rcs_info.argtypes = [vp, u64p, dp]
    lib.spp_schur_get_rcs_residual.argtypes = [vp, dp]
    lib.spp_block_ordering.argtypes = [C.c_size_t, u64p, u64p, u64p]
    lib.spp_block_symbolic_stats.argtypes = [C.c_size_t, u64p, u64p, u64p, u64p, u64p, dp]
    lib.spp_chol_symbolic.argtypes = [vp, C.c_size_t, C.c_size_t, u64p, u64p, u64p, u64p]
    lib.spp_chol_solve.argtypes = [vp, dp, dp]
    lib.spp_chol_get_factor.argtypes = [vp, u64p, u64p, u64p, dp]
    lib.spp_pose_set_graph.argtypes = [vp, C.c_int, C.c_size_t, dp, C.c_size_t, u64p, u64p, dp, dp]
    lib.spp_pose_set_ordering.argtypes = [vp, u64p]
    lib.spp_pose_set_states.argtypes = [vp, dp]
    lib.spp_pose_get_states.argtypes = [vp, dp]
    lib.spp_pose_restore_initial.argtypes = [vp]
    lib.spp_pose_linearise.argtypes = [vp]
    lib.spp_pose_get_lambda.argtypes = [vp, u64p, u64p, u64p, u64p, dp, dp]
    lib.spp_pose_chi2.argtypes = [vp, dp]
    lib.spp_pose_solve_step.argtypes = [vp, dp]
    lib.spp_pose_marginals.argtypes = [vp, dp]
    lib.spp_pose_optimize.argtypes = [vp, C.c_size_t, C.c_double, C.POINTER(Report)]
    _lib = lib
    return lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _u64p(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_uint64))


def _u8p(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_uint8))


def partition_landmarks(track_length, world: int) -> np.ndarray:
    """Landmark slice boundaries of the multi-GPU path (pure host code in the library, no GPU needed)."""
    tl = np.ascontiguousarray(track_length, np.uint32)
    bounds = np.zeros(world + 1, np.uint64)
    rc = load_library().spp_partition_landmarks(tl.shape[0], tl.ctypes.data_as(C.POINTER(C.c_uint32)), world, _u64p(bounds))
    if rc != SPP_OK:
        raise ValueError("spp_partition_landmarks: invalid arguments")
    return bounds.astype(np.int64)


def rcs_block_pattern(n_cameras: int, n_points: int, obs_camera, obs_point):
    """Pure host helper: (rows, cols) of the upper blocks of the reduced camera system of a BA graph."""
    lib = load_library()
    oc = np.ascontiguousarray(obs_camera, np.uint32)
    op = np.ascontiguousarray(obs_point, np.uint32)
    u32p = C.POINTER(C.c_uint32)
    n = C.c_uint64(0)
    rc = lib.spp_rcs_block_pattern(n_cameras, n_points, len(oc), oc.ctypes.data_as(u32p), op.ctypes.data_as(u32p), C.byref(n), None, None)
    if rc != SPP_OK:
        raise RuntimeError(f"spp_rcs_block_pattern failed: {rc}")
    r, c = np.empty(n.value, np.uint32), np.empty(n.value, np.uint32)
    rc = lib.spp_rcs_block_pattern(n_cameras, n_points, len(oc), oc.ctypes.data_as(u32p), op.ctypes.data_as(u32p), C.byref(n),
                                   r.ctypes.data_as(u32p), c.ctypes.data_as(u32p))
    if rc != SPP_OK:
        raise RuntimeError(f"spp_rcs_block_pattern failed: {rc}")
    return r, c


def block_ordering(col_ptr, row_idx) -> np.ndarray:
    """Pure host helper: the library's fill-reducing block ordering (order[new position] = block column)."""
    lib = load_library()
    col_ptr = np.ascontiguousarray(col_ptr, np.uint64)
    row_idx = np.ascontiguousarray(row_idx, np.uint64)
    n = len(col_ptr) - 1
    order = np.empty(n, np.uint64)
    rc = lib.spp_block_ordering(n, _u64p(col_ptr), _u64p(row_idx), _u64p(order))
    if rc != SPP_OK:
        raise RuntimeError(f"spp_block_ordering failed: {rc}")
    return order


def block_symbolic_stats(col_ptr, row_idx, order=None) -> dict:
    """Pure host helper: symbolic block Cholesky under an ordering (None = natural)."""
    lib = load_library()
    col_ptr = np.ascontiguousarray(col_ptr, np.uint64)
    row_idx = np.ascontiguousarray(row_idx, np.uint64)
    n = len(col_ptr) - 1
    o = None if order is None else np.ascontiguousarray(order, np.uint64)
    cnt, par, st = np.empty(n, np.uint64), np.empty(n, np.uint64), np.zeros(3)
    rc = lib.spp_block_symbolic_stats(n, _u64p(col_ptr), _u64p(row_idx), _u64p(o), _u64p(cnt), _u64p(par), _dp(st))
    if rc != SPP_OK:
        raise RuntimeError(f"spp_block_symbolic_stats failed: {rc}")
    return dict(col_count=cnt, parent=par, nnzb_factor=int(st[0]), sum_count_sq=float(st[1]), supernodes=int(st[2]))


def block_subtree_owners(col_ptr, row_idx, order, world: int, min_saving: float = 0.03):
    """The plan that shares the block-sparse factorisation out over `world` ranks (host helper): owner of every PERMUTED
    block column (-1: factored by every rank), predicted time as a fraction of the replicated factorisation, supernodes,
    shared supernodes."""
    lib = load_library()
    col_ptr = np.ascontiguousarray(col_ptr, np.uint64)
    row_idx = np.ascontiguousarray(row_idx, np.uint64)
    n = len(col_ptr) - 1
    o = None if order is None else np.ascontiguousarray(order, np.uint64)
    own = np.zeros(n, np.int32)
    st = np.zeros(3)
    rc = lib.spp_block_subtree_owners(n, _u64p(col_ptr), _u64p(row_idx), _u64p(o), int(world), float(min_saving),
                                      own.ctypes.data_as(C.POINTER(C.c_int32)), _dp(st))
    if rc != SPP_OK:
        raise RuntimeError(f"spp_block_subtree_owners failed: {rc}")
    return dict(owner=own, predicted=float(st[0]), supernodes=int(st[1]), shared=int(st[2]))


class SppError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libspp_b200 error {code}: {msg}")
        self.code = code


class NotPositiveDefinite(ArithmeticError):
    """The factorisation met a non-positive pivot (the reference's solvers return false)."""


NCCL_UNIQUE_ID_BYTES = 128


def nccl_unique_id() -> bytes:
    """ncclGetUniqueId through the library (rank 0 calls this and sends the bytes to the other ranks)."""
    lib = load_library()
    buf = C.create_string_buffer(NCCL_UNIQUE_ID_BYTES)
    rc = lib.spp_nccl_get_unique_id(buf)
    if rc != SPP_OK:
        raise SppError(rc, lib.spp_last_error(None).decode())
    return buf.raw


class Context:
    """One solver context on one GPU (``optimizer_t`` of the reference's C API)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.spp_create(device, C.byref(h))
        if rc != SPP_OK:
            raise SppError(rc, self.lib.spp_last_error(None).decode())
        self.h = h
        self._cb = None
        self._schur_n_values = 0  # set by schur_symbolic; without it the library refuses schur_covariance_pattern

    def close(self):
        if getattr(self, "h", None):
            self.lib.spp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        if rc == SPP_NOT_POSDEF:
            raise NotPositiveDefinite("matrix is not positive definite")
        if rc != SPP_OK:
            raise SppError(rc, self.lib.spp_last_error(self.h).decode())
        return rc

    def describe(self) -> str:
        buf = C.create_string_buffer(256)
        self._check(self.lib.spp_describe(self.h, buf, 256))
        return buf.value.decode()

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.spp_kernel_launches(self.h))

    @property
    def stream(self) -> int:
        return int(self.lib.spp_stream(self.h) or 0)

    def synchronize(self):
        self._check(self.lib.spp_synchronize(self.h))

    def set_allreduce(self, fn, rank: int, world: int):
        """fn(device_ptr:int, n_doubles:int) -> None sums the buffer over ranks (torch.distributed / NCCL)."""
        if fn is None:
            self._cb = ALLREDUCE_FN(0)
        else:
            def tramp(_user, ptr, n):
                try:
                    fn(int(ptr), int(n))
                    return 0
                except Exception:  # pragma: no cover - reported through the C status
                    import traceback
                    traceback.print_exc()
                    return 1
            self._cb = ALLREDUCE_FN(tramp)
        self._check(self.lib.spp_set_allreduce(self.h, self._cb, None, rank, world))

    def set_nccl(self, unique_id: bytes, rank: int, world: int):
        """The library's own NCCL communicator (ncclCommInitRank inside the library: collective over the ranks); see
        nccl_unique_id(). The all-reduces of the path then run inside the library on the context's stream."""
        buf = C.create_string_buffer(bytes(unique_id), NCCL_UNIQUE_ID_BYTES) if world > 1 else None
        self._check(self.lib.spp_set_nccl(self.h, buf, rank, world))

    # ---- bundle adjustment ----------------------------------------------------------------------
    def ba_set_graph(self, g):
        vtype = np.ascontiguousarray(g.vtype, np.uint8)
        cams = np.ascontiguousarray(g.cams, np.float64)
        pts = np.ascontiguousarray(g.pts, np.float64)
        op = np.ascontiguousarray(g.obs_pt, np.uint64)
        oc = np.ascontiguousarray(g.obs_cam, np.uint64)
        z = np.ascontiguousarray(g.z, np.float64)
        info = np.ascontiguousarray(g.info, np.float64)
        # the library reads raw pointers: a mismatched graph must raise here, not read out of bounds there
        n_c, n_p, n_o = int(np.count_nonzero(vtype == 0)), int(np.count_nonzero(vtype == 1)), int(op.shape[0])
        if vtype.ndim != 1 or n_c + n_p != vtype.shape[0]:
            raise ValueError("vtype must be a vector of 0 (camera) / 1 (point)")
        if cams.shape != (n_c, 11):
            raise ValueError(f"cams must be ({n_c}, 11): state 6 + intrinsics 5 per type-0 vertex, got {cams.shape}")
        if pts.shape != (n_p, 3):
            raise ValueError(f"pts must be ({n_p}, 3), got {pts.shape}")
        if op.ndim != 1 or oc.shape != (n_o,):
            raise ValueError("obs_pt and obs_cam must be vectors of the same length")
        if z.shape != (n_o, 2) or info.shape != (n_o, 2, 2):
            raise ValueError(f"z must be ({n_o}, 2) and info ({n_o}, 2, 2), got {z.shape} and {info.shape}")
        self._ba_dims = (int(cams.shape[0]), int(pts.shape[0]), int(op.shape[0]), int(vtype.shape[0]))
        self._ba_vertex_dims = np.where(vtype == 0, 6, 3)
        self._check(self.lib.spp_ba_set_graph(self.h, vtype.shape[0], _u8p(vtype), _dp(cams), _dp(pts), op.shape[0],
                                              _u64p(op), _u64p(oc), _dp(z), _dp(info)))

    def ba_append_graph(self, g):
        """g: the NEW vertices and observations only (same layout as for ba_set_graph; vertex ids continue the numbering)."""
        vtype = np.ascontiguousarray(g.vtype, np.uint8)
        cams = np.ascontiguousarray(g.cams, np.float64).reshape(-1, 11)
        pts = np.ascontiguousarray(g.pts, np.float64).reshape(-1, 3)
        op = np.ascontiguousarray(g.obs_pt, np.uint64)
        oc = np.ascontiguousarray(g.obs_cam, np.uint64)
        z = np.ascontiguousarray(g.z, np.float64).reshape(-1, 2)
        info = np.ascontiguousarray(g.info, np.float64).reshape(-1, 2, 2)
        n_c, n_p, n_o = int(np.count_nonzero(vtype == 0)), int(np.count_nonzero(vtype == 1)), int(op.shape[0])
        if vtype.ndim != 1 or n_c + n_p != vtype.shape[0]:
            raise ValueError("vtype must be a vector of 0 (camera) / 1 (point)")
        if cams.shape[0] != n_c or pts.shape[0] != n_p:
            raise ValueError(f"cams must be ({n_c}, 11) and pts ({n_p}, 3), got {cams.shape} and {pts.shape}")
        if oc.shape != (n_o,) or z.shape[0] != n_o or info.shape[0] != n_o:
            raise ValueError("obs_pt, obs_cam, z (O, 2) and info (O, 2, 2) must have the same length")
        self._check(self.lib.spp_ba_append_graph(self.h, vtype.shape[0], _u8p(vtype), _dp(cams), _dp(pts), n_o,
                                                 _u64p(op), _u64p(oc), _dp(z), _dp(info)))
        c0, p0, o0, v0 = self._ba_dims
        self._ba_dims = (c0 + n_c, p0 + n_p, o0 + n_o, v0 + int(vtype.shape[0]))
        self._ba_vertex_dims = np.concatenate([self._ba_vertex_dims, np.where(vtype == 0, 6, 3)])

    def ba_set_states(self, cam_states=None, pts=None):
        cs = None if cam_states is None else np.ascontiguousarray(cam_states, np.float64)
        ps = None if pts is None else np.ascontiguousarray(pts, np.float64)
        self._check(self.lib.spp_ba_set_states(self.h, _dp(cs), _dp(ps)))

    def ba_get_partition(self):
        b, e = C.c_uint64(), C.c_uint64()
        self._check(self.lib.spp_ba_get_partition(self.h, C.byref(b), C.byref(e)))
        return int(b.value), int(e.value)

    def ba_get_states(self, out_cams=None, out_pts=None):
        """Camera states and landmark positions; on a partitioned context only this rank's landmark slice
        (ba_get_partition) is filled, the rest is zero. out_cams (C, 6) / out_pts (P, 3): float64 C-contiguous buffers of the
        caller (e.g. page-locked ones: the device-to-host copy then runs at the full rate of the link), returned filled."""
        c, p, _, _ = self._ba_dims
        cs = np.empty((c, 6)) if out_cams is None else out_cams
        ps = np.zeros((p, 3)) if out_pts is None else out_pts
        for a, shape in ((cs, (c, 6)), (ps, (p, 3))):
            if a.shape != shape or a.dtype != np.float64 or not a.flags.c_contiguous or not a.flags.writeable:
                raise ValueError(f"output buffer must be a writeable C-contiguous float64 array of shape {shape}")
        self._check(self.lib.spp_ba_get_states(self.h, _dp(cs), _dp(ps)))
        return cs, ps

    def ba_gather_states(self):
        """All camera states and all landmark positions on every rank (a collective on a partitioned context)."""
        c, p, _, _ = self._ba_dims
        cs, ps = np.empty((c, 6)), np.zeros((p, 3))
        self._check(self.lib.spp_ba_gather_states(self.h, _dp(cs), _dp(ps)))
        return cs, ps

    def ba_restore_initial(self):
        self._check(self.lib.spp_ba_restore_initial(self.h))

    def ba_set_jacobian_mode(self, mode: int):
        self._check(self.lib.spp_ba_set_jacobian_mode(self.h, mode))

    def ba_set_robust_loss(self, kind: int, scale: float = 1.0):
        """Robust loss of every BA observation: LOSS_NONE (default), LOSS_HUBER or LOSS_CAUCHY with scale k > 0 in units of
        the Mahalanobis error (pixels for identity information). Context state: kept across ba_set_graph, ba_append_graph and
        ba_restore_initial. The linearisation, the marginals and ba_chi2 (then sum rho) follow it."""
        self._check(self.lib.spp_ba_set_robust_loss(self.h, int(kind), float(scale)))

    def ba_observation_errors(self):
        """(sq_error, weight): s2 = r^T Omega r and the loss weight w of every observation at the current states, in edge
        insertion order; w is bit for bit the weight a linearisation at these states uses."""
        o = self._ba_dims[2]
        s2, w = np.empty(o), np.empty(o)
        self._check(self.lib.spp_ba_get_observation_errors(self.h, _dp(s2), _dp(w)))
        return s2, w

    def ba_linearise(self):
        self._check(self.lib.spp_ba_linearise(self.h))

    def ba_get_lambda(self):
        """Returns (col_dims, col_ptr, row_idx, values, eta) in the reference's block layout."""
        nbc, nb, nv = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.spp_ba_get_lambda(self.h, C.byref(nbc), C.byref(nb), C.byref(nv), None, None, None, None, None))
        col_dims = np.empty(nbc.value, np.uint64)
        col_ptr = np.empty(nbc.value + 1, np.uint64)
        row_idx = np.empty(nb.value, np.uint64)
        vals = np.empty(nv.value)
        eta = np.empty(int(self._ba_dims[0] * 6 + self._ba_dims[1] * 3))
        self._check(self.lib.spp_ba_get_lambda(self.h, None, None, None, _u64p(col_dims), _u64p(col_ptr), _u64p(row_idx),
                                               _dp(vals), _dp(eta)))
        return col_dims, col_ptr, row_idx, vals, eta

    def ba_get_blocks(self):
        """Returns U (C,36), V (P,9), W (O,18; edge insertion order), eta_c (C,6), eta_p (P,3)."""
        c, p, o, _ = self._ba_dims
        U, V, W = np.empty((c, 36)), np.empty((p, 9)), np.empty((o, 18))
        gc, gp = np.empty((c, 6)), np.empty((p, 3))
        self._check(self.lib.spp_ba_get_blocks(self.h, _dp(U), _dp(V), _dp(W), _dp(gc), _dp(gp)))
        return U, V, W, gc, gp

    def ba_chi2(self) -> float:
        v = C.c_double()
        self._check(self.lib.spp_ba_chi2(self.h, C.byref(v)))
        return v.value

    def ba_solve_step(self, alpha: float) -> np.ndarray:
        dx = np.empty(int(self._ba_dims[0] * 6 + self._ba_dims[1] * 3))
        self._check(self.lib.spp_ba_solve_step(self.h, alpha, _dp(dx)))
        return dx

    def ba_optimize(self, max_iterations: int = 5, min_dx_norm: float = 0.01) -> dict:
        rep = Report()
        self._check(self.lib.spp_ba_optimize(self.h, max_iterations, min_dx_norm, C.byref(rep)))
        return rep.as_dict()

    def ba_marginals(self, alpha: float = 0.0):
        """Block diagonal of (lambda + alpha I)^-1 at the current states: (C, 6, 6), (P, 3, 3)."""
        c, p, _, _ = self._ba_dims
        cc, pc = np.empty((c, 6, 6)), np.empty((p, 3, 3))
        self._check(self.lib.spp_ba_marginals(self.h, alpha, _dp(cc), _dp(pc)))
        return cc, pc

    def ba_marginals_sparse(self, alpha: float = 0.0):
        """ba_marginals through the block-sparse (supernodal) factorisation and its selected inversion: no dense inverse,
        any number of cameras. (C, 6, 6), (P, 3, 3)."""
        c, p, _, _ = self._ba_dims
        cc, pc = np.empty((c, 6, 6)), np.empty((p, 3, 3))
        self._check(self.lib.spp_ba_marginals_sparse(self.h, alpha, _dp(cc), _dp(pc)))
        return cc, pc

    def ba_covariance_blocks(self, alpha: float, cam_pairs=None, observations=None, diagonal: bool = False) -> dict:
        """Selected blocks of (lambda + alpha I)^-1 at the current states in one factorisation and inversion, on the dense
        or the supernodal reduced camera system as schur_set_rcs_solver selects.
          cam_pairs (n, 2): camera indices (id order among cameras) of pairs that share a landmark or are equal
                            -> "pairs" (n, 6, 6), [k] = Cov(cam a, cam b)
          observations (m,): edge insertion indices -> "observations" (m, 6, 3), [k] = Cov(camera, point) of that edge
          diagonal: also "cameras" (C, 6, 6) and "points" (P, 3, 3), bit-identical to ba_marginals / ba_marginals_sparse
        Every block is indexed [k, row, column]; the library writes them column-major (as W in ba_get_blocks)."""
        c, p, _, _ = self._ba_dims
        pairs = np.zeros((0, 2), np.uint64) if cam_pairs is None else np.asarray(cam_pairs)
        obs = np.zeros(0, np.uint64) if observations is None else np.asarray(observations)
        if pairs.ndim != 2 or pairs.shape[1] != 2:
            raise ValueError(f"cam_pairs must be (n, 2), got {pairs.shape}")
        if obs.ndim != 1:
            raise ValueError(f"observations must be a vector, got {obs.shape}")
        if (pairs.size and pairs.min() < 0) or (obs.size and obs.min() < 0):
            raise ValueError("indices must be non-negative")
        cam_a = np.ascontiguousarray(pairs[:, 0], np.uint64)
        cam_b = np.ascontiguousarray(pairs[:, 1], np.uint64)
        obs = np.ascontiguousarray(obs, np.uint64)
        n, m = len(cam_a), len(obs)
        pc, oc = np.empty((n, 36)), np.empty((m, 18))
        cc, ptc = (np.empty((c, 6, 6)), np.empty((p, 3, 3))) if diagonal else (None, None)
        self._check(self.lib.spp_ba_covariance_blocks(self.h, alpha, n, _u64p(cam_a), _u64p(cam_b), _dp(pc), m, _u64p(obs), _dp(oc),
                                                      _dp(cc), _dp(ptc)))
        out = dict(pairs=pc.reshape(n, 6, 6).transpose(0, 2, 1), observations=oc.reshape(m, 3, 6).transpose(0, 2, 1))
        if diagonal:
            out.update(cameras=cc, points=ptc)
        return out

    def ba_joint_marginals(self, alpha: float, sets) -> list:
        """Joint marginal covariance of sets of vertices at the current states. sets: a list of integer arrays of vertex
        ids (cameras and points mixed, any order; pairs on or off the block pattern, e.g. cameras that share no
        landmark). Returns a list of (D_k, D_k) arrays, D_k = 6 per camera + 3 per point, rows and columns in the order
        of the set. Dense or supernodal reduced camera system as schur_set_rcs_solver selects."""
        return self._joint_call(self.lib.spp_ba_joint_marginals, alpha, sets, getattr(self, "_ba_vertex_dims", None))

    def schur_joint_marginals(self, alpha: float, sets) -> list:
        """ba_joint_marginals for the lambda of the last schur_solve: sets of block columns in the numbering given to
        schur_symbolic."""
        return self._joint_call(self.lib.spp_schur_joint_marginals, alpha, sets, getattr(self, "_schur_col_dims", None))

    def _joint_call(self, fn, alpha: float, sets, vertex_dims) -> list:
        ids = [np.asarray(v).reshape(-1) for v in sets]
        for v in ids:
            if v.size and (not np.issubdtype(v.dtype, np.integer) or v.min() < 0):
                raise ValueError("vertex ids must be non-negative integers")
        ptr = np.zeros(len(ids) + 1, np.uint64)
        ptr[1:] = np.cumsum([len(v) for v in ids])
        flat = np.ascontiguousarray(np.concatenate(ids) if ids else np.zeros(0), np.uint64)
        vd = np.zeros(0, np.int64) if vertex_dims is None else np.asarray(vertex_dims, np.int64)
        # ids out of range count 0 here: the library refuses them before it writes anything
        dk = np.array([int(vd[v[v < len(vd)].astype(np.int64)].sum()) for v in ids], np.int64)
        out = np.empty(max(int((dk * dk).sum()), 1))
        self._check(fn(self.h, alpha, len(ids), _u64p(ptr), _u64p(flat), _dp(out)))
        res, off = [], 0
        for D in dk:
            res.append(out[off:off + D * D].reshape(D, D).T)  # column-major in the library
            off += D * D
        return res

    # ---- slot 1: Schur linear solver on a caller-supplied lambda ---------------------------------
    def schur_symbolic(self, col_dims, col_ptr, row_idx):
        cd = np.ascontiguousarray(col_dims, np.uint64)
        cp = np.ascontiguousarray(col_ptr, np.uint64)
        ri = np.ascontiguousarray(row_idx, np.uint64)
        order = np.empty(cd.shape[0], np.uint64)
        cut = C.c_uint64()
        self._check(self.lib.spp_schur_symbolic(self.h, cd.shape[0], _u64p(cd), _u64p(cp), _u64p(ri), _u64p(order),
                                                C.byref(cut)))
        self._schur_n = int(cd.astype(np.int64).sum())
        dims = cd.astype(np.int64)
        self._schur_n_values = int((dims[ri.astype(np.int64)] * np.repeat(dims, np.diff(cp.astype(np.int64)))).sum())
        self._schur_cut = (int(cut.value), int(cd.shape[0]) - int(cut.value))
        self._schur_col_dims = dims
        return order.astype(np.int64), int(cut.value)

    def schur_marginals(self, alpha: float = 0.0):
        """Block diagonal of (lambda + alpha I)^-1 for the lambda of the last schur_solve: (cut, 6, 6), (n - cut, 3, 3)."""
        c, p = self._schur_cut
        cc, pc = np.empty((c, 6, 6)), np.empty((p, 3, 3))
        self._check(self.lib.spp_schur_marginals(self.h, alpha, _dp(cc), _dp(pc)))
        return cc, pc

    def schur_marginals_sparse(self, alpha: float = 0.0):
        """schur_marginals through the block-sparse (supernodal) factorisation and its selected inversion."""
        c, p = self._schur_cut
        cc, pc = np.empty((c, 6, 6)), np.empty((p, 3, 3))
        self._check(self.lib.spp_schur_marginals_sparse(self.h, alpha, _dp(cc), _dp(pc)))
        return cc, pc

    def schur_covariance_pattern(self, alpha: float = 0.0) -> np.ndarray:
        """(lambda + alpha I)^-1 on the block pattern of the lambda of the last schur_solve, shaped like its values (the
        reference's block layout: column-major blocks in the order of the structure given to schur_symbolic)."""
        out = np.empty(self._schur_n_values)
        self._check(self.lib.spp_schur_covariance_pattern(self.h, alpha, _dp(out)))
        return out

    def schur_solve(self, values, eta) -> np.ndarray:
        v = np.ascontiguousarray(values, np.float64)
        x = np.array(eta, np.float64, copy=True)
        self._check(self.lib.spp_schur_solve(self.h, _dp(v), _dp(x)))
        return x

    def schur_get_reduced_system(self, want_values: bool = True):
        n = C.c_uint64()
        self._check(self.lib.spp_schur_get_reduced_system(self.h, C.byref(n), None, None, None))
        n = int(n.value)
        c = n // 6
        pat = np.zeros((c, c), np.uint8)
        if want_values:
            S = np.empty((n, n))
            rhs = np.empty(n)
            self._check(self.lib.spp_schur_get_reduced_system(self.h, None, _dp(S), _dp(rhs), _u8p(pat)))
            return S.T.copy(), rhs, pat  # library writes column-major
        self._check(self.lib.spp_schur_get_reduced_system(self.h, None, None, None, _u8p(pat)))
        return None, None, pat

    # ---- dense Cholesky --------------------------------------------------------------------------
    def schur_set_rcs_solver(self, mode: int):
        self._check(self.lib.spp_schur_set_rcs_solver(self.h, mode))

    def schur_set_rcs_ordering(self, order=None):
        if order is None:
            self._check(self.lib.spp_schur_set_rcs_ordering(self.h, 0, None))
        else:
            o = np.ascontiguousarray(order, np.uint64)
            self._check(self.lib.spp_schur_set_rcs_ordering(self.h, len(o), _u64p(o)))

    def schur_get_rcs_owners(self) -> np.ndarray:
        """per supernode of the block-sparse reduced camera system: the rank that factors it, -1 = every rank"""
        n = int(self.schur_get_rcs_info()["supernodes"])
        o = np.zeros(n, np.int32)
        self._check(self.lib.spp_schur_get_rcs_owners(self.h, o.ctypes.data_as(C.POINTER(C.c_int32))))
        return o

    def schur_get_rcs_info(self) -> dict:
        st = np.zeros(8)
        self._check(self.lib.spp_schur_get_rcs_info(self.h, None, _dp(st)))
        order = np.empty(int(st[0]), np.uint64)
        self._check(self.lib.spp_schur_get_rcs_info(self.h, _u64p(order), None))
        return dict(order=order, cameras=int(st[0]), rcs_blocks=int(st[1]), supernodes=int(st[2]), factor_blocks_exact=int(st[3]),
                    factor_blocks_stored=int(st[4]), factor_flops=float(st[5]), factor_bytes=float(st[6]), updates=int(st[7]))

    def schur_get_rcs_residual(self) -> float:
        v = C.c_double()
        self._check(self.lib.spp_schur_get_rcs_residual(self.h, C.byref(v)))
        return v.value

    def dense_posdef_solve(self, A, b) -> np.ndarray:
        A = np.asfortranarray(A, np.float64)
        x = np.array(b, np.float64, copy=True)
        self._check(self.lib.spp_dense_posdef_solve(self.h, A.shape[0], A.ctypes.data_as(C.POINTER(C.c_double)), _dp(x)))
        return x

    def dense_panel_factor(self, panel) -> np.ndarray:
        """panel: (n_rows, n_cols) array; returns [R11 (upper triangle) | R11^-T A12] of the same shape."""
        p = np.asfortranarray(panel, np.float64).copy(order="F")
        self._check(self.lib.spp_dense_panel_factor(self.h, p.shape[0], p.shape[1], p.ctypes.data_as(C.POINTER(C.c_double))))
        return p

    # ---- block-sparse Cholesky (slot: CLinearSolver_UberBlock) -------------------------------------
    def chol_symbolic(self, block_size: int, col_ptr, row_idx, order=None) -> np.ndarray:
        """Returns the block ordering in use (new position -> original block column)."""
        cp = np.ascontiguousarray(col_ptr, np.uint64)
        ri = np.ascontiguousarray(row_idx, np.uint64)
        oi = None if order is None else np.ascontiguousarray(order, np.uint64)
        n = cp.shape[0] - 1
        out = np.empty(n, np.uint64)
        self._check(self.lib.spp_chol_symbolic(self.h, n, block_size, _u64p(cp), _u64p(ri), _u64p(oi), _u64p(out)))
        self._chol_dims = (n, block_size)
        return out.astype(np.int64)

    def chol_solve(self, values, eta) -> np.ndarray:
        v = np.ascontiguousarray(values, np.float64)
        x = np.array(eta, np.float64, copy=True)
        self._check(self.lib.spp_chol_solve(self.h, _dp(v), _dp(x)))
        return x

    def chol_get_factor(self, n: int, block_size: int):
        """The upper factor R (R^T R = P lambda P^T) as block CSC: col_ptr, row_idx, values (column-major blocks)."""
        nb = C.c_uint64()
        self._check(self.lib.spp_chol_get_factor(self.h, C.byref(nb), None, None, None))
        cp = np.empty(n + 1, np.uint64)
        ri = np.empty(nb.value, np.uint64)
        vals = np.empty(nb.value * block_size * block_size)
        self._check(self.lib.spp_chol_get_factor(self.h, None, _u64p(cp), _u64p(ri), _dp(vals)))
        return cp, ri, vals

    # ---- pose graphs -------------------------------------------------------------------------------
    def pose_set_graph(self, g, order=None):
        poses = np.ascontiguousarray(g.poses, np.float64)
        ef = np.ascontiguousarray(g.e_from, np.uint64)
        et = np.ascontiguousarray(g.e_to, np.uint64)
        z = np.ascontiguousarray(g.z, np.float64)
        info = np.ascontiguousarray(g.info, np.float64)
        if poses.ndim != 2 or poses.shape[1] not in (3, 6):
            raise ValueError(f"poses must be (N, 3) or (N, 6), got {poses.shape}")
        n_e, dim = int(ef.shape[0]), int(poses.shape[1])
        if ef.ndim != 1 or et.shape != (n_e,) or z.shape != (n_e, dim) or info.shape != (n_e, dim, dim):
            raise ValueError(f"e_from / e_to must be vectors of one length E, z (E, {dim}), info (E, {dim}, {dim})")
        self._pose_dims = (int(poses.shape[0]), int(poses.shape[1]))
        self._check(self.lib.spp_pose_set_graph(self.h, poses.shape[1], poses.shape[0], _dp(poses), ef.shape[0], _u64p(ef),
                                                _u64p(et), _dp(z), _dp(info)))
        if order is not None:
            self._check(self.lib.spp_pose_set_ordering(self.h, _u64p(np.ascontiguousarray(order, np.uint64))))

    def pose_set_states(self, poses):
        self._check(self.lib.spp_pose_set_states(self.h, _dp(np.ascontiguousarray(poses, np.float64))))

    def pose_get_states(self) -> np.ndarray:
        out = np.empty(self._pose_dims)
        self._check(self.lib.spp_pose_get_states(self.h, _dp(out)))
        return out

    def pose_restore_initial(self):
        self._check(self.lib.spp_pose_restore_initial(self.h))

    def pose_linearise(self):
        self._check(self.lib.spp_pose_linearise(self.h))

    def pose_get_lambda(self):
        """Returns (col_ptr, row_idx, values, eta) in the reference's block layout."""
        n, d = self._pose_dims
        nbc, nb = C.c_uint64(), C.c_uint64()
        self._check(self.lib.spp_pose_get_lambda(self.h, C.byref(nbc), C.byref(nb), None, None, None, None))
        cp = np.empty(nbc.value + 1, np.uint64)
        ri = np.empty(nb.value, np.uint64)
        vals = np.empty(nb.value * d * d)
        eta = np.empty(n * d)
        self._check(self.lib.spp_pose_get_lambda(self.h, None, None, _u64p(cp), _u64p(ri), _dp(vals), _dp(eta)))
        return cp, ri, vals, eta

    def pose_chi2(self) -> float:
        v = C.c_double()
        self._check(self.lib.spp_pose_chi2(self.h, C.byref(v)))
        return v.value

    def pose_solve_step(self) -> np.ndarray:
        n, d = self._pose_dims
        dx = np.empty(n * d)
        self._check(self.lib.spp_pose_solve_step(self.h, _dp(dx)))
        return dx

    def pose_marginals(self) -> np.ndarray:
        """Block diagonal of lambda^-1 at the current states: (N, dim, dim)."""
        n, d = self._pose_dims
        cov = np.empty((n, d, d))
        self._check(self.lib.spp_pose_marginals(self.h, _dp(cov)))
        return cov

    def pose_optimize(self, max_iterations: int = 5, min_dx_norm: float = 0.01) -> dict:
        rep = Report()
        self._check(self.lib.spp_pose_optimize(self.h, max_iterations, min_dx_norm, C.byref(rep)))
        return rep.as_dict()
