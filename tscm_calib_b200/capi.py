"""ctypes mirror of include/tscm.h (the C-ABI of libtscm_b200.so).

Plumbing only: struct layouts, library loading, and a thin `Solver` handle.
The product is the shared library; nothing here computes.
There is NO CPU fallback: if the CUDA library is missing `load_library()` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtscm_b200.so")

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)

TERMINATION = {0: "CONVERGENCE", 1: "NO_CONVERGENCE", 2: "FAILURE"}
LOSS = {"none": 0, "huber": 1, "cauchy": 2}


class TscmProblem(C.Structure):
    _fields_ = [
        ("num_cameras", C.c_int32),
        ("num_frames", C.c_int32),
        ("corners_per_board", C.c_int32),
        ("num_views", C.c_int32),
        ("board_xy", c_double_p),
        ("view_camera", c_int32_p),
        ("view_frame", c_int32_p),
        ("obs_xy", c_double_p),
        ("fixed_camera", C.c_int32),
    ]


class TscmOptions(C.Structure):
    _fields_ = [
        ("max_num_iterations", C.c_int32),
        ("function_tolerance", C.c_double),
        ("gradient_tolerance", C.c_double),
        ("parameter_tolerance", C.c_double),
        ("initial_trust_region_radius", C.c_double),
        ("max_trust_region_radius", C.c_double),
        ("min_trust_region_radius", C.c_double),
        ("min_relative_decrease", C.c_double),
        ("min_lm_diagonal", C.c_double),
        ("max_lm_diagonal", C.c_double),
        ("max_num_consecutive_invalid_steps", C.c_int32),
        ("jacobi_scaling", C.c_int32),
        ("loss_type", C.c_int32),
        ("loss_scale", C.c_double),
        ("parameter_tolerance_needs_successful_step", C.c_int32),
        ("disable_tolerances", C.c_int32),
        ("verbose", C.c_int32),
        ("num_gpus", C.c_int32),
        ("allow_large_rigs", C.c_int32),
    ]


class TscmSummary(C.Structure):
    _fields_ = [
        ("termination_type", C.c_int32),
        ("num_iterations", C.c_int32),
        ("num_successful_steps", C.c_int32),
        ("num_unsuccessful_steps", C.c_int32),
        ("initial_cost", C.c_double),
        ("final_cost", C.c_double),
        ("final_radius", C.c_double),
        ("trace_capacity", C.c_int32),
        ("trace_cost", c_double_p),
        ("trace_radius", c_double_p),
        ("trace_gradient_max_norm", c_double_p),
        ("trace_step_norm", c_double_p),
        ("trace_step_flags", c_int32_p),
    ]


class TscmCovariance(C.Structure):
    """tscm_covariance (include/tscm.h)."""
    _fields_ = [
        ("camera", c_double_p),
        ("board", c_double_p),
        ("residual_variance", C.c_double),
        ("kernel_ms", C.c_double),
    ]


class TscmRemapJob(C.Structure):
    """tscm_remap_job (include/tscm.h): one block of a remap table."""
    _fields_ = [
        ("intrinsics", C.c_double * 9),
        ("matrix", C.c_double * 9),
        ("ray_fx", C.c_double), ("ray_fy", C.c_double), ("ray_cx", C.c_double), ("ray_cy", C.c_double),
        ("offset_x", C.c_double), ("offset_y", C.c_double),
        ("cutoff_w2", C.c_double),
        ("width", C.c_int32), ("height", C.c_int32),
        ("row0", C.c_int32), ("col0", C.c_int32),
    ]


class TscmPoseGraphProblem(C.Structure):
    """tscm_pose_graph_problem (include/tscm.h)."""
    _fields_ = [
        ("num_cameras", C.c_int32), ("num_boards", C.c_int32), ("corners_per_board", C.c_int32),
        ("worlds", c_double_p), ("intrinsics", c_double_p), ("has_board", C.POINTER(C.c_uint8)),
        ("mono_rt", c_double_p), ("pixels", c_double_p),
    ]


class TscmPoseGraphResult(C.Structure):
    """tscm_pose_graph_result (include/tscm.h)."""
    _fields_ = [
        ("camera_pose", c_double_p), ("board_pose", c_double_p),
        ("board_initialised", C.POINTER(C.c_uint8)),
        ("camera_choice", c_int32_p), ("board_choice", c_int32_p),
        ("camera_candidate_error", c_double_p), ("board_candidate_error", c_double_p),
        ("kernel_ms", C.c_double), ("projections", C.c_int64),
    ]


class TscmMonoInitProblem(C.Structure):
    """tscm_mono_init_problem (include/tscm.h)."""
    _fields_ = [
        ("num_frames", C.c_int32), ("board_width", C.c_int32), ("board_height", C.c_int32),
        ("image_width", C.c_int32), ("image_height", C.c_int32),
        ("worlds", c_double_p), ("has_board", C.POINTER(C.c_uint8)), ("pixels", c_double_p),
        ("has_init_guess", C.c_int32),
    ]


class TscmMonoInitResult(C.Structure):
    """tscm_mono_init_result (include/tscm.h)."""
    _fields_ = [
        ("intrinsics", C.c_double * 9), ("mono_rt", c_double_p), ("frame_ok", C.POINTER(C.c_uint8)),
        ("focal_rows_used", C.c_int32), ("kernel_ms", C.c_double),
    ]


def default_options(**overrides) -> TscmOptions:
    """ceres::Solver::Options defaults in force at TS.cpp:271-274 /
    multi_calib.cpp:209-212 (same values tscm_options_init() writes)."""
    o = TscmOptions()
    o.max_num_iterations = 50
    o.function_tolerance = 1e-6
    o.gradient_tolerance = 1e-10
    o.parameter_tolerance = 1e-8
    o.initial_trust_region_radius = 1e4
    o.max_trust_region_radius = 1e16
    o.min_trust_region_radius = 1e-32
    o.min_relative_decrease = 1e-3
    o.min_lm_diagonal = 1e-6
    o.max_lm_diagonal = 1e32
    o.max_num_consecutive_invalid_steps = 5
    o.jacobi_scaling = 1
    o.loss_type = 0
    o.loss_scale = 1.0
    o.parameter_tolerance_needs_successful_step = 0
    o.disable_tolerances = 0
    o.verbose = 0
    o.num_gpus = 1
    o.allow_large_rigs = 0
    for k, v in overrides.items():
        if k == "loss_type" and isinstance(v, str):
            v = LOSS[v]
        if not hasattr(o, k):
            raise AttributeError(k)
        setattr(o, k, v)
    return o


def _dp(a: np.ndarray):
    return a.ctypes.data_as(c_double_p)


def _ip(a: np.ndarray):
    return a.ctypes.data_as(c_int32_p)


@dataclass
class SummaryResult:
    termination: str
    num_iterations: int
    num_successful_steps: int
    num_unsuccessful_steps: int
    initial_cost: float
    final_cost: float
    final_radius: float
    cost: np.ndarray = field(repr=False, default=None)
    radius: np.ndarray = field(repr=False, default=None)
    gradient_max_norm: np.ndarray = field(repr=False, default=None)
    step_norm: np.ndarray = field(repr=False, default=None)
    step_flags: np.ndarray = field(repr=False, default=None)


class SummaryBuffers:
    """Owns the caller-side trace arrays of a tscm_summary."""

    def __init__(self, capacity: int):
        self.capacity = int(capacity)
        self.cost = np.zeros(capacity)
        self.radius = np.zeros(capacity)
        self.gmax = np.zeros(capacity)
        self.step_norm = np.zeros(capacity)
        self.flags = np.zeros(capacity, dtype=np.int32)
        s = TscmSummary()
        s.trace_capacity = capacity
        s.trace_cost = _dp(self.cost)
        s.trace_radius = _dp(self.radius)
        s.trace_gradient_max_norm = _dp(self.gmax)
        s.trace_step_norm = _dp(self.step_norm)
        s.trace_step_flags = _ip(self.flags)
        self.c = s

    def result(self) -> SummaryResult:
        n = min(self.c.num_iterations, self.capacity)
        return SummaryResult(
            TERMINATION.get(self.c.termination_type, str(self.c.termination_type)),
            self.c.num_iterations, self.c.num_successful_steps, self.c.num_unsuccessful_steps,
            self.c.initial_cost, self.c.final_cost, self.c.final_radius,
            self.cost[:n].copy(), self.radius[:n].copy(), self.gmax[:n].copy(),
            self.step_norm[:n].copy(), self.flags[:n].copy())


class ProblemArrays:
    """Keeps the numpy arrays behind a tscm_problem alive and C-contiguous."""

    def __init__(self, board_xy, view_camera, view_frame, obs_xy, num_cameras, num_frames,
                 fixed_camera=0):
        self.board_xy = np.ascontiguousarray(board_xy, dtype=np.float64).reshape(-1, 2)
        self.view_camera = np.ascontiguousarray(view_camera, dtype=np.int32).reshape(-1)
        self.view_frame = np.ascontiguousarray(view_frame, dtype=np.int32).reshape(-1)
        K = self.board_xy.shape[0]
        V = self.view_camera.shape[0]
        self.obs_xy = np.ascontiguousarray(obs_xy, dtype=np.float64).reshape(V, K, 2)
        self.num_cameras = int(num_cameras)
        self.num_frames = int(num_frames)
        self.fixed_camera = int(fixed_camera)
        p = TscmProblem()
        p.num_cameras = self.num_cameras
        p.num_frames = self.num_frames
        p.corners_per_board = K
        p.num_views = V
        p.board_xy = _dp(self.board_xy)
        p.view_camera = _ip(self.view_camera)
        p.view_frame = _ip(self.view_frame)
        p.obs_xy = _dp(self.obs_xy)
        p.fixed_camera = self.fixed_camera
        self.c = p

    @property
    def num_views(self):
        return self.view_camera.shape[0]

    @property
    def corners_per_board(self):
        return self.board_xy.shape[0]

    @property
    def num_observations(self):
        return self.num_views * self.corners_per_board


_lib = None


def load_library(path: str | None = None):
    """Load libtscm_b200.so and declare every entry point of include/tscm.h.
    Raises (never falls back) when the library is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("TSCM_LIB_PATH") or LIB_PATH   # TSCM_LIB_PATH: A/B builds (tools/)
    if not os.path.exists(p):
        raise RuntimeError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`."
            " There is no CPU fallback for the calibration solve.")
    lib = C.CDLL(p, mode=C.RTLD_GLOBAL)
    P = C.POINTER
    lib.tscm_options_init.argtypes = [P(TscmOptions)]
    lib.tscm_options_init.restype = None
    lib.tscm_solve.argtypes = [P(TscmProblem), P(TscmOptions), c_double_p, c_double_p,
                               c_double_p, P(TscmSummary), C.c_int]
    lib.tscm_solve.restype = C.c_int
    lib.tscm_cache_configure.argtypes = [C.c_int32]
    lib.tscm_cache_configure.restype = None
    lib.tscm_cache_release.argtypes = []
    lib.tscm_cache_release.restype = None
    lib.tscm_host_alloc.argtypes = [C.c_size_t]
    lib.tscm_host_alloc.restype = C.c_void_p
    lib.tscm_host_free.argtypes = [C.c_void_p]
    lib.tscm_host_free.restype = None
    lib.tscm_solver_set_exchange_timeout.argtypes = [C.c_void_p, C.c_double]
    lib.tscm_solver_set_exchange_timeout.restype = C.c_int
    lib.tscm_solver_set_schur_form.argtypes = [C.c_void_p, C.c_int]
    lib.tscm_solver_set_schur_form.restype = C.c_int
    lib.tscm_solver_set_reduced_solve.argtypes = [C.c_void_p, C.c_int]
    lib.tscm_solver_set_reduced_solve.restype = C.c_int
    lib.tscm_set_debug.argtypes = [C.c_int32]
    lib.tscm_set_debug.restype = None
    lib.tscm_solver_create.argtypes = [P(TscmProblem), P(TscmOptions), C.c_int, P(C.c_void_p)]
    lib.tscm_solver_create.restype = C.c_int
    lib.tscm_solver_destroy.argtypes = [C.c_void_p]
    lib.tscm_solver_destroy.restype = None
    lib.tscm_solver_set_options.argtypes = [C.c_void_p, P(TscmOptions)]
    lib.tscm_solver_set_options.restype = C.c_int
    lib.tscm_solver_set_parameters.argtypes = [C.c_void_p, c_double_p, c_double_p, c_double_p]
    lib.tscm_solver_set_parameters.restype = C.c_int
    lib.tscm_solver_get_parameters.argtypes = [C.c_void_p, c_double_p, c_double_p, c_double_p]
    lib.tscm_solver_get_parameters.restype = C.c_int
    lib.tscm_solver_set_observations.argtypes = [C.c_void_p, c_double_p]
    lib.tscm_solver_set_observations.restype = C.c_int
    lib.tscm_solver_run.argtypes = [C.c_void_p, P(TscmSummary)]
    lib.tscm_solver_run.restype = C.c_int
    lib.tscm_comm_unique_id.argtypes = [C.c_void_p]
    lib.tscm_comm_unique_id.restype = C.c_int
    lib.tscm_solver_attach_comm.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.tscm_solver_attach_comm.restype = C.c_int
    lib.tscm_solver_p2p_export.argtypes = [C.c_void_p, C.c_void_p]
    lib.tscm_solver_p2p_export.restype = C.c_int
    lib.tscm_solver_p2p_attach.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.tscm_solver_p2p_attach.restype = C.c_int
    lib.tscm_solver_eval_jacobian.argtypes = [C.c_void_p, c_double_p, c_double_p, c_double_p]
    lib.tscm_solver_eval_jacobian.restype = C.c_int
    lib.tscm_solver_reduced_size.argtypes = [C.c_void_p]
    lib.tscm_solver_reduced_size.restype = C.c_int
    lib.tscm_solver_reduced_system.argtypes = [C.c_void_p, C.c_double, c_double_p, c_double_p]
    lib.tscm_solver_reduced_system.restype = C.c_int
    lib.tscm_solver_reprojection_error.argtypes = [C.c_void_p, c_double_p, c_double_p, c_double_p]
    lib.tscm_solver_reprojection_error.restype = C.c_int
    lib.tscm_solver_covariance.argtypes = [C.c_void_p, P(TscmCovariance)]
    lib.tscm_solver_covariance.restype = C.c_int
    lib.tscm_compute_covariance.argtypes = [P(TscmProblem), P(TscmOptions), c_double_p, c_double_p,
                                            c_double_p, P(TscmCovariance), C.c_int]
    lib.tscm_compute_covariance.restype = C.c_int
    lib.tscm_solver_time_stage.argtypes = [C.c_void_p, C.c_int, C.c_int, c_double_p]
    lib.tscm_solver_time_stage.restype = C.c_int
    lib.tscm_solver_launch_count.argtypes = [C.c_void_p]
    lib.tscm_solver_launch_count.restype = C.c_int64
    lib.tscm_device_fp64_peak.argtypes = [C.c_int, c_double_p]
    lib.tscm_device_fp64_peak.restype = C.c_int
    lib.tscm_remap_tables.argtypes = [P(TscmRemapJob), C.c_int32, C.c_int32, C.c_int32,
                                      P(C.c_float), P(C.c_float), C.c_int, c_double_p]
    lib.tscm_remap_tables.restype = C.c_int
    lib.tscm_pose_graph_init.argtypes = [P(TscmPoseGraphProblem), C.c_int, P(TscmPoseGraphResult)]
    lib.tscm_pose_graph_init.restype = C.c_int
    lib.tscm_mono_init.argtypes = [P(TscmMonoInitProblem), C.c_int, P(TscmMonoInitResult)]
    lib.tscm_mono_init.restype = C.c_int
    lib.tscm_last_error.argtypes = []
    lib.tscm_last_error.restype = C.c_char_p
    lib.tscm_version.argtypes = []
    lib.tscm_version.restype = C.c_char_p
    if path is None:
        _lib = lib
    return lib


# Every symbol include/tscm.h declares (checked by tests/test_abi.py).
EXPORTED_SYMBOLS = [
    "tscm_options_init", "tscm_solve", "tscm_solver_create", "tscm_solver_destroy",
    "tscm_solver_set_options", "tscm_solver_set_parameters", "tscm_solver_get_parameters",
    "tscm_solver_set_observations", "tscm_solver_run", "tscm_comm_unique_id",
    "tscm_solver_attach_comm", "tscm_solver_p2p_export", "tscm_solver_p2p_attach", "tscm_solver_eval_jacobian", "tscm_solver_reduced_size",
    "tscm_solver_reduced_system", "tscm_solver_reprojection_error", "tscm_solver_time_stage",
    "tscm_solver_launch_count", "tscm_device_fp64_peak", "tscm_remap_tables",
    "tscm_last_error", "tscm_version", "tscm_cache_configure", "tscm_cache_release",
    "tscm_host_alloc", "tscm_host_free", "tscm_solver_set_exchange_timeout",
    "tscm_solver_set_schur_form", "tscm_set_debug", "tscm_pose_graph_init", "tscm_mono_init",
    "tscm_solver_covariance", "tscm_compute_covariance", "tscm_solver_set_reduced_solve",
]

ERR_RANK_DEFICIENT = 7   # TSCM_ERR_RANK_DEFICIENT

SCHUR_FORM = {"auto": 0, "rows": 1, "fused": 2, "pairs": 3}
REDUCED_SOLVE = {"auto": 0, "single": 1, "cluster": 2}


class TscmError(RuntimeError):
    def __init__(self, message: str, code: int = 0):
        super().__init__(message)
        self.code = code


def check(rc: int, lib=None):
    if rc != 0:
        lib = lib or load_library()
        msg = lib.tscm_last_error()
        raise TscmError(f"tscm error {rc}: {msg.decode() if msg else ''}", rc)


@dataclass
class CovarianceResult:
    """Output of tscm_solver_covariance / tscm_compute_covariance (include/tscm.h)."""
    camera: np.ndarray             # n x n, live order (tscm_solver_reduced_size)
    board: np.ndarray | None       # F x 6 x 6
    residual_variance: float       # sum |r|^2 / (2N - n_free), plain residuals
    kernel_ms: float


def _covariance_buffers(n: int, F: int, boards: bool):
    cam = np.zeros((n, n))
    brd = np.zeros((F, 6, 6)) if boards else None
    c = TscmCovariance(_dp(cam), _dp(brd) if boards else None, 0.0, 0.0)
    return cam, brd, c


def live_columns(problem: "ProblemArrays"):
    """(camera, index in [rt 6 | intrinsics 9]) of every live column of the reduced system."""
    cols = []
    for m in range(problem.num_cameras):
        ks = range(6, 13) if m == problem.fixed_camera else range(13)
        cols += [(m, k) for k in ks]
    return cols


def camera_std_dev(problem: "ProblemArrays", cov, residual_variance: float | None = None) -> np.ndarray:
    """C x 15 standard deviations [rt 6 | fx fy cx cy xi lambda alpha b c] in OpenCV's sense,
    sqrt(residual_variance * diag(Sigma)), from the live camera block (a CovarianceResult or the
    n x n matrix).  Entries that are not free (the fixed camera's rt, b, c) are 0."""
    if isinstance(cov, CovarianceResult):
        if residual_variance is None:
            residual_variance = cov.residual_variance
        cov = cov.camera
    out = np.zeros((problem.num_cameras, 15))
    d = np.diag(np.asarray(cov))
    for i, (m, k) in enumerate(live_columns(problem)):
        out[m, k] = np.sqrt(residual_variance * d[i])
    return out


class Solver:
    """Resident solver handle (observations stay in HBM)."""

    def __init__(self, problem: ProblemArrays, options: TscmOptions | None = None, device: int = -1,
                 schur_form: str | int | None = None):
        self.lib = load_library()
        self.problem = problem
        self.options = options or default_options()
        h = C.c_void_p()
        check(self.lib.tscm_solver_create(C.byref(problem.c), C.byref(self.options), device,
                                          C.byref(h)), self.lib)
        self.h = h
        if schur_form is not None:
            self.set_schur_form(schur_form)

    def set_schur_form(self, form):
        """Test hook (tscm_solver_set_schur_form): 'auto' | 'rows' | 'fused' | 'pairs'."""
        f = SCHUR_FORM[form] if isinstance(form, str) else int(form)
        check(self.lib.tscm_solver_set_schur_form(self.h, f), self.lib)

    def set_reduced_solve(self, form):
        """Test hook (tscm_solver_set_reduced_solve): 'auto' | 'single' | 'cluster'."""
        f = REDUCED_SOLVE[form] if isinstance(form, str) else int(form)
        check(self.lib.tscm_solver_set_reduced_solve(self.h, f), self.lib)

    def set_exchange_timeout(self, seconds: float):
        check(self.lib.tscm_solver_set_exchange_timeout(self.h, float(seconds)), self.lib)

    def close(self):
        if getattr(self, "h", None):
            self.lib.tscm_solver_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_options(self, options: TscmOptions):
        self.options = options
        check(self.lib.tscm_solver_set_options(self.h, C.byref(options)), self.lib)

    def set_parameters(self, intrinsics, cam_rt, board_rt):
        a = np.ascontiguousarray(intrinsics, dtype=np.float64)
        b = np.ascontiguousarray(cam_rt, dtype=np.float64)
        c = np.ascontiguousarray(board_rt, dtype=np.float64)
        assert a.size == 9 * self.problem.num_cameras and b.size == 6 * self.problem.num_cameras
        assert c.size == 6 * self.problem.num_frames
        check(self.lib.tscm_solver_set_parameters(self.h, _dp(a), _dp(b), _dp(c)), self.lib)

    def get_parameters(self):
        Cn, F = self.problem.num_cameras, self.problem.num_frames
        a, b, c = np.zeros((Cn, 9)), np.zeros((Cn, 6)), np.zeros((F, 6))
        check(self.lib.tscm_solver_get_parameters(self.h, _dp(a), _dp(b), _dp(c)), self.lib)
        return a, b, c

    def set_observations(self, obs_xy):
        o = np.ascontiguousarray(obs_xy, dtype=np.float64)
        assert o.size == self.problem.num_observations * 2
        check(self.lib.tscm_solver_set_observations(self.h, _dp(o)), self.lib)

    def run(self, trace_capacity: int | None = None) -> SummaryResult:
        cap = trace_capacity if trace_capacity is not None else self.options.max_num_iterations + 2
        buf = SummaryBuffers(cap)
        check(self.lib.tscm_solver_run(self.h, C.byref(buf.c)), self.lib)
        return buf.result()

    def attach_comm(self, rank: int, num_ranks: int, unique_id: bytes):
        assert len(unique_id) == 128
        b = C.create_string_buffer(unique_id, 128)
        check(self.lib.tscm_solver_attach_comm(self.h, rank, num_ranks, b), self.lib)

    def p2p_export(self) -> bytes:
        """64-byte CUDA-IPC handle of this rank's exchange mailbox."""
        b = C.create_string_buffer(64)
        check(self.lib.tscm_solver_p2p_export(self.h, b), self.lib)
        return b.raw

    def p2p_attach(self, rank: int, num_ranks: int, handles: bytes):
        """handles: the p2p_export() of every rank, concatenated in rank order."""
        assert len(handles) == 64 * num_ranks
        b = C.create_string_buffer(handles, len(handles))
        check(self.lib.tscm_solver_p2p_attach(self.h, rank, num_ranks, b), self.lib)

    def eval_jacobian(self, want_jacobian=True):
        N = self.problem.num_observations
        r = np.zeros((N, 2))
        J = np.zeros((N, 2, 21)) if want_jacobian else None
        cost = C.c_double()
        check(self.lib.tscm_solver_eval_jacobian(self.h, _dp(r), _dp(J) if want_jacobian else None,
                                                 C.byref(cost)), self.lib)
        return r, J, cost.value

    def reduced_size(self) -> int:
        return self.lib.tscm_solver_reduced_size(self.h)

    def reduced_system(self, radius: float):
        n = self.reduced_size()
        lhs, rhs = np.zeros((n, n)), np.zeros(n)
        check(self.lib.tscm_solver_reduced_system(self.h, radius, _dp(lhs), _dp(rhs)), self.lib)
        return lhs, rhs

    def reprojection_error(self):
        per = np.zeros(self.problem.num_cameras)
        overall, rms = C.c_double(), C.c_double()
        check(self.lib.tscm_solver_reprojection_error(self.h, _dp(per), C.byref(overall),
                                                      C.byref(rms)), self.lib)
        return per, overall.value, rms.value

    def covariance(self, boards: bool = True) -> CovarianceResult:
        """tscm_solver_covariance(): covariance of the live parameters at the current point.
        Raises TscmError with code ERR_RANK_DEFICIENT when J^T J is singular."""
        cam, brd, c = _covariance_buffers(self.reduced_size(), self.problem.num_frames, boards)
        check(self.lib.tscm_solver_covariance(self.h, C.byref(c)), self.lib)
        return CovarianceResult(cam, brd, c.residual_variance, c.kernel_ms)

    def time_stage(self, stage: int, repeats: int) -> float:
        ms = C.c_double()
        check(self.lib.tscm_solver_time_stage(self.h, stage, repeats, C.byref(ms)), self.lib)
        return ms.value

    def launch_count(self) -> int:
        return int(self.lib.tscm_solver_launch_count(self.h))


def device_fp64_peak(device: int = -1) -> float:
    lib = load_library()
    v = C.c_double()
    check(lib.tscm_device_fp64_peak(device, C.byref(v)), lib)
    return v.value


def remap_job(intrinsics, matrix, ray, size, origin=(0, 0), offset=(0.0, 0.0), cutoff_w2=0.0) -> TscmRemapJob:
    """ray = (fx, fy, cx, cy) of the output pixel grid; size = (width, height);
    origin = (row0, col0) of the block in the maps."""
    j = TscmRemapJob()
    j.intrinsics[:] = [float(v) for v in np.asarray(intrinsics, dtype=np.float64).reshape(9)]
    j.matrix[:] = [float(v) for v in np.asarray(matrix, dtype=np.float64).reshape(9)]
    j.ray_fx, j.ray_fy, j.ray_cx, j.ray_cy = (float(v) for v in ray)
    j.offset_x, j.offset_y = float(offset[0]), float(offset[1])
    j.cutoff_w2 = float(cutoff_w2)
    j.width, j.height = int(size[0]), int(size[1])
    j.row0, j.col0 = int(origin[0]), int(origin[1])
    return j


def remap_tables(jobs, map_size, device: int = -1, mapx=None, mapy=None):
    """tscm_remap_tables(): fill CV_32FC1 tables (map_size = (width, height)) on the GPU.
    Returns (mapx, mapy, kernel_ms)."""
    lib = load_library()
    W, H = int(map_size[0]), int(map_size[1])
    mapx = np.zeros((H, W), dtype=np.float32) if mapx is None else mapx
    mapy = np.zeros((H, W), dtype=np.float32) if mapy is None else mapy
    assert mapx.shape == (H, W) and mapy.shape == (H, W) and mapx.dtype == np.float32
    arr = (TscmRemapJob * len(jobs))(*jobs)
    ms = C.c_double()
    check(lib.tscm_remap_tables(arr, len(jobs), W, H, mapx.ctypes.data_as(C.POINTER(C.c_float)),
                                mapy.ctypes.data_as(C.POINTER(C.c_float)), device, C.byref(ms)), lib)
    return mapx, mapy, ms.value


class PoseGraphResult:
    """Output of pose_graph_init(): poses as 12 doubles = R row-major | t."""

    def __init__(self, C_, B):
        self.camera_pose = np.zeros((C_, 12))
        self.board_pose = np.zeros((B, 12))
        self.board_init = np.zeros(B, dtype=np.uint8)
        self.camera_choice = np.full(C_, -1, dtype=np.int32)
        self.board_choice = np.full(B, -1, dtype=np.int32)
        self.camera_candidate_error = np.full((C_, B), np.nan)
        self.board_candidate_error = np.full((B, C_), np.nan)
        self.kernel_ms = 0.0
        self.projections = 0


def pose_graph_init(worlds, intrinsics, has, mono_rt, pixels, device: int = -1) -> PoseGraphResult:
    """tscm_pose_graph_init(): MultiCalib's constructor (multi_calib.cpp:6-153) with the candidate
    scoring on the GPU.  has [C][B], mono_rt [C][B][3][3], pixels [C][B][K][2], worlds [K][3]."""
    lib = load_library()
    has = np.ascontiguousarray(has, dtype=np.uint8)
    C_, B = has.shape
    worlds = np.ascontiguousarray(worlds, dtype=np.float64).reshape(-1, 3)
    K = worlds.shape[0]
    intr = np.ascontiguousarray(intrinsics, dtype=np.float64).reshape(C_, 9)
    rt = np.ascontiguousarray(mono_rt, dtype=np.float64).reshape(C_, B, 9)
    px = np.ascontiguousarray(pixels, dtype=np.float64).reshape(C_, B, K, 2)
    u8p = C.POINTER(C.c_uint8)
    prob = TscmPoseGraphProblem(C_, B, K, _dp(worlds), _dp(intr), has.ctypes.data_as(u8p), _dp(rt), _dp(px))
    r = PoseGraphResult(C_, B)
    res = TscmPoseGraphResult(_dp(r.camera_pose), _dp(r.board_pose), r.board_init.ctypes.data_as(u8p),
                              _ip(r.camera_choice), _ip(r.board_choice), _dp(r.camera_candidate_error),
                              _dp(r.board_candidate_error), 0.0, 0)
    check(lib.tscm_pose_graph_init(C.byref(prob), device, C.byref(res)), lib)
    r.kernel_ms, r.projections = res.kernel_ms, res.projections
    return r


class MonoInitResult:
    """Output of mono_init(): intrinsics [9], Rt [F][3][3], frame_ok [F]."""

    def __init__(self, F):
        self.intrinsics = np.zeros(9)
        self.Rt = np.zeros((F, 3, 3))
        self.frame_ok = np.zeros(F, dtype=np.uint8)
        self.rows_used = 0
        self.kernel_ms = 0.0


def mono_init(board, image, worlds, has, pixels, guess=None, device: int = -1) -> MonoInitResult:
    """tscm_mono_init(): TripleSphereCamera::calibrate up to the refinement (TS.cpp:36-52,
    110-203) on the GPU.  board = (W, H), image = (w, h), pixels [F][K][2]; guess: 7 or 9
    intrinsics of the has_init_guess_ path, None for the cold start."""
    lib = load_library()
    has = np.ascontiguousarray(has, dtype=np.uint8)
    F = has.shape[0]
    W, H = int(board[0]), int(board[1])
    worlds = np.ascontiguousarray(worlds, dtype=np.float64).reshape(W * H, 3)
    px = np.ascontiguousarray(pixels, dtype=np.float64).reshape(F, W * H, 2)
    r = MonoInitResult(F)
    u8p = C.POINTER(C.c_uint8)
    prob = TscmMonoInitProblem(F, W, H, int(image[0]), int(image[1]), _dp(worlds), has.ctypes.data_as(u8p), _dp(px),
                               0 if guess is None else 1)
    res = TscmMonoInitResult()
    if guess is not None:
        for k, v in enumerate(guess):
            res.intrinsics[k] = float(v)
    res.mono_rt = _dp(r.Rt)
    res.frame_ok = r.frame_ok.ctypes.data_as(u8p)
    check(lib.tscm_mono_init(C.byref(prob), device, C.byref(res)), lib)
    r.intrinsics[:] = list(res.intrinsics)
    r.rows_used, r.kernel_ms = res.focal_rows_used, res.kernel_ms
    return r


def comm_unique_id() -> bytes:
    lib = load_library()
    b = C.create_string_buffer(128)
    check(lib.tscm_comm_unique_id(b), lib)
    return b.raw


def solve(problem: ProblemArrays, intrinsics, cam_rt, board_rt, options: TscmOptions | None = None,
          device: int = -1):
    """One-shot host-buffer solve through tscm_solve() — what a reference
    adapter calls in place of ceres::Solve.  Returns (intr, cam_rt, board_rt, summary)."""
    lib = load_library()
    options = options or default_options()
    a = np.array(intrinsics, dtype=np.float64, order="C").reshape(problem.num_cameras, 9)
    b = np.array(cam_rt, dtype=np.float64, order="C").reshape(problem.num_cameras, 6)
    c = np.array(board_rt, dtype=np.float64, order="C").reshape(problem.num_frames, 6)
    buf = SummaryBuffers(options.max_num_iterations + 2)
    check(lib.tscm_solve(C.byref(problem.c), C.byref(options), _dp(a), _dp(b), _dp(c),
                         C.byref(buf.c), device), lib)
    return a, b, c, buf.result()


def covariance(problem: ProblemArrays, intrinsics, cam_rt, board_rt, options: TscmOptions | None = None,
               device: int = -1, boards: bool = True) -> CovarianceResult:
    """One-shot tscm_compute_covariance() at the given parameters, through the solver cache of
    solve(): after a solve() of the same structure only the data are uploaded."""
    lib = load_library()
    options = options or default_options()
    a = np.ascontiguousarray(intrinsics, dtype=np.float64).reshape(problem.num_cameras, 9)
    b = np.ascontiguousarray(cam_rt, dtype=np.float64).reshape(problem.num_cameras, 6)
    c = np.ascontiguousarray(board_rt, dtype=np.float64).reshape(problem.num_frames, 6)
    n = sum(7 if m == problem.fixed_camera else 13 for m in range(problem.num_cameras))
    cam, brd, cv = _covariance_buffers(n, problem.num_frames, boards)
    check(lib.tscm_compute_covariance(C.byref(problem.c), C.byref(options), _dp(a), _dp(b), _dp(c),
                                      C.byref(cv), device), lib)
    return CovarianceResult(cam, brd, cv.residual_variance, cv.kernel_ms)


def solve_resident(problem: ProblemArrays, intrinsics, cam_rt, board_rt, options: TscmOptions | None = None,
                   device: int = -1, schur_form=None):
    """The same solve through a resident Solver handle (create / set / run / get / destroy),
    optionally with a forced Schur form.  Returns (intr, cam_rt, board_rt, summary)."""
    s = Solver(problem, options, device=device, schur_form=schur_form)
    try:
        s.set_parameters(intrinsics, cam_rt, board_rt)
        res = s.run()
        a, b, c = s.get_parameters()
    finally:
        s.close()
    return a, b, c, res


def set_debug(flags: int):
    load_library().tscm_set_debug(int(flags))


def cache_release():
    load_library().tscm_cache_release()


def cache_configure(max_solvers: int):
    load_library().tscm_cache_configure(int(max_solvers))


def pinned_array(shape, dtype=np.float64) -> np.ndarray:
    """numpy array over page-locked memory from tscm_host_alloc() (kept alive by the array)."""
    lib = load_library()
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = lib.tscm_host_alloc(max(1, n))
    if not p:
        raise TscmError("tscm_host_alloc failed")

    class _Owner:
        def __init__(self, ptr): self.ptr = ptr
        def __del__(self):
            try:
                lib.tscm_host_free(self.ptr)
            except Exception:
                pass
    buf = (C.c_char * max(1, n)).from_address(p)
    buf._owner = _Owner(p)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def attach_ranks(solver: "Solver", rank: int, world: int, use_p2p: bool | None = None):
    """Make `solver` one rank of a frame-sharded solve inside an initialised
    torch.distributed NCCL process group (one process per GPU of one node).
    Peer-memory exchange (tscm_p2p.cuh) when world <= 8 unless use_p2p=False; NCCL otherwise."""
    import torch
    import torch.distributed as dist
    if use_p2p is None:
        use_p2p = world <= 8
    if use_p2p:
        mine = torch.frombuffer(bytearray(solver.p2p_export()), dtype=torch.uint8).cuda()
        allh = [torch.zeros(64, dtype=torch.uint8, device="cuda") for _ in range(world)]
        dist.all_gather(allh, mine)
        solver.p2p_attach(rank, world, b"".join(bytes(h.cpu().numpy().tobytes()) for h in allh))
        dist.barrier()      # every rank has mapped every mailbox before the first exchange
    else:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        solver.attach_comm(rank, world, bytes(uid.cpu().numpy().tobytes()))
