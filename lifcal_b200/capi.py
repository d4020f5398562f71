"""ctypes mirror of include/lfba.h and include/lfba_scene.h.

Thin binding only: every compute call goes through the C ABI of ``liblfba.so`` (hand-written CUDA for
sm_100a).  There is deliberately no Python/NumPy/torch fallback: if the shared library or a usable GPU is
missing, calls raise :class:`LfbaError`.

Reference seam: ``CameraCalibration::performBundleAdjustment`` (src/CameraCalibration.cpp:774-992).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

MAX_CAMERA_PARAMETERS = 17
CFG_NRADIAL_MASK = 0x3
CFG_TANGENTIAL = 0x4
CFG_REFINE_POSES = 0x100
CFG_ROBUST = 0x200
CFG_REFINE_POINTS = 0x400
CFG_MLADJ = 0x800
CALIBRATION_ARUCO = 0
RECALIBRATION = 1

OK, INVALID_ARGUMENT, NO_DEVICE, CUDA_ERROR, NCCL_ERROR, OUT_OF_MEMORY, FAILURE = range(7)
NUM_KERNEL_TIMERS = 12
KERNEL_TIMER_NAMES = ["lens_pose_tables", "eval_tracks", "schur_points", "allreduce", "damping", "cholesky",
                      "backsolve", "point_step", "control", "misc", "r10", "r11"]

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)


class LfbaError(RuntimeError):
    pass


class Problem(C.Structure):
    _fields_ = [
        ("config", C.c_uint32), ("calib_type", C.c_int32),
        ("spx", C.c_double), ("spy", C.c_double), ("scale", C.c_double),
        ("n_obs", C.c_int64), ("n_frames", C.c_int32), ("n_points", C.c_int32),
        ("obs_x", c_double_p), ("obs_y", c_double_p), ("ml_x", c_double_p), ("ml_y", c_double_p),
        ("point_idx", c_int32_p), ("frame_idx", c_int32_p),
        ("n_constraints", C.c_int32),
        ("c_p1", c_int32_p), ("c_p2", c_int32_p), ("c_dist", c_double_p), ("c_sigma", c_double_p),
    ]


class Options(C.Structure):
    _fields_ = [
        ("max_num_iterations", C.c_int32),
        ("function_tolerance", C.c_double), ("parameter_tolerance", C.c_double),
        ("gradient_tolerance", C.c_double),
        ("initial_trust_region_radius", C.c_double), ("max_trust_region_radius", C.c_double),
        ("min_trust_region_radius", C.c_double), ("min_relative_decrease", C.c_double),
        ("min_lm_diagonal", C.c_double), ("max_lm_diagonal", C.c_double),
        ("max_num_consecutive_invalid_steps", C.c_int32),
        ("loss_scale", C.c_double),
        ("minimizer_progress_to_stdout", C.c_int32),
        ("device", C.c_int32), ("num_gpus", C.c_int32), ("profile", C.c_int32),
        ("emulate_shards", C.c_int32), ("reserved", C.c_int32 * 7),
    ]


class Iteration(C.Structure):
    _fields_ = [
        ("iteration", C.c_int32), ("step_is_valid", C.c_int32), ("step_is_successful", C.c_int32),
        ("line_search_iterations", C.c_int32),
        ("cost", C.c_double), ("cost_change", C.c_double), ("gradient_max_norm", C.c_double),
        ("gradient_norm", C.c_double), ("step_norm", C.c_double), ("relative_decrease", C.c_double),
        ("trust_region_radius", C.c_double), ("iteration_time_s", C.c_double),
        ("cumulative_time_s", C.c_double),
    ]


class Summary(C.Structure):
    _fields_ = [
        ("termination_type", C.c_int32), ("stop_reason", C.c_int32), ("num_iterations", C.c_int32),
        ("num_successful_steps", C.c_int32), ("num_unsuccessful_steps", C.c_int32),
        ("reduced_system_size", C.c_int32),
        ("initial_cost", C.c_double), ("final_cost", C.c_double),
        ("num_jacobian_evals", C.c_int64), ("num_observations", C.c_int64), ("num_tracks", C.c_int64),
        ("num_lenses", C.c_int64), ("gpu_launches", C.c_int64),
        ("setup_time_s", C.c_double), ("solve_time_s", C.c_double), ("solve_gpu_ms", C.c_double),
        ("kernel_ms", C.c_double * NUM_KERNEL_TIMERS), ("kernel_calls", C.c_int64 * NUM_KERNEL_TIMERS),
        ("iterations", C.POINTER(Iteration)), ("iterations_capacity", C.c_int32), ("reserved_i", C.c_int32),
        ("h2d_bytes", C.c_int64), ("h2d_ms", C.c_double),
    ]


class ReprojStats(C.Structure):
    _fields_ = [("std_x", C.c_double), ("std_y", C.c_double), ("mae_x", C.c_double), ("mae_y", C.c_double),
                ("num_points", C.c_int64), ("num_inliers", C.c_int64)]


GAUGE_NONE, GAUGE_FIRST_FRAME = 0, 1


class CovarianceInfo(C.Structure):
    _fields_ = [("gauge", C.c_int32), ("gauge_frame", C.c_int32), ("n_reduced", C.c_int32), ("reserved_i", C.c_int32),
                ("num_residuals", C.c_int64), ("num_free_parameters", C.c_int64),
                ("cost", C.c_double), ("sigma2", C.c_double), ("gpu_ms", C.c_double), ("selinv_ms", C.c_double),
                ("points_ms", C.c_double), ("reserved", C.c_double * 1)]


class Comm(C.Structure):
    _fields_ = [("rank", C.c_int32), ("nranks", C.c_int32), ("nccl_unique_id", C.c_char * 128), ("handle", C.c_void_p)]


c_float_p = C.POINTER(C.c_float)


class LensGridStruct(C.Structure):
    _fields_ = [("raw_width", C.c_int32), ("raw_height", C.c_int32), ("scale", C.c_int32),
                ("lens_diameter", C.c_float), ("lens_validity_radius_2", C.c_float), ("rotation", C.c_float),
                ("rotation_on_grid", C.c_int32), ("n_lenses", C.c_int32),
                ("lens_cx", c_float_p), ("lens_cy", c_float_p), ("map_next", c_int32_p), ("map_ml", c_int32_p)]


class LensGrid:
    """NumPy-owning mirror of lfba_lens_grid: what projectPointsToRawImage reads from the reference's MicroLensGrid."""

    def __init__(self, raw_width, raw_height, scale, lens_diameter, rotation, rotation_on_grid, lens_cx, lens_cy,
                 map_next, map_ml, lens_border=1.0):
        self.raw_width, self.raw_height, self.scale = int(raw_width), int(raw_height), int(scale)
        self.lens_diameter = np.float32(lens_diameter)
        r = np.float32(self.lens_diameter * np.float32(0.5) - np.float32(lens_border))  # MicroLensGrid.cpp:110-111
        self.lens_validity_radius_2 = np.float32(r * r)
        self.rotation, self.rotation_on_grid = np.float32(rotation), int(bool(rotation_on_grid))
        self.lens_cx = np.ascontiguousarray(lens_cx, np.float32)
        self.lens_cy = np.ascontiguousarray(lens_cy, np.float32)
        self.map_next = np.ascontiguousarray(map_next, np.int32).ravel()
        self.map_ml = np.ascontiguousarray(map_ml, np.int32).ravel()
        assert self.map_next.size == self.raw_width * self.raw_height == self.map_ml.size

    def as_struct(self) -> LensGridStruct:
        g = LensGridStruct()
        g.raw_width, g.raw_height, g.scale = self.raw_width, self.raw_height, self.scale
        g.lens_diameter, g.lens_validity_radius_2 = float(self.lens_diameter), float(self.lens_validity_radius_2)
        g.rotation, g.rotation_on_grid, g.n_lenses = float(self.rotation), self.rotation_on_grid, int(self.lens_cx.size)
        g.lens_cx = self.lens_cx.ctypes.data_as(c_float_p)
        g.lens_cy = self.lens_cy.ctypes.data_as(c_float_p)
        g.map_next, g.map_ml = _ip(self.map_next), _ip(self.map_ml)
        return g


class SceneSpec(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("n_points", C.c_int32), ("n_frames", C.c_int32), ("window", C.c_int32),
        ("config", C.c_uint32), ("calib_type", C.c_int32), ("n_constraints", C.c_int32),
        ("max_lenses", C.c_int32), ("order", C.c_int32), ("point_begin", C.c_int32), ("point_end", C.c_int32),
        ("noise_px", C.c_double), ("outlier_fraction", C.c_double), ("outlier_px", C.c_double),
        ("init_intrinsics_rel", C.c_double), ("init_center_px", C.c_double), ("init_angle_rad", C.c_double),
        ("init_trans_mm", C.c_double), ("init_point_mm", C.c_double),
        ("num_threads", C.c_int32), ("reserved", C.c_int32 * 7),
    ]


def _dp(a: Optional[np.ndarray]):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_double_p)


def _ip(a: Optional[np.ndarray]):
    if a is None:
        return None
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_int32_p)


class ProblemArrays:
    """Owns NumPy copies of the arrays an lfba_problem points to."""

    def __init__(self, config, calib_type, spx, spy, scale, n_frames, n_points, obs_x, obs_y, ml_x, ml_y,
                 point_idx, frame_idx, c_p1=None, c_p2=None, c_dist=None, c_sigma=None):
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        self.config, self.calib_type = int(config), int(calib_type)
        self.spx, self.spy, self.scale = float(spx), float(spy), float(scale)
        self.n_frames, self.n_points = int(n_frames), int(n_points)
        self.obs_x, self.obs_y, self.ml_x, self.ml_y = f64(obs_x), f64(obs_y), f64(ml_x), f64(ml_y)
        self.point_idx, self.frame_idx = i32(point_idx), i32(frame_idx)
        nc = 0 if c_p1 is None else len(c_p1)
        self.c_p1 = i32(c_p1 if nc else [])
        self.c_p2 = i32(c_p2 if nc else [])
        self.c_dist = f64(c_dist if nc else [])
        self.c_sigma = f64(c_sigma if nc else [])

    @property
    def n_obs(self):
        return int(self.obs_x.shape[0])

    def subset(self, mask_or_index):
        """Same problem restricted to a subset of the observations (used for sharding tests)."""
        s = mask_or_index
        return ProblemArrays(self.config, self.calib_type, self.spx, self.spy, self.scale, self.n_frames,
                             self.n_points, self.obs_x[s], self.obs_y[s], self.ml_x[s], self.ml_y[s],
                             self.point_idx[s], self.frame_idx[s], self.c_p1, self.c_p2, self.c_dist,
                             self.c_sigma)

    def with_config(self, config, calib_type=None):
        return ProblemArrays(config, self.calib_type if calib_type is None else calib_type, self.spx, self.spy,
                             self.scale, self.n_frames, self.n_points, self.obs_x, self.obs_y, self.ml_x,
                             self.ml_y, self.point_idx, self.frame_idx, self.c_p1, self.c_p2, self.c_dist,
                             self.c_sigma)

    def as_struct(self) -> Problem:
        p = Problem()
        p.config, p.calib_type = self.config, self.calib_type
        p.spx, p.spy, p.scale = self.spx, self.spy, self.scale
        p.n_obs, p.n_frames, p.n_points = self.n_obs, self.n_frames, self.n_points
        p.obs_x, p.obs_y, p.ml_x, p.ml_y = _dp(self.obs_x), _dp(self.obs_y), _dp(self.ml_x), _dp(self.ml_y)
        p.point_idx, p.frame_idx = _ip(self.point_idx), _ip(self.frame_idx)
        p.n_constraints = int(self.c_p1.shape[0])
        p.c_p1, p.c_p2, p.c_dist, p.c_sigma = _ip(self.c_p1), _ip(self.c_p2), _dp(self.c_dist), _dp(self.c_sigma)
        return p


def summary_to_dict(s: Summary, rows) -> dict:
    n = min(s.num_iterations, len(rows))
    fields = [f for f, _ in Iteration._fields_]
    return {
        "termination_type": s.termination_type, "stop_reason": s.stop_reason,
        "num_iterations": s.num_iterations, "num_successful_steps": s.num_successful_steps,
        "num_unsuccessful_steps": s.num_unsuccessful_steps, "reduced_system_size": s.reduced_system_size,
        "initial_cost": s.initial_cost, "final_cost": s.final_cost,
        "num_jacobian_evals": s.num_jacobian_evals, "num_observations": s.num_observations,
        "num_tracks": s.num_tracks, "num_lenses": s.num_lenses, "gpu_launches": s.gpu_launches,
        "setup_time_s": s.setup_time_s, "solve_time_s": s.solve_time_s, "solve_gpu_ms": s.solve_gpu_ms,
        "h2d_bytes": s.h2d_bytes, "h2d_ms": s.h2d_ms,
        "h2d_gbs": (s.h2d_bytes / (s.h2d_ms * 1e-3) / 1e9) if s.h2d_ms > 0 else None,
        "kernel_ms": {KERNEL_TIMER_NAMES[i]: s.kernel_ms[i] for i in range(NUM_KERNEL_TIMERS) if s.kernel_calls[i]},
        "kernel_calls": {KERNEL_TIMER_NAMES[i]: s.kernel_calls[i] for i in range(NUM_KERNEL_TIMERS) if s.kernel_calls[i]},
        "iterations": [{f: getattr(rows[i], f) for f in fields} for i in range(n)],
    }


def new_summary(capacity: int = 256):
    rows = (Iteration * capacity)()
    s = Summary()
    s.iterations = C.cast(rows, C.POINTER(Iteration))
    s.iterations_capacity = capacity
    return s, rows


# ---------------------------------------------------------------------------------------------------
# scene generator (host-only library)
# ---------------------------------------------------------------------------------------------------
_scene_lib = None


def scene_lib():
    global _scene_lib
    if _scene_lib is None:
        path = os.path.join(_HERE, "liblfba_scene.so")
        if not os.path.exists(path):
            raise LfbaError(f"{path} not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
        lib = C.CDLL(path)
        lib.lfba_scene_spec_init.argtypes = [C.POINTER(SceneSpec)]
        lib.lfba_scene_spec_preset.argtypes = [C.POINTER(SceneSpec), C.c_int]
        lib.lfba_scene_create.argtypes = [C.POINTER(SceneSpec)]
        lib.lfba_scene_create.restype = C.c_void_p
        lib.lfba_scene_destroy.argtypes = [C.c_void_p]
        lib.lfba_scene_problem.argtypes = [C.c_void_p, C.POINTER(Problem)]
        for n in ("camera_init", "views_init", "points_init", "camera_true", "views_true", "points_true"):
            fn = getattr(lib, "lfba_scene_" + n)
            fn.argtypes = [C.c_void_p]
            fn.restype = c_double_p
        lib.lfba_scene_num_tracks.argtypes = [C.c_void_p]
        lib.lfba_scene_num_tracks.restype = C.c_int64
        _scene_lib = lib
    return _scene_lib


class Scene:
    """A generated synthetic scene; arrays are copied into NumPy so the C object can be freed."""

    def __init__(self, spec: SceneSpec):
        lib = scene_lib()
        h = lib.lfba_scene_create(C.byref(spec))
        if not h:
            raise LfbaError("lfba_scene_create failed")
        try:
            p = Problem()
            lib.lfba_scene_problem(h, C.byref(p))
            n, F, P, K = p.n_obs, p.n_frames, p.n_points, p.n_constraints
            cp = lambda ptr, cnt, dt: (np.ctypeslib.as_array(ptr, shape=(cnt,)).astype(dt, copy=True)
                                       if cnt > 0 else np.zeros(0, dt))
            self.problem = ProblemArrays(
                p.config, p.calib_type, p.spx, p.spy, p.scale, F, P,
                cp(p.obs_x, n, np.float64), cp(p.obs_y, n, np.float64), cp(p.ml_x, n, np.float64),
                cp(p.ml_y, n, np.float64), cp(p.point_idx, n, np.int32), cp(p.frame_idx, n, np.int32),
                cp(p.c_p1, K, np.int32), cp(p.c_p2, K, np.int32), cp(p.c_dist, K, np.float64),
                cp(p.c_sigma, K, np.float64))
            self.camera_init = cp(lib.lfba_scene_camera_init(h), 17, np.float64)
            self.views_init = cp(lib.lfba_scene_views_init(h), 6 * F, np.float64)
            self.points_init = cp(lib.lfba_scene_points_init(h), 3 * P, np.float64)
            self.camera_true = cp(lib.lfba_scene_camera_true(h), 17, np.float64)
            self.views_true = cp(lib.lfba_scene_views_true(h), 6 * F, np.float64)
            self.points_true = cp(lib.lfba_scene_points_true(h), 3 * P, np.float64)
            self.num_tracks = int(lib.lfba_scene_num_tracks(h))
            self.spec = spec
        finally:
            lib.lfba_scene_destroy(h)


def scene_spec(preset: Optional[int] = None, **kw) -> SceneSpec:
    lib = scene_lib()
    s = SceneSpec()
    if preset is None:
        lib.lfba_scene_spec_init(C.byref(s))
    elif lib.lfba_scene_spec_preset(C.byref(s), int(preset)) != 0:
        raise LfbaError(f"unknown scene preset {preset}")
    for k, v in kw.items():
        if not hasattr(s, k):
            raise AttributeError(k)
        setattr(s, k, v)
    return s


def make_scene(preset: Optional[int] = None, **kw) -> Scene:
    return Scene(scene_spec(preset, **kw))
