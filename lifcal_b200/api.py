"""Python host-side mirror of the C ABI (include/lfba.h) over ctypes.

Every call goes to liblfba.so (hand-written CUDA, sm_100a). No fallback of any kind: a missing library raises
at load(), a missing GPU makes every compute call raise LfbaError(LFBA_NO_DEVICE).

Mirrors the reference seam CameraCalibration::performBundleAdjustment (src/CameraCalibration.cpp:774-992):
``solve(problem, camera17, views6F, points3P)`` takes what that function reads and returns what it writes.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import capi
from .capi import LfbaError

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

_EXPORTS = ["lfba_version", "lfba_last_error", "lfba_status_string", "lfba_options_init", "lfba_device_count", "lfba_trim_cache",
            "lfba_solve", "lfba_eval", "lfba_comm_unique_id", "lfba_comm_create", "lfba_comm_destroy", "lfba_solver_create", "lfba_solver_set_parameters",
            "lfba_solver_get_parameters", "lfba_solver_run", "lfba_solver_time_eval", "lfba_solver_track_blocks",
            "lfba_measure_fp64_peak", "lfba_solver_destroy", "lfba_project_to_raw", "lfba_epipolar_web", "lfba_init_plenoptic",
            "lfba_solver_covariance", "lfba_covariance", "lfba_solver_covariance_points", "lfba_covariance_points"]


def load():
    """Load liblfba.so and bind every symbol include/lfba.h declares (raises if any is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.path.join(_HERE, "liblfba.so")
    if not os.path.exists(path):
        raise LfbaError(f"{path} is not built: run `python -c 'import __graft_entry__ as g; g.build()'`. "
                        "There is no CPU fallback.")
    L = C.CDLL(path)
    for name in _EXPORTS:
        if not hasattr(L, name):
            raise LfbaError(f"liblfba.so does not export {name}")
    dp, ip = capi.c_double_p, capi.c_int32_p
    L.lfba_version.restype = C.c_int
    L.lfba_last_error.restype = C.c_char_p
    L.lfba_status_string.restype = C.c_char_p
    L.lfba_status_string.argtypes = [C.c_int]
    L.lfba_options_init.argtypes = [C.POINTER(capi.Options)]
    L.lfba_device_count.restype = C.c_int
    L.lfba_solve.argtypes = [C.POINTER(capi.Problem), C.POINTER(capi.Options), dp, dp, dp, C.POINTER(capi.Summary)]
    L.lfba_eval.argtypes = [C.POINTER(capi.Problem), C.POINTER(capi.Options), dp, dp, dp, dp, dp, dp, dp, dp,
                            C.POINTER(capi.ReprojStats), C.c_double]
    L.lfba_comm_unique_id.argtypes = [C.c_char_p]
    L.lfba_comm_create.argtypes = [C.POINTER(capi.Comm), C.POINTER(C.c_void_p)]
    L.lfba_comm_destroy.argtypes = [C.c_void_p]
    L.lfba_solver_create.argtypes = [C.POINTER(capi.Problem), C.POINTER(capi.Options), C.POINTER(capi.Comm),
                                     C.POINTER(C.c_void_p)]
    L.lfba_solver_set_parameters.argtypes = [C.c_void_p, dp, dp, dp]
    L.lfba_solver_get_parameters.argtypes = [C.c_void_p, dp, dp, dp]
    L.lfba_solver_run.argtypes = [C.c_void_p, C.POINTER(capi.Summary)]
    L.lfba_solver_time_eval.argtypes = [C.c_void_p, C.c_int, C.c_int, dp]
    L.lfba_solver_track_blocks.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32), dp, dp, ip, ip]
    L.lfba_measure_fp64_peak.argtypes = [C.c_int, dp]
    L.lfba_solver_destroy.argtypes = [C.c_void_p]
    i64p = C.POINTER(C.c_int64)
    L.lfba_project_to_raw.argtypes = [C.POINTER(capi.LensGridStruct), C.c_int64, dp, dp, dp, ip, ip, C.c_int64, dp, dp, dp, dp,
                                      ip, ip, i64p, C.c_int32]
    L.lfba_epipolar_web.argtypes = [C.c_float, C.c_float, C.c_int32, ip, ip, dp, ip]
    L.lfba_init_plenoptic.argtypes = [C.c_double, C.c_double, C.c_int64, dp, ip, ip, C.c_int32, dp, C.c_int32, dp, dp, dp, dp,
                                      C.c_int32]
    L.lfba_solver_covariance.argtypes = [C.c_void_p, dp, dp, C.POINTER(capi.CovarianceInfo)]
    L.lfba_covariance.argtypes = [C.POINTER(capi.Problem), C.POINTER(capi.Options), dp, dp, dp, dp, dp,
                                  C.POINTER(capi.CovarianceInfo)]
    L.lfba_solver_covariance_points.argtypes = [C.c_void_p, dp, dp, dp, C.POINTER(capi.CovarianceInfo)]
    L.lfba_covariance_points.argtypes = [C.POINTER(capi.Problem), C.POINTER(capi.Options), dp, dp, dp, dp, dp, dp,
                                         C.POINTER(capi.CovarianceInfo)]
    _lib = L
    return L


def _check(rc: int, what: str):
    if rc != capi.OK:
        L = load()
        msg = L.lfba_last_error().decode(errors="replace")
        raise LfbaError(f"{what}: {L.lfba_status_string(rc).decode()} (status {rc}): {msg}")


def version() -> int:
    return load().lfba_version()


def device_count() -> int:
    return load().lfba_device_count()


def trim_cache() -> None:
    """Return the device blocks the library keeps between solves to the CUDA memory pool."""
    load().lfba_trim_cache()


def default_options(**kw) -> capi.Options:
    o = capi.Options()
    load().lfba_options_init(C.byref(o))
    o.minimizer_progress_to_stdout = 0
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def solve(pa: capi.ProblemArrays, camera, views, points, options: capi.Options | None = None,
          raise_on_failure: bool = True, inplace: bool = False):
    """lfba_solve: returns (camera17, views6F, points3P, summary dict). By default the inputs are left untouched (the
    library gets copies); inplace=True hands the caller's own contiguous float64 arrays to the C ABI, which updates them
    in place exactly like the reference's Ceres call does (src/CameraCalibration.cpp:965)."""
    L = load()
    if inplace:
        cam, vw, pt = camera, views, points
        for a_ in (cam, vw, pt):
            if not (isinstance(a_, np.ndarray) and a_.dtype == np.float64 and a_.flags.c_contiguous and a_.flags.writeable):
                raise ValueError("inplace=True needs writable C-contiguous float64 arrays")
    else:
        cam = np.array(camera, np.float64, copy=True)
        vw = np.array(views, np.float64, copy=True)
        pt = np.array(points, np.float64, copy=True)
    o = options if options is not None else default_options()
    s, rows = capi.new_summary(max(8, o.max_num_iterations + 8))
    p = pa.as_struct()
    rc = L.lfba_solve(C.byref(p), C.byref(o), capi._dp(cam), capi._dp(vw), capi._dp(pt), C.byref(s))
    d = capi.summary_to_dict(s, rows)
    d["status"] = rc
    if rc != capi.OK and raise_on_failure:
        _check(rc, "lfba_solve")
    return cam, vw, pt, d


def evaluate(pa: capi.ProblemArrays, camera, views, points, jacobians=True, options=None, inlier_threshold=1.0):
    """lfba_eval: residuals (n,2), Jacobians in Ceres' block layout, cost and calcReprojectionError statistics."""
    L = load()
    n = pa.n_obs
    cam = np.ascontiguousarray(camera, np.float64)
    vw = np.ascontiguousarray(views, np.float64)
    pt = np.ascontiguousarray(points, np.float64)
    res = np.zeros(2 * n)
    jc = np.zeros((n, 2, 17)) if jacobians else None
    jv = np.zeros((n, 2, 6)) if jacobians else None
    jp = np.zeros((n, 2, 3)) if jacobians else None
    cost = C.c_double(0)
    st = capi.ReprojStats()
    o = options if options is not None else default_options()
    p = pa.as_struct()
    rc = L.lfba_eval(C.byref(p), C.byref(o), capi._dp(cam), capi._dp(vw), capi._dp(pt), capi._dp(res), capi._dp(jc),
                     capi._dp(jv), capi._dp(jp), C.byref(cost), C.byref(st), float(inlier_threshold))
    _check(rc, "lfba_eval")
    return {"residuals": res.reshape(n, 2), "jac_camera": jc, "jac_view": jv, "jac_point": jp, "cost": cost.value,
            "stats": {"std_x": st.std_x, "std_y": st.std_y, "mae_x": st.mae_x, "mae_y": st.mae_y,
                      "num_points": st.num_points, "num_inliers": st.num_inliers}}


def _covariance_result(cam, poses, info: capi.CovarianceInfo, points=None) -> dict:
    inf = {f: getattr(info, f) for f, _ in capi.CovarianceInfo._fields_ if not f.startswith("reserved")}
    s2 = info.sigma2
    r = {"camera": cam, "poses": poses, "info": inf,
         "std_camera": np.sqrt(s2 * np.diag(cam)),
         "std_poses": np.sqrt(s2 * np.diagonal(poses, axis1=1, axis2=2))}
    if points is not None:
        r["points"] = points
        r["std_points"] = np.sqrt(s2 * np.diagonal(points, axis1=1, axis2=2))
    return r


def covariance(pa: capi.ProblemArrays, camera, views, points, options: capi.Options | None = None,
               with_points: bool = False) -> dict:
    """lfba_covariance: covariance blocks of (J^T W J)^-1 of camera and poses at the given parameters (ceres::Covariance
    semantics, not multiplied by sigma2). Returns {"camera": 17x17, "poses": Fx6x6, "info": {...}, "std_camera": 17,
    "std_poses": Fx6}; the standard deviations are scaled by info["sigma2"]. with_points: lfba_covariance_points, which
    also returns "points" (P x 3 x 3, relative to the gauge frame) and "std_points" (P x 3)."""
    L = load()
    cam = np.ascontiguousarray(camera, np.float64)
    vw = np.ascontiguousarray(views, np.float64)
    pt = np.ascontiguousarray(points, np.float64)
    cc = np.zeros((17, 17))
    cp = np.zeros((pa.n_frames, 6, 6))
    info = capi.CovarianceInfo()
    o = options if options is not None else default_options()
    p = pa.as_struct()
    if not with_points:
        _check(L.lfba_covariance(C.byref(p), C.byref(o), capi._dp(cam), capi._dp(vw), capi._dp(pt), capi._dp(cc),
                                 capi._dp(cp), C.byref(info)), "lfba_covariance")
        return _covariance_result(cc, cp, info)
    cq = np.zeros((pa.n_points, 3, 3))
    _check(L.lfba_covariance_points(C.byref(p), C.byref(o), capi._dp(cam), capi._dp(vw), capi._dp(pt), capi._dp(cc),
                                    capi._dp(cp), capi._dp(cq), C.byref(info)), "lfba_covariance_points")
    return _covariance_result(cc, cp, info, cq)


def project_to_raw(grid: "capi.LensGrid", feat_x, feat_y, vdepth, frame_idx=None, point_idx=None, device=-1):
    """lfba_project_to_raw: the observation arrays projectPointsToRawImage (src/CameraCalibration.cpp:640-769) produces
    for a frame-major feature list, in the reference's order. Returns a dict of NumPy arrays."""
    L = load()
    fx = np.ascontiguousarray(feat_x, np.float64)
    fy = np.ascontiguousarray(feat_y, np.float64)
    vd = np.ascontiguousarray(vdepth, np.float64)
    m = fx.size
    fi = None if frame_idx is None else np.ascontiguousarray(frame_idx, np.int32)
    pi = None if point_idx is None else np.ascontiguousarray(point_idx, np.int32)
    g = grid.as_struct()
    n = C.c_int64(0)
    _check(L.lfba_project_to_raw(C.byref(g), m, capi._dp(fx), capi._dp(fy), capi._dp(vd), capi._ip(fi), capi._ip(pi), 0, None,
                                 None, None, None, None, None, C.byref(n), device), "lfba_project_to_raw")
    k = n.value
    out = {"obs_x": np.zeros(k), "obs_y": np.zeros(k), "ml_x": np.zeros(k), "ml_y": np.zeros(k),
           "point_idx": np.zeros(k, np.int32), "frame_idx": np.zeros(k, np.int32)}
    if k:
        _check(L.lfba_project_to_raw(C.byref(g), m, capi._dp(fx), capi._dp(fy), capi._dp(vd), capi._ip(fi), capi._ip(pi), k,
                                     capi._dp(out["obs_x"]), capi._dp(out["obs_y"]), capi._dp(out["ml_x"]),
                                     capi._dp(out["ml_y"]), capi._ip(out["point_idx"]), capi._ip(out["frame_idx"]),
                                     C.byref(n), device), "lfba_project_to_raw")
    return out


def init_plenoptic(fph_init, pixel_size_totfoc, vdepth, frame_idx, point_idx, views, points, device=-1):
    """lfba_init_plenoptic: (fL_init, B_init, bL0_init) of CameraCalibration::initPlenopticParameters (:456-498)."""
    L = load()
    vd = np.ascontiguousarray(vdepth, np.float64)
    fi = np.ascontiguousarray(frame_idx, np.int32)
    pi = np.ascontiguousarray(point_idx, np.int32)
    vw = np.ascontiguousarray(views, np.float64).ravel()
    pt = np.ascontiguousarray(points, np.float64).ravel()
    fL, B, bL0 = C.c_double(0), C.c_double(0), C.c_double(0)
    _check(L.lfba_init_plenoptic(float(fph_init), float(pixel_size_totfoc), vd.size, capi._dp(vd), capi._ip(fi), capi._ip(pi),
                                 vw.size // 6, capi._dp(vw), pt.size // 3, capi._dp(pt), C.byref(fL), C.byref(B),
                                 C.byref(bL0), device), "lfba_init_plenoptic")
    return fL.value, B.value, bL0.value


def epipolar_web(lens_diameter, rotation=0.0, rotation_on_grid=False):
    """lfba_epipolar_web (host): (lines [n, 3] = ex, ey, base-line length; group_begin [n_groups + 1])."""
    L = load()
    nl, ng = C.c_int32(0), C.c_int32(0)
    _check(L.lfba_epipolar_web(float(lens_diameter), float(rotation), int(bool(rotation_on_grid)), C.byref(nl), C.byref(ng),
                               None, None), "lfba_epipolar_web")
    lines = np.zeros((nl.value, 3))
    gb = np.zeros(ng.value + 1, np.int32)
    _check(L.lfba_epipolar_web(float(lens_diameter), float(rotation), int(bool(rotation_on_grid)), C.byref(nl), C.byref(ng),
                               capi._dp(lines), capi._ip(gb)), "lfba_epipolar_web")
    return lines, gb


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _check(load().lfba_comm_unique_id(buf), "lfba_comm_unique_id")
    return buf.raw


def measure_fp64_peak(device: int = -1) -> float:
    v = C.c_double(0)
    _check(load().lfba_measure_fp64_peak(device, C.byref(v)), "lfba_measure_fp64_peak")
    return v.value


class Communicator:
    """Persistent NCCL communicator of this rank (lfba_comm_create); collective over all ranks."""

    def __init__(self, rank: int, nranks: int, unique_id: bytes):
        self._L = load()
        self.rank, self.nranks = rank, nranks
        c = capi.Comm()
        c.rank, c.nranks = rank, nranks
        C.memmove(C.addressof(c) + capi.Comm.nccl_unique_id.offset, unique_id, 128)
        self._h = C.c_void_p()
        _check(self._L.lfba_comm_create(C.byref(c), C.byref(self._h)), "lfba_comm_create")

    def close(self):
        if self._h:
            self._L.lfba_comm_destroy(self._h)
            self._h = C.c_void_p()


class DeviceSolver:
    """Device-resident session (lfba_solver_*): upload/index once, then set parameters / run repeatedly."""

    def __init__(self, pa: capi.ProblemArrays, options: capi.Options | None = None, rank: int = 0, nranks: int = 1,
                 unique_id: bytes | None = None, communicator: "Communicator | None" = None):
        self._L = load()
        self.pa = pa
        self.options = options if options is not None else default_options()
        self._h = C.c_void_p()
        p = pa.as_struct()
        comm = None
        if communicator is not None:
            c = capi.Comm()
            c.rank, c.nranks = communicator.rank, communicator.nranks
            c.handle = communicator._h
            comm = C.byref(c)
        elif nranks > 1:
            c = capi.Comm()
            c.rank, c.nranks = rank, nranks
            C.memmove(C.addressof(c) + capi.Comm.nccl_unique_id.offset, unique_id, 128)
            comm = C.byref(c)
        _check(self._L.lfba_solver_create(C.byref(p), C.byref(self.options), comm, C.byref(self._h)),
               "lfba_solver_create")

    def set_parameters(self, camera, views, points):
        cam = np.ascontiguousarray(camera, np.float64)
        vw = np.ascontiguousarray(views, np.float64)
        pt = np.ascontiguousarray(points, np.float64)
        _check(self._L.lfba_solver_set_parameters(self._h, capi._dp(cam), capi._dp(vw), capi._dp(pt)),
               "lfba_solver_set_parameters")

    def run(self, raise_on_failure=True) -> dict:
        s, rows = capi.new_summary(max(8, self.options.max_num_iterations + 8))
        rc = self._L.lfba_solver_run(self._h, C.byref(s))
        d = capi.summary_to_dict(s, rows)
        d["status"] = rc
        if rc != capi.OK and raise_on_failure:
            _check(rc, "lfba_solver_run")
        return d

    def get_parameters(self):
        cam = np.zeros(17)
        vw = np.zeros(6 * self.pa.n_frames)
        pt = np.zeros(3 * self.pa.n_points)
        _check(self._L.lfba_solver_get_parameters(self._h, capi._dp(cam), capi._dp(vw), capi._dp(pt)),
               "lfba_solver_get_parameters")
        return cam, vw, pt

    def time_eval(self, reps=10, materialize=False) -> float:
        """materialize: False/0 fused pass; True/1 eval-only kernel, Ceres layout; 2 eval-only, live camera columns only."""
        ms = C.c_double(0)
        _check(self._L.lfba_solver_time_eval(self._h, reps, int(materialize), C.byref(ms)),
               "lfba_solver_time_eval")
        return ms.value

    def track_blocks(self):
        """lfba_solver_track_blocks: raw outputs of ONE fused evaluation pass at the parameters last set — per-track
        normal-equation blocks (camera frame) and the camera block; for parity tests of the LM loop's own kernel."""
        n, rs = C.c_int64(0), C.c_int32(0)
        _check(self._L.lfba_solver_track_blocks(self._h, C.byref(n), C.byref(rs), None, None, None, None),
               "lfba_solver_track_blocks")
        T, RS = n.value, rs.value
        rec = np.zeros((T, RS))
        camsum = np.zeros(64)
        tp = np.zeros(T, np.int32)
        tf = np.zeros(T, np.int32)
        _check(self._L.lfba_solver_track_blocks(self._h, C.byref(n), C.byref(rs), capi._dp(rec), capi._dp(camsum),
                                                capi._ip(tp), capi._ip(tf)), "lfba_solver_track_blocks")
        return {"rec": rec, "camsum": camsum, "trk_point": tp, "trk_frame": tf, "rec_stride": RS}

    def covariance(self, with_points: bool = False) -> dict:
        """lfba_solver_covariance: covariance blocks of camera and poses at the parameters get_parameters() returns;
        same result as the module-level covariance() there. The session is left as it was. with_points:
        lfba_solver_covariance_points, which also returns "points" (P x 3 x 3) and "std_points" (P x 3)."""
        cc = np.zeros((17, 17))
        cp = np.zeros((self.pa.n_frames, 6, 6))
        info = capi.CovarianceInfo()
        if not with_points:
            _check(self._L.lfba_solver_covariance(self._h, capi._dp(cc), capi._dp(cp), C.byref(info)),
                   "lfba_solver_covariance")
            return _covariance_result(cc, cp, info)
        cq = np.zeros((self.pa.n_points, 3, 3))
        _check(self._L.lfba_solver_covariance_points(self._h, capi._dp(cc), capi._dp(cp), capi._dp(cq), C.byref(info)),
               "lfba_solver_covariance_points")
        return _covariance_result(cc, cp, info, cq)

    def close(self):
        if self._h:
            self._L.lfba_solver_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
