"""GPU tests of the per-point covariance blocks (lfba_solver_covariance_points / lfba_covariance_points): the device
solves, then the 3 x 3 block of every point at its final parameters is compared with the point blocks of a dense NumPy
inverse of J^T W J built from the CPU oracle's Jacobians (tests/point_covariance_ref.py). Also: the camera and pose blocks
and the info are those of lfba_solver_covariance bit for bit, fixed and inactive points get exact zeros, the blocks
are exactly symmetric, the session is left as it was, the one-shot form equals the session, and the refused cases."""
import numpy as np
import pytest

from lifcal_b200 import api, capi

from point_covariance_ref import reference_point_covariance

pytestmark = pytest.mark.gpu

# the bars of the camera / pose blocks: correlation-normalised |S_gpu - S_ref|_ij / sqrt(S_ii S_jj), and relative on the
# variances
CORR_BAR = 1e-8
VAR_BAR = 1e-8

R2T = 2 | capi.CFG_TANGENTIAL
REFINED = R2T | capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS
SCENES = {
    # eliminated and coupled points, non-robust, one window: every pose pair of a point is read
    "b_points_constraints": dict(n_points=150, n_frames=8, window=0, n_constraints=3, config=REFINED),
    # robust, fL and B constant: camera[0] and camera[2] drop out of the camera terms
    "c_recalibration": dict(n_points=150, n_frames=8, window=0, calib_type=capi.RECALIBRATION,
                            config=REFINED | capi.CFG_ROBUST),
    # windowed (band 3 of 11): banded pose-pose reads, and the gauge frame (0) inside the first window. 12 frames, not
    # more: the gauge drifts along the chain, and at 24 frames the column-scaled J^T W J has condition 5.7e8, where the
    # camera and pose blocks themselves differ from the dense reference by 3e-8 (12 frames: 1.3e8, 3e-9)
    "w_windowed_constraints": dict(n_points=120, n_frames=12, window=4, n_constraints=3,
                                   config=REFINED | capi.CFG_ROBUST | capi.CFG_MLADJ),
    # points fixed: every point block is exactly 0
    "a_points_fixed_windowed": dict(n_points=200, n_frames=40, window=4,
                                    config=R2T | capi.CFG_REFINE_POSES | capi.CFG_ROBUST | capi.CFG_MLADJ),
}
DROPPED = "w_dropped_point"  # w_windowed_constraints with the observations of one unconstrained point removed
INFO_TIMES = ("gpu_ms", "selinv_ms", "points_ms")


def _device():
    if api.device_count() < 1:
        pytest.skip("no CUDA device")


def _problem(name):
    sc = capi.make_scene(None, seed=23, **SCENES["w_windowed_constraints" if name == DROPPED else name])
    pa = sc.problem
    dropped = None
    if name == DROPPED:
        dropped = int(np.setdiff1d(np.arange(pa.n_points), np.concatenate([pa.c_p1, pa.c_p2]))[0])
        pa = pa.subset(pa.point_idx != dropped)
    return sc, pa, dropped


_SOLVED = {}


def _solved(name):
    """Solve once per scene; the covariance with and without points on the same session at its final parameters."""
    if name not in _SOLVED:
        sc, pa, dropped = _problem(name)
        ds = api.DeviceSolver(pa)
        try:
            ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
            ds.run()
            params = ds.get_parameters()
            with_pts = ds.covariance(with_points=True)
            plain = ds.covariance()
        finally:
            ds.close()
        _SOLVED[name] = (pa, params, with_pts, plain, dropped)
    return _SOLVED[name]


def _worst(got, ref):
    d = np.sqrt(np.diag(ref))
    corr = np.abs(got - ref) / np.outer(d, d)
    var = np.abs(np.diag(got) - np.diag(ref)) / np.diag(ref)
    return float(corr.max()), float(var.max())


REFINED_SCENES = ["b_points_constraints", "c_recalibration", "w_windowed_constraints", DROPPED]


@pytest.mark.parametrize("name", REFINED_SCENES)
def test_point_blocks_match_dense_reference(built, name):
    _device()
    pa, params, cov, _, dropped = _solved(name)
    ref = reference_point_covariance(pa, *params)
    got = cov["points"]
    assert got.shape == (pa.n_points, 3, 3)
    live = np.nonzero(np.any(ref != 0, axis=(1, 2)))[0]
    dead = np.setdiff1d(np.arange(pa.n_points), live)
    assert np.all(got[dead] == 0), dead
    if dropped is not None:
        assert dropped in dead
    worst = [_worst(got[p], ref[p]) for p in live]
    corr, var = max(w[0] for w in worst), max(w[1] for w in worst)
    coupled = np.unique(np.concatenate([pa.c_p1, pa.c_p2])) if pa.calib_type != capi.RECALIBRATION else []
    print(f"\n[point covariance accuracy] {name}: {live.size} points ({len(coupled)} coupled), gauge_frame="
          f"{cov['info']['gauge_frame']}, worst corr-normalised diff {corr:.3e}, worst variance rel diff {var:.3e}, "
          f"points_ms={cov['info']['points_ms']:.4f}")
    assert corr <= CORR_BAR and var <= VAR_BAR


@pytest.mark.parametrize("name", REFINED_SCENES + ["a_points_fixed_windowed"])
def test_camera_poses_and_info_unchanged_and_blocks_symmetric(built, name):
    _device()
    pa, params, cov, plain, _ = _solved(name)
    assert np.array_equal(cov["camera"], plain["camera"]) and np.array_equal(cov["poses"], plain["poses"])
    for f, v in plain["info"].items():
        if f not in INFO_TIMES:
            assert cov["info"][f] == v, f
    assert plain["info"]["points_ms"] == 0.0 and "points" not in plain
    assert cov["info"]["points_ms"] > 0.0
    pts = cov["points"]
    assert np.array_equal(pts, np.transpose(pts, (0, 2, 1)))
    s2 = cov["info"]["sigma2"]
    assert np.array_equal(cov["std_points"], np.sqrt(s2 * np.diagonal(pts, axis1=1, axis2=2)))
    assert cov["std_points"].shape == (pa.n_points, 3)


def test_points_fixed_blocks_are_zero(built):
    _device()
    pa, params, cov, plain, _ = _solved("a_points_fixed_windowed")
    assert cov["info"]["gauge"] == capi.GAUGE_NONE
    assert cov["points"].shape == (pa.n_points, 3, 3) and np.all(cov["points"] == 0)
    assert np.all(cov["std_points"] == 0)


@pytest.mark.parametrize("name", ["b_points_constraints", "w_windowed_constraints"])
def test_session_left_as_it_was_and_one_shot_equals_session(built, name):
    _device()
    sc, pa, _ = _problem(name)
    ds = api.DeviceSolver(pa)
    no_time = [f for f, _ in capi.Iteration._fields_ if not f.endswith("time_s")]
    try:
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        s1 = ds.run()
        p1 = ds.get_parameters()
        cov = ds.covariance(with_points=True)
        p_after = ds.get_parameters()
        s2 = ds.run()
        p2 = ds.get_parameters()
    finally:
        ds.close()
    for a, b in zip(p1, p_after):
        assert np.array_equal(a, b)
    assert s1["num_iterations"] == s2["num_iterations"] and s1["final_cost"] == s2["final_cost"]
    for r1, r2 in zip(s1["iterations"], s2["iterations"]):
        assert [r1[f] for f in no_time] == [r2[f] for f in no_time]
    for a, b in zip(p1, p2):
        assert np.array_equal(a, b)
    one = api.covariance(pa, *p1, with_points=True)
    for k in ("camera", "poses", "points", "std_points"):
        assert np.array_equal(one[k], cov[k]), k
    assert one["info"]["cost"] == cov["info"]["cost"] and one["info"]["sigma2"] == cov["info"]["sigma2"]
    plain = api.covariance(pa, *p1)
    assert "points" not in plain and np.array_equal(plain["camera"], cov["camera"])


def test_points_refined_without_constraints_is_refused(built):
    _device()
    sc = capi.make_scene(None, n_points=100, n_frames=6, window=0, seed=23, config=REFINED)
    with pytest.raises(capi.LfbaError) as e:
        api.covariance(sc.problem, sc.camera_init, sc.views_init, sc.points_init, with_points=True)
    assert "status 1" in str(e.value) and "scale gauge" in str(e.value)


def test_emulated_shard_session_is_refused(built):
    _device()
    sc, pa, _ = _problem("a_points_fixed_windowed")
    ds = api.DeviceSolver(pa, api.default_options(emulate_shards=2))
    try:
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        with pytest.raises(capi.LfbaError) as e:
            ds.covariance(with_points=True)
        assert "status 1" in str(e.value)
    finally:
        ds.close()
