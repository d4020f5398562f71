"""GPU tests of the parameter covariance (lfba_solver_covariance / lfba_covariance): the device solves, then the
covariance at its final parameters is compared with a dense NumPy inverse of J^T W J built from the CPU oracle's
Jacobians at the same parameters (tests/covariance_ref.py). Also: the gauge and unobserved frames' blocks are exactly 0,
sigma2 estimates the noise, refused cases, the session is left as it was, and the one-shot form equals the session."""
import numpy as np
import pytest

from lifcal_b200 import api, capi

from covariance_ref import reference_covariance

pytestmark = pytest.mark.gpu

# correlation-normalised bar |S_gpu - S_ref|_ij / sqrt(S_ii S_jj), and relative bar on the variances; worst measured
# on a B200: 1.4e-9 (points refined + constraints), 1.0e-9 (recalibration), <= 2e-11 elsewhere
# (profiles/r03_covariance_accuracy.log)
CORR_BAR = 1e-8
VAR_BAR = 1e-8

R2T = 2 | capi.CFG_TANGENTIAL
SCENES = {
    # points fixed, robust, windowed: the pose part of the reduced system is banded
    "a_points_fixed_windowed": dict(n_points=200, n_frames=40, window=4,
                                    config=R2T | capi.CFG_REFINE_POSES | capi.CFG_ROBUST | capi.CFG_MLADJ),
    # points refined + constraints: the coupled points sit in the border; non-robust for the sigma2 check
    "b_points_constraints": dict(n_points=150, n_frames=8, window=0, n_constraints=3,
                                 config=R2T | capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS),
    # recalibration: fL and B constant (they fix the scale), points refined, robust
    "c_recalibration": dict(n_points=150, n_frames=8, window=0, calib_type=capi.RECALIBRATION,
                            config=R2T | capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS | capi.CFG_ROBUST),
    # poses not refined: camera only
    "d_poses_fixed": dict(n_points=200, n_frames=6, window=0, config=R2T | capi.CFG_MLADJ),
}


def _device():
    if api.device_count() < 1:
        pytest.skip("no CUDA device")


def _problem(name):
    kw = dict(SCENES[name]) if name in SCENES else dict(n_points=200, n_frames=12, window=4,
                                                        config=R2T | capi.CFG_REFINE_POSES)
    sc = capi.make_scene(None, seed=23, **kw)
    pa = sc.problem
    if name == "e_unobserved_frame":  # frame 5 loses its observations
        pa = pa.subset(pa.frame_idx != 5)
    return sc, pa


def _solve_and_cov(name):
    sc, pa = _problem(name)
    ds = api.DeviceSolver(pa)
    try:
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        ds.run()
        cam, vw, pt = ds.get_parameters()
        cov = ds.covariance()
    finally:
        ds.close()
    return pa, cam, vw, pt, cov


def _worst(got, ref, idx):
    d = np.sqrt(np.diag(ref)[idx])
    g = got[np.ix_(idx, idx)]
    r = ref[np.ix_(idx, idx)]
    corr = np.abs(g - r) / np.outer(d, d)
    var = np.abs(np.diag(g) - np.diag(r)) / np.diag(r)
    return float(corr.max()), float(var.max())


@pytest.mark.parametrize("name", list(SCENES) + ["e_unobserved_frame"])
def test_covariance_matches_dense_reference(built, name):
    _device()
    pa, cam, vw, pt, cov = _solve_and_cov(name)
    ref_cam, ref_poses, _ = reference_covariance(pa, cam, vw, pt)
    info = cov["info"]
    live = np.nonzero(np.diag(ref_cam) > 0)[0]
    # exactly zero wherever the reference has no free parameter
    dead = np.setdiff1d(np.arange(17), live)
    assert np.all(cov["camera"][dead, :] == 0) and np.all(cov["camera"][:, dead] == 0)
    worst = [_worst(cov["camera"], ref_cam, live)]
    for f in range(pa.n_frames):
        if np.all(ref_poses[f] == 0):
            assert np.all(cov["poses"][f] == 0), f
        else:
            worst.append(_worst(cov["poses"][f], ref_poses[f], np.arange(6)))
    corr, var = max(w[0] for w in worst), max(w[1] for w in worst)
    print(f"\n[covariance accuracy] {name}: n_reduced={info['n_reduced']} gauge={info['gauge']} "
          f"gauge_frame={info['gauge_frame']} worst corr-normalised diff {corr:.3e}, worst variance rel diff {var:.3e}, "
          f"sigma2={info['sigma2']:.6g}")
    assert corr <= CORR_BAR and var <= VAR_BAR
    assert np.all(np.isfinite(cov["std_camera"])) and np.all(np.isfinite(cov["std_poses"]))


def test_gauge_and_unobserved_frames_are_zero_and_info(built):
    _device()
    pa, cam, vw, pt, cov = _solve_and_cov("b_points_constraints")
    info = cov["info"]
    assert info["gauge"] == capi.GAUGE_FIRST_FRAME and info["gauge_frame"] == int(pa.frame_idx.min())
    assert np.all(cov["poses"][info["gauge_frame"]] == 0)
    assert info["num_residuals"] == 2 * pa.n_obs + pa.c_p1.size
    # non-robust, noise_px = 0.1: 2 cost / (m - p) estimates the noise variance
    assert abs(info["sigma2"] - 0.01) <= 0.03 * 0.01, info["sigma2"]
    pa, cam, vw, pt, cov = _solve_and_cov("e_unobserved_frame")
    assert cov["info"]["gauge"] == capi.GAUGE_NONE and cov["info"]["gauge_frame"] == -1
    assert np.all(cov["poses"][5] == 0) and np.all(cov["poses"][4] != 0)


def test_points_refined_without_constraints_is_refused(built):
    _device()
    sc = capi.make_scene(None, n_points=100, n_frames=6, window=0, seed=23,
                         config=R2T | capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS)
    with pytest.raises(capi.LfbaError) as e:
        api.covariance(sc.problem, sc.camera_init, sc.views_init, sc.points_init)
    assert "status 1" in str(e.value) and "scale gauge" in str(e.value)


def test_emulated_shard_session_is_refused(built):
    _device()
    sc, pa = _problem("a_points_fixed_windowed")
    ds = api.DeviceSolver(pa, api.default_options(emulate_shards=2))
    try:
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        with pytest.raises(capi.LfbaError) as e:
            ds.covariance()
        assert "status 1" in str(e.value)
    finally:
        ds.close()


_NO_TIME = [f for f, _ in capi.Iteration._fields_ if not f.endswith("time_s")]


@pytest.mark.parametrize("name", ["a_points_fixed_windowed", "b_points_constraints", "c_recalibration"])
def test_session_left_as_it_was_and_one_shot_equals_session(built, name):
    _device()
    sc, pa = _problem(name)
    ds = api.DeviceSolver(pa)
    try:
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        s1 = ds.run()
        p1 = ds.get_parameters()
        cov = ds.covariance()
        p_after = ds.get_parameters()
        s2 = ds.run()
        p2 = ds.get_parameters()
    finally:
        ds.close()
    for a, b in zip(p1, p_after):
        assert np.array_equal(a, b)
    assert s1["num_iterations"] == s2["num_iterations"] and s1["final_cost"] == s2["final_cost"]
    for r1, r2 in zip(s1["iterations"], s2["iterations"]):
        assert [r1[f] for f in _NO_TIME] == [r2[f] for f in _NO_TIME]
    for a, b in zip(p1, p2):
        assert np.array_equal(a, b)
    one = api.covariance(pa, *p1)
    assert np.array_equal(one["camera"], cov["camera"]) and np.array_equal(one["poses"], cov["poses"])
    assert one["info"]["cost"] == cov["info"]["cost"] and one["info"]["sigma2"] == cov["info"]["sigma2"]
