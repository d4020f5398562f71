"""CPU tests of the assumption the covariance's gauge policy rests on: the null space of the loss-weighted Jacobian at
the oracle's solution. With points refined and no distance constraint it is rigid motion + scale, and the scale
direction moves bL0 and B (so their covariance is undefined); one constraint leaves rigid motion only, which holding the
first frame's pose removes without touching the intrinsics; so does recalibration, which holds fL and B constant;
with points fixed there is no null space."""
import numpy as np
import pytest

from lifcal_b200 import capi
from oracle import binding as ob

from covariance_ref import dense_jacobian, free_columns

P0 = 2 | capi.CFG_TANGENTIAL | capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS  # 0x506


def _solved(config, n_constraints=0, calib_type=capi.CALIBRATION_ARUCO, noise_px=0.1):
    sc = capi.make_scene(None, n_points=60, n_frames=6, window=0, config=config, n_constraints=n_constraints,
                         calib_type=calib_type, noise_px=noise_px, seed=11)
    cam, vw, pt, s = ob.solve(sc.problem, sc.camera_init, sc.views_init, sc.points_init)
    assert s["status"] == capi.OK
    return sc.problem, cam, vw, pt


def _null_space(pa, cam, vw, pt, drop_frame=None):
    J = dense_jacobian(pa, cam, vw, pt)
    cols = free_columns(pa, drop_frame)
    Jf = J[:, cols]
    Jn = Jf / np.linalg.norm(Jf, axis=0)
    _, s, vt = np.linalg.svd(Jn, full_matrices=False)
    null = vt[s < 1e-10 * s[0]]
    return cols, s, null


@pytest.mark.parametrize("config", [P0, P0 | capi.CFG_MLADJ])
def test_no_constraints_scale_gauge_moves_bl0_and_b(built, config):
    pa, cam, vw, pt = _solved(config)
    cols, s, null = _null_space(pa, cam, vw, pt)
    assert null.shape[0] == 7
    cam_part = np.abs(null[:, (cols == 1) | (cols == 2)]).max()
    assert cam_part > 1e-3


@pytest.mark.parametrize("config,k", [(P0, 1), (P0, 4), (P0 | capi.CFG_MLADJ | capi.CFG_ROBUST, 1)])
def test_constraints_leave_rigid_motion_only(built, config, k):
    pa, cam, vw, pt = _solved(config, n_constraints=k)
    cols, s, null = _null_space(pa, cam, vw, pt)
    assert null.shape[0] == 6
    assert np.abs(null[:, cols < 17]).max() < 1e-10
    # holding the first frame's pose removes the gauge
    cols, s, null = _null_space(pa, cam, vw, pt, drop_frame=int(pa.frame_idx.min()))
    assert null.shape[0] == 0 and s[-1] / s[0] > 1e-6


@pytest.mark.parametrize("config", [0x100, 0x102, 0x106, 0x906])
def test_points_fixed_full_rank(built, config):
    pa, cam, vw, pt = _solved(config)
    cols, s, null = _null_space(pa, cam, vw, pt)
    assert null.shape[0] == 0 and s[-1] / s[0] > 1e-6


@pytest.mark.parametrize("config", [P0, P0 | capi.CFG_MLADJ | capi.CFG_ROBUST])
def test_recalibration_fixed_fl_and_b_remove_the_scale_gauge(built, config):
    """Recalibration drops the constraints, but holds fL and B constant: that fixes the scale, so only rigid motion is
    left and the first frame's pose removes it, as with constraints."""
    pa, cam, vw, pt = _solved(config, calib_type=capi.RECALIBRATION)
    cols, s, null = _null_space(pa, cam, vw, pt)
    assert null.shape[0] == 6
    assert np.abs(null[:, cols < 17]).max() < 1e-10
    cols, s, null = _null_space(pa, cam, vw, pt, drop_frame=int(pa.frame_idx.min()))
    assert null.shape[0] == 0 and s[-1] / s[0] > 1e-6
