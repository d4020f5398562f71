"""Dense reference for the parameter covariance: the loss-weighted Jacobian of the whole problem from the CPU oracle
(reprojection blocks with sqrt(rho') row weights under the robust flag, distance-constraint rows), the columns the
solver treats as free, and (J^T J)^-1 scattered back into the 17 x 17 camera block and the F x 6 x 6 pose blocks."""
import numpy as np

from lifcal_b200 import capi
from oracle import binding as ob


def uses_constraints(pa):
    return bool(pa.config & capi.CFG_REFINE_POINTS) and pa.calib_type != capi.RECALIBRATION and pa.c_p1.size > 0


def dense_jacobian(pa, camera, views, points, loss_scale=0.5):
    """J (2N + K) x (17 + 6F + 3P) in the parameter order [camera | views | points]; columns not yet selected."""
    ev = ob.evaluate(pa, camera, views, points)
    n, F, P = pa.n_obs, pa.n_frames, pa.n_points
    J = np.zeros((2 * n + (pa.c_p1.size if uses_constraints(pa) else 0), 17 + 6 * F + 3 * P))
    rows = np.arange(n)
    w = np.ones(n)
    if pa.config & capi.CFG_ROBUST:  # Cauchy corrector: rho'' < 0, so J is scaled by sqrt(rho')
        s = (ev["residuals"] ** 2).sum(1)
        w = np.sqrt(1.0 / (1.0 + s / loss_scale ** 2))
    for k in range(2):
        J[2 * rows + k, :17] = ev["jac_camera"][:, k, :] * w[:, None]
        for j in range(6):
            J[2 * rows + k, 17 + 6 * pa.frame_idx + j] = ev["jac_view"][:, k, j] * w
        for j in range(3):
            J[2 * rows + k, 17 + 6 * F + 3 * pa.point_idx + j] = ev["jac_point"][:, k, j] * w
    if uses_constraints(pa):
        pts = np.asarray(points).reshape(-1, 3)
        for k in range(pa.c_p1.size):
            a, b = pa.c_p1[k], pa.c_p2[k]
            d = pts[a] - pts[b]
            jj = d / np.linalg.norm(d) / (pa.c_sigma[k] + 1e-6)
            J[2 * n + k, 17 + 6 * F + 3 * a:17 + 6 * F + 3 * a + 3] = jj
            J[2 * n + k, 17 + 6 * F + 3 * b:17 + 6 * F + 3 * b + 3] = -jj
    return J


def free_columns(pa, drop_frame=None):
    """Columns of dense_jacobian the solver treats as free: live camera entries (not camera[0], camera[2] in
    recalibration), poses of observed frames under REFINE_POSES (except drop_frame), observed or constrained points under
    REFINE_POINTS."""
    F, P = pa.n_frames, pa.n_points
    nc = 5 + (pa.config & capi.CFG_NRADIAL_MASK) + (2 if pa.config & capi.CFG_TANGENTIAL else 0)
    cols = [c for c in range(nc) if not (pa.calib_type == capi.RECALIBRATION and c in (0, 2))]
    if pa.config & capi.CFG_REFINE_POSES:
        seen = np.zeros(F, bool)
        seen[pa.frame_idx] = True
        for f in range(F):
            if seen[f] and f != drop_frame:
                cols += list(range(17 + 6 * f, 17 + 6 * f + 6))
    if pa.config & capi.CFG_REFINE_POINTS:
        active = np.zeros(P, bool)
        active[pa.point_idx] = True
        if uses_constraints(pa):
            active[pa.c_p1] = active[pa.c_p2] = True
        for p in np.nonzero(active)[0]:
            cols += list(range(17 + 6 * F + 3 * p, 17 + 6 * F + 3 * p + 3))
    return np.array(cols)


def gauge_frame(pa):
    """The frame the library holds fixed when points are refined (first frame with observations), else None."""
    if not pa.config & capi.CFG_REFINE_POINTS:
        return None
    return int(np.min(pa.frame_idx))


def reference_covariance(pa, camera, views, points, loss_scale=0.5):
    """(cov_camera 17x17, cov_poses Fx6x6, J restricted to the free columns) at the given parameters."""
    F = pa.n_frames
    J = dense_jacobian(pa, camera, views, points, loss_scale)
    cols = free_columns(pa, gauge_frame(pa))
    Jf = J[:, cols]
    H = Jf.T @ Jf
    d = 1.0 / np.sqrt(np.diag(H))  # symmetric scaling for a well-conditioned inverse
    Sig = d[:, None] * np.linalg.inv(d[:, None] * H * d[None, :]) * d[None, :]
    full = np.zeros((17 + 6 * F, 17 + 6 * F))
    keep = cols < 17 + 6 * F
    idx = cols[keep]
    full[np.ix_(idx, idx)] = Sig[np.ix_(np.nonzero(keep)[0], np.nonzero(keep)[0])]
    cov_cam = full[:17, :17]
    cov_poses = np.stack([full[17 + 6 * f:17 + 6 * f + 6, 17 + 6 * f:17 + 6 * f + 6] for f in range(F)])
    return cov_cam, cov_poses, Jf
