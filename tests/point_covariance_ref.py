"""Dense reference for the per-point covariance blocks: the point blocks of the same inverse of J^T W J that
covariance_ref.reference_covariance takes its camera and pose blocks from (same loss-weighted Jacobian, free columns
and gauge frame)."""
import numpy as np

from covariance_ref import dense_jacobian, free_columns, gauge_frame


def reference_point_covariance(pa, camera, views, points, loss_scale=0.5):
    """P x 3 x 3 point blocks of the dense inverse over the free columns; zero for points that are not free (inactive,
    or all points without REFINE_POINTS)."""
    F, P = pa.n_frames, pa.n_points
    J = dense_jacobian(pa, camera, views, points, loss_scale)
    cols = free_columns(pa, gauge_frame(pa))
    Jf = J[:, cols]
    H = Jf.T @ Jf
    d = 1.0 / np.sqrt(np.diag(H))  # symmetric scaling for a well-conditioned inverse
    Sig = d[:, None] * np.linalg.inv(d[:, None] * H * d[None, :]) * d[None, :]
    out = np.zeros((P, 3, 3))
    for k in np.nonzero(cols >= 17 + 6 * F)[0][::3]:  # free_columns lists a point's three columns together
        p = (cols[k] - 17 - 6 * F) // 3
        out[p] = Sig[k:k + 3, k:k + 3]
    return out
