"""Per-image camera pose refinement (DESIGN.md §3 "Camera pose refinement"): host helpers in float64.

Image k owns xi_k = (rho, phi) in R^6, applied in the camera frame: p_cam' = Exp(phi) p_cam + rho, i.e.
W2C'(xi) = C(xi) W2C with C(xi) = [[Exp(phi), rho], [0, 1]] (column convention; the rasterizer's row-vector
viewmatrix becomes viewmatrix @ C^T).  The training step applies and differentiates the correction on the device
(hg_camera_pose_apply, hg_camera_pose_grad_finish); these helpers are the same maps for saving, loading and tests.
"""
import numpy as np

# rows of the device table: rho 3 | phi 3 | 2 zero pads (float4-aligned rows)
ROW = 8


def _skew(p):
    return np.array([[0.0, -p[2], p[1]], [p[2], 0.0, -p[0]], [-p[1], p[0], 0.0]])


def so3_exp(phi):
    """Rodrigues' formula: the rotation matrix of the rotation vector `phi` (3,)."""
    p = np.asarray(phi, dtype=np.float64).reshape(3)
    t = float(np.linalg.norm(p))
    K = _skew(p)
    if t < 1e-8:
        return np.eye(3) + K + 0.5 * K @ K
    return np.eye(3) + np.sin(t) / t * K + (1.0 - np.cos(t)) / t ** 2 * K @ K


def so3_left_jacobian(phi):
    """Left Jacobian of SO(3): Exp(phi + d) = Exp(J_l(phi) d) Exp(phi) to first order in d."""
    p = np.asarray(phi, dtype=np.float64).reshape(3)
    t = float(np.linalg.norm(p))
    K = _skew(p)
    if t < 1e-8:
        return np.eye(3) + 0.5 * K + K @ K / 6.0
    return np.eye(3) + (1.0 - np.cos(t)) / t ** 2 * K + (t - np.sin(t)) / t ** 3 * K @ K


def pose_matrix(xi):
    """C(xi) = [[Exp(phi), rho], [0, 1]] (4, 4) of xi = (rho, phi)."""
    xi = np.asarray(xi, dtype=np.float64).reshape(-1)
    C = np.eye(4)
    C[:3, :3] = so3_exp(xi[3:6])
    C[:3, 3] = xi[:3]
    return C


def corrected_w2c(world_view_transform, xi):
    """The corrected world-to-camera matrix (column convention, 4 x 4 float64) of a camera whose row-vector
    `world_view_transform` is given."""
    V = np.asarray(world_view_transform, dtype=np.float64).reshape(4, 4)
    return pose_matrix(xi) @ V.T
