"""TEST INFRASTRUCTURE — numpy / scipy ports of the head-pose smoothing and landmark projection of reference
src/utils/pose_util.py, for the host arm of scripts/bench_pose_maps.py (the reference does not exist where the GPU runs)."""
import numpy as np
from scipy.spatial.transform import Rotation


def perspective(aspect):
    """create_perspective_matrix: built in fp32, returned as the 4 x 4 matrix the points are multiplied by."""
    f = 1.0 / np.tan(np.pi / 180.0 * 63 / 2.0)
    p = np.zeros(16, dtype=np.float32)
    p[0], p[5], p[10], p[11], p[14] = f / aspect, -f, 10001 / -9999.0, -1.0, 10000 / -9999.0
    return p.reshape(4, 4).T


def pose_matrix(pose):
    m = np.eye(4)
    m[:3, :3] = Rotation.from_euler("xyz", pose[:3], degrees=True).as_matrix()
    m[:3, 3] = pose[3:]
    return m


def project_points(points, trans, poses, image_shape):
    """[L, N, 3] points, [4, 4] trans, [L, 6] poses, (H, W) -> fp64 [L, N, 2]."""
    H, W = image_shape
    P = perspective(W / H)
    out = np.zeros(points.shape[:2] + (2,))
    for i, pts in enumerate(points):
        ph = np.hstack([pts, np.ones((len(pts), 1))])
        t = ph @ (trans @ pose_matrix(poses[i])).T @ P
        xy = t[:, :2] / t[:, 3:4]
        out[i, :, 0] = (xy[:, 0] + 1) * 0.5 * W
        out[i, :, 1] = (xy[:, 1] + 1) * 0.5 * H
    return out


def smooth_pose_seq(x, window):
    out = np.zeros_like(x)
    for i in range(len(x)):
        out[i] = x[max(0, i - window // 2):min(len(x), i + window // 2 + 1)].mean(axis=0)
    return out
