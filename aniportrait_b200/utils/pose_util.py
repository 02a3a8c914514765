"""Head-pose smoothing and landmark projection of reference src/utils/pose_util.py on CUDA tensors (ap_pose.cu). The
arguments keep the reference's order; the results stay on the device."""
from __future__ import annotations

import torch

from .. import ops


def smooth_pose_seq(pose_seq: torch.Tensor, window_size: int = 5) -> torch.Tensor:
    """Sliding-window mean over the rows of [L, 6] (fp32 or fp64), bit-identical to the reference's numpy."""
    return ops.pose_smooth(pose_seq, window_size)


def project_points(points_3d: torch.Tensor, transformation_matrix: torch.Tensor, pose_vectors: torch.Tensor,
                   image_shape) -> torch.Tensor:
    """points_3d [L, N, 3], transformation_matrix [4, 4], pose_vectors [>= L, 6] (xyz Euler degrees, translation),
    image_shape = (H, W) -> fp64 [L, N, 2] pixel coordinates."""
    return ops.project_points(points_3d, transformation_matrix, pose_vectors, int(image_shape[1]), int(image_shape[0]))


def project_points_with_trans(points_3d: torch.Tensor, transformation_matrix: torch.Tensor, image_shape) -> torch.Tensor:
    """points_3d [L, N, 3] with per-frame matrices [L, 4, 4], image_shape = (H, W) -> fp64 [L, N, 2]."""
    return ops.project_points(points_3d, transformation_matrix, None, int(image_shape[1]), int(image_shape[0]))
