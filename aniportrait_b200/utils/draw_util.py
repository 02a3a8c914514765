"""FaceMeshVisualizer (reference src/utils/draw_util.py) on the ap_pose.cu rasteriser, without mediapipe.

The visualiser draws the face-mesh contour edges of 468 / 478 landmarks as thickness-2 cv2 lines on a 512 x 512 BGR canvas
and resizes it to the target size. Each contour is a colour group; groups are drawn in the order below and a later group
overwrites an earlier one where they touch. The byte output equals the reference's (tests/test_pose_maps_gpu.py).
"""
from __future__ import annotations

import numpy as np
import torch

from .. import ops

# Landmark index pairs per colour group, in drawing order. Each pair keeps its (start, end) orientation: cv2's thick line
# is not symmetric in its end points.
FACE_OVAL = ((58, 132), (93, 234), (127, 162), (132, 93), (136, 172), (148, 176), (149, 150), (150, 136), (152, 148),
             (162, 21), (172, 58), (176, 149), (234, 127), (251, 389), (288, 397), (323, 361), (356, 454), (361, 288),
             (365, 379), (377, 152), (378, 400), (379, 378), (389, 356), (397, 365), (400, 377), (454, 323))
# with forehead_edge=True the oval continues over the forehead (mediapipe's full FACEMESH_FACE_OVAL)
FOREHEAD = ((10, 338), (21, 54), (54, 103), (67, 109), (103, 67), (109, 10), (284, 251), (297, 332), (332, 284),
            (338, 297))
LEFT_EYE = ((249, 390), (263, 249), (263, 466), (373, 374), (374, 380), (380, 381), (381, 382), (382, 362), (384, 398),
            (385, 384), (386, 385), (387, 386), (388, 387), (390, 373), (398, 362), (466, 388))
LEFT_EYEBROW = ((276, 283), (282, 295), (283, 282), (293, 334), (295, 285), (296, 336), (300, 293), (334, 296))
RIGHT_EYE = ((7, 163), (33, 7), (33, 246), (144, 145), (145, 153), (153, 154), (154, 155), (155, 133), (157, 173),
             (158, 157), (159, 158), (160, 159), (161, 160), (163, 144), (173, 133), (246, 161))
RIGHT_EYEBROW = ((46, 53), (52, 65), (53, 52), (63, 105), (65, 55), (66, 107), (70, 63), (105, 66))
LIPS_OUTER_BOTTOM_LEFT = ((61, 146), (146, 91), (91, 181), (181, 84), (84, 17))
LIPS_OUTER_BOTTOM_RIGHT = ((17, 314), (314, 405), (405, 321), (321, 375), (375, 291))
LIPS_INNER_BOTTOM_LEFT = ((78, 95), (95, 88), (88, 178), (178, 87), (87, 14))
LIPS_INNER_BOTTOM_RIGHT = ((14, 317), (317, 402), (402, 318), (318, 324), (324, 308))
LIPS_OUTER_TOP_LEFT = ((61, 185), (185, 40), (40, 39), (39, 37), (37, 0))
LIPS_OUTER_TOP_RIGHT = ((0, 267), (267, 269), (269, 270), (270, 409), (409, 291))
LIPS_INNER_TOP_LEFT = ((78, 191), (191, 80), (80, 81), (81, 82), (82, 13))
LIPS_INNER_TOP_RIGHT = ((13, 312), (312, 311), (311, 310), (310, 415), (415, 308))

# (edges, colour as written into the image: B, G, R)
GROUPS = (
    (FACE_OVAL, (10, 200, 10)),
    (LEFT_EYE, (180, 200, 10)),
    (LEFT_EYEBROW, (180, 220, 10)),
    (RIGHT_EYE, (10, 200, 180)),
    (RIGHT_EYEBROW, (10, 220, 180)),
    (LIPS_OUTER_BOTTOM_LEFT, (10, 180, 20)),
    (LIPS_OUTER_BOTTOM_RIGHT, (20, 10, 180)),
    (LIPS_INNER_BOTTOM_LEFT, (100, 100, 30)),
    (LIPS_INNER_BOTTOM_RIGHT, (100, 150, 50)),
    (LIPS_OUTER_TOP_LEFT, (20, 80, 100)),
    (LIPS_OUTER_TOP_RIGHT, (80, 100, 20)),
    (LIPS_INNER_TOP_LEFT, (120, 100, 200)),
    (LIPS_INNER_TOP_RIGHT, (150, 120, 100)),
)


def connection_groups(forehead_edge: bool = False):
    """The visualiser's [(edges, colour)] in drawing order."""
    if not forehead_edge:
        return list(GROUPS)
    return [(FACE_OVAL + FOREHEAD, GROUPS[0][1])] + list(GROUPS[1:])


class FaceMeshVisualizer:
    """Reference-compatible face-mesh pose-map renderer on the device. draw_landmarks keeps the reference's numpy
    signature; draw_landmarks_batch renders L frames from CUDA keypoints in one call."""

    def __init__(self, forehead_edge=False):
        self.forehead_edge = forehead_edge
        groups = connection_groups(forehead_edge)
        self._edges = np.array([(a, b, g) for g, (edges, _) in enumerate(groups) for a, b in edges], dtype=np.int32)
        self._colours = np.array([c for _, c in groups], dtype=np.uint8)
        self._max_index = int(self._edges[:, :2].max())
        self._device_tables = {}

    def _tables(self, device):
        """The edge and colour tables on `device`, uploaded once."""
        tables = self._device_tables.get(device)
        if tables is None:
            tables = (torch.from_numpy(self._edges).to(device), torch.from_numpy(self._colours).to(device))
            self._device_tables[device] = tables
        return tables

    def draw_landmarks_batch(self, image_size, keypoints, normed=False):
        """keypoints: CUDA [L, N, 2] (fp32 / fp64), pixel coordinates of an image_size = (W, H) image, or normalised
        ones with normed=True. Returns CUDA uint8 [L, H, W, 3] (BGR); W and H must be multiples of 8."""
        if not isinstance(keypoints, torch.Tensor) or keypoints.dim() != 3 or keypoints.shape[2] < 2:
            raise ValueError("draw_landmarks_batch: keypoints must be a [L, N, 2] tensor")
        if keypoints.shape[1] <= self._max_index:
            raise ValueError(f"Landmark index is out of range: the face mesh needs {self._max_index + 1} landmarks, "
                             f"got {keypoints.shape[1]}")
        if keypoints.shape[2] != 2:
            keypoints = keypoints[..., :2]
        edges, colours = self._tables(keypoints.device)
        return ops.facemesh_raster(keypoints, edges, colours, int(image_size[0]), int(image_size[1]), normed=normed)

    def draw_landmarks(self, image_size, keypoints, normed=False):
        """Reference signature: keypoints numpy [N, >= 2] -> numpy uint8 [H, W, 3] (BGR). Renders on the current CUDA
        device."""
        kp = np.asarray(keypoints)
        if kp.dtype not in (np.float32, np.float64):
            kp = kp.astype(np.float64)
        kp = torch.from_numpy(np.ascontiguousarray(kp[None, :, :2])).to(torch.device("cuda", torch.cuda.current_device()))
        return self.draw_landmarks_batch(image_size, kp, normed=normed)[0].cpu().numpy()
