"""draw_landmarks as mediapipe's solutions.drawing_utils defines it, for the call the reference makes
(landmark_drawing_spec=None: connections only)."""
import math
from collections.abc import Mapping

import cv2

from .drawing_styles import DrawingSpec

_BGR_CHANNELS = 3


def _normalized_to_pixel_coordinates(normalized_x, normalized_y, image_width, image_height):
    def is_valid_normalized_value(value):
        return (value > 0 or math.isclose(0, value)) and (value < 1 or math.isclose(1, value))

    if not (is_valid_normalized_value(normalized_x) and is_valid_normalized_value(normalized_y)):
        return None
    x_px = min(math.floor(normalized_x * image_width), image_width - 1)
    y_px = min(math.floor(normalized_y * image_height), image_height - 1)
    return x_px, y_px


def draw_landmarks(image, landmark_list, connections=None, landmark_drawing_spec=DrawingSpec(color=(0, 0, 255)),
                   connection_drawing_spec=DrawingSpec()):
    if not landmark_list:
        return
    if image.shape[2] != _BGR_CHANNELS:
        raise ValueError("Input image must contain three channel bgr data.")
    image_rows, image_cols, _ = image.shape
    idx_to_coordinates = {}
    for idx, landmark in enumerate(landmark_list.landmark):
        landmark_px = _normalized_to_pixel_coordinates(landmark.x, landmark.y, image_cols, image_rows)
        if landmark_px:
            idx_to_coordinates[idx] = landmark_px
    if connections:
        num_landmarks = len(landmark_list.landmark)
        for connection in connections:
            start_idx, end_idx = connection[0], connection[1]
            if not (0 <= start_idx < num_landmarks and 0 <= end_idx < num_landmarks):
                raise ValueError(f"Landmark index is out of range. Invalid connection from landmark #{start_idx} "
                                 f"to landmark #{end_idx}.")
            if start_idx in idx_to_coordinates and end_idx in idx_to_coordinates:
                spec = connection_drawing_spec[connection] if isinstance(connection_drawing_spec, Mapping) \
                    else connection_drawing_spec
                cv2.line(image, idx_to_coordinates[start_idx], idx_to_coordinates[end_idx], spec.color, spec.thickness)
    if landmark_drawing_spec:
        raise NotImplementedError("landmark circles: the reference passes landmark_drawing_spec=None")
