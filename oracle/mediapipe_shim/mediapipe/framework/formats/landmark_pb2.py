"""NormalizedLandmarkList with the protobuf's field types: x, y and z are `float` fields, so every value is stored as
fp32 and read back as the Python float of that fp32 value."""
import numpy as np


def _f32(v):
    return float(np.float32(v))


class NormalizedLandmark:
    def __init__(self):
        self._x = self._y = self._z = 0.0

    x = property(lambda self: self._x, lambda self, v: setattr(self, "_x", _f32(v)))
    y = property(lambda self: self._y, lambda self, v: setattr(self, "_y", _f32(v)))
    z = property(lambda self: self._z, lambda self, v: setattr(self, "_z", _f32(v)))

    def HasField(self, name):
        # visibility and presence are never set by the reference's draw_landmarks
        return False


class _Repeated(list):
    def add(self):
        lm = NormalizedLandmark()
        self.append(lm)
        return lm


class NormalizedLandmarkList:
    def __init__(self):
        self.landmark = _Repeated()
