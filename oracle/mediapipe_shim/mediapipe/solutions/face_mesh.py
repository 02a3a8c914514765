"""The FACEMESH_* connection frozensets. They are read with `ast` from the reference's vendored
src/utils/face_landmark.py (FaceLandmarksConnections); importing that file itself needs mediapipe. That mediapipe's own
sets hold the same edges is an assumption that cannot be checked without mediapipe (DESIGN.md §5)."""
import ast
import os

from oracle.ref_import import REFERENCE_ROOT


def _connections():
    path = os.path.join(REFERENCE_ROOT, "src", "utils", "face_landmark.py")
    tree = ast.parse(open(path).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "FaceLandmarksConnections")
    out = {}
    for node in cls.body:
        if isinstance(node, ast.AnnAssign) and isinstance(node.value, ast.List):
            out[node.target.id] = [(c.args[0].value, c.args[1].value) for c in node.value.elts]
    return out


_NAMES = dict(FACEMESH_LIPS="FACE_LANDMARKS_LIPS", FACEMESH_LEFT_EYE="FACE_LANDMARKS_LEFT_EYE",
              FACEMESH_LEFT_EYEBROW="FACE_LANDMARKS_LEFT_EYEBROW", FACEMESH_RIGHT_EYE="FACE_LANDMARKS_RIGHT_EYE",
              FACEMESH_RIGHT_EYEBROW="FACE_LANDMARKS_RIGHT_EYEBROW", FACEMESH_FACE_OVAL="FACE_LANDMARKS_FACE_OVAL")


def __getattr__(name):
    """The sets are read on first use, so that drawing_utils imports where no reference checkout exists."""
    if name not in _NAMES:
        raise AttributeError(name)
    value = frozenset(_connections()[_NAMES[name]])
    globals()[name] = value
    return value
