"""TEST INFRASTRUCTURE — the few mediapipe leaves that the reference's src/utils/draw_util.py imports, restated so that
tests/pose_golden.py can run the unmodified FaceMeshVisualizer without mediapipe. Nothing in the product imports this."""
from . import framework, solutions  # noqa: F401
