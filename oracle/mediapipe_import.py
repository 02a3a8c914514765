"""TEST INFRASTRUCTURE — puts oracle/mediapipe_shim on sys.path: the mediapipe leaves that the reference's
src/utils/draw_util.py imports. Used next to oracle.ref_import.activate() by tests/pose_golden.py, and alone by the host
arm of scripts/bench_pose_maps.py (which draws through the shim's drawing_utils and needs no reference checkout)."""
import os
import sys

MEDIAPIPE_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mediapipe_shim")


def activate_shim():
    """Only the mediapipe shim (part of this repository)."""
    if MEDIAPIPE_SHIM not in sys.path:
        sys.path.insert(0, MEDIAPIPE_SHIM)


def activate():
    """The unmodified reference (oracle.ref_import.activate) plus the mediapipe shim."""
    from oracle import ref_import
    ref_import.activate()
    activate_shim()
