"""Import-path shim (see dropin/src/models/unet_3d.py): the face-mesh visualiser on the device, without mediapipe.
src/utils is a namespace package, so the reference's own pose_util, mp_utils and the rest still resolve to the reference."""
from aniportrait_b200.utils.draw_util import FaceMeshVisualizer  # noqa: F401
