"""Import-path shim (see dropin/src/models/unet_3d.py)."""
from aniportrait_b200.audio_models.model import Audio2MeshModel  # noqa: F401
