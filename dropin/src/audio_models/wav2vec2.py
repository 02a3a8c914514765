"""Import-path shim (see dropin/src/models/unet_3d.py). The reference's own src/audio_models/pose_model.py imports
`from .wav2vec2 import Wav2Vec2Model`; src/audio_models has no __init__.py, so it resolves to this module and
Audio2PoseModel builds its audio encoder from the kernel implementation."""
from aniportrait_b200.audio_models.wav2vec2 import Wav2Vec2Model  # noqa: F401
