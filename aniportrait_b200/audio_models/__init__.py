"""Audio front-end of audio2vid (SURVEY.md 8f, N3): the wav2vec2-base encoder and the Audio2Mesh head on the project's
kernels, and the incremental (KV-cached) head-pose decoder loop."""
from .model import Audio2MeshModel  # noqa: F401
from .pose_maps import audio_to_pose_maps  # noqa: F401
from .pose_infer import enable_kv_cache, kv_cached_infer  # noqa: F401
from .wav2vec2 import Wav2Vec2Model  # noqa: F401
