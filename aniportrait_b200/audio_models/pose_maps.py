"""audio2vid's audio -> pose-map stage (reference scripts/audio2vid.py:161-205) with every step on the device."""
from __future__ import annotations

import random

import numpy as np
import torch

from ..utils.draw_util import FaceMeshVisualizer
from ..utils.pose_util import project_points, smooth_pose_seq

_VISUALIZER = None


def _visualizer():
    global _VISUALIZER
    if _VISUALIZER is None:
        _VISUALIZER = FaceMeshVisualizer(forehead_edge=False)
    return _VISUALIZER


def _on(device, x, dtype=None):
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.asarray(x))
    return t.to(device=device, dtype=dtype or t.dtype)


def head_pose_from_template(pose_temp, seq_len: int) -> np.ndarray:
    """The `pose_temp` branch: the template, then its mirror without the end frames, tiled and cut to seq_len rows."""
    pose_seq = np.asarray(pose_temp)
    mirrored = np.concatenate((pose_seq, pose_seq[-2:0:-1]), axis=0)
    return np.tile(mirrored, (seq_len // len(mirrored) + 1, 1))[:seq_len]


def audio_to_pose_maps(a2m_model, a2p_model, audio_feature, seq_len, lmks3d, trans_mat, width, height, id_seed=None,
                       pose_temp=None, fps=30, chunk_seconds=5):
    """Pose maps of a clip from its audio: CUDA uint8 [seq_len, height, width, 3] (BGR), the `pose_images` of
    Pose2VideoPipeline.

    audio_feature: CUDA [1, samples] (16 kHz); lmks3d [468, 3] and trans_mat [4, 4] of the reference face (numpy or
    tensors). The mesh is a2m_model.infer(audio_feature, seq_len) + lmks3d in fp64. The head pose is `pose_temp`
    (mirrored and tiled, as given) if one is passed; otherwise a2p_model.infer on chunk_seconds chunks of audio, the last
    two merged, rotations halved in the decoder's dtype, then smooth_pose_seq(., 7). id_seed: int or LongTensor; a random
    one in [0, 99] if None, like the reference.

    Divergence: audio of one chunk or less raises IndexError in the reference; here it is decoded as one chunk of
    seq_len frames."""
    device = audio_feature.device
    pred = a2m_model.infer(audio_feature, seq_len)[0]
    pred = pred.reshape(pred.shape[0], -1, 3).to(torch.float64) + _on(device, lmks3d, torch.float64)
    if pose_temp is not None:
        pose_seq = _on(device, head_pose_from_template(pose_temp, seq_len))
    else:
        if id_seed is None:
            id_seed = random.randint(0, 99)
        if not isinstance(id_seed, torch.Tensor):
            id_seed = torch.LongTensor([int(id_seed)])
        id_seed = id_seed.to(device)
        chunk_frames = chunk_seconds * fps
        chunks = list(audio_feature.split(16000 * chunk_seconds, dim=1))
        lens = [chunk_frames] * (len(chunks) - 1) + [seq_len % chunk_frames]
        if len(chunks) > 1:
            chunks[-2] = torch.cat((chunks[-2], chunks[-1]), dim=1)
            lens[-2] += lens[-1]
            del chunks[-1], lens[-1]
        else:
            lens = [seq_len]
        parts = []
        for audio, n in zip(chunks, lens):
            part = a2p_model.infer(audio, n, id_seed)[0].clone()
            part[:, :3] *= 0.5
            parts.append(part)
        pose_seq = smooth_pose_seq(torch.cat(parts, 0).contiguous(), 7)
    verts = project_points(pred, _on(device, trans_mat), pose_seq, [height, width])
    return _visualizer().draw_landmarks_batch((width, height), verts, normed=False)
