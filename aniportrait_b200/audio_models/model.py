"""Audio2MeshModel on sm_100a kernels (reference src/audio_models/model.py:11-69; audio2vid.py:66-68,162).

Same constructor (the inference_audio.yaml `a2m_model` dict), same submodules and state-dict keys, so
`load_state_dict(torch.load("audio2mesh.pt"), strict=False)` fills the same parameters. `infer` runs the wav2vec2 encoder
(aniportrait_b200.audio_models.wav2vec2) and the two linear heads on the device: in_fn as an fp16 GEMM, out_fn as a GEMM
with an fp32 output (out_dim 1404 padded to a multiple of 32 weight rows; the padding columns are not written).
"""
from __future__ import annotations

import torch
import torch.nn as nn
from transformers import Wav2Vec2Config

from .. import ops
from ..models.modeling import PackedCache, f16, f32
from .wav2vec2 import Wav2Vec2Model


class Audio2MeshModel(nn.Module):
    def __init__(self, config):
        super().__init__()
        out_dim = config['out_dim']
        latent_dim = config['latent_dim']
        model_path = config['model_path']
        only_last_fetures = config['only_last_fetures']
        from_pretrained = config['from_pretrained']

        self._only_last_features = only_last_fetures

        self.audio_encoder_config = Wav2Vec2Config.from_pretrained(model_path, local_files_only=True)
        if from_pretrained:
            self.audio_encoder = Wav2Vec2Model.from_pretrained(model_path, local_files_only=True)
        else:
            self.audio_encoder = Wav2Vec2Model(self.audio_encoder_config)
        self.audio_encoder.feature_extractor._freeze_parameters()

        hidden_size = self.audio_encoder_config.hidden_size

        self.in_fn = nn.Linear(hidden_size, latent_dim)

        self.out_fn = nn.Linear(latent_dim, out_dim)
        nn.init.constant_(self.out_fn.weight, 0)
        nn.init.constant_(self.out_fn.bias, 0)
        self._packed = PackedCache()

    @torch.no_grad()
    def _build_heads(self):
        n = self.out_fn.out_features
        n_pad = (n + 31) // 32 * 32
        w = torch.zeros(n_pad, self.out_fn.in_features, dtype=torch.float16, device=self.out_fn.weight.device)
        w[:n] = self.out_fn.weight
        b = torch.zeros(n_pad, dtype=torch.float32, device=self.out_fn.weight.device)
        b[:n] = self.out_fn.bias
        return dict(in_w=f16(self.in_fn.weight), in_b=f32(self.in_fn.bias), out_w=w, out_b=b, n=n)

    def forward(self, audio, label, audio_len=None):
        if audio_len is not None:
            raise NotImplementedError("audio_len (padded training batches with an attention mask) is not supported: "
                                      "aniportrait_b200 runs the inference path of audio2vid")
        return self.infer(audio, label.shape[1]), None

    @torch.no_grad()
    def infer(self, input_value, seq_len):
        enc = self.audio_encoder
        enc._check_call(input_value, None, None)
        heads = self._packed.get(self, self._build_heads)
        h, states = enc._encode_f16(enc._features_f16(input_value, seq_len), not self._only_last_features)
        if not self._only_last_features:
            # sum(hidden_states) / len(hidden_states) in fp32, in the reference's order, rounded once for the GEMM
            h = ops.mean_f16(states, out_f32=False, out_f16=True)
        layer_in = ops.gemm(h, heads["in_w"], heads["in_b"])
        out = ops.gemm(layer_in, heads["out_w"], heads["out_b"], n_valid=heads["n"], out_f32=True)
        return out.unsqueeze(0)
