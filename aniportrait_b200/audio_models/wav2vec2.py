"""wav2vec2-base encoder of audio2vid on sm_100a kernels (reference src/audio_models/wav2vec2.py:13-125).

The reference subclasses transformers' Wav2Vec2Model, adds `seq_len` (the encoder features are linearly resampled to the
video frame count before the feature projection, wav2vec2.py:30-32) and runs everything as fp32 library code. This class
keeps the reference's call surface, configuration, `from_pretrained` and state-dict keys (all inherited from transformers),
and on a CUDA device runs the forward on the project's kernels only:

  waveform -> layer 0: conv k=10/s=5 + per-channel GroupNorm + GELU        ap_wav_conv0_gn_gelu_f16
           -> layers 1-6: conv k=3|2/s=2 + GELU as GEMMs over strided views  ap_gemm_f16 (AP_GEMM_GELU, two K sources)
           -> linear interpolation to seq_len frames                      ap_interp_linear_time_f16
           -> feature projection: LayerNorm(512) + Linear(512, 768)         ap_layernorm_f16, ap_gemm_f16
           -> x + GELU(grouped positional conv(x)), LayerNorm              ap_pos_conv_gelu_f16, ap_layernorm_f16
           -> 12 post-LN layers: fused q|k|v GEMM, attention, out_proj + residual, LayerNorm, intermediate_dense + GELU,
              output_dense + residual, LayerNorm                             ap_gemm_f16, ap_attention_f16, ap_layernorm_f16
           -> outputs in the module's dtype                                ap_mean_f16 (fp16 -> fp32)

Activations are fp16 channels-last [T, C] with fp32 accumulation; the module may stay fp32 (as audio2vid.py:68 keeps it):
the fp16 kernel-layout copies of its weights are built once per parameter state (PackedCache). There is no CPU path and no
fallback: a CPU tensor, a batch of more than one clip, training-only arguments and other encoder layouts raise.
"""
from __future__ import annotations

import torch
from transformers import Wav2Vec2Config, Wav2Vec2Model as _HFWav2Vec2Model
from transformers.modeling_outputs import BaseModelOutput

from .. import _lib, ops
from ..models.modeling import PackedCache, f16, f32

MIN_SAMPLES = 400   # receptive field of the conv stack: 400 samples give one frame after layer 6

# the feature-extractor / encoder layout the kernels implement: wav2vec2-base (transformers' default Wav2Vec2Config)
_BASE_LAYOUT = dict(feat_extract_norm="group", conv_bias=False, conv_dim=(512,) * 7, conv_kernel=(10, 3, 3, 3, 3, 2, 2),
                    conv_stride=(5, 2, 2, 2, 2, 2, 2), hidden_size=768, num_attention_heads=12, intermediate_size=3072,
                    do_stable_layer_norm=False, hidden_act="gelu", feat_extract_activation="gelu",
                    num_conv_pos_embeddings=128, num_conv_pos_embedding_groups=16, add_adapter=False)


def check_base_layout(config: Wav2Vec2Config):
    """Raises NotImplementedError unless `config` has the wav2vec2-base layout the kernels implement (any layer count)."""
    for key, want in _BASE_LAYOUT.items():
        got = getattr(config, key, None)
        if isinstance(want, tuple):
            got = tuple(got) if got is not None else None
        if got != want:
            raise NotImplementedError(f"aniportrait_b200 Wav2Vec2Model implements the wav2vec2-base layout: config.{key} "
                                      f"is {got!r}, the kernels need {want!r}")


def resolved_pos_conv_weight(conv: torch.nn.Conv1d) -> torch.Tensor:
    """The effective weight of the weight-normed positional conv (parametrized or legacy weight_g / weight_v form)."""
    if hasattr(conv, "weight_g") and hasattr(conv, "weight_v"):
        return torch._weight_norm(conv.weight_v, conv.weight_g, 2)
    return conv.weight


def receptive_frames(samples: int) -> int:
    """Frames after the 7 feature-extractor convolutions for `samples` input samples."""
    t = samples
    for k, s in zip(_BASE_LAYOUT["conv_kernel"], _BASE_LAYOUT["conv_stride"]):
        t = (t - k) // s + 1
    return t


class Wav2Vec2Model(_HFWav2Vec2Model):
    def __init__(self, config: Wav2Vec2Config):
        super().__init__(config)
        self._packed = PackedCache()

    # ------------------------------------------------------------------ weights in kernel layout
    @torch.no_grad()
    def _build_packed(self):
        fe = self.feature_extractor.conv_layers
        fp = self.feature_projection
        pc = self.encoder.pos_conv_embed.conv
        P = dict(
            c0_w=f32(fe[0].conv.weight.reshape(fe[0].conv.weight.shape[0], -1)),
            c0_g=f32(fe[0].layer_norm.weight), c0_b=f32(fe[0].layer_norm.bias), c0_eps=float(fe[0].layer_norm.eps),
            convs=[(ops.pack_conv1d_taps(l.conv.weight), l.conv.kernel_size[0]) for l in fe[1:]],
            fp_ln=(f32(fp.layer_norm.weight), f32(fp.layer_norm.bias), float(fp.layer_norm.eps)),
            fp_w=f16(fp.projection.weight), fp_b=f32(fp.projection.bias),
            pc_w=ops.pack_pos_conv_weight(resolved_pos_conv_weight(pc)), pc_b=f32(pc.bias),
            enc_ln=(f32(self.encoder.layer_norm.weight), f32(self.encoder.layer_norm.bias),
                    float(self.encoder.layer_norm.eps)),
            layers=[])
        for layer in self.encoder.layers:
            at, ff = layer.attention, layer.feed_forward
            P["layers"].append(dict(
                qkv_w=f16(torch.cat([at.q_proj.weight, at.k_proj.weight, at.v_proj.weight])),
                qkv_b=f32(torch.cat([at.q_proj.bias, at.k_proj.bias, at.v_proj.bias])),
                o_w=f16(at.out_proj.weight), o_b=f32(at.out_proj.bias),
                ln1=(f32(layer.layer_norm.weight), f32(layer.layer_norm.bias), float(layer.layer_norm.eps)),
                i_w=f16(ff.intermediate_dense.weight), i_b=f32(ff.intermediate_dense.bias),
                out_w=f16(ff.output_dense.weight), out_b=f32(ff.output_dense.bias),
                ln2=(f32(layer.final_layer_norm.weight), f32(layer.final_layer_norm.bias),
                     float(layer.final_layer_norm.eps))))
        return P

    def packed(self):
        return self._packed.get(self, self._build_packed)

    # ------------------------------------------------------------------ kernel path
    def _check_call(self, x: torch.Tensor, attention_mask, mask_time_indices):
        if attention_mask is not None or mask_time_indices is not None:
            raise NotImplementedError("attention_mask / mask_time_indices (training-time padding and SpecAugment masking) "
                                      "are not supported: aniportrait_b200 runs the inference path of audio2vid")
        if self.training:
            raise NotImplementedError("aniportrait_b200 Wav2Vec2Model runs in eval mode only (call .eval())")
        check_base_layout(self.config)
        if not x.is_cuda:
            raise _lib.ApError("aniportrait_b200 Wav2Vec2Model needs CUDA tensors (no CPU fallback)")
        if x.dim() != 2 and x.dim() != 3:
            raise ValueError(f"expected [batch, samples] (or [batch, frames, channels] for encode), got {tuple(x.shape)}")
        if x.shape[0] != 1:
            raise ValueError(f"aniportrait_b200 Wav2Vec2Model encodes one clip at a time (batch {x.shape[0]})")

    def _features_f16(self, input_values: torch.Tensor, seq_len: int) -> torch.Tensor:
        """Feature extractor + interpolation: [1, S] waveform -> fp16 [seq_len, 512]."""
        S = input_values.shape[-1]
        if S < MIN_SAMPLES:
            raise ValueError(f"audio of {S} samples is shorter than the encoder's receptive field ({MIN_SAMPLES} samples)")
        seq_len = int(seq_len)
        if seq_len < 1:
            raise ValueError(f"seq_len must be >= 1 (got {seq_len})")
        P = self.packed()
        wav = input_values.reshape(-1).to(torch.float32).contiguous()
        x = ops.wav_conv0_gn_gelu(wav, P["c0_w"], P["c0_g"], P["c0_b"], P["c0_eps"])
        for w, k in P["convs"]:
            x = ops.conv1d_s2_gelu(x, w, k)
        return ops.interp_linear_time(x, seq_len)

    def _encode_f16(self, feats: torch.Tensor, want_states: bool):
        """Feature projection + encoder on fp16 [T, 512] -> (last hidden state fp16 [T, 768], stacked states
        fp16 [layers + 1, T, 768] or None)."""
        P = self.packed()
        T = feats.shape[0]
        g, b, eps = P["fp_ln"]
        h = ops.gemm(ops.layer_norm(feats, g, b, eps), P["fp_w"], P["fp_b"])
        h = ops.pos_conv_gelu(h, P["pc_w"], P["pc_b"])
        states = torch.empty(len(P["layers"]) + 1, T, h.shape[1], dtype=torch.float16, device=h.device) \
            if want_states else None
        g, b, eps = P["enc_ln"]
        h = ops.layer_norm(h, g, b, eps, out=states[0] if want_states else None)
        heads = self.config.num_attention_heads
        d = self.config.hidden_size // heads
        C = self.config.hidden_size
        for i, L in enumerate(P["layers"]):
            qkv = ops.gemm(h, L["qkv_w"], L["qkv_b"])
            a = ops.attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], 1, T, heads, d, d, scale=d ** -0.5)
            h1 = ops.gemm(a, L["o_w"], L["o_b"], residual=h)
            h1 = ops.layer_norm(h1, *L["ln1"])
            f = ops.gemm(h1, L["i_w"], L["i_b"], gelu=True)
            h2 = ops.gemm(f, L["out_w"], L["out_b"], residual=h1)
            h = ops.layer_norm(h2, *L["ln2"], out=states[i + 1] if want_states else None)
        return h, states

    def _to_module_dtype(self, x16: torch.Tensor) -> torch.Tensor:
        """fp16 [T, C] -> [1, T, C] in the module's dtype (fp32 through ap_mean_f16, fp16 as is)."""
        if self.dtype == torch.float16:
            return x16.unsqueeze(0)
        if self.dtype != torch.float32:
            raise NotImplementedError(f"aniportrait_b200 Wav2Vec2Model returns fp32 or fp16 (module dtype {self.dtype})")
        return ops.mean_f16(x16.unsqueeze(0)).unsqueeze(0)

    def _outputs(self, h, states, output_hidden_states, return_dict):
        last = self._to_module_dtype(h)
        all_states = tuple(self._to_module_dtype(s) for s in states) if output_hidden_states else None
        if not return_dict:
            return tuple(v for v in (last, all_states) if v is not None)
        return BaseModelOutput(last_hidden_state=last, hidden_states=all_states, attentions=None)

    # ------------------------------------------------------------------ reference surface
    @torch.no_grad()
    def forward(self, input_values, seq_len, attention_mask=None, mask_time_indices=None, output_attentions=None,
                output_hidden_states=None, return_dict=None):
        self._check_call(input_values, attention_mask, mask_time_indices)
        output_hidden_states = (output_hidden_states if output_hidden_states is not None
                                else self.config.output_hidden_states)
        return_dict = return_dict if return_dict is not None else self.config.return_dict
        feats = self._features_f16(input_values, seq_len)
        h, states = self._encode_f16(feats, bool(output_hidden_states))
        return self._outputs(h, states, output_hidden_states, return_dict)

    @torch.no_grad()
    def feature_extract(self, input_values, seq_len):
        self._check_call(input_values, None, None)
        return self._to_module_dtype(self._features_f16(input_values, seq_len))

    @torch.no_grad()
    def encode(self, extract_features, attention_mask=None, mask_time_indices=None, output_attentions=None,
               output_hidden_states=None, return_dict=None):
        self._check_call(extract_features, attention_mask, mask_time_indices)
        output_hidden_states = (output_hidden_states if output_hidden_states is not None
                                else self.config.output_hidden_states)
        return_dict = return_dict if return_dict is not None else self.config.return_dict
        # the caller's [1, T, 512] features (fp32 from feature_extract in an fp32 module) -> the kernels' fp16 operand
        feats = extract_features[0].to(torch.float16).contiguous()
        h, states = self._encode_f16(feats, bool(output_hidden_states))
        return self._outputs(h, states, output_hidden_states, return_dict)
