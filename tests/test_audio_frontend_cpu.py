"""Audio front-end (wav2vec2 encoder + Audio2Mesh head) checks that need no GPU: the drop-in's call / state-dict surface
against the reference's (stored in tests/golden/audio_front_end.pt by tests/audio_golden.py), legacy weight-norm checkpoint
keys, the kernel weight layouts, and the errors raised where the kernels do not apply."""
import json
import os
import subprocess
import sys
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GOLDEN = os.path.join(ROOT, "tests", "golden", "audio_front_end.pt")

PROBE = r'''
import inspect, json, sys, tempfile
side = sys.argv[1]
if side == "reference":
    sys.path.insert(0, sys.argv[2]); from oracle import ref_import; ref_import.activate()
else:
    sys.path.insert(0, sys.argv[2] + "/dropin"); sys.path.insert(0, sys.argv[2])
import torch
from transformers import Wav2Vec2Config
from src.audio_models.wav2vec2 import Wav2Vec2Model
from src.audio_models.model import Audio2MeshModel

def sig(fn):
    out = []
    for n, p in inspect.signature(fn).parameters.items():
        if n == "self" or p.kind in (p.VAR_KEYWORD, p.VAR_POSITIONAL):
            continue
        out.append([n, None if p.default is inspect._empty else repr(p.default)])
    return out

with tempfile.TemporaryDirectory() as d:
    Wav2Vec2Config().save_pretrained(d)
    with torch.device("meta"):
        mesh = Audio2MeshModel(dict(out_dim=1404, latent_dim=512, model_path=d, only_last_fetures=True,
                                    from_pretrained=False))
res = {
    "sig": {
        "Wav2Vec2Model.__init__": sig(Wav2Vec2Model.__init__),
        "Wav2Vec2Model.forward": sig(Wav2Vec2Model.forward),
        "Wav2Vec2Model.feature_extract": sig(Wav2Vec2Model.feature_extract),
        "Wav2Vec2Model.encode": sig(Wav2Vec2Model.encode),
        "Audio2MeshModel.__init__": sig(Audio2MeshModel.__init__),
        "Audio2MeshModel.forward": sig(Audio2MeshModel.forward),
        "Audio2MeshModel.infer": sig(Audio2MeshModel.infer),
    },
    "shapes": {k: list(v.shape) for k, v in mesh.state_dict().items()},
    "is_hf_wav2vec2": [c.__name__ for c in Wav2Vec2Model.__mro__ if c.__module__.startswith("transformers.")][:1],
}
print("PROBE_JSON" + json.dumps(res))
'''


def probe_surface(side: str) -> dict:
    """Signatures and state-dict layout of the reference's (side="reference") or the drop-in's ("dropin") audio classes,
    probed in a fresh interpreter (both define a top-level `src` package)."""
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-c", PROBE, side, ROOT], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE_JSON")][-1]
    return json.loads(line[len("PROBE_JSON"):])


def _golden():
    return torch.load(GOLDEN, weights_only=False)


def test_dropin_audio_surface_matches_reference():
    """Signatures, state-dict keys and shapes of dropin/src/audio_models/{wav2vec2,model}.py equal the reference's, so
    audio2mesh.pt / audio2pose.pt load into the same parameters and the scripts' calls bind the same way."""
    want = _golden()["surface"]
    got = probe_surface("dropin")
    assert got["sig"] == want["sig"]
    assert got["shapes"] == want["shapes"]
    assert got["is_hf_wav2vec2"] == want["is_hf_wav2vec2"] == ["Wav2Vec2Model"]


def _small_model():
    from transformers import Wav2Vec2Config
    from aniportrait_b200.audio_models import Wav2Vec2Model
    torch.manual_seed(0)
    return Wav2Vec2Model(Wav2Vec2Config(num_hidden_layers=1)).eval()


def test_legacy_weight_norm_keys_load_into_the_same_weight():
    """The published checkpoints name the positional conv's weight norm `conv.weight_g` / `conv.weight_v` (pre-
    parametrization torch); audio2vid.py loads them with strict=False, so a skipped key would go unnoticed. They must land
    in the same effective conv.weight as the parametrized names."""
    from audio_golden import audio_model_weights
    m = _small_model()
    sd = audio_model_weights(m.state_dict(), 11)
    pre = "encoder.pos_conv_embed.conv."
    g, v = sd.pop(pre + "parametrizations.weight.original0"), sd.pop(pre + "parametrizations.weight.original1")
    legacy = dict(sd, **{pre + "weight_g": g, pre + "weight_v": v})
    fresh = _small_model()
    res = fresh.load_state_dict(legacy, strict=False)
    assert not res.missing_keys and not res.unexpected_keys, res
    want = torch._weight_norm(v, g, 2)
    assert torch.equal(fresh.encoder.pos_conv_embed.conv.weight.detach(), want)
    modern = _small_model()
    modern.load_state_dict(audio_model_weights(modern.state_dict(), 11))
    assert torch.equal(modern.encoder.pos_conv_embed.conv.weight.detach(), want)


def test_packed_layouts_invert_to_module_weights():
    """Tap-major conv packing, the resolved positional-conv weight in [group, tap, in, out] order, the fused q|k|v rows and
    the padded out_fn invert to the module's own (fp16-rounded) weights."""
    from aniportrait_b200 import ops
    from aniportrait_b200.audio_models.wav2vec2 import resolved_pos_conv_weight
    from audio_golden import audio_model_weights
    m = _small_model()
    m.load_state_dict(audio_model_weights(m.state_dict(), 12))
    P = m._build_packed()
    fe = m.feature_extractor.conv_layers
    for (wp, k), layer in zip(P["convs"], fe[1:]):
        w = layer.conv.weight.detach()
        assert k == w.shape[2] and wp.shape == (512, k * 512)
        assert torch.equal(wp.view(512, k, 512).permute(0, 2, 1).float(), w.half().float())
    assert torch.equal(P["c0_w"], fe[0].conv.weight.detach().reshape(512, 10))
    wres = resolved_pos_conv_weight(m.encoder.pos_conv_embed.conv).detach()
    assert P["pc_w"].shape == (16, 128, 48, 48)
    back = P["pc_w"].permute(0, 3, 2, 1).reshape(768, 48, 128)
    assert torch.equal(back.float(), wres.half().float())
    at = m.encoder.layers[0].attention
    assert torch.equal(P["layers"][0]["qkv_w"][768:1536].float(), at.k_proj.weight.detach().half().float())
    assert torch.equal(P["layers"][0]["qkv_b"][1536:], at.v_proj.bias.detach())


def test_audio2mesh_padded_head_and_errors():
    from transformers import Wav2Vec2Config
    from aniportrait_b200 import _lib
    from aniportrait_b200.audio_models import Audio2MeshModel
    from audio_golden import audio_model_weights
    with tempfile.TemporaryDirectory() as d:
        Wav2Vec2Config(num_hidden_layers=1).save_pretrained(d)
        mesh = Audio2MeshModel(dict(out_dim=1404, latent_dim=512, model_path=d, only_last_fetures=True,
                                    from_pretrained=False)).eval()
    sd = mesh.state_dict()
    mesh.load_state_dict(audio_model_weights({k: v for k, v in sd.items() if k.startswith(("in_fn", "out_fn"))}, 13),
                         strict=False)
    heads = mesh._build_heads()
    assert heads["out_w"].shape == (1408, 512) and heads["n"] == 1404
    assert torch.equal(heads["out_w"][:1404].float(), mesh.out_fn.weight.detach().half().float())
    assert not heads["out_w"][1404:].any() and not heads["out_b"][1404:].any()
    assert torch.equal(heads["out_b"][:1404], mesh.out_fn.bias.detach())
    audio = torch.randn(1, 16000)
    with pytest.raises(_lib.ApError, match="CUDA"):
        mesh.infer(audio, 50)
    with pytest.raises(_lib.ApError, match="CUDA"):
        mesh.audio_encoder(audio, 50)
    with pytest.raises(NotImplementedError):
        mesh(audio, torch.zeros(1, 50, 1404), audio_len=torch.tensor([16000]))
    with pytest.raises(NotImplementedError):
        mesh.audio_encoder(audio, 50, attention_mask=torch.ones(1, 16000, dtype=torch.long))
    with pytest.raises(NotImplementedError):
        mesh.audio_encoder(audio, 50, mask_time_indices=torch.zeros(1, 50, dtype=torch.bool))


def test_other_encoder_layouts_raise():
    from transformers import Wav2Vec2Config
    from aniportrait_b200.audio_models import Wav2Vec2Model
    from aniportrait_b200.audio_models.wav2vec2 import check_base_layout, receptive_frames
    check_base_layout(Wav2Vec2Config())
    for kw in (dict(feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True),   # large-lv60 layout
               dict(hidden_size=1024, num_attention_heads=16, intermediate_size=4096),
               dict(num_conv_pos_embeddings=64)):
        with pytest.raises(NotImplementedError):
            check_base_layout(Wav2Vec2Config(**kw))
    with torch.device("meta"):
        m = Wav2Vec2Model(Wav2Vec2Config(feat_extract_norm="layer", do_stable_layer_norm=True)).eval()
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 16000, device="meta"), 50)
    assert receptive_frames(400) == 1 and receptive_frames(399) == 0
