"""Golden data of the audio front-end (tests/golden/audio_front_end.pt) and the seeded weights / audio it is made from.

    python tests/audio_golden.py          # needs a reference checkout (oracle/ref_import.py), runs on the CPU

Runs the UNMODIFIED reference wav2vec2 wrapper, Audio2MeshModel.infer and Audio2PoseModel.infer (one 5 s chunk) at the real
wav2vec2-base geometry (transformers' default Wav2Vec2Config) with seeded weights, in fp32 on the CPU, and stores only a
strided sample of their outputs plus the reference classes' call / state-dict surface. The functions that regenerate the
weights and the audio are imported by the tests and by scripts/bench_audio.py, so nothing but outputs is stored.
"""
from __future__ import annotations

import math
import os
import sys
import time
import zlib

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "audio_front_end.pt")

AUDIO_SEEDS = dict(encoder=701, mesh_heads=702, pose=703, audio_5s=704, audio_ragged=705)
AUDIO_CLIPS = dict(audio_5s=(80000, 150), audio_ragged=(52817, 100))     # (samples, seq_len)
AUDIO_MESH = dict(out_dim=1404, latent_dim=512, only_last_fetures=True)  # inference_audio.yaml a2m_model
AUDIO_POSE = dict(out_dim=6, latent_dim=512, only_last_fetures=True)     # inference_audio.yaml a2p_model
AUDIO_ID_SEED = 7
AUDIO_ROW_STRIDE = 4       # the stored outputs keep every 4th frame (fixture size)


def audio_clip(samples, seed):
    """Seeded audio as prepare_audio_feature hands it to the encoder: zero mean, unit variance (Wav2Vec2FeatureExtractor
    do_normalize), [1, samples] fp32. A few tones under noise so that neighbouring frames differ smoothly."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(samples, dtype=torch.float64) / 16000.0
    x = 0.3 * torch.randn(samples, generator=g, dtype=torch.float64)
    for f, a in zip((110.0, 220.0, 455.0, 1300.0), torch.rand(4, generator=g, dtype=torch.float64)):
        x += a * torch.sin(2 * math.pi * f * t * (1.0 + 0.2 * torch.sin(2 * math.pi * 0.7 * t)))
    x = (x - x.mean()) / torch.sqrt(x.var(unbiased=False) + 1e-7)
    return x.to(torch.float32).unsqueeze(0)


def audio_model_weights(sd: dict, seed: int) -> dict:
    """Seeded weights for a wav2vec2 encoder plus linear heads (keys as given, any prefix): norm scales 1 + 0.1 N(0, 1),
    biases 0.02 N(0, 1), every matrix / conv kernel N(0, 1 / fan_in) (so activations keep unit scale through 12 layers), the
    weight-normed positional conv with per-tap norms of the same fan-in scale. Per-tensor generators seeded by
    (seed, crc32(name)): independent of key order. (synthetic.randomize_state_dict gives wav2vec2's layer_norm weights
    small signed values: its norm-name list does not match them.)"""
    out = {}
    for name, t in sd.items():
        g = torch.Generator().manual_seed((seed * 1000003 + zlib.crc32(name.encode())) & 0x7FFFFFFF)
        leaf = name.rsplit(".", 1)[-1]
        if not t.is_floating_point():
            out[name] = t.clone()
        elif name.endswith("parametrizations.weight.original0"):       # weight-norm g [1, 1, k]: ||w[:, :, k]||
            v_shape = sd[name[:-1] + "1"].shape                        # v [out, in/groups, k]
            fan_in = v_shape[1] * v_shape[2]
            scale = math.sqrt(v_shape[0] * v_shape[1] / fan_in)
            out[name] = (scale * (1.0 + 0.1 * torch.randn(t.shape, generator=g))).to(t.dtype)
        elif ("norm" in name) and leaf == "weight":
            out[name] = (1.0 + 0.1 * torch.randn(t.shape, generator=g)).to(t.dtype)
        elif leaf == "bias" or t.dim() == 1:
            out[name] = (0.02 * torch.randn(t.shape, generator=g)).to(t.dtype)
        else:
            fan_in = t[0].numel()
            out[name] = (torch.randn(t.shape, generator=g) / math.sqrt(fan_in)).to(t.dtype)
    return out


def audio_encoder_config_dir(path):
    """A Wav2Vec2Config() directory for the constructors' `model_path` (eager attention: the reference's wrapper asks
    for attention maps)."""
    from transformers import Wav2Vec2Config
    cfg = Wav2Vec2Config()
    cfg._attn_implementation = "eager"
    cfg.save_pretrained(path)
    return path


def audio_mesh_state(model) -> dict:
    sd = model.state_dict()
    return audio_model_weights(sd, AUDIO_SEEDS["encoder"]) | audio_model_weights(
        {k: v for k, v in sd.items() if not k.startswith("audio_encoder.")}, AUDIO_SEEDS["mesh_heads"])


def audio_pose_state(model) -> dict:
    """Encoder weights as audio_model_weights draws them, everything else as oracle.make_golden.pose_model_weights (the
    decoder recipe of the reference_units pose case)."""
    from oracle.make_golden import pose_model_weights
    sd = model.state_dict()
    enc = audio_model_weights({k: v for k, v in sd.items() if k.startswith("audio_encoder.")}, AUDIO_SEEDS["encoder"])
    return enc | pose_model_weights(model, AUDIO_SEEDS["pose"])


def mask_from_last_row(row: torch.Tensor) -> torch.Tensor:
    """[heads, T] last query row of a causal, shift-invariant (Toeplitz) additive mask -> the [heads, T, T] mask:
    entry (i, j) = row[T - 1 - (i - j)] for j <= i, -inf above the diagonal. The generator checks that the reference's
    ALiBi mask has exactly this form before storing only its last row."""
    T = row.shape[-1]
    i = torch.arange(T).view(T, 1)
    j = torch.arange(T).view(1, T)
    idx = (T - 1 - (i - j)).clamp(0, T - 1)
    mask = row[:, idx]
    return mask.masked_fill((j > i).unsqueeze(0), float("-inf"))


def make_golden():
    import tempfile
    from oracle import ref_import
    ref_import.activate()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from src.audio_models.model import Audio2MeshModel
    from src.audio_models.pose_model import Audio2PoseModel
    from test_audio_frontend_cpu import probe_surface
    from aniportrait_b200.synthetic import _sinusoid_pe
    t0 = time.time()
    S = AUDIO_ROW_STRIDE
    G = dict(case="audio_front_end", torch_version=str(torch.__version__), seeds=dict(AUDIO_SEEDS), clips=dict(AUDIO_CLIPS),
             row_stride=S, generator="reference src/audio_models via transformers, fp32 CPU")
    wall = {}
    with tempfile.TemporaryDirectory() as cfg_dir:
        audio_encoder_config_dir(cfg_dir)
        torch.manual_seed(0)
        mesh = Audio2MeshModel(dict(AUDIO_MESH, model_path=cfg_dir, from_pretrained=False)).eval()
        mesh.audio_encoder.config._attn_implementation = "eager"
        mesh.load_state_dict(audio_mesh_state(mesh))
        enc = mesh.audio_encoder
        with torch.no_grad():
            for clip, (samples, T) in AUDIO_CLIPS.items():
                audio = audio_clip(samples, AUDIO_SEEDS[clip])
                t1 = time.perf_counter()
                emb = enc(audio, seq_len=T, output_hidden_states=True)
                wall[f"encoder_{clip}"] = time.perf_counter() - t1
                last = emb.last_hidden_state[0]
                mean = (sum(emb.hidden_states) / len(emb.hidden_states))[0]
                assert len(emb.hidden_states) == 13 and last.shape == (T, 768)
                spread = (last[1:] - last[:-1]).abs().mean().item()
                assert spread > 1e-2 and last.std().item() > 0.1, "degenerate reference encoder output"
                G[f"{clip}_last"] = last[::S].half()
                G[f"{clip}_mean"] = mean[::S].half()
                G[f"{clip}_state_norms"] = torch.stack([s[0].norm() for s in emb.hidden_states])
            samples, T = AUDIO_CLIPS["audio_5s"]
            audio = audio_clip(samples, AUDIO_SEEDS["audio_5s"])
            t1 = time.perf_counter()
            out = mesh.infer(audio, T)
            wall["mesh_infer_audio_5s"] = time.perf_counter() - t1
            assert out.shape == (1, T, AUDIO_MESH["out_dim"]) and out.std().item() > 1e-2, "degenerate Audio2Mesh output"
            G["mesh_infer"] = out[0, ::S].half()
            G["mesh_infer_norm"] = out.norm().item()

        torch.manual_seed(0)
        pose = Audio2PoseModel(dict(AUDIO_POSE, model_path=cfg_dir, from_pretrained=False)).eval()
        pose.audio_encoder.config._attn_implementation = "eager"
        pose.load_state_dict(audio_pose_state(pose))
        with torch.no_grad():
            t1 = time.perf_counter()
            want = pose.infer(audio, T, id_seed=torch.tensor([AUDIO_ID_SEED]))
            wall["pose_infer_audio_5s"] = time.perf_counter() - t1
        spread = (want[0, 1:] - want[0, :-1]).abs().mean().item()
        assert want.shape == (1, T, 6) and spread > 1e-3, "degenerate reference pose output"
        G["pose_infer"] = want
        mask = pose.biased_mask[:, :T, :T].clone()
        row = mask[:, T - 1].clone()
        assert torch.equal(mask_from_last_row(row), mask), "the reference's pose mask is not causal shift-invariant"
        G["pose_mask_last_row"] = row
        assert torch.equal(pose.PPE.pe, _sinusoid_pe(pose.PPE.pe.shape[1], pose.PPE.pe.shape[2])), \
            "the reference's positional table differs from synthetic._sinusoid_pe"
        G["cpu_reference"] = dict(wall_s=wall, threads=torch.get_num_threads(), nproc=os.cpu_count(), dtype="fp32",
                                  how="time.perf_counter() around one call of the unmodified reference modules, no warm-up")
        G["surface"] = probe_surface("reference")
    torch.save(G, GOLDEN)
    print(f"audio_front_end: {os.path.getsize(GOLDEN)} bytes in {time.time() - t0:.1f}s; reference CPU wall {wall}")


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count() or 8)
    make_golden()
