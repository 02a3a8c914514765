"""Audio front-end timing on one GPU (the wav2vec2 -> Audio2Mesh / Audio2Pose calls of audio2vid.py:162,189-195).

    python scripts/bench_audio.py --out profiles/audio_front_end_b200.json [--iters 20] [--warmup 5]

Same seeded weights and audio as tests/golden/audio_front_end.pt (tests/audio_golden.py), at 5 s and 10 s of audio:
  kernel       aniportrait_b200 Audio2MeshModel.infer (kernel encoder + heads)
  torch_fp32   the reference path as users get it today: transformers Wav2Vec2Model in fp32 on the same GPU (default TF32
               settings), the reference wrapper's interpolation + heads as torch ops (eager attention, as the golden run)
  pose_chunk   one 150-frame Audio2PoseModel.infer chunk: kernel encoder + KV-cached decoder (CUDA-graph steps)
Median of --iters calls after --warmup, each timed with CUDA events around one call; the rel-L2 between the two encoder
paths; per-kernel device times from a separate torch.profiler run of the kernel path. Writes one JSON file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _time(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return dict(median_ms=statistics.median(ts), min_ms=min(ts), max_ms=max(ts), n=len(ts))


def _gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        vals = [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
        return dict(zip(q.split(","), vals))
    except Exception as exc:  # noqa: BLE001
        return dict(error=repr(exc))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write (e.g. profiles/audio_front_end_b200.json)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_audio.py needs a CUDA device")
    from transformers import Wav2Vec2Config, Wav2Vec2Model as HFWav2Vec2Model
    from aniportrait_b200.audio_models import Audio2MeshModel, kv_cached_infer
    from audio_golden import (AUDIO_ID_SEED, AUDIO_MESH, AUDIO_SEEDS, audio_clip, audio_encoder_config_dir,
                              audio_mesh_state, audio_pose_state, mask_from_last_row)
    from test_audio_frontend_gpu import _PoseModelWithKernelEncoder
    from helpers import rel_l2
    dev = torch.device("cuda:0")
    res = dict(gpu=_gpu_info(), torch=torch.__version__, iters=args.iters, warmup=args.warmup,
               tf32_matmul=torch.backends.cuda.matmul.allow_tf32, tf32_cudnn=torch.backends.cudnn.allow_tf32,
               cases={})
    with tempfile.TemporaryDirectory() as d:
        audio_encoder_config_dir(d)
        mesh = Audio2MeshModel(dict(AUDIO_MESH, model_path=d, from_pretrained=False))
        mesh.load_state_dict(audio_mesh_state(mesh))
        mesh = mesh.to(dev).eval()
        cfg = Wav2Vec2Config.from_pretrained(d)
        cfg._attn_implementation = "eager"
        hf = HFWav2Vec2Model(cfg)
        hf.load_state_dict(mesh.audio_encoder.state_dict())
        hf = hf.to(dev).eval()
        gold = torch.load(os.path.join(ROOT, "tests", "golden", "audio_front_end.pt"), weights_only=False)
        pose = _PoseModelWithKernelEncoder(d, mask_from_last_row(gold["pose_mask_last_row"]))
    pose.load_state_dict(audio_pose_state(pose))
    pose = pose.to(dev).eval()

    def torch_path(audio, T):       # reference model.py:58-69 with wav2vec2.py:29-32 on transformers' modules
        feats = hf.feature_extractor(audio).transpose(1, 2)
        feats = F.interpolate(feats.transpose(1, 2), size=T, align_corners=True, mode="linear").transpose(1, 2)
        h, _ = hf.feature_projection(feats)
        h = hf.encoder(h).last_hidden_state
        return h, mesh.out_fn(mesh.in_fn(h))

    with torch.no_grad():
        for secs in (5, 10):
            T = 30 * secs
            audio = audio_clip(16000 * secs, AUDIO_SEEDS["audio_5s"] + secs).to(dev)
            k_enc = mesh.audio_encoder(audio, T).last_hidden_state
            t_enc, t_out = torch_path(audio, T)
            k_out = mesh.infer(audio, T)
            case = dict(samples=16000 * secs, seq_len=T,
                        kernel=_time(lambda: mesh.infer(audio, T), args.iters, args.warmup),
                        torch_fp32=_time(lambda: torch_path(audio, T), args.iters, args.warmup),
                        rel_l2_encoder_kernel_vs_torch=rel_l2(k_enc, t_enc),
                        rel_l2_mesh_kernel_vs_torch=rel_l2(k_out, t_out))
            case["speedup_torch_over_kernel"] = case["torch_fp32"]["median_ms"] / case["kernel"]["median_ms"]
            res["cases"][f"{secs}s"] = case
            print(f"{secs}s: kernel {case['kernel']['median_ms']:.3f} ms, torch fp32 {case['torch_fp32']['median_ms']:.3f} "
                  f"ms, encoder rel-L2 {case['rel_l2_encoder_kernel_vs_torch']:.2e}", flush=True)
        audio = audio_clip(80000, AUDIO_SEEDS["audio_5s"]).to(dev)
        ids = torch.tensor([AUDIO_ID_SEED], device=dev)
        res["pose_chunk_150"] = _time(lambda: kv_cached_infer(pose, audio, 150, id_seed=ids), max(5, args.iters // 4), 2)
        print(f"pose chunk: {res['pose_chunk_150']['median_ms']:.2f} ms", flush=True)

        from torch.profiler import ProfilerActivity, profile
        audio10 = audio_clip(160000, AUDIO_SEEDS["audio_5s"] + 10).to(dev)
        mesh.infer(audio10, 300)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                mesh.infer(audio10, 300)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", 0) or getattr(e, "self_cuda_time_total", 0)
            if t > 0:
                kern[e.key[:160]] = dict(us_per_call=t / 5.0, launches_per_call=e.count / 5.0)
        res["profile_10s_kernel_path"] = dict(sorted(kern.items(), key=lambda kv: -kv[1]["us_per_call"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
