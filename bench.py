#!/usr/bin/env python
"""Benchmark of the AniPortrait denoising hot path (BASELINE.json metric: denoised frames/sec @512x512, L=16, 25 DDIM
steps, CFG 3.5, fp16).

    python bench.py --gpus N --steps K --warmup W             # product arm (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's math on the host CPU cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/<name>.npy (float32)

One "step" = one complete pass of the hot path over one synthetic 16-frame clip: CLIP embed + VAE encode of the
reference image, ReferenceNet write pass, PoseGuider, 25 CFG DDIM steps of the denoising UNet (reference attention +
temporal motion modules), VAE decode of the 16 frames. Weights are random-init at the real architecture sizes
(SD1.5 UNet + AnimateDiff motion modules 1.31 B params, sd-vae-ft-mse, CLIP ViT-L/14 vision tower); inputs synthetic.
Prints ONE JSON line on rank 0 (see README / DESIGN.md for the field meanings).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "denoised frames/sec @512x512 L=16 steps=25"
W = H = 512
L = 16
DDIM_STEPS = 25
GUIDANCE = 3.5
# algorithmic FLOPs (SURVEY.md §8d / BASELINE.md §2)
FLOP_UNET_CALL = 36.43e12          # one UNet3D call, F=16, CFG
FLOP_VAE_FRAME = 2.515e12
FLOP_RUN = 25 * FLOP_UNET_CALL + 16 * FLOP_VAE_FRAME + 0.80e12 + 16 * 0.119e12 + 0.16e12 + 1.2e12

MOTION_KWARGS = dict(num_attention_heads=8, num_transformer_block=1,
                     attention_block_types=["Temporal_Self", "Temporal_Self"], temporal_position_encoding=True,
                     temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)
SCHED_KWARGS = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                    prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------------------------------------------
# synthetic inputs / weights
# ----------------------------------------------------------------------------------------------------------------
def rand_init_(module, seed):
    """Variance-preserving random init directly on the module's device (full-size weights; no checkpoints offline)."""
    with torch.no_grad():
        g = None
        for name, p in module.named_parameters():
            if g is None:
                g = torch.Generator(device=p.device).manual_seed(seed)
            if p.dim() > 1:
                fan_in = p[0].numel()
                std = min(0.05, fan_in ** -0.5)
                p.copy_(torch.randn(p.shape, generator=g, device=p.device, dtype=torch.float32) * std)
            elif name == "scale":
                p.fill_(2.0)
            elif "norm" in name and name.endswith("weight"):
                p.fill_(1.0)
            elif name.endswith("weight"):   # BatchNorm weights of the PoseGuider
                p.fill_(1.0)
            else:
                p.zero_()


def synthetic_inputs(seed, n_frames=L):
    import numpy as np
    import PIL.Image
    rng = np.random.RandomState(seed)
    ref_image = PIL.Image.fromarray(rng.randint(0, 256, (H, W, 3), dtype=np.uint8))
    poses = []
    for f in range(n_frames):
        r = np.random.RandomState(seed + 2 + f)
        img = np.zeros((H, W, 3), dtype=np.uint8)
        for _ in range(100):
            x0, y0 = r.randint(0, W, 2)
            ln = r.randint(8, 96)
            col = r.randint(64, 256, 3)
            if r.rand() < 0.5:
                img[y0:y0 + 2, x0:min(W, x0 + ln)] = col
            else:
                img[y0:min(H, y0 + ln), x0:x0 + 2] = col
        poses.append(img)
    return ref_image, poses, poses[0]


def build_product_pipeline(device):
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    from aniportrait_b200.models import UNet2DConditionModel, UNet3DConditionModel
    from aniportrait_b200.models.pose_guider import PoseGuider
    from aniportrait_b200.models.vae import AutoencoderKL
    from aniportrait_b200.pipelines import DDIMScheduler, Pose2VideoPipeline
    unet3d = UNet3DConditionModel(sample_size=64, cross_attention_dim=768, attention_head_dim=8,
                                  use_inflated_groupnorm=True, unet_use_cross_frame_attention=False,
                                  unet_use_temporal_attention=False, use_motion_module=True,
                                  motion_module_resolutions=[1, 2, 4, 8], motion_module_mid_block=True,
                                  motion_module_type="Vanilla", motion_module_kwargs=dict(MOTION_KWARGS))
    unet2d = UNet2DConditionModel(sample_size=64, cross_attention_dim=768, attention_head_dim=8)
    pose = PoseGuider(320)
    vae = AutoencoderKL()
    clip = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=1024, intermediate_size=4096,
                                                          num_hidden_layers=24, num_attention_heads=16,
                                                          image_size=224, patch_size=14, projection_dim=768)).eval()
    for i, m in enumerate((unet3d, unet2d, pose, vae, clip)):
        m.to(device=device, dtype=torch.float16)
        rand_init_(m, 100 + i)
    return Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=unet3d,
                              pose_guider=pose, scheduler=DDIMScheduler(**SCHED_KWARGS))


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                       "100", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
                for n, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if sm:
            busy = [v for v in sm if v > 0.5 * max(sm)] or sm
            out["sm_mhz"] = statistics.median(busy)
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


# ----------------------------------------------------------------------------------------------------------------
# product arm
# ----------------------------------------------------------------------------------------------------------------
def kernel_rooflines(device, peaks):
    """Live CUDA-event timing of the two dominant kernels at their hottest shapes (separate launches, after warm-up)."""
    from aniportrait_b200 import ops
    res = {}
    stream = torch.cuda.current_stream()

    def time_it(fn, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    # (1) implicit-GEMM 3x3 conv, 320->320 @64x64, 32 frames (22 % of a UNet call's FLOPs are convs of this family)
    x = torch.randn(32, 64, 64, 320, device=device, dtype=torch.float16)
    b = torch.zeros(320, device=device, dtype=torch.float32)
    out = torch.empty(32, 64, 64, 320, device=device, dtype=torch.float16)
    w_raw = torch.randn(320, 320, 3, 3, device=device, dtype=torch.float16) * 0.02
    wt = ops.pack_conv3x3_weight(w_raw)
    ms = time_it(lambda: ops.conv3x3(x, wt, 320, bias=b, out=out))
    # the values of the timed launch against a real-fp32 (TF32 off) torch evaluation of the same fp16 inputs
    parity = {}
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    def rel(a, r):
        return float((a.float() - r).norm() / r.norm())
    ref = torch.nn.functional.conv2d(x[:8].permute(0, 3, 1, 2).float(), w_raw.float(), padding=1).permute(0, 2, 3, 1)
    parity["conv3x3_320_64x64"] = rel(out[:8], ref)
    del ref
    fl = 2.0 * 32 * 64 * 64 * 320 * 9 * 320
    res["conv3x3"] = dict(kernel="gemm_kernel<BN=160,LINEAR,cta_group::2,NACC=2> (implicit-GEMM conv3x3 320->320 @64x64x32f, 256x320 tiles)", ms=ms,
                          tflops=fl / ms / 1e9)
    # (2) fused reference attention, 64x64 level: 32 frames (16 uncond: N keys, 16 cond: 2N keys), 8 heads, d=40
    n, heads, d, dpad, fr = 4096, 8, 40, 64, 32
    hp = heads * dpad
    qkv = torch.randn(fr * n, 3 * hp, device=device, dtype=torch.float16)
    bank = torch.randn(n, 2 * hp, device=device, dtype=torch.float16)
    # the head padding d..dpad is ZERO in real use (zero rows of the packed projection weights); the kernel multiplies the
    # first 48 of the 64 columns
    qkv.view(fr * n, 3 * heads, dpad)[:, :, d:] = 0
    bank.view(n, 2 * heads, dpad)[:, :, d:] = 0
    o = torch.empty(fr * n, heads * d, device=device, dtype=torch.float16)
    ms = time_it(lambda: ops.attention(qkv[:, :hp], qkv[:, hp:2 * hp], qkv[:, 2 * hp:], fr, n, heads, d, dpad,
                                       bank_k=bank[:, :hp], bank_v=bank[:, hp:], bank_tokens=n, n_banks=1,
                                       first_bank_frame=16, frames_per_bank=16, out=o), iters=5)
    # parity: one unconditional frame (N keys) and one conditional frame (own N keys + the bank's N), fp32 SDPA
    def ref_attn(fi, with_bank):
        def heads_of(t):   # [n, heads*dpad] -> [heads, n, d]
            return t.view(-1, heads, dpad)[:, :, :d].permute(1, 0, 2).float()
        rows = slice(fi * n, (fi + 1) * n)
        q_, k_, v_ = heads_of(qkv[rows, :hp]), heads_of(qkv[rows, hp:2 * hp]), heads_of(qkv[rows, 2 * hp:])
        if with_bank:
            k_ = torch.cat([k_, heads_of(bank[:, :hp])], 1)
            v_ = torch.cat([v_, heads_of(bank[:, hp:])], 1)
        r = torch.nn.functional.scaled_dot_product_attention(q_[None], k_[None], v_[None])[0]
        return r.permute(1, 0, 2).reshape(n, heads * d)
    parity["ref_attention_uncond_frame"] = rel(o[:n], ref_attn(0, False))
    parity["ref_attention_cond_frame"] = rel(o[31 * n:], ref_attn(31, True))
    fl = 4.0 * n * d * heads * (16 * 2 * n + 16 * n)
    res["ref_attention"] = dict(kernel="attention5_kernel (ref-attn 64x64 level, d=40 padded to 64, 16 cond + 16 uncond frames)",
                                ms=ms, tflops=fl / ms / 1e9)
    # (3) temporal (frame-axis) attention of the motion modules at the 64x64 level: HBM-bound, 8*C bytes per token
    B_, F_, N_, C_ = 2, 16, 4096, 320
    tq = torch.randn(B_ * F_ * N_, 3 * C_, device=device, dtype=torch.float16)
    to = torch.empty(B_ * F_ * N_, C_, device=device, dtype=torch.float16)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)     # > L2: every timed launch reads from HBM
    for _ in range(2):
        ops.temporal_attention(tq, B_, F_, N_, C_, 8, out=to)
    tms = 0.0
    for _ in range(5):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ops.temporal_attention(tq, B_, F_, N_, C_, 8, out=to)
        e1.record(stream)
        torch.cuda.synchronize()
        tms += e0.elapsed_time(e1) / 5
    # parity of the temporal core: softmax over the 16 frames of each (batch, position, head), first 256 positions
    dh = C_ // 8
    t5 = tq.view(B_, F_, N_, 3, 8, dh)[:, :, :256].float()                   # [B, F, n, 3, heads, d]
    tq_, tk_, tv_ = (t5[:, :, :, i].permute(0, 2, 3, 1, 4) for i in range(3))     # [B, n, heads, F, d]
    tref = torch.nn.functional.scaled_dot_product_attention(tq_, tk_, tv_)        # [B, n, heads, F, d]
    tref = tref.permute(0, 3, 1, 2, 4).reshape(B_, F_, 256, C_)
    parity["temporal_attention"] = rel(to.view(B_, F_, N_, C_)[:, :, :256], tref)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    res["parity"] = {k: float(f"{v:.3e}") for k, v in parity.items()}
    nbytes = (tq.numel() + to.numel()) * 2
    # (4) one full UNet3D call is timed by the caller (aggregate)
    for k_, v in res.items():
        if k_ != "parity":
            v["frac_of_peak"] = v["tflops"] / peaks["tflops_burst"]
    res["temporal_attention"] = dict(kernel="temporal_attn_mma_kernel<40> (motion-module attention, 2x16 frames x 4096 positions x 320 ch)",
                                     ms=tms, gbs=nbytes / tms / 1e6, frac_of_peak=nbytes / tms / 1e6 / peaks["hbm"])
    return res


def run_strong_c4(pipe, device, rank, world, local_rank, base_on_rank0=True):
    """BASELINE.json configs[3] (SURVEY.md 8d C4): ONE 128-frame video, 11 overlapping 16-frame windows x 25 DDIM steps, the
    22 (window, CFG-branch) units sharded over the ranks (dist_mode="window_branches": every rank replays the CUDA graphs of
    its units, one fp32 all-reduce of the prediction accumulator per step, ONE NCCL broadcast of the flat ReferenceNet bank
    buffer per video, VAE decode sharded by frame + all-gather). Strong scaling: total work fixed as N grows.
    Timed on the device (events), max over ranks. At N > 1 rank 0 afterwards runs the SAME video alone (the other ranks wait
    at the barrier), so the line carries a same-box, same-build speed-up."""
    from aniportrait_b200.pipelines.sharding import plan_units
    LC = 128
    ref_image, poses, _ = synthetic_inputs(2000, LC)
    clip_pixels = pipe.clip_image_processor.preprocess(ref_image.resize((224, 224)), return_tensors="pt").pixel_values
    clip_pixels = clip_pixels.to(device, torch.float16)
    ref_t = pipe.ref_image_processor.preprocess(ref_image, height=H, width=W).to(device, torch.float16)
    pose_t = pipe._pose_maps_to_tensor(poses, H, W, device).to(torch.float16)
    lat0 = torch.randn((1, 4, LC, H // 8, W // 8), generator=torch.Generator().manual_seed(4242),
                       dtype=torch.float16).to(device)
    mode = "window_branches" if world > 1 else None

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(dist_mode, reps):
        pipe.run_device(clip_pixels, ref_t, pose_t, lat0, DDIM_STEPS, GUIDANCE, dist_mode=dist_mode)   # builds + captures
        torch.cuda.synchronize()
        best, ph = None, None
        for _ in range(reps):
            if dist_mode is not None:
                barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pipe.run_device(clip_pixels, ref_t, pose_t, lat0, DDIM_STEPS, GUIDANCE, dist_mode=dist_mode)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if best is None or ms < best:
                best, ph = ms, dict(pipe.collect_timings())
        return best, ph, pipe.last_latents.float().cpu()

    barrier()
    ms, ph, lat_sharded = timed(mode, 2 if world > 1 else 1)
    # per-rank split: device ms inside the unit graphs = denoise - all-reduce (which includes waiting for slower ranks)
    mine = torch.tensor([ms, ph["denoise_ms"], ph.get("all_reduce_ms", 0.0), ph.get("bank_broadcast_ms", 0.0),
                         ph.get("all_gather_ms", 0.0), ph["reference_ms"], ph["decode_ms"], float(ph["units_this_rank"])],
                        device=device, dtype=torch.float64)
    allr = [torch.zeros_like(mine) for _ in range(world)]
    if world > 1:
        torch.distributed.all_gather(allr, mine)
    else:
        allr = [mine]
    rows = torch.stack(allr).cpu()
    base_ms, base_err = None, None
    if world > 1 and base_on_rank0:
        if rank == 0:
            base_ms, _, lat_single = timed(None, 1)
            base_err = float((lat_sharded - lat_single).norm() / lat_single.norm())
        barrier()
    if rank != 0:
        return None
    total_ms = float(rows[:, 0].max())
    compute = (rows[:, 1] - rows[:, 2]).tolist()
    plan = plan_units(11, True, world) if world > 1 else [[(k, "both") for k in range(11)]]
    cost = [sum({"both": 2.2, "cond": 1.2, "uncond": 1.0}[b] for _, b in r) for r in plan]
    out = {"workload": "pose2vid_long 512x512, ONE video of 128 frames = 11 overlapping 16-frame windows, 25 DDIM steps, CFG "
                       "3.5 (BASELINE.json configs[3]); 22 (window, CFG branch) units sharded over the ranks, "
                       "NCCL bank broadcast + per-step fp32 all-reduce + frame-sharded VAE decode",
           "scaling": "strong", "n_gpus": world, "frames": LC, "ms": round(total_ms, 2),
           "frames_per_s": round(LC / (total_ms / 1e3), 3),
           "dist_mode": mode or "single GPU (11 window graphs, both branches per call)",
           "units_per_rank": [int(v) for v in rows[:, 7].tolist()],
           "ideal_speedup_from_unit_costs": round(11 * 2.2 / max(cost), 3),
           "per_rank_ms": {"unit_graphs_compute": [round(v, 1) for v in compute],
                           "all_reduce_incl_wait": [round(v, 1) for v in rows[:, 2].tolist()],
                           "bank_broadcast": [round(v, 2) for v in rows[:, 3].tolist()],
                           "decode_all_gather": [round(v, 2) for v in rows[:, 4].tolist()],
                           "prologue": [round(v, 1) for v in rows[:, 5].tolist()],
                           "decode": [round(v, 1) for v in rows[:, 6].tolist()]}}
    if world > 1:
        cmax, cmean = max(compute), sum(compute) / len(compute)
        comm = float(rows[:, 2].min())     # the slowest rank never waits: its all-reduce time is (almost) pure NCCL time
        out["imbalance_ms"] = round(cmax - cmean, 1)
        out["nccl_all_reduce_ms_on_slowest_rank"] = round(comm, 1)
        out["limiter"] = ("unit imbalance" if (cmax - cmean) > comm else "NCCL all-reduce latency") + \
            f" (max-mean unit compute {cmax - cmean:.0f} ms vs {comm:.0f} ms in 25 all-reduces on the busiest rank)"
        if base_ms is not None:
            out["single_gpu_same_box_ms"] = round(base_ms, 2)
            out["speedup_vs_single_gpu"] = round(base_ms / total_ms, 3)
            out["rel_l2_vs_single_gpu_latents"] = float(f"{base_err:.3e}")
    return out


def run_c1(pipe, device):
    """BASELINE.json configs[0] (C1: 512x512, L=4, 10 DDIM steps, CFG 3.5) through the public API with host inputs: the
    like-for-like partner of the CPU arm's C1 figure."""
    ref_image, poses, ref_pose = synthetic_inputs(3000, 4)
    gen = torch.Generator().manual_seed(7)
    for _ in range(2):
        pipe(ref_image, poses, ref_pose, W, H, 4, 10, GUIDANCE, generator=gen)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        pipe(ref_image, poses, ref_pose, W, H, 4, 10, GUIDANCE, generator=gen)
    torch.cuda.synchronize()
    s_run = (time.perf_counter() - t0) / reps
    return {"workload": "pose2vid 512x512, L=4, 10 DDIM steps, CFG 3.5 (BASELINE.json configs[0]), end to end through "
                        "Pose2VideoPipeline.__call__ (host images in, fp32 host video out)",
            "seconds_per_run": round(s_run, 4), "frames_per_s": round(4 / s_run, 3)}


def run_product(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N>1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py product arm needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from aniportrait_b200 import _lib, ops
    _lib.init(local_rank)
    peaks = load_peaks()
    pipe = build_product_pipeline(device)

    # every rank animates its own 16-frame window of the SAME reference portrait (weak scaling; banks broadcast once)
    ref_image, poses, ref_pose = synthetic_inputs(1000, L)
    if world > 1:
        _, poses, _ = synthetic_inputs(1000 + 17 * rank, L)
    dist_mode = "clips" if world > 1 else None
    gen = torch.Generator().manual_seed(42 + rank)
    # device-resident inputs for the kernel-side number
    clip_pixels = pipe.clip_image_processor.preprocess(ref_image.resize((224, 224)), return_tensors="pt").pixel_values
    clip_pixels = clip_pixels.to(device, torch.float16)
    ref_t = pipe.ref_image_processor.preprocess(ref_image, height=H, width=W).to(device, torch.float16)
    pose_t = torch.cat([pipe.cond_image_processor.preprocess(p, height=H, width=W) for p in poses], 0)
    pose_t = pose_t.to(device, torch.float16)
    lat0 = torch.randn((1, 4, L, H // 8, W // 8), generator=gen, dtype=torch.float16).to(device)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def device_step():
        return pipe.run_device(clip_pixels, ref_t, pose_t, lat0, DDIM_STEPS, GUIDANCE, dist_mode=dist_mode)

    def e2e_step():
        return pipe(ref_image, poses, ref_pose, W, H, L, DDIM_STEPS, GUIDANCE, generator=gen, dist_mode=dist_mode)

    # dominant kernels timed alone (own launches, CUDA events on the launch stream) before the long run heats the part:
    # the burst peak is their denominator; the whole-UNet-call figure below uses the sustained peak
    roofs = kernel_rooflines(device, peaks) if rank == 0 else None
    torch.cuda.empty_cache()
    for _ in range(args.warmup):
        device_step()
    barrier()
    # ---- timed region 1: device-resident inputs -------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = ops.KERNEL_LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        video = device_step()
    e1.record()
    barrier()
    ms_step = e0.elapsed_time(e1) / args.steps
    # what the caller of the timed path receives from its last step: the decoded video and the final latents
    outputs = {"video": video.float().cpu(), "latents": pipe.last_latents.float().cpu()} if args.dump_outputs else None
    launches = (ops.KERNEL_LAUNCHES - n0)
    phases = pipe.collect_timings()
    clocks = sampler.stop() if rank == 0 else {}
    # ---- timed region 2: end to end through the public API with host inputs -------------------------------
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    tt = torch.tensor([ms_step, e2e_ms], device=device, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
    ms_step, e2e_ms = tt.tolist()
    # ---- extra leg: the same call returning packed 8-bit frames (output_type="uint8": 1 byte per sample to the host) ----
    e2e_u8 = None
    if world == 1:
        try:
            def u8_step():
                return pipe(ref_image, poses, ref_pose, W, H, L, DDIM_STEPS, GUIDANCE, generator=gen, output_type="uint8")
            u8_step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                u8_step()
            torch.cuda.synchronize()
            u8_ms = (time.perf_counter() - t0) * 1e3 / args.steps
            e2e_u8 = {"value": round(L / (u8_ms / 1e3), 4), "unit": "frames/s", "ms_per_step": round(u8_ms, 3),
                      "d2h_bytes_per_step": int(3 * L * H * W),
                      "note": "same call as `e2e`, frames returned as packed uint8 RGB [1, L, H, W, 3] (what the scripts' "
                              "save_videos_grid derives on the host); host inputs as in `e2e`"}
        except Exception as exc:       # an extra: never let it take the headline line down
            e2e_u8 = {"error": repr(exc)}
    # ---- extra legs (not part of `value`): C1 like-for-like (rank 0, N=1) and the strong-scaling C4 video (every N) ----
    c1 = run_c1(pipe, device) if (world == 1 and args.c1) else None
    strong_c4 = None
    if args.c4:
        pipe.clear_graph_cache()
        torch.cuda.empty_cache()
        strong_c4 = run_strong_c4(pipe, device, rank, world, local_rank)

    if rank == 0:
        value = world * L / (ms_step / 1e3)
        e2e_value = world * L / (e2e_ms / 1e3)
        h2d = int(len(poses) * H * W * 3 + 3 * 224 * 224 * 4 + 3 * H * W * 4 + 4 * L * (H // 8) * (W // 8) * 2)
        d2h = int(3 * L * H * W * 4)      # fp32 video, converted on the device, one pinned-buffer copy
        unet_ms = phases["denoise_ms"] / DDIM_STEPS
        unet_tflops = FLOP_UNET_CALL / unet_ms / 1e9
        line = {
            "metric": METRIC, "value": round(value, 4), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": "pose2vid 512x512, L=16, 25 DDIM steps, CFG 3.5, fp16, ReferenceNet bank active "
                                   "(BASELINE.json configs[1]); one 16-frame clip per GPU",
                       "weights": "random-init, real architecture sizes (UNet3D 1.31B params, sd-vae-ft-mse, CLIP ViT-L/14)",
                       "l2": "inputs larger than L2: 2.6 GB of weights + ~9 GB of activations stream per UNet call",
                       "parallelism": f"dp{world} (one independent 16-frame clip per rank, no data-path collective)"
                       if world > 1 else "single GPU"},
            "e2e": {"value": round(e2e_value, 4), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_ms, 3)},
            "gpu_launches": launches,
            "phases_ms": {k: round(v, 3) for k, v in phases.items() if k.endswith("_ms")},
            "roofline": {"bound": "tensor", "achieved": round(roofs["conv3x3"]["tflops"], 2), "peak": peaks["tflops_burst"],
                         "unit": "TFLOP/s", "frac": round(roofs["conv3x3"]["frac_of_peak"], 4),
                         # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel at this shape: a PROFILE
                         # CONSTANT from the `ncu --set full` capture (not measured in this run)
                         "traffic": 129.8e6, "traffic_unit": "bytes/launch (algorithmic 169.7e6: 84 in + 1.8 w + 84 out)",
                         "traffic_source": "profile constant: profiles/r01_ncu_full_top_kernels.md (ncu --set full, round 1)",
                         "kernel": roofs["conv3x3"]["kernel"], "launch_ms": round(roofs["conv3x3"]["ms"], 4),
                         "peak_source": peaks["source"] + " burst (kernel timed alone)"},
            "roofline_ref_attention": {"bound": "tensor", "achieved": round(roofs["ref_attention"]["tflops"], 2),
                                       "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
                                       "frac": round(roofs["ref_attention"]["frac_of_peak"], 4),
                                       "kernel": roofs["ref_attention"]["kernel"],
                                       "launch_ms": round(roofs["ref_attention"]["ms"], 4),
                                       "note": "algorithmic FLOPs (d=40 unpadded; uncond frames N keys, cond frames 2N)"},
            "roofline_temporal_attention": {"bound": "hbm", "achieved": round(roofs["temporal_attention"]["gbs"], 1),
                                            "peak": peaks["hbm"], "unit": "GB/s",
                                            "frac": round(roofs["temporal_attention"]["frac_of_peak"], 4),
                                            "kernel": roofs["temporal_attention"]["kernel"],
                                            "launch_ms": round(roofs["temporal_attention"]["ms"], 4),
                                            "note": "algorithmic bytes: q,k,v read + out written once (335.5 MB); L2 flushed "
                                                    "before every timed launch"},
            "roofline_unet_call": {"bound": "tensor", "achieved": round(unet_tflops, 2), "peak": peaks["tflops_sustained"],
                                   "unit": "TFLOP/s", "frac": round(unet_tflops / peaks["tflops_sustained"], 4),
                                   "ms": round(unet_ms, 3), "flop": FLOP_UNET_CALL,
                                   "note": "whole UNet3D call (all kernels), algorithmic 36.43 TFLOP, sustained peak"},
            "clocks": clocks,
            "parity_at_bench_shape": dict(roofs["parity"], tolerance=1e-2,
                                          how="rel-L2 of the roofline-timed launches' outputs vs a real-fp32 (TF32 off) torch "
                                              "evaluation of the same fp16 inputs on the device"),
        }
        if e2e_u8 is not None:
            line["e2e_uint8_frames"] = e2e_u8
        if c1 is not None:
            line["c1"] = c1
        if strong_c4 is not None:
            line["strong_c4"] = strong_c4
        if args.cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_sample(args.cpu_threads)
        print(json.dumps(line))
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        torch.distributed.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, outputs):
    """Writes each output as <directory>/<name>.npy in float32, so that two builds can be compared output for output on
    the same (seeded, run-to-run identical) inputs."""
    import numpy as np
    total = sum(t.numel() * 4 for t in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"outputs take {total} bytes, more than the {DUMP_LIMIT_BYTES} bytes --dump-outputs writes")
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), t.numpy().astype(np.float32))


# ----------------------------------------------------------------------------------------------------------------
# CPU baseline (the reference's math restated in oracle/functional.py, fp32, host cores)
# ----------------------------------------------------------------------------------------------------------------
def cpu_baseline_sample(threads=None):
    """The reference's math (oracle/functional.py: fp32 torch CPU restatement, pinned to the unmodified reference wiring by
    tests/test_oracle_vs_reference.py) at the REAL geometry and width on the host cores: BASELINE.json configs[0] (C1:
    512x512, L=4, CFG 3.5) — the ReferenceNet pass, ONE complete DDIM step exactly as the reference executes it (in-loop
    PoseGuider on the CFG-duplicated batch + UNet3D with reference attention over the 4-frame window) and the VAE decode
    of ONE frame are each run and timed in full; nothing is scaled in pixels. Steps and frames are repetitions of identical
    work, so   C1 = t_ref + 10 t_step + 4 t_dec   and   C2 (the headline config: L=16, 25 steps) = t_ref + 25 (4 t_step) +
    16 t_dec   (per-frame cost of a UNet call is frame-count independent except for the 0.1 % temporal core).
    CLIP and the VAE encode of the reference image (< 1 % of a run) are not included.
    The un-extrapolated wall time of the UNMODIFIED reference pipeline on C1 (recorded once in the authoring container when the
    golden fixture was generated, 8 cores) is attached from tests/golden/pipeline_c1_full.pt when present."""
    from aniportrait_b200.synthetic import meta_state_dict, randomize_state_dict
    from aniportrait_b200.models import UNet2DConditionModel, UNet3DConditionModel
    from aniportrait_b200.models.pose_guider import PoseGuider
    from aniportrait_b200.models.vae import AutoencoderKL
    from oracle import functional as OF
    threads = threads or min(os.cpu_count() or 1, 32)   # torch CPU conv/GEMM stops scaling (and oversubscribes) beyond ~32
    torch.set_num_threads(threads)
    OF.USE_SDPA = True      # time the library attention the reference itself calls (AttnProcessor2_0 -> SDPA), see oracle
    t_build = time.perf_counter()
    sd3 = randomize_state_dict(meta_state_dict(lambda: UNet3DConditionModel(
        cross_attention_dim=768, use_inflated_groupnorm=True, unet_use_cross_frame_attention=False,
        unet_use_temporal_attention=False, use_motion_module=True, motion_module_mid_block=True,
        motion_module_type="Vanilla", motion_module_kwargs=dict(MOTION_KWARGS))), seed=1)
    sd2 = randomize_state_dict(meta_state_dict(lambda: UNet2DConditionModel(cross_attention_dim=768)), seed=2)
    sdp = randomize_state_dict(meta_state_dict(lambda: PoseGuider(320)), seed=3)
    sdv = {k: v for k, v in randomize_state_dict(meta_state_dict(lambda: AutoencoderKL()), seed=4).items()
           if k.startswith(("decoder.", "post_quant_conv."))}
    t_build = time.perf_counter() - t_build
    g = torch.Generator().manual_seed(4)
    frames, latent = 4, 64
    lat = torch.randn(1, 4, frames, latent, latent, generator=g)
    clip = torch.randn(1, 768, generator=g)
    ehs = torch.cat([torch.zeros_like(clip), clip]).unsqueeze(1)
    pose_in = torch.randn(1, 3, frames, latent * 8, latent * 8, generator=g)
    with torch.no_grad():
        t0 = time.perf_counter()
        banks = OF.reference_unet_banks(sd2, torch.randn(1, 4, latent, latent, generator=g).repeat(2, 1, 1, 1), ehs)
        t_ref = time.perf_counter() - t0
        t0 = time.perf_counter()
        pf = OF.pose_guider_forward(sdp, pose_in.repeat(2, 1, 1, 1, 1))
        t_pose = time.perf_counter() - t0
        OF.unet3d_forward(sd3, lat.repeat(2, 1, 1, 1, 1), 500, ehs, pf, banks, cfg=True)
        t_step = time.perf_counter() - t0
        t0 = time.perf_counter()
        OF.vae_decode(sdv, lat[:, :, 0] / 0.18215)
        t_dec = time.perf_counter() - t0
    c1_s = t_ref + 10 * t_step + 4 * t_dec
    c2_s = t_ref + 25 * 4 * t_step + 16 * t_dec
    out = {"value": round(L / c2_s, 6), "unit": "frames/s", "cores": threads, "kind": "port",
           "sample": f"oracle/functional.py at full width, 512x512, 4-frame window, CFG: ReferenceNet pass {t_ref:.1f}s, one DDIM step "
                     f"(in-loop PoseGuider {t_pose:.1f}s + UNet3D) {t_step:.1f}s, VAE decode of one frame {t_dec:.1f}s, each run "
                     f"in full; `value` = 16 / (t_ref + 100 t_step + 16 t_dec) = 16 / {c2_s:.0f}s for the headline config (L=16, 25 "
                     f"steps); weight init {t_build:.0f}s not counted",
           "seconds": {"reference_unet": round(t_ref, 2), "ddim_step_L4": round(t_step, 2), "pose_guider_in_step": round(t_pose, 2),
                       "vae_decode_frame": round(t_dec, 2)},
           "c1": {"workload": "BASELINE.json configs[0]: 512x512, L=4, 10 DDIM steps, CFG 3.5",
                  "seconds_per_run": round(c1_s, 1), "frames_per_s": round(4 / c1_s, 6),
                  "formula": "t_ref + 10 t_step + 4 t_dec (every term measured in full on this box)"}}
    fixture = os.path.join(ROOT, "tests", "golden", "pipeline_c1_full.pt")
    if os.path.exists(fixture):
        try:
            rec = torch.load(fixture)["cpu_reference"]
            out["recorded_reference_c1"] = {
                "kind": "reference-via-shim (UNMODIFIED /root/reference/src pipeline over oracle/diffusers_shim, fp32)",
                "where": "authoring container, recorded by oracle/make_golden.py pipeline_c1_full when the golden was made",
                "wall_s": round(rec["wall_s"], 1), "frames_per_s": round(rec["frames_per_s"], 6), "threads": rec["threads"],
                "nproc": rec["nproc"], "phase_seconds": {k: round(v, 1) for k, v in rec["phase_seconds"].items()}}
        except Exception as e:   # a fixture from an older generator
            out["recorded_reference_c1"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path. The reference is pure PyTorch + diffusers;
    diffusers is not installable offline and /root/reference does not travel to the GPU box, so the arm times
    oracle/functional.py (the restatement pinned against the unmodified reference wiring) on the host cores, at the real
    geometry (see cpu_baseline_sample). Rank 0 only; one sample per `step` (a sample is minutes of CPU time)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = args.cpu_threads or min(os.cpu_count() or 1, 32)
    vals = [cpu_baseline_sample(threads) for _ in range(args.steps)]
    best = max(vals, key=lambda d: d["value"])
    v = best["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(L / v * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": "pose2vid 512x512, L=16, 25 DDIM steps, CFG 3.5 (BASELINE.json configs[1]) on the host CPU: "
                                   "every distinct piece of work timed in full at 512x512, repeated steps / frames multiplied "
                                   "(see cpu_baseline.sample)"},
            "cpu_baseline": best,
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-c4", dest="c4", action="store_false", help="skip the 128-frame strong-scaling leg")
    ap.add_argument("--no-c1", dest="c1", action="store_false", help="skip the C1 (L=4, 10 steps) like-for-like leg")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's video and latents as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the product arm's outputs; the reference arm returns timings only")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.gpus > 1:
            args.cpu_baseline = args.cpu_baseline and int(os.environ.get("RANK", "0")) == 0
        run_product(args)


if __name__ == "__main__":
    main()
