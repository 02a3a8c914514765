"""Pose2VideoPipeline — mirror of the reference's src/pipelines/pipeline_pose2vid_long.py (the pipeline every script
uses: scripts/pose2vid.py:166-176, audio2vid.py:230-240, vid2vid.py:213-223).

Same constructor and `__call__` signature and the same result object (`.videos`: fp32 CPU tensor [1, 3, F, H, W] in
[0, 1]). The denoising loop is re-designed for B200 while producing the reference's numbers:
  * latents live in one channels-last fp16 buffer [L, h, w, 4]; per window a gather kernel builds the CFG-duplicated UNet
    input, a scatter kernel accumulates the prediction into an fp32 [2, L, h, w, 4] buffer, and ONE kernel per step does
    overlap averaging + classifier-free guidance + the DDIM v-prediction update (reference :521-559);
  * PoseGuider does not depend on the timestep: it is evaluated once per window (the reference re-runs it on a
    CFG-duplicated batch every step, :531-536) — identical values, 25x less work;
  * ReferenceNet runs once; each reader block projects its bank to K/V once per video;
  * VAE decode is batched over frames (reference: one frame per call, :118-121).
  * all of the above is captured into CUDA graphs once per video geometry and replayed for every later video.
With torch.distributed initialised, dist_mode="windows" shards the frame windows of one video across ranks: rank 0 runs
the ReferenceNet once and broadcasts the 16 banks over NCCL, and the fp32 prediction accumulator is all-reduced once per
step (SURVEY.md §8e); dist_mode="clips" gives every rank its own clip with no data-path collective at all.
"""
from __future__ import annotations

import time
from dataclasses import dataclass
from typing import Callable, List, Optional, Union

import numpy as np
import torch

from .. import ops
from ..models.mutual_self_attention import ReferenceAttentionControl
from .sharding import plan_units, plan_windows, windows_of_rank
from .image_processor import VaeImageProcessor


class _Session:
    """Tensors one video's stages communicate through (inputs, latents, accumulator, banks' owners, pose features) and, for
    static sessions, the CUDA graphs captured over them."""


def _assign(dst, src):
    """First pass: keep the tensor; later passes (incl. graph capture): write into the same storage."""
    if dst is None:
        return src.contiguous().clone()
    dst.copy_(src)
    return dst


@dataclass
class Pose2VideoPipelineOutput:
    videos: Union[torch.Tensor, np.ndarray]


class Pose2VideoPipeline:
    _optional_components = []
    _video_counter = 0

    def __init__(self, vae, image_encoder, reference_unet, denoising_unet, pose_guider, scheduler,
                 image_proj_model=None, tokenizer=None, text_encoder=None):
        self.vae = vae
        self.image_encoder = image_encoder
        self.reference_unet = reference_unet
        self.denoising_unet = denoising_unet
        self.pose_guider = pose_guider
        self.scheduler = scheduler
        self.image_proj_model = image_proj_model
        self.tokenizer = tokenizer
        self.text_encoder = text_encoder
        self.vae_scale_factor = 2 ** (len(self.vae.config.block_out_channels) - 1)
        from transformers import CLIPImageProcessor
        self.clip_image_processor = CLIPImageProcessor()
        self.ref_image_processor = VaeImageProcessor(vae_scale_factor=self.vae_scale_factor, do_convert_rgb=True)
        self.cond_image_processor = VaeImageProcessor(vae_scale_factor=self.vae_scale_factor, do_convert_rgb=True,
                                                      do_normalize=True)
        self.timings = {}
        self.use_cuda_graph = True        # capture every stage of a video geometry once (a _Session), replay afterwards
        self.capture_library_stage = True  # also capture CLIP + VAE-encode (falls back to eager if not capturable)
        self.max_sessions = 2
        # sharded modes: a rank's (window, branch) units are batched into UNet calls of up to `group_units` elements
        # (unconditional windows first), instead of one batch-1 / batch-2 call per unit: larger GEMMs, fewer
        # wave-quantisation losses. 0 = one call per unit.
        self.group_units = 4
        self._sessions = {}
        self._side_stream = None

    # -------------------------------------------------------------------------------------------- plumbing
    def _nn_modules(self):
        return [m for m in (self.vae, self.image_encoder, self.reference_unet, self.denoising_unet, self.pose_guider)
                if isinstance(m, torch.nn.Module)]

    def to(self, *args, **kwargs):
        for m in self._nn_modules():
            m.to(*args, **kwargs)
        return self

    @property
    def device(self):
        for m in self._nn_modules():
            for p in m.parameters():
                return p.device
        return torch.device("cpu")

    _execution_device = device

    def progress_bar(self, iterable=None, total=None):
        from tqdm.auto import tqdm
        cfg = getattr(self, "_progress_bar_config", {"disable": True})
        return tqdm(iterable, **cfg) if iterable is not None else tqdm(total=total, **cfg)

    def set_progress_bar_config(self, **kwargs):
        self._progress_bar_config = kwargs

    def enable_vae_slicing(self):
        """Reference surface (pipeline_pose2vid_long.py:82-86). Slicing trades speed for activation memory in diffusers' VAE;
        decode_latents_device() already bounds the decoder's activations by decoding `frame_batch` frames per call, so the
        switch only selects that bound: enabled = one frame per call (the reference's sliced behaviour)."""
        self.vae_frame_batch = 1

    def disable_vae_slicing(self):
        self.vae_frame_batch = 8

    # -------------------------------------------------------------------------------------------- stages
    def prepare_latents(self, batch_size, num_channels_latents, width, height, video_length, dtype, device, generator,
                        latents=None):
        shape = (batch_size, num_channels_latents, video_length, height // self.vae_scale_factor,
                 width // self.vae_scale_factor)
        if latents is None:
            rand_device = device
            if generator is not None and generator.device.type == "cpu" and torch.device(device).type != "cpu":
                rand_device = "cpu"   # diffusers randn_tensor: sample where the generator lives, then move
            latents = torch.randn(shape, generator=generator, device=rand_device, dtype=dtype).to(device)
        else:
            latents = latents.to(device)
        return latents * self.scheduler.init_noise_sigma

    @torch.no_grad()
    def decode_latents_device(self, latents: torch.Tensor, frame_batch: int = None):
        """latents [1, 4, F, h, w] -> device tensor [1, 3, F, H, W] in [0, 1] (reference :113-123, batched)."""
        video_length = latents.shape[2]
        frame_batch = frame_batch or getattr(self, "vae_frame_batch", 8)
        z = (1 / 0.18215 * latents).permute(0, 2, 1, 3, 4).reshape(-1, *latents.shape[1:2], *latents.shape[3:])
        frames = []
        for i in range(0, z.shape[0], frame_batch):
            frames.append(self.vae.decode(z[i:i + frame_batch].to(self.vae.dtype)).sample)
        video = torch.cat(frames)
        video = video.view(-1, video_length, *video.shape[1:]).permute(0, 2, 1, 3, 4)
        return (video / 2 + 0.5).clamp(0, 1)

    def _to_host_f32(self, video: torch.Tensor) -> torch.Tensor:
        """Device fp16 video -> fp32 CPU tensor through a cached pinned staging buffer. The returned tensor is a fresh copy
        (the reference hands out a tensor the caller owns), the staging buffer is reused by the next call."""
        dev32 = video.float()
        pin = getattr(self, "_pinned_out", None)
        if pin is None or pin.shape != dev32.shape:
            pin = torch.empty(dev32.shape, dtype=torch.float32, pin_memory=True)
            self._pinned_out = pin
        pin.copy_(dev32, non_blocking=True)
        torch.cuda.current_stream(video.device).synchronize()
        return pin.clone()

    def _to_host_u8(self, video: torch.Tensor) -> torch.Tensor:
        """Device fp16 video [B, 3, F, H, W] -> uint8 CPU frames [B, F, H, W, 3]: the bytes the scripts' `save_videos_grid`
        (reference src/utils/util.py:87-104) derives from the fp32 host tensor, packed on the device -> a quarter of the
        fp32 copy's bytes over PCIe (12.6 MB instead of 50.3 MB per 16 frames at 512x512)."""
        dev8 = ops.pack_frames_u8(video)
        pin = getattr(self, "_pinned_out_u8", None)
        if pin is None or pin.shape != dev8.shape:
            pin = torch.empty(dev8.shape, dtype=torch.uint8, pin_memory=True)
            self._pinned_out_u8 = pin
        pin.copy_(dev8, non_blocking=True)
        torch.cuda.current_stream(video.device).synchronize()
        return pin.clone()

    def decode_latents(self, latents: torch.Tensor):
        """Reference-compatible: numpy fp32 on the host (reference :113-126)."""
        return self.decode_latents_device(latents).cpu().float().numpy()

    def _pose_maps_to_tensor(self, pose_images, height, width, device):
        """cond_image_processor.preprocess for the pose maps. uint8 HxWx3 arrays of the target size (what the scripts
        pass, pose2vid.py:153-158) take a fast path: the bytes go to the GPU and the reference's `2*x - 1` (no /255, see
        image_processor.py) is evaluated there in fp32 — identical values, 4x fewer bytes over PCIe, no host float pass.
        A CUDA uint8 tensor [L, H, W, 3] of the target size (the pose maps of audio_models.audio_to_pose_maps) takes the
        same path without the host copy."""
        if isinstance(pose_images, torch.Tensor) and pose_images.is_cuda and pose_images.dtype == torch.uint8:
            if pose_images.dim() != 4 or tuple(pose_images.shape[1:]) != (height, width, 3):
                raise ValueError(f"pose_images: a CUDA uint8 tensor must be [L, {height}, {width}, 3], "
                                 f"got {tuple(pose_images.shape)}")
            return pose_images.to(device).permute(0, 3, 1, 2).to(torch.float32) * 2.0 - 1.0
        frames = list(pose_images)
        if all(isinstance(p, np.ndarray) and p.dtype == np.uint8 and p.ndim == 3 and p.shape[:2] == (height, width)
               for p in frames):
            shape = (len(frames), height, width, 3)
            pin = getattr(self, "_pinned_pose", None)
            if pin is None or tuple(pin.shape) != shape:
                pin = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
                self._pinned_pose = pin
            np.stack(frames, 0, out=pin.numpy())
            u8 = pin.to(device, non_blocking=True)
            return u8.permute(0, 3, 1, 2).to(torch.float32) * 2.0 - 1.0
        return torch.cat([self.cond_image_processor.preprocess(p, height=height, width=width) for p in frames], dim=0)

    def _bank_layout(self, S):
        """Shapes of the 16 ReferenceNet banks in writer order. Rank 0 knows them after its write pass; the other ranks learn
        them ONCE per session geometry (a few integers), so that every later video needs exactly one data broadcast."""
        device = S.lat.device
        mods = S.writer._modules(S.writer.unet)
        rank = torch.distributed.get_rank()
        if rank == 0:
            meta = torch.tensor([list(m.bank[0].shape) for m in mods], dtype=torch.long, device=device).reshape(-1)
        else:
            meta = torch.zeros(3 * len(mods), dtype=torch.long, device=device)
        torch.distributed.broadcast(meta, 0)
        return [tuple(int(v) for v in meta[3 * i:3 * i + 3]) for i in range(len(mods))]

    def _pack_banks(self, S):
        """Rank 0, after the write pass: the banks into the session's ONE flat fp16 buffer (46 MB at 512x512)."""
        off = 0
        for m, shp in zip(S.writer._modules(S.writer.unet), S.bank_shapes):
            n = shp[0] * shp[1] * shp[2]
            S.bank_flat[off:off + n].copy_(m.bank[0].reshape(-1))
            off += n

    def _unpack_banks(self, S):
        """Every rank, after the broadcast: the writer blocks' banks become views of the flat buffer."""
        off = 0
        for m, shp in zip(S.writer._modules(S.writer.unet), S.bank_shapes):
            n = shp[0] * shp[1] * shp[2]
            m.bank = [S.bank_flat[off:off + n].view(*shp)]
            off += n

    def _scheduler_update_rule(self):
        """(prediction_type, clip_range) of the scheduler's DDIM update, validated against what the fused CFG + DDIM kernel
        implements (diffusers DDIMScheduler.step with eta = 0). Anything else raises instead of silently producing wrong
        latents (configs/inference/inference_v2.yaml:24-33 is v_prediction without clipping; inference_v1.yaml epsilon)."""
        cfgd = getattr(self.scheduler, "config", None)

        def get(name, default):
            if cfgd is None:
                return default
            if isinstance(cfgd, dict):
                return cfgd.get(name, default)
            return getattr(cfgd, name, default)
        pred_type = get("prediction_type", "epsilon")
        if pred_type not in ops.PREDICTION_TYPES:
            raise NotImplementedError(f"scheduler prediction_type {pred_type!r} is not supported by the fused DDIM step")
        if get("thresholding", False):
            raise NotImplementedError("dynamic thresholding is not supported by the fused DDIM step")
        if not (hasattr(self.scheduler, "alpha_pair") or hasattr(self.scheduler, "alphas_cumprod")):
            raise NotImplementedError(f"{type(self.scheduler).__name__} is not a DDIM-style scheduler (no alphas_cumprod)")
        clip_range = float(get("clip_sample_range", 1.0)) if get("clip_sample", False) else 0.0
        return pred_type, clip_range

    def _alpha_pair(self, t: int):
        if hasattr(self.scheduler, "alpha_pair"):
            return self.scheduler.alpha_pair(t)
        sch = self.scheduler   # a diffusers DDIMScheduler
        prev = t - sch.config.num_train_timesteps // sch.num_inference_steps
        a_t = float(sch.alphas_cumprod[t])
        a_p = float(sch.alphas_cumprod[prev]) if prev >= 0 else float(sch.final_alpha_cumprod)
        return a_t, a_p

    # -------------------------------------------------------------------------------------------- per-video stages
    # The work of one video is split into stages that only read / write the tensors of a _Session, so that each stage can
    # either run eagerly or be captured once into a CUDA graph and replayed for every later video of the same geometry.
    def _stage_embed(self, S):
        """Library modules: CLIP image embedding -> encoder_hidden_states; reference image -> VAE latent (once per video)."""
        if S.clip_is_embed:
            emb = S.clip_in
        else:
            emb = self.image_encoder(S.clip_in).image_embeds
        ehs = emb.unsqueeze(1)
        if S.dup == 2:
            ehs = torch.cat([torch.zeros_like(ehs), ehs], dim=0)
        S.ehs = _assign(S.ehs, ehs.to(torch.float16))
        S.ref_latents = _assign(S.ref_latents, self.vae.encode(S.ref_image).latent_dist.mean * 0.18215)

    def _stage_reference_write(self, S):
        """ReferenceNet write pass (once per video): every spatial block appends norm1(x) to its bank."""
        self.reference_unet(S.ref_latents.repeat(S.dup, 1, 1, 1), torch.zeros((), device=S.lat.device),
                            encoder_hidden_states=S.ehs, return_dict=False)

    def _stage_reference_read(self, S):
        """Banks -> reader blocks (+ their K/V projections and attn2 constants); pose maps -> PoseGuider once per window."""
        S.reader.update(S.writer)
        S.win_pose = []
        for idx in S.win_idx_long:
            fea = self.pose_guider.forward_nhwc(S.pose_cond.index_select(0, idx))
            S.win_pose.append([f.to(torch.float16).contiguous() for f in fea])
        branches = {br for k, br in S.units if k != "group"} or ({"both"} if not S.groups else set())
        for G in S.groups:      # batched units: per-group pose features / embeddings (static buffers once captured)
            n, nu = len(G["elems"]), G["n_uncond"]
            G["pose"] = [torch.cat([S.win_pose[k][m] for k, _ in G["elems"]], 0).contiguous() for m in range(5)]
            G["ehs"] = torch.stack([S.ehs[b] for _, b in G["elems"]], 0).contiguous()            # [n, 1, 768]
            self.denoising_unet.prepare_reference(n, S.frames0, G["ehs"], ehs_key=S.video_key, group=(nu, n - nu))
        if "both" in branches:
            self.denoising_unet.prepare_reference(S.dup, S.frames0, S.ehs, ehs_key=S.video_key)
        for b, br in enumerate(("uncond", "cond")):       # single-branch (batch-1) units of a CFG reader
            if br in branches:
                self.denoising_unet.prepare_reference(1, S.frames0, S.ehs[b:b + 1], ehs_key=S.video_key, ref_branch=br)

    def _window_step(self, S, k):
        idx = S.win_idx[k]
        x = ops.gather_window(S.lat, idx, S.dup, 64)
        pred = self.denoising_unet.forward_nhwc(x, S.dup, idx.numel(), S.t_dev, S.ehs, S.win_pose[k],
                                                ehs_key=S.video_key)
        ops.scatter_accumulate(pred, idx, S.acc)

    def _plan_groups(self, S, units):
        """Sharded CFG sessions: the rank's units as batched calls. Elements (window, branch) in unit order, cut into groups
        of at most `group_units`, each ordered unconditional-first (the layout the attention kernel needs: frames before
        first_bank_frame skip the bank). Returns the execution list [("group", i)] and fills S.groups (static tensors only;
        the pose / embedding tensors of a group are built by _stage_reference_read)."""
        elems = []
        for k, br in units:
            elems += [(k, 0), (k, 1)] if br == "both" else [(k, 0 if br == "uncond" else 1)]
        S.groups = []
        for i in range(0, len(elems), self.group_units):
            g = sorted(elems[i:i + self.group_units], key=lambda e: e[1])       # stable: uncond (0) first
            S.groups.append(dict(elems=g, n_uncond=sum(1 for _, b in g if b == 0),
                                 idx_all=torch.cat([S.win_idx[k] for k, _ in g]).contiguous(), pose=None, ehs=None))
        return [("group", i) for i in range(len(S.groups))]

    def _group_step(self, S, gi):
        """All elements of group gi in ONE UNet call: batch = windows of this video, unconditional ones first."""
        G = S.groups[gi]
        n, nu = len(G["elems"]), G["n_uncond"]
        F = S.win_idx[G["elems"][0][0]].numel()
        x = ops.gather_window(S.lat, G["idx_all"], 1, 64)
        pred = self.denoising_unet.forward_nhwc(x, n, F, S.t_dev, G["ehs"], G["pose"], ehs_key=S.video_key,
                                                group=(nu, n - nu))
        for e, (k, b) in enumerate(G["elems"]):
            ops.scatter_accumulate(pred[e * F:(e + 1) * F], S.win_idx[k], S.acc[b:b + 1])

    def _unit_step(self, S, k, branch):
        """One (window, CFG-branch) work unit. "both" = the reference's layout (both branches in one batch); "uncond" /
        "cond" = a batch-1 UNet call for one branch (sharded mode only), accumulated into that branch's plane;
        ("group", i) = a batched call over several units of this rank (_plan_groups)."""
        if k == "group":
            return self._group_step(S, branch)
        if branch == "both":
            return self._window_step(S, k)
        idx = S.win_idx[k]
        b = 0 if branch == "uncond" else 1
        x = ops.gather_window(S.lat, idx, 1, 64)
        pred = self.denoising_unet.forward_nhwc(x, 1, idx.numel(), S.t_dev, S.ehs[b:b + 1], S.win_pose[k],
                                                ref_branch=branch, ehs_key=S.video_key)
        ops.scatter_accumulate(pred, idx, S.acc[b:b + 1])

    def _reset_block_caches(self):
        """Drop step-invariant tensors cached on the transformer blocks (bank K/V, attn2 constants) so that the next pass
        recomputes them — required right before a graph capture, otherwise the work would be missing from the graph."""
        from ..models.blocks import BasicTransformerBlock
        for net in (self.reference_unet, self.denoising_unet, self.pose_guider):
            for m in net.modules():
                if isinstance(m, BasicTransformerBlock):
                    m._bank_kv = None
                    m._attn2_const = None

    def _weights_fingerprint(self):
        return hash(tuple((p.data_ptr(), p._version) for m in self._nn_modules() for p in m.parameters()))

    def _new_session(self, clip_in, clip_is_embed, ref_image_tensor, pose_cond, L, h, w, dup, my_windows, units, static,
                     shard):
        device = self.device
        S = _Session()
        # key of the per-block step-invariant caches (attn2 constant, bank K/V): one per session, never reused, so a later
        # video can not hit an earlier video's constants (a static session keeps its key: its graphs rewrite the same
        # buffers for every video)
        Pose2VideoPipeline._video_counter += 1
        S.video_key = ("video", id(self), Pose2VideoPipeline._video_counter)
        S.clip_is_embed, S.dup, S.static, S.shard, S.units = clip_is_embed, dup, static, shard, list(units)
        enc_dtype = self.image_encoder.dtype if isinstance(self.image_encoder, torch.nn.Module) else torch.float16

        def own(t, dtype):   # static sessions own their input buffers (graphs read them on every replay)
            t = t.to(device=device, dtype=dtype)
            return t.clone() if static else t
        S.clip_in = own(clip_in, torch.float16 if clip_is_embed else enc_dtype)
        S.ref_image = own(ref_image_tensor, self.vae.dtype)
        S.pose_cond = own(pose_cond, self.pose_guider.dtype)
        S.lat = torch.empty(L, h, w, 4, dtype=torch.float16, device=device)
        S.acc = torch.zeros(dup, L, h, w, 4, dtype=torch.float32, device=device)
        S.t_dev = torch.zeros(1, dtype=torch.float32, device=device)
        S.ehs = S.ref_latents = S.win_pose = None
        S.win_idx = [torch.tensor(wd, dtype=torch.int32, device=device) for wd in my_windows]
        S.win_idx_long = [i.long() for i in S.win_idx]
        S.frames0 = len(my_windows[0]) if my_windows else 16
        cfg = dup == 2
        S.writer = ReferenceAttentionControl(self.reference_unet, do_classifier_free_guidance=cfg, mode="write",
                                             batch_size=1, fusion_blocks="full")
        S.reader = ReferenceAttentionControl(self.denoising_unet, do_classifier_free_guidance=cfg, mode="read",
                                             batch_size=1, fusion_blocks="full")
        S.g_embed = S.g_reference = S.g_write = None
        S.g_units = []
        S.n_embed = S.n_reference = S.n_write = 0
        S.n_units = []
        S.bank_shapes = S.bank_flat = None
        S.groups = []
        if shard and dup == 2 and self.group_units and units:
            S.units = self._plan_groups(S, units)
        return S

    def _capture(self, fn, pool=None):
        """Capture fn() on the side stream; returns (graph, number of this library's kernels recorded in it).
        thread_local capture mode: a process group's watchdog thread may touch the CUDA runtime while we capture."""
        g = torch.cuda.CUDAGraph()
        n0 = ops.KERNEL_LAUNCHES
        with torch.cuda.graph(g, pool=pool, stream=self._side_stream, capture_error_mode="thread_local"):
            fn()
        n = ops.KERNEL_LAUNCHES - n0
        ops.KERNEL_LAUNCHES = n0     # recorded, not launched: replays are what count
        return g, n

    def _exchange_banks(self, S, first: bool):
        """Sharded sessions: ONE NCCL broadcast of the flat bank buffer (rank 0 -> all) per video; on the first video of a
        session also the shape handshake and the buffer allocation. All ranks end with the writer banks as views of it."""
        if first:
            S.bank_shapes = self._bank_layout(S)
            S.bank_flat = torch.empty(sum(a * b * c for a, b, c in S.bank_shapes), dtype=torch.float16, device=S.lat.device)
            if torch.distributed.get_rank() == 0:
                self._pack_banks(S)
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record()
        torch.distributed.broadcast(S.bank_flat, 0)
        ev1.record()
        self._comm_events.append(("bank_broadcast_ms", ev0, ev1))
        self._unpack_banks(S)

    def _build_static_session(self, S, mark):
        """First video of a geometry: one eager pass (lazy initialisation: cuDNN plans, kernel attributes, weight packing),
        then every stage is captured. Later videos only copy their inputs into S and replay.
        Sharded sessions (S.shard): rank 0 alone runs the ReferenceNet write pass (+ packs the banks into the flat buffer);
        the bank broadcast stays an eager NCCL call between the write graph and the read graph."""
        device = self.device
        rank0 = (not S.shard) or torch.distributed.get_rank() == 0
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=device)
        side = self._side_stream
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            self._stage_embed(S)
            if rank0:
                self._stage_reference_write(S)
        torch.cuda.current_stream(device).wait_stream(side)
        if S.shard:
            self._exchange_banks(S, first=True)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            self._stage_reference_read(S)
            if S.units:
                self._unit_step(S, *S.units[0])
            S.acc.zero_()
            S.reader.clear()
            if not S.shard:
                S.writer.clear()
        torch.cuda.current_stream(device).wait_stream(side)
        mark("warm_pass_ms")
        self._reset_block_caches()
        if self.capture_library_stage:
            try:
                S.g_embed, S.n_embed = self._capture(lambda: self._stage_embed(S))
            except Exception as e:   # a library module that cannot be captured: keep that stage eager
                import warnings
                warnings.warn(f"CLIP / VAE-encode stage not graph-capturable ({type(e).__name__}: {e}); running it eagerly")
                S.g_embed = None
                torch.cuda.synchronize(device)
        if S.shard:
            if rank0:
                def write():
                    S.writer.clear()
                    self._stage_reference_write(S)
                    self._pack_banks(S)
                S.g_write, S.n_write = self._capture(write)
            self._unpack_banks(S)

            def read():
                self._stage_reference_read(S)
            S.g_reference, S.n_reference = self._capture(read, pool=S.g_write.pool() if S.g_write is not None else None)
        else:
            def reference():
                self._stage_reference_write(S)
                self._stage_reference_read(S)
            S.g_reference, S.n_reference = self._capture(reference)
        pool = S.g_reference.pool()
        for k, branch in S.units:
            g, n = self._capture(lambda k=k, branch=branch: self._unit_step(S, k, branch), pool=pool)
            S.g_units.append(g)
            S.n_units.append(n)
        mark("graph_capture_ms")

    def _replay_prologue(self, S):
        if S.g_embed is not None:
            S.g_embed.replay()
            ops._count(S.n_embed)
        else:
            self._stage_embed(S)
        if S.shard:
            if S.g_write is not None:
                S.g_write.replay()
                ops._count(S.n_write)
            self._exchange_banks(S, first=False)
        S.g_reference.replay()
        ops._count(S.n_reference)

    # -------------------------------------------------------------------------------------------- device core
    @torch.no_grad()
    def run_device(self, clip_pixels, ref_image_tensor, pose_cond, latents, num_inference_steps, guidance_scale,
                   context_schedule="uniform", context_frames=16, context_stride=1, context_overlap=4, callback=None,
                   callback_steps=1, clip_image_embeds=None, dist_mode=None, decode=True):
        """The hot path on device-resident inputs.
        clip_pixels [1,3,224,224] (or clip_image_embeds [1,768]); ref_image_tensor [1,3,H,W] in [-1,1];
        pose_cond [L,3,H,W] (pose maps as the reference's cond_image_processor emits them); latents [1,4,L,h,w].
        Returns the decoded video on the device, fp16 [1,3,L,H,W] in [0,1] (None if decode=False).

        All stages of a video geometry are captured into CUDA graphs once (a cached _Session) and replayed for every later
        video — also in the sharded modes ("windows" / "window_branches"), where each rank captures ITS units and the two
        collectives stay eager NCCL calls between graph replays: one broadcast of the flat bank buffer per video, one fp32
        all-reduce of the prediction accumulator per DDIM step. use_cuda_graph=False runs the same stages eagerly."""
        device = self.device
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        self._comm_events = []
        detail = {} if getattr(self, "profile_phases", False) else None
        t_mark = [time.perf_counter()]

        def mark(name):   # dev aid: synchronising wall-clock split of the per-video phase (off by default)
            if detail is not None:
                torch.cuda.synchronize(device)
                now = time.perf_counter()
                detail[name] = detail.get(name, 0.0) + (now - t_mark[0]) * 1e3
                t_mark[0] = now
        self.phase_detail = detail
        cfg = guidance_scale > 1.0
        dup = 2 if cfg else 1
        pred_type, clip_range = self._scheduler_update_rule()
        self.scheduler.set_timesteps(num_inference_steps, device=device)
        timesteps = [int(t) for t in self.scheduler.timesteps]
        rank, world = 0, 1
        if dist_mode is not None and torch.distributed.is_available() and torch.distributed.is_initialized():
            rank, world = torch.distributed.get_rank(), torch.distributed.get_world_size()
        if latents.shape[0] != 1:
            raise NotImplementedError("one video per call (the reference fixes batch_size = 1)")
        L, h, w = latents.shape[2], latents.shape[3], latents.shape[4]
        windows, inv_count = plan_windows(L, num_inference_steps, context_schedule, context_frames, context_stride,
                                          context_overlap)
        shard = world > 1 and dist_mode in ("windows", "window_branches")
        if shard and dist_mode == "window_branches":
            # (window, CFG branch) units: twice as many, smaller units -> better balance when windows < 2 x ranks
            mine = plan_units(len(windows), cfg, world)[rank]
            ids = sorted({k for k, _ in mine})
            my_windows = [windows[k] for k in ids]
            units = [(ids.index(k), br) for k, br in mine]
        else:
            my_windows = windows_of_rank(windows, rank, world, shard)
            units = [(k, "both") for k in range(len(my_windows))]
        inv_count = inv_count.to(device=device, dtype=torch.float32)
        clip_is_embed = clip_image_embeds is not None
        clip_in = clip_image_embeds if clip_is_embed else clip_pixels
        static = bool(self.use_cuda_graph)

        if static:
            key = (L, h, w, dup, tuple(tuple(wd) for wd in my_windows), tuple(units), shard, rank, world,
                   self.group_units if shard else 0, clip_is_embed,
                   tuple(clip_in.shape), tuple(ref_image_tensor.shape), tuple(pose_cond.shape),
                   self._weights_fingerprint())
            S = self._sessions.get(key)
            if S is None:
                while len(self._sessions) >= self.max_sessions:     # each session pins ~10 GB of activations
                    self._sessions.pop(next(iter(self._sessions)))
                S = self._new_session(clip_in, clip_is_embed, ref_image_tensor, pose_cond, L, h, w, dup, my_windows, units,
                                      True, shard)
                S.lat.copy_(latents[0].permute(1, 2, 3, 0))
                self._build_static_session(S, mark)
                self._sessions[key] = S
            else:
                S.clip_in.copy_(clip_in)
                S.ref_image.copy_(ref_image_tensor)
                S.pose_cond.copy_(pose_cond)
                S.lat.copy_(latents[0].permute(1, 2, 3, 0))
                S.acc.zero_()
            self._replay_prologue(S)
            mark("prologue_replay_ms")
        else:
            S = self._new_session(clip_in, clip_is_embed, ref_image_tensor, pose_cond, L, h, w, dup, my_windows, units,
                                  False, shard)
            S.lat.copy_(latents[0].permute(1, 2, 3, 0))
            self._stage_embed(S)
            mark("embed_ms")
            if not shard or rank == 0:
                self._stage_reference_write(S)
            if shard:
                self._exchange_banks(S, first=True)
            self._stage_reference_read(S)
            mark("reference_ms")
        lat, acc = S.lat, S.acc

        # denoising loop -----------------------------------------------------------------------------------------
        ev[1].record()
        with self.progress_bar(total=num_inference_steps) as progress_bar:
            for i, t in enumerate(timesteps):
                S.t_dev.fill_(float(t))
                if static:
                    for g, n in zip(S.g_units, S.n_units):
                        g.replay()
                        ops._count(n)
                else:
                    for k, branch in S.units:
                        self._unit_step(S, k, branch)
                if shard:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    torch.distributed.all_reduce(acc)
                    e1.record()
                    self._comm_events.append(("all_reduce_ms", e0, e1))
                a_t, a_p = self._alpha_pair(t)
                ops.cfg_ddim_step(acc, inv_count, float(guidance_scale), a_t, a_p, lat, pred_type, clip_range)
                progress_bar.update()
                if callback is not None and i % callback_steps == 0:
                    callback(i, t, lat.permute(3, 0, 1, 2).unsqueeze(0))
        ev[2].record()
        if not static:
            S.reader.clear()
            S.writer.clear()

        # decode ---------------------------------------------------------------------------------------------
        latents_out = lat.permute(3, 0, 1, 2).unsqueeze(0)                                # [1, 4, L, h, w]
        if static:
            latents_out = latents_out.clone()     # S.lat is overwritten by the next video
        self.last_latents = latents_out
        video = None
        if decode:
            if shard and L % world == 0:   # frames sharded over ranks, gathered on every rank
                part = self.decode_latents_device(latents_out[:, :, rank::world]).contiguous()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                parts = [torch.empty_like(part) for _ in range(world)]
                torch.distributed.all_gather(parts, part)
                e1.record()
                self._comm_events.append(("all_gather_ms", e0, e1))
                video = torch.empty(1, 3, L, part.shape[-2], part.shape[-1], device=device, dtype=part.dtype)
                for r in range(world):
                    video[:, :, r::world] = parts[r]
            else:
                video = self.decode_latents_device(latents_out)
        ev[3].record()
        self._events = ev
        self._meta = dict(windows=len(windows), steps=len(timesteps), units_this_rank=len(units))
        return video

    def clear_graph_cache(self):
        """Drop every cached session (static buffers + CUDA graphs)."""
        self._sessions.clear()

    def collect_timings(self):
        """Call after a synchronize: per-phase device times of the last run_device()."""
        ev = self._events
        self.timings = dict(reference_ms=ev[0].elapsed_time(ev[1]), denoise_ms=ev[1].elapsed_time(ev[2]),
                            decode_ms=ev[2].elapsed_time(ev[3]), **self._meta)
        # collectives of the sharded modes: device time between the records around each NCCL call (includes waiting for
        # the slowest rank: a rank that finished its units early sits in the all-reduce)
        for name, e0, e1 in getattr(self, "_comm_events", []):
            self.timings[name] = self.timings.get(name, 0.0) + e0.elapsed_time(e1)
        return self.timings

    # -------------------------------------------------------------------------------------------- __call__
    @torch.no_grad()
    def __call__(self, ref_image, pose_images, ref_pose_image, width, height, video_length, num_inference_steps,
                 guidance_scale, num_images_per_prompt=1, eta: float = 0.0,
                 generator: Optional[Union[torch.Generator, List[torch.Generator]]] = None,
                 output_type: Optional[str] = "tensor", return_dict: bool = True,
                 callback: Optional[Callable[[int, int, torch.Tensor], None]] = None,
                 callback_steps: Optional[int] = 1, context_schedule="uniform", context_frames=16, context_stride=1,
                 context_overlap=4, context_batch_size=1, interpolation_factor=1, clip_image_embeds=None,
                 latents=None, dist_mode=None, clip_resize=True, **kwargs):
        """Reference signature (pipeline_pose2vid_long.py:338-363). Host-side preprocessing, then run_device(), then the
        fp32 host copy of the video.
        dist_mode (only with torch.distributed initialised):
             None       every rank computes the whole video redundantly (reference behaviour)
             "windows"  the windows of ONE long video are sharded over ranks; fp32 prediction accumulator all-reduced
                        (NCCL) once per step; every rank ends with the full latents and video
             "window_branches"  as "windows" with (window, CFG branch) work units: a rank may run the unconditional or
                        the conditional half of a window as a batch-1 UNet call (SURVEY.md §8e: 22 units instead of 11
                        windows at L=128 -> 8 GPUs stay busy)
             "clips"    every rank denoises its OWN clip (its own pose_images / latents); fully independent ranks (the
                        1 ms ReferenceNet pass is recomputed per rank rather than broadcast), no collective
           In the sharded modes rank 0 alone runs the ReferenceNet and broadcasts the 16 banks (NCCL)."""
        if eta != 0.0:
            raise NotImplementedError("eta > 0 is unused by AniPortrait")
        if context_batch_size != 1:
            raise NotImplementedError("context_batch_size > 1 cannot work in the reference either (bank batch mismatch)")
        if interpolation_factor not in (0, 1):
            raise NotImplementedError("latent interpolation is disabled in the reference (interpolation_factor=1)")
        device = self.device
        if device.type != "cuda":
            raise RuntimeError("aniportrait_b200.Pose2VideoPipeline runs on CUDA (sm_100a) only: no CPU fallback")
        clip_pixels = None
        if clip_image_embeds is None:
            # the long pipeline squashes the portrait to 224x224 first (reference :375-377); the short one lets the CLIP
            # processor resize + centre-crop (src/pipelines/pipeline_pose2vid.py:320-322)
            clip_src = ref_image.resize((224, 224)) if clip_resize else ref_image
            clip_pixels = self.clip_image_processor.preprocess(clip_src, return_tensors="pt").pixel_values
        embed_dtype = self.image_encoder.dtype if isinstance(self.image_encoder, torch.nn.Module) else torch.float16
        latents = self.prepare_latents(num_images_per_prompt, self.denoising_unet.in_channels, width, height,
                                       video_length, embed_dtype, device, generator, latents)
        ref_image_tensor = self.ref_image_processor.preprocess(ref_image, height=height, width=width)
        pose_cond = self._pose_maps_to_tensor(pose_images, height, width, device)            # [L, 3, H, W]
        video = self.run_device(clip_pixels, ref_image_tensor, pose_cond, latents, num_inference_steps,
                                guidance_scale, context_schedule, context_frames, context_stride, context_overlap,
                                callback, callback_steps, clip_image_embeds, dist_mode)
        # "we always cast to float32" (reference :124-125): the conversion runs on the device and the result lands in ONE
        # pinned host buffer (a pageable fp16 copy + host-side conversion cost ~38 ms per 16-frame clip)
        # output_type="uint8" (not in the reference): packed RGB frames [B, F, H, W, 3] instead, see _to_host_u8
        images = self._to_host_u8(video) if output_type == "uint8" else self._to_host_f32(video)
        self.collect_timings()
        if output_type not in ("tensor", "uint8"):
            images = images.numpy()
        if not return_dict:
            return images
        return Pose2VideoPipelineOutput(videos=images)
