"""End-to-end parity of the product Pose2VideoPipeline (fp16, sm_100a kernels) against the golden output of the
UNMODIFIED reference pipeline (fp32 CPU, tests/golden/pipeline_small.pt): CLIP -> ReferenceNet bank -> two overlapping
16-frame windows x 3 DDIM steps with CFG -> VAE decode. Tolerance 1e-2 rel-L2 on the final latents (north_star)."""
import os

import pytest
import torch

from helpers import build_pipeline, pipeline_inputs, rel_l2

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_pipeline_against_reference_golden(cuda_dev):
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = gold["params"]
    pipe = build_pipeline(P, cuda_dev)
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], P["L"], P["seeds"]["inputs"])
    trace = []
    # the reference samples the initial noise in fp32 (its models were fp32); feed the same noise to the fp16 product
    g = torch.manual_seed(P["seeds"]["latents"])
    lat0 = torch.randn((1, 4, P["L"], P["size"] // 8, P["size"] // 8), generator=g, dtype=torch.float32)
    out = pipe(ref_image, poses, ref_pose, P["size"], P["size"], P["L"], P["steps"], P["guidance"],
               latents=lat0.to(torch.float16), callback=lambda i, t, l: trace.append(l.clone()), callback_steps=1)
    assert out.videos.shape == (1, 3, P["L"], P["size"], P["size"]) and out.videos.dtype == torch.float32
    e_first = rel_l2(trace[0], gold["first_step_latents"])
    e_final = rel_l2(trace[-1], gold["final_latents"])
    e_video = rel_l2(out.videos[:, :, [0, 7, P["L"] - 1]], gold["video_frames"])
    pipe.collect_timings()
    print(f"pipeline rel-L2: first step {e_first:.3e}, final latents {e_final:.3e}, video frames {e_video:.3e}; "
          f"timings {pipe.timings}")
    assert e_first < 1e-2 and e_final < 1e-2 and e_video < 1e-2
    assert 0.0 <= out.videos.min() and out.videos.max() <= 1.0


def test_pipeline_c1_full_width_against_reference_golden(cuda_dev):
    """BASELINE.json configs[0] (SURVEY.md 8d C1) at the REAL sizes: 512x512, L=4, 10 DDIM steps, CFG 3.5, full-width
    UNets / PoseGuider / sd-vae-ft-mse-sized VAE / ViT-L/14 CLIP with seeded weights, against the golden output of the
    UNMODIFIED reference pipeline (fp32 CPU, tests/golden/pipeline_c1_full.pt). Tolerance 1e-2 rel-L2 (north_star)."""
    path = os.path.join(GOLDEN, "pipeline_c1_full.pt")
    if not os.path.exists(path):
        pytest.skip(f"{path} missing (run oracle/make_golden.py pipeline_c1_full)")
    gold = torch.load(path)
    P = gold["params"]
    pipe = build_pipeline(P, cuda_dev)
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], P["L"], P["seeds"]["inputs"])
    trace = []
    g = torch.manual_seed(P["seeds"]["latents"])
    lat0 = torch.randn((1, 4, P["L"], P["size"] // 8, P["size"] // 8), generator=g, dtype=torch.float32)
    out = pipe(ref_image, poses, ref_pose, P["size"], P["size"], P["L"], P["steps"], P["guidance"],
               latents=lat0.to(torch.float16), callback=lambda i, t, l: trace.append(l.clone()), callback_steps=1)
    assert out.videos.shape == (1, 3, P["L"], P["size"], P["size"]) and out.videos.dtype == torch.float32
    e_first = rel_l2(trace[0], gold["first_step_latents"])
    e_final = rel_l2(trace[-1], gold["final_latents"])
    s = gold["video_stride"]                # the fixture keeps every s-th pixel row and column
    e_video = rel_l2(out.videos[:, :, [0, P["L"] - 1], ::s, ::s], gold["video_frames"])
    e_means = rel_l2(out.videos.mean(dim=(0, 1, 3, 4)), gold["video_frame_means"])
    print(f"C1 full-width pipeline rel-L2: first step {e_first:.3e}, final latents (10 steps) {e_final:.3e}, video frames "
          f"{e_video:.3e}, frame means {e_means:.3e}; reference CPU wall {gold['cpu_reference']['wall_s']:.0f}s on "
          f"{gold['cpu_reference']['threads']} threads")
    assert e_first < 1e-2 and e_final < 1e-2 and e_video < 1e-2


def test_pipeline_no_cfg_single_window(cuda_dev):
    """guidance_scale <= 1 (no CFG duplication) and L < 16 (single window) run and give finite output."""
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = dict(gold["params"])
    pipe = build_pipeline(P, cuda_dev)
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], 4, P["seeds"]["inputs"])
    out = pipe(ref_image, poses, ref_pose, P["size"], P["size"], 4, 2, 1.0, generator=torch.manual_seed(1))
    assert out.videos.shape == (1, 3, 4, P["size"], P["size"])
    assert torch.isfinite(out.videos).all()
    # output_type="uint8": frames packed on the device == the bytes save_videos_grid (reference src/utils/util.py:94-98)
    # makes on the host from the fp32 tensor of the same run (same seed -> replay of the same session, bit-reproducible)
    u8 = pipe(ref_image, poses, ref_pose, P["size"], P["size"], 4, 2, 1.0, generator=torch.manual_seed(1),
              output_type="uint8").videos
    assert u8.shape == (1, 4, P["size"], P["size"], 3) and u8.dtype == torch.uint8 and not u8.is_cuda
    host = torch.from_numpy((out.videos * 255).numpy().astype("uint8")).permute(0, 2, 3, 4, 1)
    assert torch.equal(u8, host)


def test_vae_kernel_decode_against_oracle(cuda_dev):
    """AutoencoderKL.decode on the sm_100a kernels (conv / GroupNorm / GEMM-softmax-GEMM attention) vs the CPU oracle."""
    from aniportrait_b200 import ops
    from aniportrait_b200.models.vae import AutoencoderKL
    from aniportrait_b200.synthetic import randomize_state_dict
    from oracle import functional as OF
    vae = AutoencoderKL(block_out_channels=(64, 64, 128, 128))
    sd = randomize_state_dict(vae.state_dict(), seed=77)
    vae.load_state_dict(sd)
    vae = vae.to(cuda_dev, torch.float16)
    g = torch.Generator().manual_seed(78)
    z = torch.randn(3, 4, 16, 8, generator=g)
    n0 = ops.KERNEL_LAUNCHES
    out = vae.decode(z.to(cuda_dev, torch.float16)).sample
    assert ops.KERNEL_LAUNCHES > n0, "VAE decode did not take the sm_100a kernel path"
    with torch.no_grad():
        ref = OF.vae_decode(sd, z)
    assert out.shape == ref.shape
    err = rel_l2(out, ref)
    print(f"vae kernel decode rel-L2 = {err:.3e}")
    assert err < 1e-2


def test_pipeline_graph_replay_matches_eager_and_is_repeatable(cuda_dev):
    """Two overlapping windows, CFG: (a) the cached CUDA-graph session (first video = capture, second = pure replay) and
    the eager path run the same kernels on the same data; every reduction in the library is atomic-free / order-fixed, so
    they must agree bit for bit (threshold 1e-6 leaves room only for library kernels); (b) a replayed session must not leak
    state from the previous video (different latents in between)."""
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = gold["params"]
    pipe = build_pipeline(P, cuda_dev)
    L = 24
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], L, P["seeds"]["inputs"])
    shape = (1, 4, L, P["size"] // 8, P["size"] // 8)
    lat_a = torch.randn(shape, generator=torch.manual_seed(5)).to(torch.float16)
    lat_b = torch.randn(shape, generator=torch.manual_seed(6)).to(torch.float16)
    args = (ref_image, poses, ref_pose, P["size"], P["size"], L, 3, P["guidance"])

    def run(lat, graph):
        pipe.use_cuda_graph = graph
        v = pipe(*args, latents=lat.clone()).videos
        return pipe.last_latents.float().cpu(), v
    a1, va1 = run(lat_a, True)        # builds + captures the session
    b1, _ = run(lat_b, True)          # replay with other latents
    a2, va2 = run(lat_a, True)        # replay again with the first latents
    ae, vae_ = run(lat_a, False)      # eager
    assert len(pipe._sessions) == 1
    e_rep, e_eager, e_other = rel_l2(a2, a1), rel_l2(ae, a1), rel_l2(b1, a1)
    print(f"replay vs first {e_rep:.3e}; eager vs graph {e_eager:.3e}; other latents {e_other:.3e}; "
          f"video eager vs graph {rel_l2(vae_, va1):.3e}")
    assert e_other > 1e-1
    assert e_rep < 1e-6 and e_eager < 1e-6 and rel_l2(va2, va1) < 1e-6 and rel_l2(vae_, va1) < 1e-6


def test_eager_pipe_second_video_does_not_reuse_first_videos_clip_constant(cuda_dev):
    """ADVICE r1 (high): the per-block attn2 constant to_out(to_v(clip)) was cached on (data_ptr, _version) of the CLIP
    embedding; a second eager video with another reference image got the first video's conditioning. Two different CLIP
    embeddings through ONE eager pipe (use_cuda_graph=False) must each equal the result of a fresh pipe."""
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = gold["params"]
    L, steps, size = 4, 2, P["size"]
    ref_image, poses, ref_pose = pipeline_inputs(size, L, 555)
    lat0 = torch.randn((1, 4, L, size // 8, size // 8), generator=torch.manual_seed(11)).to(torch.float16)
    emb_a = torch.randn(1, 768, generator=torch.manual_seed(12)).to(torch.float16)
    emb_b = torch.randn(1, 768, generator=torch.manual_seed(13)).to(torch.float16)

    def run(pipe, emb):
        pipe(ref_image, poses, ref_pose, size, size, L, steps, P["guidance"], latents=lat0.clone(),
             clip_image_embeds=emb.to(cuda_dev))
        return pipe.last_latents.float().cpu()
    shared = build_pipeline(P, cuda_dev)
    shared.use_cuda_graph = False
    a_shared = run(shared, emb_a)
    b_shared = run(shared, emb_b)       # same tensor shapes: the allocator hands back the same addresses
    fresh = build_pipeline(P, cuda_dev)
    fresh.use_cuda_graph = False
    b_fresh = run(fresh, emb_b)
    assert rel_l2(a_shared, b_fresh) > 1e-3, "the two CLIP embeddings must matter"
    assert rel_l2(b_shared, b_fresh) < 1e-6, "second video on a shared eager pipe used stale conditioning"
    # the cached-graph path with a changed embedding (replay rewrites the constants)
    shared.use_cuda_graph = True
    run(shared, emb_a)
    assert rel_l2(run(shared, emb_b), b_fresh) < 1e-6


def _host_sd(module):
    return {k: v.detach().float().cpu() for k, v in module.state_dict().items()}


def test_pose2vid_single_window_pipeline_vs_oracle(cuda_dev):
    """src/pipelines/pipeline_pose2vid.py semantics: all 20 frames are ONE window (temporal attention over 20 frames, no
    overlap averaging). Final latents vs the CPU oracle's loop with context_frames = L on the same (fp16-rounded) weights,
    CLIP embedding and reference latents."""
    from aniportrait_b200.pipelines.pipeline_pose2vid import Pose2VideoPipeline as ShortPipeline
    from oracle import functional as OF
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = gold["params"]
    base = build_pipeline(P, cuda_dev)
    pipe = ShortPipeline(vae=base.vae, image_encoder=base.image_encoder, reference_unet=base.reference_unet,
                         denoising_unet=base.denoising_unet, pose_guider=base.pose_guider, scheduler=base.scheduler)
    L, steps, size = 20, 2, P["size"]
    ref_image, poses, ref_pose = pipeline_inputs(size, L, 321)
    lat0 = torch.randn((1, 4, L, size // 8, size // 8), generator=torch.manual_seed(9)).to(torch.float16)
    out = pipe(ref_image, poses, ref_pose, size, size, L, steps, P["guidance"], latents=lat0.clone())
    assert out.videos.shape == (1, 3, L, size, size)
    got = pipe.last_latents.float().cpu()
    # oracle inputs produced by the same library modules (CLIP, VAE encoder) on the device
    with torch.no_grad():
        clip_px = pipe.clip_image_processor.preprocess(ref_image, return_tensors="pt").pixel_values
        clip_embed = pipe.image_encoder(clip_px.to(cuda_dev, torch.float16)).image_embeds.float().cpu()
        ref_t = pipe.ref_image_processor.preprocess(ref_image, height=size, width=size)
        ref_lat = (pipe.vae.encode(ref_t.to(cuda_dev, torch.float16)).latent_dist.mean * 0.18215).float().cpu()
        pose_cond = torch.cat([pipe.cond_image_processor.preprocess(p, height=size, width=size) for p in poses], 0)
        pose_cond = pose_cond.permute(1, 0, 2, 3).unsqueeze(0).to(torch.float16).float()     # [1, 3, L, H, W]
        cfg = dict(OF.SD15, block_out_channels=tuple(P["chans"]))
        ref = OF.denoise_loop(_host_sd(pipe.denoising_unet), _host_sd(pipe.reference_unet), _host_sd(pipe.pose_guider),
                              lat0.float(), ref_lat, clip_embed, pose_cond, steps, guidance=P["guidance"],
                              context_frames=L, context_overlap=0, c=cfg)
    err = rel_l2(got, ref)
    print(f"single-window pipeline (L=20) vs oracle: rel-L2 = {err:.3e}")
    assert err < 1e-2


def test_pose2img_pipeline_vs_oracle(cuda_dev):
    from aniportrait_b200.pipelines.pipeline_pose2img import Pose2ImagePipeline
    from oracle import functional as OF
    gold = torch.load(os.path.join(GOLDEN, "pipeline_small.pt"))
    P = gold["params"]
    base = build_pipeline(P, cuda_dev)
    pipe = Pose2ImagePipeline(vae=base.vae, image_encoder=base.image_encoder, reference_unet=base.reference_unet,
                              denoising_unet=base.denoising_unet, pose_guider=base.pose_guider, scheduler=base.scheduler)
    size, steps = P["size"], 2
    ref_image, poses, ref_pose = pipeline_inputs(size, 1, 77)
    lat0 = torch.randn((1, 4, 1, size // 8, size // 8), generator=torch.manual_seed(3)).to(torch.float16)
    img = pipe(ref_image, poses[0], ref_pose, size, size, steps, P["guidance"], latents=lat0.clone()).images
    assert img.shape == (1, 3, 1, size, size) and torch.isfinite(img).all()
    got = pipe.last_latents.float().cpu()
    # the CPU oracle's loop on the same (fp16-rounded) weights, CLIP embedding and reference latents, one frame
    # (src/pipelines/pipeline_pose2img.py:196-372: the image pipeline is the video loop with a single frame; :229-231
    # squashes the portrait to 224x224 for CLIP like the long pipeline)
    with torch.no_grad():
        clip_px = pipe.clip_image_processor.preprocess(ref_image.resize((224, 224)), return_tensors="pt").pixel_values
        clip_embed = pipe.image_encoder(clip_px.to(cuda_dev, torch.float16)).image_embeds.float().cpu()
        ref_t = pipe.ref_image_processor.preprocess(ref_image, height=size, width=size)
        ref_lat = (pipe.vae.encode(ref_t.to(cuda_dev, torch.float16)).latent_dist.mean * 0.18215).float().cpu()
        pose_cond = pipe.cond_image_processor.preprocess(poses[0], height=size, width=size)
        pose_cond = pose_cond.permute(1, 0, 2, 3).unsqueeze(0).to(torch.float16).float()      # [1, 3, 1, H, W]
        cfg = dict(OF.SD15, block_out_channels=tuple(P["chans"]))
        ref = OF.denoise_loop(_host_sd(pipe.denoising_unet), _host_sd(pipe.reference_unet), _host_sd(pipe.pose_guider),
                              lat0.float(), ref_lat, clip_embed, pose_cond, steps, guidance=P["guidance"],
                              context_frames=1, context_overlap=0, c=cfg)
        dec = OF.vae_decode(_host_sd(pipe.vae), ref[:, :, 0] / 0.18215)
    err = rel_l2(got, ref)
    e_img = rel_l2(img[:, :, 0], (dec / 2 + 0.5).clamp(0, 1))
    print(f"pose2img vs oracle: latents rel-L2 = {err:.3e}, image {e_img:.3e}")
    assert err < 1e-2 and e_img < 1e-2


def test_vae_kernel_encode_against_oracle(cuda_dev):
    """AutoencoderKL.encode on the sm_100a kernels (stride-2 downsamplers as gathered stride-1 convolutions, mid-block
    attention as GEMM-softmax-GEMM, quant_conv folded into conv_out) vs the CPU fp32 oracle on the same weights."""
    from aniportrait_b200 import ops
    from aniportrait_b200.models.vae import AutoencoderKL
    from aniportrait_b200.synthetic import randomize_state_dict
    from oracle import functional as OF
    vae = AutoencoderKL(block_out_channels=(64, 64, 128, 128))
    sd = randomize_state_dict(vae.state_dict(), seed=91)
    vae.load_state_dict(sd)
    vae = vae.to(cuda_dev, torch.float16)
    x = (torch.rand(2, 3, 128, 192, generator=torch.Generator().manual_seed(92)) * 2 - 1)
    n0 = ops.KERNEL_LAUNCHES
    dist = vae.encode(x.to(cuda_dev, torch.float16)).latent_dist
    assert ops.KERNEL_LAUNCHES > n0, "VAE encode did not take the sm_100a kernel path"
    with torch.no_grad():
        ref = OF.vae_encode(sd, x)
    assert dist.mean.shape == (2, 4, 16, 24)
    err = rel_l2(torch.cat([dist.mean, dist.logvar], 1), ref)
    print(f"vae kernel encode rel-L2 = {err:.3e}")
    assert err < 1e-2


def test_vae_has_no_library_fallback(cuda_dev):
    """Anything the kernels cannot run raises (no torch-op path): fp32 model, widths that are not multiples of 64."""
    from aniportrait_b200.models.vae import AutoencoderKL
    z = torch.zeros(1, 4, 8, 8, device=cuda_dev)
    with pytest.raises(RuntimeError, match="no torch-op fallback"):
        AutoencoderKL(block_out_channels=(64, 64, 128, 128)).to(cuda_dev).decode(z)                 # fp32
    with pytest.raises(RuntimeError, match="no torch-op fallback"):
        AutoencoderKL(block_out_channels=(32, 64, 128, 128)).to(cuda_dev, torch.float16).decode(z.half())
