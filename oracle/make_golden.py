"""TEST INFRASTRUCTURE — generates tests/golden/*.pt by running the UNMODIFIED reference (/root/reference/src, imported
through oracle/diffusers_shim) on CPU in fp32 with seeded synthetic weights/inputs.

    python oracle/make_golden.py [case ...]

Only the small OUTPUT tensors (plus the seeds / shapes needed to regenerate weights and inputs deterministically) are
committed; weights are re-created on the test machine by aniportrait_b200.synthetic.randomize_state_dict with the same
seed (torch's CPU generator is deterministic for a given torch version; the fixture records torch.__version__).
"""
from __future__ import annotations

import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import  # noqa: E402
from aniportrait_b200.synthetic import randomize_state_dict  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def seeded_inputs_unet3d(B, Fr, h, w, chans, seed):
    """Inputs of one denoising-UNet call; shared verbatim by the GPU tests."""
    g = torch.Generator().manual_seed(seed)
    sample = torch.randn(1, 4, Fr, h, w, generator=g).repeat(B, 1, 1, 1, 1)
    clip = torch.randn(1, 768, generator=g)
    ehs = torch.cat([torch.zeros_like(clip), clip], 0).unsqueeze(1) if B == 2 else clip.unsqueeze(1)
    ref_lat = torch.randn(1, 4, h, w, generator=g)
    sizes = [(chans[0], h), (chans[0], h // 2), (chans[1], h // 4), (chans[2], h // 8), (chans[3], h // 8)]
    pose = [0.5 * torch.randn(1, c, Fr, s, s * w // h, generator=g).repeat(B, 1, 1, 1, 1) for c, s in sizes]
    return sample, ehs, ref_lat, pose


def _load(model, seed):
    sd = randomize_state_dict(model.state_dict(), seed=seed)
    model.load_state_dict(sd)
    return sd


def case_unet3d(name, chans, Fr, h, w, timestep, seeds=(101, 102, 103), stride=1):
    """ReferenceNet write pass + denoising UNet read pass under CFG, as pipeline_pose2vid_long.py:475-544 wires them.
    Stores every `stride`-th latent row and column of the output (fixtures stay under 1 MB)."""
    ref_import.activate()
    from src.models.mutual_self_attention import ReferenceAttentionControl
    t0 = time.time()
    unet3d = ref_import.build_unet3d(chans)
    unet2d = ref_import.build_unet2d(chans)
    _load(unet3d, seeds[0])
    _load(unet2d, seeds[1])
    sample, ehs, ref_lat, pose = seeded_inputs_unet3d(2, Fr, h, w, chans, seeds[2])
    writer = ReferenceAttentionControl(unet2d, do_classifier_free_guidance=True, mode="write", batch_size=1,
                                       fusion_blocks="full")
    reader = ReferenceAttentionControl(unet3d, do_classifier_free_guidance=True, mode="read", batch_size=1,
                                       fusion_blocks="full")
    with torch.no_grad():
        unet2d(ref_lat.repeat(2, 1, 1, 1), torch.zeros((), dtype=torch.long), encoder_hidden_states=ehs,
               return_dict=False)
        reader.update(writer, dtype=torch.float32)
        out = unet3d(sample, torch.tensor(timestep), encoder_hidden_states=ehs, pose_cond_fea=pose,
                     return_dict=False)[0]
    torch.save(dict(case=name, chans=tuple(chans), frames=Fr, h=h, w=w, timestep=timestep, seeds=tuple(seeds),
                    out=out[..., ::stride, ::stride].float().contiguous(), out_shape=tuple(out.shape), out_stride=stride,
                    torch_version=str(torch.__version__),
                    generator="reference src/models via oracle/diffusers_shim, fp32 CPU"),
               os.path.join(GOLDEN, name + ".pt"))
    print(f"{name}: out {tuple(out.shape)} |out|={out.norm():.4f} in {time.time() - t0:.1f}s")


PIPE_SMALL = dict(chans=(64, 128, 256, 256), vae_chans=(64, 64, 128, 128), size=128, L=20, steps=3, guidance=3.5,
                  seeds=dict(unet3d=301, unet2d=302, pose=303, vae=304, clip=305, inputs=306, latents=42))
SCHED_KWARGS = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                    prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")


def small_clip_encoder(seed):
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    cfg = CLIPVisionConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                           image_size=224, patch_size=32, projection_dim=768)
    torch.manual_seed(seed)
    m = CLIPVisionModelWithProjection(cfg)
    m.load_state_dict(randomize_state_dict(m.state_dict(), seed=seed))
    return m.eval()


def pipeline_inputs(size, L, seed):
    """Synthetic reference image (PIL RGB) and pose maps (uint8 HxWx3 arrays with a few coloured segments), as the
    scripts pass them (scripts/pose2vid.py:120-176)."""
    import numpy as np
    import PIL.Image
    rng = np.random.RandomState(seed)
    ref_image = PIL.Image.fromarray(rng.randint(0, 256, (size + 40, size + 24, 3), dtype=np.uint8))

    def pose_map(r):
        img = np.zeros((size, size, 3), dtype=np.uint8)
        for _ in range(24):
            x0, y0 = r.randint(0, size, 2)
            ln = r.randint(4, size // 3)
            col = r.randint(64, 256, 3)
            if r.rand() < 0.5:
                img[y0:y0 + 2, x0:min(size, x0 + ln)] = col
            else:
                img[y0:min(size, y0 + ln), x0:x0 + 2] = col
        return img

    poses = [pose_map(np.random.RandomState(seed + 1 + f)) for f in range(L)]
    ref_pose = pose_map(np.random.RandomState(seed + 1000))
    return ref_image, poses, ref_pose


def case_pipeline(name="pipeline_small", P=PIPE_SMALL):
    """Whole Pose2VideoPipeline.__call__ of the reference (pipeline_pose2vid_long.py:338-584): CLIP -> ReferenceNet ->
    windowed CFG/DDIM loop with in-loop PoseGuider -> frame-wise VAE decode. Two overlapping 16-frame windows."""
    ref_import.activate()
    from diffusers import AutoencoderKL, DDIMScheduler
    from src.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline
    t0 = time.time()
    sd = P["seeds"]
    unet3d = ref_import.build_unet3d(P["chans"]); _load(unet3d, sd["unet3d"])
    unet2d = ref_import.build_unet2d(P["chans"]); _load(unet2d, sd["unet2d"])
    pose = ref_import.build_pose_guider(P["chans"][0]); _load(pose, sd["pose"])
    vae = AutoencoderKL(block_out_channels=P["vae_chans"]); _load(vae, sd["vae"])
    clip = small_clip_encoder(sd["clip"])
    pipe = Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=unet3d,
                              pose_guider=pose, scheduler=DDIMScheduler(**SCHED_KWARGS))
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], P["L"], sd["inputs"])
    lat_trace = []
    out = pipe(ref_image, poses, ref_pose, P["size"], P["size"], P["L"], P["steps"], P["guidance"],
               generator=torch.manual_seed(sd["latents"]), callback=lambda i, t, l: lat_trace.append(l.clone()),
               callback_steps=1)
    videos = out.videos
    torch.save(dict(case=name, params={k: v for k, v in P.items()}, final_latents=lat_trace[-1].float(),
                    first_step_latents=lat_trace[0].float(), video_frames=videos[:, :, [0, 7, P["L"] - 1]].half(),
                    video_mean=float(videos.mean()), torch_version=str(torch.__version__),
                    generator="reference Pose2VideoPipeline via oracle/diffusers_shim, fp32 CPU"),
               os.path.join(GOLDEN, name + ".pt"))
    print(f"{name}: videos {tuple(videos.shape)} mean={videos.mean():.4f} steps traced={len(lat_trace)} "
          f"in {time.time() - t0:.1f}s")


PIPE_C1_FULL = dict(chans=(320, 640, 1280, 1280), vae_chans=(128, 256, 512, 512), size=512, L=4, steps=10,
                    guidance=3.5, clip="vit_l_14",
                    seeds=dict(unet3d=401, unet2d=402, pose=403, vae=404, clip=405, inputs=406, latents=42))


def full_clip_encoder(seed):
    """CLIP ViT-L/14 vision tower (the architecture of sd-image-variations' image_encoder), seeded random weights."""
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    cfg = CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                           image_size=224, patch_size=14, projection_dim=768)
    torch.manual_seed(seed)
    m = CLIPVisionModelWithProjection(cfg)
    m.load_state_dict(randomize_state_dict(m.state_dict(), seed=seed))
    return m.eval()


class _PhaseTimer:
    """Wall seconds spent inside the forward of each top-level module of the reference pipeline (hooks only: the
    reference code itself is not touched)."""

    def __init__(self, **modules):
        self.seconds = {k: 0.0 for k in modules}
        self.calls = {k: 0 for k in modules}
        self._t = {}
        for name, m in modules.items():
            m.register_forward_pre_hook(lambda mod, inp, name=name: self._t.__setitem__(name, time.perf_counter()))
            m.register_forward_hook(lambda mod, inp, out, name=name: self._done(name))

    def _done(self, name):
        self.seconds[name] += time.perf_counter() - self._t[name]
        self.calls[name] += 1


def case_pipeline_c1(name="pipeline_c1_full", P=PIPE_C1_FULL):
    """BASELINE.json configs[0] (SURVEY.md 8d C1): the UNMODIFIED reference Pose2VideoPipeline at the real model sizes,
    512x512, L=4, 10 DDIM steps, CFG 3.5, fp32 on the host cores. Besides the golden tensors the fixture records the wall
    seconds of the run (whole call and per top-level module): the un-extrapolated CPU baseline of the reference."""
    ref_import.activate()
    from diffusers import AutoencoderKL, DDIMScheduler
    from src.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline
    t0 = time.time()
    sd = P["seeds"]
    unet3d = ref_import.build_unet3d(P["chans"]); _load(unet3d, sd["unet3d"])
    unet2d = ref_import.build_unet2d(P["chans"]); _load(unet2d, sd["unet2d"])
    pose = ref_import.build_pose_guider(P["chans"][0]); _load(pose, sd["pose"])
    vae = AutoencoderKL(block_out_channels=P["vae_chans"]); _load(vae, sd["vae"])
    clip = full_clip_encoder(sd["clip"])
    pipe = Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=unet3d,
                              pose_guider=pose, scheduler=DDIMScheduler(**SCHED_KWARGS))
    t_build = time.time() - t0
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], P["L"], sd["inputs"])
    timer = _PhaseTimer(denoising_unet=unet3d, reference_unet=unet2d, pose_guider=pose, image_encoder=clip,
                        vae_decoder=vae.decoder, vae_encoder=vae.encoder)
    lat_trace = []
    t1 = time.perf_counter()
    out = pipe(ref_image, poses, ref_pose, P["size"], P["size"], P["L"], P["steps"], P["guidance"],
               generator=torch.manual_seed(sd["latents"]), callback=lambda i, t, l: lat_trace.append(l.clone()),
               callback_steps=1)
    wall = time.perf_counter() - t1
    videos = out.videos
    torch.save(dict(case=name, params={k: v for k, v in P.items()}, final_latents=lat_trace[-1].float(),
                    first_step_latents=lat_trace[0].float(), video_stride=4,      # every 4th pixel row and column
                    video_frames=videos[:, :, [0, P["L"] - 1], ::4, ::4].half(),
                    video_frame_means=videos.mean(dim=(0, 1, 3, 4)).float(), torch_version=str(torch.__version__),
                    cpu_reference=dict(wall_s=wall, frames=P["L"], frames_per_s=P["L"] / wall,
                                       threads=torch.get_num_threads(), nproc=os.cpu_count(),
                                       phase_seconds=dict(timer.seconds), phase_calls=dict(timer.calls),
                                       build_s=t_build, dtype="fp32",
                                       how="time.perf_counter() around the unmodified reference "
                                           "Pose2VideoPipeline.__call__ (oracle/diffusers_shim leaves), one run, no warm-up"),
                    generator="reference Pose2VideoPipeline via oracle/diffusers_shim, fp32 CPU"),
               os.path.join(GOLDEN, name + ".pt"))
    print(f"{name}: videos {tuple(videos.shape)} mean={videos.mean():.4f} steps traced={len(lat_trace)} wall={wall:.1f}s "
          f"phases={ {k: round(v, 1) for k, v in timer.seconds.items()} } total {time.time() - t0:.1f}s")


UNIT_CHANS = (64, 128, 256, 256)


def unit_unet_inputs():
    """Inputs of the plain denoising-UNet check of tests/test_oracle_vs_reference.py (no reference attention)."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 4, 3, 16, 16, generator=g)
    ehs = torch.randn(2, 1, 768, generator=g)
    pose = [torch.randn(2, c, 3, s, s, generator=g) for c, s in [(64, 16), (64, 8), (128, 4), (256, 2), (256, 2)]]
    return x, ehs, pose


def unit_ref_attention_inputs():
    """Inputs of the ReferenceNet write / denoising-UNet read check under CFG; 16 frames per branch because the reference
    hard-codes a 16-frame uc_mask (mutual_self_attention.py:77-85)."""
    g = torch.Generator().manual_seed(4)
    x = torch.randn(1, 4, 16, 8, 8, generator=g).repeat(2, 1, 1, 1, 1)
    clip = torch.randn(1, 768, generator=g)
    ehs = torch.cat([torch.zeros_like(clip), clip], 0).unsqueeze(1)
    ref_lat = torch.randn(1, 4, 8, 8, generator=g)
    return x, ehs, ref_lat


def unit_pose_guider_inputs():
    """Pose maps of the PoseGuider check, and the reference-pose image the reference's forward takes (and ignores)."""
    g = torch.Generator().manual_seed(6)
    return torch.randn(2, 3, 2, 128, 128, generator=g), torch.randn(1, 3, 128, 128, generator=g)


# context_overlap == context_size * hop (zero range step) and larger (negative step) in the last two
UNIFORM_ARGS = [(0, 25, n, 16, 1, 4) for n in (4, 16, 24, 128)] + \
    [(0, 25, 24, 16, 2, 4), (3, 25, 50, 16, 3, 4), (0, 25, 40, 16, 1, 16), (0, 25, 40, 16, 1, 20)]
FILM_CASES = [(1, 5), (2, 3)]             # (batch, frames) of the frame-interpolation check, 1..5 inserted frames each
POSE_CASES = [(0, 64, 37, True), (1, 128, 61, False)]      # (seed, latent_dim, frames, only_last_features)


def pose_model_weights(model, seed):
    """Seeded weights of everything but the audio encoder of an Audio2PoseModel; fan-in scaled so that the 8 decoder layers
    move the result (the default init is close to the identity)."""
    sd = {k: v for k, v in model.state_dict().items() if not k.startswith("audio_encoder.")}
    return randomize_state_dict(sd, seed=seed, std=1.0)


def _uniform_outcome(uniform, args):
    try:
        return [list(map(int, w)) for w in uniform(*args)]
    except ValueError:
        return "ValueError"


def case_reference_units(name="reference_units"):
    """Outputs of the UNMODIFIED reference's modules and helpers at unit-test sizes, for the checks that compare the CPU
    oracle or a host-side rewrite with the reference: denoising UNet (plain and with reference attention), PoseGuider,
    the context-window scheduler, the FILM frame-interpolation loop (on the tests' stand-in network) and the head-pose
    decoder (Audio2PoseModel.infer). Also the constructor / call / state-dict surface of the reference classes."""
    import gzip
    import importlib.util
    import json
    import tempfile
    ref_import.activate()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from src.models.mutual_self_attention import ReferenceAttentionControl
    from src.pipelines.context import uniform
    from test_dropin_conformance import _probe
    from test_host_cpu import _StandInFilm
    t0 = time.time()
    G = dict(case=name, torch_version=str(torch.__version__), generator="reference src/ via oracle/diffusers_shim, fp32 CPU")
    torch.manual_seed(0)
    unet3d, unet2d = ref_import.build_unet3d(UNIT_CHANS), ref_import.build_unet2d(UNIT_CHANS)
    _load(unet3d, 1)
    _load(unet2d, 2)
    x, ehs, pose = unit_unet_inputs()
    with torch.no_grad():
        G["unet3d_plain"] = unet3d(x, torch.tensor(500), encoder_hidden_states=ehs, pose_cond_fea=pose,
                                   return_dict=False)[0]
    x, ehs, ref_lat = unit_ref_attention_inputs()
    writer = ReferenceAttentionControl(unet2d, do_classifier_free_guidance=True, mode="write", batch_size=1,
                                       fusion_blocks="full")
    reader = ReferenceAttentionControl(unet3d, do_classifier_free_guidance=True, mode="read", batch_size=1,
                                       fusion_blocks="full")
    with torch.no_grad():
        unet2d(ref_lat.repeat(2, 1, 1, 1), torch.zeros((), dtype=torch.long), encoder_hidden_states=ehs, return_dict=False)
        reader.update(writer, dtype=torch.float32)
        G["unet3d_ref_attention"] = unet3d(x, torch.tensor(959), encoder_hidden_states=ehs, return_dict=False)[0]
    pg = ref_import.build_pose_guider(64)
    _load(pg, 5)
    pg.train()  # the scripts never call .eval(): BatchNorm uses batch statistics
    with torch.no_grad():    # every second row and column of each output: the stored sample stays small
        G["pose_guider"] = [t[..., ::2, ::2].clone() for t in pg(*unit_pose_guider_inputs())]
    G["uniform"] = [(args, _uniform_outcome(uniform, args)) for args in UNIFORM_ARGS]

    spec = importlib.util.spec_from_file_location(
        "_ref_frame_interpolation", os.path.join(ref_import.REFERENCE_ROOT, "src", "utils", "frame_interpolation.py"))
    film = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(film)
    cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self      # the reference hard-codes .cuda()
    try:
        g = torch.Generator().manual_seed(3)
        G["film"] = []
        for bs, frames in FILM_CASES:
            video = torch.rand((bs, 3, frames, 8, 12), generator=g)              # fp32, not fp16-representable
            G["film"].append(dict(video=video, out=[film.batch_images_interpolation_tool(video, _StandInFilm(), n)
                                                    for n in range(1, 6)]))
    finally:
        torch.Tensor.cuda = cuda

    from transformers import Wav2Vec2Config
    from src.audio_models.pose_model import Audio2PoseModel
    G["pose_infer"] = []
    with tempfile.TemporaryDirectory() as cfg_dir:
        cfg = Wav2Vec2Config(hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128,
                             conv_dim=(32, 32, 32), conv_stride=(5, 4, 2), conv_kernel=(10, 4, 2),
                             num_feat_extract_layers=3, num_conv_pos_embeddings=16, num_conv_pos_embedding_groups=4)
        cfg._attn_implementation = "eager"        # the reference's wav2vec2 wrapper asks for attention maps
        cfg.save_pretrained(cfg_dir)
        for seed, latent, T, only_last in POSE_CASES:
            torch.manual_seed(seed)
            m = Audio2PoseModel(dict(latent_dim=latent, model_path=cfg_dir, only_last_fetures=only_last,
                                     from_pretrained=False, out_dim=6)).eval()
            m.audio_encoder.config._attn_implementation = "eager"
            m.load_state_dict(pose_model_weights(m, seed), strict=False)
            with torch.no_grad():
                audio = torch.randn(1, 16000)
                emb = m.audio_encoder(audio, seq_len=T, output_hidden_states=True)
                want = m.infer(audio, T, id_seed=torch.tensor([7]))
            spread = (want[0, 1:] - want[0, :-1]).abs().mean().item()
            assert spread > 1e-3, "degenerate reference output: the check would prove nothing"
            features = emb.last_hidden_state if only_last else torch.stack(emb.hidden_states)
            G["pose_infer"].append(dict(seed=seed, latent=latent, frames=T, only_last=only_last, features=features,
                                        pe=m.PPE.pe[:, :T].clone(), out=want))
            G["pose_biased_mask"] = m.biased_mask[:, :T, :T].clone()     # the same buffer in every model; largest T last
    torch.save(G, os.path.join(GOLDEN, name + ".pt"))
    with gzip.open(os.path.join(GOLDEN, "dropin_reference_surface.json.gz"), "wt") as f:
        json.dump(_probe("reference"), f, sort_keys=True)
    print(f"{name}: written in {time.time() - t0:.1f}s")


CASES = {
    "reference_units": case_reference_units,
    "pipeline_small": case_pipeline,
    "pipeline_c1_full": case_pipeline_c1,
    # the benchmarked geometry (BASELINE.json configs[1]): full width, 64x64 latents, one 16-frame window under CFG
    "unet3d_full_f16_64x64": lambda: case_unet3d("unet3d_full_f16_64x64", (320, 640, 1280, 1280), 16, 64, 64, 479,
                                                  seeds=(121, 122, 123), stride=2),
    # full SD1.5 width (the real model size), 256x256-pixel equivalent latents, 4-frame window
    "unet3d_full_f4_32x32": lambda: case_unet3d("unet3d_full_f4_32x32", (320, 640, 1280, 1280), 4, 32, 32, 479),
    # reduced width, 16-frame window (temporal attention at the production window length), non-square latent
    "unet3d_small_f16_16x24": lambda: case_unet3d("unet3d_small_f16_16x24", (64, 128, 256, 256), 16, 16, 24, 959,
                                                   seeds=(111, 112, 113)),
}

if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 8)
    names = sys.argv[1:] or list(CASES)
    for n in names:
        CASES[n]()
