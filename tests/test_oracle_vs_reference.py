"""Pins the CPU oracle (oracle/functional.py) against the UNMODIFIED reference wiring (imported through
oracle/diffusers_shim): the reference's outputs at these sizes are stored in tests/golden/reference_units.pt by
oracle/make_golden.py, the diffusers-restating pieces (scheduler, VAE, image processor) run live from the shim. Weights are
re-created from seeds with the product classes, whose state-dict keys and shapes are the reference's
(tests/test_dropin_conformance.py); randomize_state_dict depends on names and shapes only."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import make_golden as MG  # noqa: E402
from oracle import functional as OF  # noqa: E402
from oracle import ref_import  # noqa: E402
from aniportrait_b200.synthetic import randomize_state_dict  # noqa: E402
from helpers import build_unet2d, build_unet3d  # noqa: E402

SMALL = MG.UNIT_CHANS
CFG_SMALL = dict(OF.SD15, block_out_channels=SMALL)


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


def _load(model, seed):
    sd = randomize_state_dict(model.state_dict(), seed=seed)
    model.load_state_dict(sd)
    return sd


def _pose_guider_sd(channels, seed):
    from aniportrait_b200.models.pose_guider import PoseGuider
    return randomize_state_dict(PoseGuider(channels).state_dict(), seed=seed)


@pytest.fixture(scope="module")
def gold():
    return torch.load(os.path.join(ROOT, "tests", "golden", "reference_units.pt"))


@pytest.fixture(scope="module")
def nets():
    return build_unet3d(SMALL, 1)[1], build_unet2d(SMALL, 2)[1]


def test_unet3d_plain_forward(nets, gold):
    """No reference attention: UNet3DConditionModel.forward vs oracle.unet3d_forward."""
    sd3, _ = nets
    x, ehs, pose = MG.unit_unet_inputs()
    ref = gold["unet3d_plain"]
    with torch.no_grad():
        ours = OF.unet3d_forward(sd3, x, 500, ehs, pose, banks=None, cfg=False, c=CFG_SMALL)
        OF.USE_SDPA = True        # the variant bench.py's CPU-baseline leg times (library SDPA, as the reference calls it)
        try:
            ours_sdpa = OF.unet3d_forward(sd3, x, 500, ehs, pose, banks=None, cfg=False, c=CFG_SMALL)
        finally:
            OF.USE_SDPA = False
    assert rel_l2(ours, ref) < 1e-5
    assert rel_l2(ours_sdpa, ref) < 1e-5


def test_reference_attention_read_write(nets, gold):
    """Writer/reader through ReferenceAttentionControl (CFG on) vs oracle banks + read-mode blocks."""
    sd3, sd2 = nets
    x, ehs, ref_lat = MG.unit_ref_attention_inputs()
    with torch.no_grad():
        banks = OF.reference_unet_banks(sd2, ref_lat.repeat(2, 1, 1, 1), ehs, c=CFG_SMALL)
        ours = OF.unet3d_forward(sd3, x, 959, ehs, None, banks=OF.pair_banks(banks), cfg=True, c=CFG_SMALL)
    assert len(banks) == 16
    assert rel_l2(ours, gold["unet3d_ref_attention"]) < 1e-5


def test_pose_guider(gold):
    """The reference module in train mode (the scripts never call .eval(): BatchNorm uses batch statistics); the fixture
    holds every second row and column of each output."""
    sd = _pose_guider_sd(64, 5)
    x, _ = MG.unit_pose_guider_inputs()
    with torch.no_grad():
        ours = OF.pose_guider_forward(sd, x, 64)
    assert len(ours) == len(gold["pose_guider"])
    for a, b in zip(ours, gold["pose_guider"]):
        a = a[..., ::2, ::2]
        assert a.shape == b.shape
        assert rel_l2(a, b) < 1e-5


def test_ddim_and_windows(gold):
    ref_import.activate_shim()
    from diffusers.schedulers import DDIMScheduler
    uniform = dict(gold["uniform"])
    s = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                      prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")
    s.set_timesteps(25)
    o = OF.DDIM()
    assert s.timesteps.tolist() == o.timesteps(25)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(1, 4, 2, 8, 8, generator=g)
    v = torch.randn(1, 4, 2, 8, 8, generator=g)
    for t in (999, 479, 39):
        assert rel_l2(o.step(v, t, x, 25), s.step(v, t, x).prev_sample) < 1e-6
    for n in (4, 16, 24, 128):
        assert uniform[(0, 25, n, 16, 1, 4)] == OF.context_windows(n, 16, 4)


def test_vae_decode():
    ref_import.activate_shim()
    from diffusers import AutoencoderKL
    vae = AutoencoderKL(block_out_channels=(32, 64, 128, 128))
    sd = _load(vae, 8)
    g = torch.Generator().manual_seed(9)
    z = torch.randn(2, 4, 8, 8, generator=g)
    with torch.no_grad():
        ref = vae.decode(z).sample
        ours = OF.vae_decode(sd, z)
    assert rel_l2(ours, ref) < 1e-5


def test_vae_encode():
    ref_import.activate_shim()
    from diffusers import AutoencoderKL
    vae = AutoencoderKL(block_out_channels=(32, 64, 128, 128))
    sd = _load(vae, 10)
    g = torch.Generator().manual_seed(11)
    x = torch.rand(2, 3, 64, 48, generator=g) * 2 - 1
    with torch.no_grad():
        dist = vae.encode(x).latent_dist
        ours = OF.vae_encode(sd, x)
    assert ours.shape == (2, 8, 8, 6)
    assert rel_l2(ours[:, :4], dist.mean) < 1e-5
    assert rel_l2(ours, torch.cat([dist.mean, dist.logvar], 1)) < 1e-5


def test_denoise_loop_against_the_reference_pipeline_golden():
    """The oracle's whole denoising loop (windows with wrap-around, in-loop PoseGuider on the CFG-duplicated batch, overlap
    accumulation, CFG, DDIM) + VAE decode against the committed output of the UNMODIFIED reference pipeline
    (tests/golden/pipeline_small.pt: L=20 -> two overlapping 16-frame windows, 3 steps). The host-side preparation below restates
    pipeline_pose2vid_long.py:373-447 with the (shim) library objects the reference itself uses. This is the checker the GPU
    tests use for the single-window / image pipelines, so it is pinned at pipeline level too."""
    gold_path = os.path.join(ROOT, "tests", "golden", "pipeline_small.pt")
    ref_import.activate_shim()
    from diffusers import AutoencoderKL
    from diffusers.image_processor import VaeImageProcessor
    from transformers import CLIPImageProcessor
    gold = torch.load(gold_path)
    P = gold["params"]
    seeds = P["seeds"]
    sd3 = build_unet3d(P["chans"], seeds["unet3d"])[1]
    sd2 = build_unet2d(P["chans"], seeds["unet2d"])[1]
    sdp = _pose_guider_sd(P["chans"][0], seeds["pose"])
    vae = AutoencoderKL(block_out_channels=P["vae_chans"])
    sdv = _load(vae, seeds["vae"])
    clip = MG.small_clip_encoder(seeds["clip"])
    size, L = P["size"], P["L"]
    ref_image, poses, _ = MG.pipeline_inputs(size, L, seeds["inputs"])
    with torch.no_grad():
        clip_px = CLIPImageProcessor().preprocess(ref_image.resize((224, 224)), return_tensors="pt").pixel_values
        clip_embed = clip(clip_px).image_embeds
        ref_t = VaeImageProcessor(vae_scale_factor=8, do_convert_rgb=True).preprocess(ref_image, height=size, width=size)
        ref_lat = vae.encode(ref_t).latent_dist.mean * 0.18215
        cond = VaeImageProcessor(vae_scale_factor=8, do_convert_rgb=True, do_normalize=True)
        pose_cond = torch.cat([cond.preprocess(p, height=size, width=size) for p in poses], 0)      # [L, 3, H, W]
        pose_cond = pose_cond.permute(1, 0, 2, 3).unsqueeze(0)
        lat0 = torch.randn((1, 4, L, size // 8, size // 8), generator=torch.manual_seed(seeds["latents"]))
        out = OF.denoise_loop(sd3, sd2, sdp, lat0, ref_lat, clip_embed, pose_cond, P["steps"], guidance=P["guidance"],
                              c=dict(OF.SD15, block_out_channels=tuple(P["chans"])))
        frames = [0, 7, L - 1]
        video = (OF.vae_decode(sdv, out[0, :, frames].permute(1, 0, 2, 3) / 0.18215) / 2 + 0.5).clamp(0, 1)
    assert rel_l2(out, gold["final_latents"]) < 1e-4
    assert rel_l2(video.permute(1, 0, 2, 3).unsqueeze(0), gold["video_frames"].float()) < 2e-3     # the fixture stores fp16
