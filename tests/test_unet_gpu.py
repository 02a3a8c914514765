"""GPU parity of the denoising UNet3D + ReferenceNet (through the reference's call surface) against
(1) golden outputs of the UNMODIFIED reference (tests/golden/*.pt, made by oracle/make_golden.py) and
(2) the CPU fp32 oracle restatement (oracle/functional.py) on other seeded inputs.
Tolerance: rel-L2 <= 1e-2 (BASELINE.json north_star: "within 1e-2 rel-L2 of reference")."""
import os

import pytest
import torch

from helpers import build_unet2d, build_unet3d, rel_l2, seeded_inputs_unet3d

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-2


def _run_product(unet3d, unet2d, sample, ehs, ref_lat, pose, timestep, dev):
    from aniportrait_b200.models import ReferenceAttentionControl
    writer = ReferenceAttentionControl(unet2d, do_classifier_free_guidance=True, mode="write", batch_size=1,
                                       fusion_blocks="full")
    reader = ReferenceAttentionControl(unet3d, do_classifier_free_guidance=True, mode="read", batch_size=1,
                                       fusion_blocks="full")
    h16 = lambda t: t.to(dev, torch.float16)  # noqa: E731
    with torch.no_grad():
        unet2d(h16(ref_lat).repeat(2, 1, 1, 1), torch.zeros((), dtype=torch.long, device=dev),
               encoder_hidden_states=h16(ehs), return_dict=False)
        reader.update(writer)
        out = unet3d(h16(sample), torch.tensor(timestep, device=dev), encoder_hidden_states=h16(ehs),
                     pose_cond_fea=[h16(p) for p in pose], return_dict=False)[0]
    torch.cuda.synchronize()
    reader.clear()
    writer.clear()
    return out


# unet3d_full_f16_64x64 is the BENCHMARKED geometry (BASELINE.json configs[1]: 512x512 -> 64x64 latents, one 16-frame window
# under CFG = 32 frames per call, full SD1.5 width): M = 131072-row GEMMs on the wide cta_group::2 tiles, 8192-key reference
# attention (attention5_kernel) with 16 + 16 frames, temporal attention over 16 frames.
@pytest.mark.parametrize("name", ["unet3d_small_f16_16x24", "unet3d_full_f4_32x32", "unet3d_full_f16_64x64"])
def test_unet3d_against_reference_golden(cuda_dev, name):
    path = os.path.join(GOLDEN, name + ".pt")
    if not os.path.exists(path):
        pytest.skip(f"{path} missing (run oracle/make_golden.py)")
    gold = torch.load(path)
    chans, Fr, h, w = gold["chans"], gold["frames"], gold["h"], gold["w"]
    unet3d, _ = build_unet3d(chans, gold["seeds"][0], cuda_dev)
    unet2d, _ = build_unet2d(chans, gold["seeds"][1], cuda_dev)
    sample, ehs, ref_lat, pose = seeded_inputs_unet3d(2, Fr, h, w, chans, gold["seeds"][2])
    out = _run_product(unet3d, unet2d, sample, ehs, ref_lat, pose, gold["timestep"], cuda_dev)
    s = gold["out_stride"]                  # the fixture keeps every s-th latent row and column
    err = rel_l2(out[..., ::s, ::s], gold["out"])
    print(f"{name}: rel-L2 vs reference golden = {err:.3e}")
    assert tuple(out.shape) == gold["out_shape"]
    assert err < TOL, err


def test_unet3d_against_oracle_small(cuda_dev):
    """Different seeds/shape than the goldens; the oracle runs on the host CPU in fp32."""
    from oracle import functional as OF
    chans = (64, 128, 256, 256)
    cfg = dict(OF.SD15, block_out_channels=chans)
    unet3d, sd3 = build_unet3d(chans, 201, cuda_dev)
    unet2d, sd2 = build_unet2d(chans, 202, cuda_dev)
    sample, ehs, ref_lat, pose = seeded_inputs_unet3d(2, 8, 24, 16, chans, 203)
    out = _run_product(unet3d, unet2d, sample, ehs, ref_lat, pose, 39, cuda_dev)
    with torch.no_grad():
        banks = OF.reference_unet_banks(sd2, ref_lat.repeat(2, 1, 1, 1), ehs, c=cfg)
        ref = OF.unet3d_forward(sd3, sample, 39, ehs, pose, banks=OF.pair_banks(banks), cfg=True, c=cfg)
    err = rel_l2(out, ref)
    print(f"small vs oracle: rel-L2 = {err:.3e}")
    assert err < TOL, err


def test_unet3d_no_cfg_no_bank(cuda_dev):
    """guidance <= 1 path: batch 1, every frame reads the bank; and the plain (no control object) forward."""
    from oracle import functional as OF
    from aniportrait_b200.models import ReferenceAttentionControl
    chans = (64, 128, 256, 256)
    cfg = dict(OF.SD15, block_out_channels=chans)
    unet3d, sd3 = build_unet3d(chans, 211, cuda_dev)
    unet2d, sd2 = build_unet2d(chans, 212, cuda_dev)
    sample, ehs, ref_lat, pose = seeded_inputs_unet3d(1, 4, 16, 16, chans, 213)
    h16 = lambda t: t.to(cuda_dev, torch.float16)  # noqa: E731
    with torch.no_grad():
        plain = unet3d(h16(sample), 500, encoder_hidden_states=h16(ehs), return_dict=False)[0]
        ref_plain = OF.unet3d_forward(sd3, sample, 500, ehs, None, banks=None, cfg=False, c=cfg)
    assert rel_l2(plain, ref_plain) < TOL
    writer = ReferenceAttentionControl(unet2d, do_classifier_free_guidance=False, mode="write", fusion_blocks="full")
    reader = ReferenceAttentionControl(unet3d, do_classifier_free_guidance=False, mode="read", fusion_blocks="full")
    with torch.no_grad():
        unet2d(h16(ref_lat), torch.zeros((), dtype=torch.long, device=cuda_dev), encoder_hidden_states=h16(ehs))
        reader.update(writer)
        out = unet3d(h16(sample), 500, encoder_hidden_states=h16(ehs), pose_cond_fea=[h16(p) for p in pose]).sample
        banks = OF.reference_unet_banks(sd2, ref_lat, ehs, c=cfg)
        ref = OF.unet3d_forward(sd3, sample, 500, ehs, pose, banks=banks, cfg=False, c=cfg)
    reader.clear()
    writer.clear()
    assert rel_l2(out, ref) < TOL
