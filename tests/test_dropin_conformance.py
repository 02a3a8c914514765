"""The drop-in boundary (SURVEY.md 8b): `dropin/src/...` must expose, under the reference's import paths, classes whose
constructor / forward / __call__ signatures accept everything the reference's scripts pass, and whose state-dict keys are
exactly the reference's (so denoising_unet.pth / motion_module.pth / reference_unet.pth / pose_guider.pth load). Compared
against the surface of the UNMODIFIED reference classes (imported through oracle/diffusers_shim), stored in
tests/golden/dropin_reference_surface.json.gz by oracle/make_golden.py. The probe runs in its own interpreter: the drop-in
and the reference both define a top-level `src` package."""
import gzip
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBE = r'''
import inspect, json, sys
side = sys.argv[1]
if side == "reference":
    sys.path.insert(0, sys.argv[2]); from oracle import ref_import; ref_import.activate()
else:
    sys.path.insert(0, sys.argv[2] + "/dropin"); sys.path.insert(0, sys.argv[2])
import torch
from src.models.unet_3d import UNet3DConditionModel
from src.models.unet_2d_condition import UNet2DConditionModel
from src.models.pose_guider import PoseGuider
from src.models.mutual_self_attention import ReferenceAttentionControl
from src.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline
from src.pipelines.pipeline_pose2vid import Pose2VideoPipeline as ShortPipeline
from src.pipelines.pipeline_pose2img import Pose2ImagePipeline
from src.pipelines.context import get_context_scheduler
from src.utils.frame_interpolation import batch_images_interpolation_tool, init_frame_interpolation_model

def sig(fn):
    out = []
    for n, p in inspect.signature(fn).parameters.items():
        if n == "self" or p.kind in (p.VAR_KEYWORD, p.VAR_POSITIONAL):
            continue
        d = None if p.default is inspect._empty else repr(p.default)
        out.append([n, d])
    return out

MOTION = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
              temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)
chans = (32, 64, 64, 64)
with torch.device("meta"):
    u3 = UNet3DConditionModel(sample_size=8, block_out_channels=chans, cross_attention_dim=768, attention_head_dim=8,
                              use_inflated_groupnorm=True, unet_use_cross_frame_attention=False,
                              unet_use_temporal_attention=False, use_motion_module=True,
                              motion_module_resolutions=[1, 2, 4, 8], motion_module_mid_block=True,
                              motion_module_type="Vanilla", motion_module_kwargs=dict(MOTION))
    u2 = UNet2DConditionModel(sample_size=8, block_out_channels=chans, cross_attention_dim=768, attention_head_dim=8)
    pg = PoseGuider(noise_latent_channels=64, use_ca=True)
res = {
    "sig": {
        "UNet3D.forward": sig(UNet3DConditionModel.forward),
        "UNet3D.from_pretrained_2d": sig(UNet3DConditionModel.from_pretrained_2d),
        "UNet2D.forward": sig(UNet2DConditionModel.forward),
        "PoseGuider.__init__": sig(PoseGuider.__init__),
        "PoseGuider.forward": sig(PoseGuider.forward),
        "ReferenceAttentionControl.__init__": sig(ReferenceAttentionControl.__init__),
        "ReferenceAttentionControl.update": sig(ReferenceAttentionControl.update),
        "ReferenceAttentionControl.clear": sig(ReferenceAttentionControl.clear),
        "Pose2VideoPipeline.__init__": sig(Pose2VideoPipeline.__init__),
        "Pose2VideoPipeline.__call__": sig(Pose2VideoPipeline.__call__),
        "ShortPipeline.__call__": sig(ShortPipeline.__call__),
        "Pose2ImagePipeline.__call__": sig(Pose2ImagePipeline.__call__),
        "context.uniform": sig(get_context_scheduler("uniform")),
        "batch_images_interpolation_tool": sig(batch_images_interpolation_tool),
        "init_frame_interpolation_model": sig(init_frame_interpolation_model),
    },
    "keys": {"unet3d": sorted(u3.state_dict().keys()), "unet2d": sorted(u2.state_dict().keys()),
             "pose_guider": sorted(pg.state_dict().keys())},
    "shapes": {"unet3d": {k: list(v.shape) for k, v in u3.state_dict().items()},
               "unet2d": {k: list(v.shape) for k, v in u2.state_dict().items()},
               "pose_guider": {k: list(v.shape) for k, v in pg.state_dict().items()}},
    "attrs": {"unet3d.in_channels": int(u3.in_channels), "has_blocks": all(hasattr(u3, a) for a in
              ("down_blocks", "mid_block", "up_blocks", "config", "dtype", "device"))},
}
print("PROBE_JSON" + json.dumps(res))
'''


def _probe(side):
    """side "product": the drop-in classes; side "reference": the reference's (oracle/make_golden.py stores that result)."""
    from oracle import ref_import
    r = subprocess.run([sys.executable, "-c", PROBE, side, ROOT], capture_output=True, text=True, timeout=600,
                       cwd=ROOT if side == "product" else ref_import.REFERENCE_ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE_JSON")][-1]
    return json.loads(line[len("PROBE_JSON"):])


def test_dropin_surface_matches_reference_classes():
    with gzip.open(os.path.join(ROOT, "tests", "golden", "dropin_reference_surface.json.gz"), "rt") as f:
        ref = json.load(f)
    ours = _probe("product")
    # 1. every parameter the reference accepts exists on ours, in the same position, with the same default
    for name, rsig in ref["sig"].items():
        osig = ours["sig"][name]
        onames = [n for n, _ in osig]
        if name == "UNet2D.forward":
            # the ReferenceNet forward keeps the positional core; the reference's nine unused optional kwargs
            # (class_labels .. return_dict handled) may be absent only if they default to None there
            core = [p for p in rsig if p[1] is None or p[0] in onames]
            for (n, d) in rsig:
                if n not in onames:
                    assert d == "None", f"{name}: reference parameter {n} (default {d}) missing"
            rsig = [p for p in rsig if p[0] in onames]
            osig = [p for p in osig if p[0] in [q[0] for q in rsig]]
        assert [n for n, _ in rsig] == onames[:len(rsig)] or name == "UNet2D.forward" and \
            [n for n, _ in rsig] == [n for n, _ in osig], f"{name}: parameter order differs: {rsig} vs {osig}"
        for (n, d), (n2, d2) in zip(rsig, osig):
            # a parameter that is required in the reference may carry a default here (strictly more permissive)
            assert n == n2 and (d in (None, "Ellipsis") or d == d2), f"{name}: {n}={d} (reference) vs {n2}={d2} (drop-in)"
    # 2. identical state-dict keys and shapes -> the published checkpoints load
    for m in ("unet3d", "unet2d", "pose_guider"):
        assert ours["keys"][m] == ref["keys"][m], (m, sorted(set(ours["keys"][m]) ^ set(ref["keys"][m]))[:8])
        assert ours["shapes"][m] == ref["shapes"][m], m
    assert ours["attrs"] == ref["attrs"]
