"""TEST INFRASTRUCTURE — import the UNMODIFIED reference (/root/reference/src) through oracle/diffusers_shim.
Only usable in the authoring container (the GPU box has no /root/reference); used to pin oracle/functional.py and to
generate tests/golden/*.pt (oracle/make_golden.py)."""
import os
import sys

REFERENCE_ROOT = os.environ.get("ANIPORTRAIT_REFERENCE", "/root/reference")
SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "diffusers_shim")


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "models"))


def activate_shim():
    """Only the diffusers shim (part of this repository): what the checks that need no reference module import."""
    if SHIM not in sys.path:
        sys.path.insert(0, SHIM)


def activate():
    if not available():
        raise RuntimeError(f"reference not found at {REFERENCE_ROOT}")
    activate_shim()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


MOTION_KWARGS = dict(num_attention_heads=8, num_transformer_block=1,
                     attention_block_types=["Temporal_Self", "Temporal_Self"], temporal_position_encoding=True,
                     temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)


def build_unet3d(block_out_channels=(320, 640, 1280, 1280)):
    """UNet3DConditionModel as from_pretrained_2d builds it from SD1.5's unet/config.json + inference_v2.yaml."""
    activate()
    from src.models.unet_3d import UNet3DConditionModel
    return UNet3DConditionModel(
        sample_size=64, in_channels=4, out_channels=4, block_out_channels=tuple(block_out_channels),
        cross_attention_dim=768, attention_head_dim=8, use_inflated_groupnorm=True,
        unet_use_cross_frame_attention=False, unet_use_temporal_attention=False, use_motion_module=True,
        motion_module_resolutions=[1, 2, 4, 8], motion_module_mid_block=True, motion_module_decoder_only=False,
        motion_module_type="Vanilla", motion_module_kwargs=dict(MOTION_KWARGS))


def build_unet2d(block_out_channels=(320, 640, 1280, 1280)):
    activate()
    from src.models.unet_2d_condition import UNet2DConditionModel
    return UNet2DConditionModel(sample_size=64, in_channels=4, out_channels=4,
                                block_out_channels=tuple(block_out_channels), cross_attention_dim=768,
                                attention_head_dim=8)


def build_pose_guider(channels=320):
    activate()
    from src.models.pose_guider import PoseGuider
    return PoseGuider(noise_latent_channels=channels, use_ca=True)
