"""Face-mesh pose maps on the B200 against the reference's stored output (tests/golden/pose_maps.pt): the rasteriser on
every stored cv2.line segment, pose maps at 512 x 512 and the normed pose byte for byte, other sizes per byte, smoothing
bit for bit, projection to 1e-12, the audio -> pose-map stage end to end, determinism, a kernel census, and the
pipeline's CUDA uint8 pose-map input."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pose_golden as PG  # noqa: E402
from test_pose_maps_cpu import decode_png  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    return torch.load(PG.GOLDEN, weights_only=False)


@pytest.fixture(scope="module")
def vis():
    from aniportrait_b200.utils.draw_util import FaceMeshVisualizer
    return FaceMeshVisualizer(forehead_edge=False)


def test_rasteriser_is_bit_exact_on_every_stored_segment(cuda_dev, golden):
    """Each segment as a one-edge mesh of two normalised landmarks (v = pixel / 512 is exact in fp32)."""
    from aniportrait_b200 import ops
    S = golden["segments"]
    seg = S["seg"]
    edges = torch.tensor([[0, 1, 0]], dtype=torch.int32, device=cuda_dev)
    white = torch.full((1, 3), 255, dtype=torch.uint8, device=cuda_dev)
    bad = []
    for c0 in range(0, len(seg), 500):
        chunk = seg[c0:c0 + 500]
        kp = (chunk.view(-1, 2, 2).to(torch.float32) / 512.0).to(cuda_dev)
        cover = (ops.facemesh_raster(kp, edges, white, 512, 512, normed=True)[..., 0] > 0).cpu().numpy()
        for j in range(len(chunk)):
            if not np.array_equal(cover[j], PG.unpack_mask(S["box"], S["offs"], S["bits"], c0 + j)):
                bad.append(tuple(chunk[j].tolist()))
    print(f"rasteriser: {len(seg) - len(bad)} / {len(seg)} segments bit-exact")
    assert not bad, f"{len(bad)} segments differ, e.g. {bad[:5]}"


def test_pose_maps_512_are_byte_identical(cuda_dev, golden, vis):
    kp = golden["project_points"].to(cuda_dev)
    got = vis.draw_landmarks_batch((512, 512), kp).cpu().numpy()
    for i, want in enumerate(golden["maps_512"]):
        assert np.array_equal(got[i], decode_png(want)), f"frame {i}"
    from aniportrait_b200.utils.draw_util import FaceMeshVisualizer
    got = FaceMeshVisualizer(forehead_edge=True).draw_landmarks_batch((512, 512), kp[:4]).cpu().numpy()
    for i, want in enumerate(golden["maps_512_forehead"]):
        assert np.array_equal(got[i], decode_png(want)), f"forehead frame {i}"


def test_normed_reference_pose_is_byte_identical(cuda_dev, golden, vis):
    lm = torch.from_numpy(PG.normed_landmarks()).to(cuda_dev)
    got = vis.draw_landmarks_batch((512, 512), lm[None], normed=True)[0].cpu().numpy()
    assert np.array_equal(got, decode_png(golden["normed_pose"]))


@pytest.mark.parametrize("size", [(768, 768), (384, 640)])
def test_resized_pose_maps_within_one_lsb(cuda_dev, golden, vis, size):
    W, H = size
    got = vis.draw_landmarks_batch((W, H), golden[f"kp_{W}x{H}"].to(cuda_dev)).cpu().numpy().astype(int)
    want = np.stack([decode_png(m) for m in golden[f"maps_{W}x{H}"]]).astype(int)
    diff = np.abs(got - want)
    print(f"{W}x{H}: {int((diff > 0).sum())} of {diff.size} bytes differ, max {int(diff.max())}")
    assert got.shape == want.shape and diff.max() <= 1


@pytest.mark.parametrize("name", ["f32_w7", "f32_w7_short", "f64_w3", "f64_w3_short"])
def test_smoothing_is_bit_exact(cuda_dev, golden, name):
    from aniportrait_b200.utils.pose_util import smooth_pose_seq
    x, w = PG.smoothing_inputs()[name]
    got = smooth_pose_seq(torch.from_numpy(x).to(cuda_dev), w).cpu()
    want = golden["smooth"][name]
    assert got.dtype == want.dtype and torch.equal(got, want)


def _close(got, want):
    err = ((got - want).abs() / want.abs().clamp_min(1.0)).max().item()
    print(f"projection max relative error {err:.2e}")
    return err <= 1e-12


def test_projection_within_1e12(cuda_dev, golden):
    from aniportrait_b200.utils.pose_util import project_points, project_points_with_trans
    _, trans = PG.face_cloud()
    pts = torch.from_numpy(PG.face_frames()).to(cuda_dev)
    got = project_points(pts, torch.from_numpy(trans).to(cuda_dev), torch.from_numpy(PG.head_poses()).to(cuda_dev),
                         [512, 512])
    assert got.dtype == torch.float64 and got.is_cuda and _close(got.cpu(), golden["project_points"])
    T = PG.TRANS_FRAMES
    got = project_points_with_trans(pts[:T].to(torch.float32), torch.from_numpy(PG.frame_matrices(T)).to(cuda_dev),
                                    [512, 512])
    assert _close(got.cpu(), golden["project_points_with_trans"])
    for W, H in ((768, 768), (384, 640)):
        n = PG.SIZED_FRAMES
        got = project_points(pts[:n], torch.from_numpy(trans).to(cuda_dev),
                             torch.from_numpy(PG.head_poses()[:n]).to(cuda_dev), [H, W])
        assert _close(got.cpu(), golden[f"kp_{W}x{H}"])


@pytest.mark.parametrize("branch", ["template", "chunked"])
def test_audio_to_pose_maps_end_to_end(cuda_dev, golden, branch):
    from aniportrait_b200.audio_models import audio_to_pose_maps
    lmks3d, trans = PG.face_cloud()
    E = PG.E2E
    temp = np.load(PG.POSE_TEMP) if branch == "template" else None
    maps = audio_to_pose_maps(PG.StandInMesh(), PG.StandInPose(), PG.e2e_audio().to(cuda_dev), E["seq_len"], lmks3d,
                              trans, E["width"], E["height"], id_seed=E["id_seed"], pose_temp=temp)
    assert maps.is_cuda and maps.dtype == torch.uint8 and maps.shape == (E["seq_len"], E["height"], E["width"], 3)
    got = maps.cpu().numpy()
    assert np.array_equal(got[E["seq_len"] // 2], decode_png(golden[f"e2e_{branch}_png"]))
    digests = PG.frame_digests(got)
    bad = (digests != golden[f"e2e_{branch}_digests"]).any(1).nonzero().flatten().tolist()
    assert not bad, f"{len(bad)} frames differ, first {bad[:5]}"


def test_single_frame_draw_landmarks_equals_the_batched_call(cuda_dev, golden, vis):
    kp = golden["project_points"][:3]
    batch = vis.draw_landmarks_batch((384, 640), kp.to(cuda_dev)).cpu().numpy()
    for i in range(3):
        one = vis.draw_landmarks((384, 640), kp[i].numpy())
        assert isinstance(one, np.ndarray) and one.dtype == np.uint8 and np.array_equal(one, batch[i])


def test_two_calls_give_identical_bytes(cuda_dev, golden, vis):
    from aniportrait_b200.utils.pose_util import project_points, smooth_pose_seq
    _, trans = PG.face_cloud()
    pts = torch.from_numpy(PG.face_frames()).to(cuda_dev)
    pose = torch.from_numpy(PG.head_poses()).to(cuda_dev)
    t = torch.from_numpy(trans).to(cuda_dev)

    def run():
        kp = project_points(pts, t, smooth_pose_seq(pose, 7), [640, 384])
        return kp, vis.draw_landmarks_batch((384, 640), kp)

    a, b = run(), run()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_pose_map_path_launches_only_library_kernels(cuda_dev, vis):
    from torch.profiler import ProfilerActivity, profile
    from aniportrait_b200.utils.pose_util import project_points, project_points_with_trans, smooth_pose_seq
    _, trans = PG.face_cloud()
    pts = torch.from_numpy(PG.face_frames()).to(cuda_dev)
    pose = torch.from_numpy(PG.head_poses()).to(cuda_dev)
    t = torch.from_numpy(trans).to(cuda_dev)
    mats = torch.from_numpy(PG.frame_matrices()).to(cuda_dev)

    def run():
        kp = project_points(pts, t, smooth_pose_seq(pose, 7), [512, 512])
        project_points_with_trans(pts, mats, [512, 512])
        vis.draw_landmarks_batch((768, 768), kp)

    run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA
             or getattr(e, "self_device_time_total", 0) > 0]
    names = [n for n in names if "memcpy" not in n.lower() and "memset" not in n.lower()]
    foreign = [n for n in names if "ap::" not in n]
    assert names and not foreign, f"non-library kernels on the pose-map path: {foreign}"


def test_pose_maps_to_tensor_takes_cuda_uint8_like_numpy_frames(cuda_dev, golden):
    from aniportrait_b200.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline
    pipe = object.__new__(Pose2VideoPipeline)
    frames = [decode_png(m) for m in golden["maps_384x640"]]
    want = pipe._pose_maps_to_tensor(frames, 640, 384, cuda_dev)
    got = pipe._pose_maps_to_tensor(torch.from_numpy(np.stack(frames)).to(cuda_dev), 640, 384, cuda_dev)
    assert got.shape == want.shape == (len(frames), 3, 640, 384) and torch.equal(got, want)


def test_small_pipeline_with_device_pose_maps_matches_numpy_frames(cuda_dev):
    from helpers import build_pipeline, pipeline_inputs
    gold = torch.load(os.path.join(ROOT, "tests", "golden", "pipeline_small.pt"))
    P = gold["params"]
    pipe = build_pipeline(P, cuda_dev)
    L = 4
    ref_image, poses, ref_pose = pipeline_inputs(P["size"], L, P["seeds"]["inputs"])
    dev_poses = torch.from_numpy(np.stack(poses)).to(cuda_dev)
    a = pipe(ref_image, poses, ref_pose, P["size"], P["size"], L, 2, 3.5, generator=torch.manual_seed(1)).videos
    b = pipe(ref_image, dev_poses, ref_pose, P["size"], P["size"], L, 2, 3.5, generator=torch.manual_seed(1)).videos
    assert torch.isfinite(a).all() and torch.equal(a, b)
