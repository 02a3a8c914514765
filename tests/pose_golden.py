"""Golden data of the face-mesh pose-map stage (tests/golden/pose_maps.pt) and the seeded inputs it is made from.

    python tests/pose_golden.py          # needs a reference checkout (oracle/mediapipe_import.py), runs on the CPU

Runs the UNMODIFIED reference src/utils/draw_util.FaceMeshVisualizer (through oracle/mediapipe_shim) and
src/utils/pose_util (scipy, cv2) and stores:
  * the visualiser's face_connection_spec as an ordered (edge, colour) list, for both forehead_edge values;
  * cv2.line(thickness=2) coverage of ~4000 seeded integer segments on the 512 x 512 canvas, as packed-bit masks cropped
    to each segment's bounding box;
  * smooth_pose_seq outputs (fp32 window 7, fp64 window 3, including L < window);
  * project_points / project_points_with_trans outputs (fp64) of a seeded 468-point face cloud;
  * pose maps drawn from those projections at 512 x 512 (PNG), 768 x 768 and 384 x 640 (W x H), and the normed=True
    pose of a 478-point landmark set;
  * one end-to-end run of audio2vid's audio -> pose-map stage (scripts/audio2vid.py:161-205) on stand-in audio models,
    for the pose-template branch and the chunked head-pose branch, as per-frame SHA-256 digests.
The functions that regenerate the inputs are imported by the tests and scripts/bench_pose_maps.py; only outputs are stored.
"""
from __future__ import annotations

import hashlib
import inspect
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "pose_maps.pt")
POSE_TEMP = os.path.join(ROOT, "tests", "golden", "pose_temp.npy")   # configs/inference/head_pose_temp/pose_temp.npy

SEEDS = dict(segments=801, face=802, poses=803, smooth=804, normed=805, mesh=806, head_pose=807)
FRAMES = 20                    # frames of the projection / 512 x 512 pose-map case (fixture size)
TRANS_FRAMES = 8               # frames of the project_points_with_trans case
SIZED_FRAMES = 2               # frames per non-square / enlarged size
E2E = dict(samples=196800, seq_len=369, width=512, height=512, id_seed=7)   # 12.3 s at 16 kHz / 30 fps: 3 chunks


def face_cloud(seed=SEEDS["face"]):
    """468 points of face size (about 14 x 18 x 6 units, the scale of mediapipe's canonical face) and the reference
    face's transformation matrix: a small rotation and a translation to z = -40 (fp32, as mediapipe returns it)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(468, 3, generator=g, dtype=torch.float64)
    u = u / u.norm(dim=1, keepdim=True) * torch.rand(468, 1, generator=g, dtype=torch.float64) ** (1 / 3)
    lmks3d = u * torch.tensor([7.0, 9.0, 3.0], dtype=torch.float64)
    a = 0.05
    trans = torch.tensor([[1.0, -a, 0.0, 0.4], [a, 1.0, 0.0, -0.3], [0.0, 0.0, 1.0, -40.0], [0.0, 0.0, 0.0, 1.0]],
                         dtype=torch.float32)
    return lmks3d.numpy(), trans.numpy()


def head_poses(L=FRAMES, seed=SEEDS["poses"]):
    """[L, 6] fp32 poses (degrees, then translation). Every 5th frame is pushed sideways or turned far so that some
    landmarks leave the canvas; frame 3 moves the face almost entirely out."""
    g = torch.Generator().manual_seed(seed)
    pose = torch.cat([torch.randn(L, 3, generator=g) * 12.0, torch.randn(L, 3, generator=g) * 1.5], dim=1)
    shifts = torch.tensor([24.0, -22.0, 18.0, -26.0, 30.0, -20.0, 22.0])
    pose[::5, 3] += shifts.repeat(L // 35 + 1)[: len(pose[::5])]
    pose[2::7, 1] += 60.0
    pose[3, 4] = 40.0
    return pose.to(torch.float32).numpy()


def face_frames(L=FRAMES, seed=SEEDS["mesh"]):
    """[L, 468, 3] fp64: the face cloud plus a small per-frame deformation (the Audio2Mesh output's role)."""
    lmks3d, _ = face_cloud()
    g = torch.Generator().manual_seed(seed)
    d = 0.2 * torch.randn(L, 468, 3, generator=g)
    return d.to(torch.float32).numpy() + lmks3d


def frame_matrices(L=FRAMES):
    """[L, 4, 4] fp64 per-frame matrices for project_points_with_trans: trans @ pose matrix of head_poses."""
    from scipy.spatial.transform import Rotation
    _, trans = face_cloud()
    out = np.zeros((L, 4, 4))
    for i, p in enumerate(head_poses(L)):
        m = np.eye(4)
        m[:3, :3] = Rotation.from_euler("xyz", p[:3], degrees=True).as_matrix()
        m[:3, 3] = p[3:]
        out[i] = trans @ m
    return out


def smoothing_inputs(seed=SEEDS["smooth"]):
    """{name: (array, window)}: fp32 window 7 and fp64 window 3, each at a long and a shorter-than-window length."""
    g = torch.Generator().manual_seed(seed)
    return {
        "f32_w7": ((torch.randn(300, 6, generator=g) * 10).numpy(), 7),
        "f32_w7_short": ((torch.randn(5, 6, generator=g) * 10).numpy(), 7),
        "f64_w3": ((torch.randn(61, 6, generator=g, dtype=torch.float64) * 10).numpy(), 3),
        "f64_w3_short": ((torch.randn(2, 6, generator=g, dtype=torch.float64) * 10).numpy(), 3),
    }


def normed_landmarks(seed=SEEDS["normed"]):
    """478 normalised fp32 landmarks (x, y, z) as LMKExtractor returns them, a few outside [0, 1] or on its edges."""
    lmks3d, trans = face_cloud()
    pts = np.concatenate([lmks3d, lmks3d[:10] * 0.3], 0)
    g = torch.Generator().manual_seed(seed)
    xy = 0.5 + pts[:, :2] / 30.0 + 0.002 * torch.randn(478, 2, generator=g, dtype=torch.float64).numpy()
    xy[5], xy[6], xy[7], xy[8] = (1.0, 0.5), (0.0, 0.25), (1.0 + 1e-7, 0.5), (0.5, -1e-7)
    xy[9] = (np.nan, 0.5)
    out = np.concatenate([xy, pts[:, 2:] / 30.0], 1)
    return out.astype(np.float32)


def segments(seed=SEEDS["segments"]):
    """~4000 integer segments inside the 512 x 512 canvas: mostly short, many on the borders, horizontal, vertical,
    steep, zero-length and a few longer diagonals. int32 [S, 4] (x0, y0, x1, y1)."""
    rng = np.random.default_rng(seed)
    out = []

    def add(x0, y0, x1, y1):
        out.append([int(np.clip(v, 0, 511)) for v in (x0, y0, x1, y1)])

    for _ in range(2400):
        x0, y0 = rng.integers(0, 512, 2)
        dx, dy = rng.integers(-16, 17, 2)
        add(x0, y0, x0 + dx, y0 + dy)
    for _ in range(700):
        x0, y0 = rng.integers(0, 512, 2)
        e = rng.choice([0, 1, 2, 509, 510, 511])
        if rng.random() < 0.5:
            x0 = e
        else:
            y0 = e
        dx, dy = rng.integers(-8, 9, 2)
        add(x0, y0, x0 + dx, y0 + dy)
    for _ in range(300):
        x0, y0 = rng.integers(0, 512, 2)
        n = rng.integers(-200, 201)
        add(x0, y0, x0 + n, y0) if rng.random() < 0.5 else add(x0, y0, x0, y0 + n)
    for _ in range(300):
        x0, y0 = rng.integers(0, 512, 2)
        add(x0, y0, x0 + rng.integers(-3, 4), y0 + rng.integers(-90, 91))
    for _ in range(150):
        x0, y0 = rng.integers(0, 512, 2)
        add(x0, y0, x0, y0)
    for _ in range(150):
        x0, y0 = rng.integers(0, 512, 2)
        dx, dy = rng.integers(-64, 65, 2)
        add(x0, y0, x0 + dx, y0 + dy)
    for c in ((0, 0, 511, 511), (511, 0, 0, 511), (0, 0, 0, 0), (511, 511, 511, 511), (0, 511, 511, 511),
              (3, 0, 5, 0), (0, 7, 0, 9), (511, 100, 509, 101)):
        add(*c)
    return np.array(out, dtype=np.int32)


def pack_masks(masks_and_boxes):
    """[(mask bool [h, w], (y0, x0))] -> (box int32 [S, 4] = (y0, x0, h, w), offs int64 [S + 1], bits uint8)."""
    boxes, offs, chunks = [], [0], []
    for m, (y0, x0) in masks_and_boxes:
        boxes.append((y0, x0, m.shape[0], m.shape[1]))
        b = np.packbits(m.ravel())
        chunks.append(b)
        offs.append(offs[-1] + len(b))
    return (torch.tensor(boxes, dtype=torch.int32), torch.tensor(offs, dtype=torch.int64),
            torch.from_numpy(np.concatenate(chunks)))


def unpack_mask(box, offs, bits, i, shape=(512, 512)):
    """The full-canvas bool mask of segment i."""
    y0, x0, h, w = (int(v) for v in box[i])
    b = np.asarray(bits[int(offs[i]):int(offs[i + 1])])
    m = np.zeros(shape, dtype=bool)
    m[y0:y0 + h, x0:x0 + w] = np.unpackbits(b, count=h * w).reshape(h, w).astype(bool)
    return m


def png(img: np.ndarray) -> torch.Tensor:
    import cv2
    ok, buf = cv2.imencode(".png", img, [cv2.IMWRITE_PNG_COMPRESSION, 9])
    assert ok
    return torch.from_numpy(buf.reshape(-1).copy())


def unpng(t: torch.Tensor) -> np.ndarray:
    import cv2
    return cv2.imdecode(t.numpy(), cv2.IMREAD_UNCHANGED)


def frame_digests(frames) -> torch.Tensor:
    """uint8 [L, 32]: SHA-256 of each uint8 [H, W, 3] frame's bytes (C order)."""
    return torch.tensor([list(hashlib.sha256(np.ascontiguousarray(f).tobytes()).digest()) for f in frames],
                        dtype=torch.uint8)


class StandInMesh:
    """Stand-in Audio2MeshModel: infer(audio, seq_len) -> [1, seq_len, 1404] fp32 on the audio's device, seeded by the
    audio length (small mesh offsets, the scale of Audio2Mesh's output)."""

    def infer(self, input_value, seq_len):
        g = torch.Generator().manual_seed(SEEDS["mesh"] * 1000 + input_value.shape[1] % 997)
        out = 0.15 * torch.randn(1, seq_len, 1404, generator=g)
        return out.to(input_value.device)


class StandInPose:
    """Stand-in Audio2PoseModel: infer(audio, seq_len, id_seed) -> [1, seq_len, 6] fp32 on the audio's device, a smooth
    seeded head motion (degrees, then translation) that depends on the chunk's length and the identity seed."""

    def infer(self, input_value, seq_len, id_seed):
        g = torch.Generator().manual_seed(SEEDS["head_pose"] * 100000 + input_value.shape[1] * 101 + int(id_seed.item()))
        t = torch.arange(seq_len, dtype=torch.float32)[:, None]
        amp = torch.randn(1, 6, generator=g) * torch.tensor([[8.0, 8.0, 4.0, 0.5, 0.5, 0.3]])
        freq = 0.02 + 0.05 * torch.rand(1, 6, generator=g)
        out = amp * torch.sin(freq * t) + 0.3 * torch.randn(seq_len, 6, generator=g)
        return out.to(torch.float32).unsqueeze(0).to(input_value.device)


def e2e_audio():
    g = torch.Generator().manual_seed(SEEDS["head_pose"])
    return torch.randn(1, E2E["samples"], generator=g)


def reference_audio_to_pose_maps(vis, pose_util, a2m, a2p, audio, seq_len, lmks3d, trans_mat, width, height, id_seed,
                                 pose_temp):
    """The audio -> pose-map steps of scripts/audio2vid.py:161-205 (5 s chunks at 30 fps, rotation halved, window-7
    smoothing), run on the reference's numpy pose_util and draw_util."""
    pred = a2m.infer(audio, seq_len).squeeze().detach().cpu().numpy()
    pred = pred.reshape(pred.shape[0], -1, 3) + lmks3d
    if pose_temp is not None:
        mirrored = np.concatenate((pose_temp, pose_temp[-2:0:-1]), axis=0)
        pose_seq = np.tile(mirrored, (seq_len // len(mirrored) + 1, 1))[:seq_len]
    else:
        chunks = list(audio.split(16000 * 5, dim=1))
        lens = [150] * (len(chunks) - 1) + [seq_len % 150]
        chunks[-2] = torch.cat((chunks[-2], chunks[-1]), dim=1)
        lens[-2] += lens[-1]
        del chunks[-1], lens[-1]
        parts = []
        for a, n in zip(chunks, lens):
            p = a2p.infer(a, n, torch.LongTensor([id_seed])).squeeze().detach().cpu().numpy()
            p[:, :3] *= 0.5
            parts.append(p)
        pose_seq = pose_util.smooth_pose_seq(np.concatenate(parts, 0), 7)
    verts = pose_util.project_points(pred, trans_mat, pose_seq, [height, width])
    return [vis.draw_landmarks((width, height), v, normed=False) for v in verts], pose_seq


def _inserted_edges(draw_util, forehead_edge):
    """How many (edge, colour) insertions FaceMeshVisualizer.__init__ makes: the lists it defines (read with ast) plus
    the mediapipe sets it iterates. Equal to the dict's size iff no edge is in two groups."""
    import ast
    import mediapipe as mp
    tree = ast.parse(inspect.getsource(draw_util))
    lists = {n.targets[0].id: ast.literal_eval(n.value) for n in ast.walk(tree)
             if isinstance(n, ast.Assign) and isinstance(n.targets[0], ast.Name) and n.targets[0].id.startswith("FACEMESH_")}
    fm = mp.solutions.face_mesh
    oval = fm.FACEMESH_FACE_OVAL if forehead_edge else lists["FACEMESH_CUSTOM_FACE_OVAL"]
    sets = (fm.FACEMESH_LEFT_EYE, fm.FACEMESH_LEFT_EYEBROW, fm.FACEMESH_RIGHT_EYE, fm.FACEMESH_RIGHT_EYEBROW)
    lips = [v for k, v in lists.items() if k.startswith("FACEMESH_LIPS_")]
    assert len(lips) == 8
    return len(oval) + sum(len(s) for s in sets) + sum(len(v) for v in lips)


def make_golden():
    import cv2
    from oracle import mediapipe_import
    mediapipe_import.activate()
    from src.utils import draw_util, pose_util
    t0 = time.time()
    G = dict(case="pose_maps", seeds=dict(SEEDS), e2e=dict(E2E), frames=FRAMES, cv2_version=cv2.__version__,
             numpy_version=np.__version__, generator="reference src/utils/draw_util.py + pose_util.py, CPU")

    # edge / colour table
    for fe in (False, True):
        vis = draw_util.FaceMeshVisualizer(forehead_edge=fe)
        spec = [(tuple(int(v) for v in e), tuple(int(c) for c in d.color)) for e, d in vis.face_connection_spec.items()]
        assert _inserted_edges(draw_util, fe) == len(spec), "an edge sits in two groups"
        G[f"spec_forehead_{fe}"] = spec
    sig = inspect.signature
    G["surface"] = {"__init__": str(sig(draw_util.FaceMeshVisualizer.__init__)),
                    "draw_landmarks": str(sig(draw_util.FaceMeshVisualizer.draw_landmarks))}

    # cv2.line coverage of random segments
    segs = segments()
    cropped = []
    for x0, y0, x1, y1 in segs:
        img = np.zeros((512, 512, 3), np.uint8)
        cv2.line(img, (int(x0), int(y0)), (int(x1), int(y1)), (255, 255, 255), thickness=2)
        m = img[..., 0] > 0
        ys, xs = np.nonzero(m)
        cropped.append((m[ys.min():ys.max() + 1, xs.min():xs.max() + 1], (int(ys.min()), int(xs.min()))))
    box, offs, bits = pack_masks(cropped)
    G["segments"] = dict(seg=torch.from_numpy(segs), box=box, offs=offs, bits=bits)

    # smoothing
    G["smooth"] = {k: torch.from_numpy(pose_util.smooth_pose_seq(x, w)) for k, (x, w) in smoothing_inputs().items()}

    # projection and pose maps at 512 x 512
    lmks3d, trans = face_cloud()
    pts, poses = face_frames(), head_poses()
    proj = pose_util.project_points(pts, trans, poses, [512, 512])
    proj_t = pose_util.project_points_with_trans(pts[:TRANS_FRAMES].astype(np.float32), frame_matrices(TRANS_FRAMES),
                                                 [512, 512])
    G["project_points"] = torch.from_numpy(proj)
    G["project_points_with_trans"] = torch.from_numpy(proj_t)
    vis = draw_util.FaceMeshVisualizer(forehead_edge=False)
    maps = [vis.draw_landmarks((512, 512), v, normed=False) for v in proj]
    assert any(not ((v >= 0) & (v < 512)).all() for v in proj), "no landmark leaves the canvas"
    assert all(m.any() for m in maps[:2]), "empty pose maps"
    G["maps_512"] = [png(m) for m in maps]
    vis_fe = draw_util.FaceMeshVisualizer(forehead_edge=True)
    G["maps_512_forehead"] = [png(vis_fe.draw_landmarks((512, 512), v, normed=False)) for v in proj[:4]]
    lm = normed_landmarks()
    G["normed_pose"] = png(vis.draw_landmarks((512, 512), lm, normed=True))

    # other sizes: image_size = (W, H), projected for image_shape = [H, W]
    for W, H in ((768, 768), (384, 640)):
        kp = pose_util.project_points(pts[:SIZED_FRAMES], trans, poses[:SIZED_FRAMES], [H, W])
        G[f"kp_{W}x{H}"] = torch.from_numpy(kp)
        G[f"maps_{W}x{H}"] = [png(vis.draw_landmarks((W, H), v, normed=False)) for v in kp]

    # end to end: audio -> pose maps
    audio = e2e_audio()
    pose_temp = np.load(POSE_TEMP)
    for branch, temp in (("template", pose_temp), ("chunked", None)):
        frames, pose_seq = reference_audio_to_pose_maps(vis, pose_util, StandInMesh(), StandInPose(), audio,
                                                        E2E["seq_len"], lmks3d, trans, E2E["width"], E2E["height"],
                                                        E2E["id_seed"], temp)
        assert len(frames) == E2E["seq_len"] and frames[0].shape == (E2E["height"], E2E["width"], 3)
        G[f"e2e_{branch}_digests"] = frame_digests(frames)
        if temp is None:
            G[f"e2e_{branch}_pose_seq"] = torch.from_numpy(pose_seq)
        G[f"e2e_{branch}_png"] = png(frames[E2E["seq_len"] // 2])
    torch.save(G, GOLDEN)
    print(f"pose_maps: {os.path.getsize(GOLDEN)} bytes in {time.time() - t0:.1f}s, {len(segs)} segments")


if __name__ == "__main__":
    make_golden()
