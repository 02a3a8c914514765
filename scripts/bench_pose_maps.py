"""Pose-map stage of audio2vid: head-pose smoothing, landmark projection and face-mesh rendering of a 10 s clip.

    python scripts/bench_pose_maps.py [--frames 300] [--iters 20]

Device arm: ap_pose.cu (smooth_pose_seq, project_points, FaceMeshVisualizer.draw_landmarks_batch) from device tensors,
timed with CUDA events after warm-up. Host arm: a PORT of the reference's host path (oracle/pose_np.py projection and
smoothing, oracle/mediapipe_shim drawing through cv2.line per edge, cv2.resize), the reference itself not being available
where this runs; it stops before the maps are copied to the GPU. The inputs are the seeded face of tests/pose_golden.py.
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001
        return [torch.cuda.get_device_name(0), f"unknown ({e})", "unknown"]


def host_arm(pts, trans, poses, W, H):
    from oracle import pose_np
    from oracle import mediapipe_import
    mediapipe_import.activate_shim()
    import cv2
    from mediapipe.framework.formats import landmark_pb2
    from mediapipe.solutions import drawing_utils
    from mediapipe.solutions.drawing_styles import DrawingSpec
    from aniportrait_b200.utils.draw_util import connection_groups
    spec = {e: DrawingSpec(color=c, thickness=2, circle_radius=1) for edges, c in connection_groups(False) for e in edges}
    t0 = time.perf_counter()
    verts = pose_np.project_points(pts, trans, pose_np.smooth_pose_seq(poses, 7), [H, W])
    maps = []
    for v in verts:
        img = np.zeros((512, 512, 3), np.uint8)
        lms = landmark_pb2.NormalizedLandmarkList()
        for x, y in v:
            lm = lms.landmark.add()
            lm.x, lm.y, lm.z = x / W, y / H, 1.0
        drawing_utils.draw_landmarks(image=img, landmark_list=lms, connections=spec.keys(), landmark_drawing_spec=None,
                                     connection_drawing_spec=spec)
        maps.append(cv2.resize(img, (W, H)))
    return time.perf_counter() - t0, np.stack(maps)


def device_arm(pts, trans, poses, W, H, iters, vis):
    from aniportrait_b200.utils.pose_util import project_points, smooth_pose_seq

    def run():
        kp = project_points(pts, trans, smooth_pose_seq(poses, 7), [H, W])
        return vis.draw_landmarks_batch((W, H), kp)

    for _ in range(3):
        run()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = run()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pose_maps needs a CUDA device")
    import pose_golden as PG
    from aniportrait_b200.utils.draw_util import FaceMeshVisualizer
    L = args.frames
    _, trans = PG.face_cloud()
    pts, poses = PG.face_frames(L), PG.head_poses(L)
    dev = torch.device("cuda:0")
    vis = FaceMeshVisualizer(forehead_edge=False)
    name, power, clock = gpu_info()
    result = dict(bench="pose_maps", frames=L, gpu=name, power_limit=power, max_sm_clock=clock, sizes={})
    for W, H in ((512, 512), (384, 640)):
        med, best, out = device_arm(torch.from_numpy(pts).to(dev), torch.from_numpy(trans).to(dev),
                                    torch.from_numpy(poses).to(dev), W, H, args.iters, vis)
        host_s, host_maps = host_arm(pts, trans, poses, W, H)
        same = int((out.cpu().numpy() != host_maps).sum())
        result["sizes"][f"{W}x{H}"] = dict(
            device_ms_per_frame=med / L, device_ms_per_frame_best=best / L, device_ms_total_median=med,
            host_port_ms_per_frame=host_s * 1e3 / L, host_port_threads=1,
            h2d_bytes_avoided=L * H * W * 3, bytes_differing_from_host_port=same)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
