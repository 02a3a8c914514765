"""Face-mesh pose maps without a GPU: the product's edge / colour table, the written specification of cv2's thick line and
INTER_LINEAR resize (oracle/cv2_line.py) against the reference's stored output, the drop-in surface and the errors."""
import inspect
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from pose_golden import GOLDEN, normed_landmarks, unpack_mask  # noqa: E402


@pytest.fixture(scope="module")
def golden():
    return torch.load(GOLDEN, weights_only=False)


def decode_png(t: torch.Tensor) -> np.ndarray:
    """The stored BGR frame (PNG keeps it as RGB channel order swapped)."""
    import io
    from PIL import Image
    return np.array(Image.open(io.BytesIO(t.numpy().tobytes())))[..., ::-1].copy()


def _runs(spec):
    """Ordered (edge, colour) list -> [(colour, set of edges)] per consecutive colour group."""
    out = []
    for edge, colour in spec:
        if not out or out[-1][0] != tuple(colour):
            out.append((tuple(colour), set()))
        out[-1][1].add(tuple(edge))
    return out


@pytest.mark.parametrize("forehead_edge", [False, True])
def test_edge_and_colour_table_equals_the_reference(golden, forehead_edge):
    from aniportrait_b200.utils.draw_util import connection_groups
    want = _runs(golden[f"spec_forehead_{forehead_edge}"])
    got = [(tuple(c), set(edges)) for edges, c in connection_groups(forehead_edge)]
    assert got == want
    assert sum(len(e) for e, _ in connection_groups(forehead_edge)) == len(golden[f"spec_forehead_{forehead_edge}"])


def test_line_restatement_reproduces_every_stored_cv2_segment(golden):
    from oracle.cv2_line import thick_line_mask
    S = golden["segments"]
    bad = []
    for i, (x0, y0, x1, y1) in enumerate(S["seg"].tolist()):
        if not np.array_equal(thick_line_mask((512, 512), x0, y0, x1, y1), unpack_mask(S["box"], S["offs"], S["bits"], i)):
            bad.append((x0, y0, x1, y1))
    assert len(S["seg"]) >= 4000 and not bad, f"{len(bad)} segments differ, e.g. {bad[:5]}"


def test_pose_map_restatement_reproduces_the_reference_maps(golden):
    """Landmark normalisation and validity, group overwrite order and the resize, at every stored size."""
    from aniportrait_b200.utils.draw_util import connection_groups
    from oracle.cv2_line import face_mesh_map
    groups = connection_groups(False)
    cases = [(golden["project_points"][i].numpy(), 512, 512, golden["maps_512"][i]) for i in (0, 3, 5)]
    for W, H in ((768, 768), (384, 640)):
        cases += [(kp.numpy(), W, H, m) for kp, m in zip(golden[f"kp_{W}x{H}"], golden[f"maps_{W}x{H}"])]
    for kp, W, H, want in cases:
        assert np.array_equal(face_mesh_map(kp, groups, W, H), decode_png(want)), (W, H)
    got = face_mesh_map(normed_landmarks(), groups, 512, 512, normed=True)
    assert np.array_equal(got, decode_png(golden["normed_pose"]))


def test_dropin_visualizer_signatures_match_the_reference(golden):
    from aniportrait_b200.utils.draw_util import FaceMeshVisualizer
    assert str(inspect.signature(FaceMeshVisualizer.__init__)) == golden["surface"]["__init__"]
    assert str(inspect.signature(FaceMeshVisualizer.draw_landmarks)) == golden["surface"]["draw_landmarks"]


def test_dropin_draw_util_does_not_import_mediapipe():
    import subprocess
    code = ("import sys; from src.utils.draw_util import FaceMeshVisualizer as F; "
            "from aniportrait_b200.utils.draw_util import FaceMeshVisualizer as G; "
            "assert F is G and 'mediapipe' not in sys.modules")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "dropin"), ROOT]))
    subprocess.run([sys.executable, "-c", code], check=True, env=env, cwd=ROOT)


def test_pose_ops_refuse_cpu_tensors():
    from aniportrait_b200 import ops
    from aniportrait_b200._lib import ApError
    from aniportrait_b200.utils import draw_util, pose_util
    with pytest.raises(ApError):
        pose_util.smooth_pose_seq(torch.zeros(8, 6), 7)
    with pytest.raises(ApError):
        pose_util.project_points(torch.zeros(2, 468, 3), torch.eye(4), torch.zeros(2, 6), [512, 512])
    with pytest.raises(ApError):
        pose_util.project_points_with_trans(torch.zeros(2, 468, 3), torch.eye(4).repeat(2, 1, 1), [512, 512])
    with pytest.raises(ApError):
        ops.facemesh_raster(torch.zeros(1, 468, 2), torch.zeros(1, 3, dtype=torch.int32),
                            torch.zeros(1, 3, dtype=torch.uint8), 512, 512)
    with pytest.raises(ApError):
        draw_util.FaceMeshVisualizer().draw_landmarks_batch((512, 512), torch.zeros(1, 468, 2))


class _CudaLooking(torch.Tensor):
    """A host tensor that reports is_cuda: reaches the pipeline's shape check without a device."""

    @property
    def is_cuda(self):
        return True


def test_pipeline_rejects_a_cuda_uint8_pose_tensor_of_the_wrong_size():
    from aniportrait_b200.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline
    pipe = object.__new__(Pose2VideoPipeline)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    for shape in ((4, 64, 48, 3), (4, 48, 64, 3), (4, 3, 64, 64), (64, 64, 3)):
        t = torch.zeros(shape, dtype=torch.uint8)
        t = t.to(dev) if dev == "cuda" else t.as_subclass(_CudaLooking)
        with pytest.raises(ValueError):
            pipe._pose_maps_to_tensor(t, 64, 64, torch.device(dev))
