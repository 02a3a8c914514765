"""Audio front-end on the B200: each new kernel against fp32 torch on the same fp16 inputs, the whole wav2vec2 encoder,
Audio2MeshModel.infer and a KV-cached Audio2PoseModel chunk against the reference's outputs (tests/golden/audio_front_end.pt,
seeded real-geometry weights), run-to-run bit identity, and a kernel census of the encoder + Audio2Mesh call."""
import os
import sys
import tempfile

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import rel_l2  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, "tests", "golden", "audio_front_end.pt")
TOL_OP = 2e-3
TOL_MODEL = 1e-2


def _h(t, dev):
    return t.to(dev, torch.float16)


# ----------------------------------------------------------------------------------------------------------- single ops
@pytest.mark.parametrize("samples", [16000, 52817])
def test_wav_conv0_groupnorm_gelu(cuda_dev, samples):
    from aniportrait_b200 import ops
    g = torch.Generator().manual_seed(samples)
    wav = torch.randn(samples, generator=g)
    w = torch.randn(512, 10, generator=g) / 10 ** 0.5
    gamma, beta = 1 + 0.1 * torch.randn(512, generator=g), 0.1 * torch.randn(512, generator=g)
    got = ops.wav_conv0_gn_gelu(wav.to(cuda_dev), w.to(cuda_dev), gamma.to(cuda_dev), beta.to(cuda_dev))
    y = F.conv1d(wav.double().view(1, 1, -1), w.double().view(512, 1, 10), stride=5)
    want = F.gelu(F.group_norm(y, 512, gamma.double(), beta.double(), eps=1e-5))[0].t()
    assert got.shape == want.shape == ((samples - 10) // 5 + 1, 512)
    assert rel_l2(got, want) < TOL_OP


@pytest.mark.parametrize("M,N,K", [(37, 512, 1024), (150, 3072, 768), (300, 3072, 768), (499, 512, 1536),
                                   (1000, 256, 192)])
def test_gemm_gelu_epilogue(cuda_dev, M, N, K):
    from aniportrait_b200 import ops
    g = torch.Generator().manual_seed(M * N + K)
    a, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5
    b = 0.5 * torch.randn(N, generator=g)
    a16, w16 = _h(a, cuda_dev), _h(w, cuda_dev)
    got = ops.gemm(a16, w16, b.to(cuda_dev), gelu=True)
    want = F.gelu(a16.float() @ w16.float().t() + b.to(cuda_dev))
    assert rel_l2(got, want) < TOL_OP
    got_nb = ops.gemm(a16, w16, gelu=True)
    assert rel_l2(got_nb, F.gelu(a16.float() @ w16.float().t())) < TOL_OP


@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("t_in", [7, 38, 77, 155, 3999])
def test_strided_view_conv_layers(cuda_dev, k, t_in):
    """Feature-extractor layers 1-6 as GEMMs over strided views of the channels-last input, at odd and even lengths; the
    input lives at the END of a larger allocation guarded by a NaN tail, so a read past frame t_in - 1 would show."""
    from aniportrait_b200 import ops
    g = torch.Generator().manual_seed(t_in * 10 + k)
    x = torch.randn(t_in, 512, generator=g)
    w = torch.randn(512, 512, k, generator=g) / (512 * k) ** 0.5
    buf = torch.full((t_in + 64, 512), float("nan"), dtype=torch.float16, device=cuda_dev)
    buf[:t_in] = _h(x, cuda_dev)
    xv = buf[:t_in]
    got = ops.conv1d_s2_gelu(xv, ops.pack_conv1d_taps(w.to(cuda_dev)), k)
    want = F.gelu(F.conv1d(xv.float().t().unsqueeze(0), w.to(cuda_dev).half().float(), stride=2))[0].t()
    assert got.shape == want.shape == ((t_in - k) // 2 + 1, 512)
    assert torch.isfinite(got.float()).all()
    assert rel_l2(got, want) < TOL_OP


@pytest.mark.parametrize("T", [37, 150, 300, 499])
def test_positional_conv(cuda_dev, T):
    from aniportrait_b200 import ops
    g = torch.Generator().manual_seed(T)
    x = torch.randn(T, 768, generator=g)
    w = torch.randn(768, 48, 128, generator=g) / (48 * 128) ** 0.5
    b = 0.1 * torch.randn(768, generator=g)
    x16 = _h(x, cuda_dev)
    got = ops.pos_conv_gelu(x16, ops.pack_pos_conv_weight(w.to(cuda_dev)), b.to(cuda_dev))
    xf = x16.float().t().unsqueeze(0)
    conv = F.conv1d(xf, w.to(cuda_dev).half().float(), b.to(cuda_dev), padding=64, groups=16)[..., :-1]
    want = (xf + F.gelu(conv))[0].t()
    assert rel_l2(got, want) < TOL_OP


@pytest.mark.parametrize("t_in,t_out", [(149, 150), (150, 150), (299, 150), (249, 100), (49, 1), (1, 5), (300, 599)])
def test_time_interpolation(cuda_dev, t_in, t_out):
    from aniportrait_b200 import ops
    x16 = _h(torch.randn(t_in, 512, generator=torch.Generator().manual_seed(t_in)), cuda_dev)
    got = ops.interp_linear_time(x16, t_out)
    want = F.interpolate(x16.float().t().unsqueeze(0), size=t_out, mode="linear", align_corners=True)[0].t()
    assert got.shape == (t_out, 512)
    assert rel_l2(got, want) < TOL_OP


@pytest.mark.parametrize("T", [37, 100, 150, 300, 499])
def test_attention_ragged_single_frame(cuda_dev, T):
    from aniportrait_b200 import ops
    g = torch.Generator().manual_seed(T)
    qkv = _h(torch.randn(T, 3 * 768, generator=g), cuda_dev)
    got = ops.attention(qkv[:, :768], qkv[:, 768:1536], qkv[:, 1536:], 1, T, 12, 64, 64, scale=0.125)
    q, k, v = (qkv[:, i * 768:(i + 1) * 768].float().view(T, 12, 64).transpose(0, 1) for i in range(3))
    want = torch.softmax(q @ k.transpose(1, 2) * 0.125, -1) @ v
    assert rel_l2(got, want.transpose(0, 1).reshape(T, 768)) < TOL_OP


def test_mean_of_states(cuda_dev):
    from aniportrait_b200 import ops
    x = _h(torch.randn(13, 150, 768, generator=torch.Generator().manual_seed(1)), cuda_dev)
    m32, m16 = ops.mean_f16(x, out_f32=True, out_f16=True)
    s = sum(x.float().unbind(0))                       # fp32 sums in the reference's order
    # the kernel divides; torch's CUDA division by a scalar multiplies by the reciprocal: the two differ by at most an ulp
    assert ((m32 - s / 13).abs() <= 2 ** -22 * (s / 13).abs()).all()
    assert torch.equal(m16, m32.half())
    assert torch.equal(ops.mean_f16(x[:1]), x[0].float())


# ----------------------------------------------------------------------------------------------------------- models
def _gold():
    return torch.load(GOLDEN, weights_only=False)


@pytest.fixture(scope="module")
def mesh_model(cuda_dev):
    from aniportrait_b200.audio_models import Audio2MeshModel
    from audio_golden import AUDIO_MESH, audio_encoder_config_dir, audio_mesh_state
    with tempfile.TemporaryDirectory() as d:
        audio_encoder_config_dir(d)
        m = Audio2MeshModel(dict(AUDIO_MESH, model_path=d, from_pretrained=False))
    m.load_state_dict(audio_mesh_state(m))
    return m.to(cuda_dev).eval()


def test_encoder_and_mesh_head_match_reference(cuda_dev, mesh_model):
    from audio_golden import AUDIO_CLIPS, AUDIO_ROW_STRIDE, AUDIO_SEEDS, audio_clip
    G = _gold()
    enc = mesh_model.audio_encoder
    report = []
    for clip, (samples, T) in AUDIO_CLIPS.items():
        audio = audio_clip(samples, AUDIO_SEEDS[clip]).to(cuda_dev)
        out = enc(audio, seq_len=T, output_hidden_states=True)
        assert out.last_hidden_state.dtype == torch.float32 and out.last_hidden_state.shape == (1, T, 768)
        assert len(out.hidden_states) == 13 and out.attentions is None
        e_last = rel_l2(out.last_hidden_state[0, ::AUDIO_ROW_STRIDE], G[f"{clip}_last"])
        mean = sum(out.hidden_states) / len(out.hidden_states)
        e_mean = rel_l2(mean[0, ::AUDIO_ROW_STRIDE], G[f"{clip}_mean"])
        norms = torch.stack([s[0].norm() for s in out.hidden_states]).cpu()
        e_norms = ((norms - G[f"{clip}_state_norms"]).abs() / G[f"{clip}_state_norms"]).max().item()
        report.append(f"{clip}: last {e_last:.2e} mean13 {e_mean:.2e} state norms {e_norms:.2e}")
        assert e_last < TOL_MODEL and e_mean < TOL_MODEL and e_norms < TOL_MODEL, report[-1]
    samples, T = AUDIO_CLIPS["audio_5s"]
    audio = audio_clip(samples, AUDIO_SEEDS["audio_5s"]).to(cuda_dev)
    pred = mesh_model.infer(audio, T)
    assert pred.shape == (1, T, 1404) and pred.dtype == torch.float32
    e_mesh = rel_l2(pred[0, ::AUDIO_ROW_STRIDE], G["mesh_infer"])
    report.append(f"Audio2MeshModel.infer: {e_mesh:.2e}")
    print("audio front-end vs reference (rel-L2): " + "; ".join(report))
    assert e_mesh < TOL_MODEL
    # only_last_fetures=False: the 13-state mean path of infer
    mesh_model._only_last_features = False
    try:
        pred_mean = mesh_model.infer(audio, T)
    finally:
        mesh_model._only_last_features = True
    out = enc(audio, seq_len=T, output_hidden_states=True)
    mean = (sum(out.hidden_states) / len(out.hidden_states))[0]
    want = mesh_model.out_fn(mesh_model.in_fn(mean.half().float()))
    assert rel_l2(pred_mean[0], want) < TOL_OP


def test_two_calls_bit_identical(cuda_dev, mesh_model):
    from audio_golden import AUDIO_SEEDS, audio_clip
    audio = audio_clip(52817, AUDIO_SEEDS["audio_ragged"]).to(cuda_dev)
    a = mesh_model.infer(audio, 100)
    b = mesh_model.infer(audio, 100)
    assert torch.equal(a, b)
    s1 = mesh_model.audio_encoder(audio, 100, output_hidden_states=True)
    s2 = mesh_model.audio_encoder(audio, 100, output_hidden_states=True)
    assert all(torch.equal(x, y) for x, y in zip(s1.hidden_states, s2.hidden_states))


def test_encoder_and_mesh_launch_only_library_kernels(cuda_dev, mesh_model):
    from torch.profiler import ProfilerActivity, profile
    from audio_golden import AUDIO_SEEDS, audio_clip
    audio = audio_clip(80000, AUDIO_SEEDS["audio_5s"]).to(cuda_dev)
    mesh_model.infer(audio, 150)
    mesh_model.audio_encoder(audio, 150, output_hidden_states=True)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        mesh_model.audio_encoder(audio, 150, output_hidden_states=True)
        mesh_model.infer(audio, 150)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA
             or getattr(e, "self_device_time_total", 0) > 0]
    names = [n for n in names if "memcpy" not in n.lower() and "memset" not in n.lower()]
    foreign = [n for n in names if "ap::" not in n]
    assert names and not foreign, f"non-library kernels on the audio path: {foreign}"


def test_errors_on_device(cuda_dev, mesh_model):
    enc = mesh_model.audio_encoder
    with pytest.raises(ValueError, match="receptive field"):
        enc(torch.randn(1, 399, device=cuda_dev), 5)
    with pytest.raises(ValueError, match="one clip"):
        enc(torch.randn(2, 16000, device=cuda_dev), 50)
    with pytest.raises(NotImplementedError):
        enc(torch.randn(1, 16000, device=cuda_dev), 50, attention_mask=torch.ones(1, 16000, device=cuda_dev))
    out = enc(torch.randn(1, 400, device=cuda_dev), 1)      # the shortest clip the conv stack accepts
    assert out.last_hidden_state.shape == (1, 1, 768) and torch.isfinite(out.last_hidden_state).all()


class _PoseModelWithKernelEncoder(torch.nn.Module):
    """The submodules of the reference's Audio2PoseModel (src/audio_models/pose_model.py:56-89) that infer reads, built
    from torch layers with the reference's hyper-parameters; the audio encoder is the kernel Wav2Vec2Model, as the drop-in
    gives the reference class."""

    def __init__(self, cfg_dir, biased_mask, E=512):
        super().__init__()
        from transformers import Wav2Vec2Config
        from aniportrait_b200.audio_models import Wav2Vec2Model
        from aniportrait_b200.synthetic import _sinusoid_pe
        self.out_dim = 6
        self._only_last_features = True
        self.audio_encoder = Wav2Vec2Model(Wav2Vec2Config.from_pretrained(cfg_dir))
        self.pose_map = torch.nn.Linear(6, E)
        self.in_fn = torch.nn.Linear(768, E)
        self.PPE = torch.nn.Module()
        self.PPE.register_buffer("pe", _sinusoid_pe(600, E))
        self.biased_mask = biased_mask
        layer = torch.nn.TransformerDecoderLayer(d_model=E, nhead=8, dim_feedforward=2 * E, batch_first=True)
        self.transformer_decoder = torch.nn.TransformerDecoder(layer, num_layers=8)
        self.pose_map_r = torch.nn.Linear(E, 6)
        self.id_embed = torch.nn.Embedding(100, E)


def test_kv_cached_pose_chunk_with_kernel_encoder(cuda_dev):
    from aniportrait_b200.audio_models import kv_cached_infer
    from audio_golden import AUDIO_CLIPS, AUDIO_ID_SEED, AUDIO_SEEDS, audio_clip, audio_encoder_config_dir, \
        audio_pose_state, mask_from_last_row
    G = _gold()
    samples, T = AUDIO_CLIPS["audio_5s"]
    with tempfile.TemporaryDirectory() as d:
        audio_encoder_config_dir(d)
        m = _PoseModelWithKernelEncoder(d, mask_from_last_row(G["pose_mask_last_row"]))
    m.load_state_dict(audio_pose_state(m))
    m = m.to(cuda_dev).eval()
    audio = audio_clip(samples, AUDIO_SEEDS["audio_5s"]).to(cuda_dev)
    got = kv_cached_infer(m, audio, T, id_seed=torch.tensor([AUDIO_ID_SEED], device=cuda_dev))
    err = rel_l2(got, G["pose_infer"])
    print(f"KV-cached Audio2PoseModel chunk (kernel encoder) vs reference: rel-L2 {err:.2e}")
    assert got.shape == (1, T, 6) and err < TOL_MODEL
