"""CPU-only tests (-m "not gpu"): C-ABI library loads and exports every declared symbol; host-side logic (scheduler,
window scheduler, image pre-processing, weight repacking, state-dict surface) against the oracle; world_size-2 gloo test
of the window-sharded denoising step."""
import os
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import functional as OF  # noqa: E402


def rel_l2(a, b):
    a, b = a.detach().float(), b.detach().float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def _reference_units():
    """Outputs of the unmodified reference at unit-test sizes (oracle/make_golden.py reference_units)."""
    return torch.load(os.path.join(ROOT, "tests", "golden", "reference_units.pt"))


def test_library_exports_every_declared_symbol():
    from aniportrait_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.lib()
    syms = _lib.declared_symbols()
    assert len(syms) >= 17
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/aniportrait_b200.h but not exported"
    assert lib.ap_version() == 200


def test_ops_refuse_cpu_tensors():
    from aniportrait_b200 import _lib, ops
    with pytest.raises(_lib.ApError):
        ops.gemm(torch.zeros(128, 64, dtype=torch.float16), torch.zeros(64, 64, dtype=torch.float16))


def test_product_forward_fails_loudly_without_gpu():
    from helpers import build_unet3d
    unet, _ = build_unet3d((64, 128, 256, 256), 1)
    with pytest.raises(Exception):
        unet(torch.zeros(1, 4, 2, 16, 16), 10, encoder_hidden_states=torch.zeros(1, 1, 768))


def test_scheduler_matches_oracle():
    from aniportrait_b200.pipelines.scheduler import DDIMScheduler
    s = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                      prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")
    o = OF.DDIM()
    for n in (10, 25, 50):
        s.set_timesteps(n)
        assert s.timesteps.tolist() == o.timesteps(n)
    s.set_timesteps(25)
    assert torch.allclose(s.alphas_cumprod, o.alphas_cumprod, rtol=0, atol=0)
    assert s.alphas_cumprod[-1].item() == 0.0   # zero terminal SNR
    g = torch.Generator().manual_seed(0)
    x, v = torch.randn(1, 4, 3, 8, 8, generator=g), torch.randn(1, 4, 3, 8, 8, generator=g)
    for t in (999, 519, 39):
        assert torch.allclose(s.step(v, t, x).prev_sample, o.step(v, t, x, 25), atol=1e-6)
    a_t, a_p = s.alpha_pair(39)
    assert a_p == 1.0 and 0 < a_t < 1


@pytest.mark.parametrize("n", [1, 4, 16, 17, 24, 40, 128])
def test_window_scheduler_matches_oracle(n):
    from aniportrait_b200.pipelines.context import uniform
    from aniportrait_b200.pipelines.sharding import plan_windows
    assert list(uniform(0, 25, n, 16, 1, 4)) == OF.context_windows(n, 16, 4)
    windows, inv = plan_windows(n, 25)
    assert inv.shape == (n,) and (inv > 0).all()
    if n == 128:
        assert len(windows) == 11 and windows[-1] == list(range(120, 128)) + list(range(0, 8))


def test_image_processor_paths():
    import PIL.Image
    from aniportrait_b200.pipelines.image_processor import VaeImageProcessor
    p = VaeImageProcessor(vae_scale_factor=8, do_convert_rgb=True, do_normalize=True)
    img = PIL.Image.fromarray(np.random.RandomState(0).randint(0, 256, (70, 90, 3), dtype=np.uint8))
    t = p.preprocess(img, height=64, width=64)
    assert t.shape == (1, 3, 64, 64) and -1.0 <= t.min() and t.max() <= 1.0
    arr = np.zeros((64, 64, 3), dtype=np.uint8)
    arr[10, 10] = 255
    t = p.preprocess(arr, height=64, width=64)   # numpy path: NOT divided by 255 (diffusers 0.24 behaviour)
    assert t.shape == (1, 3, 64, 64) and t.max().item() == 509.0 and t.min().item() == -1.0


def test_weight_repacking():
    from aniportrait_b200 import ops
    w = torch.randn(10, 4, 3, 3)
    wp = ops.pack_conv3x3_weight(w)
    assert wp.shape == (32, 9 * 64)
    v = wp.view(32, 3, 3, 64)
    assert torch.equal(v[:10, :, :, :4], w.permute(0, 2, 3, 1).half()) and v[10:].abs().sum() == 0
    wg, bg = ops.interleave_geglu(torch.arange(64 * 8).float().view(64, 8), torch.arange(64).float())
    assert bg[:16].tolist() == list(range(16)) and bg[16:32].tolist() == list(range(32, 48))
    wq = ops.pad_head_rows(torch.ones(8 * 40, 16), 8, 64)
    assert wq.shape == (512, 16) and wq.view(8, 64, 16)[:, 40:].abs().sum() == 0
    assert [ops.head_pad(d) for d in (8, 40, 80, 88, 160)] == [64, 64, 128, 128, 192]


def test_reference_attention_control_pairing():
    """update() pairs reader/writer blocks positionally after the stable width sort; clear() empties banks."""
    from helpers import build_unet2d, build_unet3d
    from aniportrait_b200.models import ReferenceAttentionControl
    u3, _ = build_unet3d((64, 128, 256, 256), 1)
    u2, _ = build_unet2d((64, 128, 256, 256), 2)
    w = ReferenceAttentionControl(u2, mode="write", do_classifier_free_guidance=True, fusion_blocks="full")
    r = ReferenceAttentionControl(u3, mode="read", do_classifier_free_guidance=True, fusion_blocks="full")
    wm, rm = w._modules(u2), r._modules(u3)
    assert len(wm) == len(rm) == 16
    assert [m.norm1.normalized_shape[0] for m in rm] == [256] * 6 + [128] * 5 + [64] * 5
    for i, m in enumerate(wm):
        m.bank.append(torch.full((2, 4, m.norm1.normalized_shape[0]), float(i)))
    r.update(w)
    for i, m in enumerate(rm):
        assert m.bank[0].dtype == torch.float16 and m.bank[0].flatten()[0].item() == float(i)
        assert m._ref_mode == "read" and m._ref_cfg
    r.clear()
    assert all(len(m.bank) == 0 for m in rm)


def _gloo_worker(rank, world, port, L, out_q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from aniportrait_b200.pipelines.sharding import accumulate, combine, plan_windows, windows_of_rank
    windows, inv = plan_windows(L, 25)
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(1, 4, L, 4, 4, generator=g)

    def fake_unet(x):   # deterministic stand-in for the UNet call of one window: [2, 4, F, h, w]
        return torch.stack([torch.sin(x[0] * 1.3), torch.cos(x[0] * 0.7)]) + x.mean(dim=2, keepdim=True)

    acc = torch.zeros(2, L, 4, 4, 4)
    for wd in windows_of_rank(windows, rank, world, True):
        pred = fake_unet(lat[:, :, wd])                                   # [2, 4, F, h, w]
        accumulate(acc, pred.permute(0, 2, 1, 3, 4), wd)                  # acc is [B, L, C, h, w]
    dist.all_reduce(acc)
    out = combine(acc, inv, 3.5)
    if rank == 0:
        out_q.put(out.numpy())      # by value: a tensor handle would die with this process
    dist.destroy_process_group()


def test_window_sharding_world2_gloo():
    """N>1 path on CPU: 2 ranks each process their windows; one sum all-reduce per step reproduces the single-process
    overlap-average + CFG result."""
    import torch.multiprocessing as mp
    from aniportrait_b200.pipelines.sharding import accumulate, combine, plan_windows
    L, world, port = 40, 2, 29533
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, L, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    windows, inv = plan_windows(L, 25)
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(1, 4, L, 4, 4, generator=g)
    acc = torch.zeros(2, L, 4, 4, 4)
    for wd in windows:
        x = lat[:, :, wd]
        pred = torch.stack([torch.sin(x[0] * 1.3), torch.cos(x[0] * 0.7)]) + x.mean(dim=2, keepdim=True)
        accumulate(acc, pred.permute(0, 2, 1, 3, 4), wd)
    ref = combine(acc, inv, 3.5)
    assert torch.allclose(torch.from_numpy(got), ref, atol=1e-5)


def test_plan_units_covers_every_window_branch_once_and_balances():
    """(window, CFG branch) work units (SURVEY.md §8e): every unit is assigned exactly once, every rank derives the same
    plan, and 11 windows on 8 ranks balance better than whole windows (2 windows = 4.4 cost units on the busiest rank)."""
    from aniportrait_b200.pipelines.sharding import plan_units
    for n_windows, world in [(11, 8), (2, 2), (5, 4), (3, 8), (1, 2)]:
        plan = plan_units(n_windows, True, world)
        assert plan == plan_units(n_windows, True, world) and len(plan) == world
        seen = []
        for units in plan:
            for k, br in units:
                seen += [(k, "uncond"), (k, "cond")] if br == "both" else [(k, br)]
        assert sorted(seen) == sorted([(k, b) for k in range(n_windows) for b in ("uncond", "cond")])
    cost = {"both": 2.2, "cond": 1.2, "uncond": 1.0}
    busiest = max(sum(cost[br] for _, br in units) for units in plan_units(11, True, 8))
    assert busiest <= 3.45 < 4.4
    # no CFG: whole windows round-robin
    assert plan_units(3, False, 2) == [[(0, "both"), (2, "both")], [(1, "both")]]


def test_ctypes_call_sites_match_the_header_prototypes():
    """ABI drift guard: every `lib().ap_*(...)` call in aniportrait_b200/ops.py passes exactly as many arguments as the
    prototype in include/aniportrait_b200.h declares (ctypes would not notice a missing / extra trailing argument)."""
    import ast
    import re
    header = open(os.path.join(ROOT, "include", "aniportrait_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(?:int|const char\*)\s+(ap_\w+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
    assert len(protos) >= 20
    tree = ast.parse(open(os.path.join(ROOT, "aniportrait_b200", "ops.py")).read())
    seen = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr.startswith("ap_"):
            seen[node.func.attr] = len(node.args)
    assert seen, "no C-ABI call sites found in ops.py"
    for name, n in seen.items():
        assert name in protos, f"{name} is called from ops.py but not declared in the header"
        assert n == protos[name], f"{name}: ops.py passes {n} arguments, the header declares {protos[name]}"


def test_short_pipelines_forward_to_the_shared_core_with_single_window_arguments():
    """pipeline_pose2vid / pipeline_pose2img are thin wrappers: the whole clip is ONE window (context_frames = L, no
    overlap), the CLIP input is not squashed, clips longer than the temporal PE table are rejected, and the image pipeline is
    a one-frame clip whose result is exposed as `.images`."""
    from unittest import mock
    from aniportrait_b200.pipelines import pipeline_pose2img, pipeline_pose2vid
    from aniportrait_b200.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline as Long
    calls = []

    def fake_call(self, *args, **kwargs):
        calls.append((args, kwargs))
        return "VIDEO" if kwargs.get("return_dict", args[12] if len(args) > 12 else True) else "RAW"

    with mock.patch.object(Long, "__call__", fake_call):
        short = pipeline_pose2vid.Pose2VideoPipeline.__new__(pipeline_pose2vid.Pose2VideoPipeline)
        out = short("ref", ["p"] * 20, "refpose", 512, 512, 20, 25, 3.5)
        args, kw = calls[-1]
        assert out == "VIDEO" and args[5] == 20
        assert kw["context_frames"] == 20 and kw["context_overlap"] == 0 and kw["clip_resize"] is False
        with pytest.raises(ValueError):
            short("ref", ["p"] * 40, "refpose", 512, 512, 40, 25, 3.5)
        img = pipeline_pose2img.Pose2ImagePipeline.__new__(pipeline_pose2img.Pose2ImagePipeline)
        res = img("ref", "pose", "refpose", 512, 512, 25, 3.5)
        args, kw = calls[-1]
        assert args[1] == ["pose"] and args[5] == 1 and kw["context_frames"] == 1
        assert isinstance(res, pipeline_pose2img.Pose2ImagePipelineOutput) and res.images == "RAW"


def test_window_scheduler_degenerate_overlap_fails_like_the_reference():
    """context_overlap == context_size * hop: the reference's range() raises ValueError (zero step); the rewritten loop must
    not spin forever. A larger overlap (negative step) yields no window at that level in both."""
    from aniportrait_b200.pipelines.context import uniform
    with pytest.raises(ValueError):
        list(uniform(0, 25, 40, 16, 1, 16))
    assert list(uniform(0, 25, 40, 16, 1, 20)) == []
    # what the reference's uniform() returned (or raised) for the same arguments
    ref = dict(_reference_units()["uniform"])
    assert ref[(0, 25, 40, 16, 1, 16)] == "ValueError"
    assert ref[(0, 25, 40, 16, 1, 20)] == []
    for args in [(0, 25, 24, 16, 2, 4), (3, 25, 50, 16, 3, 4), (0, 25, 128, 16, 1, 4)]:
        assert list(uniform(*args)) == ref[args]


def test_repeated_frame_in_a_window_counts_once():
    from aniportrait_b200.pipelines.sharding import accumulate, plan_windows
    windows, inv = plan_windows(24, 25, "uniform", 16, 2, 4)
    counts = torch.zeros(24)
    for wd in windows:
        for f in set(wd):
            counts[f] += 1
    assert torch.equal(inv, 1.0 / counts)
    wd = next(w for w in windows if len(set(w)) < len(w))
    acc = accumulate(torch.zeros(1, 24, 2), torch.ones(1, len(wd), 2), wd)
    assert acc.max().item() == 1.0


def test_checked_state_dict_loading():
    """from_pretrained must not silently leave weights at random init: legacy VAE attention names are remapped (diffusers
    _convert_deprecated_attention_blocks [dep]); anything missing / unknown raises unless whitelisted."""
    from aniportrait_b200.models.modeling import load_checked
    from aniportrait_b200.models.vae import AutoencoderKL
    vae = AutoencoderKL(block_out_channels=(32, 32, 64, 64))
    ren = {"to_q": "query", "to_k": "key", "to_v": "value", "to_out.0": "proj_attn"}

    def legacy_name(k):
        if ".attentions.0." in k:
            for new, old in ren.items():
                k = k.replace(f".{new}.", f".{old}.")
        return k
    legacy = {legacy_name(k): torch.randn_like(v) for k, v in vae.state_dict().items()}
    assert any(".query." in k for k in legacy)
    load_checked(vae, legacy)
    for k, v in vae.state_dict().items():
        assert torch.equal(v, legacy[legacy_name(k)])
    broken = dict(legacy)
    broken.pop("decoder.conv_in.weight")
    with pytest.raises(RuntimeError, match="missing"):
        load_checked(vae, broken)
    extra = dict(legacy, **{"decoder.bogus.weight": torch.zeros(1)})
    with pytest.raises(RuntimeError, match="unexpected"):
        load_checked(vae, extra)
    load_checked(vae, extra, allow_unexpected=("bogus",))


def test_pipeline_rejects_schedulers_the_fused_step_cannot_reproduce():
    from aniportrait_b200.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline
    from aniportrait_b200.pipelines.scheduler import DDIMScheduler

    class P(Pose2VideoPipeline):
        def __init__(self, scheduler):
            self.scheduler = scheduler
    assert P(DDIMScheduler(prediction_type="v_prediction", clip_sample=False))._scheduler_update_rule() == ("v_prediction", 0.0)
    assert P(DDIMScheduler())._scheduler_update_rule() == ("epsilon", 1.0)      # diffusers defaults: epsilon + clip_sample

    class Flow:
        config = dict(prediction_type="flow")
    with pytest.raises(NotImplementedError):
        P(Flow())._scheduler_update_rule()

    class NoAlphas:
        config = dict(prediction_type="epsilon")
    with pytest.raises(NotImplementedError):
        P(NoAlphas())._scheduler_update_rule()


def test_layernorm_folding_algebra():
    """Host side of the LayerNorm folding (aniportrait_b200/models/blocks.py::fold_layer_norm, FeedForward.folded, the motion
    module's positional-encoding bias table) evaluated with plain torch: rstd (x W'^T - mean colsum) + bias' == LN(x) W^T + b."""
    import torch.nn.functional as F
    from aniportrait_b200 import ops
    from aniportrait_b200.models.blocks import FeedForward, TemporalTransformer3DModel, fold_layer_norm
    g = torch.Generator().manual_seed(0)
    M, C, N = 50, 64, 96
    x = torch.randn(M, C, generator=g) + 0.4
    w, b = torch.randn(N, C, generator=g) * C ** -0.5, torch.randn(N, generator=g) * 0.1
    gamma, beta = 1 + 0.2 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    wg, bias = fold_layer_norm(w, b, gamma, beta)                       # [N, C + 8]
    assert wg.shape == (N, C + ops.LN_EXTRA_K)
    mean, var = x.mean(1, keepdim=True), x.var(1, unbiased=False, keepdim=True)
    rstd = (var + 1e-5).rsqrt()

    def a_ext(t, mean):      # what ap_layernorm_finalize_f16 appends: -mean split in two fp16 halves, (hi, lo, hi, 0 x 5)
        hi = (-mean).half()
        lo = (-mean - hi.float()).half()
        return torch.cat([t, hi.float(), lo.float(), hi.float(), torch.zeros(t.shape[0], 5)], 1)
    got = rstd * (a_ext(x, mean) @ wg.float().t()) + bias[None]
    ref = F.layer_norm(x, (C,), gamma, beta, 1e-5) @ w.t() + b
    assert rel_l2(got, ref) < 2e-3          # W' is rounded to fp16
    # GEGLU: the folded, interleaved projection pairs value / gate columns like the kernel's epilogue expects
    ff = FeedForward(C)
    w1, b1 = ff.folded(gamma, beta)
    acc = rstd * (a_ext(x, mean) @ w1.float().t()) + b1[None]                              # [M, 8C] interleaved 16 | 16
    a = acc.view(M, -1, 2, 16)
    got = (a[:, :, 0] * F.gelu(a[:, :, 1])).reshape(M, -1)
    h, gate = (F.layer_norm(x, (C,), gamma, beta, 1e-5) @ ff.net[0].proj.weight.t() + ff.net[0].proj.bias).chunk(2, -1)
    assert rel_l2(got, h * F.gelu(gate)) < 2e-3
    # motion module: LN(m) + pe[f] projected by Wqkv == folded GEMM + per-frame bias table
    mm = TemporalTransformer3DModel(C, heads=8, max_len=32, groups=32)
    for p in mm.parameters():
        torch.nn.init.normal_(p, std=0.3)
    pk = mm.packed()
    B, Fr, n_tok = 2, 5, 3
    m = torch.randn(B * Fr * n_tok, C, generator=g) + 0.7
    a0 = pk["attn"][0]
    tab = mm._pe_bias(pk, 0, B, Fr)                                                        # [B*F, 3C]
    mean, rstd = m.mean(1, keepdim=True), (m.var(1, unbiased=False, keepdim=True) + 1e-5).rsqrt()
    rows = torch.arange(B * Fr * n_tok) // n_tok
    got = rstd * (a_ext(m, mean) @ a0["wqkv_g"].float().t()) + tab[rows]
    frame = rows % Fr
    n = F.layer_norm(m, (C,), a0["g"], a0["b"], 1e-5) + a0["pe"][frame]
    assert rel_l2(got, n @ a0["wqkv"].float().t()) < 2e-3


def test_vae_quant_conv_folding_algebra():
    """AutoencoderKL: quant_conv folded into encoder.conv_out, post_quant_conv folded into decoder.conv_in over a
    constant-one channel (aniportrait_b200/models/vae.py) == the two-convolution chains, borders included."""
    import torch.nn.functional as F
    from aniportrait_b200.models.vae import AutoencoderKL
    vae = AutoencoderKL(block_out_channels=(64, 64, 64, 64))
    for p in vae.parameters():
        torch.nn.init.normal_(p, std=0.2)
    g = torch.Generator().manual_seed(1)
    # encoder tail
    pk = vae.encoder._packed(vae.quant_conv)
    wo, bo = pk["conv_out"]                                  # [32 (padded), 9 * 64] tap-major / channel-minor
    w_f = wo[:8].float().view(8, 3, 3, 64).permute(0, 3, 1, 2)
    x = torch.randn(2, 64, 6, 5, generator=g)
    ref = vae.quant_conv(vae.encoder.conv_out(x))
    got = F.conv2d(x, w_f, bo[:8], padding=1)
    assert rel_l2(got, ref) < 2e-3
    # decoder head
    pk = vae.decoder._packed(vae.post_quant_conv)
    wi, bi = pk["conv_in"]                                   # [64, 9 * 64]: channels 0..3 latent, 4 the ones channel
    w_f = wi.float().view(-1, 3, 3, 64).permute(0, 3, 1, 2)[:, :5]
    z = torch.randn(2, 4, 6, 5, generator=g)
    ref = vae.decoder.conv_in(vae.post_quant_conv(z))
    z1 = torch.cat([z, torch.ones(2, 1, 6, 5)], 1)
    got = F.conv2d(z1, w_f, bi[:64], padding=1)
    assert rel_l2(got, ref) < 2e-3


def test_unit_groups_cover_every_unit_once_uncond_first():
    """Sharded mode: a rank's (window, branch) units are batched into UNet calls of <= group_units elements, unconditional
    windows first inside every group (the attention kernel's bank rule: frames before first_bank_frame skip the bank)."""
    from aniportrait_b200.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline, _Session
    from aniportrait_b200.pipelines.sharding import plan_units

    class P(Pose2VideoPipeline):
        def __init__(self):
            self.group_units = 4
    for world in (2, 4, 8):
        for rank, mine in enumerate(plan_units(11, True, world)):
            ids = sorted({k for k, _ in mine})
            units = [(ids.index(k), br) for k, br in mine]
            S = _Session()
            S.win_idx = [torch.arange(16, dtype=torch.int32) + 12 * k for k in ids]
            execs = P()._plan_groups(S, units)
            assert execs == [("group", i) for i in range(len(S.groups))]
            seen = []
            for G in S.groups:
                assert 1 <= len(G["elems"]) <= 4
                bs = [b for _, b in G["elems"]]
                assert bs == sorted(bs) and G["n_uncond"] == bs.count(0)
                assert G["idx_all"].numel() == 16 * len(G["elems"])
                for e, (k, b) in enumerate(G["elems"]):
                    assert torch.equal(G["idx_all"][16 * e:16 * e + 16], S.win_idx[k])
                seen += G["elems"]
            want = []
            for k, br in units:
                want += [(k, 0), (k, 1)] if br == "both" else [(k, 0 if br == "uncond" else 1)]
            assert sorted(seen) == sorted(want)


def _gloo_bank_worker(rank, world, port, out_q):
    """Bank exchange protocol of the sharded sessions on CPU tensors: shape handshake (once per session), rank 0 packs its
    banks into ONE flat buffer, one broadcast, every rank's writer blocks end up with views of it."""
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from aniportrait_b200.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline, _Session

    class Blk:
        def __init__(self):
            self.bank = []

    class Writer:
        def __init__(self, mods):
            self.unet, self.mods = None, mods

        def _modules(self, unet):
            return self.mods

    class P(Pose2VideoPipeline):
        def __init__(self):
            pass
    shapes = [(2, 16, 256), (2, 16, 256), (2, 64, 128), (2, 256, 64)]
    mods = [Blk() for _ in shapes]
    if rank == 0:
        g = torch.Generator().manual_seed(3)
        for m, shp in zip(mods, shapes):
            m.bank = [torch.randn(*shp, generator=g).to(torch.float16)]
    S = _Session()
    S.lat = torch.zeros(1)
    S.writer = Writer(mods)
    pipe = P()
    S.bank_shapes = pipe._bank_layout(S)
    assert S.bank_shapes == shapes
    S.bank_flat = torch.empty(sum(a * b * c for a, b, c in shapes), dtype=torch.float16)
    if rank == 0:
        pipe._pack_banks(S)
    dist.broadcast(S.bank_flat, 0)
    pipe._unpack_banks(S)
    g = torch.Generator().manual_seed(3)
    same = all(torch.equal(m.bank[0], torch.randn(*shp, generator=g).to(torch.float16)) for m, shp in zip(mods, shapes))
    lo, hi = S.bank_flat.data_ptr(), S.bank_flat.data_ptr() + S.bank_flat.numel() * 2
    views = all(lo <= m.bank[0].data_ptr() < hi for m in mods)
    out_q.put((rank, bool(same), bool(views)))       # plain Python values: no tensor handles cross the process boundary
    dist.barrier()
    dist.destroy_process_group()


def test_bank_exchange_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_bank_worker, args=(r, 2, 29547, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(2):
        r = q.get(timeout=120)
        got[r[0]] = r
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0][1] and got[1][1], "every rank must hold rank 0's banks after the single broadcast"
    assert got[0][2] and got[1][2], "the banks must be views of the flat broadcast buffer"


class _StandInFilm(torch.nn.Module):
    """Stand-in for the FILM TorchScript file (absent): same call layout (x0, x1 [n, c, h, w] fp16, dt [n, 1] or [1, 1]),
    elementwise + shifts only, so that a frame's value cannot depend on the batch it is computed in; leaves [0, 1] on purpose
    (the wrapper clamps)."""

    def __init__(self):
        super().__init__()
        self.anchor = torch.nn.Parameter(torch.zeros(1))       # tells the wrapper which device the network lives on

    def forward(self, x0, x1, dt):
        t = dt.view(-1, 1, 1, 1).to(x0.dtype)
        mix = x0 * (1 - t) + x1 * t
        return mix + 0.3 * torch.sin(7 * torch.roll(x0, 1, -1) - 5 * torch.roll(x1, 1, -2) + 3 * t) - 0.05


def test_frame_interpolation_matches_reference_order_and_values():
    """N2 (SURVEY.md 8f): the batched `-acc` wrapper returns the frames of the unmodified reference
    src/utils/frame_interpolation.py:23-69 (one network call per inserted frame and pair, host round trips) — same insertion
    order, same dt bit patterns, same clamping, same pass-through of the given frames — with `inter_frames` network calls.
    The reference's frames on this stand-in network are stored in tests/golden/reference_units.pt."""
    from aniportrait_b200.pipelines.frame_interpolation import batch_images_interpolation_tool, insertion_schedule
    gold = _reference_units()["film"]
    assert len(gold) == 2

    class Counting(_StandInFilm):
        calls = 0

        def forward(self, x0, x1, dt):
            Counting.calls += 1
            assert x0.dtype == torch.float16 and dt.dtype == torch.float16
            return super().forward(x0, x1, dt)

    for (bs, frames), case in zip([(1, 5), (2, 3)], gold):
        video = case["video"]                                                 # fp32, not fp16-representable
        assert video.shape == (bs, 3, frames, 8, 12)
        for n in range(1, 6):
            want = case["out"][n - 1]
            Counting.calls = 0
            got = batch_images_interpolation_tool(video, Counting(), inter_frames=n)
            assert Counting.calls == n                                        # (frames - 1) * n in the reference
            assert got.dtype == want.dtype == torch.float32 and got.shape == (bs, 3, (frames - 1) * (n + 1) + 1, 8, 12)
            assert torch.equal(got, want), (bs, frames, n)
            assert torch.equal(batch_images_interpolation_tool(video, _StandInFilm(), n, max_pairs_per_call=1), want)
            assert len(insertion_schedule(n)) == n
    # the midpoint first, then the quarters: the order for three inserted frames
    assert [(a, b, c) for a, b, c, _ in insertion_schedule(3)] == [(0, 4, 2), (0, 2, 1), (2, 4, 3)]
    assert torch.equal(batch_images_interpolation_tool(video, _StandInFilm(), 0), video)


class _PoseModelStandIn(torch.nn.Module):
    """The attributes of the reference's Audio2PoseModel (src/audio_models/pose_model.py:56-89) that infer reads, made of
    torch modules with the reference's hyper-parameters (8 post-norm decoder layers, 8 heads, feed-forward 2 * latent,
    batch_first); its audio encoder returns the features the reference's wav2vec2 produced for the stored case."""

    def __init__(self, case, biased_mask):
        super().__init__()
        E, feats = case["latent"], case["features"]
        self.out_dim = 6
        self._only_last_features = case["only_last"]
        self.pose_map = torch.nn.Linear(6, E)
        self.in_fn = torch.nn.Linear(feats.shape[-1], E)
        self.PPE = torch.nn.Module()
        self.PPE.register_buffer("pe", case["pe"])
        self.biased_mask = biased_mask
        layer = torch.nn.TransformerDecoderLayer(d_model=E, nhead=8, dim_feedforward=2 * E, batch_first=True)
        self.transformer_decoder = torch.nn.TransformerDecoder(layer, num_layers=8)
        self.pose_map_r = torch.nn.Linear(E, 6)
        self.id_embed = torch.nn.Embedding(100, E)
        if case["only_last"]:
            enc = types.SimpleNamespace(last_hidden_state=feats, hidden_states=None)
        else:
            enc = types.SimpleNamespace(last_hidden_state=feats[-1], hidden_states=tuple(feats))
        self.audio_encoder = lambda input_value, seq_len, output_hidden_states: enc


def test_kv_cached_pose_infer_matches_reference_infer():
    """N3 (SURVEY.md 8f): the incremental (KV-cached, one-key cross-attention precomputed) head-pose decoder returns what the
    UNMODIFIED reference Audio2PoseModel.infer (src/audio_models/pose_model.py:97-124) computes by re-decoding all tokens at
    every frame — seeded weights, CPU fp32. The reference's result, audio features and mask / positional-encoding buffers
    are stored in tests/golden/reference_units.pt."""
    from oracle.make_golden import POSE_CASES, pose_model_weights
    from aniportrait_b200.audio_models import enable_kv_cache, kv_cached_infer
    gold = _reference_units()
    assert len(gold["pose_infer"]) == len(POSE_CASES)
    worst = 0.0
    for case in gold["pose_infer"]:
        T = case["frames"]
        m = _PoseModelStandIn(case, gold["pose_biased_mask"][:, :T, :T]).eval()
        m.load_state_dict(pose_model_weights(m, case["seed"]))
        want = case["out"]
        with torch.no_grad():
            got = kv_cached_infer(m, None, T, id_seed=torch.tensor([7]))
            enable_kv_cache(m)
            again = m.infer(None, T, id_seed=torch.tensor([7]))
        assert got.shape == want.shape == (1, T, 6), (got.shape, want.shape)
        assert torch.equal(got, again)
        spread = (want[0, 1:] - want[0, :-1]).abs().mean().item()
        assert spread > 1e-3, "degenerate reference output: the test would prove nothing"
        worst = max(worst, ((got - want).norm() / want.norm()).item())
    print(f"kv-cached pose decoder vs reference re-decoding: rel-L2 {worst:.2e}")
    assert worst < 1e-4
