"""Python-side operator wrappers over the C ABI (torch tensors in, torch tensors out).

torch is used for device memory and streams only; every arithmetic op below is a hand-written sm_100a kernel in
aniportrait_b200/csrc reached through libaniportrait_b200.so. Activations are fp16 channels-last token matrices.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import I, LL, check, fptr, lib, ptr, stream_ptr

SHAPE_LOG = None  # dev aid: set to a list to record (kind, M, N, K, flags) of every GEMM / conv launch
GN_MAX_BLOCKS = 2368  # AP_GN_MAX_BLOCKS in include/aniportrait_b200.h
KERNEL_LAUNCHES = 0  # incremented by every wrapper; bench.py reports it as gpu_launches


def _count(n=1):
    global KERNEL_LAUNCHES
    KERNEL_LAUNCHES += n


def _ensure(t: torch.Tensor):
    if not t.is_cuda:
        raise _lib.ApError("aniportrait_b200 ops need CUDA tensors (no CPU fallback)")
    _lib.init(t.device.index if t.device.index is not None else torch.cuda.current_device())


# --------------------------------------------------------------------------------------------------------------
# weight repacking (done once at load time)
# --------------------------------------------------------------------------------------------------------------
def pack_conv3x3_weight(w: torch.Tensor, cin_pad_to: int = 64, cout_pad_to: int = 32) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> [Cout_p, 9*Cin_p] fp16, tap-major / channel-minor, zero padded."""
    cout, cin = w.shape[0], w.shape[1]
    cin_p = (cin + cin_pad_to - 1) // cin_pad_to * cin_pad_to
    cout_p = (cout + cout_pad_to - 1) // cout_pad_to * cout_pad_to
    wp = torch.zeros(cout_p, 3, 3, cin_p, dtype=torch.float16, device=w.device)
    wp[:cout, :, :, :cin] = w.permute(0, 2, 3, 1).to(torch.float16)
    return wp.reshape(cout_p, 9 * cin_p).contiguous()


def interleave_geglu(w: torch.Tensor, b: torch.Tensor | None):
    """FeedForward.net.0.proj weight [8C, C] (value half then gate half) -> rows interleaved in blocks of 16:
    [v0..15, g0..15, v16..31, g16..31, ...] so that a 32-column accumulator chunk holds matching value/gate pairs."""
    n2 = w.shape[0]
    half = n2 // 2
    assert half % 16 == 0
    idx = torch.arange(half, device=w.device).reshape(-1, 16)
    order = torch.cat([idx, idx + half], dim=1).reshape(-1)
    wi = w[order].contiguous()
    bi = b[order].contiguous() if b is not None else None
    return wi, bi


# --------------------------------------------------------------------------------------------------------------
# GEMM / conv
# --------------------------------------------------------------------------------------------------------------
class RowStats:
    """Per-row {sum, sumsq} partials of a GEMM output, written by its epilogue: the LayerNorm statistics of the next op."""

    def __init__(self, buf: torch.Tensor, parts: int, ld: int):
        self.buf, self.parts, self.ld = buf, parts, ld


class ColStats:
    """Per-channel {sum, sumsq} partials over 32-row blocks of a GEMM / conv output: the GroupNorm statistics of the next
    op. buf: fp32 [entries, C, 2]."""

    def __init__(self, buf: torch.Tensor):
        self.buf = buf


LN_EXTRA_K = 8    # columns the LayerNorm folding appends to K: (-mean_hi, -mean_lo, -mean_hi, 0 x 5) x (cs_hi, cs_hi, cs_lo, 0 x 5)


class LNFold:
    """LayerNorm folded into the consuming GEMM. The GEMM's weights are [W diag(gamma) | colsum_hi, colsum_hi, colsum_lo, 0..]
    (K + LN_EXTRA_K columns: models.blocks.fold_layer_norm), its bias beta.W^T + b; `stats` are the RowStats of the A
    operand x from its producer's epilogue. ops.gemm turns them into the [M, 8] operand (-mean_hi, -mean_lo, -mean_hi, 0..)
    and the per-row rstd (ap_layernorm_finalize_f16), appends the operand as a second K source, and the epilogue applies
    out = rstd * acc + bias."""

    def __init__(self, stats: RowStats, eps: float = 1e-5):
        self.stats, self.eps = stats, eps

    def operands(self, M: int, K: int):
        """(a2 [M, 8] fp16, rstd [M] fp32); computed once per RowStats."""
        cached = getattr(self.stats, "_ln_ops", None)
        if cached is None:
            dev = self.stats.buf.device
            a2 = torch.empty(M, LN_EXTRA_K, dtype=torch.float16, device=dev)
            rstd = torch.empty(M, dtype=torch.float32, device=dev)
            check(lib().ap_layernorm_finalize_f16(ptr(self.stats.buf), I(self.stats.parts), LL(self.stats.ld), LL(M), I(K),
                                                  _lib.c_float(self.eps), ptr(a2), fptr(rstd), stream_ptr()),
                  "ap_layernorm_finalize_f16")
            _count()
            cached = (a2, rstd)
            self.stats._ln_ops = cached
        return cached


def _epilogue_ext(M, N, device, row_stats, col_stats, ln, bias, flags, K, block_n):
    """Builds the ap_epilogue_ext for a call; returns (ext | None, RowStats | None, ColStats | None)."""
    bias_ld = 0
    if bias is not None and bias.dim() == 2 and bias.stride(0) != bias.shape[1]:
        bias_ld = bias.stride(0)           # a column slice of a wider table shared by several ops
    if not (row_stats or col_stats or ln is not None or bias_ld):
        return None, None, None
    ext = _lib.EpilogueExt()
    m_pad = (M + 127) // 128 * 128
    rs = cs = None
    if row_stats:
        parts = lib().ap_gemm_row_stat_parts(LL(M), I(N), I(K), I(flags), I(block_n))
        if parts <= 0:
            check(parts if parts < 0 else -1, "ap_gemm_row_stat_parts")
        rs = RowStats(torch.empty(2 * parts, m_pad, 2, dtype=torch.float32, device=device), 2 * parts, m_pad)
        ext.row_stat_out, ext.row_stat_ld = rs.buf.data_ptr(), m_pad
    if col_stats:
        cs = ColStats(torch.empty(m_pad // 32, N, 2, dtype=torch.float32, device=device))
        ext.col_stat_out, ext.col_stat_ld = cs.buf.data_ptr(), N
    if ln is not None:
        ext.ln_rstd = ln.rstd.data_ptr()
    ext.bias_ld = bias_ld
    return ext, rs, cs


def _with_stats(out, rs, cs, row_stats, col_stats):
    if not (row_stats or col_stats):
        return out
    res = [out]
    if row_stats:
        res.append(rs)
    if col_stats:
        res.append(cs)
    return tuple(res)


def gemm(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor | None = None, residual: torch.Tensor | None = None,
         a2: torch.Tensor | None = None, geglu: bool = False, out: torch.Tensor | None = None,
         bias_group_rows: int = 0, n_valid: int = 0, block_n: int = 0, out_f32: bool = False,
         row_stats: bool = False, col_stats: bool = False, ln: LNFold | None = None, gelu: bool = False):
    """out = [a | a2] @ w.T (+bias) (+residual); a:[M,K1] fp16 (row stride may exceed K1), w:[N,K1+K2] fp16.
    gelu: out = gelu_erf([a | a2] @ w.T + bias) (no residual).
    row_stats / col_stats: also return the epilogue's RowStats / ColStats of `out` (-> (out, RowStats?, ColStats?)).
    ln: fold a LayerNorm of `a` into this GEMM (see LNFold). bias may be a column slice of a wider fp32 table."""
    _ensure(a)
    assert a.dtype == torch.float16 and w.dtype == torch.float16 and a.dim() == 2 and w.dim() == 2
    assert a.stride(1) == 1 and w.is_contiguous()
    M, K1 = a.shape
    N = w.shape[0]
    K2 = 0
    if ln is not None:
        assert a2 is None and bias is not None, "LayerNorm folding: single-source A, folded bias required"
        a2, ln.rstd = ln.operands(M, K1)
    if a2 is not None:
        assert a2.dtype == torch.float16 and a2.shape[0] == M and a2.stride(1) == 1
        K2 = a2.shape[1]
    assert w.shape[1] == K1 + K2, (w.shape, K1, K2)
    nout = N // 2 if geglu else N
    if n_valid:
        nout = n_valid
    if out is None:
        out = torch.empty(M, nout, dtype=torch.float32 if out_f32 else torch.float16, device=a.device)
    assert out.stride(1) == 1 and out.dtype == (torch.float32 if out_f32 else torch.float16)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.stride(-1) == 1 and bias.shape[-1] == N
        assert bias.is_contiguous() or bias.dim() == 2
    if residual is not None:
        assert residual.dtype == torch.float16 and residual.stride(1) == 1 and residual.shape[0] == M
    assert not (gelu and (geglu or residual is not None)), "the GELU epilogue takes no residual and excludes GEGLU"
    flags = (1 if geglu else 0) | (2 if out_f32 else 0) | (4 if gelu else 0)
    ext, rs, cs = _epilogue_ext(M, N, a.device, row_stats, col_stats, ln, bias, flags, K1 + K2, block_n)
    rc = lib().ap_gemm_f16(ptr(a), LL(a.stride(0)), I(K1), ptr(a2), LL(a2.stride(0) if a2 is not None else 0), I(K2),
                           ptr(w), LL(M), I(N), fptr(bias), LL(bias_group_rows), ptr(residual),
                           LL(residual.stride(0) if residual is not None else 0), ptr(out), LL(out.stride(0)),
                           I(nout), I(flags), I(block_n), stream_ptr(), _lib.ext_ptr(ext))
    check(rc, "ap_gemm_f16")
    if SHAPE_LOG is not None:
        SHAPE_LOG.append(("gemm_geglu" if geglu else ("gemm_gelu" if gelu else "gemm"), M, N, K1 + K2,
                          int(residual is not None)))
    _count()
    return _with_stats(out, rs, cs, row_stats, col_stats)


def conv_col_stats_ok(nf: int, ho: int, wo: int) -> bool:
    """Can a 3x3 conv with this output grid emit GroupNorm column statistics from its epilogue? (mirrors the tile-box choice
    of ap_conv3x3_nhwc_f16: every 32-row sub-box of a tile must lie in one frame, entries frame-major)."""
    def pow2_div(v, cap):
        d = 1
        while d * 2 <= cap and v % (d * 2) == 0:
            d *= 2
        return d
    bw = pow2_div(wo, 128)
    bh = pow2_div(ho, 128 // bw)
    bnf = 128 // (bw * bh)
    tiles = (wo // bw) * (ho // bh)
    return (ho * wo) % 32 == 0 and bw * bh >= 32 and (bnf == 1 or tiles == 1)


def conv_m_tiles(nf: int, ho: int, wo: int) -> int:
    def pow2_div(v, cap):
        d = 1
        while d * 2 <= cap and v % (d * 2) == 0:
            d *= 2
        return d
    bw = pow2_div(wo, 128)
    bh = pow2_div(ho, 128 // bw)
    bnf = 128 // (bw * bh)
    return (nf + bnf - 1) // bnf * (wo // bw) * (ho // bh)


def conv3x3(x: torch.Tensor, w_packed: torch.Tensor, cout: int, bias: torch.Tensor | None = None,
            residual: torch.Tensor | None = None, x2: torch.Tensor | None = None, stride: int = 1,
            out: torch.Tensor | None = None, bias_group_rows: int = 0, block_n: int = 0, col_stats: bool = False):
    """x: [Nf, H, W, C1] fp16 channels-last (C1 % 64 == 0); w_packed: pack_conv3x3_weight(...); returns
    [Nf, H/stride, W/stride, cout] (and, with col_stats, the ColStats of the output for the next GroupNorm: only where
    conv_col_stats_ok(...) holds). bias may be a column slice of a wider fp32 table."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 4
    nf, h, wd, c1 = x.shape
    c2 = 0
    if x2 is not None:
        assert x2.is_contiguous() and x2.shape[:3] == x.shape[:3]
        c2 = x2.shape[3]
    cout_p = w_packed.shape[0]
    assert w_packed.shape[1] == 9 * (c1 + c2), (w_packed.shape, c1, c2)
    ho, wo = h // stride, wd // stride
    if out is None:
        out = torch.empty(nf, ho, wo, cout, dtype=torch.float16, device=x.device)
    assert out.is_contiguous()
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.stride(-1) == 1 and bias.shape[-1] == cout_p
        assert bias.is_contiguous() or bias.dim() == 2
    if residual is not None:
        assert residual.is_contiguous() and residual.shape == out.shape
    ext, cs = None, None
    bias_ld = bias.stride(0) if (bias is not None and bias.dim() == 2 and bias.stride(0) != bias.shape[1]) else 0
    if col_stats or bias_ld:
        ext = _lib.EpilogueExt()
        ext.bias_ld = bias_ld
        if col_stats:
            assert cout == cout_p, "column statistics need an unpadded output width"
            cs = ColStats(torch.empty(4 * conv_m_tiles(nf, ho, wo), cout, 2, dtype=torch.float32, device=x.device))
            ext.col_stat_out, ext.col_stat_ld = cs.buf.data_ptr(), cout
    rc = lib().ap_conv3x3_nhwc_f16(ptr(x), I(c1), ptr(x2), I(c2), I(nf), I(h), I(wd), I(stride), ptr(w_packed),
                                   I(cout_p), fptr(bias), LL(bias_group_rows), ptr(residual), ptr(out), LL(cout),
                                   I(cout), I(block_n), stream_ptr(), _lib.ext_ptr(ext))
    check(rc, "ap_conv3x3_nhwc_f16")
    if SHAPE_LOG is not None:
        SHAPE_LOG.append((f"conv3x3_s{stride}", nf * ho * wo, cout_p, 9 * (c1 + c2), int(residual is not None)))
    _count()
    return (out, cs) if col_stats else out


# --------------------------------------------------------------------------------------------------------------
# normalisation
# --------------------------------------------------------------------------------------------------------------
_stats_ws = {}


def _stats_workspace(device, n):
    key = (device.index, torch.cuda.current_stream().cuda_stream)
    buf = _stats_ws.get(key)
    if buf is None or buf.numel() < n:
        # sized once for any realistic frame count: CUDA graphs keep this pointer, so it must never be re-allocated
        buf = torch.empty(max(n, 2 * 32 * (4096 + 2 * GN_MAX_BLOCKS)), dtype=torch.float32, device=device)
        _stats_ws[key] = buf
    return buf


def group_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, eps: float, silu: bool,
               x2: torch.Tensor | None = None, out: torch.Tensor | None = None, stats: ColStats | None = None,
               stats2: ColStats | None = None) -> torch.Tensor:
    """x: [Nf, HW, C1] (or [Nf,H,W,C1]) fp16 channels-last; optional x2 concatenated along C. gamma/beta fp32 [C].
    stats / stats2: ColStats written by the epilogue of the op that produced x / x2: when every source has them, the
    statistics pass over the activation is skipped (finalize from the partials + apply only)."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous()
    nf, c1 = x.shape[0], x.shape[-1]
    hw = x.numel() // (nf * c1)
    c2 = 0
    if x2 is not None:
        assert x2.is_contiguous() and x2.shape[0] == nf
        c2 = x2.shape[-1]
    c = c1 + c2
    assert gamma.dtype == torch.float32 and gamma.numel() == c and beta.numel() == c
    if out is None:
        out = torch.empty(*x.shape[:-1], c, dtype=torch.float16, device=x.device)
    fused = stats is not None and (x2 is None or stats2 is not None) and hw % 32 == 0 and groups <= 32
    ws = _stats_workspace(x.device, 2 * groups * (nf + 2 * GN_MAX_BLOCKS))
    if fused:
        for st, cc in ((stats, c1), (stats2, c2)):
            if st is not None:
                assert st.buf.shape[1] == cc and st.buf.shape[0] >= nf * hw // 32, (st.buf.shape, nf, hw, cc)
        rc = lib().ap_groupnorm_apply_nhwc_f16(ptr(x), I(c1), ptr(stats.buf), LL(c1), ptr(x2), I(c2),
                                               ptr(stats2.buf if stats2 is not None else None), LL(c2), I(nf), I(hw),
                                               I(groups), _lib.c_float(eps), fptr(gamma), fptr(beta),
                                               I(1 if silu else 0), fptr(ws), ptr(out), stream_ptr())
        check(rc, "ap_groupnorm_apply_nhwc_f16")
        _count(3 if x2 is not None else 2)
        return out
    stats = ws
    rc = lib().ap_groupnorm_nhwc_f16(ptr(x), I(c1), ptr(x2), I(c2), I(nf), I(hw), I(groups), _lib.c_float(eps),
                                     fptr(gamma), fptr(beta), I(1 if silu else 0), fptr(stats), ptr(out),
                                     stream_ptr())
    check(rc, "ap_groupnorm_nhwc_f16")
    _count(5 if x2 is not None else 3)
    return out


def layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5,
               pe: torch.Tensor | None = None, rows_per_pe: int = 0, pe_period: int = 0,
               out: torch.Tensor | None = None) -> torch.Tensor:
    """x: [rows, C] fp16; pe: optional fp32 [pe_period, C] added after the affine (row r uses pe[(r//rows_per_pe)%period])."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 2
    rows, c = x.shape
    if out is None:
        out = torch.empty_like(x)
    if pe is not None:
        assert pe.dtype == torch.float32 and pe.is_contiguous() and pe.shape[-1] == c and pe.shape[0] >= pe_period
    rc = lib().ap_layernorm_f16(ptr(x), LL(rows), I(c), _lib.c_float(eps), fptr(gamma), fptr(beta), fptr(pe),
                                I(rows_per_pe), I(pe_period), ptr(out), stream_ptr())
    check(rc, "ap_layernorm_f16")
    _count()
    return out


BN_MAX_BLOCKS = 2048  # AP_BN_MAX_BLOCKS in include/aniportrait_b200.h
_bn_ws = {}


def batch_norm_train(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5, relu: bool = True,
                     out: torch.Tensor | None = None) -> torch.Tensor:
    """nn.BatchNorm2d in TRAIN mode (batch statistics over every row of the call, biased variance) + optional ReLU.
    x: [..., C] fp16 channels-last, C % 8 == 0; gamma/beta fp32 [C]."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous()
    c = x.shape[-1]
    rows = x.numel() // c
    assert gamma.dtype == torch.float32 and gamma.numel() == c and beta.dtype == torch.float32 and beta.numel() == c
    if out is None:
        out = torch.empty_like(x)
    key = (x.device.index, torch.cuda.current_stream().cuda_stream)
    ws = _bn_ws.get(key)
    if ws is None:   # sized once for the widest layer: CUDA graphs keep this pointer
        ws = torch.empty(2 * 2048 * (BN_MAX_BLOCKS + 1), dtype=torch.float32, device=x.device)
        _bn_ws[key] = ws
    rc = lib().ap_batchnorm_train_nhwc_f16(ptr(x), LL(rows), I(c), fptr(gamma), fptr(beta), _lib.c_float(eps),
                                           I(1 if relu else 0), fptr(ws), LL(ws.numel()), ptr(out), stream_ptr())
    check(rc, "ap_batchnorm_train_nhwc_f16")
    _count(3)
    return out


def pack_conv_direct_weight(w: torch.Tensor, cin_pad: int, cout_pad: int) -> torch.Tensor:
    """[Cout, Cin, K, K] -> [cout_pad, K, K, cin_pad] fp16 (zero padded) for conv2d_direct."""
    cout, cin, k, _ = w.shape
    wp = torch.zeros(cout_pad, k, k, cin_pad, dtype=torch.float16, device=w.device)
    wp[:cout, :, :, :cin] = w.permute(0, 2, 3, 1).to(torch.float16)
    return wp.contiguous()


def conv2d_direct(x: torch.Tensor, w_packed: torch.Tensor, stride: int, pad: int = 1,
                  bias: torch.Tensor | None = None) -> torch.Tensor:
    """Small-channel direct convolution. x: [Nf, H, W, Cin] fp16 (Cin in {8, 16, 32}); w_packed from
    pack_conv_direct_weight; returns [Nf, Ho, Wo, Cout]."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 4 and w_packed.dtype == torch.float16
    nf, h, wd, cin = x.shape
    cout, k, _, cin_w = w_packed.shape
    assert cin_w == cin and w_packed.is_contiguous()
    ho, wo = (h + 2 * pad - k) // stride + 1, (wd + 2 * pad - k) // stride + 1
    out = torch.empty(nf, ho, wo, cout, dtype=torch.float16, device=x.device)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == cout
    rc = lib().ap_conv2d_direct_nhwc_f16(ptr(x), I(cin), I(nf), I(h), I(wd), ptr(w_packed), I(cout), I(k), I(stride),
                                         I(pad), fptr(bias), ptr(out), stream_ptr())
    check(rc, "ap_conv2d_direct_nhwc_f16")
    _count()
    return out


def softmax_rows(x: torch.Tensor) -> torch.Tensor:
    """In-place row softmax of an fp16 matrix [rows, cols] (cols even)."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.dim() == 2 and x.stride(1) == 1
    check(lib().ap_softmax_rows_f16(ptr(x), ptr(x), LL(x.shape[0]), I(x.shape[1]), LL(x.stride(0)), stream_ptr()),
          "ap_softmax_rows_f16")
    _count()
    return x


# --------------------------------------------------------------------------------------------------------------
# attention
# --------------------------------------------------------------------------------------------------------------
def head_pad(d: int) -> int:
    """Head dim padded to a whole number of 64-column swizzle atoms (40->64, 80->128, 88->128, 160->192)."""
    p = (d + 63) // 64 * 64
    if p > 192:
        raise _lib.ApError(f"head_dim {d} > 192 is not supported by the fused attention kernel")
    return p


def pad_head_rows(w: torch.Tensor, heads: int, dpad: int) -> torch.Tensor:
    """Projection weight [heads*d, K] -> [heads*dpad, K] with zero rows after each head's d rows."""
    hd, k = w.shape
    d = hd // heads
    out = torch.zeros(heads, dpad, k, dtype=w.dtype, device=w.device)
    out[:, :d] = w.view(heads, d, k)
    return out.reshape(heads * dpad, k).contiguous()


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, n_frames: int, tokens: int, heads: int,
              head_dim: int, dpad: int, bank_k: torch.Tensor | None = None, bank_v: torch.Tensor | None = None,
              bank_tokens: int = 0, n_banks: int = 0, first_bank_frame: int = 0, frames_per_bank: int = 1,
              scale: float | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """q/k/v: column-slices [n_frames*tokens, heads*dpad] of one fp16 buffer (same row stride); returns
    [n_frames*tokens, heads*head_dim]."""
    _ensure(q)
    rows = n_frames * tokens
    for t in (q, k, v):
        assert t.dtype == torch.float16 and t.shape == (rows, heads * dpad) and t.stride(1) == 1
        assert t.stride(0) == q.stride(0)
    if out is None:
        out = torch.empty(rows, heads * head_dim, dtype=torch.float16, device=q.device)
    ld_bank = 0
    if bank_k is not None:
        assert bank_k.shape == (n_banks * bank_tokens, heads * dpad) and bank_k.stride(1) == 1
        assert bank_v.shape == bank_k.shape and bank_v.stride(0) == bank_k.stride(0)
        ld_bank = bank_k.stride(0)
    if scale is None:
        scale = head_dim ** -0.5
    rc = lib().ap_attention_f16(ptr(q), ptr(k), ptr(v), LL(q.stride(0)), ptr(bank_k), ptr(bank_v), LL(ld_bank),
                                I(bank_tokens), I(n_banks), I(n_frames), I(tokens), I(heads), I(head_dim), I(dpad),
                                I(first_bank_frame), I(frames_per_bank), _lib.c_float(scale), ptr(out),
                                LL(out.stride(0)), stream_ptr())
    check(rc, "ap_attention_f16")
    _count()
    return out


def temporal_attention(qkv: torch.Tensor, B: int, F: int, N: int, C: int, heads: int,
                       out: torch.Tensor | None = None) -> torch.Tensor:
    _ensure(qkv)
    assert qkv.dtype == torch.float16 and qkv.shape == (B * F * N, 3 * C) and qkv.stride(1) == 1
    if out is None:
        out = torch.empty(B * F * N, C, dtype=torch.float16, device=qkv.device)
    scale = (C // heads) ** -0.5
    rc = lib().ap_temporal_attention_f16(ptr(qkv), LL(qkv.stride(0)), ptr(out), LL(out.stride(0)), I(B), I(F), I(N),
                                         I(C), I(heads), _lib.c_float(scale), stream_ptr())
    check(rc, "ap_temporal_attention_f16")
    _count()
    return out


# --------------------------------------------------------------------------------------------------------------
# elementwise / layout
# --------------------------------------------------------------------------------------------------------------
def add(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    _ensure(a)
    assert a.dtype == torch.float16 and a.shape == b.shape and a.is_contiguous() and b.is_contiguous()
    if out is None:
        out = torch.empty_like(a)
    check(lib().ap_add_f16(ptr(a), ptr(b), ptr(out), LL(a.numel()), stream_ptr()), "ap_add_f16")
    _count()
    return out


def add_bcast(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """a: [dup*n...], b: [n...] broadcast over the leading duplicate (CFG) dimension."""
    _ensure(a)
    assert a.dtype == torch.float16 and a.is_contiguous() and b.is_contiguous() and a.numel() % b.numel() == 0
    if out is None:
        out = torch.empty_like(a)
    check(lib().ap_add_bcast_f16(ptr(a), ptr(b), ptr(out), LL(a.numel()), LL(b.numel()), stream_ptr()),
          "ap_add_bcast_f16")
    _count()
    return out


def timestep_embedding(t: torch.Tensor, dim: int) -> torch.Tensor:
    """t: fp32 [B] on device -> fp16 [B, dim] (cos | sin)."""
    _ensure(t)
    assert t.dtype == torch.float32 and t.is_contiguous()
    out = torch.empty(t.numel(), dim, dtype=torch.float16, device=t.device)
    check(lib().ap_timestep_embedding_f16(fptr(t), I(t.numel()), I(dim), ptr(out), stream_ptr()),
          "ap_timestep_embedding_f16")
    _count()
    return out


def silu(x: torch.Tensor) -> torch.Tensor:
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous()
    out = torch.empty_like(x)
    check(lib().ap_silu_f16(ptr(x), ptr(out), LL(x.numel()), stream_ptr()), "ap_silu_f16")
    _count()
    return out


def upsample2x(x: torch.Tensor) -> torch.Tensor:
    _ensure(x)
    nf, h, w, c = x.shape
    assert x.dtype == torch.float16 and x.is_contiguous()
    out = torch.empty(nf, 2 * h, 2 * w, c, dtype=torch.float16, device=x.device)
    check(lib().ap_upsample2x_nhwc_f16(ptr(x), ptr(out), I(nf), I(h), I(w), I(c), stream_ptr()), "ap_upsample2x")
    _count()
    return out


def ncfhw_to_nhwc(x: torch.Tensor, cpad: int) -> torch.Tensor:
    """[B, C, F, H, W] -> [(B F), H, W, cpad] (zero padded channels)."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 5
    b, c, f, h, w = x.shape
    out = torch.empty(b * f, h, w, cpad, dtype=torch.float16, device=x.device)
    check(lib().ap_ncfhw_to_nhwc_f16(ptr(x), ptr(out), I(b), I(c), I(f), I(h * w), I(cpad), stream_ptr()),
          "ap_ncfhw_to_nhwc_f16")
    _count()
    return out


def nhwc_to_ncfhw(x: torch.Tensor, B: int, C: int, F: int) -> torch.Tensor:
    """[(B F), H, W, ld>=C] -> [B, C, F, H, W]."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 4 and x.shape[0] == B * F
    _, h, w, ld = x.shape
    out = torch.empty(B, C, F, h, w, dtype=torch.float16, device=x.device)
    check(lib().ap_nhwc_to_ncfhw_f16(ptr(x), ptr(out), I(B), I(C), I(F), I(h * w), I(ld), stream_ptr()),
          "ap_nhwc_to_ncfhw_f16")
    _count()
    return out


def gather_window(latents: torch.Tensor, frame_idx: torch.Tensor, dup: int, cpad: int = 64) -> torch.Tensor:
    """latents [L, H, W, 4] fp16 -> UNet input [(dup F), H, W, cpad]."""
    _ensure(latents)
    L, h, w, c = latents.shape
    assert c == 4 and latents.dtype == torch.float16 and latents.is_contiguous() and frame_idx.dtype == torch.int32
    F = frame_idx.numel()
    out = torch.empty(dup * F, h, w, cpad, dtype=torch.float16, device=latents.device)
    check(lib().ap_gather_window_f16(ptr(latents), _lib.ctypes.cast(_lib.c_void_p(frame_idx.data_ptr()),
                                                                     _lib.POINTER(_lib.c_int)),
                                     ptr(out), I(dup), I(F), I(h * w), I(cpad), stream_ptr()), "ap_gather_window_f16")
    _count()
    return out


def scatter_accumulate(pred: torch.Tensor, frame_idx: torch.Tensor, acc: torch.Tensor):
    """pred [(B F), H, W, ld] fp16 (first 4 channels) accumulated into acc fp32 [B, L, H, W, 4] at frame_idx."""
    _ensure(pred)
    B, L, h, w, _ = acc.shape
    F = frame_idx.numel()
    assert pred.shape[0] == B * F and acc.dtype == torch.float32 and acc.is_contiguous() and pred.is_contiguous()
    check(lib().ap_scatter_accumulate_f16(ptr(pred), I(pred.shape[-1]),
                                          _lib.ctypes.cast(_lib.c_void_p(frame_idx.data_ptr()), _lib.POINTER(_lib.c_int)),
                                          fptr(acc), I(B), I(F), I(L), I(h * w), stream_ptr()),
          "ap_scatter_accumulate_f16")
    _count()


PREDICTION_TYPES = {"v_prediction": 0, "epsilon": 1, "sample": 2}   # AP_PRED_* in include/aniportrait_b200.h


def cfg_ddim_step(acc: torch.Tensor, inv_count: torch.Tensor, guidance: float, alpha_t: float, alpha_prev: float,
                  latents: torch.Tensor, prediction_type: str = "v_prediction", clip_range: float = 0.0):
    """In place: latents <- DDIM (eta = 0) step of the CFG-combined, overlap-averaged prediction; acc zeroed.
    clip_range > 0 clamps the predicted x0 (DDIMScheduler clip_sample)."""
    if prediction_type not in PREDICTION_TYPES:
        raise ValueError(f"prediction_type {prediction_type!r} is not one of {sorted(PREDICTION_TYPES)}")
    _ensure(latents)
    B, L, h, w, _ = acc.shape
    assert latents.shape == (L, h, w, 4) and latents.dtype == torch.float16 and inv_count.dtype == torch.float32
    check(lib().ap_cfg_ddim_step_f16(fptr(acc), fptr(inv_count), I(1 if B == 2 else 0), _lib.c_float(guidance),
                                     _lib.c_float(alpha_t), _lib.c_float(alpha_prev),
                                     I(PREDICTION_TYPES[prediction_type]), _lib.c_float(clip_range), ptr(latents),
                                     I(L), I(h * w), stream_ptr()), "ap_cfg_ddim_step_f16")
    _count()


def pack_frames_u8(video: torch.Tensor, rescale: bool = False) -> torch.Tensor:
    """video [B, 3, F, H, W] fp16 (any strides, e.g. the decoder's [F, 3, H, W] frames viewed as a video) -> [B, F, H, W, 3]
    uint8 on the device: the bytes `save_videos_grid` (reference src/utils/util.py:87-104) makes on the host from the fp32
    copy, `(x * 255).astype(uint8)` after `(x + 1) / 2` if rescale."""
    _ensure(video)
    assert video.dim() == 5 and video.shape[1] == 3 and video.dtype == torch.float16, "pack_frames_u8: [B, 3, F, H, W] fp16"
    B, _, F, H, W = video.shape
    out = torch.empty(B, F, H, W, 3, dtype=torch.uint8, device=video.device)
    strides = (_lib.c_longlong * 5)(*video.stride())
    check(lib().ap_pack_frames_u8(ptr(video), strides, I(B), I(F), I(H), I(W), I(1 if rescale else 0), ptr(out),
                                  stream_ptr()), "ap_pack_frames_u8")
    _count()
    return out


# --------------------------------------------------------------------------------------------------------------
# audio front-end (wav2vec2 encoder of audio2vid)
# --------------------------------------------------------------------------------------------------------------
def wav_conv0_gn_gelu(wav: torch.Tensor, w: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor,
                      eps: float = 1e-5) -> torch.Tensor:
    """wav2vec2 feature-extractor layer 0: Conv1d(1, 512, 10, stride 5, no bias) + GroupNorm(512, 512) + GELU.
    wav: fp32 [S]; w: fp32 [512, 10]; gamma/beta fp32 [512]; returns fp16 channels-last [(S - 10) // 5 + 1, 512]."""
    _ensure(wav)
    assert wav.dtype == torch.float32 and wav.dim() == 1 and wav.is_contiguous()
    assert w.dtype == torch.float32 and w.shape == (512, 10) and w.is_contiguous()
    assert gamma.dtype == torch.float32 and gamma.numel() == 512 and beta.dtype == torch.float32 and beta.numel() == 512
    S = wav.numel()
    if S < 10:
        raise ValueError(f"wav_conv0_gn_gelu: {S} samples, fewer than the kernel width 10")
    out = torch.empty((S - 10) // 5 + 1, 512, dtype=torch.float16, device=wav.device)
    need = lib().ap_wav_conv0_workspace_floats(LL(S))
    if need < 0:
        check(need, "ap_wav_conv0_workspace_floats")
    ws = torch.empty(need, dtype=torch.float32, device=wav.device)
    check(lib().ap_wav_conv0_gn_gelu_f16(fptr(wav), LL(S), fptr(w), fptr(gamma), fptr(beta), _lib.c_float(eps), fptr(ws),
                                         LL(ws.numel()), ptr(out), stream_ptr()), "ap_wav_conv0_gn_gelu_f16")
    _count(3)
    return out


def pack_conv1d_taps(w: torch.Tensor) -> torch.Tensor:
    """Conv1d weight [Cout, Cin, k] -> [Cout, k * Cin] fp16, tap-major / channel-minor: row o, column t * Cin + c holds
    w[o, c, t], the order in which a channels-last strided view presents k consecutive input frames."""
    cout, cin, k = w.shape
    return w.detach().permute(0, 2, 1).reshape(cout, k * cin).to(torch.float16).contiguous()


def conv1d_s2_gelu(x: torch.Tensor, w_packed: torch.Tensor, k: int) -> torch.Tensor:
    """Conv1d(C, C, k in {2, 3}, stride 2, no bias) + GELU on channels-last x [T_in, C] fp16 as ONE GEMM over strided views of
    x (no im2col): A row t = frames 2t, 2t+1 (= x viewed as [T_out, 2C] with row stride 2C), plus frame 2t + 2 for k = 3 as the
    second K source (x from frame 2 on, same row stride). w_packed: pack_conv1d_taps(w). Returns [T_out, C]."""
    assert k in (2, 3) and x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 2
    t_in, c = x.shape
    if t_in < k:
        raise ValueError(f"conv1d_s2_gelu: {t_in} frames, fewer than the kernel width {k}")
    t_out = (t_in - k) // 2 + 1
    # the views end inside x: k = 2 reads frames <= 2 t_out - 1 <= t_in - 1; k = 3 reads frames <= 2 (t_out - 1) + 2 <= t_in - 1
    a = x.as_strided((t_out, 2 * c), (2 * c, 1))
    a2 = x.as_strided((t_out, c), (2 * c, 1), x.storage_offset() + 2 * c) if k == 3 else None
    assert w_packed.shape == (c, k * c)
    return gemm(a, w_packed, a2=a2, gelu=True)


def interp_linear_time(x: torch.Tensor, t_out: int) -> torch.Tensor:
    """F.interpolate(mode="linear", align_corners=True) along time: x [T_in, C] fp16 -> [t_out, C]."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 2 and x.shape[1] % 8 == 0
    out = torch.empty(int(t_out), x.shape[1], dtype=torch.float16, device=x.device)
    check(lib().ap_interp_linear_time_f16(ptr(x), I(x.shape[0]), I(x.shape[1]), ptr(out), I(int(t_out)), stream_ptr()),
          "ap_interp_linear_time_f16")
    _count()
    return out


POS_CONV_GROUPS, POS_CONV_K = 16, 128


def pack_pos_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """Resolved positional-conv weight [768, 48, 128] (out, in-of-group, tap) -> [16 groups, 128 taps, 48 in, 48 out] fp16."""
    cout, cin_g, k = w.shape
    g = POS_CONV_GROUPS
    assert k == POS_CONV_K and cout == g * cin_g
    return w.detach().reshape(g, cout // g, cin_g, k).permute(0, 3, 2, 1).to(torch.float16).contiguous()


def pos_conv_gelu(x: torch.Tensor, w_packed: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """x + GELU(grouped positional conv(x) + bias), k = 128, padding 64, last frame dropped. x: [T, 768] fp16."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and x.dim() == 2 and x.shape[1] == 768
    assert w_packed.dtype == torch.float16 and w_packed.shape == (16, 128, 48, 48) and w_packed.is_contiguous()
    assert bias.dtype == torch.float32 and bias.numel() == 768 and bias.is_contiguous()
    out = torch.empty_like(x)
    check(lib().ap_pos_conv_gelu_f16(ptr(x), I(x.shape[0]), ptr(w_packed), fptr(bias), ptr(out), stream_ptr()),
          "ap_pos_conv_gelu_f16")
    _count()
    return out


def mean_f16(x: torch.Tensor, out_f32: bool = True, out_f16: bool = False):
    """Mean over the leading dim of fp16 x [n_src, ...], summed in fp32 in order; returns the fp32 and / or fp16 result
    (a tuple when both are asked for). n_src = 1: an fp16 -> fp32 copy."""
    _ensure(x)
    assert x.dtype == torch.float16 and x.is_contiguous() and (out_f32 or out_f16)
    o32 = torch.empty(x.shape[1:], dtype=torch.float32, device=x.device) if out_f32 else None
    o16 = torch.empty(x.shape[1:], dtype=torch.float16, device=x.device) if out_f16 else None
    check(lib().ap_mean_f16(ptr(x), I(x.shape[0]), LL(x[0].numel()), fptr(o32), ptr(o16), stream_ptr()), "ap_mean_f16")
    _count()
    if out_f32 and out_f16:
        return o32, o16
    return o32 if out_f32 else o16


# --------------------------------------------------------------------------------------------------------------
# face-mesh pose maps (audio2vid / vid2vid conditioning: reference src/utils/pose_util.py, draw_util.py)
# --------------------------------------------------------------------------------------------------------------
_F32_F64 = (torch.float32, torch.float64)


def _float_operand(t: torch.Tensor, what: str, shape_ok) -> torch.Tensor:
    _ensure(t)
    if t.dtype not in _F32_F64 or not shape_ok(t.shape):
        raise ValueError(f"{what}: expected fp32 / fp64 of the documented shape, got {t.dtype} {tuple(t.shape)}")
    return t.contiguous()


def pose_smooth(x: torch.Tensor, window: int) -> torch.Tensor:
    """smooth_pose_seq: sliding-window mean over rows of x [L, 6] (fp32 or fp64), bit-identical to numpy's."""
    x = _float_operand(x, "pose_smooth", lambda s: len(s) == 2 and s[0] > 0 and s[1] == 6)
    if int(window) < 1:
        raise ValueError(f"pose_smooth: window {window} < 1")
    out = torch.empty_like(x)
    check(lib().ap_pose_smooth(ptr(x), I(x.shape[0]), I(int(window)), I(x.dtype == torch.float64), ptr(out), stream_ptr()),
          "ap_pose_smooth")
    _count()
    return out


def project_points(points: torch.Tensor, trans: torch.Tensor, pose: torch.Tensor | None, width: int,
                   height: int) -> torch.Tensor:
    """Perspective projection in fp64: points [L, N, 3]; with `pose` [L, 6] one trans [4, 4], else per-frame trans
    [L, 4, 4]. Returns fp64 [L, N, 2] pixel coordinates of a width x height image."""
    points = _float_operand(points, "project_points: points", lambda s: len(s) == 3 and s[0] > 0 and s[1] > 0 and s[2] == 3)
    L = points.shape[0]
    if pose is None:
        trans = _float_operand(trans, "project_points: trans", lambda s: tuple(s) == (L, 4, 4))
    else:
        trans = _float_operand(trans, "project_points: trans", lambda s: tuple(s) == (4, 4))
        pose = _float_operand(pose, "project_points: pose", lambda s: len(s) == 2 and s[0] >= L and s[1] == 6)
    out = torch.empty(L, points.shape[1], 2, dtype=torch.float64, device=points.device)
    f64 = lambda t: I(t is not None and t.dtype == torch.float64)  # noqa: E731
    check(lib().ap_project_points(ptr(points), f64(points), I(L), I(points.shape[1]), ptr(trans), f64(trans), ptr(pose),
                                  f64(pose), I(int(width)), I(int(height)), ptr(out), stream_ptr()), "ap_project_points")
    _count()
    return out


def facemesh_raster(keypoints: torch.Tensor, edges: torch.Tensor, colours: torch.Tensor, width: int, height: int,
                    normed: bool = False) -> torch.Tensor:
    """Face-mesh pose maps: keypoints [L, N, 2] (fp32 / fp64; pixels of a width x height image, or normalised) drawn as
    thickness-2 cv2 lines of `edges` (int32 [E, 3]: a, b, colour group) in `colours` (uint8 [G, 3]) on a 512 x 512
    canvas, resized to width x height (multiples of 8). Returns uint8 [L, height, width, 3]."""
    keypoints = _float_operand(keypoints, "facemesh_raster: keypoints",
                               lambda s: len(s) == 3 and s[0] > 0 and s[1] > 0 and s[2] == 2)
    _ensure(edges)
    _ensure(colours)
    if edges.dtype != torch.int32 or edges.dim() != 2 or edges.shape[1] != 3 or not edges.is_contiguous():
        raise ValueError("facemesh_raster: edges must be contiguous int32 [E, 3]")
    if colours.dtype != torch.uint8 or colours.dim() != 2 or colours.shape[1] != 3 or not colours.is_contiguous():
        raise ValueError("facemesh_raster: colours must be contiguous uint8 [G, 3]")
    W, H = int(width), int(height)
    if W <= 0 or H <= 0 or W % 8 or H % 8:
        raise ValueError(f"facemesh_raster: width {W} and height {H} must be positive multiples of 8")
    L, N = keypoints.shape[:2]
    canvas = torch.empty(L, 512, 512, dtype=torch.uint8, device=keypoints.device)
    out = torch.empty(L, H, W, 3, dtype=torch.uint8, device=keypoints.device)
    check(lib().ap_facemesh_raster(ptr(keypoints), I(keypoints.dtype == torch.float64), I(L), I(N), I(bool(normed)), I(W),
                                   I(H), ptr(edges), I(edges.shape[0]), ptr(colours), I(colours.shape[0]), ptr(canvas),
                                   ptr(out), stream_ptr()), "ap_facemesh_raster")
    _count(2)
    return out
