"""Kernel-level fp64 parity of the accuracy mode (precision="f32x3"): the streaming kernels of csrc/accurate.cu, the
fp32 conv-0 layer of csrc/frontend.cu, the split-operand GEMMs (A' = [x_hi|x_lo|x_hi], W' = [w_hi|w_hi|w_lo]) as the
encoder and the default path's fp32-input Linears use them, the three-pass positional conv, and the whole encoder.

The mode claims fp32 accuracy, so every reference is fp64 on the exact fp32 inputs the kernel reads: rounding an input
to 16 bits counts as error.  Where an operation has a default-mode twin, the twin runs in the same test on the
bf16-rounded inputs against the same reference, and the f32x3 error must be at least 64x smaller: a defect that drops
part of a tensor (a lost lo term, a wrong halo row, a masked key let in) to bf16-level error fails that rule even when
an absolute bound would have room for it.

Each absolute bound is about 4x the error measured on an NVIDIA B200 (1000 W power limit); the measured value is
given beside it.  Errors of GEMM-like outputs are normalised by the sum of absolute products, |x|.|w|^T + |b| (+ |r|
with a residual), which is what fp32 accumulation scales with.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from aptai_b200 import accurate
from aptai_b200 import lib as _lib
from aptai_b200 import ops
from aptai_b200.backbone import Wav2Vec2Backbone
from aptai_b200.config import W2V2Config
from oracle import w2v2 as ow
from oracle.weights import backbone_state_dict, waveforms

F64, I16, I32 = torch.float64, torch.int16, torch.int32
TWIN_RATIO = 64.0


def _randn(shape, dev, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g, dtype=torch.float32) * scale).to(dev)


def _gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x * math.sqrt(0.5)))


def _split_ref(x):
    """The bf16 pair of fp32 x: hi = RN(x), lo = RN(x - hi) (x - hi is exact)."""
    hi = x.bfloat16()
    return hi, (x - hi.float()).bfloat16()


def _split3_ref(x, weight_layout):
    hi, lo = _split_ref(x)
    return torch.cat([hi, hi, lo] if weight_layout else [hi, lo, hi], dim=-1)


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(I16), b.contiguous().view(I16))


def _decode3(t3, cols):
    """[hi | lo | hi] -> hi + lo in fp64; the third block must repeat the first bit for bit."""
    assert _same_bits(t3[..., :cols], t3[..., 2 * cols:]), "split output: third block differs from the first"
    return t3[..., :cols].double() + t3[..., cols:2 * cols].double()


def _check(what, err, bound, twin=None):
    """err <= bound, and (with a bf16 twin's error) twin >= 64 * err.  Prints the numbers for the record."""
    msg = f"{what}: f32x3 {err:.3e} (bound {bound:.1e})"
    if twin is not None:
        msg += f", bf16 twin {twin:.3e} (x{twin / max(err, 1e-300):.0f})"
    print("[f32x3] " + msg)
    assert err <= bound, msg
    if twin is not None:
        assert twin >= TWIN_RATIO * err, msg + f": the bf16 twin is not {TWIN_RATIO:.0f}x worse"


def _gemm_err(out, ref, mag, rows=None):
    """(max, median) of |out - ref| / mag over the selected rows."""
    e = ((out.double() - ref) / mag)
    if rows is not None:
        e = e[rows]
    e = e.abs().float().flatten()
    return e.max().item(), e.median().item()


# ================================================================================================ 1. split3
SPLIT3_SHAPES = [(1, 1), (7, 40), (999, 768), (40000, 1024)]     # 40000 x 1024 > the 8192 x 256 grid: stride loop


def _split3_input(rows, cols, dev, seed):
    """N(0,1) scaled by 2^[-20, 20] per row, with exact-in-bf16 values (lo == 0) and +-0 mixed in."""
    x = _randn((rows, cols), dev, seed)
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    x *= torch.pow(2.0, torch.randint(-20, 21, (rows, 1), generator=g).float()).to(dev)
    x[:, 3::7] = x[:, 3::7].bfloat16().float()
    x[:, 0] = 0.0
    if cols > 1:
        x[:, 1] = -0.0
    return x


@pytest.mark.parametrize("weight_layout", [0, 1])
@pytest.mark.parametrize("rows,cols", SPLIT3_SHAPES)
def test_split3_bit_exact(cuda, rows, cols, weight_layout):
    x = _split3_input(rows, cols, cuda, rows + cols)
    ref = _split3_ref(x, weight_layout)
    assert _same_bits(accurate.split3(x, weight_layout=bool(weight_layout)), ref)
    assert _same_bits(ops.split3_bf16(x, weight_layout=bool(weight_layout)), ref)
    for scale in (0.125, 0.7):      # the q block of the fused QKV weight is split with the softmax scale folded in
        ref_s = _split3_ref(x * scale, weight_layout)
        assert _same_bits(accurate.split3(x, weight_layout=bool(weight_layout), scale=scale), ref_s), scale
    hi, lo = _split_ref(x)
    assert bool((lo[:, 3::7].float() == 0).all()) and _same_bits(hi[:, 3::7], x[:, 3::7].bfloat16())


@pytest.mark.parametrize("weight_layout", [0, 1])
def test_split3_strided_rows(cuda, weight_layout):
    """ld_in > cols through the C entry: the gap columns hold NaN and must never be read."""
    rows, cols, ld = 3001, 320, 352
    full = _split3_input(rows, ld, cuda, 5)
    full[:, cols:] = float("nan")
    out = torch.empty((rows, 3 * cols), dtype=torch.bfloat16, device=cuda)
    _lib.check(_lib.load().aptai_split3_bf16(full.data_ptr(), rows, cols, ld, weight_layout, 0.7, out.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "split3_bf16")
    assert _same_bits(out, _split3_ref(full[:, :cols] * 0.7, weight_layout))


# ================================================================================================ 2. rowop
ROWOP_BOUND = 1e-6          # measured 2.7e-7 (256 columns, LayerNorm + GELU); bf16 twin >= 2.2e-3
ROWOP_SPLIT_BOUND = 2.5e-5  # measured 6.8e-6: hi + lo carries 16 significant bits (2^-17 relative)


def _rowop_ref(x64, gamma, beta, norm, gelu, eps=1e-5):
    y, scale = x64, torch.ones_like(x64[:, :1])
    if norm:
        mean = x64.mean(-1, keepdim=True)
        xc = x64 - mean
        var = (xc * xc).mean(-1, keepdim=True)
        y = xc / torch.sqrt(var + eps) * gamma.double() + beta.double()
        scale = 1.0 + mean.abs() / var.sqrt()       # fp32 mean error grows with |mean| / std
    if gelu:
        y = _gelu64(y)
    return y, scale


@pytest.mark.parametrize("rows", [1, 7, 8, 9, 1001, 40000])
@pytest.mark.parametrize("cols", [256, 512, 768, 1024])
def test_rowop_layernorm_gelu(cuda, cols, rows):
    """Every third row is 300 + N(0, 1): a one-pass E[x^2] - mean^2 variance loses ~1e-2 of the variance there."""
    x = _randn((rows, cols), cuda, cols + rows)
    x *= _randn((rows, 1), cuda, 7).abs() + 0.1
    x[0::3] = 300.0 + _randn((len(range(0, rows, 3)), cols), cuda, 9)
    gamma = 1.0 + _randn((cols,), cuda, 11, 0.2)
    beta = _randn((cols,), cuda, 12, 0.2)
    x64 = x.double()
    for norm in (0, 1):
        for gelu in (0, 1):
            what = f"rowop cols={cols} rows={rows} norm={norm} gelu={gelu}"
            g, b = (gamma, beta) if norm else (None, None)
            o32, o3 = accurate.rowop(x, g, b, gelu=bool(gelu), want_f32=True, want_split=True)
            ref, scale = _rowop_ref(x64, gamma, beta, norm, gelu)
            denom = (1.0 + ref.abs()) * scale
            err = ((o32.double() - ref).abs() / denom).max().item()
            twin = None
            if norm and not gelu:
                tw, _ = ops.layernorm(x.bfloat16(), gamma, beta, 1e-5, want_f32=True, want_bf16=False)
                twin = ((tw.double() - ref).abs() / denom).max().item()
            _check(what, err, ROWOP_BOUND, twin)
            # the split output is split3 of the kernel's own fp32 result, and the same without the fp32 output
            assert _same_bits(o3, _split3_ref(o32, 0)), what
            _, o3b = accurate.rowop(x, g, b, gelu=bool(gelu), want_f32=False, want_split=True)
            assert _same_bits(o3b, o3), what
            e3 = ((_decode3(o3, cols) - ref).abs() / denom).max().item()
            _check(what + " split", e3, ROWOP_SPLIT_BOUND)


def test_rowop_rejects_unsupported_width(cuda):
    x = torch.zeros((8, 640), device=cuda)
    with pytest.raises(RuntimeError, match=r"cols=640 unsupported \(256, 512, 768, 1024\)"):
        accurate.rowop(x, None, None, gelu=True)


# ================================================================================================ 3. conv0
CONV0_BOUND = 2.5e-5        # measured 6.4e-6 (hi + lo, GroupNorm); bf16 twin >= 1.7e-3
# (B, L, valid samples per utterance): T0 = 3199, 3199, 257, 79, 1, 64, 65
CONV0_CASES = [(3, 16000, [16000, 11111, 4000]), (2, 16003, None), (5, 1290, None), (1, 400, None), (1, 10, None),
               (2, 325, None), (3, 330, [330, 200, 330])]


@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("norm", [0, 1, 2])
@pytest.mark.parametrize("B,L,lens", CONV0_CASES)
def test_conv0_accurate(cuda, B, L, lens, norm, bias):
    T0 = (L - 10) // 5 + 1
    if norm == 2 and T0 == 1:
        pytest.skip("GroupNorm over a single frame has zero variance")
    wav = _randn((B, L), cuda, L + B)
    wav *= torch.tensor([0.05, 1.0, 0.3, 2.0, 0.01][:B], device=cuda)[:, None]      # per-utterance amplitude
    wav[0] += 0.5                                                                  # a DC offset
    if lens is not None:
        for b, n in enumerate(lens):
            wav[b, n:] = 0.0
    w = _randn((512, 10), cuda, 21, 0.3)
    b_ = _randn((512,), cuda, 22, 0.1) if bias else None
    gamma = 1.0 + _randn((512,), cuda, 23, 0.2) if norm else None
    beta = _randn((512,), cuda, 24, 0.2) if norm else None
    out = accurate.conv0(wav, w, b_, gamma, beta, norm)
    y = F.conv1d(wav.double()[:, None], w.double()[:, None, :], None if b_ is None else b_.double(), stride=5)
    if norm == 1:
        y = F.layer_norm(y.transpose(1, 2), (512,), gamma.double(), beta.double(), 1e-5).transpose(1, 2)
    elif norm == 2:
        y = F.group_norm(y, 512, gamma.double(), beta.double(), 1e-5)
    ref = _gelu64(y).transpose(1, 2)
    assert out.shape == (B, T0, 1536)
    err = ((_decode3(out, 512) - ref).abs() / (1.0 + ref.abs())).max().item()
    twin_out = ops.conv0(wav, w, b_, gamma, beta, norm)
    twin = ((twin_out.double() - ref).abs() / (1.0 + ref.abs())).max().item()
    _check(f"conv0 B={B} L={L} norm={norm} bias={bias}", err, CONV0_BOUND, twin)


# ================================================================================================ 4. gelu_add
GELU_ADD_BOUND = 1.2e-6     # measured 3.0e-7 (the erfc approximation of gelu_erf, ptx.cuh)


@pytest.mark.parametrize("n", [1, 3003, 5_000_001])          # 5e6 > the 8192 x 256 grid
def test_gelu_add(cuda, n):
    x = _randn((n,), cuda, n, 3.0)
    res = _randn((n,), cuda, n + 1)
    ref = res.double() + _gelu64(x.double())
    out = accurate.gelu_add(x, res)
    err = ((out.double() - ref).abs() / (1.0 + ref.abs())).max().item()
    _check(f"gelu_add n={n}", err, GELU_ADD_BOUND)
    h = res.clone()
    assert accurate.gelu_add(x, h, out=h) is h           # in place, as encode uses it
    assert torch.equal(h, out)


# ================================================================================================ 5. cast_pad_split
@pytest.mark.parametrize("T", [1, 24, 199, 999])              # T = 999: (999 + 128) x 1024 > the 4096 x 256 grid
@pytest.mark.parametrize("segs", [1, 3])
def test_cast_pad_split(cuda, segs, T):
    """Interior = the torch split bit for bit; both halos exactly zero.  The input is a view of a larger buffer whose
    next row is nonzero, so a row read past an utterance's end shows up in its trailing halo even for the last one."""
    H, halo = 1024, 64
    buf = _randn((segs + 1, T, H), cuda, T + segs)
    buf += torch.where(buf >= 0, 1.0, -1.0)                  # |x| >= 1: no element is zero
    x = buf[:segs]
    hi, lo = accurate.cast_pad_split(x, halo)
    assert hi.shape == lo.shape == (segs, T + 2 * halo, H)
    rh, rl = _split_ref(x)
    assert _same_bits(hi[:, halo:halo + T], rh) and _same_bits(lo[:, halo:halo + T], rl)
    for t in (hi, lo):
        for part in (t[:, :halo], t[:, halo + T:]):
            assert bool((part.contiguous().view(I16) == 0).all()), "cast_pad_split: nonzero halo row"


# ================================================================================================ 6. posconv_fold_split
FOLD_BOUND = 3e-5           # measured 7.8e-6 relative (hi + lo); bf16 twin >= 3.9e-3


@pytest.mark.parametrize("H,groups", [(1024, 16), (768, 16), (256, 4)])
def test_posconv_fold_split(cuda, H, groups):
    cin, taps, cpad = H // groups, 128, 64
    g = 0.5 + _randn((1, 1, taps), cuda, 31).abs()
    v = _randn((H, cin, taps), cuda, 32)
    hi, lo = accurate.posconv_fold_split(g, v)
    w = g.double() * v.double() / torch.linalg.vector_norm(v.double(), dim=(0, 1), keepdim=True)
    ref = w.permute(0, 2, 1)                                              # [H, taps, cin]
    hi3, lo3 = hi.view(H, taps, cpad), lo.view(H, taps, cpad)
    for t in (hi3, lo3):
        assert bool((t[:, :, cin:].contiguous().view(I16) == 0).all()), "posconv_fold_split: nonzero padding column"
    err = ((hi3[:, :, :cin].double() + lo3[:, :, :cin].double() - ref).abs() / ref.abs()).max().item()
    tw = ops.posconv_fold(g, v).view(H, taps, cpad)[:, :, :cin]
    twin = ((tw.double() - ref).abs() / ref.abs()).max().item()
    _check(f"posconv_fold_split H={H} groups={groups}", err, FOLD_BOUND, twin)


# ================================================================================================ 7. attention_f32
ATTN_BOUND = 8e-6           # measured 2.1e-6 of max|v| (T = 513, keys x4); bf16 twin >= 2.6e-3
ATTN_CASES = [(2, 199, 16, [199, 150]), (3, 64, 12, [64, 1, 33]), (1, 999, 16, [999]), (2, 513, 4, [513, 400]),
              (3, 257, 2, [257, 256, 129]), (2, 33, 2, [33, 32]), (1, 1, 16, [1])]


@pytest.mark.parametrize("B,T,heads,key_len", ATTN_CASES)
def test_attention_f32(cuda, B, T, heads, key_len):
    """Every query row (padded queries too, as in HF) against fp64 softmax(q k^T + key mask) v."""
    H = heads * 64
    qkv = _randn((B, T, 3, H), cuda, T + heads)
    qkv[:, :, 0] *= 0.3                                   # q pre-scaled, as the fused QKV weights do
    if T == 513:
        qkv[:, 256:, 1] *= 4.0                            # later keys dominate: the running maximum moves
    qkv = qkv.view(B * T, 3 * H).contiguous()
    kl = torch.tensor(key_len, dtype=I32, device=cuda)
    ctx = accurate.attention_f32(qkv, kl, B, T, heads)
    q, k, v = qkv.double().view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    s = q @ k.transpose(-1, -2)
    s = s.masked_fill(torch.arange(T, device=cuda)[None, None, None, :] >= kl[:, None, None, None].long(),
                      float("-inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * T, H)
    vmax = v.abs().max()
    err = ((ctx.double() - ref).abs().max() / vmax).item()
    tw = ops.attention(qkv.bfloat16(), kl, B, T, heads)
    twin = ((tw.double() - ref).abs().max() / vmax).item()
    _check(f"attention_f32 B={B} T={T} heads={heads} key_len={key_len}", err, ATTN_BOUND, twin)


# ================================================================================================ 8. split-operand GEMMs
GEMM_BOUND_MAX = 1.3e-5     # measured 3.3e-6 (M = 25536, 4096 -> 1024, in place)
GEMM_BOUND_MED = 1.3e-6     # measured 3.2e-7; bf16 twin medians >= 2.4e-5
# (K, N, epilogue): the encoder's Linears at H = 1024 and their 768-wide twins
GEMM_SHAPES = [(512, 1024, "ragged"), (1024, 3072, "plain"), (1024, 1024, "residual"), (1024, 4096, "gelu"),
               (4096, 1024, "inplace"), (512, 768, "ragged"), (768, 2304, "plain"), (768, 768, "residual"),
               (768, 3072, "gelu"), (3072, 768, "inplace")]
# M -> (rows per utterance, valid rows per utterance) of the ragged feature projection
GEMM_M = {1: (1, [1]), 129: (43, [43, 1, 20]), 700: (350, [350, 201]),
          25536: (399, [399] + [int(v) for v in torch.randint(1, 400, (63,),
                                                               generator=torch.Generator().manual_seed(5))])}


def _gemm_case(M, K, N, dev, seed):
    x = _randn((M, K), dev, seed)
    w = _randn((N, K), dev, seed + 1, K ** -0.5)
    b = _randn((N,), dev, seed + 2, 0.1)
    acc = x.double() @ w.double().T
    mag = x.double().abs() @ w.double().abs().T + b.double().abs()
    return x, w, b, acc + b.double(), mag


@pytest.mark.parametrize("M", list(GEMM_M))
@pytest.mark.parametrize("K,N,kind", GEMM_SHAPES)
def test_linear3(cuda, K, N, kind, M):
    x, w, b, ref, mag = _gemm_case(M, K, N, cuda, K + N + M)
    x3, w3 = accurate.split3(x), accurate.split3(w, weight_layout=True)
    xb, wb = x.bfloat16(), w.bfloat16()
    kw, rows = {}, None
    if kind == "ragged":
        seg, valid = GEMM_M[M]
        kw = dict(seg_rows=seg, seg_valid_rows=torch.tensor(valid, dtype=I32, device=cuda))
        rows = (torch.arange(M, device=cuda) % seg) < kw["seg_valid_rows"].long().repeat_interleave(seg)
    elif kind == "gelu":
        kw = dict(act=1)
        ref = _gelu64(ref)
    elif kind in ("residual", "inplace"):
        r = _randn((M, N), cuda, M + 3)
        ref, mag = ref + r.double(), mag + r.double().abs()
    if kind == "residual":
        out = accurate.linear3(x3, w3, b, residual=r)
        tw = ops.linear(xb, wb, b, residual=r, want_f32=True, want_bf16=False)[0]
    elif kind == "inplace":
        h = r.clone()
        out = accurate.linear3(x3, w3, b, residual=h, out_f32=h)
        assert out.data_ptr() == h.data_ptr()
        h2 = r.clone()
        tw = ops.linear(xb, wb, b, residual=h2, out_f32=h2, want_f32=True, want_bf16=False)[0]
    else:
        out = accurate.linear3(x3, w3, b, **kw)
        tw = ops.linear(xb, wb, b, want_f32=True, want_bf16=False, **kw)[0]
    if rows is not None:
        assert bool((out[~rows] == 0).all()) and bool((out[~rows].view(I32) == 0).all()), "padded rows not zero"
    e_max, e_med = _gemm_err(out, ref, mag, rows)
    t_max, t_med = _gemm_err(tw, ref, mag, rows)
    what = f"linear3 M={M} {K}->{N} {kind}"
    _check(what + " max", e_max, GEMM_BOUND_MAX)
    _check(what + " median", e_med, GEMM_BOUND_MED, t_med)


@pytest.mark.parametrize("K,N", [(1024, 128), (256, 2048), (512, 256)])     # frame_lin, BiLSTM input, RNN head
def test_linear_f32x3_default_path(cuda, K, N):
    M = 64 * 399
    x, w, b, ref, mag = _gemm_case(M, K, N, cuda, K + N)
    out = ops.linear_f32x3(x, w, b)
    tw = ops.linear(x.bfloat16(), w.bfloat16(), b, want_f32=True, want_bf16=False)[0]
    e_max, e_med = _gemm_err(out, ref, mag)
    t_max, t_med = _gemm_err(tw, ref, mag)
    _check(f"linear_f32x3 {K}->{N} max", e_max, GEMM_BOUND_MAX)
    _check(f"linear_f32x3 {K}->{N} median", e_med, GEMM_BOUND_MED, t_med)


@pytest.mark.parametrize("T_in", [801, 640, 399, 3])
@pytest.mark.parametrize("k", [3, 2])
def test_conv_igemm_split_operands(cuda, k, T_in):
    """Conv layers 1-6 of the accuracy mode: x3 = split3 of the fp32 activations (with the zeroed slack rows the
    strided view may touch), weights split per tap ([hi|hi|lo] over the 512 input channels), fp32 output."""
    B, C, s = 3, 512, 2
    x = _randn((B, T_in, C), cuda, T_in + k)
    w = _randn((C, C, k), cuda, k, (C * k) ** -0.5)
    b = _randn((C,), cuda, k + 1, 0.1)
    x3 = accurate.split3(x.view(B * T_in, C), slack_rows=2).view(B, T_in, 3 * C)
    w3 = accurate.split3(w.permute(0, 2, 1).reshape(C * k, C).contiguous(), weight_layout=True).view(C, k * 3 * C)
    T_out = (T_in - k) // s + 1
    out = torch.empty((B, T_out, C), dtype=torch.float32, device=cuda)
    ops.conv_igemm(x3, w3, b, k, s, act=0, out_f32=out)
    x64, w64 = x.double().transpose(1, 2), w.double()
    ref = F.conv1d(x64, w64, b.double(), stride=s).transpose(1, 2)
    mag = (F.conv1d(x64.abs(), w64.abs(), stride=s) + b.double().abs()[None, :, None]).transpose(1, 2)
    xb = ops.alloc_rows_bf16(B, T_in, C, cuda)
    xb.copy_(x.bfloat16())
    tw = torch.empty_like(out)
    ops.conv_igemm(xb, w.permute(0, 2, 1).reshape(C, k * C).bfloat16().contiguous(), b, k, s, act=0, out_f32=tw)
    e_max, e_med = _gemm_err(out, ref, mag)
    t_max, t_med = _gemm_err(tw, ref, mag)
    _check(f"conv_igemm k={k} T_in={T_in} max", e_max, GEMM_BOUND_MAX)
    _check(f"conv_igemm k={k} T_in={T_in} median", e_med, GEMM_BOUND_MED, t_med)


# ================================================================================================ 9. positional conv
POSCONV_BOUND_MAX = 6e-6    # measured 1.5e-6
POSCONV_BOUND_MED = 4.5e-7  # measured 1.1e-7; bf16 twin medians >= 5.2e-6


@pytest.mark.parametrize("T", [1, 24, 199, 999])
@pytest.mark.parametrize("H,groups", [(1024, 16), (768, 16), (256, 4)])
def test_pos_conv_three_pass(cuda, H, groups, T):
    """accurate.pos_conv_add (h_hi.w_hi + h_lo.w_hi + h_hi.w_lo, then h += gelu(. + b)) against the fp64 weight-normed
    grouped conv plus residual; the second utterance is shorter and its padded rows are zero, as in encode."""
    B, taps = 2, 128
    lens = [T, max(1, T // 2)]
    h = _randn((B, T, H), cuda, T + H)
    for i, n in enumerate(lens):
        h[i, n:] = 0.0
    g = 0.5 + _randn((1, 1, taps), cuda, 41).abs()
    v = _randn((H, H // groups, taps), cuda, 42)
    bias = _randn((H,), cuda, 43, 0.1)
    w64 = g.double() * v.double() / torch.linalg.vector_norm(v.double(), dim=(0, 1), keepdim=True)
    h64 = h.double().transpose(1, 2)
    pos = F.conv1d(h64, w64, bias.double(), padding=taps // 2, groups=groups)[:, :, :-1]
    ref = (h64 + _gelu64(pos)).transpose(1, 2)
    mag = (F.conv1d(h64.abs(), w64.abs(), padding=taps // 2, groups=groups)[:, :, :-1]
           + bias.double().abs()[None, :, None] + h64.abs()).transpose(1, 2)
    w_hi, w_lo = accurate.posconv_fold_split(g, v)
    out = h.clone()
    assert accurate.pos_conv_add(out, w_hi, w_lo, bias, groups, taps) is out
    tw = h.clone()
    ops.posconv(ops.cast_pad(h, taps // 2), ops.posconv_fold(g, v), bias, tw, T, H, groups, taps, tw)
    e_max, e_med = _gemm_err(out, ref, mag)
    t_max, t_med = _gemm_err(tw, ref, mag)
    _check(f"pos_conv_add H={H} T={T} max", e_max, POSCONV_BOUND_MAX)
    _check(f"pos_conv_add H={H} T={T} median", e_med, POSCONV_BOUND_MED, t_med)


# ================================================================================================ 10. encoder
def _cfg(variant, H, heads, F_, layers=2):
    kw = dict(hidden_size=H, num_hidden_layers=layers, num_attention_heads=heads, intermediate_size=F_,
              num_conv_pos_embedding_groups=16 if H > 256 else 4, hidden_dropout=0.0, activation_dropout=0.0,
              attention_dropout=0.0, feat_proj_dropout=0.0, final_dropout=0.0, layerdrop=0.0,
              apply_spec_augment=False)
    return W2V2Config.large(**kw) if variant == "layer" else W2V2Config.base(**kw)


def _encoder_errors(cfg, lens, cuda):
    """Max-abs error of every hidden state (all frames) against the fp64 oracle, f32x3 and bf16; the model."""
    sd = backbone_state_dict(cfg, seed=0)
    wav = waveforms(len(lens), max(lens), lens, seed=1234)
    ref = ow.forward({k: v.double() for k, v in sd.items()}, cfg, wav.double(), lens)
    m = Wav2Vec2Backbone(cfg)
    m.load_state_dict(sd, strict=True)
    m = m.to(cuda).eval()
    am = torch.tensor(lens, device=cuda)[:, None]
    errs = {}
    for mode in ("bf16", "f32x3"):
        m.set_precision(mode)
        out = m(wav.to(cuda), attention_mask=am, output_hidden_states=True)
        assert len(out.hidden_states) == len(ref) == cfg.num_hidden_layers + 1
        errs[mode] = [(o.double().cpu() - r).abs().max().item() for o, r in zip(out.hidden_states, ref)]
    return errs, m, wav, out


# max-abs bound over all hidden states = 4x the measured error (9.6e-5, 1.34e-4, 5.9e-5, 1.03e-4; bf16: 1.3e-2 to
# 2.3e-2).  The activations between the GEMMs are hi + lo pairs (16 significant bits, 2^-17 relative), not fp32, so the
# encoder lands about 10x above an fp32 forward's 4-9e-6.
E2E_CASES = [("layer", 1024, 16, 4096, [64000, 20000], 4e-4), ("group", 768, 12, 3072, [32000, 20000], 5.5e-4),
             ("layer", 256, 4, 512, [8000, 400, 3217], 2.4e-4), ("group", 256, 4, 512, [8000, 400, 3217], 4e-4)]


@pytest.mark.parametrize("variant,H,heads,F_,lens,bound", E2E_CASES)
def test_encoder_f32x3_matches_fp64_oracle(cuda, variant, H, heads, F_, lens, bound):
    errs, _, _, _ = _encoder_errors(_cfg(variant, H, heads, F_), lens, cuda)
    what = f"encoder {variant} H={H} lens={lens}"
    print(f"[f32x3] {what}: per hidden state f32x3 {errs['f32x3']}, bf16 {errs['bf16']}")
    _check(what, max(errs["f32x3"]), bound, max(errs["bf16"]))


def test_encoder_f32x3_20s(cuda):
    """20 s (999 frames) next to 2 s; the 2 s utterance's valid frames must match the same waveform run alone."""
    cfg = _cfg("layer", 1024, 16, 4096)
    lens = [320000, 32000]
    errs, m, wav, out = _encoder_errors(cfg, lens, cuda)
    assert out.last_hidden_state.shape[1] == 999
    print(f"[f32x3] encoder 20 s: per hidden state f32x3 {errs['f32x3']}, bf16 {errs['bf16']}")
    _check("encoder 20 s", max(errs["f32x3"]), 4.5e-4, max(errs["bf16"]))     # measured 1.07e-4; bf16 2.1e-2
    alone = m(wav[1:2, :32000].contiguous().to(cuda), attention_mask=torch.tensor([[32000]], device=cuda))
    d = (out.last_hidden_state[1, :99] - alone.last_hidden_state[0, :99]).abs().max().item()
    _check("encoder 20 s: 2 s utterance batched vs alone", d, 1e-5)        # measured 0 (bit-identical)
