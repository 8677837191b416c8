"""Kernel-level parity of the kernels that run only in training: the conv feature encoder's backward (LayerNorm / GELU
backward, tcgen05 weight gradient, strided-output input gradient, conv-0 GroupNorm backward and im2col), attention
with dropout on the probabilities, and the small elementwise kernels of the backward.

Every reference is built in fp64 on the same 16-bit-rounded operands the kernel reads, so a tolerance only has to cover
the kernel's own rounding:
  * fp32-accumulated outputs (weight / input gradients, dgamma / dbeta): relative L2 <= 2e-5 (as test_wgrad), and every
    element within 1e-4 * max|ref| (a lost 64-frame block or a wrong row moves single elements by far more);
  * bf16 outputs: within 2^-8 * |ref| (bf16 rounding) plus a floor of 2e-5 * the largest |ref| of the row (or, for
    GroupNorm, the channel) for elements where LayerNorm's d - mean(d) - xhat * mean(d * xhat) cancels.  The floor
    covers fp32 arithmetic and the ~2e-7 absolute error of the kernels' erf-based GELU derivative.
The attention-dropout mask is restated on the host (numpy uint32) from its definition; the dropout tests use that
restatement, never the device's replay kernel.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from aptai_b200 import lib as _lib
from aptai_b200 import ops

F64 = torch.float64
C = 512
LOG2E = 1.4426950408889634
BF16_REL = 2.0 ** -8


def _rand(shape, dev, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


def _rel(out, ref):
    return ((out.double() - ref.double()).norm() / ref.double().norm().clamp_min(1e-300)).item()


def _check_f32_acc(out, ref, what):
    """fp32-accumulated output: relative L2 <= 2e-5 and every element within 1e-4 * max|ref|."""
    out, ref = out.double(), ref.double()
    r = _rel(out, ref)
    e = ((out - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()
    assert r <= 2e-5 and e <= 1e-4, f"{what}: relative L2 {r:.3e}, max error / max|ref| {e:.3e}"


def _check_bf16(out, ref, scale, what):
    """bf16 output: |out - ref| <= 2^-8 |ref| + 2e-5 * scale (scale broadcasts: the row's or channel's max|ref|)."""
    out, ref = out.double(), ref.double()
    err = (out - ref).abs()
    bound = BF16_REL * ref.abs() + 2e-5 * scale
    ratio = err / bound.clamp_min(1e-300)
    worst = np.unravel_index(int(ratio.argmax()), tuple(ratio.shape))
    assert bool((err <= bound).all()), f"{what}: worst error / bound {ratio.max().item():.3e} at {worst}"


def _gelu_grad(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def _pitched(rows_per_seg, pitch, segs, dev, seed):
    """dy fp32 [segs*pitch, 512] with NaN in the gap rows (which must never be read), and its logical rows."""
    dy = _rand((segs, pitch, C), dev, 1.0, seed)
    dy[:, rows_per_seg:] = float("nan")
    return dy.view(segs * pitch, C), dy[:, :rows_per_seg].reshape(segs * rows_per_seg, C)


def _storage_tail(t, n_main):
    """The elements behind the first n_main of t's allocation (the slack rows of ops.alloc_rows_bf16)."""
    flat = torch.empty(0, dtype=t.dtype, device=t.device).set_(t.untyped_storage())
    return flat[n_main:]


# ---------------------------------------------------------------------------------------------- fp64 conv references
def _tap_rows(T_out, stride, tap):
    return slice(tap, tap + stride * (T_out - 1) + 1, stride)


def _conv_wgrad64(dz, x, k, stride):
    """dW [O, k*C] (tap-major) = sum_{b,t} dz[b,t,o] x[b, t*stride + tap, c];  dz [B,T_out,O], x [B,T_in,C] fp64."""
    B, T_out, O = dz.shape
    d = dz.reshape(-1, O)
    return torch.cat([d.t() @ x[:, _tap_rows(T_out, stride, tap)].reshape(-1, x.shape[2]) for tap in range(k)], 1)


def _conv_dgrad64(dz, w, stride, T_pad):
    """dx [B, T_pad, C]: dx[b, t*stride + tap] += dz[b, t] @ w[:, :, tap];  w [O, C, k] fp64 (the conv weight)."""
    B, T_out, _ = dz.shape
    dx = torch.zeros((B, T_pad, w.shape[1]), dtype=dz.dtype, device=dz.device)
    for tap in range(w.shape[2]):
        dx[:, _tap_rows(T_out, stride, tap)] += dz @ w[:, :, tap]
    return dx


def test_conv_references_match_torch_autograd():
    """The per-tap fp64 helpers against F.conv1d autograd on CPU (both layer geometries, both parities of T_in)."""
    g = torch.Generator().manual_seed(0)
    for k, s, T_in in ((3, 2, 11), (3, 2, 12), (2, 2, 10), (2, 2, 11)):
        x = torch.randn((2, T_in, 8), generator=g, dtype=F64, requires_grad=True)
        w = torch.randn((6, 8, k), generator=g, dtype=F64, requires_grad=True)
        y = F.conv1d(x.transpose(1, 2), w, stride=s).transpose(1, 2)
        dz = torch.randn(y.shape, generator=g, dtype=F64)
        y.backward(dz)
        T_pad = (T_in + s - 1) // s * s
        dx = _conv_dgrad64(dz, w.detach(), s, T_pad)
        torch.testing.assert_close(dx[:, :T_in], x.grad, atol=1e-12, rtol=1e-12)
        assert dx[:, T_in:].abs().max().item() == 0 if T_pad > T_in else True
        dw = _conv_wgrad64(dz, x.detach(), k, s)
        torch.testing.assert_close(dw, w.grad.permute(0, 2, 1).reshape(6, -1), atol=1e-12, rtol=1e-12)


# ---------------------------------------------------------------------------------------- A. conv feature encoder
def _ln_params(dev, seed):
    gamma = _rand((C,), dev, 0.3, seed) + 1.0
    beta = _rand((C,), dev, 0.3, seed + 1)
    return gamma, beta


@pytest.mark.parametrize("B,T", [(1, 1), (2, 999), (3, 12799)])
def test_ln_gelu_fwd(cuda, B, T):
    z = (_rand((B, T, C), cuda, 2.0, 1) + 0.5).bfloat16()
    gamma, beta = _ln_params(cuda, 2)
    y = ops.ln_gelu_fwd(z, gamma, beta)
    ref = F.gelu(F.layer_norm(z.double(), (C,), gamma.double(), beta.double(), 1e-5))
    _check_bf16(y, ref, ref.abs().amax(-1, keepdim=True), "ln_gelu_fwd y")
    assert _storage_tail(y, B * T * C).abs().max().item() == 0, "slack rows behind the output must stay zero"


def _ln_gelu_bwd_ref(z64, dy64, gamma, beta):
    zr = z64.detach().requires_grad_(True)
    gr, br = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    F.gelu(F.layer_norm(zr, (C,), gr, br, 1e-5)).backward(dy64)
    return zr.grad, gr.grad, br.grad


def _check_ln_gelu_bwd(dz, dg, db, refs, dg0, db0):
    rdz, rdg, rdb = refs
    _check_bf16(dz, rdz, rdz.abs().amax(-1, keepdim=True), "ln_gelu_bwd dz")
    _check_f32_acc(dg, dg0.double() + rdg, "ln_gelu_bwd dgamma (accumulated)")
    _check_f32_acc(db, db0.double() + rdb, "ln_gelu_bwd dbeta (accumulated)")


# segs x rows_per_seg at row pitch seg_pitch: odd rows with a gap row, one row, and more rows than one grid sweep
# (8 rows per block, at most 8 blocks per SM)
@pytest.mark.parametrize("segs,rows_per_seg,seg_pitch", [(1, 1, 2), (2, 999, 1000), (3, 12799, 12800)])
def test_ln_gelu_bwd(cuda, segs, rows_per_seg, seg_pitch):
    rows = segs * rows_per_seg
    z = (_rand((rows, C), cuda, 2.0, 1) - 0.3).bfloat16()
    gamma, beta = _ln_params(cuda, 2)
    dy, dy_log = _pitched(rows_per_seg, seg_pitch, segs, cuda, 3)
    dg0, db0 = torch.full((C,), 0.5, device=cuda), torch.full((C,), -0.25, device=cuda)
    dg, db = dg0.clone(), db0.clone()
    dz = ops.ln_gelu_bwd(dy, rows_per_seg, seg_pitch, segs, gamma, beta, 1e-5, dg, db, z=z)
    _check_ln_gelu_bwd(dz, dg, db, _ln_gelu_bwd_ref(z.double(), dy_log.double(), gamma, beta), dg0, db0)


def _conv0_64(wav, w0, bias0):
    """fp64 conv layer 0 (k=10, s=5): [B, L] -> [B, T0, 512]."""
    return F.conv1d(wav.double()[:, None], w0.double()[:, None, :], None if bias0 is None else bias0.double(),
                    stride=5).transpose(1, 2)


def test_conv0_reference_matches_explicit_frames():
    g = torch.Generator().manual_seed(0)
    wav, w0, b0 = torch.randn((2, 53), generator=g), torch.randn((C, 10), generator=g), torch.randn((C,), generator=g)
    frames = wav.double().unfold(1, 10, 5)                                     # [B, T0, 10]
    torch.testing.assert_close(_conv0_64(wav, w0, b0), frames @ w0.double().t() + b0.double(), atol=1e-12, rtol=1e-12)


@pytest.mark.parametrize("L", [16003, 16010])              # (L - 10) % 5 != 0 and == 0
def test_ln_gelu_bwd_conv0_from_waveform(cuda, L):
    B = 2
    T0 = (L - 10) // 5 + 1
    pitch = T0 + 3
    wav = _rand((B, L), cuda, 0.3, 1)
    w0 = _rand((C, 10), cuda, 0.3, 2)
    bias0 = _rand((C,), cuda, 0.1, 3)
    gamma, beta = _ln_params(cuda, 4)
    dy, dy_log = _pitched(T0, pitch, B, cuda, 6)
    dg0, db0 = torch.full((C,), -0.75, device=cuda), torch.full((C,), 0.125, device=cuda)
    dg, db = dg0.clone(), db0.clone()
    dz = ops.ln_gelu_bwd(dy, T0, pitch, B, gamma, beta, 1e-5, dg, db, wav=wav, w0t=w0.t().contiguous(), bias0=bias0)
    z64 = _conv0_64(wav, w0, bias0).reshape(B * T0, C)
    _check_ln_gelu_bwd(dz, dg, db, _ln_gelu_bwd_ref(z64, dy_log.double(), gamma, beta), dg0, db0)


def test_ln_gelu_bwd_rejects_a_waveform_too_short_for_the_frames(cuda):
    """Frame t of conv 0 reads samples 5t .. 5t+9: one frame more than the waveform holds is an argument error.  The
    waveform is a view at the front of a longer buffer, so that even an unchecked call would stay inside it."""
    B, L = 2, 16003
    T0 = (L - 10) // 5 + 1
    flat = torch.zeros((B * L + 512,), device=cuda)
    wav = flat[: B * L].view(B, L)
    w0t = _rand((10, C), cuda, 0.3, 1)
    gamma, beta = _ln_params(cuda, 2)
    dg, db = torch.zeros((C,), device=cuda), torch.zeros((C,), device=cuda)
    dy = torch.zeros((B * (T0 + 1), C), device=cuda)
    with pytest.raises(RuntimeError, match="ln_gelu_bwd"):
        ops.ln_gelu_bwd(dy, T0 + 1, T0 + 1, B, gamma, beta, 1e-5, dg, db, wav=wav, w0t=w0t, bias0=None)
    ops.ln_gelu_bwd(dy[: B * T0], T0, T0, B, gamma, beta, 1e-5, dg, db, wav=wav, w0t=w0t, bias0=None)
    torch.cuda.synchronize()


def _conv_case(cuda, B, T_out, k, s, odd):
    """Inputs of one strided conv layer: T_in of the requested parity that yields T_out frames."""
    T_in = s * (T_out - 1) + k
    if (T_in % 2 == 1) != odd:
        T_in += 1                                           # one more input row, still T_out output frames
    assert (T_in - k) // s + 1 == T_out
    x = ops.alloc_rows_bf16(B, T_in, C, cuda)
    x.copy_(_rand((B, T_in, C), cuda, 1.0, 11).bfloat16())
    dz = _rand((B, T_out, C), cuda, 1.0, 12).bfloat16()
    w = _rand((C, C, k), cuda, 0.05, 13)                   # conv weight [out, in, tap]
    return x, dz, w, T_in


CONV_GEOMETRY = [(3, 2), (2, 2)]                             # layers 1-4, layers 5-6
CONV_T_OUT = [1, 2, 63, 64, 65, 128, 129, 999]


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("T_out", CONV_T_OUT)
@pytest.mark.parametrize("odd", [True, False])
@pytest.mark.parametrize("k,s", CONV_GEOMETRY)
def test_conv_wgrad(cuda, k, s, odd, T_out, B):
    x, dz, _, T_in = _conv_case(cuda, B, T_out, k, s, odd)
    dw = ops.conv_wgrad(dz, x, k, s)
    _check_f32_acc(dw, _conv_wgrad64(dz.double(), x.double(), k, s), f"conv_wgrad T_in={T_in}")


def test_conv_wgrad_full_size_layer1(cuda):
    """A 20 s utterance at layer 1: T_in = 63999, T_out = 31999 (500 frame blocks split across CTAs)."""
    x, dz, _, T_in = _conv_case(cuda, 1, 31999, 3, 2, True)
    assert T_in == 63999
    dw = ops.conv_wgrad(dz, x, 3, 2)
    _check_f32_acc(dw, _conv_wgrad64(dz.double(), x.double(), 3, 2), "conv_wgrad layer 1, 20 s")


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("T_out", CONV_T_OUT)
@pytest.mark.parametrize("odd", [True, False])
@pytest.mark.parametrize("k,s", CONV_GEOMETRY)
def test_conv_dgrad(cuda, k, s, odd, T_out, B):
    _, dz, w, T_in = _conv_case(cuda, B, T_out, k, s, odd)
    wt_taps = [w[:, :, tap].t().contiguous().bfloat16() for tap in range(k)]       # as backbone's conv_wt
    dx, T_pad = ops.conv_dgrad(dz, wt_taps, k, s, T_in)
    assert T_pad == (T_in + s - 1) // s * s and dx.shape == (B, T_pad, C)
    ref = _conv_dgrad64(dz.double(), w.bfloat16().double(), s, T_pad)
    _check_f32_acc(dx[:, :T_in], ref[:, :T_in], f"conv_dgrad T_in={T_in}")
    assert T_pad == T_in or dx[:, T_in:].abs().max().item() == 0, "rows T_in .. T_pad-1 must be exactly zero"


@pytest.mark.parametrize("segs,rows_per_seg,seg_pitch", [(1, 1, 2), (2, 999, 1000), (3, 12799, 12800)])
def test_gelu_bwd_rows(cuda, segs, rows_per_seg, seg_pitch):
    rows = segs * rows_per_seg
    z = _rand((rows, C), cuda, 2.0, 1).bfloat16()
    dy, dy_log = _pitched(rows_per_seg, seg_pitch, segs, cuda, 2)
    dz = ops.gelu_bwd_rows(dy, rows_per_seg, seg_pitch, segs, z)
    ref = dy_log.double() * _gelu_grad(z.double())
    _check_bf16(dz, ref, ref.abs().amax(-1, keepdim=True), "gelu_bwd_rows dz")


def test_groupnorm_reference_is_per_utterance():
    """GroupNorm(512 groups) normalises each utterance on its own: per-utterance autograd (what the GroupNorm tests
    compare with) sums to the batched F.group_norm gradients."""
    g = torch.Generator().manual_seed(0)
    z = torch.randn((3, 8, 40), generator=g, dtype=F64, requires_grad=True)
    gam = torch.randn((8,), generator=g, dtype=F64, requires_grad=True)
    bet = torch.randn((8,), generator=g, dtype=F64, requires_grad=True)
    dy = torch.randn((3, 8, 40), generator=g, dtype=F64)
    F.gelu(F.group_norm(z, 8, gam, bet, 1e-5)).backward(dy)
    dz, dgam, dbet = _groupnorm_gelu_ref(z.detach(), dy, gam.detach(), bet.detach())
    torch.testing.assert_close(dz, z.grad, atol=1e-12, rtol=1e-12)
    torch.testing.assert_close(dgam.sum(0), gam.grad, atol=1e-12, rtol=1e-12)
    torch.testing.assert_close(dbet.sum(0), bet.grad, atol=1e-12, rtol=1e-12)


def _groupnorm_gelu_ref(z, dy, gamma, beta):
    """Autograd of GELU(GroupNorm(z)) per utterance: z, dy [B, C, T] fp64 -> (dz, dgamma [B, C], dbeta [B, C])."""
    dz, dg, db = [], [], []
    for b in range(z.shape[0]):
        zb = z[b: b + 1].clone().requires_grad_(True)
        gb, bb = gamma.double().clone().requires_grad_(True), beta.double().clone().requires_grad_(True)
        F.gelu(F.group_norm(zb, z.shape[1], gb, bb, 1e-5)).backward(dy[b: b + 1])
        dz.append(zb.grad[0]); dg.append(gb.grad); db.append(bb.grad)
    return torch.stack(dz), torch.stack(dg), torch.stack(db)


def test_conv0_groupnorm_bwd(cuda):
    """Conv 0 + GroupNorm over time + GELU ('group' variant), statistics over all T0 frames of zero-tailed rows.
    Channel 0 has gamma = 0, channels 1 / 2 gamma = +-1e-4 with |beta| = 8, channels 3..9 negative gamma."""
    B, L = 2, 16003
    T0 = (L - 10) // 5 + 1
    pitch = T0 + 1
    wav = _rand((B, L), cuda, 0.3, 1)
    wav[1, 11000:] = 0.0
    w0 = _rand((C, 10), cuda, 0.3, 2)
    bias0 = _rand((C,), cuda, 0.1, 3)
    gamma, beta = _ln_params(cuda, 4)
    gamma[0], beta[0] = 0.0, 2.0
    gamma[1], beta[1] = 1e-4, 8.0
    gamma[2], beta[2] = -1e-4, -8.0
    gamma[3:10] = -gamma[3:10]
    _, ws = ops.conv0(wav, w0, bias0, gamma, beta, 2, out_dtype=torch.bfloat16, return_ws=True)
    affine, norm_stats = ops.conv0_groupnorm_saved(ws, B)
    dy, dy_log = _pitched(T0, pitch, B, cuda, 5)
    dz, sums = ops.conv0_groupnorm_bwd(dy, pitch, wav, T0, w0, affine, norm_stats)
    z64 = _conv0_64(wav, w0, bias0).transpose(1, 2)                           # [B, C, T0]
    rdz, rdg, rdb = _groupnorm_gelu_ref(z64, dy_log.view(B, T0, C).double().transpose(1, 2), gamma, beta)
    rdz = rdz.transpose(1, 2)                                                  # [B, T0, C]
    # floor in units of |gamma * rstd * dy| (dz with GELU' = 1), per (utterance, channel): in the far tails (beta = -8)
    # the erf-based GELU derivative is accurate in absolute terms (~2e-17 at -8), not relative to its ~4e-14 value
    a64 = gamma.double() / (z64.var(-1, unbiased=False) + 1e-5).sqrt()             # [B, C]
    scale = a64.abs()[:, None, :] * dy_log.view(B, T0, C).double().abs().amax(1, keepdim=True)
    _check_bf16(dz.view(B, T0, C), rdz, scale, "conv0_groupnorm_bwd dz")
    for b in range(B):
        _check_f32_acc(sums[b, :, 0], rdb[b], f"conv0_groupnorm_bwd dbeta, utterance {b}")
        _check_f32_acc(sums[b, :, 1], rdg[b], f"conv0_groupnorm_bwd dgamma, utterance {b}")


@pytest.mark.parametrize("L", [16003, 16010])
def test_conv0_im2col_and_weight_gradient(cuda, L):
    B = 3
    T0 = (L - 10) // 5 + 1
    wav = _rand((B, L), cuda, 0.3, 1)
    X = ops.conv0_im2col(wav, T0)
    ref = torch.zeros((B, T0, 64), dtype=torch.bfloat16, device=cuda)
    ref[:, :, :10] = wav.bfloat16().unfold(1, 10, 5)
    assert torch.equal(X, ref.view(B * T0, 64))
    dz0 = _rand((B * T0, C), cuda, 1.0, 2).bfloat16()
    dw0 = torch.zeros((C, 64), device=cuda)
    ops.wgrad(dz0, X, dw0)
    frames = wav.bfloat16().double().unfold(1, 10, 5).reshape(B * T0, 10)
    _check_f32_acc(dw0[:, :10], dz0.double().t() @ frames, "conv-0 weight gradient")
    assert dw0[:, 10:].abs().max().item() == 0


# ---------------------------------------------------------------------------------------------- B. attention dropout
def _mix32(x):
    """lowbias32 on numpy uint32 (wrapping) arithmetic."""
    x = x ^ (x >> np.uint32(16))
    x = x * np.uint32(0x7FEB352D)
    x = x ^ (x >> np.uint32(15))
    x = x * np.uint32(0x846CA68B)
    return x ^ (x >> np.uint32(16))


def attention_dropout_keep_host(B, T, heads, p, seed):
    """keep/(1-p) fp32 [B, heads, T, T] of the attention dropout, from its definition: with bh = b*heads + h,
    seed_bh = mix(lo32(seed) ^ bh*0x9E3779B9) ^ hi32(seed), and (q, k) is kept iff
    mix((q*T + k) ^ seed_bh) >> 8 >= floor(float64(float32(p)) * 2^24)."""
    thresh = np.uint32(math.floor(float(np.float32(p)) * 2.0 ** 24))
    inv_keep = np.float32(1.0) / (np.float32(1.0) - np.float32(p))
    bh = np.arange(B * heads, dtype=np.uint32)
    seed_bh = _mix32(np.uint32(seed & 0xFFFFFFFF) ^ (bh * np.uint32(0x9E3779B9))) ^ np.uint32(seed >> 32)
    qk = np.arange(T, dtype=np.uint32)[:, None] * np.uint32(T) + np.arange(T, dtype=np.uint32)[None, :]
    out = np.empty((B * heads, T, T), dtype=np.float32)
    for i in range(B * heads):
        out[i] = np.where((_mix32(qk ^ seed_bh[i]) >> np.uint32(8)) >= thresh, inv_keep, np.float32(0.0))
    return out.reshape(B, heads, T, T)


SEED = 0xC0FFEE12_3456789A                                   # high 32 bits nonzero


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("B,T,heads", [(2, 130, 3), (1, 999, 2)])
def test_attention_dropout_mask_matches_host_restatement(cuda, B, T, heads, p):
    host = attention_dropout_keep_host(B, T, heads, p, SEED)
    dev = ops.attention_dropout_mask(B, T, heads, p, SEED, cuda).cpu().numpy()
    assert np.array_equal(dev.view(np.uint32), host.view(np.uint32))
    assert abs(float((host > 0).mean()) - (1.0 - p)) < 0.01


def _attn_case(cuda, T, seed):
    heads = 16 if T % 2 == 0 else 12
    lens = sorted({n for n in (1, 64, 127, 128, T) if n <= T})
    B, H = len(lens), heads * 64
    qkv = _rand((B * T, 3 * H), cuda, 1.0, seed)
    qkv[:, :H] *= 0.25                                       # q is stored pre-scaled
    return qkv.bfloat16(), torch.tensor(lens, dtype=torch.int32, device=cuda), lens, B, heads


def _attn_ref(qkv, klen, B, T, heads, mask):
    """fp64 (softmax(s) * mask) @ v with keys >= key_len masked; returns (leaf x, s, ctx [B*T, H])."""
    x = qkv.double().view(B, T, 3, heads, 64).requires_grad_(True)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    s = q @ k.transpose(-1, -2)
    pad = torch.arange(T, device=qkv.device)[None, :] >= klen[:, None]
    s = s.masked_fill(pad[:, None, None, :], float("-inf"))
    o = ((s.softmax(-1) * mask) @ v).transpose(1, 2).reshape(B * T, heads * 64)
    return x, s, o


def _tiles(T):
    return [slice(i, min(T, i + 128)) for i in range(0, T, 128)]


ATTN_T = [64, 99, 128, 129, 256, 257, 399, 999]


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("T", ATTN_T)
def test_attention_dropout_forward(cuda, T, p):
    """Checked per 128-row query tile, so that a wrong mask in one tile is not diluted by the correct ones."""
    seed = SEED + T
    qkv, klen, lens, B, heads = _attn_case(cuda, T, 1)
    lse = torch.empty((B, heads, T), dtype=torch.float32, device=cuda)
    ctx = ops.attention(qkv, klen, B, T, heads, lse=lse, drop_p=p, drop_seed=seed)
    mask = torch.from_numpy(attention_dropout_keep_host(B, T, heads, p, seed)).to(cuda).double()
    _, s, ref = _attn_ref(qkv, klen, B, T, heads, mask)
    ref = ref.detach()
    for b in range(B):
        for i, rows in enumerate(_tiles(T)):
            o, r = ctx[b * T:(b + 1) * T][rows].double(), ref[b * T:(b + 1) * T][rows]
            torch.testing.assert_close(o, r, atol=2e-2, rtol=2e-2, msg=lambda m: f"utterance {b} tile {i}: {m}")
            assert _rel(o, r) < 1e-2, (b, i, _rel(o, r))
    # dropout does not change the softmax normaliser
    torch.testing.assert_close(lse.double(), torch.logsumexp(s.detach(), -1) * LOG2E, atol=2e-2, rtol=1e-3)


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("T", ATTN_T)
def test_attention_dropout_backward(cuda, T, p):
    """dq per 128-row query tile, dk / dv per 128-key tile; padded keys get exactly zero gradient."""
    seed = SEED + 7 * T
    qkv, klen, lens, B, heads = _attn_case(cuda, T, 2)
    H = heads * 64
    lse = torch.empty((B, heads, T), dtype=torch.float32, device=cuda)
    ctx = ops.attention(qkv, klen, B, T, heads, lse=lse, drop_p=p, drop_seed=seed)
    d_ctx = _rand((B * T, H), cuda, 1.0, 3).bfloat16()
    dqkv = ops.attention_bwd(qkv, ctx, d_ctx, lse, klen, B, T, heads, q_scale=1.0, drop_p=p, drop_seed=seed)
    mask = torch.from_numpy(attention_dropout_keep_host(B, T, heads, p, seed)).to(cuda).double()
    x, _, o = _attn_ref(qkv, klen, B, T, heads, mask)
    o.backward(d_ctx.double())
    ref = x.grad.reshape(B * T, 3 * H)
    for b, n in enumerate(lens):
        out_b, ref_b = dqkv[b * T:(b + 1) * T].double(), ref[b * T:(b + 1) * T]
        # one key: the softmax is constant, so dq and dk are exactly zero in the reference and only rounding (of the
        # bf16 ctx behind D = dO . O) in the kernel; dv is checked
        grads = (("dk", slice(H, 2 * H)), ("dv", slice(2 * H, 3 * H))) if n > 1 else (("dv", slice(2 * H, 3 * H)),)
        for i, rows in enumerate(_tiles(T)):
            if n > 1:
                r = _rel(out_b[rows, :H], ref_b[rows, :H])
                assert r < 1.5e-2, ("dq", b, i, r)
            keys = slice(rows.start, min(rows.stop, n))
            if keys.start < keys.stop:
                for name, sl in grads:
                    r = _rel(out_b[keys, sl], ref_b[keys, sl])
                    assert r < 1.5e-2, (name, b, i, r)
        if n < T:
            assert out_b[n:, H:].abs().max().item() == 0, f"padded keys of utterance {b} got a gradient"


@pytest.mark.parametrize("T", [128, 257])
def test_attention_dropout_seed_determinism(cuda, T):
    """The same seed twice: bit-identical ctx and dqkv.  Beyond one 128-key block the dq partial sums of the key
    blocks meet in fp32 atomics (order-dependent in the last bits), so there only dk / dv are compared bit for bit.
    Another seed changes both outputs."""
    qkv, klen, lens, B, heads = _attn_case(cuda, T, 4)
    H = heads * 64
    d_ctx = _rand((B * T, H), cuda, 1.0, 5).bfloat16()

    def run(seed):
        lse = torch.empty((B, heads, T), dtype=torch.float32, device=cuda)
        ctx = ops.attention(qkv, klen, B, T, heads, lse=lse, drop_p=0.1, drop_seed=seed)
        return ctx, ops.attention_bwd(qkv, ctx, d_ctx, lse, klen, B, T, heads, q_scale=1.0, drop_p=0.1, drop_seed=seed)

    c1, g1 = run(SEED)
    c2, g2 = run(SEED)
    c3, g3 = run(SEED + 1)
    exact = slice(0, 3 * H) if T <= 128 else slice(H, 3 * H)
    assert torch.equal(c1, c2) and torch.equal(g1[:, exact], g2[:, exact])
    assert not torch.equal(c1, c3) and not torch.equal(g1[:, H:], g3[:, H:])


# --------------------------------------------------------------------------------- C. small elementwise kernels
def test_gelu_bwd(cuda):
    pre = torch.cat([torch.linspace(-8.0, 8.0, 40000), torch.linspace(-300.0, 300.0, 4000),
                     torch.tensor([-300.0, 300.0, 0.0, -0.0])]).to(cuda).bfloat16()
    dy = _rand(pre.shape, cuda, 1.0, 1)
    out = ops.gelu_bwd(dy, pre)
    ref = dy.double() * _gelu_grad(pre.double())
    # the erf-based derivative is accurate to ~2e-7 absolute; the product adds one fp32 rounding
    err = (out.double() - ref).abs()
    bound = 1e-6 * dy.double().abs() + 2.0 ** -23 * ref.abs()
    assert bool((err <= bound).all()), f"worst error / bound {(err / bound).max().item():.3f}"


@pytest.mark.parametrize("rows,cols,ldo,scale", [(999, 768, 3 * 768, 1.0), (130, 1024, 3 * 1024, 0.125),
                                                 (7, 64, 64, 0.3)])
def test_scale_cast_bf16(cuda, rows, cols, ldo, scale):
    """out[r][0..cols) at row pitch ldo = bf16(scale * x): as attention_bwd writes the q block of dqkv (ldo = 3H).
    Columns cols .. ldo-1 are not written."""
    x = _rand((rows, cols), cuda, 3.0, 1)
    x[0, :4] = torch.tensor([1.00390625, 1.01171875, -3e38, float("inf")])    # two round-to-even ties, huge, inf
    out = torch.full((rows, ldo), 7.0, dtype=torch.bfloat16, device=cuda)
    _lib.check(_lib.load().aptai_scale_cast_bf16(x.data_ptr(), rows, cols, float(scale), out.data_ptr(), ldo,
                                                 ops._stream()), "scale_cast_bf16")
    expect = torch.full_like(out, 7.0)
    expect[:, :cols] = (x * scale).bfloat16()
    assert torch.equal(out.view(torch.int16), expect.view(torch.int16))
    if ldo == cols:
        assert torch.equal(ops.scale_cast_bf16(x, scale).view(torch.int16), expect.view(torch.int16))
