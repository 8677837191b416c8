"""Parity of the tcgen05 GEMM family (plain Linear, implicit-GEMM conv, grouped pos-conv, fused LN epilogue)
against fp32 torch references on bf16-rounded operands.  Calls go through the C ABI (aptai_b200.ops -> ctypes)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from aptai_b200 import ops


def _rand(shape, dev, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


def _close_bf16(out, ref, what, atol=2e-2, rtol=2e-2):
    out, ref = out.float(), ref.float()
    err = (out - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = (err > tol).sum().item()
    assert bad == 0, f"{what}: {bad} mismatches, max err {err.max().item():.4g}"


@pytest.mark.parametrize("pair", [1, 2])
@pytest.mark.parametrize("M,K,N", [(128, 64, 256), (300, 512, 1024), (1000, 1024, 3072), (777, 768, 2304),
                                   (129, 256, 128), (64, 128, 64), (5000, 4096, 1024), (40000, 1024, 1024)])
def test_linear_bias(cuda, M, K, N, pair):
    a = _rand((M, K), cuda, 1.0, 1).bfloat16()
    w = _rand((N, K), cuda, 0.05, 2).bfloat16()
    b = _rand((N,), cuda, 0.5, 3)
    o32, o16 = ops.linear(a, w, b, want_f32=True, want_bf16=True, cta_pair=pair)
    ref = a.float() @ w.float().t() + b
    torch.testing.assert_close(o32, ref, atol=2e-3, rtol=2e-3)
    _close_bf16(o16, ref, "bf16 out")


def test_linear_gelu_residual_mask(cuda):
    B, T, K, N = 3, 210, 512, 768
    M = B * T
    a = _rand((M, K), cuda, 1.0, 4).bfloat16()
    w = _rand((N, K), cuda, 0.05, 5).bfloat16()
    b = _rand((N,), cuda, 0.5, 6)
    res = _rand((M, N), cuda, 1.0, 7)
    _, o16 = ops.linear(a, w, b, act=1)
    ref = F.gelu(a.float() @ w.float().t() + b)
    _close_bf16(o16, ref, "gelu")
    o32, _ = ops.linear(a, w, b, residual=res, want_f32=True, want_bf16=False)
    torch.testing.assert_close(o32, a.float() @ w.float().t() + b + res, atol=2e-3, rtol=2e-3)
    # in-place residual (out aliases residual) + padded-row zeroing
    lens = torch.tensor([210, 100, 1], dtype=torch.int32, device=cuda)
    h = res.clone()
    ops.linear(a, w, b, residual=h, out_f32=h, want_bf16=False, seg_rows=T, seg_valid_rows=lens)
    ref = (a.float() @ w.float().t() + b + res).view(B, T, N)
    for i, n in enumerate(lens.tolist()):
        ref[i, n:] = 0
    torch.testing.assert_close(h.view(B, T, N), ref, atol=2e-3, rtol=2e-3)


@pytest.mark.parametrize("pair", [1, 2])
@pytest.mark.parametrize("k,T_in,B,ln", [(3, 801, 2, True), (3, 640, 3, False), (2, 399, 2, True), (2, 130, 1, False),
                                         (3, 2563, 2, True)])
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
def test_conv_igemm(cuda, k, T_in, B, ln, pair, dt):
    C = 512
    x = ops.alloc_rows_bf16(B, T_in, C, cuda, dtype=dt)
    x.copy_(_rand((B, T_in, C), cuda, 1.0, 8).to(dt))
    w = _rand((C, C, k), cuda, (2.0 / (C * k)) ** 0.5, 9)                  # torch layout [out][in][k]
    bias = _rand((C,), cuda, 0.1, 10)
    gam = 1 + _rand((C,), cuda, 0.1, 11)
    bet = _rand((C,), cuda, 0.1, 12)
    wk = w.permute(0, 2, 1).reshape(C, k * C).to(dt).contiguous()
    y = ops.conv_igemm(x, wk, bias, k, 2, ln_gamma=gam if ln else None, ln_beta=bet if ln else None, act=1, cta_pair=pair)
    assert y.dtype == dt
    ref = F.conv1d(x.float().transpose(1, 2), w.to(dt).float(), bias, stride=2)
    if ln:
        ref = F.layer_norm(ref.transpose(1, 2), (C,), gam, bet, 1e-5).transpose(1, 2)
    ref = F.gelu(ref).transpose(1, 2)
    assert y.shape == ref.shape
    _close_bf16(y, ref, "conv_igemm")


@pytest.mark.parametrize("H,groups,T,B", [(1024, 16, 199, 2), (768, 16, 130, 2), (256, 4, 77, 3)])
def test_posconv(cuda, H, groups, T, B):
    taps = 128
    gw = H // groups
    x = _rand((B, T, H), cuda, 1.0, 13)
    v = _rand((H, gw, taps), cuda, 2 * (1.0 / (taps * H)) ** 0.5, 14)
    g = torch.linalg.vector_norm(v, dim=(0, 1), keepdim=True) * (1 + _rand((1, 1, taps), cuda, 0.05, 15))
    bias = _rand((H,), cuda, 0.1, 16)
    wf = ops.posconv_fold(g.contiguous(), v.contiguous(), 64)
    w_ref = g * v / torch.linalg.vector_norm(v, dim=(0, 1), keepdim=True)
    # fold check (bf16 rounding of the exact quotient)
    wf_ref = torch.zeros((H, taps, 64), device=cuda)
    wf_ref[:, :, :gw] = w_ref.permute(0, 2, 1)
    torch.testing.assert_close(wf.float().view(H, taps, 64), wf_ref.bfloat16().float(), atol=1e-3, rtol=1e-2)
    xp = ops.cast_pad(x, taps // 2)
    assert xp.shape == (B, T + taps, H)
    assert torch.equal(xp[:, taps // 2: taps // 2 + T], x.bfloat16())
    assert float(xp[:, : taps // 2].abs().max()) == 0 and float(xp[:, taps // 2 + T:].abs().max()) == 0
    h = x.clone().view(B * T, H)
    ops.posconv(xp, wf, bias, h, T, H, groups, taps, h)
    pos = F.conv1d(x.bfloat16().float().transpose(1, 2), w_ref.bfloat16().float(), bias, padding=taps // 2,
                   groups=groups)[:, :, :-1]
    ref = x + F.gelu(pos).transpose(1, 2)
    torch.testing.assert_close(h.view(B, T, H), ref, atol=5e-3, rtol=5e-3)


def test_gelu_accuracy(cuda):
    """erf-GELU of the GEMM epilogue against the fp64 definition (identity weights, fp32 output)."""
    x = torch.linspace(-8, 8, 64 * 512, device=cuda).view(512, 64)
    a = x.bfloat16()
    w = torch.eye(64, device=cuda).bfloat16()
    o32, _ = ops.linear(a, w, None, act=1, want_f32=True, want_bf16=False)
    ref = torch.nn.functional.gelu(a.double())
    assert (o32.double() - ref).abs().max().item() < 1e-6
    # 16-bit outputs take the cheaper sigmoid-of-polynomial form (gelu_fast2, max abs error 2.6e-5 before rounding):
    # within half a bf16 ulp (2^-8 relative) of the fp64 definition plus that bound, over the whole range incl. |x| >> 8
    x = torch.cat([torch.linspace(-8, 8, 63 * 512), torch.linspace(-300, 300, 512)]).to(cuda).view(512, 64)
    a = x.bfloat16()
    _, o16 = ops.linear(a, w, None, act=1, want_f32=False, want_bf16=True)
    ref = torch.nn.functional.gelu(a.double())
    err = (o16.double() - ref).abs()
    assert bool((err <= ref.abs() * 2.0 ** -8 + 3e-5).all()), float((err - ref.abs() * 2.0 ** -8).max())


@pytest.mark.parametrize("T,B", [(399, 3), (256, 2), (257, 1), (600, 20), (1, 2)])
def test_posconv_slab_matches_generic(cuda, T, B):
    """The slab kernel (one load of every input row, tap shift as a descriptor offset with the SWIZZLE_128B base
    offset) against the generic implicit-GEMM path on the same operands: same bf16 products, same fp32 accumulation
    order per tap, so the two agree to fp32 rounding of the residual add."""
    H, groups, taps = 1024, 16, 128
    x = _rand((B, T, H), cuda, 1.0, 40)
    v = _rand((H, H // groups, taps), cuda, 2 * (1.0 / (taps * H)) ** 0.5, 41)
    g = torch.linalg.vector_norm(v, dim=(0, 1), keepdim=True) * (1 + _rand((1, 1, taps), cuda, 0.05, 42))
    bias = _rand((H,), cuda, 0.1, 43)
    wf = ops.posconv_fold(g.contiguous(), v.contiguous(), 64)
    xp = ops.cast_pad(x, taps // 2)
    h1 = x.clone().view(B * T, H)
    h2 = x.clone().view(B * T, H)
    old = ops.POSCONV_SLAB
    try:
        ops.POSCONV_SLAB = 1
        ops.posconv(xp, wf, bias, h1, T, H, groups, taps, h1)
        ops.POSCONV_SLAB = 0
        ops.posconv(xp, wf, bias, h2, T, H, groups, taps, h2)
    finally:
        ops.POSCONV_SLAB = old
    torch.testing.assert_close(h1, h2, atol=2e-6, rtol=2e-6)


@pytest.mark.parametrize("H,groups,T,B", [(1024, 16, 399, 2), (768, 16, 130, 2)])
def test_posconv_fp16_operands(cuda, H, groups, T, B):
    """precision="fp16": fold, cast + pad and both pos-conv kernels (slab for 64-channel groups, generic otherwise) on
    IEEE fp16 operands against the fp32 conv on fp16-rounded operands."""
    taps = 128
    gw = H // groups
    x = _rand((B, T, H), cuda, 1.0, 50)
    v = _rand((H, gw, taps), cuda, 2 * (1.0 / (taps * H)) ** 0.5, 51)
    g = torch.linalg.vector_norm(v, dim=(0, 1), keepdim=True) * (1 + _rand((1, 1, taps), cuda, 0.05, 52))
    bias = _rand((H,), cuda, 0.1, 53)
    wf = ops.posconv_fold(g.contiguous(), v.contiguous(), 64, dtype=torch.float16)
    assert wf.dtype == torch.float16
    w_ref = g * v / torch.linalg.vector_norm(v, dim=(0, 1), keepdim=True)
    wf_ref = torch.zeros((H, taps, 64), device=cuda)
    wf_ref[:, :, :gw] = w_ref.permute(0, 2, 1)
    torch.testing.assert_close(wf.float().view(H, taps, 64), wf_ref.half().float(), atol=1e-6, rtol=2e-3)
    xp = ops.cast_pad(x, taps // 2, dtype=torch.float16)
    assert xp.dtype == torch.float16 and torch.equal(xp[:, taps // 2: taps // 2 + T], x.half())
    assert float(xp[:, : taps // 2].abs().max()) == 0 and float(xp[:, taps // 2 + T:].abs().max()) == 0
    h = x.clone().view(B * T, H)
    ops.posconv(xp, wf, bias, h, T, H, groups, taps, h)
    pos = F.conv1d(x.half().float().transpose(1, 2), w_ref.half().float(), bias, padding=taps // 2,
                   groups=groups)[:, :, :-1]
    ref = x + F.gelu(pos).transpose(1, 2)
    torch.testing.assert_close(h.view(B, T, H), ref, atol=1e-4, rtol=1e-4)
    with pytest.raises(TypeError):
        ops.posconv(xp, wf.bfloat16(), bias, h, T, H, groups, taps, h)


def test_linear_fp16_operands(cuda):
    """The transformer GEMM shapes on fp16 operands (QKV, FFN1 + GELU, FFN2 + in-place residual)."""
    M, H, Fi = 700, 1024, 4096
    x = _rand((M, H), cuda, 1.0, 60)
    w1, b1 = _rand((Fi, H), cuda, 0.03, 61), _rand((Fi,), cuda, 0.1, 62)
    w2, b2 = _rand((H, Fi), cuda, 0.02, 63), _rand((H,), cuda, 0.1, 64)
    _, u = ops.linear(x.half(), w1.half(), b1, act=1)
    assert u.dtype == torch.float16
    ref_u = F.gelu(x.half().float() @ w1.half().float().t() + b1)
    torch.testing.assert_close(u.float(), ref_u, atol=2e-3, rtol=2e-3)
    h = _rand((M, H), cuda, 1.0, 65)
    h0 = h.clone()
    ops.linear(u, w2.half(), b2, residual=h, out_f32=h, want_bf16=False)
    torch.testing.assert_close(h, h0 + u.float() @ w2.half().float().t() + b2, atol=2e-4, rtol=2e-4)
