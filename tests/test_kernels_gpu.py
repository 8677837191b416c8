"""Parity of the HBM-bound kernels, attention and the alignment kernels, through the C ABI."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from aptai_b200 import ops
from oracle import ctc as octc
from oracle import heads as oheads


def _rand(shape, dev, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("norm,bias", [(1, True), (2, False), (2, True), (0, False)])
def test_conv0(cuda, norm, bias, dt):
    B, L = 3, 16000
    lens = [16000, 12345, 4000]
    wav = _rand((B, L), cuda, 0.1, 1)
    for b, n in enumerate(lens):
        wav[b, n:] = 0
    w = _rand((512, 1, 10), cuda, (2.0 / 10) ** 0.5, 2)
    bs = _rand((512,), cuda, 0.2, 3) if bias else None
    gam = 1 + _rand((512,), cuda, 0.1, 4)
    bet = _rand((512,), cuda, 0.1, 5)
    y = ops.conv0(wav, w.view(512, 10).contiguous(), bs, gam, bet, norm, out_dtype=dt)
    assert y.dtype == dt
    ref = F.conv1d(wav[:, None], w, bs, stride=5)
    if norm == 1:
        ref = F.layer_norm(ref.transpose(1, 2), (512,), gam, bet, 1e-5).transpose(1, 2)
    elif norm == 2:
        ref = F.group_norm(ref, 512, gam, bet, 1e-5)
    ref = F.gelu(ref).transpose(1, 2)
    assert y.shape == ref.shape
    err = (y.float() - ref).abs()
    tol = 1e-2 + 1e-2 * ref.abs()
    assert (err > tol).sum().item() == 0, f"max err {err.max().item()}"
    # beyond bf16 rounding the fp32 math must agree closely: compare in fp32 before rounding via mean error
    assert err.mean().item() < 2e-3


@pytest.mark.parametrize("norm", [1, 2, 0])
@pytest.mark.parametrize("B,L", [(3, 16000), (2, 16003), (5, 1290), (1, 10), (150, 4000)])
def test_conv0_tensor_core_vs_simt(cuda, norm, B, L, monkeypatch):
    """csrc/conv0_tc.cu (split-operand tcgen05 contraction, TMA bulk waveform tiles when L % 4 == 0, plain loads
    otherwise) against the SIMT kernel it replaces: same fp32 math up to 2^-24 splits, so the fp16 outputs may differ
    by one rounding step on a few elements and by nothing systematic."""
    if norm == 2 and L == 10:
        pytest.skip("GroupNorm over ONE frame: the variance is 0 and rstd = eps^-1/2 amplifies fp32 noise")
    wav = _rand((B, L), cuda, 0.1, 11)
    w = _rand((512, 10), cuda, (2.0 / 10) ** 0.5, 12)
    bs = _rand((512,), cuda, 0.2, 13)
    gam = 1 + _rand((512,), cuda, 0.1, 14)
    bet = _rand((512,), cuda, 0.1, 15)
    monkeypatch.setattr(ops, "CONV0_TC", 1)
    y_tc = ops.conv0(wav, w, bs, gam, bet, norm, out_dtype=torch.float16).float()
    monkeypatch.setattr(ops, "CONV0_TC", 0)
    y_simt = ops.conv0(wav, w, bs, gam, bet, norm, out_dtype=torch.float16).float()
    torch.cuda.synchronize()
    assert y_tc.shape == (B, (L - 10) // 5 + 1, 512)
    d = (y_tc - y_simt).abs()
    # one fp16 rounding step, plus the fp32 noise (1e-7 of an O(1) pre-activation) that dominates where the GELU
    # output itself is ~1e-4 (measured against fp64, profiles/scripts/conv0_tc_debug.py: both kernels 0.25 ulp mean)
    ulp = 2.0 ** -10 * y_simt.abs().clamp_min(2.0 ** -14)
    assert (d > 1.01 * ulp + 1e-6).sum().item() == 0, f"max err {d.max().item()}"
    assert (d > 0).float().mean().item() < 2e-2          # a rounding flip on fewer than 2 % of the elements
    assert torch.isfinite(y_tc).all()


@pytest.mark.parametrize("cols", [512, 768, 1024, 256])
@pytest.mark.parametrize("in_bf16", [False, True, torch.float16])
def test_layernorm(cuda, cols, in_bf16):
    rows = 1000
    x = _rand((rows, cols), cuda, 2.0, 6) + 0.5
    if in_bf16 is True:
        x = x.bfloat16()
    elif in_bf16 is torch.float16:
        x = x.half()
        o32, o16 = ops.layernorm(x, 1 + _rand((cols,), cuda, 0.1, 7), _rand((cols,), cuda, 0.1, 8), 1e-5, want_f32=True,
                                 want_bf16=True, out16_dtype=torch.float16)
        ref = F.layer_norm(x.float(), (cols,), 1 + _rand((cols,), cuda, 0.1, 7), _rand((cols,), cuda, 0.1, 8), 1e-5)
        torch.testing.assert_close(o32, ref, atol=2e-5, rtol=2e-5)
        torch.testing.assert_close(o16.float(), ref.half().float(), atol=3e-3, rtol=2e-3)
        return
    g = 1 + _rand((cols,), cuda, 0.1, 7)
    b = _rand((cols,), cuda, 0.1, 8)
    o32, o16 = ops.layernorm(x, g, b, 1e-5, want_f32=True, want_bf16=True)
    ref = F.layer_norm(x.float(), (cols,), g, b, 1e-5)
    torch.testing.assert_close(o32, ref, atol=2e-5, rtol=2e-5)
    torch.testing.assert_close(o16.float(), ref.bfloat16().float(), atol=2e-2, rtol=1e-2)


@pytest.mark.parametrize("legacy", [False, "v3"])
@pytest.mark.parametrize("B,T,heads,lens,scale", [(2, 199, 16, [199, 150], 1.0), (3, 64, 12, [64, 1, 33], 1.0),
                                                  (1, 999, 4, [999], 1.0), (2, 130, 2, [70, 130], 1.0),
                                                  (40, 399, 16, None, 0.5), (2, 513, 2, [513, 400], 3.0),
                                                  (3, 257, 2, [257, 256, 129], 1.0), (2, 128, 2, [128, 127], 1.0),
                                                  (24, 600, 16, None, 1.0), (150, 130, 4, None, 1.0)])
def test_attention(cuda, B, T, heads, lens, scale, legacy):
    H = heads * 64
    qkv = _rand((B * T, 3 * H), cuda, scale, 9).bfloat16()
    if lens is None:
        lens = [max(1, T - (7 * b) % 200) for b in range(B)]
    if scale > 1.0:
        qkv[T // 2:, H: 2 * H] *= 4.0          # later keys score much higher: exercises the lazy O rescale
    kl = torch.tensor(lens, dtype=torch.int32, device=cuda)
    lse = None
    if legacy == "v3":
        # third generation (P in TMEM, polynomial exponentials for 3 of every 8 pairs); context buffer pre-filled so
        # that rows the TMA store must NOT touch (none here: every row < T is written) would show
        lse = torch.empty((B, heads, T), dtype=torch.float32, device=cuda)
        ctx = ops.attention(qkv, kl, B, T, heads, impl=3, lse=lse,
                            out=torch.full((B * T, H), float("nan"), dtype=torch.bfloat16, device=cuda))
    else:
        ctx = ops.attention(qkv, kl, B, T, heads, impl=1)
    q, k, v = qkv.float().view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    s = q @ k.transpose(-1, -2)                      # q is expected pre-scaled
    mask = torch.arange(T, device=cuda)[None, :] < kl[:, None]
    s = s.masked_fill(~mask[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * T, H)
    torch.testing.assert_close(ctx.float(), ref, atol=2e-2, rtol=2e-2)
    if lse is not None:
        torch.testing.assert_close(lse, torch.logsumexp(s, -1) * 1.4426950408889634, atol=2e-2, rtol=1e-3)


def test_heads_lowpass_losses(cuda):
    B, T, H, V = 2, 150, 1024, 46
    h = _rand((B, T, H), cuda, 1.0, 10)
    tvw, tvb = _rand((9, H), cuda, 0.03, 11), _rand((9,), cuda, 0.03, 12)
    pw, pb = _rand((V, H), cuda, 0.03, 13), _rand((V,), cuda, 0.03, 14)
    taps = oheads.lowpass_taps().to(cuda)
    tv_raw, logits, am = ops.heads(h.view(B * T, H), tvw, tvb, ops.ACT_TANH, pw, pb, ops.ACT_LEAKY)
    r_raw, r_tv, r_logits = oheads.aptai_heads(h.cpu(), tvw.cpu(), tvb.cpu(), pw.cpu(), pb.cpu(), taps.cpu())
    torch.testing.assert_close(tv_raw.cpu().view(B, T, 9), r_raw, atol=2e-5, rtol=1e-4)
    torch.testing.assert_close(logits.cpu().view(B, T, V), r_logits, atol=2e-5, rtol=1e-4)
    assert torch.equal(am.cpu().view(B, T), torch.argmax(logits.cpu().view(B, T, V), -1))
    tv = ops.lowpass(tv_raw.view(B, T, 9), taps)
    torch.testing.assert_close(tv.cpu(), oheads.lowpass(tv_raw.cpu().view(B, T, 9), taps.cpu()), atol=1e-6, rtol=1e-5)
    # losses
    g = torch.Generator().manual_seed(15)
    phn = torch.randint(1, V, (B, T), generator=g)
    phn[1, 100:] = 0
    tgt = torch.randn((B, T, 9), generator=g)
    tgt[1, 100:] = -100.0
    out = ops.masked_mse_ce(tv.view(B * T, 9), tgt.to(cuda).view(B * T, 9).contiguous(), logits, phn.to(cuda).view(-1))
    loss, mse, ce = oheads.aptai_losses(tv.cpu(), logits.cpu().view(B, T, V), phn, tgt)
    torch.testing.assert_close(out.cpu(), torch.stack([loss, mse, ce]), atol=1e-5, rtol=1e-5)


@pytest.mark.parametrize("B,T,heads,lens,scale", [(2, 199, 16, [199, 150], 1.0), (3, 64, 12, [64, 1, 33], 1.0),
                                                  (1, 999, 4, [999], 1.0), (2, 513, 2, [513, 400], 3.0),
                                                  (2, 128, 2, [128, 127], 1.0), (40, 399, 16, None, 0.5)])
def test_attention_fp16_operands(cuda, B, T, heads, lens, scale):
    """precision="fp16": both attention kernels (two threads per row for T <= 128, query-tile pairs with P in TMEM
    above) on IEEE fp16 q / k / v / P / context — eight times tighter than the bf16 tolerance of test_attention."""
    H = heads * 64
    qkv = _rand((B * T, 3 * H), cuda, scale, 9).half()
    if lens is None:
        lens = [max(1, T - (7 * b) % 200) for b in range(B)]
    if scale > 1.0:
        qkv[T // 2:, H: 2 * H] *= 4.0          # later keys score much higher: exercises the lazy O rescale
    kl = torch.tensor(lens, dtype=torch.int32, device=cuda)
    q, k, v = qkv.float().view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    s = q @ k.transpose(-1, -2)
    mask = torch.arange(T, device=cuda)[None, :] < kl[:, None]
    s = s.masked_fill(~mask[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * T, H)
    for impl in (None, 3):                       # by shape, and the query-tile-pair kernel forced
        lse = torch.empty((B, heads, T), dtype=torch.float32, device=cuda)
        ctx = ops.attention(qkv, kl, B, T, heads, impl=impl, lse=lse,
                            out=torch.full((B * T, H), float("nan"), dtype=torch.float16, device=cuda))
        assert ctx.dtype == torch.float16
        torch.testing.assert_close(ctx.float(), ref, atol=2.5e-3, rtol=2.5e-3)
        torch.testing.assert_close(lse, torch.logsumexp(s, -1) * 1.4426950408889634, atol=2e-2, rtol=1e-3)
    with pytest.raises(TypeError):
        ops.attention(qkv, kl, B, T, heads, out=torch.empty((B * T, H), dtype=torch.bfloat16, device=cuda))


def _ctc_case(B, T, V, Smax, seed, repeats=False):
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((B, T, V)).astype(np.float32) * 2
    tl = rng.integers(1, Smax + 1, size=B).astype(np.int32)
    il = rng.integers(max(2, T // 2), T + 1, size=B).astype(np.int32)
    il[0] = T
    tg = np.full((B, Smax), -100, dtype=np.int32)
    for b in range(B):
        tg[b, : tl[b]] = rng.integers(1, V, size=tl[b])
        if repeats and tl[b] > 3:
            tg[b, 1] = tg[b, 0]
            tg[b, 3] = tg[b, 2]
    return logits, tg, il, tl


@pytest.mark.parametrize("B,T,V,Smax,rep", [(4, 60, 12, 9, True), (16, 399, 46, 59, False), (3, 50, 46, 100, True),
                                                (3, 999, 46, 200, True), (3, 999, 46, 450, True)])
def test_logsoftmax_ctc(cuda, B, T, V, Smax, rep):
    logits, tg, il, tl = _ctc_case(B, T, V, Smax, 3, rep)
    if Smax >= 200:                             # 16 / 32 states per lane: one full-width feasible transcript
        tl[0] = Smax
        tg[0] = 1 + (np.arange(Smax) * 7 % (V - 1))
    if B >= 3:
        tl[1] = min(Smax, il[1] + 1)            # infeasible: more labels than frames -> zero_infinity
        tg[1, : tl[1]] = 1 + (np.arange(tl[1]) % (V - 1))
    o = octc.ctc_loss_grad(logits, tg, il, tl, blank=0, zero_infinity=True, reduction="mean")
    scale = torch.from_numpy(o["scale"].astype(np.float32)).to(cuda)
    r = ops.logsoftmax_ctc(torch.from_numpy(logits).to(cuda), torch.from_numpy(tg).to(cuda),
                           torch.from_numpy(il).to(cuda), torch.from_numpy(tl).to(cuda), blank=0, zero_infinity=True,
                           scale=scale, want_log_probs=True, want_grad=True)
    nll = r["nll"].cpu().numpy()
    np.testing.assert_allclose(nll, o["nll"], rtol=1e-3, atol=1e-3)
    assert abs(float(r["loss_sum"].cpu()) - o["loss"]) <= 1e-3 * abs(o["loss"]) + 1e-5
    np.testing.assert_allclose(r["log_probs"].cpu().numpy(), o["log_probs"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(r["grad"].cpu().numpy(), o["grad"], rtol=1e-3, atol=2e-5)


def test_forward_sum(cuda):
    """ForwardSumLoss (models/modules.py:77-117): prepended blank column, per-utterance class count."""
    rng = np.random.default_rng(5)
    B, T, N = 3, 80, 60
    att = torch.log_softmax(torch.from_numpy(rng.standard_normal((B, T, N)).astype(np.float32)), -1)
    text = np.array([30, 59, 5], dtype=np.int32)
    mel = np.array([80, 70, 33], dtype=np.int32)
    loss_ref, nll_ref = octc.forward_sum_loss(att[:, None].numpy(), text, mel, -1.0)
    tg = torch.arange(1, N + 1, dtype=torch.int32)[None].repeat(B, 1).contiguous().to(cuda)
    scale = torch.from_numpy((1.0 / (np.maximum(text, 1) * B)).astype(np.float32)).to(cuda)
    r = ops.logsoftmax_ctc(att.to(cuda).contiguous(), tg, torch.from_numpy(mel).to(cuda), torch.from_numpy(text).to(cuda),
                           blank=0, zero_infinity=True, scale=scale, want_log_probs=False, prepend_blank=True,
                           blank_value=-1.0, vocab_len=torch.from_numpy(text + 1).to(cuda))
    np.testing.assert_allclose(r["nll"].cpu().numpy(), nll_ref, rtol=1e-3)
    assert abs(float(r["loss_sum"].cpu()) - loss_ref) <= 1e-3 * abs(loss_ref)


@pytest.mark.parametrize("B,T,C,Smax", [(64, 399, 46, 59), (8, 40, 5, 12), (4, 999, 46, 100), (3, 765, 46, 59),
                                        (4, 999, 46, 200), (4, 999, 46, 450)])
def test_viterbi_bit_exact(cuda, B, T, C, Smax):
    rng = np.random.default_rng(11)
    x = rng.standard_normal((B, T, C)).astype(np.float32)
    x[1] = 0.0                                             # all ties
    x[2] = rng.integers(0, 3, size=(T, C)).astype(np.float32)   # heavy ties
    lp = torch.log_softmax(torch.from_numpy(x), -1)
    tl = rng.integers(1, Smax + 1, size=B).astype(np.int32)
    il = rng.integers(max(2 * Smax, T // 2), T + 1, size=B).astype(np.int32) if T >= 4 * Smax else np.full(B, T, np.int32)
    il[0] = T
    tg = np.zeros((B, Smax), dtype=np.int32)
    if Smax >= 200:
        tl[0] = Smax                                        # il[0] = T: the widest transcript is used in full
    for b in range(B):
        tl[b] = min(tl[b], il[b] // 2)
        tg[b, : tl[b]] = rng.integers(1, C, size=tl[b])
        if tl[b] > 2:
            tg[b, 1] = tg[b, 0]
    paths, scores, status = ops.ctc_viterbi(lp.to(cuda).contiguous(), torch.from_numpy(tg).to(cuda),
                                            torch.from_numpy(il).to(cuda), torch.from_numpy(tl).to(cuda), blank=0)
    paths, scores, status = paths.cpu().numpy(), scores.cpu().numpy(), status.cpu().numpy()
    for b in range(B):
        p, s = octc.viterbi_align(lp[b, : il[b]].numpy(), tg[b, : tl[b]], blank=0)
        assert status[b] == 0
        assert np.array_equal(paths[b, : il[b]], p), f"utt {b}: path mismatch"
        assert np.array_equal(scores[b, : il[b]], s), f"utt {b}: score mismatch"
        assert (paths[b, il[b]:] == -1).all()


def test_viterbi_known_answer_and_infeasible(cuda):
    # SURVEY.md §4: uniform(T=6,C=3), targets [1,2] -> [1,2,2,2,2,2]
    lp = torch.log_softmax(torch.zeros((2, 6, 3)), -1).to(cuda)
    tg = torch.tensor([[1, 2, 0, 0, 0, 0, 0], [1, 1, 1, 1, 1, 1, 1]], dtype=torch.int32, device=cuda)
    il = torch.tensor([6, 6], dtype=torch.int32, device=cuda)
    tl = torch.tensor([2, 7], dtype=torch.int32, device=cuda)
    paths, _, status = ops.ctc_viterbi(lp, tg, il, tl, blank=0)
    assert paths[0].tolist() == [1, 2, 2, 2, 2, 2]
    assert status.tolist() == [0, 1]


def test_greedy(cuda):
    rng = np.random.default_rng(13)
    B, T, V = 5, 200, 46
    x = rng.standard_normal((B, T, V)).astype(np.float32)
    x[:, :, 0] += 1.5
    lens = np.array([200, 150, 1, 77, 33], dtype=np.int32)
    tok, frm, n = ops.ctc_greedy(torch.from_numpy(x).to(cuda), torch.from_numpy(lens).to(cuda), blank=0)
    for b in range(B):
        t_ref, f_ref = octc.greedy_decode(x[b, : lens[b]], blank=0)
        nb = int(n[b])
        assert nb == len(t_ref)
        assert np.array_equal(tok[b, :nb].cpu().numpy(), t_ref)
        assert np.array_equal(frm[b, :nb].cpu().numpy(), f_ref)


@pytest.mark.parametrize("B,T,lens", [(3, 70, [30, 59, 1]), (64, 399, None)])
def test_cross_attention_block(cuda, B, T, lens):
    """Fused Force_APTAI cross-attention (embedding + PE + q/k + masked softmax + LayerNorm + log-softmax) against the
    CPU restatement of models/modules.py:139-153 + models/force_aptai.py:118-130."""
    g = torch.Generator().manual_seed(3)
    V = 46
    if lens is None:          # BASELINE config-3 shape: the launch switches to 64 frames per CTA
        lens = torch.randint(10, 60, (B,), generator=g).tolist()
    frame = torch.randn((B, T, 128), generator=g)
    ids = torch.zeros((B, 60), dtype=torch.int32)
    for b, n in enumerate(lens):
        ids[b, :n] = torch.randint(1, V, (n,), generator=g).int()
    emb = torch.randn((V, 128), generator=g) * 0.3
    emb[0] = 0
    pe = oheads.positional_encoding(128, 60)
    wq, bq = torch.randn((128, 128), generator=g) * 0.09, torch.randn((128,), generator=g) * 0.02
    wk, bk = torch.randn((128, 128), generator=g) * 0.09, torch.randn((128,), generator=g) * 0.02
    lnw, lnb = 1 + 0.1 * torch.randn((256,), generator=g), 0.1 * torch.randn((256,), generator=g)
    c = lambda t: t.to(cuda).contiguous()
    att_out, energy, att = ops.cross_attention(c(frame), c(ids), c(emb), c(pe[:, 0, :]), c(wq), c(bq), c(wk), c(bk),
                                               c(lnw), c(lnb))
    mask = (ids != 0).int()
    phn = torch.nn.functional.embedding(ids.long(), emb) + pe[:60, 0][None]
    r_out, r_energy = oheads.cross_attention(frame, phn, mask, wq, bq, wk, bk, lnw, lnb)
    r_att = torch.log_softmax(r_energy + ((1 - mask) * -1000.0).unsqueeze(1), dim=-1)
    torch.testing.assert_close(energy.cpu(), r_energy, atol=2e-4, rtol=1e-4)
    torch.testing.assert_close(att_out.cpu(), r_out, atol=2e-4, rtol=1e-4)
    torch.testing.assert_close(att.cpu(), r_att, atol=2e-4, rtol=1e-4)
    assert torch.equal(att.cpu().argmax(-1), r_att.argmax(-1))
    # module form (models/modules.py:129-153 signature): precomputed phoneme embeddings + 0/1 mask
    from aptai_b200.modules import CrossAttention
    m = CrossAttention(128, 128, 128)
    with torch.no_grad():
        m.q.weight.copy_(wq); m.q.bias.copy_(bq); m.k.weight.copy_(wk); m.k.bias.copy_(bk)
        m.layer_norm.weight.copy_(lnw); m.layer_norm.bias.copy_(lnb)
    m = m.to(cuda)
    o2, e2 = m(c(frame), c(phn), c(mask))
    torch.testing.assert_close(o2.cpu(), r_out, atol=2e-4, rtol=1e-4)
    torch.testing.assert_close(e2.cpu(), r_energy, atol=2e-4, rtol=1e-4)


@pytest.mark.parametrize("B,T,lens", [(1, 99, [99]), (3, 130, [130, 7, 64]), (9, 50, [50, 1, 50, 33, 2, 49, 17, 50, 25]),
                                       (64, 399, None)])
def test_bilstm_cluster_kernel_vs_torch(cuda, B, T, lens):
    """Persistent cluster BiLSTM (csrc/lstm.cu) + RNN tail against torch nn.LSTM on packed sequences (CPU fp32):
    models/modules.py:190-214 with the intended packed_output semantics."""
    from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence
    from aptai_b200.modules import RNN
    torch.manual_seed(3)
    rnn = RNN(256, 9, drop=0.0).eval()
    g = torch.Generator().manual_seed(5)
    if lens is None:
        lens = torch.randint(60, T + 1, (B,), generator=g).tolist()
        lens[0] = T
    x = torch.randn((B, T, 256), generator=g)
    with torch.no_grad():
        packed = pack_padded_sequence(x, torch.tensor(lens), batch_first=True, enforce_sorted=False)
        ref_h, _ = pad_packed_sequence(rnn.lstm(packed)[0], batch_first=True, total_length=T)
        ref_out = rnn.linear(ref_h)
    rnn = rnn.to(cuda)
    out, hid = rnn(x.to(cuda), lens)
    torch.testing.assert_close(hid.cpu(), ref_h, atol=2e-4, rtol=1e-3)
    torch.testing.assert_close(out.cpu(), ref_out, atol=5e-4, rtol=1e-3)


@pytest.mark.parametrize("B,T,lens", [(3, 40, [40, 17, 1]), (9, 120, None)])
def test_bilstm_backward_through_time_vs_torch(cuda, B, T, lens):
    """BPTT cluster kernel + the GEMMs on its gate gradients (ops.bilstm_256_bwd) against torch autograd through
    nn.LSTM on packed sequences (CPU fp32): dx and all eight parameter gradients."""
    from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence
    from aptai_b200 import ops
    torch.manual_seed(4)
    lstm = torch.nn.LSTM(256, 256, bidirectional=True, num_layers=1, batch_first=True)
    g = torch.Generator().manual_seed(6)
    if lens is None:
        lens = torch.randint(30, T + 1, (B,), generator=g).tolist()
        lens[0] = T
    x = torch.randn((B, T, 256), generator=g, requires_grad=True)
    dh = torch.randn((B, T, 512), generator=g)
    packed = pack_padded_sequence(x, torch.tensor(lens), batch_first=True, enforce_sorted=False)
    ref_h, _ = pad_packed_sequence(lstm(packed)[0], batch_first=True, total_length=T)
    (ref_h * dh).sum().backward()
    ln = torch.tensor(lens, dtype=torch.int32, device=cuda)
    hid, sv = ops.bilstm_256(x.detach().to(cuda), lstm, ln, save=True)
    torch.testing.assert_close(hid.cpu(), ref_h.detach(), atol=2e-4, rtol=1e-3)
    grads = {n: torch.zeros_like(p, device=cuda) for n, p in lstm.named_parameters()}
    dx = ops.bilstm_256_bwd(sv, dh.to(cuda), grads)
    torch.cuda.synchronize()

    def close(name, got, ref):
        got, ref = got.double().cpu().flatten(), ref.double().flatten()
        rel = float((got - ref).norm() / ref.norm())
        assert rel < 1e-2, (name, rel)
        return rel

    worst = max(close("dx", dx, x.grad), *[close(n, grads[n], p.grad) for n, p in lstm.named_parameters()])
    print(f"BiLSTM backward B={B} T={T}: worst relative L2 error {worst:.2e}")


@pytest.mark.parametrize("B,T", [(2, 37), (5, 130), (64, 399)])
def test_cross_attention_backward_vs_autograd(cuda, B, T):
    """csrc/xattn.cu backward against torch autograd through the reference formulas (models/modules.py:129-153 and
    the doubly masked log-softmax of models/force_aptai.py:128-130): gradients of the projected queries / keys and
    of the LayerNorm parameters, for upstream gradients on both outputs (att_out and att)."""
    import torch.nn.functional as F
    from aptai_b200 import ops
    g = torch.Generator().manual_seed(31 + T)
    frame = torch.randn((B, T, 128), generator=g)
    phn = torch.randn((B, 60, 128), generator=g)
    ids = torch.zeros((B, 60), dtype=torch.int32)
    for b in range(B):
        n = int(torch.randint(3, 59, (1,), generator=g))
        ids[b, :n] = torch.randint(1, 46, (n,), generator=g, dtype=torch.int32)
    wq, wk = torch.randn((128, 128), generator=g) * 0.05, torch.randn((128, 128), generator=g) * 0.05
    bq, bk = torch.randn((128,), generator=g) * 0.1, torch.randn((128,), generator=g) * 0.1
    lnw = (1 + 0.1 * torch.randn((256,), generator=g)).requires_grad_(True)
    lnb = (0.1 * torch.randn((256,), generator=g)).requires_grad_(True)
    d_out, d_att = torch.randn((B, T, 256), generator=g), torch.randn((B, T, 60), generator=g)
    q = (frame @ wq.t() + bq).requires_grad_(True)
    k = (phn @ wk.t() + bk).requires_grad_(True)
    mask = ((ids == 0).float() * -1000.0)[:, None, :]
    energy = q @ k.transpose(1, 2) + mask
    ctx = torch.softmax(energy, dim=-1) @ k
    out = F.layer_norm(torch.cat([ctx, q], dim=-1), (256,), lnw, lnb, 1e-5)
    att = torch.log_softmax(energy + mask, dim=-1)
    ((out * d_out).sum() + (att * d_att).sum()).backward()
    c = lambda t: t.detach().to(cuda).contiguous()
    dlw, dlb = torch.zeros(256, device=cuda), torch.zeros(256, device=cuda)
    dq, dk = ops.cross_attention_bwd(c(frame), c(ids), c(phn), c(wq), c(bq), c(wk), c(bk), c(lnw), 1e-5, c(d_out),
                                     c(d_att), dlw, dlb)
    for name, got, ref in (("d_q", dq, q.grad), ("d_k", dk, k.grad), ("d_ln_w", dlw, lnw.grad), ("d_ln_b", dlb, lnb.grad)):
        rel = float((got.cpu().double() - ref.double()).norm() / ref.double().norm())
        assert rel < 1e-4, (name, rel)


def test_bilstm_backward_full_size_linearity(cuda):
    """BASELINE config-3 size (64 utterances x 399 frames, ragged): the CPU autograd oracle takes too long here, so
    the check is the size-independent property of a backward pass — it is linear in the upstream gradient:
    bwd(2 a - 3 b) == 2 bwd(a) - 3 bwd(b) for dx and every parameter gradient — plus exact zeros on padding frames."""
    from aptai_b200 import ops
    torch.manual_seed(8)
    B, T = 64, 399
    lstm = torch.nn.LSTM(256, 256, bidirectional=True, num_layers=1, batch_first=True).to(cuda)
    g = torch.Generator().manual_seed(12)
    lens = torch.randint(200, T + 1, (B,), generator=g).tolist()
    lens[0], lens[1] = T, 1
    ln = torch.tensor(lens, dtype=torch.int32, device=cuda)
    x = torch.randn((B, T, 256), generator=g).to(cuda)
    _, sv = ops.bilstm_256(x, lstm, ln, save=True)
    a, b = torch.randn((B, T, 512), generator=g).to(cuda), torch.randn((B, T, 512), generator=g).to(cuda)

    def run(dh):
        grads = {n: torch.zeros_like(p) for n, p in lstm.named_parameters()}
        return ops.bilstm_256_bwd(sv, dh.contiguous(), grads), grads

    (dxa, ga), (dxb, gb_), (dxc, gc) = run(a), run(b), run(2 * a - 3 * b)
    rel = lambda got, want: float((got - want).double().norm() / want.double().norm())
    # bf16 operands in the gradient GEMMs: each pass rounds its gate gradients independently (2^-9 per element)
    worst = rel(dxc, 2 * dxa - 3 * dxb)
    for n in ga:
        worst = max(worst, rel(gc[n], 2 * ga[n] - 3 * gb_[n]))
    print(f"BiLSTM backward 64x399 linearity: worst relative L2 deviation {worst:.2e}")
    assert worst < 1e-2
    for bi in (1, 5, 33):
        assert float(dxc[bi, lens[bi]:].abs().max()) == 0.0


def test_frame_lengths_kernel(cuda):
    """One-launch `_get_feat_extract_output_lengths` (HF:1005-1024) against the integer recurrence, incl. inputs too
    short for the conv stack (floor division goes negative exactly like torch.div(..., rounding_mode='floor'))."""
    from aptai_b200.config import W2V2Config
    cfg = W2V2Config.large()
    n = torch.tensor([16000, 400, 399, 128000, 320000, 25, 10, 1, 47999], dtype=torch.int64, device=cuda)
    o64, o32 = ops.frame_lengths(n, cfg.conv_kernel, cfg.conv_stride)
    ref = n.clone()
    for k, s in zip(cfg.conv_kernel, cfg.conv_stride):
        ref = torch.div(ref - k, s, rounding_mode="floor") + 1
    assert torch.equal(o64, ref) and torch.equal(o32.long(), ref)
    assert [cfg.conv_out_length(int(v)) for v in n[:5]] == o64[:5].tolist()


@pytest.mark.parametrize("rows,H,with_ln", [(150, 1024, True), (64, 768, True), (1000, 1024, False), (1, 1024, True),
                                            (5000, 1024, True), (129, 768, False)])
def test_fused_tail(cuda, rows, H, with_ln):
    """One-launch tail (final LayerNorm + both heads + argmax + log-softmax) against the separate kernels it
    replaces and against torch: fp32 throughout, so logits agree to accumulation-order noise and the argmax /
    log-softmax are consistent with the kernel's own logits."""
    h = _rand((rows, H), cuda, 1.5, 30) + 0.3
    g = 1 + _rand((H,), cuda, 0.1, 31)
    b = _rand((H,), cuda, 0.1, 32)
    tvw, tvb = _rand((9, H), cuda, 0.03, 33), _rand((9,), cuda, 0.03, 34)
    pw, pb = _rand((46, H), cuda, 0.03, 35), _rand((46,), cuda, 0.03, 36)
    oa, ob, am, lp, hn = ops.tail(h, g if with_ln else None, b if with_ln else None, 1e-5, tvw, tvb, ops.ACT_TANH, pw, pb,
                                  ops.ACT_LEAKY, want_logp=True, want_h_norm=with_ln)
    x = F.layer_norm(h, (H,), g, b, 1e-5) if with_ln else h
    if with_ln:
        torch.testing.assert_close(hn, x, atol=2e-5, rtol=2e-5)
    ref_a = torch.tanh(x) @ tvw.t() + tvb
    ref_b = F.leaky_relu(x, 0.01) @ pw.t() + pb
    torch.testing.assert_close(oa, ref_a, atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(ob, ref_b, atol=5e-5, rtol=1e-4)
    assert torch.equal(am, torch.argmax(ob, -1))
    torch.testing.assert_close(lp, torch.log_softmax(ob, -1), atol=2e-6, rtol=1e-5)
    # the kernels it replaces
    xs = ops.layernorm(h, g, b, 1e-5, want_f32=True, want_bf16=False)[0] if with_ln else h
    o2a, o2b, am2 = ops.heads(xs, tvw, tvb, ops.ACT_TANH, pw, pb, ops.ACT_LEAKY)
    torch.testing.assert_close(oa, o2a, atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(ob, o2b, atol=5e-5, rtol=1e-4)
