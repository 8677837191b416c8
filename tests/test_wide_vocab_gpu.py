"""Phoneme recognisers with 49..1024 classes: the wide tensor-core head (`ops.pr_head_wide` + `ops.logits_rows`), its
backward (`ops.pr_head_wide_bwd`), CTC / Viterbi / decoding at V = 1024, and Wav2Vec2_PR / Force_APTAI on a 392-class
recogniser.  Errors are measured against fp64 on the exact fp32 inputs the kernels read; each bound is about 4x the
error measured on an NVIDIA B200 (printed with a "[wide]" prefix)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from helpers import backbone_sd, cfg_large
from aptai_b200 import Force_APTAI, Wav2Vec2_PR, ops
from aptai_b200.backbone import register_in_memory_checkpoint
from oracle import ctc as octc
from oracle import ctc_decode as ocd
from oracle import weights as W

# |out - ref| / (|a| |b| + |bias|) (max, median over all entries); measured on a B200 (1000 W): logits 2.8e-6 / 3.5e-7,
# dh 7.5e-6 / 7.1e-7, dW 1.65e-5 / 5.2e-7 (7 rows: every product's split error shows), db 9.8e-8 / 1.5e-8.  A bf16
# head is at ~1e-3.
BOUNDS = {"logits": (1.2e-5, 1.4e-6), "dh": (3e-5, 2.8e-6), "dW": (6.5e-5, 2.1e-6), "db": (4e-7, 6e-8)}
GEMM_MAX = BOUNDS["logits"][0]
LOGP_MAX, PROB_MAX = 1e-5, 2e-6   # |out - ref| / max over the row of (|h| |W| + |b|); measured 2.5e-6, 4.6e-7
ROWS = (1, 7, 129, 20000)   # 20000 rows > 148 SMs x 8 CTAs x 8 warps: the row kernel's grid-stride loop runs twice


def _report(what, err, bound):
    print(f"[wide] {what}: {err:.3e} (bound {bound:.1e})")
    assert err <= bound, f"{what}: {err:.3e} > {bound:.1e}"


def _randn(shape, dev, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g, dtype=torch.float64) * scale).float().to(dev)


def _head_case(rows, H, V, dev, seed):
    h = _randn((rows, H), dev, seed)
    w = _randn((V, H), dev, seed + 1, H ** -0.5)
    b = _randn((V,), dev, seed + 2, 0.1)
    ref = h.double() @ w.double().T + b.double()
    mag = h.double().abs() @ w.double().abs().T + b.double().abs()
    return h, w, b, ref, mag


def _err(out, ref, mag):
    e = ((out.double() - ref) / mag).abs().float().flatten()
    return e.max().item(), e.median().item()


# ================================================================================================ 1. forward
@pytest.mark.parametrize("H", [256, 768, 1024])
@pytest.mark.parametrize("V", [49, 63, 64, 65, 127, 392, 1000, 1024])
def test_head_forward_vs_fp64(cuda, V, H):
    for rows in ROWS:
        h, w, b, ref, mag = _head_case(rows, H, V, cuda, 1000 * V + H + rows)
        raw = ops.pr_head_wide(h, w, b)
        assert raw.shape == (rows, V) and raw.stride(0) == (V + 63) // 64 * 64
        lg, am, lp, pr = ops.logits_rows(raw, want_argmax=True, want_logp=True, want_prob=True)
        assert lg.is_contiguous() and torch.equal(lg, raw)
        e_max, e_med = _err(lg, ref, mag)
        _report(f"logits V={V} H={H} rows={rows} max", e_max, GEMM_MAX)
        _report(f"logits V={V} H={H} rows={rows} median", e_med, BOUNDS["logits"][1])
        lp_ref = torch.log_softmax(ref, -1)
        row_mag = mag.max(-1, keepdim=True).values
        _report(f"log_softmax V={V} H={H} rows={rows}", ((lp.double() - lp_ref) / row_mag).abs().max().item(),
                LOGP_MAX)
        _report(f"softmax V={V} H={H} rows={rows}", ((pr.double() - lp_ref.exp()) / row_mag).abs().max().item(),
                PROB_MAX)
        # argmax: fp64's first maximum wherever the top-2 margin is clear of the error bound
        top2 = ref.topk(2, dim=-1).values
        safe = (top2[:, 0] - top2[:, 1]) > 4 * GEMM_MAX * mag.max(-1).values
        assert safe.float().mean() > 0.9
        assert torch.equal(am[safe], ref.argmax(-1)[safe]), f"argmax V={V} H={H} rows={rows}"
        assert torch.equal(am, lg.argmax(-1))                  # torch's first-max rule on the kernel's own logits


@pytest.mark.parametrize("V", [65, 392, 1024])
def test_head_planted_ties_first_max(cuda, V):
    """Duplicated weight rows give bit-equal logits; the first of them must win: the same lane (columns 5 and 37),
    across lanes (31 and 35), and across 64-column GEMM tiles (40 and V - 2)."""
    H, rows = 768, 3000
    for j1, j2 in [(5, 37), (31, 35), (40, V - 2)]:
        h, w, b, _, _ = _head_case(rows, H, V, cuda, V + j1)
        u = _randn((H,), cuda, 7 + j1)
        u = u / u.norm()
        h = h + 8.0 * u                                       # every row points along u ...
        w[j1] = w[j2] = 3.0 * u                               # ... so the planted pair is the maximum
        b[j1] = b[j2] = 0.5
        lg, am, _, _ = ops.logits_rows(ops.pr_head_wide(h, w, b), want_argmax=True)
        assert torch.equal(lg[:, j1], lg[:, j2])
        assert (lg[:, j1] >= lg.max(-1).values).all()
        assert (am == j1).all(), (j1, j2, am.unique().tolist())


def test_head_output_padding_does_not_leak(cuda):
    rows, H, V = 500, 256, 100
    h, w, b, ref, mag = _head_case(rows, H, V, cuda, 5)
    buf = torch.full((rows, 136), float("nan"), device=cuda)     # pitch 136 > Vp = 128
    raw = ops.pr_head_wide(h, w, b, out=buf)
    assert raw.data_ptr() == buf.data_ptr() and raw.stride(0) == 136
    assert not buf[:, V:128].any() and buf[:, 128:].isnan().all()   # zero weight rows; nothing past Vp is written
    lg, am, lp, pr = ops.logits_rows(raw, want_argmax=True, want_logp=True, want_prob=True)
    for t in (lg, lp, pr):
        assert torch.isfinite(t).all()
    assert _err(lg, ref, mag)[0] <= GEMM_MAX
    assert torch.allclose(pr.double().sum(-1), torch.ones(rows, dtype=torch.float64, device=cuda), atol=1e-5)


def test_logits_rows_matches_softmax_rows(cuda):
    """Same formulas and summation order as softmax_rows: bit-identical log-softmax / softmax."""
    for V in (49, 300, 1024):
        x = _randn((777, V), cuda, V, 3.0)
        _, _, lp, pr = ops.logits_rows(x, want_logits=False, want_logp=True, want_prob=True)
        assert torch.equal(lp, ops.softmax_rows(x, log=True)) and torch.equal(pr, ops.softmax_rows(x))


def test_wide_head_limits(cuda):
    h = _randn((4, 256), cuda, 1)
    with pytest.raises(ValueError, match="1024"):
        ops.pr_head_wide(h, _randn((1025, 256), cuda, 2), None)
    with pytest.raises(RuntimeError, match="1024"):
        ops.logits_rows(_randn((4, 1025), cuda, 3))


# ================================================================================================ 2. backward
def _bwd_case(rows, H, V, dev, seed, ld):
    h = _randn((rows, H), dev, seed)
    w = _randn((V, H), dev, seed + 1, H ** -0.5)
    dbuf = _randn((rows, ld), dev, seed + 2, 1e-3)
    return h, w, dbuf[:, :V]


@pytest.mark.parametrize("H", [256, 1024])
@pytest.mark.parametrize("V", [49, 64, 65, 392, 1024])
@pytest.mark.parametrize("rows", [7, 20000])
def test_head_backward_vs_fp64(cuda, V, H, rows):
    ld = V + 24                                   # d_logits with a row pitch wider than V
    h, w, d = _bwd_case(rows, H, V, cuda, V + H + rows, ld)
    dw0 = _randn((V, H), cuda, 11, 1e-2)          # accumulate into non-zero gradients
    db0 = _randn((V,), cuda, 12, 1e-2)
    dw, db = dw0.clone(), db0.clone()
    dh = ops.pr_head_wide_bwd(h, w, d, dw, db)
    hd, wd, dd = h.double(), w.double(), d.double()
    checks = [("dh", dh, dd @ wd, dd.abs() @ wd.abs()),
              ("dW", dw, dw0.double() + dd.T @ hd, dw0.double().abs() + dd.abs().T @ hd.abs()),
              ("db", db, db0.double() + dd.sum(0), db0.double().abs() + dd.abs().sum(0))]
    for name, out, ref, mag in checks:
        e_max, e_med = _err(out, ref, mag)
        _report(f"{name} V={V} H={H} rows={rows} max", e_max, BOUNDS[name][0])
        _report(f"{name} V={V} H={H} rows={rows} median", e_med, BOUNDS[name][1])


# ================================================================================================ 3. narrow path
def _vocab(V):
    return {"(blank)": 0, "(...)": 1, **{f"p{i}": i for i in range(2, V)}}


def _tiny_pr(cuda, V, seed=3):
    cfg = cfg_large(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=512,
                    num_conv_pos_embedding_groups=4, vocab_size=V)
    sd = backbone_sd(cfg, seed)
    name = register_in_memory_checkpoint(f"mem://tiny-large-seed{seed}", sd)
    pr = Wav2Vec2_PR(cfg, None, name, _vocab(V))
    hw, hb = W.linear_params(200 + V, V, 256)
    with torch.no_grad():
        pr.pr_head.weight.copy_(hw); pr.pr_head.bias.copy_(hb)
    return pr.to(cuda), cfg, sd, hw, hb


def _batch(cuda, V, B=2, seed=21):
    lens = [32000, 23000][:B]
    wav = W.waveforms(B, max(lens), lens, seed=seed).to(cuda)
    labels, _ = W.phoneme_sequences(B, 3, 12, 2, V - 1, seed=seed, pad=-100)
    return wav, torch.tensor(lens, device=cuda), labels.to(cuda)


@pytest.mark.parametrize("V", [46, 48, 49])
def test_head_path_selection_bit_identical(cuda, V):
    """V <= 48: logits, loss and head gradients are those of direct ops.heads / ops.heads_bwd calls; V = 49: those
    of direct ops.pr_head_wide / ops.logits_rows / ops.pr_head_wide_bwd calls."""
    pr, _, _, _, _ = _tiny_pr(cuda, V)
    pr.wav2vec2.freeze_feature_encoder()
    pr.train()
    wav, lens, labels = _batch(cuda, V)
    r = pr(wav, lens, labels)
    r["loss"].backward()
    h = r["hidden_states"].reshape(-1, 256).contiguous()
    w = pr.pr_head.weight.detach().float().contiguous()
    b = pr.pr_head.bias.detach().float().contiguous()
    d_lg = r["grad_logits"].reshape(h.shape[0], V).contiguous()
    dw, db = torch.zeros_like(w), torch.zeros_like(b)
    if V <= ops.PR_HEAD_NARROW:
        lg = ops.heads(h, None, None, 0, w, b, ops.ACT_NONE, want_argmax=False)[1]
        ops.heads_bwd(h, None, None, 0, None, None, d_lg, w, ops.ACT_NONE, dw, db)
    else:
        lg = ops.logits_rows(ops.pr_head_wide(h, w, b))[0]
        ops.pr_head_wide_bwd(h, w, d_lg, dw, db)
    assert torch.equal(r["phoneme_logits"].reshape(-1, V), lg)
    B, T = r["phoneme_logits"].shape[:2]
    il = pr.wav2vec2._get_feat_extract_output_lengths(lens).int()
    tl = (labels >= 0).sum(-1).int()
    again = ops.logsoftmax_ctc(lg.view(B, T, V), labels.int().contiguous(), il, tl, blank=0, zero_infinity=True,
                               scale=(1.0 / (tl.clamp(min=1).float() * B)).contiguous())
    assert torch.equal(r["loss"].detach().reshape(1), again["loss_sum"])
    # the weight / bias gradients are sums with atomics in both paths: equal up to their order
    torch.testing.assert_close(pr.pr_head.weight.grad, dw, rtol=1e-5, atol=1e-9)
    torch.testing.assert_close(pr.pr_head.bias.grad, db, rtol=1e-5, atol=1e-9)


# ================================================================================================ 4. CTC at V = 1024
V_CTC = 1024


def _labels(rng, L):
    tg = rng.integers(1, V_CTC, size=L).astype(np.int32)
    tg[7::50] = tg[6::50][: len(tg[7::50])]                  # adjacent repeats
    return tg


@pytest.mark.parametrize("S,T", [(200, 400), (1000, 1300)])
def test_ctc_loss_grad_v1024(cuda, S, T):
    rng = np.random.default_rng(S)
    B = 2
    logits = (rng.standard_normal((B, T, V_CTC)) * 2).astype(np.float32)
    seqs = [_labels(rng, S), _labels(rng, S - 37)]
    tg = np.zeros((B, S), np.int32)
    for b, s in enumerate(seqs):
        tg[b, : len(s)] = s
    il = np.array([T, T - 41], np.int32)
    tl = np.array([len(s) for s in seqs], np.int32)
    o = octc.ctc_loss_grad(logits, tg, il, tl, blank=0, zero_infinity=True, reduction="mean")
    r = ops.logsoftmax_ctc(torch.from_numpy(logits).to(cuda), torch.from_numpy(tg).to(cuda),
                           torch.from_numpy(il).to(cuda), torch.from_numpy(tl).to(cuda), blank=0, zero_infinity=True,
                           scale=torch.from_numpy(o["scale"]).float().to(cuda), want_grad=True)
    assert np.isfinite(o["loss"]) and o["loss"] > 0
    # measured: loss 1.4e-7 relative, log_probs 2.5e-6, gradient 1.0e-3 (S = 200) / 5.8e-4 (S = 1000) of max |grad|
    _report(f"ctc loss S={S} rel", abs(float(r["loss_sum"]) - o["loss"]) / o["loss"], 6e-7)
    _report(f"ctc log_probs S={S}", np.abs(r["log_probs"].cpu().numpy() - o["log_probs"]).max(), 1e-5)
    g = r["grad"].cpu().numpy()
    _report(f"ctc grad S={S} / max|grad|", np.abs(g - o["grad"]).max() / np.abs(o["grad"]).max(), 4e-3)
    assert not g[1, il[1]:].any()


@pytest.mark.parametrize("S,T", [(200, 400), (1000, 1300)])
def test_ctc_viterbi_v1024_bit_exact(cuda, S, T):
    rng = np.random.default_rng(S + 1)
    x = rng.standard_normal((3, T, V_CTC)).astype(np.float32)
    x[1, ::3] = 0.0                                           # all-tie frames
    x[2] = rng.integers(0, 3, size=(T, V_CTC)).astype(np.float32)
    lp = torch.log_softmax(torch.from_numpy(x), -1).numpy()
    seqs = [_labels(rng, S), _labels(rng, S - 11), _labels(rng, S // 2)]
    tg = np.zeros((3, S), np.int32)
    for b, s in enumerate(seqs):
        tg[b, : len(s)] = s
    il = np.array([T, T - 9, T - 100], np.int32)
    tl = np.array([len(s) for s in seqs], np.int32)
    paths, scores, status = ops.ctc_viterbi(torch.from_numpy(lp).to(cuda), torch.from_numpy(tg).to(cuda),
                                            torch.from_numpy(il).to(cuda), torch.from_numpy(tl).to(cuda), blank=0)
    assert status.tolist() == [0, 0, 0]
    paths, scores = paths.cpu().numpy(), scores.cpu().numpy()
    for b in range(3):
        p, s = octc.viterbi_align(lp[b, : il[b]], seqs[b], blank=0)
        assert np.array_equal(paths[b, : il[b]], p) and np.array_equal(scores[b, : il[b]], s), b


def test_ctc_greedy_and_decode_ref_v1024(cuda):
    rng = np.random.default_rng(5)
    B, T = 3, 700
    x = rng.standard_normal((B, T, V_CTC)).astype(np.float32)
    x[1, :, :] = np.round(x[1] * 2) / 2                       # many exact ties
    x[2, 100:200] = 0.0
    lg = torch.from_numpy(x).to(cuda)
    il = torch.tensor([T, 650, 333], dtype=torch.int32, device=cuda)
    tok, frm, n = (t.cpu().numpy() for t in ops.ctc_greedy(lg, il, blank=0))
    for b, L in enumerate([T, 650, 333]):
        et, ef = octc.greedy_decode(x[b, :L], blank=0)
        assert n[b] == len(et) and np.array_equal(tok[b, : n[b]], et) and np.array_equal(frm[b, : n[b]], ef), b
    tok, steps, n = (t.cpu().numpy() for t in ops.ctc_decode_ref(lg, None, blank=0, sil=1))
    for b in range(B):
        et, es = ocd.reference_decode(x[b], blank=0, sil=1)
        assert np.array_equal(tok[b, : n[b]], et) and np.array_equal(steps[b, : n[b]], es), b


# ================================================================================================ 5. model level, V = 392
V_PR = 392


def _grad_match(ours, ref, what, norm_tol=0.05, cos_min=0.98):
    ours, ref = ours.double().cpu().flatten(), ref.double().cpu().flatten()
    dev = abs(float(ours.norm() / ref.norm()) - 1)
    cos = float(ours @ ref / (ours.norm() * ref.norm()))
    print(f"[wide] {what}: grad-norm deviation {dev:.2e}, cosine {cos:.5f}")
    assert dev < norm_tol and cos > cos_min, (what, dev, cos)


def test_pr392_forward_and_train_step_vs_oracle(cuda):
    from oracle import w2v2 as ow
    pr, cfg, sd0, hw, hb = _tiny_pr(cuda, V_PR)
    pr.wav2vec2.freeze_feature_encoder()
    wav, lens, labels = _batch(cuda, V_PR, seed=31)
    lens_l = lens.tolist()
    sd = {k: v.clone() for k, v in sd0.items()}
    trainable = [k for k in sd if not k.startswith("feature_extractor.") and k != "masked_spec_embed"]
    for k in trainable:
        sd[k].requires_grad_(True)
    w_ref, b_ref = hw.clone().requires_grad_(True), hb.clone().requires_grad_(True)
    hidden, _, flen = ow.forward(sd, cfg, wav.cpu(), lens_l, return_features=True)
    lp = F.log_softmax(F.linear(hidden[-1], w_ref, b_ref), dim=-1).transpose(0, 1)
    lab = labels.cpu()
    ref_loss = F.ctc_loss(lp, lab[lab >= 0], flen, (lab >= 0).sum(-1), blank=0, reduction="mean", zero_infinity=True)
    ref_loss.backward()
    ref = float(ref_loss.detach())
    with torch.no_grad():
        r_eval = pr.eval()(wav, lens, labels)
    _report("pr392 eval loss rel", abs(float(r_eval["loss"]) - ref) / ref, 1e-3)
    r = pr.train()(wav, lens, labels)
    _report("pr392 train loss rel", abs(float(r["loss"].detach()) - ref) / ref, 1e-3)
    r["loss"].backward()
    _grad_match(pr.pr_head.weight.grad, w_ref.grad, "pr_head.weight")
    _grad_match(pr.pr_head.bias.grad, b_ref.grad, "pr_head.bias")
    params = dict(pr.named_parameters())
    norms = {k: float(sd[k].grad.double().norm()) for k in trainable}
    floor = 1e-4 * float(np.median(list(norms.values())))
    for k, n in norms.items():
        if n >= floor:
            _grad_match(params["wav2vec2." + k].grad, sd[k].grad, k)


def test_pr392_get_embeddings_grad_vs_oracle(cuda):
    from oracle import w2v2 as ow
    pr, cfg, sd0, hw, hb = _tiny_pr(cuda, V_PR)
    pr.eval()
    wav, lens, _ = _batch(cuda, V_PR, seed=41)
    pr.grad_buffer().zero()
    out = pr.get_embeddings_grad(wav, lens, _vocab(V_PR), 1, 2)
    frames = pr.wav2vec2._get_feat_extract_output_lengths(lens).tolist()
    mask = torch.zeros(out["phoneme_logits_last"].shape[:2], device=cuda)
    for b, n in enumerate(frames):
        mask[b, :n] = 1
    def loss_of(last, inter):
        return ((last.log_softmax(-1)[..., 3] + 0.5 * inter[..., 7]) * mask.to(last.device)).sum()
    loss_of(out["phoneme_logits_last"], out["phoneme_logits_inter"]).backward()
    sd = {k: v.clone() for k, v in sd0.items()}
    w_ref, b_ref = hw.clone().requires_grad_(True), hb.clone().requires_grad_(True)
    with torch.no_grad():
        hidden = ow.forward(sd, cfg, wav.cpu(), lens.tolist())
    loss_of(F.linear(hidden[-1], w_ref, b_ref), F.linear(hidden[1], w_ref, b_ref)).backward()
    _grad_match(pr.pr_head.weight.grad, w_ref.grad, "get_embeddings_grad pr_head.weight")
    _grad_match(pr.pr_head.bias.grad, b_ref.grad, "get_embeddings_grad pr_head.bias")
    assert any(p.grad is not None and p.grad.abs().max() > 0 for n, p in pr.named_parameters() if "encoder" in n)


def test_pr392_single_utterance_decode_and_graph_replay(cuda):
    pr, _, _, _, _ = _tiny_pr(cuda, V_PR)
    pr.eval()
    vocab = _vocab(V_PR)
    wav = W.waveforms(1, 40000, None, seed=51)[0].numpy()
    pr.use_cuda_graphs = False
    eager = pr.get_ctc_logits(wav)
    T = int(pr.wav2vec2._get_feat_extract_output_lengths(torch.tensor([40000]))[0])
    pr.use_cuda_graphs = True
    first, replay = pr.get_ctc_logits(wav), pr.get_ctc_logits(wav)
    assert eager.shape == (T, V_PR)
    assert np.array_equal(first, eager) and np.array_equal(replay, eager)
    et, es = ocd.reference_decode(eager, blank=0, sil=1)
    seq = pr.pred_phn_seq(wav, vocab)
    assert np.array_equal(seq["phn_seq_idx"], et)
    dur = pr.predict_phonemes_durations(wav, vocab)
    assert np.array_equal(dur["phn_seq_idx"], et)
    ratio = 40000 / T / 16000
    np.testing.assert_allclose(dur["phn_seq_dur"], es * ratio, rtol=1e-12)
    assert (et < V_PR).all() and len(et) > 2


def test_force_aptai_on_pr392(cuda):
    pr, _, _, _, _ = _tiny_pr(cuda, V_PR)
    pr.eval()
    with torch.no_grad():
        pr.pr_head.bias[0] += 2.5       # mostly blank frames: the decoded sequences fit Force_APTAI's 60 slots
    torch.manual_seed(0)
    fa = Force_APTAI("unused", cuda, _vocab(V_PR), w2v2_pr=pr).to(cuda).eval()
    wav, lens, _ = _batch(cuda, V_PR, seed=61)
    T = int(pr.wav2vec2._get_feat_extract_output_lengths(lens).max())
    tv = [torch.randn(2, T, device=cuda) for _ in range(9)]
    with torch.no_grad():
        out = fa(0, wav, lens, None, None, *tv)
        _, _, logits = pr._logits(wav, lens)
    assert torch.isfinite(out["loss"])
    dec = pr._decode(logits)
    for a, e in zip(out["pred_ctc_phn_seq"], dec):
        assert np.array_equal(np.asarray(a), e)
    seqs = [[300, 5, 391, 391, 17], [2, 250, 100]]
    lp = ops.softmax_rows(logits.contiguous(), log=True)
    paths, scores, status = fa.forced_align(wav, lens, seqs, log_probs=lp)
    assert status.tolist() == [0, 0]
    lp = lp.cpu().numpy()
    for b, n in enumerate(pr.wav2vec2._get_feat_extract_output_lengths(lens).tolist()):
        p, s = octc.viterbi_align(lp[b, :n], np.array(seqs[b]), blank=0)
        assert np.array_equal(paths[b, :n].cpu().numpy(), p) and np.array_equal(scores[b, :n].cpu().numpy(), s)
    # a Force_APTAI whose embedding table is smaller than the recogniser's vocabulary rejects the ids it cannot embed
    small = Force_APTAI("unused", cuda, _vocab(46), w2v2_pr=pr).to(cuda).eval()
    with pytest.raises(ValueError, match="embedding table of 46"):
        with torch.no_grad():
            small(0, wav, lens, None, None, *tv, phn_seqs=[[3, 100], [5]])
