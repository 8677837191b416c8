"""CTC loss / gradient and CTC-Viterbi alignment for transcripts longer than 511 labels (the CTA-wide kernels), and
the encoder beyond 20 s.

References: the fp64 NumPy oracle (`oracle.ctc.ctc_loss_grad`) for the loss and gradient, `oracle.ctc.viterbi_align`
(bit-exact) for the alignment.  A CTC value passes when it is within `test_logsoftmax_ctc`'s tolerances of the
oracle, or within twice the error of torch.nn.functional.ctc_loss (CPU, fp32, autograd) on the same inputs: over
thousands of frames the reference's own fp32 arithmetic drifts, and the kernel is held to at least that standard.

Labels are laid out so that adjacent repeats (no s-2 skip) and distinct neighbours (skip allowed) both fall on
the boundary between two threads' state slices (16 states = 8 labels per thread)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from helpers import VOCAB, backbone_sd, cfg_large
from aptai_b200 import APTAI, Force_APTAI, Wav2Vec2_PR, ops
from aptai_b200 import lib as _lib
from aptai_b200.backbone import Wav2Vec2Backbone, register_in_memory_checkpoint
from oracle import ctc as octc
from oracle import w2v2 as ow
from oracle import weights as W

V = 46
LP_TOL = dict(rtol=1e-4, atol=1e-4)       # test_logsoftmax_ctc's tolerances
NLL_TOL = dict(rtol=1e-3, atol=1e-3)
GRAD_TOL = dict(rtol=1e-3, atol=2e-5)


def _labels(rng, L, C=V):
    """L labels in 1..C-1 with adjacent repeats at thread boundaries (label index j = 0 mod 8) and elsewhere."""
    tg = rng.integers(1, C, size=L).astype(np.int32)
    for j in range(8, L, 40):
        tg[j] = tg[j - 1]
    for j in range(13, L, 97):
        tg[j] = tg[j - 1]
    for j in range(16, L, 40):                    # distinct neighbours across the boundary: the skip is allowed
        if tg[j] == tg[j - 1]:
            tg[j] = 1 + tg[j - 1] % (C - 1)
    return tg


def _repeats(tg):
    return int(np.sum(tg[1:] == tg[:-1]))


def _pack(seqs, width, pad=-100):
    tg = np.full((len(seqs), width), pad, dtype=np.int32)
    for b, s in enumerate(seqs):
        tg[b, : len(s)] = s
    return tg


def _close(ours, ref, torch_val, tol, what):
    """|ours - ref| within `tol`, or within 2x torch's own error against the same reference."""
    ours, ref, tv = (np.asarray(x, dtype=np.float64) for x in (ours, ref, torch_val))
    fin = np.isfinite(ref)
    assert np.array_equal(ours[~fin], ref[~fin]), f"{what}: non-finite entries differ"
    if not fin.any():
        return
    err = np.abs(ours[fin] - ref[fin])
    assert np.isfinite(err).all(), f"{what}: non-finite where the reference is finite"
    if np.all(err <= tol["atol"] + tol["rtol"] * np.abs(ref[fin])):
        return
    terr = np.abs(tv - ref)[fin]
    terr = terr[np.isfinite(terr)]
    bound = 2 * float(terr.max()) if terr.size else 0.0
    assert err.max() <= bound, f"{what}: max error {err.max():.3g} beyond the tolerance and 2x torch's ({bound:.3g})"


def _oracle(logits, tg, il, tl, zero_infinity, reduction):
    """oracle.ctc.ctc_loss_grad per utterance; a 0-label utterance (which the oracle's recursion does not take) is
    the all-blank path: nll = -sum_t lp[t, blank], gradient softmax - onehot(blank)."""
    B, T, _ = logits.shape
    lp = octc.log_softmax(np.asarray(logits, dtype=np.float64))
    nll, grad = np.zeros(B), np.zeros(logits.shape)
    for b in range(B):
        n = int(il[b])
        if tl[b] == 0:
            nll[b] = -lp[b, :n, 0].sum()
            grad[b, :n] = np.exp(lp[b, :n])
            grad[b, :n, 0] -= 1.0
        else:
            o = octc.ctc_loss_grad(logits[b:b + 1], tg[b:b + 1], il[b:b + 1], tl[b:b + 1], blank=0,
                                   zero_infinity=zero_infinity, reduction="sum")
            nll[b], grad[b] = o["nll"][0], o["grad"][0]
    scale = 1.0 / (np.maximum(tl, 1) * B) if reduction == "mean" else np.ones(B)
    return {"nll": nll, "loss": float(np.sum(nll * scale)), "grad": grad * scale[:, None, None],
            "log_probs": np.transpose(lp, (1, 0, 2)), "scale": scale}


def _torch_ctc(logits, tg, il, tl, scale, zero_infinity):
    x = torch.from_numpy(logits).requires_grad_(True)
    lp = torch.log_softmax(x, -1)
    nll = F.ctc_loss(lp.transpose(0, 1), torch.from_numpy(np.maximum(tg, 0)).long(), torch.from_numpy(il).long(),
                     torch.from_numpy(tl).long(), blank=0, reduction="none", zero_infinity=zero_infinity)
    loss = (nll * torch.from_numpy(scale.astype(np.float32))).sum()
    loss.backward()
    return {"nll": nll.detach().numpy(), "loss": float(loss.detach()), "log_probs": lp.detach().transpose(0, 1).numpy(),
            "grad": x.grad.numpy()}


def _run_ctc(cuda, logits, tg, il, tl, scale, zero_infinity):
    d = lambda a: torch.from_numpy(a).to(cuda)
    return ops.logsoftmax_ctc(d(logits), d(tg), d(il), d(tl), blank=0, zero_infinity=zero_infinity,
                              scale=d(scale.astype(np.float32)), want_log_probs=True, want_grad=True)


def _check_ctc(cuda, logits, tg, il, tl, reduction="sum", zero_infinity=True):
    o = _oracle(logits, tg, il, tl, zero_infinity, reduction)
    scale = o["scale"]
    t = _torch_ctc(logits, tg, il, tl, scale, zero_infinity)
    r = _run_ctc(cuda, logits, tg, il, tl, scale, zero_infinity)
    nll = r["nll"].cpu().numpy()
    _close(nll, o["nll"], t["nll"], NLL_TOL, "nll")
    _close([float(r["loss_sum"].cpu())], [o["loss"]], [t["loss"]], NLL_TOL, "loss_sum")
    _close(r["log_probs"].cpu().numpy(), o["log_probs"], t["log_probs"], LP_TOL, "log_probs")
    grad = r["grad"].cpu().numpy()
    _close(grad, o["grad"], t["grad"], GRAD_TOL, "grad")
    for b in range(len(il)):
        assert not grad[b, il[b]:].any(), f"utt {b}: gradient not zero beyond input_len"
    return r, o


# ------------------------------------------------------------------------------------------------ CTC loss / gradient
def _case_512():
    """Smax 512: a full-width transcript, a tight one (T = L + R), a 1-frame one-label utterance."""
    rng = np.random.default_rng(101)
    T = 1100
    a = _labels(rng, 512)
    b = _labels(rng, 500)
    seqs = [a, b, np.array([7], np.int32)]
    il = np.array([T, len(b) + _repeats(b), 1], np.int32)
    logits = rng.standard_normal((3, T, V)).astype(np.float32)
    return logits, _pack(seqs, 512), il, np.array([len(s) for s in seqs], np.int32)


def _case_1000():
    """Smax 1000: a full-width transcript, an infeasible one (more labels than frames), a 0-label one."""
    rng = np.random.default_rng(102)
    T = 2500
    a = _labels(rng, 1000)
    b = _labels(rng, 900)
    seqs = [a, b, np.zeros(0, np.int32)]
    il = np.array([T, 850, 2000], np.int32)
    logits = (1.5 * rng.standard_normal((3, T, V))).astype(np.float32)
    return logits, _pack(seqs, 1000), il, np.array([len(s) for s in seqs], np.int32)


def _case_2047():
    """Smax 2047 in a label tensor padded to 2600 columns, ragged input lengths."""
    rng = np.random.default_rng(103)
    T = 4500
    seqs = [_labels(rng, 2047), _labels(rng, 1500)]
    il = np.array([T, 3900], np.int32)
    logits = rng.standard_normal((2, T, V)).astype(np.float32)
    return logits, _pack(seqs, 2600), il, np.array([len(s) for s in seqs], np.int32)


def _case_4095():
    rng = np.random.default_rng(104)
    T = 6000
    seqs = [_labels(rng, 4095)]
    logits = rng.standard_normal((1, T, V)).astype(np.float32)
    return logits, _pack(seqs, 4095), np.array([T], np.int32), np.array([4095], np.int32)


def test_ctc_long_512_tight_and_one_frame(cuda):
    logits, tg, il, tl = _case_512()
    r, o = _check_ctc(cuda, logits, tg, il, tl, reduction="mean")
    assert np.isfinite(o["nll"]).all() and (o["nll"] > 0).all()


@pytest.mark.parametrize("zero_infinity", [True, False])
def test_ctc_long_1000_infeasible_and_empty(cuda, zero_infinity):
    logits, tg, il, tl = _case_1000()
    r, o = _check_ctc(cuda, logits, tg, il, tl, zero_infinity=zero_infinity)
    nll = r["nll"].cpu().numpy()
    if zero_infinity:
        assert nll[1] == 0 and not r["grad"][1].any()
    else:
        assert np.isinf(nll[1]) and np.isinf(float(r["loss_sum"].cpu()))
    assert np.isfinite(nll[[0, 2]]).all()


def test_ctc_long_2047_padded_labels(cuda):
    logits, tg, il, tl = _case_2047()
    _check_ctc(cuda, logits, tg, il, tl)


def test_ctc_long_4095(cuda):
    logits, tg, il, tl = _case_4095()
    _check_ctc(cuda, logits, tg, il, tl)


def test_ctc_long_deterministic(cuda):
    logits, tg, il, tl = _case_2047()
    scale = np.full(len(il), 0.5)
    r1 = _run_ctc(cuda, logits, tg, il, tl, scale, True)
    r2 = _run_ctc(cuda, logits, tg, il, tl, scale, True)
    for k in ("nll", "loss_sum", "log_probs", "grad"):
        assert torch.equal(r1[k], r2[k]), k


def test_ctc_long_boundary_511_512(cuda):
    """511 labels run the register kernel, also from a label tensor padded to 600 columns (narrowed to 511);
    512 labels run the CTA kernel.  Both agree with the oracle."""
    rng = np.random.default_rng(105)
    T = 1200
    logits = rng.standard_normal((1, T, V)).astype(np.float32)
    il = np.array([T], np.int32)
    s511 = _labels(rng, 511)
    r511 = _run_ctc(cuda, logits, _pack([s511], 511), il, np.array([511], np.int32), np.ones(1), True)
    r600 = _run_ctc(cuda, logits, _pack([s511], 600), il, np.array([511], np.int32), np.ones(1), True)
    for k in ("nll", "grad", "log_probs"):
        assert torch.equal(r511[k], r600[k]), k
    _check_ctc(cuda, logits, _pack([s511], 511), il, np.array([511], np.int32))
    _check_ctc(cuda, logits, _pack([_labels(rng, 512)], 512), il, np.array([512], np.int32))


def test_forward_sum_long(cuda):
    """ForwardSumLoss form beyond 511 labels: virtual blank column, per-utterance class count, targets 1..N."""
    rng = np.random.default_rng(106)
    B, T, N = 2, 1500, 700
    att = torch.log_softmax(torch.from_numpy(rng.standard_normal((B, T, N)).astype(np.float32)), -1)
    text = np.array([700, 600], dtype=np.int32)
    mel = np.array([1500, 1300], dtype=np.int32)
    loss_ref, nll_ref = octc.forward_sum_loss(att[:, None].numpy(), text, mel, -1.0)
    tg = torch.arange(1, N + 1, dtype=torch.int32)[None].repeat(B, 1).contiguous().to(cuda)
    scale = (1.0 / (np.maximum(text, 1) * B)).astype(np.float32)
    r = ops.logsoftmax_ctc(att.to(cuda).contiguous(), tg, torch.from_numpy(mel).to(cuda),
                           torch.from_numpy(text).to(cuda), blank=0, zero_infinity=True,
                           scale=torch.from_numpy(scale).to(cuda), want_log_probs=False, want_grad=True,
                           prepend_blank=True, blank_value=-1.0, vocab_len=torch.from_numpy(text + 1).to(cuda))
    np.testing.assert_allclose(r["nll"].cpu().numpy(), nll_ref, rtol=1e-3)
    assert abs(float(r["loss_sum"].cpu()) - loss_ref) <= 1e-3 * abs(loss_ref)
    grad = r["grad"].cpu().numpy()
    for b in range(B):
        n, tb = int(text[b]), int(mel[b])
        cur = np.concatenate((np.full((tb, 1), -1.0), att[b, :tb, :n].double().numpy()), axis=1)
        _, g = octc.ctc_single(octc.log_softmax(cur), np.arange(1, n + 1), blank=0)
        np.testing.assert_allclose(grad[b, :tb, :n], g[:, 1:] * scale[b], **GRAD_TOL)
        assert not grad[b, :tb, n:].any() and not grad[b, tb:].any()


def test_ctc_beyond_limit_rejected(cuda):
    L = _lib.load()
    assert ops.CTC_MAX_LABELS == 4095
    B, T, S = 1, 9000, 4096
    assert L.aptai_ctc_workspace_bytes(B, T, S) == 0 and L.aptai_viterbi_workspace_bytes(B, T, S) == 0
    assert L.aptai_ctc_workspace_bytes(B, T, 4095) > 0 and L.aptai_viterbi_workspace_bytes(B, T, 4095) > 0
    logits = torch.zeros((B, T, V), device=cuda)
    tg = torch.ones((B, S), dtype=torch.int32, device=cuda)
    il = torch.tensor([T], dtype=torch.int32, device=cuda)
    tl = torch.tensor([S], dtype=torch.int32, device=cuda)
    with pytest.raises(ValueError, match="4095"):
        ops.logsoftmax_ctc(logits, tg, il, tl)
    with pytest.raises(ValueError, match="4095"):
        ops.ctc_viterbi(logits, tg, il, tl)
    nll = torch.empty((B,), device=cuda)
    ws = torch.empty((1 << 20,), dtype=torch.uint8, device=cuda)
    rc = L.aptai_logsoftmax_ctc_ex(logits.data_ptr(), B, T, V, 0, 0.0, None, tg.data_ptr(), S, il.data_ptr(),
                                   tl.data_ptr(), 0, 1, None, nll.data_ptr(), None, None, None, ws.data_ptr(),
                                   ws.numel(), None)
    assert rc == -1 and "4095" in _lib.last_error()
    paths = torch.empty((B, T), dtype=torch.int32, device=cuda)
    rc = L.aptai_ctc_viterbi_f32(logits.data_ptr(), tg.data_ptr(), il.data_ptr(), tl.data_ptr(), B, T, V, S, 0,
                                 paths.data_ptr(), None, None, ws.data_ptr(), ws.numel(), None)
    assert rc == -1 and "4095" in _lib.last_error()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ Viterbi
def _check_viterbi(cuda, lp, seqs, il, width):
    B, T, _ = lp.shape
    tg = _pack(seqs, width, pad=0)
    tl = np.array([len(s) for s in seqs], np.int32)
    paths, scores, status = ops.ctc_viterbi(torch.from_numpy(lp).to(cuda), torch.from_numpy(tg).to(cuda),
                                            torch.from_numpy(il).to(cuda), torch.from_numpy(tl).to(cuda), blank=0)
    paths, scores, status = paths.cpu().numpy(), scores.cpu().numpy(), status.cpu().numpy()
    for b in range(B):
        n = int(il[b])
        assert (paths[b, n:] == -1).all() and (scores[b, n:] == 0).all(), f"utt {b}: frames beyond input_len"
        if n < len(seqs[b]) + _repeats(seqs[b]):
            assert status[b] == 1 and (paths[b] == -1).all() and (scores[b] == 0).all(), f"utt {b}: infeasible"
            continue
        p, s = octc.viterbi_align(lp[b, :n], seqs[b], blank=0)
        assert status[b] == 0
        assert np.array_equal(paths[b, :n], p), f"utt {b}: path mismatch at frame {np.argmax(paths[b, :n] != p)}"
        assert np.array_equal(scores[b, :n], s), f"utt {b}: score mismatch"


@pytest.mark.parametrize("Smax,T", [(512, 1100), (1000, 2200), (2047, 4400), (4095, 6000)])
def test_viterbi_long_bit_exact(cuda, Smax, T):
    """Random, all-tie, heavy-tie + tight (T = L + R), infeasible and short utterances in one ragged batch."""
    rng = np.random.default_rng(Smax)
    x = rng.standard_normal((4, T, V)).astype(np.float32)
    x[1] = 0.0                                                    # all ties
    x[2] = rng.integers(0, 3, size=(T, V)).astype(np.float32)     # heavy ties
    lp = torch.log_softmax(torch.from_numpy(x), -1).numpy()
    seqs = [_labels(rng, Smax), _labels(rng, Smax // 2), _labels(rng, Smax - 9), _labels(rng, Smax // 3)]
    il = np.array([T, T - 37, len(seqs[2]) + _repeats(seqs[2]), len(seqs[3]) - 1], np.int32)
    _check_viterbi(cuda, lp, seqs, il, Smax)


# ------------------------------------------------------------------------------------------------ model level
SEC60, SEC2 = 960000, 32000          # 2999 and 99 frames


def _tiny_cfg():
    return cfg_large(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=512,
                     num_conv_pos_embedding_groups=4, vocab_size=V)


def _tiny_pr(cuda):
    cfg = _tiny_cfg()
    name = register_in_memory_checkpoint("mem://tiny-large-seed3", backbone_sd(cfg, 3))
    pr = Wav2Vec2_PR(cfg, None, name, VOCAB)
    hw, hb = W.linear_params(104, V, 256)
    with torch.no_grad():
        pr.pr_head.weight.copy_(hw); pr.pr_head.bias.copy_(hb)
    return pr.to(cuda)


def _long_inputs(cuda):
    lens = [SEC60, SEC2]
    wav = W.waveforms(2, SEC60, lens, seed=4321).to(cuda)
    rng = np.random.default_rng(107)
    seqs = [_labels(rng, 1200), _labels(rng, 30)]
    return wav, torch.tensor(lens, device=cuda), seqs


def test_pr_forward_long_transcript(cuda):
    pr = _tiny_pr(cuda).eval()
    wav, lens, seqs = _long_inputs(cuda)
    labels = torch.from_numpy(_pack(seqs, 1200)).to(cuda)
    with torch.no_grad():
        r = pr(wav, lens, labels, want_grad=True)
    lg = r["phoneme_logits"].cpu().numpy()
    assert lg.shape == (2, 2999, V)
    il = np.array([2999, 99], np.int32)
    tl = np.array([1200, 30], np.int32)
    o = _oracle(lg, _pack(seqs, 1200), il, tl, True, "mean")
    t = _torch_ctc(lg, _pack(seqs, 1200), il, tl, o["scale"], True)
    _close([float(r["loss"])], [o["loss"]], [t["loss"]], NLL_TOL, "loss")
    gl = r["grad_logits"].cpu().numpy()
    _close(gl, o["grad"], t["grad"], GRAD_TOL, "grad_logits")
    assert not gl[1, 99:].any()


def test_pr_train_backward_long_transcript(cuda):
    pr = _tiny_pr(cuda)
    pr.wav2vec2.freeze_feature_encoder()
    pr.train()
    wav, lens, seqs = _long_inputs(cuda)
    labels = torch.from_numpy(_pack(seqs, 1200)).to(cuda)
    r = pr(wav, lens, labels)
    assert np.isfinite(float(r["loss"].detach())) and float(r["loss"].detach()) > 0
    r["loss"].backward()
    n = 0
    for name, p in pr.named_parameters():
        if p.grad is not None:
            assert torch.isfinite(p.grad).all(), name
            n += 1
    assert n > 0 and pr.pr_head.weight.grad.abs().max() > 0


def test_aptai_predict_long_alignment(cuda):
    cfg = _tiny_cfg()
    name = register_in_memory_checkpoint("mem://tiny-large-seed3", backbone_sd(cfg, 3))
    torch.manual_seed(0)
    m = APTAI(cuda, VOCAB, name, cfg, None, phn_drop=0.0, tv_drop=0.0).to(cuda).eval()
    wav, lens, seqs = _long_inputs(cuda)
    tg = torch.from_numpy(_pack(seqs, 1200, pad=0)).to(cuda)
    tl = torch.tensor([len(s) for s in seqs], dtype=torch.int32, device=cuda)
    out = m.predict(wav, lens, phn_targets=tg, phn_target_lens=tl)
    lp = out["log_probs"].cpu().numpy()
    paths, scores = out["align_paths"].cpu().numpy(), out["align_scores"].cpu().numpy()
    assert out["align_status"].tolist() == [0, 0]
    for b, n in enumerate([2999, 99]):
        p, s = octc.viterbi_align(lp[b, :n], seqs[b], blank=0)
        assert np.array_equal(paths[b, :n], p) and np.array_equal(scores[b, :n], s), b
        assert (paths[b, n:] == -1).all()


def test_force_aptai_forced_align_long(cuda):
    pr = _tiny_pr(cuda).eval()
    fa = Force_APTAI("unused", cuda, VOCAB, w2v2_pr=pr).to(cuda).eval()
    wav, lens, seqs = _long_inputs(cuda)
    _, _, logits = pr._logits(wav, lens)
    lp = ops.softmax_rows(logits.contiguous(), log=True)
    paths, scores, status = fa.forced_align(wav, lens, [s.tolist() for s in seqs], log_probs=lp)
    lp = lp.cpu().numpy()
    assert status.tolist() == [0, 0]
    for b, n in enumerate([2999, 99]):
        p, s = octc.viterbi_align(lp[b, :n], seqs[b], blank=0)
        assert np.array_equal(paths[b, :n].cpu().numpy(), p) and np.array_equal(scores[b, :n].cpu().numpy(), s), b
        assert (paths[b, n:] == -1).all()


def test_encoder_60s(cuda):
    """test_maximum_length_20s at 60 s (2999 frames: 24 query tiles of 128) with a 2 s partner."""
    cfg = _tiny_cfg()
    lens = [SEC60, SEC2]
    sd = W.backbone_state_dict(cfg, seed=0)
    wav = W.waveforms(2, SEC60, lens, seed=1234)
    ref = ow.forward(sd, cfg, wav, lens)
    m = Wav2Vec2Backbone(cfg)
    m.load_state_dict(sd, strict=True)
    m = m.to(cuda).eval()
    out = m(wav.to(cuda), attention_mask=torch.tensor(lens, device=cuda)[:, None], output_hidden_states=True)
    assert ref[-1].shape[1] == 2999
    err = (out.last_hidden_state.cpu() - ref[-1]).abs()
    assert err.max().item() < 8e-2 and err.mean().item() < 1.2e-2, (err.max().item(), err.mean().item())
