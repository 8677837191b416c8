"""North-star parity at the BASELINE config sizes, against goldens produced by the reference's OWN classes
(tests/golden/make_golden_v2.py: 24x1024 backbone, 8 s / 20 s single utterances, a ragged batch of 4, the 16 x 8 s
CTC batch of config 2, Force_APTAI at 8 s).  T = 399 / 999 puts the query-tile-pair attention kernel — the one
bench.py runs — on the path of a 24-layer reference-pinned test.

Tolerances are the literal ones of BASELINE.json's north_star:
    articulatory trajectories  max-abs <= 1e-2, Pearson >= 0.999 per channel          (both precision modes)
    CTC / CTC-type losses      <= 1e-3 relative                                       (both modes for the CTC loss;
                                                                                       f32x3 for Force's align_loss)
    phoneme argmax agreement   >= 99.9 %                                              (precision="f32x3")
precision="fp16" (the default kernels on IEEE fp16 operands, same speed) is asserted on what three more mantissa bits
buy: the literal CTC-type loss tolerance everywhere (Force_APTAI's align_loss included), trajectories within 2.5e-3,
logits within 4e-3 and a raw argmax agreement >= 99.5 % (profiles/scripts/operand_format_study.py: 99.8 % expected).
In the default bf16 mode the argmax criterion is not reachable on an untrained head (median top-2 margin 0.07 vs a
bf16 logit error of ~1e-2, SURVEY.md Appendix D): there the tests assert full agreement on every frame whose fp32
top-2 margin exceeds 4x the measured logit error and record the raw figure in gpurun_out/parity_report.json.
"""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from helpers import (R4_FRAMES, ROOT, TV, VOCAB, backbone_sd, cfg_large, f8_tv_targets, force_tail_state, golden2,
                     pearson, r4_targets)
from aptai_b200 import APTAI, Force_APTAI, Wav2Vec2_PR
from aptai_b200.backbone import register_in_memory_checkpoint
from oracle import weights as W

REPORT = os.path.join(ROOT, "gpurun_out", "parity_report.json")
MODES = ["f32x3", "fp16", "bf16"]


def _report(key, val):
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    d = json.load(open(REPORT)) if os.path.exists(REPORT) else {}
    d[key] = val
    json.dump(d, open(REPORT, "w"), indent=1)


def _argmax(logits, ref_logits=None, ref_pred=None, ref_margin=None, err=None):
    """(raw agreement, agreement on frames with margin > 4 * err, logit max-abs error)."""
    if ref_logits is not None:
        err = float(np.abs(logits - ref_logits).max())
        ref_pred = ref_logits.argmax(-1)
        srt = np.sort(ref_logits, -1)
        ref_margin = srt[..., -1] - srt[..., -2]
    pred = logits.argmax(-1)
    hit = pred == ref_pred
    safe = ref_margin > 4 * err
    return float(hit.mean()), (float(hit[safe].mean()) if safe.any() else 1.0), err


def _check_argmax(mode, key, raw, safe, err, frames):
    _report(f"{key}[{mode}]", {"argmax_agreement_raw": raw, "argmax_agreement_margin_gt_4err": safe,
                                "logit_max_abs_err": err, "frames": int(frames)})
    if mode == "f32x3":
        assert raw >= 0.999, (key, raw, err)               # north star, literal
    elif mode == "fp16":
        assert safe == 1.0 and raw >= 0.995 and err <= 4e-3, (key, raw, safe, err)
    else:
        assert safe == 1.0 and raw >= 0.97, (key, raw, safe, err)


@pytest.fixture(scope="module")
def aptai_large(cuda):
    cfg = cfg_large()
    name = register_in_memory_checkpoint("mem://large-seed0", backbone_sd(cfg, 0))
    m = APTAI(cuda, VOCAB, name, cfg, None, phn_drop=0.0, tv_drop=0.0)
    tvw, tvb = W.linear_params(101, 9, 1024)
    pw, pb = W.linear_params(102, 46, 1024)
    with torch.no_grad():
        m.tv_head[2].weight.copy_(tvw); m.tv_head[2].bias.copy_(tvb)
        m.phn_head[2].weight.copy_(pw); m.phn_head[2].bias.copy_(pb)
    return m.to(cuda).eval()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag,L,seed", [("l8", 128000, 4234), ("l20", 320000, 5234)])
def test_aptai_single_utterance_8s_20s(aptai_large, mode, tag, L, seed):
    g = golden2()
    aptai_large.set_precision(mode)
    try:
        wav = W.waveforms(1, L, None, seed=seed)
        r = aptai_large.get_aptai_output(wav[0].numpy())
    finally:
        aptai_large.set_precision("bf16")
    T = g[f"{tag}_logits"].shape[0]
    assert r["phn_fc_logits"].shape == (T, 46) and r["phn_fc_probs"].shape == (46, T, 1)
    tvs = np.stack([np.asarray(r["tvs_pred"][k], dtype=np.float32) for k in TV], -1)
    d = float(np.abs(tvs - g[f"{tag}_tvs"]).max())
    pc = float(pearson(tvs, g[f"{tag}_tvs"]).min())
    _report(f"aptai_{tag}_tv[{mode}]", {"tv_max_abs": d, "pearson_min": pc})
    assert d <= (2.5e-3 if mode == "fp16" else 1e-2) and pc >= 0.999, (d, pc)
    raw, safe, err = _argmax(r["phn_fc_logits"], g[f"{tag}_logits"])
    _check_argmax(mode, f"aptai_{tag}", raw, safe, err, T)
    assert np.array_equal(r["phn_fc_pred"], r["phn_fc_logits"].argmax(-1))


@pytest.mark.parametrize("mode", MODES)
def test_aptai_forward_ragged_batch(aptai_large, cuda, mode):
    g = golden2()
    lens, flen = [128000, 113000, 96000, 71000], R4_FRAMES
    wav = W.waveforms(4, 128000, lens, seed=6234).to(cuda)
    phn, tvt = (torch.from_numpy(a).to(cuda) for a in r4_targets())
    aptai_large.set_precision(mode)
    try:
        out = aptai_large(0, wav, torch.tensor(lens, device=cuda), phn, *[tvt[:, :, i].contiguous() for i in range(9)])
        pr = aptai_large.predict(wav, torch.tensor(lens, device=cuda))
    finally:
        aptai_large.set_precision("bf16")
    tvs = out["tvs_pred"].cpu().numpy()
    d = max(float(np.abs(tvs[b, :n] - g["r4_tvs"][b, :n]).max()) for b, n in enumerate(flen))
    pc = min(float(pearson(tvs[b, :n], g["r4_tvs"][b, :n]).min()) for b, n in enumerate(flen))
    losses = np.asarray([float(out["loss"]), float(out["mse_loss"]), float(out["ce_loss"])])
    rel = np.abs(losses - g["r4_losses"]) / np.abs(g["r4_losses"])
    lg = pr["phn_fc_logits"].cpu().numpy()
    valid = np.zeros((4, 399), dtype=bool)
    for b, n in enumerate(flen):
        valid[b, :n] = True
    raw, safe, err = _argmax(lg[valid], g["r4_logits"][valid])
    _report(f"aptai_forward_b4_ragged[{mode}]", {"tv_max_abs_valid": d, "pearson_min": pc, "losses": losses.tolist(),
                                                 "ref_losses": g["r4_losses"].tolist(), "loss_rel": rel.tolist()})
    assert d <= (2.5e-3 if mode == "fp16" else 1e-2) and pc >= 0.999, (d, pc)
    assert rel.max() <= (5e-3 if mode == "bf16" else 1e-3), rel
    _check_argmax(mode, "aptai_forward_b4_ragged", raw, safe, err, valid.sum())
    pred = out["phn_fc_pred"].cpu().numpy()
    agree = float((pred[valid] == g["r4_pred"].astype(np.int64)[valid]).mean())
    assert agree >= {"f32x3": 0.999, "fp16": 0.995, "bf16": 0.97}[mode], agree
    # padded-batch semantics: the same utterance alone gives the same valid frames ('layer' variant, SURVEY fact 7)
    if mode == "bf16":
        one = aptai_large.predict(wav[3:4, :71000].contiguous(), torch.tensor([71000], device=cuda))
        assert (one["phn_fc_logits"][0] - pr["phn_fc_logits"][3, :221]).abs().max().item() < 3e-2


@pytest.mark.parametrize("mode", MODES)
def test_pr_forward_config2_16x8s(cuda, mode):
    """BASELINE config 2: w2v2 phoneme recogniser CTC forward (+ d loss / d logits), batch 16 x <= 8 s, 24x1024."""
    g = golden2()
    cfg = cfg_large()
    name = register_in_memory_checkpoint("mem://large-seed0", backbone_sd(cfg, 0))
    m = Wav2Vec2_PR(cfg, None, name, VOCAB)
    hw, hb = W.linear_params(103, 46, 1024)
    with torch.no_grad():
        m.pr_head.weight.copy_(hw); m.pr_head.bias.copy_(hb)
    m = m.to(cuda).eval().set_precision(mode)
    lens = g["c2_lens"].tolist()
    wav = W.waveforms(16, 128000, lens, seed=7234).to(cuda)
    labels = torch.from_numpy(g["c2_labels"]).to(cuda)
    r = m(wav, torch.tensor(lens, device=cuda), labels, want_grad=True)
    loss, ref = float(r["loss"]), float(g["c2_loss"][0])
    rel = abs(loss - ref) / abs(ref)
    assert r["log_probs"].shape == (399, 16, 46)
    lg = r["phoneme_logits"].cpu().numpy()
    flen = [(n - 400) // 320 + 1 for n in lens]
    valid = np.zeros((16, 399), dtype=bool)
    for b, n in enumerate(flen):
        valid[b, :n] = True
    err = float(np.abs(lg[:, ::8] - g["c2_logits_sub"])[valid[:, ::8]].max())
    raw, safe, _ = _argmax(lg[valid], ref_pred=g["c2_pred"].astype(np.int64)[valid], ref_margin=g["c2_margin"][valid],
                           err=err)
    gerr = float(np.abs(r["grad_logits"].cpu().numpy()[:, ::8] - g["c2_grad_sub"]).max())
    _report(f"pr_config2_16x8s[{mode}]", {"ctc_loss": loss, "ref": ref, "rel": rel, "grad_logits_max_abs_err": gerr})
    assert rel <= 1e-3, (loss, ref)                          # north star, literal, both modes
    _check_argmax(mode, "pr_config2_16x8s", raw, safe, err, valid.sum())
    assert gerr <= {"f32x3": 2e-5, "fp16": 4e-4, "bf16": 2e-3}[mode], gerr


@pytest.mark.parametrize("mode", MODES)
def test_force_aptai_8s(cuda, mode):
    g = golden2()
    cfg = cfg_large()
    name = register_in_memory_checkpoint("mem://large-seed0", backbone_sd(cfg, 0))
    pr = Wav2Vec2_PR(cfg, None, name, VOCAB)
    hw, hb = W.linear_params(103, 46, 1024)
    with torch.no_grad():
        pr.pr_head.weight.copy_(hw); pr.pr_head.bias.copy_(hb)
    fa = Force_APTAI("unused", cuda, VOCAB, w2v2_pr=pr)
    fa.load_state_dict(force_tail_state(fa.state_dict()), strict=False)
    fa = fa.to(cuda).eval().set_precision(mode)
    wav = W.waveforms(1, 128000, None, seed=4234)
    known = g["f8_known"]
    al = fa.get_alignment(wav[0].numpy(), phn_seq=known)["alignment"]
    assert al.shape == g["f8_alignment"].shape == (45, 399)
    dp = float(np.abs(np.exp(al) - np.exp(g["f8_alignment"])).max())
    agree = float((al.argmax(0) == g["f8_alignment"].argmax(0)).mean())
    out = fa.get_faptai_output(wav[0].numpy(), phn_seq=known)
    tvs = np.stack([np.asarray(out["tvs_pred"][k], dtype=np.float32) for k in TV], -1)
    d = float(np.abs(tvs - g["f8_tvs"]).max())
    fp_agree = float((np.asarray(out["pred_frame_phns"], dtype=np.int64) == g["f8_frame_phns"]).mean())
    tvt = torch.from_numpy(f8_tv_targets()).to(cuda)
    res = fa(0, wav.to(cuda), torch.tensor([128000], device=cuda), None, None,
             *[tvt[:, :, i].contiguous() for i in range(9)], phn_seqs=[known])
    losses = np.asarray([float(res["loss"]), float(res["tv_loss"]), float(res["align_loss"])])
    rel = np.abs(losses - g["f8_losses"]) / np.abs(g["f8_losses"])
    _report(f"force_aptai_8s[{mode}]", {"alignment_prob_max_abs": dp, "frame_argmax_agreement": agree,
                                        "frame_phn_agreement": fp_agree, "tv_max_abs": d, "losses": losses.tolist(),
                                        "ref_losses": g["f8_losses"].tolist(), "loss_rel": rel.tolist()})
    assert d <= (2.5e-3 if mode == "fp16" else 1e-2), d
    if mode == "f32x3":
        assert rel.max() <= 1e-3, rel                        # align_loss is CTC-based: the CTC tolerance, literal
        assert agree >= 0.999 and fp_agree >= 0.999 and dp < 2e-3, (agree, fp_agree, dp)
    elif mode == "fp16":
        assert rel.max() <= 1e-3, rel                        # the literal tolerance at the default kernels' speed
        assert agree >= 0.99 and dp < 1e-2, (agree, dp)
    else:
        assert rel.max() <= 1e-2 and agree >= 0.95 and dp < 5e-2, (rel, agree, dp)
