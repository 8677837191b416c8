#!/usr/bin/env python
"""Timing of the recogniser head and the CTC kernels for wide vocabularies (CUDA events, one GPU):

  head forward / backward at M = 75,776 rows (the frames of one bench.py batch) and H = 1024 for
  V = 46 (the fused SIMT heads kernel), 392 and 1024 (split-operand tensor-core head + row kernel);
  logsoftmax_ctc (loss + gradient) and ctc_viterbi at B = 16, T = 999 for V = 46 and 1024, 200 labels (register
  kernels) and 600 labels (CTA-wide kernels): the V = 46 row isolates what the wider vocabulary adds.

  python profiles/wide_vocab_bench.py --out profiles/wide_vocab_bench.json

Inputs are larger than the 126 MB L2 for the head (h alone is 310 MB); the CTC inputs (65 MB at V = 1024) are not.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from aptai_b200 import ops  # noqa: E402

M, H = 75776, 1024


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def head_case(V, dev, warmup, iters):
    g = torch.Generator(device=dev).manual_seed(V)
    h = torch.randn((M, H), device=dev, generator=g)
    w = torch.randn((V, H), device=dev, generator=g) * H ** -0.5
    b = torch.randn((V,), device=dev, generator=g) * 0.1
    d = torch.randn((M, V), device=dev, generator=g) * 1e-3
    dw, db = torch.zeros_like(w), torch.zeros_like(b)
    if V <= ops.PR_HEAD_NARROW:
        fwd = lambda: ops.heads(h, None, None, 0, w, b, ops.ACT_NONE, want_argmax=False)
        bwd = lambda: ops.heads_bwd(h, None, None, 0, None, None, d, w, ops.ACT_NONE, dw, db)
        kernel = "aptai_heads / aptai_heads_bwd (SIMT)"
    else:
        fwd = lambda: ops.logits_rows(ops.pr_head_wide(h, w, b))
        bwd = lambda: ops.pr_head_wide_bwd(h, w, d, dw, db)
        kernel = "aptai_pr_head_wide + aptai_logits_rows / aptai_pr_head_wide_bwd (split-operand tcgen05)"
    raw = (ops.pr_head_wide(h, w, b) if V > ops.PR_HEAD_NARROW else None)
    rows_ms = timed(lambda: ops.logits_rows(raw), warmup, iters) if raw is not None else None
    f_ms, b_ms = timed(fwd, warmup, iters), timed(bwd, warmup, iters)
    Vp = (V + 63) // 64 * 64 if V > ops.PR_HEAD_NARROW else V
    # split-operand products: K tripled (forward, dgrad) / three wgrad products
    tc_flop_f, tc_flop_b = 2.0 * M * Vp * 3 * H, 2 * (2.0 * M * Vp * 3 * H)
    return {"V": V, "M": M, "H": H, "kernel": kernel, "forward_ms": round(f_ms, 4), "backward_ms": round(b_ms, 4),
            "logits_rows_ms": None if rows_ms is None else round(rows_ms, 4),
            "bf16_tensor_flop_forward": tc_flop_f if V > ops.PR_HEAD_NARROW else None,
            "bf16_tensor_flop_backward": tc_flop_b if V > ops.PR_HEAD_NARROW else None}


def ctc_case(V, S, dev, warmup, iters):
    B, T = 16, 999
    rng = np.random.default_rng(S + V)
    logits = torch.from_numpy(rng.standard_normal((B, T, V)).astype(np.float32) * 2).to(dev)
    tg = torch.from_numpy(rng.integers(1, V, size=(B, S)).astype(np.int32)).to(dev)
    il = torch.full((B,), T, dtype=torch.int32, device=dev)
    tl = torch.full((B,), S, dtype=torch.int32, device=dev)
    lp = torch.log_softmax(logits, -1).contiguous()
    ctc = lambda: ops.logsoftmax_ctc(logits, tg, il, tl, blank=0, want_grad=True)
    vit = lambda: ops.ctc_viterbi(lp, tg, il, tl, blank=0)
    return {"V": V, "B": B, "T": T, "labels": S, "path": "register" if S <= 511 else "cta",
            "logsoftmax_ctc_grad_ms": round(timed(ctc, warmup, iters), 4),
            "ctc_viterbi_ms": round(timed(vit, warmup, iters), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wide_vocab_bench.json"))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_vocab_bench: no CUDA device")
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "timing": "CUDA events, mean of --iters calls",
           "head": [head_case(V, dev, a.warmup, a.iters) for V in (46, 392, 1024)],
           "ctc": [ctc_case(V, S, dev, a.warmup, a.iters) for S in (200, 600) for V in (46, 1024)]}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
