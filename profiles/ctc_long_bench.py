"""CTC loss + gradient and CTC-Viterbi timing across the 511-label boundary and for long transcripts.

Times (CUDA events, shapes warmed, mean over repeated calls) `ops.logsoftmax_ctc` (log-probs, loss and gradient)
and `ops.ctc_viterbi`, next to the library baselines on the same GPU: `F.ctc_loss` (cuda, fp32, log_softmax +
forward + backward) and `torchaudio.functional.forced_align` (one utterance per call, so a batch is a loop).
Cases: S = 511 (register kernel) against S = 512 (CTA kernel) at the same T, then T = 2999 / S = 1000 and
T = 8999 / S = 4095, each at B = 1 and B = 16; V = 46.  Prints one JSON document (card name and power limit
included) and writes it to --out.

    python profiles/ctc_long_bench.py --out /tmp/ctc_long_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from aptai_b200 import ops  # noqa: E402

V = 46
CASES = [(1, 1500, 511), (1, 1500, 512), (16, 1500, 511), (16, 1500, 512),
         (1, 2999, 1000), (16, 2999, 1000), (1, 8999, 4095), (16, 8999, 4095)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def timed(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def inputs(B, T, S, dev):
    g = torch.Generator().manual_seed(B * 100003 + T * 31 + S)
    logits = torch.randn((B, T, V), generator=g).to(dev)
    tg = torch.randint(1, V, (B, S), generator=g, dtype=torch.int32).to(dev)
    il = torch.full((B,), T, dtype=torch.int32, device=dev)
    tl = torch.full((B,), S, dtype=torch.int32, device=dev)
    return logits, tg, il, tl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--no-baselines", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"card": card(), "V": V, "unit": "ms per call (mean)", "cases": []}
    for B, T, S in CASES:
        logits, tg, il, tl = inputs(B, T, S, dev)
        lp = torch.log_softmax(logits, -1).contiguous()
        reps = args.reps if T * S < 5_000_000 else max(3, args.reps // 3)
        row = {"B": B, "T": T, "S": S, "kernel": "register (warp)" if S <= 511 else "CTA-wide"}
        row["aptai_ctc_loss_grad"] = timed(lambda: ops.logsoftmax_ctc(logits, tg, il, tl, want_grad=True), reps)
        row["aptai_ctc_loss_only"] = timed(lambda: ops.logsoftmax_ctc(logits, tg, il, tl, want_grad=False), reps)
        row["aptai_viterbi"] = timed(lambda: ops.ctc_viterbi(lp, tg, il, tl), reps)
        if not args.no_baselines:
            x = logits.clone().requires_grad_(True)
            tgl, ill, tll = tg.long(), il.long(), tl.long()

            def torch_ctc():
                x.grad = None
                loss = F.ctc_loss(torch.log_softmax(x, -1).transpose(0, 1), tgl, ill, tll, blank=0,
                                  reduction="sum", zero_infinity=True)
                loss.backward()
            row["torch_ctc_loss_fwd_bwd"] = timed(torch_ctc, reps)
            try:
                import torchaudio.functional as AF

                def ta_align():
                    for b in range(B):
                        AF.forced_align(lp[b:b + 1], tg[b:b + 1], il[b:b + 1], tl[b:b + 1], blank=0)
                row["torchaudio_forced_align"] = timed(ta_align, max(2, reps // 2), warm=1)
            except Exception as e:      # noqa: BLE001  (a missing baseline is reported, not fatal)
                row["torchaudio_forced_align"] = f"unavailable: {type(e).__name__}: {e}"[:200]
        del logits, lp
        torch.cuda.empty_cache()
        res["cases"].append(row)
        print(json.dumps(row), flush=True)
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
