#!/usr/bin/env python
"""bench.py — audio-seconds per second of the APTAI forward + alignment hot path (BASELINE.json metric).

Workload (BASELINE config 5): 4096 synthetic utterances, duration U[2, 20] s at 16 kHz, XLS-R-sized 24x1024 'layer'
backbone with random-init weights, APTAI inference (encoder -> TV head + low-pass, phoneme head + argmax) followed
by log-softmax + CTC-Viterbi forced alignment against known synthetic phoneme sequences.  One step = one pass over
all utterances, length-bucketed (padding semantics of the reference: pad to the batch maximum).
Every rank runs the full workload on its own GPU (utterance-sharded path, no collective): weak scaling (`value`).

  python bench.py --gpus 1 --steps K --warmup W            our arm (CUDA kernels through the C ABI)
  python bench.py ... --dump-outputs DIR                   also writes what the last timed step computed (a seeded
                                                           sample of utterances) as DIR/<name>.npy, to compare builds
  python bench.py --impl reference ...                     reference arm: the reference's own classes
                                                           (baseline/_ref/{aptai,modules}.py on transformers, unmodified)
                                                           on the host CPU cores, length-stratified sample

Beside the contract's keys the line carries the rest of the scorecard (VERDICT r1 #3):
  roofline          GEMM family, valid-frame algorithmic FLOPs (SURVEY 8d) / CUDA-event time of its launches
  cpu_baseline      reference classes on the host cores, bounded stratified sample (rank 0, N = 1)
  accuracy_mode     precision="f32x3" on a sample of the same batches: audio-s/s and agreement with the bf16 mode;
                    its `fp16_mode` entry: the default kernels on fp16 operands on the same batches
  library_baseline  the reference's classes in torch eager + bf16 autocast on the SAME GPU, same batches (N = 1)
  strong            ONE 4096-utterance set split over the N ranks by sweep.shard_lpt (N > 1)
  train             BASELINE config 4: APTAI training step, batch 32 / GPU, NCCL gradient all-reduce at N ranks
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from aptai_b200 import sweep  # noqa: E402
from aptai_b200.config import W2V2Config  # noqa: E402

NO_REG = dict(hidden_dropout=0.0, activation_dropout=0.0, attention_dropout=0.0, feat_proj_dropout=0.0,
              final_dropout=0.0, layerdrop=0.0, apply_spec_augment=False)
VOCAB = {"(blank)": 0, "(...)": 1, **{f"p{i}": i for i in range(2, 46)}}
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
REF_FILES = ("models/aptai.py", "models/modules.py", "models/w2v2_pr.py", "models/force_aptai.py", "utility.py")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ workload
def build_workload(cfg, n_utts, seed, max_rows):
    lengths = sweep.synth_durations(n_utts, 2.0, 20.0, seed=seed)
    batches = sweep.make_batches(cfg, lengths, bucket_width=32, max_rows=max_rows)
    return lengths, batches


def synth_batch_host(lengths, batch, seed, pin=True):
    """Host buffers of one batch: waveform fp32 [B,L] (0.1*N(0,1), zero beyond each length), lengths, known
    phoneme sequences int32 [B,59] (ids 1..45, length U{10..59} capped by the frame count)."""
    B, L = len(batch.indices), batch.samples
    g = torch.Generator().manual_seed(seed)
    wav = torch.empty((B, L), dtype=torch.float32)
    if pin:
        wav = wav.pin_memory()
    wav.normal_(0.0, 0.1, generator=g)
    lens = torch.tensor([lengths[i] for i in batch.indices], dtype=torch.int64)
    for b in range(B):
        wav[b, int(lens[b]):] = 0.0
    rng = np.random.Generator(np.random.PCG64(seed))
    tg = np.zeros((B, 59), dtype=np.int32)
    tl = np.zeros((B,), dtype=np.int32)
    for b in range(B):
        n = int(rng.integers(10, 60))
        tl[b] = n
        seq = rng.integers(1, 46, size=n)
        for j in range(1, n):                       # no adjacent repeats: always feasible for T >= 99 frames
            if seq[j] == seq[j - 1]:
                seq[j] = 1 + (seq[j] % 45)
        tg[b, :n] = seq
    out = (wav, lens, torch.from_numpy(tg), torch.from_numpy(tl))
    return tuple(t.pin_memory() if pin and not t.is_pinned() else t for t in out)


def head_params(H):
    from aptai_b200.synth import linear_params
    return linear_params(101, 9, H), linear_params(102, 46, H)


def make_model(cfg, dev):
    from aptai_b200 import APTAI
    from aptai_b200.backbone import register_in_memory_checkpoint
    from aptai_b200.synth import backbone_state_dict
    name = register_in_memory_checkpoint("mem://bench", backbone_state_dict(cfg, 0))
    m = APTAI(dev, VOCAB, name, cfg, None, phn_drop=0.0, tv_drop=0.0)
    (tvw, tvb), (pw, pb) = head_params(cfg.hidden_size)
    with torch.no_grad():
        m.tv_head[2].weight.copy_(tvw); m.tv_head[2].bias.copy_(tvb)
        m.phn_head[2].weight.copy_(pw); m.phn_head[2].bias.copy_(pb)
    return m.to(dev).eval()


def hot_path(model, wav, lens, tg, tl):
    """One batch through the public API: APTAI.predict = encoder + heads + low-pass + argmax + forced alignment.
    Returns what predict() returns to its caller."""
    return model.predict(wav, lens, phn_targets=tg, phn_target_lens=tl)


# --dump-outputs: predict()'s per-frame outputs and their widths
DUMP_FRAME_KEYS = {"tvs_pred": 9, "phn_fc_logits": 46, "log_probs": 46, "phn_fc_pred": 1, "align_paths": 1,
                   "align_scores": 1}
DUMP_BYTES = 60 * 10 ** 6          # with the .npy headers, under 64 MB in all


def dump_outputs(out_dir, cfg, lengths, batches, outs, seed=0):
    """Writes one step's outputs (`outs[k]` = predict() of batches[k]) as float32 `out_dir/<name>.npy`.
    The files stay within DUMP_BYTES: utterances are taken in a fixed, seeded order while they fit (the config-5
    step's outputs are several times larger), on their valid frames only (what lies beyond an utterance's length is
    padding that no caller reads).  Per-frame arrays are the sampled utterances'
    frames concatenated in utterance-id order, per-utterance arrays (`utterance_index`, `frames`, `align_status`)
    follow the same order.  The sample depends only on the workload, so two builds dump the same utterances."""
    frame_bytes = 4 * sum(DUMP_FRAME_KEYS.values())
    budget = (DUMP_BYTES - 3 * 4 * len(lengths)) // frame_bytes
    pick, total = [], 0
    for i in np.random.Generator(np.random.PCG64(seed)).permutation(len(lengths)):
        n = cfg.conv_out_length(lengths[i])
        if total + n <= budget:
            pick.append(int(i))
            total += n
    pick.sort()
    where = {i: (k, j) for k, b in enumerate(batches) for j, i in enumerate(b.indices)}
    cols = {name: [] for name in (*DUMP_FRAME_KEYS, "align_status")}
    for i in pick:
        k, j = where[i]
        n = cfg.conv_out_length(lengths[i])
        for name in DUMP_FRAME_KEYS:
            cols[name].append(outs[k][name][j, :n].float().cpu().numpy())
        cols["align_status"].append(outs[k]["align_status"][j: j + 1].float().cpu().numpy())
    os.makedirs(out_dir, exist_ok=True)
    arrays = {name: np.concatenate(v) for name, v in cols.items()}
    arrays["utterance_index"] = np.asarray(pick, dtype=np.float32)
    arrays["frames"] = np.asarray([cfg.conv_out_length(lengths[i]) for i in pick], dtype=np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32))


class GemmTimer:
    """CUDA-event bracket around every launch of the GEMM family (roofline leg).  The FLOPs the roofline is quoted on
    are NOT counted here (padded rows would be included): they are the valid-frame closed form of SURVEY 8d."""

    def __init__(self):
        self.ev = []

    def hook(self, a):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        self.ev.append((e0, e1))
        return e1.record

    def total_ms(self):
        return sum(e0.elapsed_time(e1) for e0, e1 in self.ev)


# ------------------------------------------------------------------------------------------------ reference classes
def ensure_reference_copy():
    """baseline/_ref/ = the reference's model files, UNMODIFIED, copied flat (the reference expects a flat import
    path, README.md:9).  Git-ignored; travels to the GPU box with the snapshot.  Copied whenever the reference tree
    is present (the build container); the GPU box uses what travelled."""
    src = os.environ.get("APTAI_REFERENCE", "/root/reference")
    if os.path.isdir(src):
        os.makedirs(REF_DIR, exist_ok=True)
        manifest = {}
        for rel in REF_FILES:
            dst = os.path.join(REF_DIR, os.path.basename(rel))
            shutil.copyfile(os.path.join(src, rel), dst)
            manifest[rel] = hashlib.sha256(open(dst, "rb").read()).hexdigest()
        json.dump(manifest, open(os.path.join(REF_DIR, "MANIFEST.json"), "w"), indent=1)
    return have_reference_copy()


def have_reference_copy():
    """Whether build() left the reference's classes in baseline/_ref/ (the benchmark itself writes nothing there)."""
    return os.path.exists(os.path.join(REF_DIR, "aptai.py"))


def load_reference_aptai(cfg, device):
    """The reference's APTAI class (baseline/_ref/aptai.py on the installed transformers), same synthetic weights as
    our arm.  Shims per SURVEY Appendix C: a local save_pretrained directory stands in for the hub id."""
    import transformers  # noqa: F401
    from transformers import Wav2Vec2Config, Wav2Vec2Model
    from aptai_b200.synth import backbone_state_dict
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import aptai as ref_aptai
    kw = dict(vocab_size=cfg.vocab_size, hidden_size=cfg.hidden_size, num_hidden_layers=cfg.num_hidden_layers,
              num_attention_heads=cfg.num_attention_heads, intermediate_size=cfg.intermediate_size,
              feat_extract_norm=cfg.feat_extract_norm, conv_bias=cfg.conv_bias,
              do_stable_layer_norm=cfg.do_stable_layer_norm, **NO_REG)
    hf = Wav2Vec2Config(**kw)
    tmp = tempfile.mkdtemp(prefix="aptai_ref_")
    try:
        m0 = Wav2Vec2Model(hf)
        m0.load_state_dict(backbone_state_dict(cfg, 0), strict=True)
        m0.save_pretrained(tmp)
        del m0
        m = ref_aptai.APTAI(device, VOCAB, tmp, hf, None, phn_drop=0.0, tv_drop=0.0)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    (tvw, tvb), (pw, pb) = head_params(cfg.hidden_size)
    with torch.no_grad():
        m.tv_head[2].weight.copy_(tvw); m.tv_head[2].bias.copy_(tvb)
        m.phn_head[2].weight.copy_(pw); m.phn_head[2].bias.copy_(pb)
    return m.to(device).eval()


class ReferenceHotPath:
    """The reference's path for one padded batch: `APTAI.forward` (models/aptai.py:58-115: backbone, heads, low-pass,
    masked losses, argmax) under no_grad, then the forced alignment the north star adds — the oracle the Viterbi
    kernel is bit-exact with, `torchaudio.functional.forced_align`, one call per utterance — on the log-softmax of the
    phoneme logits (captured by a forward hook; `forward` does not return them)."""

    def __init__(self, model, cfg, align=True):
        self.m, self.cfg, self.align = model, cfg, align
        self.logits = None
        model.phn_head.register_forward_hook(lambda mod, i, o: setattr(self, "logits", o))

    def __call__(self, wav, lens, tg, tl, autocast=None):
        import contextlib
        import torchaudio
        B = wav.shape[0]
        T = self.cfg.conv_out_length(wav.shape[1])
        dev = wav.device
        phn = torch.ones((B, T), dtype=torch.long, device=dev)
        tv = torch.zeros((B, T), dtype=torch.float32, device=dev)
        ctx = torch.autocast(dev.type, dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
        with torch.no_grad(), ctx:
            out = self.m(0, wav, lens, phn, *([tv] * 9))
        res = [out["tvs_pred"], out["phn_fc_pred"]]
        if self.align:
            lp = torch.log_softmax(self.logits.float(), -1)
            for b in range(B):
                Tb = self.cfg.conv_out_length(int(lens[b]))
                n = int(tl[b])
                p, _ = torchaudio.functional.forced_align(lp[b: b + 1, :Tb], tg[b: b + 1, :n].to(dev), blank=0)
                res.append(p)
        return res


def stratified_sample(lengths, batches, per_bucket, quantiles):
    """Length-stratified sample of the workload: `per_bucket` utterances from the batch at each duration quantile
    (the quadratic attention cost of the long utterances is in the sample, unlike a median-only pick)."""
    picks = []
    for q in quantiles:
        b = batches[min(len(batches) - 1, int(q * len(batches)))]
        idx = b.indices[-per_bucket:]
        L = max(lengths[i] for i in idx)
        picks.append(sweep.Batch(list(idx), L, None, 0.0))
    return picks


def reference_cpu_arm(cfg, lengths, batches, steps, warmup, budget_s):
    """Times the reference's own classes on the host cores.  Returns (audio-s/s, ms per step, description)."""
    torch.set_num_threads(os.cpu_count())
    if not have_reference_copy():
        raise RuntimeError("baseline/_ref is missing (__graft_entry__.build() copies it from the reference tree "
                           "named by APTAI_REFERENCE)")
    m = load_reference_aptai(cfg, torch.device("cpu"))
    ref = ReferenceHotPath(m, cfg)
    sample = stratified_sample(lengths, batches, per_bucket=1, quantiles=(0.1, 0.5, 0.9))
    host = [synth_batch_host(lengths, b, 7000 + i, pin=False) for i, b in enumerate(sample)]
    audio_s = sum(lengths[i] for b in sample for i in b.indices) / 16000.0

    def step():
        for (wav, lens, tg, tl) in host:
            ref(wav, lens, tg, tl)

    t0 = time.perf_counter()
    step()                                           # first warm-up step also sizes the run
    t_first = time.perf_counter() - t0
    n_total = warmup + steps
    if t_first * n_total > budget_s:                 # bound the whole run: fewer timed repetitions, never a smaller sample
        steps_run = max(1, int(budget_s / t_first) - 1)
        warm_run = 1
    else:
        steps_run, warm_run = steps, max(1, warmup)
    for _ in range(warm_run - 1):
        step()
    ts = []
    for _ in range(steps_run):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    dt = float(np.mean(ts))
    desc = (f"reference classes (baseline/_ref/aptai.py + transformers {__import__('transformers').__version__}, "
            f"torch CPU fp32): {len(sample)} utterances at the 10/50/90 % duration quantiles "
            f"({', '.join(f'{lengths[i] / 16000:.1f}' for b in sample for i in b.indices)} s = {audio_s:.1f} audio-s "
            f"per step), APTAI.forward + torchaudio forced_align; {steps_run} timed steps of {dt:.1f} s")
    return audio_s / dt, dt * 1e3, desc, steps_run


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the aptai_b200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its banner ("NCCL version ...") on fd 1 when the
        # communicator is created, so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    from aptai_b200 import lib, ops
    cfg = W2V2Config.large(**NO_REG)
    lengths, batches = build_workload(cfg, args.utterances, seed=rank, max_rows=args.max_rows)
    audio_s = sum(lengths) / 16000.0
    model = make_model(cfg, dev)
    host = [synth_batch_host(lengths, b, 1000 * rank + i) for i, b in enumerate(batches)]
    devb = [tuple(t.to(dev, non_blocking=True) for t in h) for h in host]
    torch.cuda.synchronize()
    padded_frames = sum(len(b.indices) * b.frames for b in batches)
    valid_frames = sum(cfg.conv_out_length(l) for l in lengths)

    n_streams = max(1, int(os.environ.get("APTAI_BENCH_STREAMS", "1")))
    side = [torch.cuda.Stream(device=dev) for _ in range(n_streams)] if n_streams > 1 else []

    def step_resident(bs=devb, sink=None):
        """`sink`: a list that receives each batch's outputs (kept alive only when they are to be dumped)"""
        if not side:
            for (wav, lens, tg, tl) in bs:
                r = hot_path(model, wav, lens, tg, tl)
                if sink is not None:
                    sink.append(r)
            return
        # independent batches alternate over `n_streams` streams: the tail of one batch's kernel is filled by the
        # other batch's next one, and HBM-bound kernels of one overlap tensor-bound kernels of the other
        cur = torch.cuda.current_stream(dev)
        for st in side:
            st.wait_stream(cur)
        for i, (wav, lens, tg, tl) in enumerate(bs):
            with torch.cuda.stream(side[i % n_streams]):
                r = hot_path(model, wav, lens, tg, tl)
            if sink is not None:
                sink.append(r)
        for st in side:
            cur.wait_stream(st)

    copy_stream = torch.cuda.Stream(device=dev)

    def step_e2e(sink, hs=host):
        """What a caller of the public API does with a list of pinned host batches: the host -> device copy of batch
        i+1 is issued on a copy stream while batch i computes (every copy and every result read-back is still inside
        the timed region; only their serialisation with the kernels is gone)."""
        main = torch.cuda.current_stream(dev)

        def upload(h):
            with torch.cuda.stream(copy_stream):
                t = tuple(x.to(dev, non_blocking=True) for x in h)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return t, ev

        nxt = upload(hs[0])
        for i in range(len(hs)):
            (w, l, g, t), ev = nxt
            if i + 1 < len(hs):
                nxt = upload(hs[i + 1])
            main.wait_event(ev)
            for x in (w, l, g, t):
                x.record_stream(main)
            r = hot_path(model, w, l, g, t)
            sink.append((r["tvs_pred"].to("cpu", non_blocking=True), r["phn_fc_pred"].to("cpu", non_blocking=True),
                         r["align_paths"].to("cpu", non_blocking=True)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    def max_over_ranks(*vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    for _ in range(args.warmup):
        step_resident()
    barrier()
    launches0 = lib.launch_count()
    clocks = ClockSampler(local)
    clocks.start()
    timer = GemmTimer()
    ops.set_gemm_hook(timer.hook)
    last = [] if args.dump_outputs and rank == 0 else None

    def step_timed():
        if last is not None:
            last.clear()                             # keep the outputs of the last timed step only
        step_resident(sink=last)

    ms = timed(step_timed, args.steps)
    ops.set_gemm_hook(None)
    clk = clocks.stop()
    launches = lib.launch_count() - launches0
    gemm_ms = timer.total_ms()
    gemm_launches = len(timer.ev)
    timer.ev.clear()
    if last is not None:
        dump_outputs(args.dump_outputs, cfg, lengths, batches, last)
        last.clear()
    # end-to-end: pinned host -> device copies and device -> host results inside the timed region
    sink = []
    step_e2e(sink)
    barrier()
    ms_e2e = timed(lambda: (sink.clear(), step_e2e(sink)), args.steps)
    sink.clear()
    h2d = sum(sum(t.numel() * t.element_size() for t in h) for h in host)
    d2h = sum(len(b.indices) * b.frames * (9 * 4 + 8 + 4) for b in batches)
    ms_max, ms_e2e_max = max_over_ranks(ms, ms_e2e)

    # ---- strong scaling: ONE utterance set (rank 0's) split over the ranks by longest-processing-time-first
    strong = None
    if world > 1:
        l0, b0 = build_workload(cfg, args.utterances, seed=0, max_rows=args.max_rows)
        shards = sweep.shard_lpt(b0, world, cfg, l0)
        mine = shards[rank]
        hs = [synth_batch_host(l0, b, 1000 * 0 + 100000 + i, pin=False) for i, b in enumerate(mine)]
        ds = [tuple(t.to(dev) for t in h) for h in hs]
        del hs
        step_resident(ds)
        ms_s = timed(lambda: step_resident(ds), args.steps)
        (ms_s_max,) = max_over_ranks(ms_s)
        loads = [sum(b.flops for b in s) for s in shards]
        strong = {"value": sum(l0) / 16000.0 * args.steps / (ms_s_max * 1e-3), "unit": "audio-s/s",
                  "ms_per_step": ms_s_max / args.steps, "scaling": "strong",
                  "workload": f"one set of {args.utterances} utterances (seed 0) split over {world} ranks by "
                              "sweep.shard_lpt on the forward-FLOP estimate (whole batches, then the tail of one batch handed "
                              "from the most to the least loaded rank until max/mean <= 1.003), no collective",
                  "flops_imbalance_max_over_mean": max(loads) / (sum(loads) / world),
                  "time_imbalance_max_over_this_rank0": ms_s_max / ms_s if rank == 0 else None}
        del ds

    # ---- accuracy mode on a sample of the same batches
    accuracy = None
    if rank == 0 and not args.no_accuracy:
        accuracy = accuracy_mode_leg(model, cfg, lengths, batches, devb, dev)
    model.set_precision("bf16")

    line = None
    if rank == 0:
        peak_tf, peak_hbm, how = peaks()
        gemm_flops = args.steps * sum(sweep.gemm_flops_utt(cfg, l) for l in lengths)
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        traffic, traffic_src, traffic_alg = None, None, None
        tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            traffic_alg = tj.get("algorithmic_bytes")
        line = {
            "metric": "audio-sec/sec APTAI fwd+align", "value": world * audio_s * args.steps / (ms_max * 1e-3),
            "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"config5: {args.utterances} utterances U[2,20]s 16kHz per GPU, XLS-R-sized 24x1024 "
                                   "'layer' backbone, APTAI heads+low-pass+argmax + log-softmax + CTC-Viterbi alignment",
                       "batches": len(batches), "bucket_width_frames": 32, "max_rows": args.max_rows,
                       "padded_over_valid_frames": padded_frames / valid_frames,
                       "l2": "inputs larger than L2 (each batch's activations >> 126 MB; weights 631 MB)",
                       "audio_s_per_gpu_per_step": audio_s, "parallelism": f"utterance-sharded x{world}, no collective"},
            "e2e": {"value": world * audio_s * args.steps / (ms_e2e_max * 1e-3), "unit": "audio-s/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tcgen05_kernel (all launches of the GEMM family)",
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "traffic": traffic, "traffic_source": traffic_src, "traffic_algorithmic_bytes": traffic_alg,
                         "peak_source": how,
                         "flops": "valid frames only (SURVEY 8d closed form over the step's utterance lengths)",
                         "gemm_share_of_step": gemm_ms / ms, "gemm_launches": gemm_launches,
                         "whole_step_tflops": args.steps * sum(sweep.flops_utt(cfg, l) for l in lengths) / (ms * 1e-3) / 1e12},
        }
        if strong is not None:
            line["strong"] = strong
        if accuracy is not None:
            line["accuracy_mode"] = accuracy
    # free the inference state before the training leg
    del devb, host
    torch.cuda.empty_cache()

    if not args.no_train:
        tr = train_leg(cfg, dev, rank, world, args)
        if rank == 0:
            line["train"] = tr
    if rank == 0 and world == 1 and not args.no_library_baseline:
        try:
            line["library_baseline"] = library_baseline_leg(cfg, lengths, batches, dev, model)
        except Exception as e:                                              # noqa: BLE001
            line["library_baseline"] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            v, ms_ref, desc, _ = reference_cpu_arm(cfg, lengths, batches, steps=3, warmup=1, budget_s=args.cpu_budget)
            line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": torch.get_num_threads(),
                                    "kind": "reference", "sample": desc}
        except Exception as e:                                              # noqa: BLE001
            line["cpu_baseline"] = cpu_baseline_port(cfg, lengths, batches, budget_s=args.cpu_budget)
            line["cpu_baseline"]["note"] = f"reference classes unavailable ({type(e).__name__}: {str(e)[:120]})"
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def accuracy_mode_leg(model, cfg, lengths, batches, devb, dev):
    """precision='f32x3' on three of the step's batches (short / median / long): throughput and agreement with the
    default mode on the valid frames."""
    pick = sorted({len(batches) // 6, len(batches) // 2, (5 * len(batches)) // 6})
    audio = sum(lengths[i] for k in pick for i in batches[k].indices) / 16000.0

    def run(mode):
        model.set_precision(mode)
        outs = []
        for k in pick:
            wav, lens, tg, tl = devb[k]
            outs.append(model.predict(wav, lens, phn_targets=tg, phn_target_lens=tl))
        return outs

    ref = run("bf16")
    run("f32x3")                                     # warm-up (plan build)
    run("fp16")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_run(mode, reps):
        """`reps` back-to-back passes over the sample (the power cap needs a second to act: a single 0.2 s pass of a
        16-bit mode runs at boost clocks the sustained step never sees)"""
        run(mode)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            o = run(mode)
        e1.record()
        torch.cuda.synchronize()
        return o, e0.elapsed_time(e1) / reps

    acc, ms = timed_run("f32x3", 2)
    _, ms16 = timed_run("bf16", 8)
    half, ms_h = timed_run("fp16", 8)
    _, ms16b = timed_run("bf16", 8)                  # bf16 again behind fp16: the pair brackets box drift
    ms16 = 0.5 * (ms16 + ms16b)

    def compare(outs):
        """valid-frame agreement of one mode's outputs with the accuracy mode's"""
        n = d = same = 0
        tv_d = lg_d = 0.0
        for k, a, r in zip(pick, acc, outs):
            flen = torch.tensor([cfg.conv_out_length(lengths[i]) for i in batches[k].indices], device=dev)
            T = a["phn_fc_pred"].shape[1]
            valid = torch.arange(T, device=dev)[None, :] < flen[:, None]
            n += int(((a["phn_fc_pred"] == r["phn_fc_pred"]) & valid).sum())
            d += int(valid.sum())
            tv_d = max(tv_d, float((a["tvs_pred"] - r["tvs_pred"]).abs()[valid].max()))
            lg_d = max(lg_d, float((a["phn_fc_logits"] - r["phn_fc_logits"]).abs()[valid].max()))
            same += int(((a["align_paths"] == r["align_paths"]) & valid).sum())
        return {"phoneme_argmax_agreement_valid_frames": n / d, "frames": d, "tv_max_abs": tv_d, "logit_max_abs": lg_d,
                "viterbi_path_agreement_valid_frames": same / max(1, d)}

    model.set_precision("bf16")
    return {"precision": "f32x3 (every contraction as three bf16 products on hi/lo operand pairs, fp32 elsewhere)",
            "value": audio / (ms * 1e-3), "unit": "audio-s/s", "bf16_value_same_batches": audio / (ms16 * 1e-3),
            "sample": f"batches {pick} of {len(batches)} ({audio:.0f} audio-s)",
            "bf16_vs_f32x3": compare(ref),
            "fp16_mode": {"precision": "fp16 (the default kernels on IEEE fp16 operands: weights, activations, attention "
                                       "probabilities; fp32 accumulation, residual stream and statistics)",
                          "value": audio / (ms_h * 1e-3), "unit": "audio-s/s", "fp16_vs_f32x3": compare(half)},
            "parity": "north-star tolerances are asserted literally against the reference's goldens in the f32x3 mode "
                      "(tests/test_parity_gpu.py); the bf16 mode meets the TV / CTC-loss tolerances, the fp16 mode "
                      "also every CTC-type loss tolerance at 7x smaller logit / trajectory error"}


def library_baseline_leg(cfg, lengths, batches, dev, ours):
    """The existing Blackwell library path: the reference's classes, torch eager + bf16 autocast (cuBLAS / cuDNN / SDPA)
    on the same GPU, on a stratified third of the same batches; our arm timed on exactly those batches beside it."""
    if not have_reference_copy():
        return {"unavailable": "baseline/_ref missing"}
    pick = list(range(1, len(batches), 6))
    hs = [synth_batch_host(lengths, batches[k], 1000 * 0 + k, pin=False) for k in pick]
    ds = [tuple(t.to(dev) for t in h) for h in hs]
    audio = sum(lengths[i] for k in pick for i in batches[k].indices) / 16000.0
    m = load_reference_aptai(cfg, dev)
    ref = ReferenceHotPath(m, cfg, align=True)
    note = "APTAI.forward (bf16 autocast) + torchaudio forced_align on the GPU"
    try:
        ref(*[t[:2] if t.dim() else t for t in (ds[0][0][:2], ds[0][1][:2], ds[0][2][:2], ds[0][3][:2])], autocast=True)
    except Exception as e:                                                  # noqa: BLE001
        ref.align = False
        note = f"APTAI.forward (bf16 autocast); alignment excluded (torchaudio forced_align on CUDA: {type(e).__name__})"

    def run_ref():
        for (wav, lens, tg, tl) in ds:
            ref(wav, lens, tg, tl, autocast=True)

    def run_ours():
        for (wav, lens, tg, tl) in ds:
            hot_path(ours, wav, lens, tg, tl)

    def ev(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    ms_ref, ms_ours = ev(run_ref), ev(run_ours)
    del m, ref, ds
    torch.cuda.empty_cache()
    return {"value": audio / (ms_ref * 1e-3), "unit": "audio-s/s", "what": note,
            "ours_same_batches": audio / (ms_ours * 1e-3),
            "sample": f"batches {pick[0]}::6 of {len(batches)} ({len(pick)} batches, {audio:.0f} audio-s), device-resident"}


def train_leg(cfg, dev, rank, world, args):
    """BASELINE config 4: APTAI training step (articulatory MSE + phoneme CE), 24x1024, batch 32 x <= 8 s per GPU,
    frozen conv encoder, fused Adam; at N > 1 data-parallel with the NCCL gradient all-reduce overlapped with the
    backward.  Reports ms / step (CUDA events, max over ranks), the forward / backward / optimizer split, the exposed
    all-reduce time (same step with the exchange switched off) and a gradient check (all-reduced gradient == mean
    over ranks of the single-rank gradients of the same batches)."""
    import torch.distributed as dist
    from aptai_b200 import APTAI, lib
    from aptai_b200.backbone import register_in_memory_checkpoint
    from aptai_b200.synth import backbone_state_dict
    from aptai_b200.train import FusedAdam
    B, L = 32, 128000
    T = cfg.conv_out_length(L)
    name = register_in_memory_checkpoint("mem://bench-train", backbone_state_dict(cfg, 0))
    model = APTAI(dev, VOCAB, name, cfg, None, phn_drop=0.0, tv_drop=0.0)
    (tvw, tvb), (pw, pb) = head_params(cfg.hidden_size)
    with torch.no_grad():
        model.tv_head[2].weight.copy_(tvw); model.tv_head[2].bias.copy_(tvb)
        model.phn_head[2].weight.copy_(pw); model.phn_head[2].bias.copy_(pb)
    model = model.to(dev).train()

    def batch(r):
        rng = np.random.Generator(np.random.PCG64(21 + r))
        g = torch.Generator().manual_seed(1234 + r)
        lens = rng.integers(64000, 128001, size=B)
        lens[0] = L
        wav = torch.empty((B, L)).normal_(0.0, 0.1, generator=g)
        phn = np.zeros((B, T), dtype=np.int64)
        tvt = np.full((B, T, 9), -100.0, dtype=np.float32)
        for b in range(B):
            wav[b, int(lens[b]):] = 0
            n = cfg.conv_out_length(int(lens[b]))
            phn[b, :n] = rng.integers(1, 46, size=n)
            tvt[b, :n] = rng.standard_normal((n, 9), dtype=np.float32)
        return (0, wav.to(dev), torch.as_tensor(lens).to(dev), torch.from_numpy(phn).to(dev),
                *[torch.from_numpy(tvt[:, :, i]).to(dev) for i in range(9)]), float(lens.sum()) / 16000.0

    mine, audio_s = batch(rank)
    opt = FusedAdam([p for p in model.parameters() if p.requires_grad], lr=1e-5)
    check = None
    if world > 1:
        model.enable_data_parallel()
        red = model._reducer
        # gradient check first (weights identical on all ranks after the broadcast)
        object.__setattr__(model, "_reducer", None)
        gb = model.grad_buffer()
        ref = torch.zeros_like(gb.flat)
        for r in range(world):
            gb.zero()
            model(*(mine if r == rank else batch(r)[0]))["loss"].backward()
            ref += gb.flat / world
        object.__setattr__(model, "_reducer", red)
        opt.zero_grad()
        model(*mine)["loss"].backward()
        gb.wait_pending()                                   # the reducer leaves the last waits to the optimizer
        torch.cuda.synchronize()
        err = torch.tensor([float((gb.flat - ref).norm() / ref.norm())], dtype=torch.float64, device=dev)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        # tolerance: the two gradients differ by the order of the fp32 atomics of the split-frame weight-gradient and
        # dQ reductions, whose results are rounded to bf16 before the next GEMM (observed 1e-4 at this size; a wrong
        # reduction — a missing rank, SUM instead of AVG — shows as >= 0.3)
        check = {"dp_grad_check": "ok" if float(err) < 1e-3 else "FAILED", "rel_err_max_over_ranks": float(err),
                 "dp_grad_check_tolerance": 1e-3}
        del ref
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def step(times=None):
        e = [ev() for _ in range(4)]
        e[0].record()
        opt.zero_grad()
        out = model(*mine)
        e[1].record()
        out["loss"].backward()
        e[2].record()
        opt.step()
        e[3].record()
        if times is not None:
            times.append(e)

    def timed(n):
        times = []
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0, t1 = ev(), ev()
        t0.record()
        for _ in range(n):
            step(times)
        t1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([t0.elapsed_time(t1) / n], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), times

    for _ in range(3):
        step()
    l0 = lib.launch_count()
    n = max(5, min(args.train_steps, 50))
    ms, times = timed(n)
    launches = (lib.launch_count() - l0) / n
    out = {"workload": "config4: APTAI training step, 24x1024, batch 32 x <= 8 s per GPU, frozen conv encoder, fused "
                       "Adam" + (f", data-parallel x{world}: NCCL all-reduce of the flat fp32 gradient (AVG), buckets "
                                 "of 4 encoder layers overlapped with the backward" if world > 1 else ""),
           "n_gpus": world, "steps": n, "ms_per_step": ms, "audio_s_per_s": world * audio_s / (ms * 1e-3),
           "fwd_ms": float(np.mean([e[0].elapsed_time(e[1]) for e in times])),
           "bwd_ms": float(np.mean([e[1].elapsed_time(e[2]) for e in times])),
           "opt_ms": float(np.mean([e[2].elapsed_time(e[3]) for e in times])),
           "launches_per_step": launches, "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
    if world > 1:
        gb = model.grad_buffer()
        red = model._reducer
        object.__setattr__(model, "_reducer", None)              # same step without the exchange
        for _ in range(2):
            step()
        ms0, _ = timed(n)
        object.__setattr__(model, "_reducer", red)
        out.update(check)
        out.update({"ms_per_step_without_allreduce": ms0, "exposed_allreduce_ms": ms - ms0,
                    "allreduce_bytes_per_step": int(gb.numel) * 4})
    del model, opt
    torch.cuda.empty_cache()
    return out


def cpu_baseline_port(cfg, lengths, batches, budget_s=15.0):
    """Fallback when the reference's classes cannot be loaded: the oracle port (torch-CPU fp32 restatement)."""
    from oracle import ctc as octc
    from oracle import heads as oh
    from oracle import w2v2 as ow
    from oracle.weights import backbone_state_dict
    torch.set_num_threads(os.cpu_count())
    sd = backbone_state_dict(cfg, 0)
    (tvw, tvb), (pw, pb) = head_params(cfg.hidden_size)
    taps = oh.lowpass_taps()
    sample = stratified_sample(lengths, batches, per_bucket=1, quantiles=(0.1, 0.5, 0.9))
    host = [synth_batch_host(lengths, b, 7000 + i, pin=False) for i, b in enumerate(sample)]
    audio_s = sum(lengths[i] for b in sample for i in b.indices) / 16000.0

    def once():
        with torch.no_grad():
            for (wav, lens, tg, tl) in host:
                ll = [int(x) for x in lens]
                h = ow.forward(sd, cfg, wav, ll)[-1]
                _, tv, logits = oh.aptai_heads(h, tvw, tvb, pw, pb, taps)
                lp = torch.log_softmax(logits, -1).numpy()
                for i, n in enumerate(ll):
                    octc.viterbi_align(lp[i, : cfg.conv_out_length(n)], tg[i, : int(tl[i])].numpy(), blank=0)

    once()
    t0 = time.perf_counter()
    n = 0
    while True:
        once()
        n += 1
        if time.perf_counter() - t0 >= budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": n * audio_s / dt, "unit": "audio-s/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} passes over {len(sample)} utterances at the 10/50/90 % duration quantiles "
                      f"({audio_s:.1f} audio-s per pass, fp32, {dt:.1f} s of CPU work)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cfg = W2V2Config.large(**NO_REG)
    lengths, batches = build_workload(cfg, args.utterances, seed=0, max_rows=args.max_rows)
    world = int(os.environ.get("WORLD_SIZE", 1))
    try:
        v, ms_step, desc, steps_run = reference_cpu_arm(cfg, lengths, batches, steps=args.steps, warmup=args.warmup,
                                                        budget_s=args.reference_budget)
        base = {"value": v, "unit": "audio-s/s", "cores": torch.get_num_threads(), "kind": "reference", "sample": desc}
    except Exception as e:                                                  # noqa: BLE001
        base = cpu_baseline_port(cfg, lengths, batches, budget_s=min(60.0, args.reference_budget))
        base["note"] = f"reference classes unavailable ({type(e).__name__}: {str(e)[:160]}); oracle port timed instead"
        v, ms_step, steps_run = base["value"], None, args.steps
    line = {"impl": "reference", "metric": "audio-sec/sec APTAI fwd+align", "value": v, "unit": "audio-s/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "timed_steps_run": steps_run,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config5 sample: {base['sample']}", "parallelism": "host CPU threads"},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--utterances", type=int, default=4096)
    ap.add_argument("--max-rows", type=int, default=75776)   # 4 x (74 CTA pairs x 256 rows)
    ap.add_argument("--cpu-budget", type=float, default=25.0)
    ap.add_argument("--reference-budget", type=float, default=150.0)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-accuracy", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0; float32, "
                         "valid frames of a fixed, seeded sample of utterances)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
