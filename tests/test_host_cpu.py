"""CPU suite (no GPU): C-ABI surface, host-side bucketing/sharding logic, drop-in module layout, and the
world_size-2 gloo run of the utterance-sharded path's host logic."""
import os
import re
import subprocess
import sys

import pytest
import torch

from helpers import ROOT, VOCAB, cfg_base, cfg_large
from aptai_b200 import sweep
from aptai_b200.config import W2V2Config


def test_cabi_library_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    from aptai_b200 import lib
    L = lib.load()
    hdr = open(os.path.join(ROOT, "include", "aptai_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(aptai_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/aptai_b200.h but not exported"
        assert name in lib.PROTOTYPES, f"{name} has no ctypes prototype in aptai_b200/lib.py"
    assert L.aptai_version() >= 100
    assert isinstance(lib.last_error(), str)


def test_cabi_struct_layouts_match_the_ctypes_mirrors(tmp_path):
    """The two structs that cross the C ABI by pointer (aptai_gemm_args, aptai_prep_entry): size and every field offset
    as a C compiler sees include/aptai_b200.h == the ctypes mirrors in aptai_b200/lib.py (a drifted field would
    silently shift every argument behind it)."""
    import ctypes as C
    import shutil
    from aptai_b200 import lib
    gcc = shutil.which("gcc") or shutil.which("cc")
    if gcc is None:
        pytest.skip("no C compiler")
    mirrors = {"aptai_gemm_args": lib.GemmArgs, "aptai_prep_entry": lib.PrepEntry}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "aptai_b200.h"', 'int main(void) {']
    for cname, cls in mirrors.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    seen = {}
    for ln in out:
        if ln.strip():
            cname, fname, val = ln.split()
            seen[(cname, fname)] = int(val)
    for cname, cls in mirrors.items():
        assert seen[(cname, "size")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert seen[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)
    assert C.sizeof(lib.PrepEntry) == 64


def test_compute_entry_points_fail_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from aptai_b200 import lib
    L = lib.load()
    rc = L.aptai_layernorm(None, 0, 1, 512, None, None, 1e-5, None, None, 0, None)
    assert rc != 0
    assert "CUDA" in lib.last_error() or "device" in lib.last_error()
    from aptai_b200 import ops
    with pytest.raises(RuntimeError):
        ops.layernorm(torch.zeros(4, 512), torch.ones(512), torch.zeros(512))       # CPU tensor: no CPU path


def test_backbone_state_dict_layout_matches_hf_names():
    from aptai_b200.backbone import Wav2Vec2Backbone
    for cfg, n in ((cfg_base(), 211), (cfg_large(), 422)):
        m = Wav2Vec2Backbone(cfg)
        keys = list(m.state_dict().keys())
        assert len(keys) == n
        assert "encoder.pos_conv_embed.conv.parametrizations.weight.original0" in keys
        assert "feature_projection.projection.weight" in keys
    total = sum(p.numel() for p in Wav2Vec2Backbone(cfg_base()).parameters())
    assert total == 94371712                      # SURVEY.md §8c known answer (base)


def test_hf_config_objects_are_accepted():
    from transformers import Wav2Vec2Config
    hf = Wav2Vec2Config(vocab_size=46, hidden_size=1024, num_hidden_layers=24, num_attention_heads=16,
                        intermediate_size=4096, feat_extract_norm="layer", conv_bias=True, do_stable_layer_norm=True)
    c = W2V2Config.from_any(hf)
    assert c.hidden_size == 1024 and c.do_stable_layer_norm and c.conv_kernel == (10, 3, 3, 3, 3, 2, 2)
    c.validate_for_kernels()


def test_bucketing_and_lpt_sharding():
    cfg = cfg_large()
    lengths = sweep.synth_durations(4096, 2.0, 20.0, seed=0)
    assert min(lengths) >= 32000 and max(lengths) <= 320000
    batches = sweep.make_batches(cfg, lengths, bucket_width=32, max_rows=49152)
    seen = sorted(i for b in batches for i in b.indices)
    assert seen == list(range(4096))                                   # every utterance exactly once
    for b in batches:
        Ts = [cfg.conv_out_length(lengths[i]) for i in b.indices]
        assert max(Ts) - min(Ts) <= 32 and len(b.indices) * b.frames <= 49152
        assert b.frames == max(Ts)
    padded = sum(len(b.indices) * b.frames for b in batches)
    valid = sum(cfg.conv_out_length(l) for l in lengths)
    assert padded / valid < 1.03
    shards = sweep.shard_lpt(batches, 8)
    loads = [sum(b.flops for b in s) for s in shards]
    assert max(loads) / min(loads) < 1.10   # 50 coarse batches over 8 ranks
    assert sorted(i for s in shards for b in s for i in b.indices) == list(range(4096))
    # refined assignment (tails of batches handed from the most to the least loaded rank): still a partition, every
    # batch still inside its length bucket and row budget, max / mean within 0.5 %
    for world in (2, 4, 8):
        fine = sweep.shard_lpt(batches, world, cfg, lengths)
        assert sorted(i for s in fine for b in s for i in b.indices) == list(range(4096))
        fl = [sum(b.flops for b in s) for s in fine]
        assert max(fl) / (sum(fl) / world) <= 1.005, (world, fl)
        for s in fine:
            for b in s:
                Ts = [cfg.conv_out_length(lengths[i]) for i in b.indices]
                assert max(Ts) - min(Ts) <= 32 and len(b.indices) * b.frames <= 49152 and b.frames == max(Ts)
                assert abs(b.flops - sum(sweep.flops_utt(cfg, lengths[i]) for i in b.indices)) <= 1e-6 * b.flops
    # closed-form FLOPs (SURVEY.md §8d): large, 8 s -> 303.06 GFLOP
    assert abs(sweep.flops_utt(cfg, 128000) / 1e9 - 303.06) < 0.5


def test_two_rank_gloo_sharded_run():
    """world_size 2 on CPU (gloo): each rank takes its LPT shard, the shards partition the workload, and the
    max-over-ranks reduction used by bench.py works."""
    script = os.path.join(ROOT, "tests", "_gloo_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731", script], capture_output=True,
                       text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "GLOO_OK" in r.stdout


def test_two_rank_gloo_data_parallel_gradients():
    """world_size 2 on CPU (gloo): flat gradient buffer layout, layer-bucketed overlapped all-reduce with averaging,
    parameter broadcast — the host logic of the data-parallel training step (BASELINE config 4)."""
    script = os.path.join(ROOT, "tests", "_gloo_dp_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29741", script], capture_output=True,
                       text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "GLOO_DP_OK" in r.stdout


def test_specaugment_masks_match_transformers():
    """aptai_b200.specaug restates transformers' `_compute_mask_indices` (HF:101-217) on the same global NumPy RNG."""
    import numpy as np
    from transformers.models.wav2vec2.modeling_wav2vec2 import _compute_mask_indices
    from aptai_b200.specaug import compute_mask_indices
    cases = [((4, 399), 0.05, 10, [399, 250, 399, 120], 2), ((2, 99), 0.05, 10, [99, 74], 2), ((3, 999), 0.2, 10, None, 0),
             ((5, 60), 0.5, 4, [60, 3, 5, 60, 30], 1), ((1, 20), 0.01, 10, [15], 0), ((2, 49), 0.65, 10, [49, 9], 2)]
    for seed, (shape, prob, length, lens, mn) in enumerate(cases):
        am = None
        if lens is not None:
            am = torch.zeros(shape, dtype=torch.long)
            for b, n in enumerate(lens):
                am[b, :n] = 1
        np.random.seed(100 + seed)
        ref = _compute_mask_indices(shape, prob, length, attention_mask=am, min_masks=mn)
        np.random.seed(100 + seed)
        got = compute_mask_indices(shape, prob, length, frame_lens=lens, min_masks=mn)
        assert np.array_equal(ref, got), (shape, prob, length, lens, mn)
        # the generator state advanced identically:
        np.random.seed(100 + seed); _compute_mask_indices(shape, prob, length, attention_mask=am, min_masks=mn)
        a = np.random.rand()
        np.random.seed(100 + seed); compute_mask_indices(shape, prob, length, frame_lens=lens, min_masks=mn)
        assert a == np.random.rand()


def test_force_aptai_parameter_layout_matches_reference_counts():
    """Drop-in boundary of Force_APTAI (models/force_aptai.py:20-78): 1 356 937 trainable tail parameters over the 21
    tensors the reference trains, 315 485 921 frozen ones for the 24x1024 recogniser (SURVEY.md §8a row a8), and the
    names the golden gradients of the reference's class are keyed by."""
    import numpy as np
    from aptai_b200 import Force_APTAI, Wav2Vec2_PR
    from aptai_b200.backbone import register_in_memory_checkpoint
    from helpers import ROOT, VOCAB, backbone_sd
    cfg = cfg_large(vocab_size=46)
    name = register_in_memory_checkpoint("mem://large-seed0-layout", backbone_sd(cfg, 0))
    fa = Force_APTAI("unused", "cpu", VOCAB, w2v2_pr=Wav2Vec2_PR(cfg, None, name, VOCAB))
    train = {n: p for n, p in fa.named_parameters() if p.requires_grad}
    frozen = [p for p in fa.parameters() if not p.requires_grad]
    assert sum(p.numel() for p in train.values()) == 1356937
    assert sum(p.numel() for p in frozen) == 315485921          # recogniser + the 51 float64 low-pass taps
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_force_train_v1.npz"))
    assert sorted(train) == sorted(str(n) for n in g["grad_names"])
    gb = fa.grad_buffer()                       # flat gradient storage: every trainable .grad is a view into it
    assert all(gb.owns(p) for p in train.values()) and gb.numel >= 1356937


def test_aptai_and_pr_parameter_counts_match_reference():
    """SURVEY.md §8a rows a1 / a5: APTAI = backbone + 9 225 (TV head) + 47 150 (phoneme head) + 51 fp64 low-pass
    taps; Wav2Vec2_PR = backbone + Linear(H, 46)."""
    from aptai_b200 import APTAI, Wav2Vec2_PR
    from aptai_b200.backbone import register_in_memory_checkpoint
    from helpers import VOCAB, backbone_sd
    cfg = cfg_large(vocab_size=46)
    name = register_in_memory_checkpoint("mem://large-seed0-layout", backbone_sd(cfg, 0))
    m = APTAI("cpu", VOCAB, name, cfg, None)
    n_backbone = sum(p.numel() for p in m.wav2vec2.parameters())
    assert sum(p.numel() for p in m.tv_head.parameters()) == 9225
    assert sum(p.numel() for p in m.phn_head.parameters()) == 47150
    assert m.tv_lowpass.lowpass.weight.dtype == torch.float64 and m.tv_lowpass.lowpass.weight.numel() == 51
    assert sum(p.numel() for p in m.parameters()) == n_backbone + 9225 + 47150 + 51
    pr = Wav2Vec2_PR(cfg, None, name, VOCAB)
    assert sum(p.numel() for p in pr.parameters()) == n_backbone + 1024 * 46 + 46
    assert n_backbone + 1024 * 46 + 46 + 51 == 315485921          # what Force_APTAI freezes (row a8)


def test_bench_dump_outputs_sample_and_layout(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 files within the byte budget, valid frames of the sampled utterances laid out
    in utterance order, and the same sample on every run of the same workload."""
    import numpy as np
    import bench
    cfg = cfg_large()
    lengths, batches = bench.build_workload(cfg, 64, seed=0, max_rows=4096)
    g = torch.Generator().manual_seed(0)
    outs = []
    for b in batches:
        B, T = len(b.indices), b.frames
        outs.append({"tvs_pred": torch.randn(B, T, 9, generator=g), "phn_fc_logits": torch.randn(B, T, 46, generator=g),
                     "log_probs": torch.randn(B, T, 46, generator=g), "phn_fc_pred": torch.randint(0, 46, (B, T)),
                     "align_paths": torch.randint(-1, 46, (B, T), dtype=torch.int32),
                     "align_scores": torch.randn(B, T, generator=g), "align_status": torch.zeros(B, dtype=torch.int32)})
    budget = 2 * 2 ** 20                             # far below the workload's outputs: forces a sample
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    bench.dump_outputs(str(tmp_path / "a"), cfg, lengths, batches, outs)
    bench.dump_outputs(str(tmp_path / "b"), cfg, lengths, batches, outs)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(f"{k}.npy" for k in (*bench.DUMP_FRAME_KEYS, "align_status", "utterance_index", "frames"))
    d = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert all(a.dtype == np.float32 for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= budget
    for n in names:
        assert np.array_equal(d[n[:-4]], np.load(tmp_path / "b" / n))
    idx, fr = d["utterance_index"].astype(int), d["frames"].astype(int)
    assert 0 < len(idx) < len(lengths) and list(idx) == sorted(set(idx))
    assert len(d["tvs_pred"]) == fr.sum() and d["phn_fc_logits"].shape == (fr.sum(), 46)
    where = {i: (k, j) for k, b in enumerate(batches) for j, i in enumerate(b.indices)}
    off = 0
    for i, n in zip(idx, fr):
        k, j = where[i]
        assert n == cfg.conv_out_length(lengths[i])
        for name in bench.DUMP_FRAME_KEYS:
            assert np.array_equal(d[name][off: off + n], outs[k][name][j, :n].float().numpy()), (name, i)
        off += n


def test_precision_modes_are_validated_on_the_host():
    """set_precision accepts the three documented modes on every drop-in module's backbone and refuses anything else
    (no kernels run: host logic only)."""
    from aptai_b200.backbone import Wav2Vec2Backbone
    cfg = W2V2Config.large(num_hidden_layers=1, hidden_size=256, num_attention_heads=4, intermediate_size=512,
                           num_conv_pos_embedding_groups=4)
    m = Wav2Vec2Backbone(cfg)
    assert m.precision == "bf16" and m.defers_final_ln()
    for mode in ("fp16", "f32x3", "bf16"):
        assert m.set_precision(mode) is m and m.precision == mode
        assert m.defers_final_ln() == (mode in ("bf16", "fp16"))
    for bad in ("fp8", "float16", ""):
        with pytest.raises(ValueError):
            m.set_precision(bad)
    assert m.precision == "bf16"


@pytest.mark.parametrize("H,heads", [(640, 10), (1280, 20), (128, 2)])
def test_accuracy_mode_rejects_unsupported_hidden_size_on_the_host(H, heads):
    """The accuracy mode's row kernel exists for hidden sizes 256 / 512 / 768 / 1024 only: set_precision('f32x3')
    must refuse any other at the call, naming the supported sizes, and leave the mode unchanged."""
    from aptai_b200.backbone import Wav2Vec2Backbone
    cfg = W2V2Config.large(num_hidden_layers=1, hidden_size=H, num_attention_heads=heads, intermediate_size=2 * H,
                           num_conv_pos_embedding_groups=heads)
    m = Wav2Vec2Backbone(cfg)
    with pytest.raises(ValueError, match=r"256, 512, 768, 1024"):
        m.set_precision("f32x3")
    assert m.precision == "bf16"
    assert m.set_precision("fp16").precision == "fp16"
