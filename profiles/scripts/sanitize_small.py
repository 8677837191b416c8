"""Small invocation of every kernel family of the inference path (2-layer 1024-wide 'layer' encoder, 3 ragged utterances
of <= 3 s: conv-0, the implicit-GEMM conv tiles, pos-conv slab, LayerNorm, QKV / out-proj / FFN GEMMs, both attention
kernels, tail, low-pass, log-softmax, CTC-Viterbi) in the three precision modes, for compute-sanitizer:
  compute-sanitizer --tool memcheck  python profiles/scripts/sanitize_small.py
  compute-sanitizer --tool racecheck python profiles/scripts/sanitize_small.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from aptai_b200 import APTAI
from aptai_b200.backbone import register_in_memory_checkpoint
from aptai_b200.config import W2V2Config
from aptai_b200.synth import backbone_state_dict, waveforms

dev = torch.device("cuda:0")
cfg = W2V2Config.large(num_hidden_layers=2, hidden_dropout=0.0, activation_dropout=0.0, attention_dropout=0.0,
                       final_dropout=0.0, layerdrop=0.0, apply_spec_augment=False)
name = register_in_memory_checkpoint("mem://san", backbone_state_dict(cfg, 0))
vocab = {"(blank)": 0, "(...)": 1, **{f"p{i}": i for i in range(2, 46)}}
m = APTAI(dev, vocab, name, cfg, None, phn_drop=0.0, tv_drop=0.0).to(dev).eval()
m.use_cuda_graphs = False
lens = [48000, 30000, 16000]                     # T = 149 / 93 / 49: the query-tile-pair kernel; 1 s alone: T <= 128
wav = waveforms(3, 48000, lens, seed=5).to(dev)
tg = torch.tensor([[3, 7, 7, 12, 5], [9, 2, 30, 0, 0], [4, 4, 0, 0, 0]], dtype=torch.int32, device=dev)
tl = torch.tensor([5, 3, 2], dtype=torch.int32, device=dev)
for mode in ("bf16", "fp16", "f32x3"):
    m.set_precision(mode)
    r = m.predict(wav, torch.tensor(lens, device=dev), phn_targets=tg, phn_target_lens=tl)
    r1 = m.predict(wav[2:3, :16000].contiguous(), torch.tensor([16000], device=dev))
    torch.cuda.synchronize()
    print(mode, "ok", float(r["tvs_pred"].abs().max()), r["align_status"].tolist(), r1["phn_fc_logits"].shape, flush=True)
