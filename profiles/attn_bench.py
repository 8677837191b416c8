"""Attention micro-benchmark: the by-shape default against the two-threads-per-row kernel (impl 1) and the
query-tile-pair kernel with P in TMEM (impl 3) (CUDA events, L2 flushed)."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from aptai_b200 import ops
dev = torch.device("cuda:0")
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
def timeit(fn, iters=8):
    for _ in range(3): fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]
for B, T in [(120, 399), (48, 999), (80, 600), (189, 250)]:
    heads, H = 16, 1024
    qkv = (torch.randn((B * T, 3 * H), device=dev) * 0.5).bfloat16()
    kl = torch.full((B,), T, dtype=torch.int32, device=dev)
    out = torch.empty((B * T, H), dtype=torch.bfloat16, device=dev)
    fl = 4.0 * B * heads * T * T * 64
    r = timeit(lambda: ops.attention(qkv, kl, B, T, heads, out=out))
    a = timeit(lambda: ops.attention(qkv, kl, B, T, heads, out=out, impl=1))
    d = timeit(lambda: ops.attention(qkv, kl, B, T, heads, out=out, impl=3))
    print(f"B={B:4d} T={T:4d}: default {r:7.3f} ms {fl / r / 1e9:7.1f} TFLOP/s | impl 1 {a:7.3f} ms "
          f"{fl / a / 1e9:7.1f} TFLOP/s | impl 3 (P in TMEM) {d:7.3f} ms {fl / d / 1e9:7.1f} TFLOP/s", flush=True)
