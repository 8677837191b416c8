"""Debug driver: attention v3 at the bench shapes, one launch at a time, checked against impl 1."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from aptai_b200 import ops
dev = torch.device("cuda:0")
for B, T, lens in [(8, 399, None), (120, 399, None), (120, 399, "ragged"), (48, 999, None), (189, 250, None)]:
    heads, H = 16, 1024
    torch.manual_seed(0)
    qkv = (torch.randn((B * T, 3 * H), device=dev) * 0.5).bfloat16()
    if lens == "ragged":
        kl = torch.tensor([T - (7 * b) % 32 for b in range(B)], dtype=torch.int32, device=dev)
    else:
        kl = torch.full((B,), T, dtype=torch.int32, device=dev)
    ref = ops.attention(qkv, kl, B, T, heads, impl=1)
    out = ops.attention(qkv, kl, B, T, heads, impl=3)
    torch.cuda.synchronize()
    print(B, T, lens, "max diff vs impl 1", float((out.float() - ref.float()).abs().max()), flush=True)
