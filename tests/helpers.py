"""Shared builders for the parity tests: deterministic configs/weights/inputs that match tests/golden/make_golden.py."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from aptai_b200.config import W2V2Config  # noqa: E402
from oracle import weights as W  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "golden_v1.npz")
VOCAB = {"(blank)": 0, "(...)": 1, **{f"p{i}": i for i in range(2, 46)}}
TV = ("LA", "LP", "JA", "TTCL", "TTCD", "TMCL", "TMCD", "TBCL", "TBCD")
NO_REG = dict(hidden_dropout=0.0, activation_dropout=0.0, attention_dropout=0.0, feat_proj_dropout=0.0,
              final_dropout=0.0, layerdrop=0.0, apply_spec_augment=False)


def golden():
    return np.load(GOLDEN)


_G2 = {}


def golden2():
    """Config-size fixtures from the reference's own classes (tests/golden/make_golden_v2.py)."""
    if "g" not in _G2:
        _G2["g"] = dict(np.load(os.path.join(ROOT, "tests", "golden", "golden_v2.npz")))
    return _G2["g"]


R4_FRAMES = [399, 352, 299, 221]


def r4_targets(T=399):
    """Phoneme / TV targets of golden_v2's ragged batch R4: int64 [4,T] and fp32 [4,T,9] (-100 beyond each length)."""
    rng = np.random.Generator(np.random.PCG64(31))
    phn = np.zeros((4, T), dtype=np.int64)
    tvt = np.full((4, T, 9), -100.0, dtype=np.float32)
    for b, n in enumerate(R4_FRAMES):
        phn[b, :n] = rng.integers(1, 46, size=n)
        tvt[b, :n] = rng.standard_normal((n, 9), dtype=np.float32)
    return phn, tvt


def f8_tv_targets():
    """TV targets of golden_v2's Force_APTAI case F8: fp32 [1,399,9]."""
    return np.random.Generator(np.random.PCG64(51)).standard_normal((1, 399, 9), dtype=np.float32)


def cfg_large(**kw):
    return W2V2Config.large(**{**NO_REG, **kw})


def cfg_base(**kw):
    return W2V2Config.base(**{**NO_REG, **kw})


_SD_CACHE = {}


def backbone_sd(cfg, seed):
    key = (cfg.hidden_size, cfg.num_hidden_layers, cfg.feat_extract_norm, seed)
    if key not in _SD_CACHE:
        _SD_CACHE[key] = W.backbone_state_dict(cfg, seed)
    return _SD_CACHE[key]


def pearson(a, b):
    a = a - a.mean(0, keepdims=True)
    b = b - b.mean(0, keepdims=True)
    return (a * b).sum(0) / np.sqrt((a * a).sum(0) * (b * b).sum(0))


def save_backbone_dir(cfg, seed, path):
    """Write <path>/pytorch_model.bin so that `from_pretrained(path, config=cfg)` of the drop-in loads it."""
    os.makedirs(path, exist_ok=True)
    torch.save(backbone_sd(cfg, seed), os.path.join(path, "pytorch_model.bin"))
    return path


def force_tail_state(state_dict):
    """Deterministic weights for the Force_APTAI tail (everything except the frozen recogniser, the PE buffer and
    the low-pass taps), keyed by parameter NAME so that module definition order does not matter."""
    import zlib
    out = {}
    for k, v in state_dict.items():
        if k.startswith("w2v2_pr.") or k in ("pe_phn.pe", "tv_lowpass.lowpass.weight"):
            continue
        g = np.random.Generator(np.random.PCG64(zlib.crc32(k.encode())))
        if k.endswith("layer_norm.weight"):
            t = torch.ones(tuple(v.shape))
        elif k.endswith("bias") or "bias_" in k:
            t = torch.from_numpy(g.standard_normal(tuple(v.shape), dtype=np.float32) * np.float32(0.02))
        else:
            t = torch.from_numpy(g.standard_normal(tuple(v.shape), dtype=np.float32)
                                 * np.float32(1.0 / np.sqrt(v.shape[-1])))
        out[k] = t
    out["phn_emb_layer.weight"][0] = 0
    return out
