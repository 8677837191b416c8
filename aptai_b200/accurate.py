"""Accuracy mode (`precision="f32x3"`) of the acoustic encoder.

Same kernels, same wiring as `Wav2Vec2Backbone.encode`, but no activation is ever rounded to 16 bits: the residual
stream, LayerNorm / GELU / softmax run in fp32 and every contraction is the tcgen05 GEMM on split operands
(A' = [x_hi | x_lo | x_hi], W' = [w_hi | w_hi | w_lo]: three bf16 products per multiply, ~2^-17 relative); attention
is the fp32 kernel.  About 3-4x the tensor work of the default mode — it exists to show that the north-star
tolerances which an untrained head's near-tie frames deny to any 16-bit-operand path (phoneme argmax >= 99.9 %,
SURVEY.md Appendix D) are met by the same arithmetic once the operand rounding is removed, and as a reference
point for the default mode's error (bench.py reports both).

Reference lines replaced: HF:254-323, 409-434 (feature encoder / projection), HF:329-379 (positional conv),
HF:500-655 (attention, feed-forward, both layer wirings), HF:668-803 (encoders).
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional

import torch

from . import lib as _lib
from . import ops
from .lib import check

BF16, F32, I32 = torch.bfloat16, torch.float32, torch.int32


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def split3(x: torch.Tensor, weight_layout: bool = False, scale: float = 1.0, slack_rows: int = 0) -> torch.Tensor:
    """fp32 [rows, cols] -> bf16 [rows, 3*cols] = [hi | lo | hi] (activations) or [hi | hi | lo] (weights)."""
    ops._req(x, F32, "x")
    cols = x.shape[-1]
    rows = x.numel() // cols
    flat = torch.empty(((rows + slack_rows) * 3 * cols,), dtype=BF16, device=x.device)
    if slack_rows:
        flat[rows * 3 * cols:].zero_()
    check(_lib.load().aptai_split3_bf16(x.data_ptr(), rows, cols, cols, int(weight_layout), float(scale),
                                        flat.data_ptr(), _stream()), "split3_bf16")
    return flat[: rows * 3 * cols].view(rows, 3 * cols)


def rowop(x: torch.Tensor, gamma=None, beta=None, eps: float = 1e-5, *, gelu: bool = False, want_f32: bool = False,
          want_split: bool = True, slack_rows: int = 0):
    """(LayerNorm) -> (GELU) per row of fp32 [rows, cols]; returns (fp32 | None, split bf16 [rows, 3*cols] | None)."""
    ops._req(x, F32, "x")
    cols = x.shape[-1]
    rows = x.numel() // cols
    o32 = torch.empty((rows, cols), dtype=F32, device=x.device) if want_f32 else None
    o3 = None
    if want_split:
        flat = torch.empty(((rows + slack_rows) * 3 * cols,), dtype=BF16, device=x.device)
        if slack_rows:
            flat[rows * 3 * cols:].zero_()
        o3 = flat[: rows * 3 * cols].view(rows, 3 * cols)
    check(_lib.load().aptai_rowop_split3(x.data_ptr(), rows, cols, ops._ptr(gamma), ops._ptr(beta), float(eps),
                                         int(gamma is not None), int(gelu), ops._ptr(o32), ops._ptr(o3), _stream()),
          "rowop_split3")
    return o32, o3


def conv0(wav, w, bias, gamma, beta, norm: int, eps: float = 1e-5) -> torch.Tensor:
    ops._req(wav, F32, "wav")
    B, L = wav.shape
    T0 = (L - 10) // 5 + 1
    flat = torch.empty(((B * T0 + 2) * 1536,), dtype=BF16, device=wav.device)
    flat[B * T0 * 1536:].zero_()
    ws = torch.empty((max(256, B * (65 * 2 + 1024) + 16),), dtype=F32, device=wav.device) if norm == 2 else None
    check(_lib.load().aptai_conv0_accurate(wav.data_ptr(), B, L, w.data_ptr(), ops._ptr(bias), ops._ptr(gamma),
                                           ops._ptr(beta), norm, float(eps), flat.data_ptr(), T0, ops._ptr(ws),
                                           _stream()), "conv0_accurate")
    return flat[: B * T0 * 1536].view(B, T0, 1536)


def attention_f32(qkv: torch.Tensor, key_len: torch.Tensor, B: int, T: int, heads: int) -> torch.Tensor:
    ops._req(qkv, F32, "qkv"); ops._req(key_len, I32, "key_len")
    H = heads * 64
    assert qkv.numel() == B * T * 3 * H
    ctx = torch.empty((B * T, H), dtype=F32, device=qkv.device)
    check(_lib.load().aptai_attention_fwd_f32(qkv.data_ptr(), ctx.data_ptr(), key_len.data_ptr(), B, T, heads,
                                              _stream()), "attention_fwd_f32")
    return ctx


def gelu_add(x: torch.Tensor, res: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    ops._req(x, F32, "x"); ops._req(res, F32, "res")
    out = out if out is not None else torch.empty_like(res)
    check(_lib.load().aptai_gelu_add_f32(x.data_ptr(), res.data_ptr(), x.numel(), out.data_ptr(), _stream()),
          "gelu_add_f32")
    return out


def cast_pad_split(x: torch.Tensor, halo: int):
    ops._req(x, F32, "x")
    B, T, H = x.shape
    hi = torch.empty((B, T + 2 * halo, H), dtype=BF16, device=x.device)
    lo = torch.empty_like(hi)
    check(_lib.load().aptai_cast_pad_split(x.data_ptr(), B, T, H, halo, hi.data_ptr(), lo.data_ptr(), _stream()),
          "cast_pad_split")
    return hi, lo


def posconv_fold_split(g: torch.Tensor, v: torch.Tensor, cpad: int = 64):
    ops._req(g, F32, "g"); ops._req(v, F32, "v")
    H, cin, taps = v.shape
    hi = torch.empty((H, taps * cpad), dtype=BF16, device=v.device)
    lo = torch.empty_like(hi)
    ws = torch.empty((taps,), dtype=F32, device=v.device)
    check(_lib.load().aptai_posconv_fold_split(g.data_ptr(), v.data_ptr(), H, cin, taps, cpad, hi.data_ptr(),
                                               lo.data_ptr(), ws.data_ptr(), _stream()), "posconv_fold_split")
    return hi, lo


def pos_conv_add(h: torch.Tensor, w_hi: torch.Tensor, w_lo: torch.Tensor, bias: torch.Tensor, groups: int,
                 taps: int) -> torch.Tensor:
    """h fp32 [B,T,H] += gelu(grouped positional conv(h) + bias), in place (HF:329-379, 689-690 | 763-764), as three
    bf16 products: h_hi.w_hi + h_lo.w_hi + h_hi.w_lo (w_hi / w_lo from posconv_fold_split)."""
    B, T, H = h.shape
    hp_hi, hp_lo = cast_pad_split(h, taps // 2)
    acc = torch.empty_like(h)
    ops.posconv(hp_hi, w_hi, bias, None, T, H, groups, taps, acc, act=0)
    ops.posconv(hp_lo, w_hi, None, acc, T, H, groups, taps, acc, act=0)
    ops.posconv(hp_hi, w_lo, None, acc, T, H, groups, taps, acc, act=0)
    return gelu_add(acc, h, out=h)


def linear3(x3: torch.Tensor, w3: torch.Tensor, bias, **kw):
    """fp32-accurate Linear: x3 = split3(x), w3 = split3(W, weight_layout=True); fp32 output."""
    return ops.linear(x3, w3, bias, want_f32=kw.pop("want_f32", True), want_bf16=False, **kw)[0]


class PlanF32x3:
    """Split-operand copies of the parameters, derived once per parameter version (like backbone._Plan)."""

    def __init__(self, m):
        cfg = m.cfg
        dev = m.masked_spec_embed.device
        f = lambda t: t.detach().to(device=dev, dtype=F32).contiguous()
        w3 = lambda t, scale=1.0: split3(f(t), weight_layout=True, scale=scale)
        cl = m.feature_extractor.conv_layers
        self.conv0_w = f(cl[0].conv.weight.reshape(cfg.conv_dim[0], cfg.conv_kernel[0]))
        self.conv_b = [f(l.conv.bias) if l.conv.bias is not None else None for l in cl]
        self.conv_ln_w = [f(l.layer_norm.weight) if hasattr(l, "layer_norm") else None for l in cl]
        self.conv_ln_b = [f(l.layer_norm.bias) if hasattr(l, "layer_norm") else None for l in cl]
        self.conv_w = [None]
        for l in cl[1:]:
            cout, cin, k = l.conv.weight.shape
            wt = f(l.conv.weight.permute(0, 2, 1)).reshape(cout * k, cin)       # rows (out, tap): [hi | hi | lo] per tap
            self.conv_w.append(split3(wt, weight_layout=True).view(cout, k * 3 * cin))
        fp = m.feature_projection
        self.fp_ln_w, self.fp_ln_b = f(fp.layer_norm.weight), f(fp.layer_norm.bias)
        self.fp_w, self.fp_b = w3(fp.projection.weight), f(fp.projection.bias)
        pc = m.encoder.pos_conv_embed.conv
        self.pos_b = f(pc.bias)
        self.pos_w_hi, self.pos_w_lo = posconv_fold_split(f(pc.parametrizations.weight.original0),
                                                          f(pc.parametrizations.weight.original1))
        self.enc_ln_w, self.enc_ln_b = f(m.encoder.layer_norm.weight), f(m.encoder.layer_norm.bias)
        scale = float(cfg.head_dim) ** -0.5
        self.layers = []
        for l in m.encoder.layers:
            a, ff = l.attention, l.feed_forward
            qkv_w = torch.cat([f(a.q_proj.weight) * scale, f(a.k_proj.weight), f(a.v_proj.weight)], 0).contiguous()
            qkv_b = torch.cat([f(a.q_proj.bias) * scale, f(a.k_proj.bias), f(a.v_proj.bias)], 0).contiguous()
            self.layers.append(SimpleNamespace(
                qkv_w=split3(qkv_w, weight_layout=True), qkv_b=qkv_b, o_w=w3(a.out_proj.weight), o_b=f(a.out_proj.bias),
                ff1_w=w3(ff.intermediate_dense.weight), ff1_b=f(ff.intermediate_dense.bias),
                ff2_w=w3(ff.output_dense.weight), ff2_b=f(ff.output_dense.bias),
                ln1_w=f(l.layer_norm.weight), ln1_b=f(l.layer_norm.bias),
                ln2_w=f(l.final_layer_norm.weight), ln2_b=f(l.final_layer_norm.bias)))


def plan(m) -> PlanF32x3:
    params = list(m.parameters())
    key = (tuple(p.data_ptr() for p in params), tuple(p._version for p in params))
    cached = getattr(m, "_plan_f32x3", None)
    if cached is None or cached[0] != key:
        with torch.no_grad():
            cached = (key, PlanF32x3(m))
        object.__setattr__(m, "_plan_f32x3", cached)
    return cached[1]


@torch.no_grad()
def encode(m, wav: torch.Tensor, frame_lens: torch.Tensor, *, collect_hidden: bool = False,
           want_features: bool = False):
    """Accuracy-mode twin of `Wav2Vec2Backbone.encode` (same arguments and return values; features are fp32)."""
    cfg, P = m.cfg, plan(m)
    B, L = wav.shape
    layer_norm = cfg.feat_extract_norm == "layer"
    y3 = conv0(wav, P.conv0_w, P.conv_b[0], P.conv_ln_w[0], P.conv_ln_b[0], 1 if layer_norm else 2)
    feats = None
    n_conv = len(cfg.conv_kernel)
    for i in range(1, n_conv):
        k, s = cfg.conv_kernel[i], cfg.conv_stride[i]
        T_out = (y3.shape[1] - k) // s + 1
        z = torch.empty((B, T_out, cfg.conv_dim[i]), dtype=F32, device=wav.device)
        ops.conv_igemm(y3, P.conv_w[i], P.conv_b[i], k, s, act=0, out_f32=z)
        last = i == n_conv - 1
        g = (P.conv_ln_w[i], P.conv_ln_b[i]) if layer_norm else (None, None)
        o32, o3 = rowop(z.view(B * T_out, -1), g[0], g[1], 1e-5, gelu=True, want_f32=last, want_split=not last,
                        slack_rows=2)
        if last:
            feats = o32.view(B, T_out, -1)
        else:
            y3 = o3.view(B, T_out, -1)
    T = feats.shape[1]
    M, H = B * T, cfg.hidden_size
    eps, heads = cfg.layer_norm_eps, cfg.num_attention_heads
    _, xn3 = rowop(feats.view(M, -1), P.fp_ln_w, P.fp_ln_b, eps)
    h = linear3(xn3, P.fp_w, P.fp_b, seg_rows=T, seg_valid_rows=frame_lens)
    pos_conv_add(h.view(B, T, H), P.pos_w_hi, P.pos_w_lo, P.pos_b, cfg.num_conv_pos_embedding_groups,
                 cfg.num_conv_pos_embeddings)
    hidden = [] if collect_hidden else None

    def attn_ffn(x3, lw, res_attn):
        qkv = linear3(x3, lw.qkv_w, lw.qkv_b)
        ctx = attention_f32(qkv, frame_lens, B, T, heads)
        return linear3(split3(ctx), lw.o_w, lw.o_b, residual=res_attn)

    def ffn(x3, lw, res):
        u = linear3(x3, lw.ff1_w, lw.ff1_b, act=1)
        return linear3(split3(u), lw.ff2_w, lw.ff2_b, residual=res)

    if cfg.do_stable_layer_norm:
        for lw in P.layers:
            if collect_hidden:
                hidden.append(h.view(B, T, H))
            h = attn_ffn(rowop(h, lw.ln1_w, lw.ln1_b, eps)[1], lw, h)
            h = ffn(rowop(h, lw.ln2_w, lw.ln2_b, eps)[1], lw, h)
        last_h, _ = rowop(h, P.enc_ln_w, P.enc_ln_b, eps, want_f32=True, want_split=False)
    else:
        h, x3 = rowop(h, P.enc_ln_w, P.enc_ln_b, eps, want_f32=True)
        for lw in P.layers:
            if collect_hidden:
                hidden.append(h.view(B, T, H))
            t = attn_ffn(x3, lw, h)
            h, x3 = rowop(t, lw.ln1_w, lw.ln1_b, eps, want_f32=True)
            t = ffn(x3, lw, h)
            h, x3 = rowop(t, lw.ln2_w, lw.ln2_b, eps, want_f32=True)
        last_h = h
    last_h = last_h.view(B, T, H)
    if collect_hidden:
        hidden.append(last_h)
    return last_h, (tuple(hidden) if collect_hidden else None), (feats if want_features else None)
