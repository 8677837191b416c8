"""Torch-facing wrappers of the C-ABI kernels: argument checks, output allocation (PyTorch's caching allocator
owns every buffer), launch on torch's current CUDA stream.  No arithmetic happens here.
"""
from __future__ import annotations

import ctypes as C
import os
from types import SimpleNamespace
from typing import Optional

import torch

from . import lib as _lib
from .lib import GemmArgs, check

BF16, F16, F32, I32, I64, F64 = torch.bfloat16, torch.float16, torch.float32, torch.int32, torch.int64, torch.float64


def _h16(t: torch.Tensor, name: str) -> int:
    """16-bit operand format of a tensor: 0 = bf16, 1 = fp16."""
    if not t.is_cuda:
        raise RuntimeError(f"aptai_b200: {name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype not in (BF16, F16):
        raise TypeError(f"aptai_b200: {name} must be bfloat16 or float16, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"aptai_b200: {name} must be contiguous")
    return int(t.dtype == F16)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"aptai_b200: {name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"aptai_b200: {name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"aptai_b200: {name} must be contiguous")
    return t


def alloc_rows_bf16(B: int, T: int, C: int, device, slack_rows: int = 2, dtype=None) -> torch.Tensor:
    """bf16 [B,T,C] view of a flat buffer with `slack_rows` zeroed rows behind it: the strided (conv) TMA view of
    the next layer may address one row past the last utterance, and must not leave the allocation."""
    flat = torch.empty((B * T + slack_rows) * C, dtype=dtype or BF16, device=device)
    flat[B * T * C:].zero_()
    return flat[: B * T * C].view(B, T, C)


_gemm_hook = None


def set_gemm_hook(hook) -> None:
    """bench.py's roofline leg: `hook(args)` returns a callable invoked after the launch (CUDA-event bracketing)."""
    global _gemm_hook
    _gemm_hook = hook


def gemm_raw(args: GemmArgs) -> None:
    done = _gemm_hook(args) if _gemm_hook is not None else None
    check(_lib.load().aptai_gemm_bf16(C.byref(args), _stream()), "gemm_bf16")
    if done is not None:
        done()


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act: int = 0,
           residual: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None,
           out_bf16: Optional[torch.Tensor] = None, want_f32: bool = False, want_bf16: bool = True,
           seg_rows: Optional[int] = None, seg_valid_rows: Optional[torch.Tensor] = None,
           block_n: int = 0, cta_pair: int = 0, aux: Optional[torch.Tensor] = None,
           out_pre: Optional[torch.Tensor] = None):
    """out = epilogue(a @ w.T): a bf16 [M,K], w bf16 [N,K] (nn.Linear layout), bias fp32 [N].

    seg_rows / seg_valid_rows: rows are grouped in segments of seg_rows; rows >= seg_valid_rows[s] are written as 0.
    """
    fmt = _h16(a, "a")
    if _h16(w, "w") != fmt:
        raise TypeError("linear: a and w must have the same 16-bit dtype")
    M, K = a.shape
    N, K2 = w.shape
    if K != K2 or K % 64:
        raise ValueError(f"linear: K mismatch or not a multiple of 64 ({K}, {K2})")
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty((M, N), dtype=F32, device=a.device)
    if want_bf16 and out_bf16 is None:
        out_bf16 = torch.empty((M, N), dtype=a.dtype, device=a.device)
    g = GemmArgs()
    g.a = a.data_ptr(); g.a_row_stride = K; g.a_cols = K; g.P = 1; g.taps = 1; g.kb_per_tap = K // 64
    g.a_col_per_nblk = 0
    g.segs = 1; g.rows_per_seg = M; g.a_rows = M; g.a_seg_stride = 0; g.out_seg_stride = 0
    if seg_valid_rows is not None:
        assert seg_rows is not None and M % seg_rows == 0
        _req(seg_valid_rows, I32, "seg_valid_rows")
        g.seg_valid_rows = seg_valid_rows.data_ptr(); g.mask_seg_rows = seg_rows
    else:
        g.seg_valid_rows = None; g.mask_seg_rows = 0
    g.w = w.data_ptr(); g.N = N; g.block_n = block_n
    g.bias = _ptr(_req(bias, F32, "bias")) if bias is not None else None
    g.gamma = None; g.beta = None
    g.residual = _ptr(_req(residual, F32, "residual")) if residual is not None else None
    g.out_f32 = _ptr(out_f32); g.out_bf16 = _ptr(out_bf16); g.ldo = N
    g.act = act; g.ln = 0; g.ln_eps = 0.0; g.cta_pair = cta_pair; g.half_fmt = fmt
    if act == 2:
        if aux is None or aux.shape != (M, N):
            raise ValueError("linear: act=2 (GELU dgrad) needs aux of the output's shape")
        g.aux = _req(aux, BF16, "aux").data_ptr()
    if out_pre is not None:
        if out_pre.shape != (M, N) or out_pre.dtype != a.dtype:
            raise ValueError("linear: out_pre must match the 16-bit output")
        g.out_pre = out_pre.data_ptr()
    gemm_raw(g)
    return out_f32, out_bf16


def split3_bf16(x: torch.Tensor, weight_layout: bool = False, scale: float = 1.0) -> torch.Tensor:
    """fp32 [rows, cols] -> bf16 [rows, 3*cols] = [hi | lo | hi] (activations) or [hi | hi | lo] (weights)."""
    _req(x, F32, "x")
    cols = x.shape[-1]
    rows = x.numel() // cols
    out = torch.empty((rows, 3 * cols), dtype=BF16, device=x.device)
    check(_lib.load().aptai_split3_bf16(x.data_ptr(), rows, cols, cols, int(weight_layout), float(scale),
                                        out.data_ptr(), _stream()), "split3_bf16")
    return out


def linear_f32x3(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """fp32-accurate Linear on the bf16 tensor cores: x = x_hi + x_lo, w = w_hi + w_lo (bf16 pairs) and
    out = [x_hi | x_lo | x_hi] @ [w_hi | w_hi | w_lo]^T (K tripled; the dropped x_lo*w_lo term is ~2^-18 relative).
    For small projections whose input must not be re-quantised (Force_APTAI's frame_lin)."""
    _req(x, F32, "x")
    a = split3_bf16(x, weight_layout=False)                 # one launch each (csrc/accurate.cu), no ATen chain
    ww = split3_bf16(w.detach().float().contiguous(), weight_layout=True)
    out, _ = linear(a, ww, bias, want_f32=True, want_bf16=False)
    return out


def conv_igemm(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], k: int, stride: int, *,
               ln_gamma: Optional[torch.Tensor] = None, ln_beta: Optional[torch.Tensor] = None,
               eps: float = 1e-5, act: int = 1, out: Optional[torch.Tensor] = None, cta_pair: int = 0,
               out_pre: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Strided conv1d as implicit GEMM.  x bf16 [B,T_in,C] channels-last, w bf16 [N, k*C] (tap-major K), out bf16
    [B,T_out,N]; epilogue = (+bias) -> (LayerNorm over N, if gamma) -> GELU.  `out_f32` (fp32 [B,T_out,N]) replaces
    the 16-bit output (accuracy mode)."""
    fmt = _h16(x, "x")
    if _h16(w, "w") != fmt:
        raise TypeError("conv_igemm: x and w must have the same 16-bit dtype")
    B, T_in, Cc = x.shape
    N = w.shape[0]
    assert w.shape[1] == k * Cc and Cc % 64 == 0
    T_out = (T_in - k) // stride + 1
    if out_f32 is not None:
        _req(out_f32, F32, "out_f32")
        assert out_f32.shape == (B, T_out, N)
    elif out is None:
        out = alloc_rows_bf16(B, T_out, N, x.device, dtype=x.dtype)
    g = GemmArgs()
    g.a = x.data_ptr(); g.a_row_stride = Cc; g.a_seg_stride = T_in * Cc; g.a_rows = T_in; g.a_cols = Cc
    g.P = stride; g.taps = k; g.kb_per_tap = Cc // 64; g.a_col_per_nblk = 0
    g.w = w.data_ptr(); g.N = N; g.block_n = 0
    g.segs = B; g.rows_per_seg = T_out
    g.bias = _ptr(bias)
    g.gamma = _ptr(ln_gamma); g.beta = _ptr(ln_beta); g.residual = None
    g.out_f32 = _ptr(out_f32); g.out_bf16 = None if out_f32 is not None else out.data_ptr()
    g.ldo = N; g.out_seg_stride = T_out
    g.seg_valid_rows = None; g.mask_seg_rows = 0; g.act = act; g.ln = 1 if ln_gamma is not None else 0; g.ln_eps = eps
    g.cta_pair = cta_pair; g.half_fmt = fmt
    if out_pre is not None:
        g.out_pre = _req(out_pre, x.dtype, "out_pre").data_ptr()
    gemm_raw(g)
    return out_f32 if out_f32 is not None else out


def posconv(x_pad: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], residual: Optional[torch.Tensor],
            T: int, H: int, groups: int, taps: int, out_f32: torch.Tensor, *, out_pre: Optional[torch.Tensor] = None,
            act: int = 1, row_shift: int = 0, seg_valid_rows: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Grouped positional conv + bias + GELU + residual.  x_pad bf16 [B, T+2*halo, H] (halo = taps//2, zeroed),
    w bf16 [H, taps*64] (per output channel: tap-major, 64-padded group input channels)."""
    fmt = _h16(x_pad, "x_pad")
    if _h16(w, "w") != fmt:
        raise TypeError("posconv: x_pad and w must have the same 16-bit dtype")
    B, Tp, H2 = x_pad.shape
    assert H2 == H and Tp == T + taps
    gw = H // groups
    if (POSCONV_SLAB and gw == 64 and taps == 128 and act == 1 and row_shift == 0 and out_pre is None
            and seg_valid_rows is None and residual is not None and residual.data_ptr() == out_f32.data_ptr()):
        # in-place h += gelu(conv + bias), 64-channel groups: the slab kernel loads every input row once
        _req(out_f32, F32, "out_f32")
        done = _gemm_hook(None) if _gemm_hook is not None else None       # part of the GEMM family (bench roofline leg)
        check(_lib.load().aptai_posconv_slab_fmt(x_pad.data_ptr(), w.data_ptr(), _ptr(bias), out_f32.data_ptr(), B, T, H,
                                                 fmt, _stream()), "posconv_slab")
        if done is not None:
            done()
        return out_f32
    g = GemmArgs()
    # row_shift: first physical row of every segment (the transposed conv of the backward pass reads the halo-padded
    # gradient one row later than the forward reads its input)
    g.a = x_pad.data_ptr() + row_shift * H * 2; g.a_row_stride = H; g.a_seg_stride = Tp * H
    g.a_rows = Tp - row_shift; g.a_cols = H
    g.P = 1; g.taps = taps; g.kb_per_tap = 1; g.a_col_per_nblk = gw
    g.w = w.data_ptr(); g.N = H; g.block_n = gw; g.segs = B; g.rows_per_seg = T
    g.bias = _ptr(bias); g.gamma = None; g.beta = None; g.residual = _ptr(residual)
    g.out_f32 = out_f32.data_ptr(); g.out_bf16 = None; g.ldo = H; g.out_seg_stride = T
    g.seg_valid_rows = None; g.mask_seg_rows = 0; g.act = act; g.ln = 0; g.ln_eps = 0.0; g.cta_pair = 0; g.half_fmt = fmt
    if seg_valid_rows is not None:
        g.seg_valid_rows = _req(seg_valid_rows, I32, "seg_valid_rows").data_ptr(); g.mask_seg_rows = T
    if out_pre is not None:
        g.out_pre = _req(out_pre, x_pad.dtype, "out_pre").data_ptr()
    gemm_raw(g)
    return out_f32


CONV0_TC = int(os.environ.get("APTAI_CONV0_TC", "1"))     # 0: the SIMT conv-0 kernel (A/B runs)


def conv0(wav: torch.Tensor, w: torch.Tensor, bias, gamma, beta, norm: int, eps: float = 1e-5,
          out_dtype=None, return_ws: bool = False):
    _req(wav, F32, "wav"); _req(w, F32, "w")
    B, L = wav.shape
    T0 = (L - 10) // 5 + 1
    out = alloc_rows_bf16(B, T0, 512, wav.device, dtype=out_dtype or BF16)
    L_ = _lib.load()
    ws = torch.empty((L_.aptai_conv0_workspace_bytes(B, norm) // 4,), dtype=F32, device=wav.device)
    flags = int(out.dtype == F16) | (0 if CONV0_TC else 2)
    check(L_.aptai_conv0_norm_gelu(wav.data_ptr(), B, L, w.data_ptr(), _ptr(bias), _ptr(gamma), _ptr(beta),
                                   norm, eps, out.data_ptr(), T0, ws.data_ptr(), flags, _stream()), "conv0_norm_gelu")
    if return_ws:
        return out, ws
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5, *, want_f32=False,
              want_bf16=True, out_f32=None, out_bf16=None, out16_dtype=None):
    if not x.is_cuda:
        raise RuntimeError("aptai_b200: layernorm input must be a CUDA tensor (there is no CPU path)")
    assert x.dtype in (F32, BF16, F16) and x.is_contiguous()
    cols = x.shape[-1]
    rows = x.numel() // cols
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty(x.shape, dtype=F32, device=x.device)
    if want_bf16 and out_bf16 is None:
        out_bf16 = torch.empty(x.shape, dtype=out16_dtype or BF16, device=x.device)
    x_fmt = {F32: 0, BF16: 1, F16: 2}[x.dtype]
    o16 = int(out_bf16 is not None and out_bf16.dtype == F16)
    check(_lib.load().aptai_layernorm(x.data_ptr(), x_fmt, rows, cols, gamma.data_ptr(), beta.data_ptr(), eps,
                                      _ptr(out_f32), _ptr(out_bf16), o16, _stream()), "layernorm")
    return out_f32, out_bf16


def frame_lengths(samples: torch.Tensor, kernels, strides, want_i64: bool = True, want_i32: bool = True):
    """Frames per utterance after the conv feature encoder (HF:1005-1024), one launch.  samples: int64 [B] CUDA.
    Returns (int64 [B] | None, int32 [B] | None)."""
    _req(samples, torch.int64, "samples")
    B = samples.numel()
    nl = len(kernels)
    ks = (C.c_int32 * nl)(*[int(k) for k in kernels])
    ss = (C.c_int32 * nl)(*[int(v) for v in strides])
    o64 = torch.empty((B,), dtype=torch.int64, device=samples.device) if want_i64 else None
    o32 = torch.empty((B,), dtype=I32, device=samples.device) if want_i32 else None
    check(_lib.load().aptai_frame_lengths(samples.data_ptr(), B, C.cast(ks, C.c_void_p), C.cast(ss, C.c_void_p), nl,
                                          _ptr(o64), _ptr(o32), _stream()), "frame_lengths")
    return o64, o32


def cast_pad(x: torch.Tensor, halo: int, dtype=None) -> torch.Tensor:
    _req(x, F32, "x")
    B, T, H = x.shape
    out = torch.empty((B, T + 2 * halo, H), dtype=dtype or BF16, device=x.device)
    check(_lib.load().aptai_cast_pad_h16(x.data_ptr(), B, T, H, halo, out.data_ptr(), _h16(out, "out"), _stream()),
          "cast_pad_h16")
    return out


def posconv_fold(g: torch.Tensor, v: torch.Tensor, cpad: int = 64, out: Optional[torch.Tensor] = None,
                 dtype=None) -> torch.Tensor:
    """weight_norm(dim=2) fold: g [1,1,taps], v [H, cin, taps] -> bf16 (or `dtype` = fp16) [H, taps*cpad]."""
    _req(g, F32, "g"); _req(v, F32, "v")
    H, cin, taps = v.shape
    w = out if out is not None else torch.empty((H, taps * cpad), dtype=dtype or BF16, device=v.device)
    ws = torch.empty((taps,), dtype=F32, device=v.device)
    check(_lib.load().aptai_posconv_fold_fmt(g.data_ptr(), v.data_ptr(), H, cin, taps, cpad, w.data_ptr(), ws.data_ptr(),
                                             _h16(w, "w"), _stream()), "posconv_fold")
    return w


def set_traversal(reverse: bool) -> None:
    """Traversal hint for the next GEMM / LayerNorm / attention-v3 launches of this thread (include/aptai_b200.h)."""
    _lib.load().aptai_set_traversal(1 if reverse else 0)


class Serpentine:
    """Alternates the traversal direction from one kernel of a chain to the next: `s()` before each launch."""

    def __init__(self):
        self.k = 0

    def __call__(self):
        set_traversal(bool(self.k & 1))
        self.k += 1

    def done(self):
        set_traversal(False)


POSCONV_SLAB = int(os.environ.get("APTAI_POSCONV_SLAB", "1"))     # 0: always the generic implicit-GEMM path (A/B runs)


def attention(qkv: torch.Tensor, key_len: Optional[torch.Tensor], B: int, T: int, heads: int,
              out: Optional[torch.Tensor] = None, lse: Optional[torch.Tensor] = None,
              impl: Optional[int] = None, drop_p: float = 0.0, drop_seed: int = 0) -> torch.Tensor:
    """impl None: the kernel by shape (attention_v3.cu's query-tile pairs with P in TMEM when an utterance has more
    than one 128-query tile, else attention_tc.cu's two threads per row); 1 / 3 force one of them (tests)."""
    if impl not in (None, 1, 3):
        raise ValueError(f"attention: impl must be None, 1 or 3, not {impl!r}")
    fmt = _h16(qkv, "qkv")
    H = heads * 64
    assert qkv.numel() == B * T * 3 * H
    if out is None:
        out = torch.empty((B * T, H), dtype=qkv.dtype, device=qkv.device)
    elif out.dtype != qkv.dtype:
        raise TypeError("attention: out must have qkv's dtype")
    if key_len is None:
        key_len = torch.full((B,), T, dtype=I32, device=qkv.device)
    _req(key_len, I32, "key_len")
    if lse is not None:
        _req(lse, F32, "lse")
        assert lse.numel() == B * heads * T
    if drop_p > 0:        # training: dropout on the attention probabilities lives in the query-tile-pair kernel
        _req(qkv, BF16, "qkv")
        check(_lib.load().aptai_attention_fwd_dropout(qkv.data_ptr(), out.data_ptr(), _ptr(lse), key_len.data_ptr(), B,
                                                      T, heads, float(drop_p), int(drop_seed) & 0xFFFFFFFFFFFFFFFF,
                                                      _stream()), "attention_fwd_dropout")
        return out
    which = impl or (3 if T > 128 else 1)
    if which == 3:
        check(_lib.load().aptai_attention_fwd_v3(qkv.data_ptr(), out.data_ptr(), _ptr(lse), key_len.data_ptr(), B, T,
                                                 heads, fmt, _stream()), "attention_fwd_v3")
        return out
    if fmt:               # fp16 operands: the two-threads-per-row kernel for short utterances
        check(_lib.load().aptai_attention_fwd_fmt(qkv.data_ptr(), out.data_ptr(), _ptr(lse), key_len.data_ptr(), B, T,
                                                  heads, fmt, _stream()), "attention_fwd_fmt")
        return out
    if lse is not None:
        check(_lib.load().aptai_attention_fwd_lse(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), key_len.data_ptr(),
                                                  B, T, heads, _stream()), "attention_fwd_lse")
        return out
    check(_lib.load().aptai_attention_fwd(qkv.data_ptr(), out.data_ptr(), key_len.data_ptr(), B, T, heads, _stream()), "attention_fwd")
    return out


ACT_NONE, ACT_TANH, ACT_LEAKY = 0, 1, 2


def heads(h: torch.Tensor, wa, ba, act_a: int, wb, bb, act_b: int, want_argmax: bool = True):
    """h fp32 [rows,H] -> (out_a [rows,na] | None, out_b [rows,nb] | None, argmax_b int64 [rows] | None)."""
    _req(h, F32, "h")
    rows, H = h.shape
    na = 0 if wa is None else wa.shape[0]
    nb = 0 if wb is None else wb.shape[0]
    oa = torch.empty((rows, na), dtype=F32, device=h.device) if na else None
    ob = torch.empty((rows, nb), dtype=F32, device=h.device) if nb else None
    am = torch.empty((rows,), dtype=I64, device=h.device) if (nb and want_argmax) else None
    check(_lib.load().aptai_heads(h.data_ptr(), rows, H, _ptr(wa), _ptr(ba), na, act_a, _ptr(oa), _ptr(wb), _ptr(bb),
                                  nb, act_b, _ptr(ob), _ptr(am), _stream()), "heads")
    return oa, ob, am


PR_HEAD_NARROW = 48        # head-B slots of aptai_heads: recogniser heads up to here run on that kernel
PR_HEAD_MAX_VOCAB = 1024  # wide head (aptai_pr_head_wide, aptai_logits_rows): one row of logits per warp, 32 per lane


def pr_head_wide(h: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], out: Optional[torch.Tensor] = None):
    """Recogniser head h fp32 [rows,H] -> raw logits h @ w.T + b (fp32-accurate split-operand GEMM), 1 <= V <= 1024.
    Returns the [rows, V] view of a pitched buffer (row stride >= 64*ceil(V/64)): `out` fp32 [rows, ld] if given,
    else a new one; pass it to `logits_rows`."""
    _req(h, F32, "h"); _req(w, F32, "w")
    rows, H = h.shape
    V = w.shape[0]
    if w.shape[1] != H:
        raise ValueError(f"pr_head_wide: weight {tuple(w.shape)} does not match h [{rows}, {H}]")
    if b is not None:
        _req(b, F32, "b")
    if out is None:
        out = torch.empty((rows, (V + 63) // 64 * 64), dtype=F32, device=h.device)
    elif out.dtype != F32 or out.dim() != 2 or out.shape[0] != rows or out.stride(1) != 1:
        raise ValueError("pr_head_wide: out must be fp32 [rows, ld] with unit column stride")
    L = _lib.load()
    nbytes = L.aptai_pr_head_wide_workspace_bytes(rows, H, V, 0)
    if nbytes == 0:
        raise ValueError(f"pr_head_wide: V={V}, H={H} unsupported (1 <= V <= {PR_HEAD_MAX_VOCAB}, H % 64 == 0)")
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=h.device)
    check(L.aptai_pr_head_wide(h.data_ptr(), rows, H, w.data_ptr(), _ptr(b), V, out.data_ptr(), out.stride(0),
                               ws.data_ptr(), nbytes, _stream()), "pr_head_wide")
    return out[:, :V]


def logits_rows(x: torch.Tensor, *, want_logits: bool = True, want_argmax: bool = False, want_logp: bool = False,
                want_prob: bool = False):
    """One pass over fp32 rows x [rows, V] (V <= 1024; any row stride, unit column stride) -> (logits contiguous
    [rows, V] | None, first-max argmax int64 [rows] | None, log_softmax | None, softmax | None)."""
    if not x.is_cuda or x.dtype != F32 or x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("logits_rows: x must be a CUDA fp32 [rows, V] tensor with unit column stride")
    rows, V = x.shape
    dev = x.device
    new = lambda on, dt=F32, shape=(rows, V): torch.empty(shape, dtype=dt, device=dev) if on else None
    lg, am, lp, pr = new(want_logits), new(want_argmax, I64, (rows,)), new(want_logp), new(want_prob)
    check(_lib.load().aptai_logits_rows(x.data_ptr(), rows, V, x.stride(0), _ptr(lg), _ptr(am), _ptr(lp), _ptr(pr),
                                        _stream()), "logits_rows")
    return lg, am, lp, pr


def pr_head_wide_bwd(h: torch.Tensor, w: torch.Tensor, d_logits: torch.Tensor, dw: Optional[torch.Tensor],
                     db: Optional[torch.Tensor], want_dh: bool = True) -> Optional[torch.Tensor]:
    """Backward of `pr_head_wide`: returns dh = d_logits @ w (fp32 [rows,H]) and accumulates dw += d_logits.T @ h,
    db += d_logits.sum(0) (either may be None).  d_logits fp32 [rows, V], any row stride, unit column stride."""
    _req(h, F32, "h"); _req(w, F32, "w")
    rows, H = h.shape
    V = w.shape[0]
    if (d_logits.dtype != F32 or not d_logits.is_cuda or tuple(d_logits.shape) != (rows, V)
            or d_logits.stride(1) != 1):
        raise ValueError(f"pr_head_wide_bwd: d_logits must be CUDA fp32 [{rows}, {V}] with unit column stride")
    if dw is not None:
        _req(dw, F32, "dw")
        assert tuple(dw.shape) == (V, H)
    if db is not None:
        _req(db, F32, "db")
        assert db.numel() == V
    dh = torch.empty_like(h) if want_dh else None
    L = _lib.load()
    nbytes = L.aptai_pr_head_wide_workspace_bytes(rows, H, V, 1)
    if nbytes == 0:
        raise ValueError(f"pr_head_wide_bwd: V={V}, H={H} unsupported (1 <= V <= {PR_HEAD_MAX_VOCAB}, H % 64 == 0)")
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=h.device)
    check(L.aptai_pr_head_wide_bwd(h.data_ptr(), rows, H, w.data_ptr(), V, d_logits.data_ptr(), d_logits.stride(0),
                                   _ptr(dh), _ptr(dw), _ptr(db), ws.data_ptr(), nbytes, _stream()), "pr_head_wide_bwd")
    return dh


def tail(h: torch.Tensor, ln_gamma, ln_beta, eps: float, wa, ba, act_a: int, wb, bb, act_b: int, *,
         want_argmax: bool = True, want_logp: bool = False, want_h_norm: bool = False):
    """Fused tail: (final LayerNorm) -> heads A / B -> argmax -> log_softmax.  h fp32 [rows,H].
    Returns (out_a | None, out_b | None, argmax int64 | None, logp | None, h_norm | None)."""
    _req(h, F32, "h")
    rows, H = h.shape
    na = 0 if wa is None else wa.shape[0]
    nb = 0 if wb is None else wb.shape[0]
    dev = h.device
    oa = torch.empty((rows, na), dtype=F32, device=dev) if na else None
    ob = torch.empty((rows, nb), dtype=F32, device=dev) if nb else None
    am = torch.empty((rows,), dtype=I64, device=dev) if (nb and want_argmax) else None
    lp = torch.empty((rows, nb), dtype=F32, device=dev) if (nb and want_logp) else None
    hn = torch.empty((rows, H), dtype=F32, device=dev) if (want_h_norm and ln_gamma is not None) else None
    check(_lib.load().aptai_tail(h.data_ptr(), rows, H, _ptr(ln_gamma), _ptr(ln_beta), float(eps), _ptr(wa), _ptr(ba), na,
                                 act_a, _ptr(oa), _ptr(wb), _ptr(bb), nb, act_b, _ptr(ob), _ptr(am), _ptr(lp), _ptr(hn),
                                 _stream()), "tail")
    return oa, ob, am, lp, hn


def lowpass(x: torch.Tensor, taps: torch.Tensor) -> torch.Tensor:
    _req(x, F32, "x"); _req(taps, F64, "taps")
    B, T, Cc = x.shape
    y = torch.empty_like(x)
    check(_lib.load().aptai_lowpass_fir(x.data_ptr(), B, T, Cc, taps.data_ptr(), taps.numel(), y.data_ptr(),
                                        _stream()), "lowpass_fir")
    return y


def softmax_rows(x: torch.Tensor, log: bool = False) -> torch.Tensor:
    _req(x, F32, "x")
    V = x.shape[-1]
    y = torch.empty_like(x)
    check(_lib.load().aptai_softmax_rows(x.data_ptr(), x.numel() // V, V, int(log), y.data_ptr(), _stream()),
          "softmax_rows")
    return y


def cross_attention(frame, phn_ids, emb, pe, wq, bq, wk, bk, ln_w, ln_b, eps: float = 1e-5, phn_hidden=None):
    """Force_APTAI cross-attention block.  frame fp32 [B,T,128], phn_ids int32 [B,60] -> (att_out [B,T,256],
    energy [B,T,60], att = log_softmax(energy + mask) [B,T,60])."""
    _req(frame, F32, "frame"); _req(phn_ids, I32, "phn_ids")
    B, T, D = frame.shape
    assert D == 128 and phn_ids.shape == (B, 60)
    f = lambda t: t.detach().to(device=frame.device, dtype=F32).contiguous()
    dev = frame.device
    att_out = torch.empty((B, T, 256), dtype=F32, device=dev)
    energy = torch.empty((B, T, 60), dtype=F32, device=dev)
    att = torch.empty((B, T, 60), dtype=F32, device=dev)
    emb = f(emb) if emb is not None else None
    pe = f(pe) if pe is not None else None
    ph = f(phn_hidden) if phn_hidden is not None else None
    check(_lib.load().aptai_cross_attention(frame.data_ptr(), phn_ids.data_ptr(), _ptr(ph), _ptr(emb),
                                            emb.shape[0] if emb is not None else 1,
                                            _ptr(pe), f(wq).data_ptr(), f(bq).data_ptr(), f(wk).data_ptr(),
                                            f(bk).data_ptr(), f(ln_w).data_ptr(), f(ln_b).data_ptr(), eps, B, T,
                                            att_out.data_ptr(), energy.data_ptr(), att.data_ptr(), _stream()),
          "cross_attention")
    return att_out, energy, att


def cross_attention_bwd(frame, phn_ids, phn_hidden, wq, bq, wk, bk, ln_w, eps, d_att_out, d_att, d_ln_w, d_ln_b):
    """Backward of `cross_attention` (phn_hidden form).  Returns (d_q fp32 [B,T,128], d_k fp32 [B,60,128]): gradients
    of the projected queries / keys; d_ln_w / d_ln_b (fp32 [256]) accumulate."""
    _req(frame, F32, "frame"); _req(phn_ids, I32, "phn_ids"); _req(phn_hidden, F32, "phn_hidden")
    _req(d_att_out, F32, "d_att_out"); _req(d_ln_w, F32, "d_ln_w"); _req(d_ln_b, F32, "d_ln_b")
    B, T, D = frame.shape
    assert D == 128 and phn_ids.shape == (B, 60) and d_att_out.shape == (B, T, 256)
    if d_att is not None:
        _req(d_att, F32, "d_att")
        assert d_att.shape == (B, T, 60)
    f = lambda t: t.detach().to(device=frame.device, dtype=F32).contiguous()
    d_q = torch.empty((B, T, 128), dtype=F32, device=frame.device)
    d_k = torch.zeros((B, 60, 128), dtype=F32, device=frame.device)
    check(_lib.load().aptai_cross_attention_bwd(frame.data_ptr(), phn_ids.data_ptr(), phn_hidden.data_ptr(),
                                                f(wq).data_ptr(), f(bq).data_ptr(), f(wk).data_ptr(), f(bk).data_ptr(),
                                                f(ln_w).data_ptr(), eps, B, T, d_att_out.data_ptr(), _ptr(d_att),
                                                d_q.data_ptr(), d_k.data_ptr(), d_ln_w.data_ptr(), d_ln_b.data_ptr(),
                                                _stream()), "cross_attention_bwd")
    return d_q, d_k


def masked_mse_ce(tv_pred, tv_tgt, logits, phn_tgt, return_ws: bool = False):
    _req(tv_pred, F32, "tv_pred"); _req(tv_tgt, F32, "tv_tgt"); _req(logits, F32, "logits"); _req(phn_tgt, I64, "phn")
    rows = phn_tgt.numel()
    ntv = tv_pred.shape[-1]
    V = logits.shape[-1]
    ws = torch.empty((4,), dtype=F64, device=logits.device)
    out = torch.empty((3,), dtype=F32, device=logits.device)
    check(_lib.load().aptai_masked_mse_ce(tv_pred.data_ptr(), tv_tgt.data_ptr(), logits.data_ptr(), phn_tgt.data_ptr(),
                                          rows, ntv, V, ws.data_ptr(), out.data_ptr(), _stream()), "masked_mse_ce")
    if return_ws:
        return out, ws
    return out


CTC_MAX_LABELS = 4095     # labels per utterance of the CTC / Viterbi kernels (2S+1 states over one CTA, 16 per thread)
CTC_FAST_LABELS = 127     # up to here (<= 8 states per lane) a padded label tensor is passed as is


def _trim_targets(targets: torch.Tensor, target_len: torch.Tensor, what: str) -> torch.Tensor:
    """The kernels' label limit applies to the LONGEST transcript, not to the padded width of the label tensor: a
    label tensor wider than CTC_FAST_LABELS is narrowed to max(target_len) (one device->host read, only in that
    case).  The narrowed width selects the kernel: up to 511 labels the state vector lives in one warp's
    registers, beyond that it spans a CTA."""
    if targets.shape[1] <= CTC_FAST_LABELS:
        return targets
    m = max(1, int(target_len.max()))
    if m > CTC_MAX_LABELS:
        raise ValueError(f"{what}: a transcript of {m} labels exceeds the kernels' limit of {CTC_MAX_LABELS} labels per "
                         "utterance (INTEGRATION.md, limits)")
    return targets[:, :m].contiguous()


def logsoftmax_ctc(logits: torch.Tensor, targets: torch.Tensor, input_len: torch.Tensor, target_len: torch.Tensor, *,
                   blank: int = 0, zero_infinity: bool = True, scale: Optional[torch.Tensor] = None,
                   want_log_probs: bool = True, want_grad: bool = False, prepend_blank: bool = False,
                   blank_value: float = 0.0, vocab_len: Optional[torch.Tensor] = None):
    """Returns dict(nll [B], loss_sum [1], log_probs [T,B,Veff] | None, grad [B,T,V] | None).

    Device workspace (`aptai_ctc_workspace_bytes`) is O(B*T*SP): about 2*B*T*SP*4 bytes for alpha and beta, with
    SP = 32 * (4 | 8 | 16 | 32) up to 511 labels and SP = 512 * ceil((2*S+1) / 512) beyond (S = the longest
    transcript), e.g. 2.4 GB for B = 16, T = 8999, S = 1000 and 9.4 GB at S = 4095."""
    _req(logits, F32, "logits"); _req(targets, I32, "targets")
    _req(input_len, I32, "input_len"); _req(target_len, I32, "target_len")
    B, T, V = logits.shape
    targets = _trim_targets(targets, target_len, "logsoftmax_ctc")
    Smax = targets.shape[1]
    Veff = V + int(prepend_blank)
    dev = logits.device
    L = _lib.load()
    nbytes = L.aptai_ctc_workspace_bytes(B, T, Smax)
    if nbytes == 0:
        raise ValueError(f"logsoftmax_ctc: Smax={Smax} unsupported (limit {CTC_MAX_LABELS} labels)")
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    nll = torch.empty((B,), dtype=F32, device=dev)
    loss_sum = torch.empty((1,), dtype=F32, device=dev)
    lp = torch.empty((T, B, Veff), dtype=F32, device=dev) if want_log_probs else None
    grad = torch.empty((B, T, V), dtype=F32, device=dev) if want_grad else None
    if scale is not None:
        _req(scale, F32, "scale")
    if vocab_len is not None:
        _req(vocab_len, I32, "vocab_len")
    check(L.aptai_logsoftmax_ctc_ex(logits.data_ptr(), B, T, V, int(prepend_blank), float(blank_value),
                                    _ptr(vocab_len), targets.data_ptr(), Smax, input_len.data_ptr(),
                                    target_len.data_ptr(), blank, int(zero_infinity), _ptr(lp), nll.data_ptr(),
                                    _ptr(scale), loss_sum.data_ptr(), _ptr(grad), ws.data_ptr(), nbytes, _stream()),
          "logsoftmax_ctc")
    return {"nll": nll, "loss_sum": loss_sum, "log_probs": lp, "grad": grad}


def ctc_viterbi(log_probs: torch.Tensor, targets: torch.Tensor, input_len: torch.Tensor, target_len: torch.Tensor,
                blank: int = 0):
    """log_probs fp32 [B,T,C]; returns (paths int32 [B,T], scores fp32 [B,T], status int32 [B])."""
    _req(log_probs, F32, "log_probs"); _req(targets, I32, "targets")
    _req(input_len, I32, "input_len"); _req(target_len, I32, "target_len")
    B, T, Cc = log_probs.shape
    targets = _trim_targets(targets, target_len, "ctc_viterbi")
    Smax = targets.shape[1]
    dev = log_probs.device
    L = _lib.load()
    nbytes = L.aptai_viterbi_workspace_bytes(B, T, Smax)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    paths = torch.empty((B, T), dtype=I32, device=dev)
    scores = torch.empty((B, T), dtype=F32, device=dev)
    status = torch.empty((B,), dtype=I32, device=dev)
    check(L.aptai_ctc_viterbi_f32(log_probs.data_ptr(), targets.data_ptr(), input_len.data_ptr(), target_len.data_ptr(),
                                  B, T, Cc, Smax, blank, paths.data_ptr(), scores.data_ptr(), status.data_ptr(),
                                  ws.data_ptr(), nbytes, _stream()), "ctc_viterbi")
    return paths, scores, status


def ctc_greedy(logits: torch.Tensor, input_len: Optional[torch.Tensor], blank: int = 0, maxtok: Optional[int] = None):
    _req(logits, F32, "logits")
    B, T, V = logits.shape
    maxtok = maxtok or T
    dev = logits.device
    tokens = torch.zeros((B, maxtok), dtype=I32, device=dev)
    frames = torch.zeros((B, maxtok), dtype=I32, device=dev)
    ntok = torch.empty((B,), dtype=I32, device=dev)
    check(_lib.load().aptai_ctc_greedy(logits.data_ptr(), B, T, V, _ptr(input_len), blank, tokens.data_ptr(),
                                       frames.data_ptr(), ntok.data_ptr(), maxtok, _stream()), "ctc_greedy")
    return tokens, frames, ntok


def ctc_decode_ref(logits: torch.Tensor, input_len: Optional[torch.Tensor], blank: int = 0, sil: int = 1):
    """The reference's decoder output on device (`aptai_ctc_decode_ref`): tokens int32 [B,T+2] (leading / trailing
    `sil`), timesteps int32 [B,T+2] (raw-path index = frame + 1), ntokens int32 [B]."""
    _req(logits, F32, "logits")
    B, T, V = logits.shape
    dev = logits.device
    maxtok = T + 2
    tokens = torch.zeros((B, maxtok), dtype=I32, device=dev)
    steps = torch.zeros((B, maxtok), dtype=I32, device=dev)
    ntok = torch.empty((B,), dtype=I32, device=dev)
    check(_lib.load().aptai_ctc_decode_ref(logits.data_ptr(), B, T, V, _ptr(input_len), blank, sil, tokens.data_ptr(),
                                           steps.data_ptr(), ntok.data_ptr(), maxtok, _stream()), "ctc_decode_ref")
    return tokens, steps, ntok


# ============================================================================================ training step
def attention_dropout_mask(B: int, T: int, heads: int, drop_p: float, drop_seed: int, device) -> torch.Tensor:
    """keep/(1-p) fp32 [B, heads, T, T] of the counter-based attention dropout (what a step with this seed used)."""
    out = torch.empty((B, heads, T, T), dtype=F32, device=device)
    check(_lib.load().aptai_attention_dropout_mask(B, T, heads, float(drop_p), int(drop_seed) & 0xFFFFFFFFFFFFFFFF,
                                                   out.data_ptr(), _stream()), "attention_dropout_mask")
    return out


def attention_bwd(qkv: torch.Tensor, ctx: torch.Tensor, d_ctx: torch.Tensor, lse: torch.Tensor,
                  key_len: torch.Tensor, B: int, T: int, heads: int, q_scale: float, drop_p: float = 0.0,
                  drop_seed: int = 0) -> torch.Tensor:
    """Backward of `attention`: returns dqkv bf16 [B*T, 3H]; the q block is the gradient w.r.t. the UNSCALED q
    (q_scale = head_dim^-0.5 folded in), matching the unscaled q_proj weight used for dgrad/wgrad."""
    _req(qkv, BF16, "qkv"); _req(ctx, BF16, "ctx"); _req(d_ctx, BF16, "d_ctx"); _req(lse, F32, "lse")
    _req(key_len, I32, "key_len")
    H = heads * 64
    M = B * T
    dev = qkv.device
    L = _lib.load()
    dvec = torch.empty((B, heads, T), dtype=F32, device=dev)
    dq32 = torch.empty((M, H), dtype=F32, device=dev)      # cleared by the row-dot kernel (no memset launch)
    check(L.aptai_attention_bwd_dot_zero(d_ctx.data_ptr(), ctx.data_ptr(), B, T, heads, dvec.data_ptr(), dq32.data_ptr(),
                                         _stream()), "attention_bwd_dot")
    dqkv = torch.empty((M, 3 * H), dtype=BF16, device=dev)
    check(L.aptai_attention_bwd_dropout(qkv.data_ptr(), d_ctx.data_ptr(), lse.data_ptr(), dvec.data_ptr(),
                                        key_len.data_ptr(), B, T, heads, dq32.data_ptr(), dqkv.data_ptr(), float(drop_p),
                                        int(drop_seed) & 0xFFFFFFFFFFFFFFFF, _stream()), "attention_bwd")
    check(L.aptai_scale_cast_bf16(dq32.data_ptr(), M, H, float(q_scale), dqkv.data_ptr(), 3 * H, _stream()),
          "scale_cast_bf16")
    return dqkv


def wgrad(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, scale: float = 1.0) -> None:
    """dw[N,K] (fp32, contiguous rows) += scale * dy[M,N]^T @ x[M,K]   (bf16 operands)."""
    _req(dy, BF16, "dy"); _req(x, BF16, "x"); _req(dw, F32, "dw")
    M, N = dy.shape
    M2, K = x.shape
    if M != M2 or tuple(dw.shape) != (N, K):
        raise ValueError(f"wgrad: shapes dy {tuple(dy.shape)}, x {tuple(x.shape)}, dw {tuple(dw.shape)}")
    check(_lib.load().aptai_gemm_wgrad_bf16(dy.data_ptr(), N, x.data_ptr(), K, M, N, K, float(scale), dw.data_ptr(), K,
                                            _stream()), "gemm_wgrad_bf16")


def posconv_wgrad(dy: torch.Tensor, x_pad: torch.Tensor, groups: int, taps: int) -> torch.Tensor:
    """Folded weight gradient [H, taps*64] fp32 of the grouped positional conv."""
    _req(dy, BF16, "dy"); _req(x_pad, BF16, "x_pad")
    B, T, H = dy.shape
    assert x_pad.shape == (B, T + taps, H)
    dwf = torch.zeros((H, taps * 64), dtype=F32, device=dy.device)
    check(_lib.load().aptai_posconv_wgrad_bf16(dy.data_ptr(), x_pad.data_ptr(), B, T, H, groups, taps, dwf.data_ptr(),
                                               _stream()), "posconv_wgrad_bf16")
    return dwf


def posconv_weightnorm_bwd(dwf: torch.Tensor, g: torch.Tensor, v: torch.Tensor, dg: torch.Tensor, dv: torch.Tensor):
    _req(dwf, F32, "dwf"); _req(g, F32, "g"); _req(v, F32, "v"); _req(dg, F32, "dg"); _req(dv, F32, "dv")
    H, cin, taps = v.shape
    ws = torch.empty((2 * taps,), dtype=F64, device=v.device)
    check(_lib.load().aptai_posconv_weightnorm_bwd(dwf.data_ptr(), g.data_ptr(), v.data_ptr(), H, cin, taps, 64,
                                                   dg.data_ptr(), dv.data_ptr(), ws.data_ptr(), _stream()),
          "posconv_weightnorm_bwd")


def colsum(x: torch.Tensor, out: torch.Tensor, scale: float = 1.0) -> None:
    """out[N] (fp32) += scale * x.sum(0); x bf16 or fp32 [M,N]."""
    if x.dtype not in (BF16, F32) or not x.is_cuda or not x.is_contiguous():
        raise TypeError("colsum: x must be a contiguous CUDA bf16/fp32 tensor")
    _req(out, F32, "out")
    M, N = x.shape
    assert out.numel() == N
    check(_lib.load().aptai_colsum(x.data_ptr(), int(x.dtype == BF16), M, N, N, float(scale), out.data_ptr(),
                                   _stream()), "colsum")


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, gamma: torch.Tensor, eps: float, *, dres=None, dgamma=None,
                  dbeta=None, want_f32=True, want_bf16=False, out_f32=None, dcolsum=None):
    """Returns (dx fp32 | None, dx bf16 | None); dx = dres + LN'(dy).  dgamma/dbeta accumulate; `dcolsum` (fp32
    [cols]) accumulates the column sums of dx: the bias gradient of the Linear that wrote this LayerNorm's input."""
    _req(dy, F32, "dy"); _req(x, F32, "x"); _req(gamma, F32, "gamma")
    cols = x.shape[-1]
    rows = x.numel() // cols
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty(x.shape, dtype=F32, device=x.device)
    ob = torch.empty(x.shape, dtype=BF16, device=x.device) if want_bf16 else None
    if dcolsum is not None:
        _req(dcolsum, F32, "dcolsum")
        assert dcolsum.numel() == cols
    check(_lib.load().aptai_layernorm_bwd_colsum(dy.data_ptr(), x.data_ptr(), rows, cols, gamma.data_ptr(), eps,
                                                 _ptr(dres), _ptr(out_f32), _ptr(ob), _ptr(dgamma), _ptr(dbeta),
                                                 _ptr(dcolsum), _stream()), "layernorm_bwd")
    return out_f32, ob


def heads_bwd(h, da, wa, act_a, dwa, dba, db, wb, act_b, dwb, dbb, want_dh: bool = True):
    _req(h, F32, "h")
    rows, H = h.shape
    na = 0 if da is None else da.shape[-1]
    nb = 0 if db is None else db.shape[-1]
    dh = torch.empty_like(h) if want_dh else None
    check(_lib.load().aptai_heads_bwd(h.data_ptr(), rows, H, _ptr(da), na, _ptr(wa), act_a, _ptr(dwa), _ptr(dba),
                                      _ptr(db), nb, _ptr(wb), act_b, _ptr(dwb), _ptr(dbb), _ptr(dh), _stream()),
          "heads_bwd")
    return dh


def masked_mse_ce_bwd(tv_pred, tv_tgt, logits, phn_tgt, ws, grad_scale: Optional[torch.Tensor] = None):
    rows = phn_tgt.numel()
    ntv = tv_pred.shape[-1]
    V = logits.shape[-1]
    d_tv = torch.empty_like(tv_pred)
    d_logits = torch.empty_like(logits)
    check(_lib.load().aptai_masked_mse_ce_bwd(tv_pred.data_ptr(), tv_tgt.data_ptr(), logits.data_ptr(),
                                              phn_tgt.data_ptr(), rows, ntv, V, ws.data_ptr(), _ptr(grad_scale),
                                              d_tv.data_ptr(), d_logits.data_ptr(), _stream()), "masked_mse_ce_bwd")
    return d_tv, d_logits


def scale_cast_bf16(x: torch.Tensor, scale: float = 1.0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _req(x, F32, "x")
    cols = x.shape[-1]
    rows = x.numel() // cols
    if out is None:
        out = torch.empty(x.shape, dtype=BF16, device=x.device)
    check(_lib.load().aptai_scale_cast_bf16(x.data_ptr(), rows, cols, float(scale), out.data_ptr(), cols, _stream()),
          "scale_cast_bf16")
    return out


def gelu_bwd(dy: torch.Tensor, pre: torch.Tensor) -> torch.Tensor:
    """dy fp32 * gelu'(pre bf16) -> fp32."""
    _req(dy, F32, "dy"); _req(pre, BF16, "pre")
    assert dy.numel() == pre.numel()
    out = torch.empty_like(dy)
    check(_lib.load().aptai_gelu_bwd(dy.data_ptr(), pre.data_ptr(), dy.numel(), out.data_ptr(), _stream()), "gelu_bwd")
    return out


def bilstm_256(x: torch.Tensor, lstm: "torch.nn.LSTM", lens: torch.Tensor, save: bool = False):
    """Bidirectional single-layer LSTM(256 -> 256) over padded [B,T,256] fp32 input with per-utterance lengths
    (packed-sequence semantics): input projection of both directions as one fp32-accurate tensor-core GEMM, the
    recurrence in the cluster kernel.  Returns hidden fp32 [B,T,512]; with `save` (training) also the namespace
    `bilstm_256_bwd` needs (gate activations, cell states)."""
    _req(x, F32, "x"); _req(lens, I32, "lens")
    B, T, D = x.shape
    if D != 256 or lstm.hidden_size != 256 or not lstm.bidirectional or lstm.num_layers != 1:
        raise NotImplementedError("aptai_b200 BiLSTM kernel is built for Force_APTAI's LSTM(256, 256, bidirectional)")
    f = lambda t: t.detach().to(device=x.device, dtype=F32).contiguous()
    w_ih = torch.cat([f(lstm.weight_ih_l0), f(lstm.weight_ih_l0_reverse)], dim=0)                  # [2048, 256]
    b = torch.cat([f(lstm.bias_ih_l0) + f(lstm.bias_hh_l0), f(lstm.bias_ih_l0_reverse) + f(lstm.bias_hh_l0_reverse)])
    gates = linear_f32x3(x.view(B * T, D), w_ih, b.contiguous())                                   # [B*T, 2048]
    out = torch.empty((B, T, 512), dtype=F32, device=x.device)
    whf, whr = f(lstm.weight_hh_l0), f(lstm.weight_hh_l0_reverse)
    if save:
        ga = torch.empty((B, T, 2, 1024), dtype=F32, device=x.device)
        cs = torch.empty((B, T, 2, 256), dtype=F32, device=x.device)
        check(_lib.load().aptai_bilstm_256_train(gates.data_ptr(), whf.data_ptr(), whr.data_ptr(), lens.data_ptr(), B, T,
                                                 out.data_ptr(), ga.data_ptr(), cs.data_ptr(), _stream()),
              "bilstm_256_train")
        return out, SimpleNamespace(x=x, lens=lens, gates_act=ga, cells=cs, hidden=out, w_ih=w_ih, whf=whf, whr=whr)
    check(_lib.load().aptai_bilstm_256(gates.data_ptr(), whf.data_ptr(), whr.data_ptr(), lens.data_ptr(), B, T,
                                       out.data_ptr(), _stream()), "bilstm_256")
    return out


def bilstm_256_bwd(sv, d_hidden: torch.Tensor, grads: dict) -> torch.Tensor:
    """Backward of `bilstm_256(..., save=True)`: d_hidden fp32 [B,T,512] -> dx fp32 [B,T,256]; accumulates into the
    fp32 gradient tensors grads['weight_ih_l0'], ['weight_hh_l0'], ['bias_ih_l0'], ['bias_hh_l0'] and their
    '_reverse' twins.  Recurrence: the cluster BPTT kernel; weight / input gradients: tensor-core GEMMs on its output."""
    _req(d_hidden, F32, "d_hidden")
    B, T, _ = d_hidden.shape
    M = B * T
    dev = d_hidden.device
    dG = torch.zeros((2, M, 1024), dtype=F32, device=dev)
    check(_lib.load().aptai_bilstm_256_bwd(d_hidden.data_ptr(), sv.gates_act.data_ptr(), sv.cells.data_ptr(),
                                           sv.whf.data_ptr(), sv.whr.data_ptr(), sv.lens.data_ptr(), B, T, dG.data_ptr(),
                                           _stream()), "bilstm_256_bwd")
    dGb = scale_cast_bf16(dG)
    xb = scale_cast_bf16(sv.x.view(M, 256))
    # h_{t-1} as seen by each direction: the forward chain reads the previous frame, the reverse chain the next one
    hprev = torch.zeros((2, B, T, 256), dtype=F32, device=dev)
    hprev[0, :, 1:] = sv.hidden[:, :-1, :256]
    hprev[1, :, :-1] = sv.hidden[:, 1:, 256:]
    hpb = scale_cast_bf16(hprev.view(2, M, 256))
    dx = None
    for d, sfx in enumerate(("", "_reverse")):
        wgrad(dGb[d], xb, grads["weight_ih_l0" + sfx])
        wgrad(dGb[d], hpb[d], grads["weight_hh_l0" + sfx])
        db = torch.zeros((1024,), dtype=F32, device=dev)       # b_ih and b_hh enter the gates as a sum: same gradient
        colsum(dG[d], db)
        grads["bias_ih_l0" + sfx].add_(db)
        grads["bias_hh_l0" + sfx].add_(db)
        wt = sv.w_ih[d * 1024:(d + 1) * 1024].t().contiguous().to(BF16)            # [256, 1024]
        dx, _ = linear(dGb[d], wt, None, residual=dx, want_f32=True, want_bf16=False)
    return dx.view(B, T, 256)


def prepare_weights(table: torch.Tensor, n_entries: int, total_tiles: int, half_fmt: int = 0) -> None:
    """Launch the multi-tensor weight preparation over a device table of `aptai_prep_entry` rows; `half_fmt` 1: the
    16-bit destinations are IEEE fp16 instead of bf16."""
    check(_lib.load().aptai_prepare_weights_fmt(table.data_ptr(), n_entries, total_tiles, half_fmt, _stream()),
          "prepare_weights")


def dropout(x: torch.Tensor, p: float, seed: int, *, residual: Optional[torch.Tensor] = None, want_f32: bool = False,
            want_bf16: bool = False, out_f32: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None):
    """Counter-based inverted dropout: residual + keep(seed, i) * x / (1 - p).  x fp32 or bf16; returns (fp32 | None,
    bf16 | None).  In place when an output is x itself.  The backward of a site = the same call on the gradient."""
    if not x.is_cuda or x.dtype not in (F32, BF16) or not x.is_contiguous():
        raise TypeError("dropout: x must be a contiguous CUDA fp32/bf16 tensor")
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty(x.shape, dtype=F32, device=x.device)
    if want_bf16 and out_bf16 is None:
        out_bf16 = torch.empty(x.shape, dtype=BF16, device=x.device)
    if residual is not None:
        _req(residual, F32, "residual")
    check(_lib.load().aptai_dropout(x.data_ptr(), int(x.dtype == BF16), _ptr(residual), x.numel(), float(p),
                                    int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(out_f32), _ptr(out_bf16), _stream()), "dropout")
    return out_f32, out_bf16


# ---- conv feature encoder, training path ('layer' norm variant) -------------------------------------------------
def ln_gelu_fwd(z: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """y = GELU(LayerNorm_512(z)); z bf16 [B,T,512] -> y bf16 [B,T,512] (with the slack rows the strided TMA view needs)."""
    _req(z, BF16, "z")
    B, T, Cc = z.shape
    assert Cc == 512
    y = alloc_rows_bf16(B, T, Cc, z.device)
    check(_lib.load().aptai_ln_gelu_fwd_512(z.data_ptr(), B * T, gamma.data_ptr(), beta.data_ptr(), eps, y.data_ptr(),
                                            _stream()), "ln_gelu_fwd")
    return y


def ln_gelu_bwd(dy: torch.Tensor, rows_per_seg: int, seg_pitch: int, segs: int, gamma, beta, eps, dgamma, dbeta, *,
                z: Optional[torch.Tensor] = None, wav: Optional[torch.Tensor] = None,
                w0t: Optional[torch.Tensor] = None, bias0: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dz bf16 [segs*rows_per_seg, 512] = LN'(dy * GELU'(LN(z))); dy fp32, logical row r of segment s at physical row
    s*seg_pitch + r.  z given, or recomputed from the waveform for conv layer 0 (wav fp32 [B,L], w0t fp32 [10,512])."""
    _req(dy, F32, "dy")
    rows = segs * rows_per_seg
    dz = torch.empty((rows, 512), dtype=BF16, device=dy.device)
    check(_lib.load().aptai_ln_gelu_bwd_512(dy.data_ptr(), rows_per_seg, seg_pitch, _ptr(z), _ptr(wav),
                                            wav.shape[1] if wav is not None else 0, _ptr(w0t), _ptr(bias0), rows,
                                            gamma.data_ptr(), beta.data_ptr(), eps, dz.data_ptr(), dgamma.data_ptr(),
                                            dbeta.data_ptr(), _stream()), "ln_gelu_bwd")
    return dz


def conv_wgrad(dz: torch.Tensor, x: torch.Tensor, k: int, stride: int) -> torch.Tensor:
    """Tap-major weight gradient fp32 [C, k*C] of a strided conv layer: dz bf16 [B,T_out,C], x bf16 [B,T_in,C]."""
    _req(dz, BF16, "dz"); _req(x, BF16, "x")
    B, T_out, Cc = dz.shape
    T_in = x.shape[1]
    dwf = torch.zeros((Cc, k * Cc), dtype=F32, device=dz.device)
    check(_lib.load().aptai_conv_wgrad_bf16(dz.data_ptr(), x.data_ptr(), B, T_out, T_in, Cc, k, stride, dwf.data_ptr(),
                                            _stream()), "conv_wgrad_bf16")
    return dwf


def conv_dgrad(dz: torch.Tensor, wt_taps, k: int, stride: int, T_in: int):
    """Input gradient of a strided conv layer as one GEMM per tap with strided output rows:
    dx[b, t*stride + tap, c] (+)= sum_o dz[b,t,o] * W[o,c,tap].  dz bf16 [B,T_out,C]; wt_taps[tap] bf16 [C(c), C(o)].
    Returns (dx fp32 [B, T_pad, C], T_pad): T_pad = T_in rounded up to the stride."""
    _req(dz, BF16, "dz")
    B, T_out, Cc = dz.shape
    T_pad = (T_in + stride - 1) // stride * stride
    dx = torch.zeros((B, T_pad, Cc), dtype=F32, device=dz.device)
    for tap in range(k):
        w = _req(wt_taps[tap], BF16, "wt")
        g = GemmArgs()
        g.a = dz.data_ptr(); g.a_row_stride = Cc; g.a_seg_stride = T_out * Cc; g.a_rows = T_out; g.a_cols = Cc
        g.P = 1; g.taps = 1; g.kb_per_tap = Cc // 64; g.a_col_per_nblk = 0
        g.w = w.data_ptr(); g.N = Cc; g.block_n = 0; g.segs = B; g.rows_per_seg = T_out
        g.bias = None; g.gamma = None; g.beta = None
        out = dx.data_ptr() + tap * Cc * 4
        g.residual = out if tap >= stride else None          # taps congruent mod stride hit the same rows: accumulate
        g.out_f32 = out; g.out_bf16 = None; g.ldo = stride * Cc; g.out_seg_stride = T_pad // stride
        g.seg_valid_rows = None; g.mask_seg_rows = 0; g.act = 0; g.ln = 0; g.ln_eps = 0.0; g.cta_pair = 0; g.half_fmt = 0
        gemm_raw(g)
    return dx, T_pad


def conv0_im2col(wav: torch.Tensor, T0: int) -> torch.Tensor:
    _req(wav, F32, "wav")
    B, L = wav.shape
    X = torch.empty((B * T0, 64), dtype=BF16, device=wav.device)
    check(_lib.load().aptai_conv0_im2col_bf16(wav.data_ptr(), B, L, T0, X.data_ptr(), _stream()), "conv0_im2col")
    return X


def gelu_bwd_rows(dy: torch.Tensor, rows_per_seg: int, seg_pitch: int, segs: int, z: torch.Tensor) -> torch.Tensor:
    """dz bf16 [segs*rows_per_seg, 512] = dy * GELU'(z) ('group' variant conv layers 1..6)."""
    _req(dy, F32, "dy"); _req(z, BF16, "z")
    rows = segs * rows_per_seg
    dz = torch.empty((rows, 512), dtype=BF16, device=dy.device)
    check(_lib.load().aptai_gelu_bwd_rows_512(dy.data_ptr(), rows_per_seg, seg_pitch, z.data_ptr(), rows, dz.data_ptr(),
                                              _stream()), "gelu_bwd_rows")
    return dz


def conv0_groupnorm_saved(ws: torch.Tensor, B: int):
    """What the backward of conv layer 0 + GroupNorm needs from `conv0(..., norm=2, return_ws=True)`'s workspace:
    (affine fp32 [B, 512, 2] = {scale, shift}, norm_stats fp32 [B, 512, 2] = {mean - bias, rstd})."""
    o = B * 65 * 2                                    # behind the fp64 waveform moments
    return ws[o: o + B * 1024].view(B, 512, 2), ws[o + B * 1024: o + B * 2048].view(B, 512, 2)


def conv0_groupnorm_bwd(dy: torch.Tensor, seg_pitch: int, wav: torch.Tensor, T0: int, w0: torch.Tensor,
                        affine: torch.Tensor, norm_stats: torch.Tensor):
    """Backward of conv layer 0 + GroupNorm-over-time + GELU (affine, norm_stats: `conv0_groupnorm_saved`).  Returns
    (dz0 bf16 [B*T0, 512], sums fp32 [B, 512, 2] = per-utterance {dbeta, dgamma} contributions)."""
    _req(dy, F32, "dy"); _req(wav, F32, "wav"); _req(affine, F32, "affine"); _req(norm_stats, F32, "norm_stats")
    B, L = wav.shape
    if affine.numel() != B * 1024 or norm_stats.numel() != B * 1024:
        raise ValueError("conv0_groupnorm_bwd: affine and norm_stats must be [B, 512, 2]")
    sums = torch.empty((B, 512, 2), dtype=F32, device=wav.device)
    dz = torch.empty((B * T0, 512), dtype=BF16, device=wav.device)
    check(_lib.load().aptai_conv0_groupnorm_bwd(dy.data_ptr(), seg_pitch, wav.data_ptr(), B, L, T0, w0.data_ptr(),
                                                affine.data_ptr(), norm_stats.data_ptr(), sums.data_ptr(),
                                                dz.data_ptr(), _stream()), "conv0_groupnorm_bwd")
    return dz, sums
