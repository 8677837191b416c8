"""wav2vec2-style acoustic encoder on the aptai_b200 kernels.

`Wav2Vec2Backbone` is the drop-in for the `transformers.Wav2Vec2Model` instance the reference wraps
(models/aptai.py:33-40, models/w2v2_pr.py:28-33): same constructor source (`from_pretrained(id, config=...,
cache_dir=...)`), same `state_dict` keys/shapes (SURVEY.md Appendix A.5, incl. the weight-norm parametrisation
`encoder.pos_conv_embed.conv.parametrizations.weight.original0/1`), same call
`forward(input_values, attention_mask=lengths[:, None], output_hidden_states=True, return_dict=True)`.
The torch submodules below are parameter containers only — they are never called; the arithmetic runs in the
sm_100a kernels through `aptai_b200.ops`:

  conv0+norm+GELU (HBM-bound SIMT)  ->  conv1..6 implicit GEMM, LN/GELU epilogue (tcgen05)
  -> LayerNorm -> projection GEMM (bias, padded frames zeroed) -> grouped pos-conv GEMM (+GELU +residual)
  -> N x [LN -> QKV GEMM -> masked flash attention -> out-proj GEMM(+residual) -> LN -> FFN GEMM(+GELU)
          -> FFN GEMM(+residual)]  (pre-LN 'stable' or post-LN wiring)  -> final LN

Precision policy (SURVEY.md Appendix D): bf16 GEMM/attention operands, fp32 accumulation, fp32 residual stream,
LayerNorm statistics and softmax in fp32.
Training: `encode_train` runs the same kernels and keeps every activation the backward needs (no recomputation —
the reference's gradient checkpointing exists to fit small GPUs, 180 GB of HBM3e holds a 32 x 8 s batch outright);
`backward` runs the hand-written backward kernels (dgrad on transposed weights, MN-major tcgen05 wgrad, tcgen05
attention backward, LayerNorm/GELU backward) into a flat gradient buffer, including the stochastic regularisers
of the HF training forward (counter-based dropout at every site, LayerDrop, SpecAugment along time and features)
and the backward of the conv feature encoder when it is not frozen (the reference freezes it for APTAI,
models/aptai.py:39-40, and trains it for the recogniser, train/train_phoneme_recognizer.py:170).
`precision="f32x3"` (see `encode_f32x3`) is the accuracy mode: every contraction on bf16 hi/lo operand pairs
(three tensor-core products per GEMM, ~2^-17 relative), fp32 everywhere else.
"""
from __future__ import annotations

import os
from types import SimpleNamespace
from typing import Optional

import torch
import torch.nn as nn

from . import ops
from .config import W2V2Config

BF16, F16, F32, I32 = torch.bfloat16, torch.float16, torch.float32, torch.int32
F32X3_HIDDEN_SIZES = (256, 512, 768, 1024)      # the widths aptai_rowop_split3 is instantiated for


# ----------------------------------------------------------------------------------------- parameter containers
class _ConvLayer(nn.Module):
    def __init__(self, cin, cout, k, s, bias, with_ln):
        super().__init__()
        self.conv = nn.Conv1d(cin, cout, k, stride=s, bias=bias)
        if with_ln:
            self.layer_norm = nn.LayerNorm(cout)      # GroupNorm(512,512) has the same parameter names/shapes


class _FeatureExtractor(nn.Module):
    def __init__(self, cfg: W2V2Config):
        super().__init__()
        layers = []
        cin = 1
        for i, (c, k, s) in enumerate(zip(cfg.conv_dim, cfg.conv_kernel, cfg.conv_stride)):
            layers.append(_ConvLayer(cin, c, k, s, cfg.conv_bias, cfg.feat_extract_norm == "layer" or i == 0))
            cin = c
        self.conv_layers = nn.ModuleList(layers)


class _FeatureProjection(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.layer_norm = nn.LayerNorm(cfg.conv_dim[-1], eps=cfg.layer_norm_eps)
        self.projection = nn.Linear(cfg.conv_dim[-1], cfg.hidden_size)


class _PosConv(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        conv = nn.Conv1d(cfg.hidden_size, cfg.hidden_size, cfg.num_conv_pos_embeddings,
                         padding=cfg.num_conv_pos_embeddings // 2, groups=cfg.num_conv_pos_embedding_groups)
        self.conv = nn.utils.parametrizations.weight_norm(conv, name="weight", dim=2)


class _Attention(nn.Module):
    def __init__(self, H):
        super().__init__()
        self.k_proj = nn.Linear(H, H)
        self.v_proj = nn.Linear(H, H)
        self.q_proj = nn.Linear(H, H)
        self.out_proj = nn.Linear(H, H)


class _FeedForward(nn.Module):
    def __init__(self, H, F):
        super().__init__()
        self.intermediate_dense = nn.Linear(H, F)
        self.output_dense = nn.Linear(F, H)


class _EncoderLayer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.attention = _Attention(cfg.hidden_size)
        self.layer_norm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)
        self.feed_forward = _FeedForward(cfg.hidden_size, cfg.intermediate_size)
        self.final_layer_norm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)


class _Encoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.pos_conv_embed = _PosConv(cfg)
        self.layer_norm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)
        self.layers = nn.ModuleList([_EncoderLayer(cfg) for _ in range(cfg.num_hidden_layers)])


# ----------------------------------------------------------------------------------------- kernel-side weights
class _WeightTable:
    """Device table for `aptai_prepare_weights`: one launch turns the fp32 master weights into the kernels' operand
    copies (bf16 [N][K], transposed bf16 [K][N], fused / scaled fp32 biases)."""

    def __init__(self, dev):
        self.dev, self.rows, self.keep, self.tiles = dev, [], [], 0
        self.table = None

    def add(self, src, dst=None, dst_off=0, dst_ld=0, dst_t=None, dst_t_off=0, dst_t_ld=0, dst_f32=None, f32_off=0,
            scale=1.0, scale_t=1.0):
        src = src.detach()
        if src.dtype != F32 or not src.is_contiguous() or src.device != self.dev:
            raise TypeError("aptai_b200: master weights must be contiguous fp32 tensors on the model's CUDA device")
        rows, cols = (1, src.numel()) if src.dim() == 1 else (src.shape[0], src.shape[1])
        from .lib import PrepEntry
        e = PrepEntry()
        e.src = src.data_ptr()
        e.dst = dst.data_ptr() + 2 * dst_off if dst is not None else None
        e.dst_t = dst_t.data_ptr() + 2 * dst_t_off if dst_t is not None else None
        e.dst_f32 = dst_f32.data_ptr() + 4 * f32_off if dst_f32 is not None else None
        e.rows, e.cols, e.dst_ld, e.dst_t_ld = rows, cols, dst_ld or cols, dst_t_ld or rows
        e.scale, e.scale_t = scale, scale_t
        e.tiles_x = (cols + 63) // 64                     # 64 x 64 tiles (aptai_prepare_weights)
        e.tile0 = self.tiles
        self.tiles += e.tiles_x * ((rows + 63) // 64)
        self.rows.append(e)
        self.keep.append((src, dst, dst_t, dst_f32))

    def run(self, half_fmt: int = 0):
        import ctypes as C
        from .lib import PrepEntry
        if self.table is None:
            arr = (PrepEntry * len(self.rows))(*self.rows)
            raw = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone()
            self.table = raw.to(self.dev)
        ops.prepare_weights(self.table, len(self.rows), self.tiles, half_fmt)


class _Plan:
    """Kernel-ready copies of the parameters (bf16 GEMM operands, fused QKV with the softmax scale folded into q,
    tap-major conv weights, folded weight-norm) in PERSISTENT buffers.  `refresh()` re-derives them from the fp32
    master weights with one multi-tensor launch (after load_state_dict / every optimizer step); the table is rebuilt
    only when a parameter's storage moves.  With `train=True` it also keeps what the backward needs: transposed bf16
    weights for the dgrad GEMMs (dX = dY @ W is the forward kernel on W^T; the q block unscaled), a bf16 projection
    weight, and the flipped / in-out-swapped folded pos-conv weight (transposed conv = the forward kernel on it)."""

    def __init__(self, m: "Wav2Vec2Backbone", train: bool = False, half: int = 0):
        cfg = m.cfg
        dev = m.masked_spec_embed.device
        if train and half:
            raise ValueError("aptai_b200: the training plan keeps bf16 operands (fp16 gradients would underflow)")
        self.train = train
        self.half = half          # 1: the transformer's operand copies are IEEE fp16 (precision="fp16", inference)
        f = lambda t: t.detach().to(device=dev, dtype=F32).contiguous()    # fp32 params: a view, tracks updates
        self._f = f
        self._conv_key = None
        fp = m.feature_projection
        self.fp_ln_w, self.fp_ln_b = f(fp.layer_norm.weight), f(fp.layer_norm.bias)
        self.fp_b = f(fp.projection.bias)
        pc = m.encoder.pos_conv_embed.conv
        self.pos_b = f(pc.bias)
        self.enc_ln_w, self.enc_ln_b = f(m.encoder.layer_norm.weight), f(m.encoder.layer_norm.bias)
        H, Fi = cfg.hidden_size, cfg.intermediate_size
        scale = float(cfg.head_dim) ** -0.5     # folded into q (0.125 for head_dim 64: exact in bf16)
        tb = _WeightTable(dev)
        e16 = lambda *shape: torch.empty(shape, dtype=F16 if half else BF16, device=dev)
        if train:
            self.fp_w_bf16, self.fp_wt = e16(H, cfg.conv_dim[-1]), e16(cfg.conv_dim[-1], H)
            tb.add(fp.projection.weight, dst=self.fp_w_bf16, dst_t=self.fp_wt)
        self.layers = []
        for l in m.encoder.layers:
            a, ff = l.attention, l.feed_forward
            ns = SimpleNamespace(
                qkv_w=e16(3 * H, H), qkv_b=torch.empty((3 * H,), dtype=F32, device=dev), o_w=e16(H, H),
                ff1_w=e16(Fi, H), ff2_w=e16(H, Fi), o_b=f(a.out_proj.bias), ff1_b=f(ff.intermediate_dense.bias),
                ff2_b=f(ff.output_dense.bias), ln1_w=f(l.layer_norm.weight), ln1_b=f(l.layer_norm.bias),
                ln2_w=f(l.final_layer_norm.weight), ln2_b=f(l.final_layer_norm.bias))
            if train:
                ns.qkv_wt, ns.o_wt, ns.ff1_wt, ns.ff2_wt = e16(H, 3 * H), e16(H, H), e16(H, Fi), e16(Fi, H)
            for blk, (proj, sc) in enumerate(((a.q_proj, scale), (a.k_proj, 1.0), (a.v_proj, 1.0))):
                tb.add(proj.weight, dst=ns.qkv_w, dst_off=blk * H * H, dst_ld=H, scale=sc,
                       dst_t=ns.qkv_wt if train else None, dst_t_off=blk * H, dst_t_ld=3 * H, scale_t=1.0)
                tb.add(proj.bias, dst_f32=ns.qkv_b, f32_off=blk * H, scale=sc)
            tb.add(a.out_proj.weight, dst=ns.o_w, dst_t=ns.o_wt if train else None)
            tb.add(ff.intermediate_dense.weight, dst=ns.ff1_w, dst_t=ns.ff1_wt if train else None)
            tb.add(ff.output_dense.weight, dst=ns.ff2_w, dst_t=ns.ff2_wt if train else None)
            self.layers.append(ns)
        self._table = tb
        self.refresh(m)

    def refresh(self, m: "Wav2Vec2Backbone") -> None:
        cfg = m.cfg
        dev = m.masked_spec_embed.device
        f = self._f
        cl = m.feature_extractor.conv_layers
        ck = tuple((p.data_ptr(), p._version) for p in m.feature_extractor.parameters()) + tuple(
            (p.data_ptr(), p._version) for p in m.feature_projection.projection.parameters())
        if ck != self._conv_key:      # frozen in training: re-derived only after load_state_dict / .to()
            h = lambda t: t.detach().to(device=dev, dtype=F16).contiguous()   # conv stack / projection operands
            self.conv0_w = f(cl[0].conv.weight.reshape(cfg.conv_dim[0], cfg.conv_kernel[0]))
            self.conv_b = [f(l.conv.bias) if l.conv.bias is not None else None for l in cl]
            self.conv_ln_w = [f(l.layer_norm.weight) if hasattr(l, "layer_norm") else None for l in cl]
            self.conv_ln_b = [f(l.layer_norm.bias) if hasattr(l, "layer_norm") else None for l in cl]
            # conv i >= 1: [out][in][k] -> [out][k][in]  (K index = tap*C_in + c)
            self.conv_w = [None] + [h(l.conv.weight.permute(0, 2, 1).reshape(l.conv.weight.shape[0], -1))
                                    for l in cl[1:]]
            self.fp_w = h(m.feature_projection.projection.weight)
            if self.train and any(p.requires_grad for p in m.feature_extractor.parameters()):
                # unfrozen conv encoder: bf16 forward operands (the gradients flow in bf16, fp16 would underflow),
                # per-tap transposed weights for the input-gradient GEMMs, conv-0's weight as [10][512]
                bq = lambda t: t.detach().to(device=dev, dtype=BF16).contiguous()
                self.conv_w_bf16 = [None] + [bq(l.conv.weight.permute(0, 2, 1).reshape(l.conv.weight.shape[0], -1))
                                             for l in cl[1:]]
                self.conv_wt = [None] + [[bq(l.conv.weight[:, :, tap].t()) for tap in range(l.conv.weight.shape[2])]
                                         for l in cl[1:]]
                self.conv0_wt = f(cl[0].conv.weight.reshape(cfg.conv_dim[0], cfg.conv_kernel[0]).t())
            self._conv_key = ck
            self.generation = getattr(self, "generation", 0) + 1      # buffers re-allocated: captured graphs are stale
        self._table.run(self.half)
        pc = m.encoder.pos_conv_embed.conv
        g = f(pc.parametrizations.weight.original0)
        v = f(pc.parametrizations.weight.original1)
        self.pos_w = ops.posconv_fold(g, v, cpad=64, out=getattr(self, "pos_w", None),
                                      dtype=F16 if self.half else BF16)
        if self.train:
            Hh, gw, taps = v.shape
            groups = Hh // gw
            vt = v.view(groups, gw, gw, taps).permute(0, 2, 1, 3).flip(-1).reshape(Hh, gw, taps).contiguous()
            self.pos_wt = ops.posconv_fold(g.flip(-1).contiguous(), vt, cpad=64, out=getattr(self, "pos_wt", None))
            self.pos_g, self.pos_v = g, v


_IN_MEMORY = {}


def register_in_memory_checkpoint(name: str, state_dict) -> str:
    """Offline stand-in for a hub id: `from_pretrained(name, ...)` loads this state dict (tests, benchmarks)."""
    _IN_MEMORY[name] = state_dict
    return name


class Wav2Vec2Backbone(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config                       # whatever the caller passed (HF config object or ours)
        self.cfg = W2V2Config.from_any(config)
        self.cfg.validate_for_kernels()
        cfg = self.cfg
        self.masked_spec_embed = nn.Parameter(torch.empty(cfg.hidden_size).uniform_())
        self.feature_extractor = _FeatureExtractor(cfg)
        self.feature_projection = _FeatureProjection(cfg)
        self.encoder = _Encoder(cfg)
        self.precision = "bf16"                    # "bf16" (default) | "f32x3" (accuracy mode, aptai_b200/accurate.py)
        self._plan: Optional[_Plan] = None
        self._plan_key = None
        self._plan_ptrs = None
        self._plan_h: Optional[_Plan] = None       # the fp16-operand inference plan lives beside the bf16 one
        self._plan_h_key = None
        self._plan_h_ptrs = None
        self._feature_encoder_frozen = False

    # ---- reference-facing helpers --------------------------------------------------------------------------
    @classmethod
    def from_pretrained(cls, model_id, config=None, cache_dir=None, **_):
        """Local `save_pretrained` directory (model.safetensors / pytorch_model.bin).  There is no network in
        this environment, so hub ids are refused with a clear error instead of a silent random init."""
        if config is None:
            raise ValueError("Wav2Vec2Backbone.from_pretrained needs config=")
        m = cls(config)
        path = str(model_id)
        if path in _IN_MEMORY:
            m.load_state_dict(_IN_MEMORY[path], strict=True)
        elif os.path.isdir(path):
            st = os.path.join(path, "model.safetensors")
            pt = os.path.join(path, "pytorch_model.bin")
            if os.path.exists(st):
                from safetensors.torch import load_file
                sd = load_file(st)
            elif os.path.exists(pt):
                sd = torch.load(pt, map_location="cpu")
            else:
                raise FileNotFoundError(f"no model.safetensors / pytorch_model.bin under {path}")
            sd = {k[len("wav2vec2."):] if k.startswith("wav2vec2.") else k: v for k, v in sd.items()}
            missing, unexpected = m.load_state_dict(sd, strict=False)
            missing = [k for k in missing if k != "masked_spec_embed"]
            if missing:
                raise RuntimeError(f"checkpoint {path} is missing {missing[:5]}...")
        else:
            raise FileNotFoundError(
                f"'{model_id}' is not a local directory; hub downloads are unavailable (no network). "
                "Pass a directory written by save_pretrained().")
        return m

    def set_precision(self, precision: str):
        """'bf16': 16-bit tensor-core operands (default, the measured hot path).  'fp16': the same kernels on IEEE
        fp16 operands (weights, activations, attention probabilities; fp32 accumulation, residual stream and
        statistics as before) — same speed, 7x smaller logit / trajectory error (three more mantissa bits), for
        checkpoints whose activations stay inside fp16's range (inference only; training keeps bf16).
        'f32x3': accuracy mode — every contraction on bf16 hi/lo operand pairs, fp32 elsewhere (inference only)."""
        if precision not in ("bf16", "fp16", "f32x3"):
            raise ValueError(f"aptai_b200: unknown precision {precision!r} ('bf16', 'fp16' or 'f32x3')")
        if precision == "f32x3" and self.cfg.hidden_size not in F32X3_HIDDEN_SIZES:
            # the accuracy mode's LayerNorm kernel (aptai_rowop_split3) holds a row in one warp's registers;
            # head_dim == 64 is already enforced for every mode by cfg.validate_for_kernels()
            raise ValueError(f"aptai_b200: precision 'f32x3' supports hidden sizes {F32X3_HIDDEN_SIZES}, "
                             f"not {self.cfg.hidden_size}")
        self.precision = precision       # the fp16 operand copies (0.6 GB for 24x1024) stay cached across mode switches
        return self

    def gradient_checkpointing_enable(self, *a, **k):    # models/aptai.py:38 — no autograd graph to checkpoint here
        return None

    def freeze_feature_encoder(self):                    # models/aptai.py:39-40
        for p in self.feature_extractor.parameters():
            p.requires_grad = False
        self._feature_encoder_frozen = True

    def _get_feat_extract_output_lengths(self, input_lengths):
        """HF:1005-1024 on tensors or ints.  CUDA tensors go through one kernel launch (csrc/elementwise.cu
        `frame_lengths_kernel`) instead of three ATen launches per conv layer."""
        n = input_lengths
        if torch.is_tensor(n) and n.is_cuda and not n.is_floating_point():
            shape = n.shape
            o64, _ = ops.frame_lengths(n.reshape(-1).to(torch.int64).contiguous(), self.cfg.conv_kernel,
                                       self.cfg.conv_stride, want_i32=False)
            return o64.view(shape).to(n.dtype)
        for k, s in zip(self.cfg.conv_kernel, self.cfg.conv_stride):
            n = torch.div(n - k, s, rounding_mode="floor") + 1 if torch.is_tensor(n) else (n - k) // s + 1
        return n

    def defers_final_ln(self) -> bool:
        """True when `encode(final_ln=False)` really leaves the last LayerNorm to the caller (pre-LN encoder, default
        precision)."""
        return bool(self.cfg.do_stable_layer_norm) and self.precision in ("bf16", "fp16")

    def final_ln_params(self):
        """(gamma, beta, eps) of the encoder's last LayerNorm as the kernels take them (fp32, contiguous)."""
        P = self.plan()
        return P.enc_ln_w, P.enc_ln_b, self.cfg.layer_norm_eps

    def frame_lengths_i32(self, input_lengths: torch.Tensor) -> torch.Tensor:
        """int32 [B] frame counts (the form every kernel takes) of sample counts on this module's device."""
        dev = next(self.parameters()).device
        lens = input_lengths.reshape(-1).to(device=dev, dtype=torch.int64).contiguous()
        return ops.frame_lengths(lens, self.cfg.conv_kernel, self.cfg.conv_stride, want_i64=False)[1]

    # ---- plan ------------------------------------------------------------------------------------------------
    def plan(self, train: bool = False) -> _Plan:
        params = list(self.parameters())
        ptrs = tuple(p.data_ptr() for p in params)
        vers = tuple(p._version for p in params)
        if self.precision == "fp16" and not train:
            P = self._plan_h
            with torch.no_grad():
                if P is None or ptrs != self._plan_h_ptrs:
                    self._plan_h = _Plan(self, half=1)
                elif vers != self._plan_h_key:
                    P.refresh(self)
            self._plan_h_ptrs, self._plan_h_key = ptrs, vers
            return self._plan_h
        P = self._plan
        with torch.no_grad():
            if P is None or ptrs != self._plan_ptrs or (train and not P.train):
                self._plan = _Plan(self, train=train or (P is not None and P.train))
            elif vers != self._plan_key:
                P.refresh(self)
        self._plan_ptrs, self._plan_key = ptrs, vers
        return self._plan

    def train_plan(self) -> _Plan:
        return self.plan(train=True)

    def fused_grad_groups(self, prefix: str = ""):
        """Parameter-name groups that must be adjacent in the flat gradient buffer (fused QKV wgrad)."""
        groups = []
        for i in range(len(self.encoder.layers)):
            base = f"{prefix}encoder.layers.{i}.attention."
            groups.append([base + "q_proj.weight", base + "k_proj.weight", base + "v_proj.weight"])
            groups.append([base + "q_proj.bias", base + "k_proj.bias", base + "v_proj.bias"])
        return groups

    def check_trainable(self):
        """Every regulariser of the HF training forward is built; kept as the hook where an unbuilt one is refused."""

    # Stochastic regularisers of the training path.  Dropout is counter-based (csrc/dropout.cu): a site's mask is a
    # function of (seed, element index), the seed of (training step, layer, site), so the backward regenerates it.
    SITE_ATTN, SITE_ACT, SITE_FFN, SITE_PROJ, SITE_ENC, SITE_HEAD_A, SITE_HEAD_B, SITE_ATTN_P = range(8)

    def drop_seed(self, step: int, layer: int, site: int) -> int:
        base = getattr(self, "_drop_base", None)
        if base is None:
            base = int(torch.initial_seed()) & 0xFFFFFFFF          # torch.manual_seed() controls the masks
            object.__setattr__(self, "_drop_base", base)
        return ((base * 1000003 + step) << 12) | ((layer + 1) << 4) | site

    # ---- training: forward that keeps activations, and the backward --------------------------------------------
    @torch.no_grad()
    def encode_train(self, wav: torch.Tensor, frame_lens: torch.Tensor, regularise: bool = True,
                     collect_hidden: bool = False):
        """Same arithmetic as `encode` (the feature projection runs on bf16 instead of fp16 operands so that its
        wgrad shares the bf16 kernel), plus the training-mode regularisers: feat_proj / hidden / activation dropout
        (HF:434,546,570,603-607,647-653,694,766), LayerDrop (HF:701-706,773-778: `torch.rand([])` per layer, the same
        host RNG stream HF consumes) and SpecAugment (HF:1280-1324).  Returns (last_hidden fp32 [B,T,H], saved).
        `regularise=False`: a gradient-carrying forward of a module in eval mode (get_embeddings_grad);
        `collect_hidden`: saved.hidden = the N+1 hidden states (HF `output_hidden_states`)."""
        self.check_trainable()
        cfg = self.cfg
        if not regularise:
            import copy
            cfg = copy.copy(cfg)
            cfg.hidden_dropout = cfg.activation_dropout = cfg.attention_dropout = cfg.feat_proj_dropout = 0.0
            cfg.layerdrop = 0.0
            cfg.apply_spec_augment = False
        P = TP = self.train_plan()
        B, L = wav.shape
        norm = 1 if cfg.feat_extract_norm == "layer" else 2
        train_conv = any(p.requires_grad for p in self.feature_extractor.parameters())
        conv_sv = None
        if train_conv:
            # unfrozen conv encoder: bf16 operands, conv outputs z_i kept un-normalised, LayerNorm + GELU as a separate
            # streaming kernel (the backward recomputes statistics and activations from z_i; conv 0 from the waveform)
            y, ws0 = ops.conv0(wav, P.conv0_w, P.conv_b[0], P.conv_ln_w[0], P.conv_ln_b[0], norm, out_dtype=BF16,
                               return_ws=True)
            conv_sv = SimpleNamespace(wav=wav, ys=[y], zs=[None], gn_saved=None)
            if norm == 2:        # GroupNorm: per-(utterance, channel) scale / shift and statistics of the forward kernel
                conv_sv.gn_saved = ops.conv0_groupnorm_saved(ws0, B)
            for i in range(1, len(cfg.conv_kernel)):
                if norm == 1:
                    z = ops.conv_igemm(y, P.conv_w_bf16[i], P.conv_b[i], cfg.conv_kernel[i], cfg.conv_stride[i], act=0)
                    y = ops.ln_gelu_fwd(z, P.conv_ln_w[i], P.conv_ln_b[i])
                else:            # 'group' variant: layers 1..6 are conv -> GELU; keep the pre-activation
                    T_o = (y.shape[1] - cfg.conv_kernel[i]) // cfg.conv_stride[i] + 1
                    z = torch.empty((B, T_o, y.shape[2]), dtype=BF16, device=wav.device)
                    y = ops.conv_igemm(y, P.conv_w_bf16[i], P.conv_b[i], cfg.conv_kernel[i], cfg.conv_stride[i], act=1,
                                       out_pre=z)
                conv_sv.zs.append(z)
                conv_sv.ys.append(y)
        else:
            y = ops.conv0(wav, P.conv0_w, P.conv_b[0], P.conv_ln_w[0], P.conv_ln_b[0], norm, out_dtype=F16)
            for i in range(1, len(cfg.conv_kernel)):
                y = _conv_layer(y, P, i, cfg)
        T = y.shape[1]
        M, H = B * T, cfg.hidden_size
        eps, heads = cfg.layer_norm_eps, cfg.num_attention_heads
        taps, groups = cfg.num_conv_pos_embeddings, cfg.num_conv_pos_embedding_groups
        step = getattr(self, "_drop_step", 0) + 1
        object.__setattr__(self, "_drop_step", step)
        p_h, p_a, p_fp = float(cfg.hidden_dropout), float(cfg.activation_dropout), float(cfg.feat_proj_dropout)
        p_at = float(cfg.attention_dropout)
        seed = lambda layer, site: self.drop_seed(step, layer, site)
        sv = SimpleNamespace(B=B, T=T, frame_lens=frame_lens, layers=[], step=step, p_h=p_h, p_a=p_a, p_fp=p_fp, p_at=p_at,
                             spec_rows=None, spec_keep=None, skipped=[], conv=conv_sv, hidden=None, feats=y)
        hidden = [] if collect_hidden else None
        sv.y32 = y.view(M, -1).float()
        _, sv.xn = ops.layernorm(sv.y32, P.fp_ln_w, P.fp_ln_b, eps)
        h0, _ = ops.linear(sv.xn, TP.fp_w_bf16, P.fp_b, want_f32=True, want_bf16=False, seg_rows=T,
                           seg_valid_rows=frame_lens)
        if p_fp > 0:
            ops.dropout(h0, p_fp, seed(-1, self.SITE_PROJ), out_f32=h0)
        if cfg.apply_spec_augment and cfg.mask_time_prob > 0:
            from .specaug import compute_mask_indices
            mask = compute_mask_indices((B, T), cfg.mask_time_prob, cfg.mask_time_length,
                                        frame_lens=frame_lens.cpu().numpy(), min_masks=cfg.mask_time_min_masks)
            rows = torch.from_numpy(mask.reshape(-1).nonzero()[0].astype("int64")).to(wav.device)
            if rows.numel():
                # hidden_states[mask] = masked_spec_embed (HF:1303): an indexed row copy
                h0.index_copy_(0, rows, self.masked_spec_embed.detach().float().expand(rows.numel(), H))
                sv.spec_rows = rows
        if cfg.apply_spec_augment and cfg.mask_feature_prob > 0:
            # feature-axis spans (HF:1314-1322): whole channels of an utterance zeroed, masked_spec_embed rows included
            from .specaug import compute_mask_indices
            fmask = compute_mask_indices((B, H), cfg.mask_feature_prob, cfg.mask_feature_length,
                                         min_masks=cfg.mask_feature_min_masks)
            sv.spec_keep = torch.from_numpy(~fmask).to(wav.device, F32).view(B, 1, H)
            h0.view(B, T, H).mul_(sv.spec_keep)
        sv.hp = ops.cast_pad(h0.view(B, T, H), taps // 2)
        sv.pos_pre = torch.empty((M, H), dtype=BF16, device=wav.device)
        h = torch.empty_like(h0)
        ops.posconv(sv.hp, P.pos_w, P.pos_b, h0, T, H, groups, taps, h, out_pre=sv.pos_pre)
        F_ = cfg.intermediate_size

        def attn(x, li):
            _, qkv = ops.linear(x, lw.qkv_w, lw.qkv_b)
            lse = torch.empty((B, heads, T), dtype=F32, device=wav.device)
            ctx = ops.attention(qkv, frame_lens, B, T, heads, lse=lse, drop_p=p_at,
                                drop_seed=seed(li, self.SITE_ATTN_P))
            return qkv, ctx, lse

        def ffn1(x, li):
            u = torch.empty((M, F_), dtype=BF16, device=wav.device)
            _, g = ops.linear(x, lw.ff1_w, lw.ff1_b, act=1, out_pre=u)
            if p_a > 0:
                ops.dropout(g, p_a, seed(li, self.SITE_ACT), out_bf16=g)
            return u, g

        def proj_res(a, w, b_, res, li, site):
            """res + dropout(a @ w^T + b)"""
            if p_h > 0:
                tmp, _ = ops.linear(a, w, b_, want_f32=True, want_bf16=False)
                return ops.dropout(tmp, p_h, seed(li, site), residual=res, out_f32=tmp)[0]
            return ops.linear(a, w, b_, residual=res, want_f32=True, want_bf16=False)[0]

        def skip_layer():          # HF:701-706 / 773-778
            return bool(torch.rand([]) < cfg.layerdrop) if cfg.layerdrop > 0 else False

        if cfg.do_stable_layer_norm:
            if p_h > 0:
                ops.dropout(h, p_h, seed(-1, self.SITE_ENC), out_f32=h)
            for li, lw in enumerate(P.layers):
                if collect_hidden:
                    hidden.append(h.view(B, T, H))
                if skip_layer():
                    sv.layers.append(None)
                    sv.skipped.append(li)
                    continue
                _, x1 = ops.layernorm(h, lw.ln1_w, lw.ln1_b, eps)
                qkv, ctx, lse = attn(x1, li)
                hm = proj_res(ctx, lw.o_w, lw.o_b, h, li, self.SITE_ATTN)
                _, x2 = ops.layernorm(hm, lw.ln2_w, lw.ln2_b, eps)
                u, g = ffn1(x2, li)
                hn = proj_res(g, lw.ff2_w, lw.ff2_b, hm, li, self.SITE_FFN)
                sv.layers.append(SimpleNamespace(h_in=h, x1=x1, qkv=qkv, ctx=ctx, lse=lse, h_mid=hm, x2=x2, u=u, g=g))
                h = hn
            sv.h_final_in = h
            last, _ = ops.layernorm(h, P.enc_ln_w, P.enc_ln_b, eps, want_f32=True, want_bf16=False)
        else:
            sv.h_enc_in = h
            h, x = ops.layernorm(h, P.enc_ln_w, P.enc_ln_b, eps, want_f32=True, want_bf16=True)
            if p_h > 0:
                ops.dropout(h, p_h, seed(-1, self.SITE_ENC), out_f32=h, out_bf16=x)
            for li, lw in enumerate(P.layers):
                if collect_hidden:
                    hidden.append(h.view(B, T, H))
                if skip_layer():
                    sv.layers.append(None)
                    sv.skipped.append(li)
                    continue
                qkv, ctx, lse = attn(x, li)
                t = proj_res(ctx, lw.o_w, lw.o_b, h, li, self.SITE_ATTN)
                h1, x1 = ops.layernorm(t, lw.ln1_w, lw.ln1_b, eps, want_f32=True, want_bf16=True)
                u, g = ffn1(x1, li)
                t2 = proj_res(g, lw.ff2_w, lw.ff2_b, h1, li, self.SITE_FFN)
                h2, x2 = ops.layernorm(t2, lw.ln2_w, lw.ln2_b, eps, want_f32=True, want_bf16=True)
                sv.layers.append(SimpleNamespace(x_in=x, qkv=qkv, ctx=ctx, lse=lse, t=t, x1=x1, u=u, g=g, t2=t2))
                h, x = h2, x2
            last = h
        object.__setattr__(self, "_last_regularisers", dict(step=step, skipped=list(sv.skipped), spec_rows=sv.spec_rows,
                                                             spec_keep=sv.spec_keep))
        if collect_hidden:
            hidden.append(last.view(B, T, H))
            sv.hidden = tuple(hidden)
        return last.view(B, T, H), sv

    @torch.no_grad()
    def backward(self, sv, d_last: torch.Tensor, gb, prefix: str = "", on_layer_done=None, d_hidden=None) -> None:
        """Accumulate d loss / d parameter for every trainable parameter of the backbone into the GradBuffer `gb`
        (whose parameter names carry `prefix`), given d loss / d last_hidden (fp32 [B*T, H]).  `on_layer_done(i)`
        is called once layer i's gradients are final (data-parallel all-reduce overlap, train.GradReducer).
        `d_hidden`: {i: d loss / d hidden_states[i]} for losses that also read intermediate hidden states
        (models/w2v2_pr.py:91-121).  Frees the saved activations as it consumes them."""
        cfg = self.cfg
        P = TP = self.train_plan()
        B, T, flen = sv.B, sv.T, sv.frame_lens
        M, H = B * T, cfg.hidden_size
        eps, heads = cfg.layer_norm_eps, cfg.num_attention_heads
        taps, groups = cfg.num_conv_pos_embeddings, cfg.num_conv_pos_embedding_groups
        q_scale = float(cfg.head_dim) ** -0.5
        p_h, p_a, p_fp = sv.p_h, sv.p_a, sv.p_fp
        seed = lambda layer, site: self.drop_seed(sv.step, layer, site)
        G = lambda name: gb.view(prefix + name)
        d_last = d_last.reshape(M, H).contiguous()
        d_hidden = {int(k): v.reshape(M, H).to(F32) for k, v in (d_hidden or {}).items() if v is not None}
        if len(sv.layers) in d_hidden:
            d_last = d_last + d_hidden.pop(len(sv.layers))

        def lin_grads(dy_b, x_b, name, bias_done=False):
            ops.wgrad(dy_b, x_b, G(name + ".weight"))
            if not bias_done:
                ops.colsum(dy_b, G(name + ".bias"))

        # Without hidden dropout the gradient of out-proj's / FFN2's OUTPUT is the residual-stream gradient a LayerNorm
        # backward has just produced: that kernel accumulates its column sums (the bias gradient) on the way out
        # (`dcolsum`), which saves the colsum launch that would re-read the tensor.
        fuse_bias = p_h == 0

        def masked16(d32, d16, li, site):
            """bf16 gradient w.r.t. the input of a hidden-dropout site (same mask as the forward)."""
            if p_h > 0:
                return ops.dropout(d32, p_h, seed(li, site), want_bf16=True)[1]
            return d16

        def ffn_block(i, s, lt, dy_b, x_in_b, bias_done=False):
            """FFN2 wgrad/dgrad (through activation dropout and the GELU) and FFN1 wgrad; returns du (bf16)."""
            base = f"encoder.layers.{i}.feed_forward."
            lin_grads(dy_b, s.g, base + "output_dense", bias_done)
            _, du = ops.linear(dy_b, lt.ff2_wt, None, act=2, aux=s.u)
            if p_a > 0:
                ops.dropout(du, p_a, seed(i, self.SITE_ACT), out_bf16=du)
            lin_grads(du, x_in_b, base + "intermediate_dense")
            return du

        def attn_block(i, s, lt, dctx_src_b, x_in_b, bias_done=False):
            """out-proj dgrad -> attention backward -> fused QKV wgrad; returns dqkv."""
            base = f"encoder.layers.{i}.attention."
            lin_grads(dctx_src_b, s.ctx, base + "out_proj", bias_done)
            _, dctx = ops.linear(dctx_src_b, lt.o_wt, None)
            dqkv = ops.attention_bwd(s.qkv, s.ctx, dctx, s.lse, flen, B, T, heads, q_scale, drop_p=sv.p_at,
                                     drop_seed=seed(i, self.SITE_ATTN_P))
            names_w = [prefix + base + n + ".weight" for n in ("q_proj", "k_proj", "v_proj")]
            names_b = [prefix + base + n + ".bias" for n in ("q_proj", "k_proj", "v_proj")]
            ops.wgrad(dqkv, x_in_b, gb.fused(names_w, (3 * H, H)))
            ops.colsum(dqkv, gb.fused(names_b, (3 * H,)))
            return dqkv

        nl = len(sv.layers)
        if cfg.do_stable_layer_norm:
            ff2_b = lambda j: G(f"encoder.layers.{j}.feed_forward.output_dense.bias")
            # the LayerNorm backward that produces layer j's incoming residual gradient also sums its columns when
            # layer j is the next one to run and nothing is added to the gradient in between
            feeds = lambda j: fuse_bias and j >= 0 and sv.layers[j] is not None and (j + 1) not in d_hidden
            ff2_done = feeds(nl - 1)
            dh32, dhb = ops.layernorm_bwd(d_last, sv.h_final_in, P.enc_ln_w, eps, dgamma=G("encoder.layer_norm.weight"),
                                          dbeta=G("encoder.layer_norm.bias"), want_bf16=True,
                                          dcolsum=ff2_b(nl - 1) if ff2_done else None)
            for i in range(nl - 1, -1, -1):
                s, lw, lt = sv.layers[i], P.layers[i], TP.layers[i]
                if s is not None:            # None: the layer was dropped by LayerDrop (identity)
                    base = f"encoder.layers.{i}."
                    du = ffn_block(i, s, lt, masked16(dh32, dhb, i, self.SITE_FFN), s.x2, bias_done=ff2_done)
                    dx2, _ = ops.linear(du, lt.ff1_wt, None, want_f32=True, want_bf16=False)
                    dhm32, dhmb = ops.layernorm_bwd(dx2, s.h_mid, lw.ln2_w, eps, dres=dh32,
                                                    dgamma=G(base + "final_layer_norm.weight"),
                                                    dbeta=G(base + "final_layer_norm.bias"), want_bf16=True,
                                                    dcolsum=G(base + "attention.out_proj.bias") if fuse_bias else None)
                    dqkv = attn_block(i, s, lt, masked16(dhm32, dhmb, i, self.SITE_ATTN), s.x1, bias_done=fuse_bias)
                    dx1, _ = ops.linear(dqkv, lt.qkv_wt, None, want_f32=True, want_bf16=False)
                    ff2_done = feeds(i - 1) and i not in d_hidden
                    dh32, dhb = ops.layernorm_bwd(dx1, s.h_in, lw.ln1_w, eps, dres=dhm32,
                                                  dgamma=G(base + "layer_norm.weight"),
                                                  dbeta=G(base + "layer_norm.bias"), want_bf16=True,
                                                  dcolsum=ff2_b(i - 1) if ff2_done else None)
                    sv.layers[i] = None
                else:
                    ff2_done = False         # a dropped layer passes the gradient on: the next FFN2 sums it itself
                if i in d_hidden:             # hidden_states[i] = the residual stream entering layer i
                    dh32 = dh32 + d_hidden[i]
                    dhb = ops.scale_cast_bf16(dh32)
                if on_layer_done is not None:
                    on_layer_done(i)
            if p_h > 0:
                ops.dropout(dh32, p_h, seed(-1, self.SITE_ENC), out_f32=dh32)
        else:
            dh32 = d_last
            for i in range(nl - 1, -1, -1):
                s, lw, lt = sv.layers[i], P.layers[i], TP.layers[i]
                if i + 1 in d_hidden:         # hidden_states[i+1] = the output of layer i
                    dh32 = dh32 + d_hidden[i + 1]
                if s is not None:
                    base = f"encoder.layers.{i}."
                    dt2, dt2b = ops.layernorm_bwd(dh32, s.t2, lw.ln2_w, eps, dgamma=G(base + "final_layer_norm.weight"),
                                                  dbeta=G(base + "final_layer_norm.bias"), want_bf16=True,
                                                  dcolsum=G(base + "feed_forward.output_dense.bias") if fuse_bias else None)
                    du = ffn_block(i, s, lt, masked16(dt2, dt2b, i, self.SITE_FFN), s.x1, bias_done=fuse_bias)
                    dh1, _ = ops.linear(du, lt.ff1_wt, None, residual=dt2, want_f32=True, want_bf16=False)
                    dt, dtb = ops.layernorm_bwd(dh1, s.t, lw.ln1_w, eps, dgamma=G(base + "layer_norm.weight"),
                                                dbeta=G(base + "layer_norm.bias"), want_bf16=True,
                                                dcolsum=G(base + "attention.out_proj.bias") if fuse_bias else None)
                    dqkv = attn_block(i, s, lt, masked16(dt, dtb, i, self.SITE_ATTN), s.x_in, bias_done=fuse_bias)
                    dh32, _ = ops.linear(dqkv, lt.qkv_wt, None, residual=dt, want_f32=True, want_bf16=False)
                    sv.layers[i] = None
                if on_layer_done is not None:
                    on_layer_done(i)
            if 0 in d_hidden:
                dh32 = dh32 + d_hidden[0]
            if p_h > 0:
                ops.dropout(dh32, p_h, seed(-1, self.SITE_ENC), out_f32=dh32)
            dh32, _ = ops.layernorm_bwd(dh32, sv.h_enc_in, P.enc_ln_w, eps, dgamma=G("encoder.layer_norm.weight"),
                                        dbeta=G("encoder.layer_norm.bias"))
        # positional conv: h1 = h0 + gelu(conv(h0) + b)
        pc = "encoder.pos_conv_embed.conv."
        dpre32 = ops.gelu_bwd(dh32, sv.pos_pre)
        dpre_b = ops.scale_cast_bf16(dpre32)
        ops.colsum(dpre_b, G(pc + "bias"))
        dwf = ops.posconv_wgrad(dpre_b.view(B, T, H), sv.hp, groups, taps)
        ops.posconv_weightnorm_bwd(dwf, TP.pos_g, TP.pos_v, G(pc + "parametrizations.weight.original0"),
                                   G(pc + "parametrizations.weight.original1"))
        dpre_pad = ops.cast_pad(dpre32.view(B, T, H), taps // 2)
        dh0 = torch.empty_like(dh32)
        ops.posconv(dpre_pad, TP.pos_wt, None, dh32, T, H, groups, taps, dh0, act=0, row_shift=1,
                    seg_valid_rows=flen)       # padded frames were zeroed after the projection (HF:678,754)
        if sv.spec_keep is not None:
            dh0.view(sv.B, sv.T, -1).mul_(sv.spec_keep)
        if sv.spec_rows is not None:
            # SpecAugment rows were overwritten by masked_spec_embed: their gradient goes to it, not to the projection
            sel = dh0.index_select(0, sv.spec_rows)
            ops.colsum(sel, G("masked_spec_embed"))
            dh0.index_fill_(0, sv.spec_rows, 0.0)
        if p_fp > 0:
            ops.dropout(dh0, p_fp, seed(-1, self.SITE_PROJ), out_f32=dh0)
        # feature projection + its LayerNorm (the conv encoder below is frozen)
        dh0b = ops.scale_cast_bf16(dh0)
        lin_grads(dh0b, sv.xn, "feature_projection.projection")
        dxn, _ = ops.linear(dh0b, TP.fp_wt, None, want_f32=True, want_bf16=False)
        dy, _ = ops.layernorm_bwd(dxn, sv.y32, P.fp_ln_w, eps, dgamma=G("feature_projection.layer_norm.weight"),
                                  dbeta=G("feature_projection.layer_norm.bias"))
        def release():
            # the step is over: drop every saved activation (the closure that owns `sv` may outlive the backward when
            # the caller keeps the loss tensor, train/train_aptai.py:446 `sum_train_loss += train_loss`)
            for k in list(vars(sv)):
                setattr(sv, k, None)

        if sv.conv is None:
            release()
            return                              # frozen conv feature encoder (models/aptai.py:39-40)
        # ---- conv feature encoder (HF:275-299), layers 6..1 then layer 0
        cs = sv.conv
        rows_per_seg, pitch = T, T
        for i in range(len(cfg.conv_kernel) - 1, 0, -1):
            k, s_ = cfg.conv_kernel[i], cfg.conv_stride[i]
            name = f"feature_extractor.conv_layers.{i}."
            z, x_in = cs.zs[i], cs.ys[i - 1]
            T_out, T_in = z.shape[1], x_in.shape[1]
            if cfg.feat_extract_norm == "layer":
                dz = ops.ln_gelu_bwd(dy, rows_per_seg, pitch, B, P.conv_ln_w[i], P.conv_ln_b[i], 1e-5,
                                     G(name + "layer_norm.weight"), G(name + "layer_norm.bias"), z=z)
            else:
                dz = ops.gelu_bwd_rows(dy, rows_per_seg, pitch, B, z.view(-1, z.shape[2]))
            if P.conv_b[i] is not None:
                ops.colsum(dz, G(name + "conv.bias"))
            dwf = ops.conv_wgrad(dz.view(B, T_out, -1), x_in, k, s_)
            G(name + "conv.weight").add_(dwf.view(dwf.shape[0], k, -1).permute(0, 2, 1))
            dy, pitch = ops.conv_dgrad(dz.view(B, T_out, -1), TP.conv_wt[i], k, s_, T_in)
            rows_per_seg = T_in
            cs.zs[i] = cs.ys[i] = None
        name = "feature_extractor.conv_layers.0."
        T0 = rows_per_seg
        if cfg.feat_extract_norm == "layer":
            dz0 = ops.ln_gelu_bwd(dy, T0, pitch, B, P.conv_ln_w[0], P.conv_ln_b[0], 1e-5, G(name + "layer_norm.weight"),
                                  G(name + "layer_norm.bias"), wav=cs.wav, w0t=TP.conv0_wt, bias0=P.conv_b[0])
        else:
            dz0, sums = ops.conv0_groupnorm_bwd(dy, pitch, cs.wav, T0, P.conv0_w, *cs.gn_saved)
            G(name + "layer_norm.bias").add_(sums[:, :, 0].sum(0))
            G(name + "layer_norm.weight").add_(sums[:, :, 1].sum(0))
        if P.conv_b[0] is not None:
            ops.colsum(dz0, G(name + "conv.bias"))
        X = ops.conv0_im2col(cs.wav, T0)
        dw0 = torch.zeros((dz0.shape[1], 64), dtype=F32, device=dz0.device)
        ops.wgrad(dz0, X, dw0)
        G(name + "conv.weight").add_(dw0[:, : cfg.conv_kernel[0]].reshape(-1, 1, cfg.conv_kernel[0]))
        cs.wav = cs.ys = cs.zs = cs.gn_saved = None
        release()

    # ---- the hot path ----------------------------------------------------------------------------------------
    @torch.no_grad()
    def encode(self, wav: torch.Tensor, frame_lens: torch.Tensor, *, collect_hidden: bool = False,
               want_features: bool = False, final_ln: bool = True):
        """wav fp32 [B,L] (CUDA), frame_lens int32 [B] (CUDA, valid frames per utterance).
        Returns (last_hidden fp32 [B,T,H], hidden tuple | None, features bf16 [B,T,512] | None).
        `final_ln=False` (pre-LN 'stable' encoders in the default precision, no hidden-state collection): the encoder's
        last LayerNorm (HF:792) is left to the caller's fused tail kernel (`ops.tail`) — see `final_ln_params()` —
        and `last_hidden` is the un-normalised residual stream."""
        if self.precision == "f32x3":
            from . import accurate
            return accurate.encode(self, wav, frame_lens, collect_hidden=collect_hidden, want_features=want_features)
        if self.precision not in ("bf16", "fp16"):
            raise ValueError(f"aptai_b200: unknown precision {self.precision!r} ('bf16', 'fp16' or 'f32x3')")
        cfg, P = self.cfg, self.plan()
        X16 = F16 if P.half else BF16          # operand format of the transformer (the conv stack is fp16 either way)
        B, L = wav.shape
        norm = 1 if cfg.feat_extract_norm == "layer" else 2
        # feature encoder + projection run on fp16 operands (activations are O(1) after the norms; three more
        # mantissa bits than bf16 at the same tensor-core rate); the transformer runs on bf16 operands
        y = ops.conv0(wav, P.conv0_w, P.conv_b[0], P.conv_ln_w[0], P.conv_ln_b[0], norm, out_dtype=F16)
        for i in range(1, len(cfg.conv_kernel)):
            y = _conv_layer(y, P, i, cfg)
        T = y.shape[1]
        M = B * T
        H = cfg.hidden_size
        feats = y
        _, xn = ops.layernorm(y.view(M, -1), P.fp_ln_w, P.fp_ln_b, cfg.layer_norm_eps, out16_dtype=F16)
        h, _ = ops.linear(xn, P.fp_w, P.fp_b, want_f32=True, want_bf16=False, seg_rows=T, seg_valid_rows=frame_lens)
        taps = cfg.num_conv_pos_embeddings
        hp = ops.cast_pad(h.view(B, T, H), taps // 2, dtype=X16)
        ops.posconv(hp, P.pos_w, P.pos_b, h, T, H, cfg.num_conv_pos_embedding_groups, taps, h)
        hidden = [] if collect_hidden else None
        eps = cfg.layer_norm_eps
        heads = cfg.num_attention_heads
        if not cfg.do_stable_layer_norm:
            h, x = ops.layernorm(h, P.enc_ln_w, P.enc_ln_b, eps, want_f32=True, want_bf16=True, out16_dtype=X16)
            for lw in P.layers:
                if collect_hidden:
                    hidden.append(h.view(B, T, H).clone())
                _, qkv = ops.linear(x, lw.qkv_w, lw.qkv_b)
                ctx = ops.attention(qkv, frame_lens, B, T, heads)
                t32, _ = ops.linear(ctx, lw.o_w, lw.o_b, residual=h, want_f32=True, want_bf16=False)
                h, x = ops.layernorm(t32, lw.ln1_w, lw.ln1_b, eps, want_f32=True, want_bf16=True, out16_dtype=X16)
                _, u = ops.linear(x, lw.ff1_w, lw.ff1_b, act=1)
                t32, _ = ops.linear(u, lw.ff2_w, lw.ff2_b, residual=h, want_f32=True, want_bf16=False)
                h, x = ops.layernorm(t32, lw.ln2_w, lw.ln2_b, eps, want_f32=True, want_bf16=True, out16_dtype=X16)
            last = h
        else:
            # every activation of a 75 k-row batch (h 300 MB, qkv 450 MB, u 600 MB) exceeds the 126 MB L2: consecutive
            # kernels walk their rows in ALTERNATING directions, so each one starts on the rows its producer wrote last
            serp = ops.Serpentine()
            for lw in P.layers:
                if collect_hidden:
                    hidden.append(h.view(B, T, H).clone())
                serp(); _, x = ops.layernorm(h, lw.ln1_w, lw.ln1_b, eps, out16_dtype=X16)
                serp(); _, qkv = ops.linear(x, lw.qkv_w, lw.qkv_b)
                serp(); ctx = ops.attention(qkv, frame_lens, B, T, heads)
                serp(); ops.linear(ctx, lw.o_w, lw.o_b, residual=h, out_f32=h, want_bf16=False)
                serp(); _, x = ops.layernorm(h, lw.ln2_w, lw.ln2_b, eps, out16_dtype=X16)
                serp(); _, u = ops.linear(x, lw.ff1_w, lw.ff1_b, act=1)
                serp(); ops.linear(u, lw.ff2_w, lw.ff2_b, residual=h, out_f32=h, want_bf16=False)
            serp.done()
            if final_ln or collect_hidden:
                last, _ = ops.layernorm(h, P.enc_ln_w, P.enc_ln_b, eps, want_f32=True, want_bf16=False)
            else:
                last = h
        last = last.view(B, T, H)
        if collect_hidden:
            hidden.append(last)
        return last, (tuple(hidden) if collect_hidden else None), (feats if want_features else None)

    def forward(self, input_values, attention_mask=None, output_hidden_states=False, return_dict=True, **_):
        """HF-compatible call.  `attention_mask` is what the reference passes: `lengths[:, None]`, a (B,1) tensor
        of sample counts (models/aptai.py:77; the cumsum trick of HF:1031), or a (B,L) 0/1 mask, or None."""
        if self.training and torch.is_grad_enabled():
            raise RuntimeError("aptai_b200: Wav2Vec2Backbone.forward is the inference path; training goes through the "
                               "drop-in modules (APTAI / Wav2Vec2_PR .forward in train mode -> encode_train/backward)")
        if not input_values.is_cuda:
            raise RuntimeError("aptai_b200: input_values must be on a CUDA (sm_100) device; there is no CPU path")
        wav = input_values.to(F32).contiguous()
        B, L = wav.shape
        if attention_mask is None:
            lens = torch.full((B,), L, dtype=torch.int64, device=wav.device)
        else:
            am = attention_mask.reshape(B, -1)
            lens = am.sum(-1) if am.shape[1] == L and L > 1 else am[:, -1]
            lens = lens.to(device=wav.device, dtype=torch.int64)
        flen = self.frame_lengths_i32(lens)
        last, hidden, feats = self.encode(wav, flen, collect_hidden=output_hidden_states, want_features=True)
        out = SimpleNamespace(last_hidden_state=last, extract_features=feats, hidden_states=hidden, attentions=None)
        if not return_dict:
            return tuple(v for v in (last, feats, hidden) if v is not None)
        return _Output(out)


class _Output(SimpleNamespace):
    """BaseModelOutput-like: attribute access plus `outputs[0]` (models/w2v2_pr.py:53)."""

    def __init__(self, ns):
        super().__init__(**vars(ns))

    def __getitem__(self, i):
        return tuple(v for v in (self.last_hidden_state, self.extract_features, self.hidden_states) if v is not None)[i]


def _conv_layer(y, P, i, cfg):
    # y comes from ops.conv0 / ops.conv_igemm, whose buffers carry slack rows for the strided TMA view
    return ops.conv_igemm(y, P.conv_w[i], P.conv_b[i], cfg.conv_kernel[i], cfg.conv_stride[i],
                          ln_gamma=P.conv_ln_w[i], ln_beta=P.conv_ln_b[i], act=1)
