"""Drop-in for the reference's models/w2v2_pr.py (class Wav2Vec2_PR) on the aptai_b200 kernels.

State dict: `wav2vec2.*`, `pr_head.{weight,bias}`.  `forward` = backbone -> Linear(H, vocab) -> fused
log_softmax + CTC loss (mean, zero_infinity, blank from the config).  The target lengths are counted on the device
(the reference loops over device scalars, models/w2v2_pr.py:62-70), and the conv encoder runs once in
`get_embeddings` (the reference runs it twice, :129).

Decoding: the reference builds a torchaudio/flashlight lexicon-free beam decoder on every call (:143-155).  Here the
default is the on-device `aptai_ctc_decode_ref` kernel, which reproduces that decoder's OUTPUT: with no LM and
max-merge the best beam is the frame-wise argmax path, and flashlight's raw path carries a leading and a trailing
`(...)` silence entry which torchaudio's `_get_tokens` / `_get_timesteps` collapse with the frame labels — so token
lists start / end with the silence id and time stamps are frame + 1 (oracle/ctc_decode.py restates both layers;
flashlight-text itself is not installable here, so that layer stays parity-unpinned).  Any other decoder can be
injected (`phoneme_decoder=`).
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .backbone import Wav2Vec2Backbone
from .config import W2V2Config
from .graphs import GraphCache
from .train import GradBuffer, GradReducer, attach_backward, broadcast_parameters

BLANK_TOKEN, SIL_TOKEN = "(blank)", "(...)"          # models/w2v2_pr.py:152-153


class _HiddenStatesFn(torch.autograd.Function):
    """Gradient-carrying hidden states for `get_embeddings_grad`: autograd delivers d loss / d hidden_states and the
    hand-written backbone backward accumulates the parameter gradients into the model's flat gradient buffer."""

    @staticmethod
    def forward(ctx, anchor, model, sv, idx, *hidden):
        ctx.model, ctx.sv, ctx.idx = model, sv, idx
        return tuple(h.detach().clone() for h in hidden)

    @staticmethod
    def backward(ctx, *grads):
        model, sv, idx = ctx.model, ctx.sv, ctx.idx
        ctx.model = ctx.sv = None
        if sv is None:
            raise RuntimeError("aptai_b200: backward through get_embeddings_grad a second time")
        w2v = model.wav2vec2
        n = len(w2v.encoder.layers)
        d_hidden = {}
        for i, g in zip(idx, grads):
            if g is not None:
                i = i % (n + 1)
                d_hidden[i] = d_hidden[i] + g.float() if i in d_hidden else g.float()
        B, T, H = sv.B, sv.T, w2v.cfg.hidden_size
        d_last = d_hidden.pop(n, None)
        if d_last is None:
            d_last = torch.zeros((B * T, H), dtype=torch.float32, device=sv.frame_lens.device)
        w2v.backward(sv, d_last.contiguous(), model.grad_buffer(), prefix="wav2vec2.", d_hidden=d_hidden)
        return (None,) * (4 + len(idx))


def _head_fwd(hm, w, b):
    """pr_head logits fp32 [rows, V] of h fp32 [rows, H]: the fused heads kernel up to ops.PR_HEAD_NARROW classes, the
    fp32-accurate tensor-core head beyond (ops.pr_head_wide + one pass of ops.logits_rows)."""
    if w.shape[0] <= ops.PR_HEAD_NARROW:
        return ops.heads(hm, None, None, 0, w, b, ops.ACT_NONE, want_argmax=False)[1]
    return ops.logits_rows(ops.pr_head_wide(hm, w, b))[0]


def _head_bwd(hm, w, d_lg, dw, db):
    """dh of `_head_fwd` (fp32 [rows, H]); dw / db accumulate."""
    if w.shape[0] <= ops.PR_HEAD_NARROW:
        return ops.heads_bwd(hm, None, None, 0, None, None, d_lg, w, ops.ACT_NONE, dw, db)
    return ops.pr_head_wide_bwd(hm, w, d_lg, dw, db)


class _HeadFn(torch.autograd.Function):
    """pr_head (Linear H -> vocab) through the heads kernels, differentiable w.r.t. its input and parameters."""

    @staticmethod
    def forward(ctx, h, weight, bias):
        B, T, H = h.shape
        hm = h.detach().reshape(B * T, H).float().contiguous()
        w = weight.detach().float().contiguous()
        logits = _head_fwd(hm, w, bias.detach().float().contiguous())
        ctx.save_for_backward(hm, w)
        return logits.view(B, T, -1)

    @staticmethod
    def backward(ctx, d_logits):
        hm, w = ctx.saved_tensors
        B, T, V = d_logits.shape
        dw = torch.zeros_like(w)
        db = torch.zeros((V,), dtype=torch.float32, device=w.device)
        dh = _head_bwd(hm, w, d_logits.reshape(B * T, V).float().contiguous(), dw, db)
        return dh.view(B, T, -1), dw, db


def idx_phonemes(vocab, seq):
    """utility.py:200-210."""
    keys, vals = list(vocab.keys()), list(vocab.values())
    return [keys[vals.index(int(i))] for i in seq]


class Wav2Vec2_PR(nn.Module):
    def __init__(self, pretrain_cfg, cache_dir, huggingface_model_id, vocab=None,
                 phoneme_decoder: Optional[Callable] = None):
        super().__init__()
        vocab_size = int(getattr(pretrain_cfg, "vocab_size", 0))
        if vocab_size > ops.PR_HEAD_MAX_VOCAB:
            raise ValueError(f"Wav2Vec2_PR: vocab_size={vocab_size} exceeds the recogniser head's limit of "
                             f"{ops.PR_HEAD_MAX_VOCAB} symbols")
        self.cache_dir = cache_dir
        self.huggingface_model_id = huggingface_model_id
        self.pretrain_cfg = pretrain_cfg
        self.wav2vec2 = Wav2Vec2Backbone.from_pretrained(huggingface_model_id, config=pretrain_cfg,
                                                         cache_dir=cache_dir)
        self.wav2vec2.gradient_checkpointing_enable()
        cfg = self.wav2vec2.cfg
        self.dropout = nn.Dropout(cfg.final_dropout)
        self.pr_head = nn.Linear(cfg.hidden_size, cfg.vocab_size)       # parameter container
        self.vocab = vocab
        self.phoneme_decoder = phoneme_decoder

    # ---------------------------------------------------------------------------------------------- kernels
    @torch.no_grad()
    def _logits(self, input_values, input_lengths, output_hidden_states=False):
        if self.training and self.dropout.p > 0:
            raise RuntimeError("aptai_b200: this is the inference path (no final dropout); in training mode call "
                               "forward() with autograd enabled, or .eval() first")
        out = self.wav2vec2(input_values, attention_mask=input_lengths.reshape(-1)[:, None], return_dict=True,
                            output_hidden_states=output_hidden_states)
        h = out.last_hidden_state
        logits = self._head(h)
        return out, h, logits

    def _head(self, h):
        B, T, H = h.shape
        f = lambda p: p.detach().float().contiguous()
        logits = _head_fwd(h.reshape(B * T, H).contiguous(), f(self.pr_head.weight), f(self.pr_head.bias))
        return logits.view(B, T, -1)

    def enable_data_parallel(self, group=None, layers_per_bucket: int = 4, broadcast: bool = True,
                             overlap_optimizer: bool = False):
        """Data-parallel training over `torch.distributed` (one process per GPU): weights are broadcast from rank 0
        and every backward all-reduces (averages) the flat gradient buffer, bucketed by encoder layers and
        overlapped with the remaining backward kernels (BASELINE config 4; the reference trains single-GPU).
        `overlap_optimizer`: see `APTAI.enable_data_parallel`."""
        if broadcast:
            broadcast_parameters(self, 0, group)
        gb = self.grad_buffer()
        red = GradReducer(gb, "wav2vec2.encoder.layers.", len(self.wav2vec2.encoder.layers), layers_per_bucket, group,
                          defer_wait=overlap_optimizer)
        object.__setattr__(self, "_reducer", red)
        return red

    def grad_buffer(self) -> GradBuffer:
        gb = getattr(self, "_grad_buffer", None)
        if gb is None:
            gb = GradBuffer(list(self.named_parameters()), self.wav2vec2.fused_grad_groups("wav2vec2."))
            object.__setattr__(self, "_grad_buffer", gb)
            return gb
        dropped = False
        for n, p in gb.params:
            if not gb.owns(p):
                dropped = True
                p.grad = gb.flat[gb.offsets[n]: gb.offsets[n] + p.numel()].view(p.shape)
        if dropped:
            gb.zero()
        return gb

    def forward(self, input_values, input_lengths, phoneme_labels, want_grad=False):
        """models/w2v2_pr.py:40-88.  `want_grad=True` additionally returns d loss / d phoneme_logits from the
        fused kernel (key 'grad_logits'), the implementation-independent quantity of SURVEY.md §3.3.
        In training mode with autograd enabled, `loss.backward()` runs the hand-written backward kernels
        (train/train_phoneme_recognizer.py: loss.backward(); optimizer.step())."""
        cfg = self.wav2vec2.cfg
        train = self.training and torch.is_grad_enabled()
        sv = None
        if train:
            dev0 = next(self.wav2vec2.parameters()).device
            wav = input_values.to(device=dev0, dtype=torch.float32).contiguous()
            lens = input_lengths.reshape(-1).to(device=dev0, dtype=torch.int64)
            flen = self.wav2vec2.frame_lengths_i32(lens)
            gb = self.grad_buffer()
            h, sv = self.wav2vec2.encode_train(wav, flen)
            p_fin = float(self.dropout.p)                      # final_dropout (models/w2v2_pr.py:56)
            s_fin = self.wav2vec2.drop_seed(sv.step, -1, self.wav2vec2.SITE_HEAD_A)
            h_in = ops.dropout(h, p_fin, s_fin, want_f32=True)[0] if p_fin > 0 else h
            logits = self._head(h_in)
            h = h_in                                           # the reference returns the dropped hidden states (:53-58)
            want_grad = True
        else:
            out, h, logits = self._logits(input_values, input_lengths)
        dev = h.device
        B, T, V = logits.shape
        state_lens = self.wav2vec2._get_feat_extract_output_lengths(input_lengths.reshape(-1).to(dev))
        labels = phoneme_labels.to(device=dev, dtype=torch.int32).contiguous()
        target_lengths = (labels >= 0).sum(-1).to(torch.int32).contiguous()
        if cfg.ctc_loss_reduction == "mean":
            scale = 1.0 / (target_lengths.clamp(min=1).float() * B)
        elif cfg.ctc_loss_reduction == "sum":
            scale = torch.ones((B,), dtype=torch.float32, device=dev)
        else:
            raise ValueError(f"unsupported ctc_loss_reduction {cfg.ctc_loss_reduction!r}")
        r = ops.logsoftmax_ctc(logits.contiguous(), labels, state_lens.to(torch.int32).contiguous(), target_lengths,
                               blank=int(cfg.blank), zero_infinity=bool(cfg.ctc_zero_infinity),
                               scale=scale.contiguous(), want_log_probs=True, want_grad=want_grad)
        res = {"loss": r["loss_sum"][0], "phoneme_logits": logits, "log_probs": r["log_probs"], "hidden_states": h}
        if want_grad:
            res["grad_logits"] = r["grad"]
        if train:
            hm = h_in.reshape(B * T, -1)
            w = self.pr_head.weight.detach().float().contiguous()

            def run_backward(grad_out):
                d_lg = (r["grad"] * grad_out.detach().to(device=dev, dtype=torch.float32)).view(B * T, V).contiguous()
                dh = _head_bwd(hm, w, d_lg, gb.view("pr_head.weight"), gb.view("pr_head.bias"))
                if p_fin > 0:
                    ops.dropout(dh, p_fin, s_fin, out_f32=dh)
                red = getattr(self, "_reducer", None)
                self.wav2vec2.backward(sv, dh, gb, prefix="wav2vec2.", on_layer_done=red.layer_done if red else None)
                if red is not None:
                    red.finish()

            res["loss"] = attach_backward(res["loss"], self.pr_head.weight, run_backward)
        return res

    def _token_ids(self, vocab=None):
        """(blank, sil) ids as the reference's decoder sees them: positions in `list(vocab.keys())` (:144-153)."""
        vocab = vocab if vocab is not None else self.vocab
        if vocab is None:
            return int(self.wav2vec2.cfg.blank), 1
        keys = list(vocab.keys())
        return keys.index(BLANK_TOKEN), keys.index(SIL_TOKEN)

    def _decode(self, phoneme_logits, frame_lens=None, vocab=None, with_timesteps=False):
        """List of int arrays, one per utterance: what `decoder(logits)[b][0].tokens` holds in the reference (all
        frames are decoded: the reference passes no lengths to its decoder, :155)."""
        if self.phoneme_decoder is not None:
            return [np.asarray(x) for x in self.phoneme_decoder(phoneme_logits)]
        blank, sil = self._token_ids(vocab)
        tok, steps, n = ops.ctc_decode_ref(phoneme_logits.contiguous(), frame_lens, blank=blank, sil=sil)
        tok, steps, n = tok.cpu().numpy(), steps.cpu().numpy(), n.cpu().numpy()
        toks = [tok[b, : n[b]].astype(np.int64) for b in range(tok.shape[0])]
        if with_timesteps:
            return toks, [steps[b, : n[b]].astype(np.int32) for b in range(tok.shape[0])]
        return toks

    def get_embeddings(self, audio_inputs, audio_lengths):
        """models/w2v2_pr.py:124-167."""
        self.eval()
        with torch.no_grad():
            out, h, logits = self._logits(audio_inputs, audio_lengths)
            frame_seq_lens = self.wav2vec2._get_feat_extract_output_lengths(audio_lengths)
            phn_seq_idx = self._decode(logits)
            return {
                "features_hidden": out.extract_features.float().permute(0, 2, 1),
                "last_transf_hidden": h.permute(0, 2, 1),
                "phoneme_logits": logits.cpu().numpy().transpose(0, 2, 1),
                "phn_pred_seq_idx": phn_seq_idx,
                "frame_seq_lens": frame_seq_lens.cpu().numpy(),
            }

    def get_embeddings_grad(self, audio_inputs, audio_lengths, vocab, intermediate_hidden, latter_hidden):
        """models/w2v2_pr.py:91-121.  With autograd enabled the hidden states and logits carry gradients like the
        reference's: `.backward()` of anything computed from them runs the hand-written backbone backward (into
        `p.grad` of the backbone parameters, views of the flat gradient buffer) and the heads backward (pr_head).
        The module's mode decides the regularisers, as in the reference (eval: none).  `features_hidden` is returned
        detached."""
        w2v = self.wav2vec2
        if not torch.is_grad_enabled():
            out = w2v(audio_inputs, attention_mask=audio_lengths.reshape(-1)[:, None], return_dict=True,
                      output_hidden_states=True)
            last, inter, latter = (out.last_hidden_state, out.hidden_states[intermediate_hidden],
                                   out.hidden_states[latter_hidden])
            feats = out.extract_features
            head = lambda x: self._head(x.contiguous())
        else:
            dev = next(w2v.parameters()).device
            wav = audio_inputs.to(device=dev, dtype=torch.float32).contiguous()
            lens = audio_lengths.reshape(-1).to(device=dev, dtype=torch.int64)
            flen = w2v.frame_lengths_i32(lens)
            self.grad_buffer()
            _, sv = w2v.encode_train(wav, flen, regularise=self.training, collect_hidden=True)
            idx = (len(w2v.encoder.layers), intermediate_hidden, latter_hidden)
            feats = sv.feats
            last, inter, latter = _HiddenStatesFn.apply(self.pr_head.weight, self, sv, idx,
                                                        *[sv.hidden[i] for i in idx])
            head = lambda x: _HeadFn.apply(x, self.pr_head.weight, self.pr_head.bias)
        return {
            "features_hidden": feats.float().permute(0, 2, 1),
            "last_transf_hidden": last.permute(0, 2, 1),
            "phoneme_logits_last": head(last),
            "phoneme_logits_inter": head(inter),
            "phoneme_logits_latter": head(latter),
            "intermediate_hidden": inter.permute(0, 2, 1),
            "latter_hidden": latter.permute(0, 2, 1),
        }

    def _single(self, wav):
        dev = next(self.wav2vec2.parameters()).device
        if type(wav) is torch.Tensor:
            wav = wav[0]
        wav_input = torch.as_tensor(np.asarray(wav), dtype=torch.float32).reshape(1, -1).to(dev)
        wav_len = torch.tensor([wav_input.shape[1]], dtype=torch.int64, device=dev)
        if not self.use_cuda_graphs or self.wav2vec2.precision not in ("bf16", "fp16"):
            return wav_input, self._logits(wav_input, wav_len)[2]
        cache = getattr(self, "_graph_cache", None)
        if cache is None:
            cache = GraphCache()
            object.__setattr__(self, "_graph_cache", cache)
        P = self.wav2vec2.plan()
        (logits,) = cache.run((id(P), P.generation, int(wav_input.shape[1])),
                              lambda w, l: (self._logits(w, l)[2],), wav_input, wav_len)
        return wav_input, logits

    use_cuda_graphs = True      # single-utterance calls are launch-bound: replay one CUDA graph per input length

    def get_ctc_logits(self, wav):
        """models/w2v2_pr.py:170-188."""
        self.eval()
        with torch.no_grad():
            _, logits = self._single(wav)
            return logits[0].cpu().numpy()

    def pred_phn_seq(self, wav, vocab):
        """models/w2v2_pr.py:238-277."""
        self.eval()
        with torch.no_grad():
            _, logits = self._single(wav)
            idx = self._decode(logits, vocab=vocab)[0]
            return {"phn_seq_idx": idx, "phn_seq_ipa": idx_phonemes(vocab, idx)}

    def predict_phonemes_durations(self, wav, vocab):
        """models/w2v2_pr.py:191-235: time stamps = the decoder's `timesteps` (index of each token's first entry in
        the raw path, i.e. frame + 1; 0 for the leading silence) * seconds per frame."""
        self.eval()
        with torch.no_grad():
            wav_input, logits = self._single(wav)
            frame_sec_ratio = wav_input.shape[1] / logits.shape[1] / 16000
            if self.phoneme_decoder is not None:
                raise NotImplementedError("predict_phonemes_durations needs the built-in decoder's time stamps")
            toks, steps = self._decode(logits, vocab=vocab, with_timesteps=True)
            idx, ts = toks[0], steps[0]
            return {"phn_seq_idx": idx, "phn_seq_ipa": idx_phonemes(vocab, idx),
                    "phn_seq_dur": [t * frame_sec_ratio for t in ts]}

    def set_precision(self, precision: str):
        """'bf16' (default), 'fp16' (same kernels on IEEE fp16 operands: same speed, 7x smaller output error;
        inference only) or 'f32x3' (accuracy mode of the encoder, aptai_b200/accurate.py; inference only)."""
        self.wav2vec2.set_precision(precision)
        return self

    def get_config(self):
        return {"huggingface_model_id": self.huggingface_model_id, "cache_dir": self.cache_dir,
                "pretrain_cfg": self.pretrain_cfg}

    def freeze_feature_encoder(self):            # the reference's version lacks `self` (models/w2v2_pr.py:290-291)
        self.wav2vec2.freeze_feature_encoder()
