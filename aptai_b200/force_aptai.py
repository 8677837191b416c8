"""Drop-in for the reference's models/force_aptai.py (class Force_APTAI) on the aptai_b200 kernels.

Frozen Wav2Vec2_PR -> CTC-decoded phoneme sequence (padded to 60) -> embedding + sinusoidal PE -> cross-attention
frames x phonemes -> log-softmax alignment matrix -> BiLSTM -> 9 TVs -> FIR low-pass; loss = 0.4 MSE + 0.6
forward-sum (CTC over the attention matrix).  Additive API: `forced_align()` — the CTC-Viterbi alignment of the
north star, which the reference does not have (SURVEY.md fact 4) — and `phn_seqs=` to inject known phoneme
sequences instead of decoding (BASELINE config 3).
"""
from __future__ import annotations

import os
import pickle

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .aptai import TV_NAMES
from .modules import CrossAttention, ForwardSumLoss, LowPassFilterLayer, PositionalEncoding, RNN
from .train import GradBuffer, attach_backward, broadcast_parameters
from .w2v2_pr import Wav2Vec2_PR


class Force_APTAI(nn.Module):
    def __init__(self, pr_model_path, device, vocab, w2v2_pr: Wav2Vec2_PR = None):
        super().__init__()
        self.vocab = vocab
        self.device = device
        self.hidden_drop = 0.2
        self.rnn_drop = 0.1
        self.max_phn_seq_len = 60
        self.frame_hidden_dim = 128
        self.phn_hidden_dim = 128
        self.att_hidden_dim = 128
        self.rnn_in_dim = 2 * self.att_hidden_dim
        self.pr_model_path = pr_model_path
        if w2v2_pr is None:
            assert os.path.exists(pr_model_path)
            pr_ckpt_path = os.path.join(pr_model_path, "best-model-ckpt")
            self.w2v2_pr_cfg = pickle.load(open(os.path.join(pr_ckpt_path, "model_cfg.pkl"), "rb"))
            self.w2v2_pr = Wav2Vec2_PR(self.w2v2_pr_cfg["pretrain_cfg"], self.w2v2_pr_cfg["cache_dir"],
                                       self.w2v2_pr_cfg["huggingface_model_id"], vocab).to(self.device)
            self.w2v2_pr.load_state_dict(torch.load(os.path.join(pr_ckpt_path, "pytorch_model.bin"),
                                                    map_location=torch.device(self.device)))
        else:
            self.w2v2_pr_cfg = w2v2_pr.get_config()
            self.w2v2_pr = w2v2_pr.to(self.device)
        H = self.w2v2_pr.wav2vec2.cfg.hidden_size
        self.xatt = CrossAttention(self.frame_hidden_dim, self.phn_hidden_dim, self.att_hidden_dim)
        self.align_loss = ForwardSumLoss()
        self.frame_lin = nn.Linear(H, self.frame_hidden_dim)
        self.frame_drop = nn.Dropout(self.hidden_drop)
        self.phn_emb_layer = nn.Embedding(len(self.vocab), self.phn_hidden_dim, padding_idx=0)
        self.pe_phn = PositionalEncoding(self.phn_hidden_dim, max_len=60, dropout=self.hidden_drop)
        self.rnn = RNN(self.rnn_in_dim, 9, self.rnn_drop)
        self.tv_lowpass = LowPassFilterLayer(self.device, 10, 49, 9)
        for param in self.w2v2_pr.parameters():
            param.requires_grad = False

    def set_precision(self, precision: str):
        """'bf16' (default), 'fp16' (fp16 operands in the frozen recogniser's encoder, same speed) or 'f32x3' (its
        accuracy mode); the tail is fp32 already."""
        self.w2v2_pr.set_precision(precision)
        return self

    # ---------------------------------------------------------------------------------------------- shared trunk
    @torch.no_grad()
    def _recogniser(self, audio_inputs, audio_lengths, phn_seqs=None):
        """Frozen recogniser in eval mode (the reference's get_embeddings switches it to eval and runs under no_grad,
        models/w2v2_pr.py:125-127), CTC-decoded (or injected) phoneme sequences padded to 60 slots."""
        pr = self.w2v2_pr
        if pr.training:
            pr.eval()
        _, h, logits = pr._logits(audio_inputs, audio_lengths)
        dev = h.device
        frame_seq_lens = pr.wav2vec2._get_feat_extract_output_lengths(audio_lengths.reshape(-1)).cpu().tolist()
        phn_pred_list = [np.asarray(s) for s in phn_seqs] if phn_seqs is not None else pr._decode(logits)
        phn_seq_lens = [len(l) for l in phn_pred_list]
        padded = []
        n_emb = self.phn_emb_layer.num_embeddings
        for lst in phn_pred_list:
            assert len(lst) < self.max_phn_seq_len, "Need longer max phoneme sequence length."
            # the cross-attention kernel indexes its embedding table with these ids unchecked
            if len(lst) and (int(np.min(lst)) < 0 or int(np.max(lst)) >= n_emb):
                raise ValueError(f"Force_APTAI: phoneme id {int(np.max(lst))} (or a negative one) outside the "
                                 f"embedding table of {n_emb} entries (len(vocab)); the recogniser's vocabulary must "
                                 "not be larger than Force_APTAI's")
            padded.append(np.pad(lst, (0, self.max_phn_seq_len - len(lst)), mode="constant"))
        phn_pred_seq = torch.tensor(np.stack(padded), dtype=torch.int32, device=dev)
        return h, logits, frame_seq_lens, phn_pred_list, phn_seq_lens, phn_pred_seq

    @torch.no_grad()
    def _trunk(self, audio_inputs, audio_lengths, phn_seqs=None):
        h, logits, frame_seq_lens, phn_pred_list, phn_seq_lens, phn_pred_seq = self._recogniser(
            audio_inputs, audio_lengths, phn_seqs)
        B, T, H = h.shape
        fl = self.frame_lin                 # Linear(H,128) on the tcgen05 GEMM, bf16x3 split (fp32-accurate)
        fh = ops.linear_f32x3(h.reshape(B * T, H).contiguous(), fl.weight, fl.bias.detach().float().contiguous())
        # fused cross-attention kernel: embedding + PE, q/k projections, masked softmax, LayerNorm(256) and the
        # log-softmax alignment matrix (eval mode: the two dropouts are identities)
        xa = self.xatt
        att_out, energy, att = ops.cross_attention(fh.view(B, T, -1), phn_pred_seq.contiguous(),
                                                   self.phn_emb_layer.weight, self.pe_phn.pe[:, 0, :], xa.q.weight,
                                                   xa.q.bias, xa.k.weight, xa.k.bias, xa.layer_norm.weight,
                                                   xa.layer_norm.bias, xa.layer_norm.eps)
        return dict(h=h, logits=logits, frame_seq_lens=frame_seq_lens, phn_pred_list=phn_pred_list,
                    phn_seq_lens=phn_seq_lens, phn_pred_seq=phn_pred_seq, att_out=att_out, att=att)

    def forward(self, epoch, audio_inputs, audio_lengths, phoneme_labels, phn_frames_49hz, LA, LP, JA, TTCL, TTCD,
                TMCL, TMCD, TBCL, TBCD, phn_seqs=None):
        """models/force_aptai.py:80-178."""
        tv_targets = torch.stack([LA, LP, JA, TTCL, TTCD, TMCL, TMCD, TBCL, TBCD], dim=-1).float()
        if self.training:
            return self._forward_train(audio_inputs, audio_lengths, tv_targets, phn_seqs)
        t = self._trunk(audio_inputs, audio_lengths, phn_seqs)
        att = t["att"]
        dev = att.device
        rnn_out = self.rnn(t["att_out"], t["frame_seq_lens"])
        tvs_out = self.tv_lowpass(rnn_out[0].contiguous())
        tv_targets = tv_targets.to(dev)
        tv_pad_mask = tv_targets != -100.0
        d = (tvs_out - tv_targets)[tv_pad_mask]
        tv_loss = (d * d).mean()
        align_loss = self.align_loss(att.unsqueeze(1), t["phn_seq_lens"], t["frame_seq_lens"])
        a = 0.4
        loss = a * tv_loss + (1 - a) * align_loss
        align_out = torch.max(att, axis=2)[1]
        frame_phn = torch.gather(t["phn_pred_seq"].long(), 1, align_out).cpu().numpy()      # one D->H copy
        pred_frame_phns = [[int(x) for x in frame_phn[b, : t["frame_seq_lens"][b]]] for b in range(att.shape[0])]
        return {"loss": loss, "tv_loss": tv_loss, "align_loss": align_loss, "tvs_pred": tvs_out,
                "pred_frame_phns": pred_frame_phns, "pred_ctc_phn_seq": t["phn_pred_list"]}


    # ---------------------------------------------------------------------------------------------- training
    def grad_buffer(self) -> GradBuffer:
        """Flat fp32 gradient buffer over the trainable tail (the recogniser is frozen, models/force_aptai.py:76-78)."""
        gb = getattr(self, "_grad_buffer", None)
        if gb is None:
            gb = GradBuffer(list(self.named_parameters()))
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

    def enable_data_parallel(self, group=None, broadcast: bool = True):
        """Data-parallel training of the tail over `torch.distributed` (one process per GPU; the reference trains on
        one GPU): weights broadcast from rank 0, and every backward ends with one NCCL all-reduce (average) of the flat
        5 MB gradient buffer — too small to be worth bucketing or overlapping."""
        if broadcast:
            broadcast_parameters(self, 0, group)
        object.__setattr__(self, "_dp", (True, group))
        return self.grad_buffer()

    def _drop_seed(self, site: int) -> int:
        # sites 100..102 of the backbone's counter-based generator (frame_drop, pe_phn.dropout, rnn dropout)
        return self.w2v2_pr.wav2vec2.drop_seed(self._drop_step, site, 0)

    def _forward_train(self, audio_inputs, audio_lengths, tv_targets, phn_seqs=None):
        with torch.no_grad():
            loss_val, run_backward, out = self._train_step(audio_inputs, audio_lengths, tv_targets, phn_seqs)
        out["loss"] = attach_backward(loss_val, self.frame_lin.weight, run_backward)
        return out

    def _train_step(self, audio_inputs, audio_lengths, tv_targets, phn_seqs=None):
        """Training step of train/train_force_aptai.py: the forward keeps what the backward needs; `loss.backward()`
        launches the hand-written backward of the tail (low-pass adjoint, head MLP, BiLSTM through time,
        cross-attention, embedding, frame projection).  Dropouts (frame_drop 0.2, positional-encoding 0.2, RNN 0.1) are
        counter-based like the backbone's and regenerated in the backward."""
        h, logits, frame_seq_lens, phn_pred_list, phn_seq_lens, ids = self._recogniser(audio_inputs, audio_lengths,
                                                                                       phn_seqs)
        dev = h.device
        B, T, H = h.shape
        M = B * T
        gb = self.grad_buffer()
        object.__setattr__(self, "_drop_step", getattr(self, "_drop_step", 0) + 1)
        f = lambda p: p.detach().float().contiguous()
        fl, xa, rnn = self.frame_lin, self.xatt, self.rnn
        p_f, p_pe, p_r = float(self.frame_drop.p), float(self.pe_phn.dropout.p), float(rnn.linear[1].p)
        s_f, s_pe, s_r = self._drop_seed(100), self._drop_seed(101), self._drop_seed(102)
        h2 = h.reshape(M, H).contiguous()
        fh = ops.linear_f32x3(h2, fl.weight, f(fl.bias))
        if p_f > 0:
            ops.dropout(fh, p_f, s_f, out_f32=fh)
        phn = (f(self.phn_emb_layer.weight)[ids.long()] + self.pe_phn.pe[:, 0, :].float()[None]).contiguous()
        if p_pe > 0:
            ops.dropout(phn, p_pe, s_pe, out_f32=phn)
        att_out, _, att = ops.cross_attention(fh.view(B, T, -1), ids, None, None, xa.q.weight, xa.q.bias, xa.k.weight,
                                              xa.k.bias, xa.layer_norm.weight, xa.layer_norm.bias, xa.layer_norm.eps,
                                              phn_hidden=phn)
        ln = (torch.as_tensor(frame_seq_lens, dtype=torch.int32).reshape(B).to(dev) if B > 1
              else torch.full((1,), T, dtype=torch.int32, device=dev))
        hidden, lsv = ops.bilstm_256(att_out, rnn.lstm, ln, save=True)
        l0, l3 = rnn.linear[0], rnn.linear[3]
        z1 = ops.linear_f32x3(hidden.view(M, -1), l0.weight, f(l0.bias))
        if p_r > 0:
            ops.dropout(z1, p_r, s_r, out_f32=z1)
        w3 = f(l3.weight)
        raw, _, _ = ops.heads(z1, w3, f(l3.bias), ops.ACT_TANH, None, None, 0, want_argmax=False)
        taps = self.tv_lowpass.lowpass.weight.detach().reshape(-1).to(device=dev, dtype=torch.float64).contiguous()
        tvs_out = ops.lowpass(raw.view(B, T, 9), taps)
        tv_targets = tv_targets.to(dev)
        tv_mask = tv_targets != -100.0
        diff = torch.where(tv_mask, tvs_out - tv_targets, torch.zeros((), device=dev))
        count = tv_mask.sum().clamp(min=1).float()
        tv_loss = (diff * diff).sum() / count
        # forward-sum loss with its gradient w.r.t. the alignment log-probs (models/modules.py:65-117)
        text = torch.as_tensor(phn_seq_lens, dtype=torch.int32, device=dev).reshape(B).contiguous()
        mel = torch.as_tensor(frame_seq_lens, dtype=torch.int32, device=dev).reshape(B).contiguous()
        N = att.shape[2]
        tg = torch.arange(1, N + 1, dtype=torch.int32, device=dev)[None].expand(B, N).contiguous()
        scale = (1.0 / (text.clamp(min=1).float() * B)).contiguous()
        r = ops.logsoftmax_ctc(att, tg, mel, text, blank=0, zero_infinity=True, scale=scale, want_log_probs=False,
                               want_grad=True, prepend_blank=True, blank_value=float(self.align_loss.blank_logprob),
                               vocab_len=(text + 1).contiguous())
        align_loss = r["loss_sum"][0]
        a = 0.4
        loss_val = a * tv_loss + (1 - a) * align_loss
        G = lambda name: gb.view(name)
        bf = ops.scale_cast_bf16

        def run_backward(grad_out):
            gs = grad_out.detach().to(device=dev, dtype=torch.float32)       # upstream scalar, kept on the device
            d_tvs = (diff * (gs * (2.0 * a) / count)).contiguous()
            d_raw = ops.lowpass(d_tvs, taps).view(M, 9)                     # symmetric FIR: adjoint = the filter
            d_z1 = ops.heads_bwd(z1, d_raw, w3, ops.ACT_TANH, G("rnn.linear.3.weight"), G("rnn.linear.3.bias"),
                                 None, None, 0, None, None)
            if p_r > 0:
                ops.dropout(d_z1, p_r, s_r, out_f32=d_z1)
            d_z1b = bf(d_z1)
            ops.wgrad(d_z1b, bf(hidden.view(M, -1)), G("rnn.linear.0.weight"))
            ops.colsum(d_z1, G("rnn.linear.0.bias"))
            d_hidden, _ = ops.linear(d_z1b, f(l0.weight).t().contiguous().to(torch.bfloat16), None, want_f32=True,
                                     want_bf16=False)
            lg = {n: G("rnn.lstm." + n) for n, _ in rnn.lstm.named_parameters()}
            d_att_out = ops.bilstm_256_bwd(lsv, d_hidden.view(B, T, -1), lg)
            d_att = (r["grad"] * (gs * (1 - a))).contiguous()
            d_q, d_k = ops.cross_attention_bwd(fh.view(B, T, -1), ids, phn, xa.q.weight, xa.q.bias, xa.k.weight,
                                               xa.k.bias, xa.layer_norm.weight, xa.layer_norm.eps,
                                               d_att_out.contiguous(), d_att, G("xatt.layer_norm.weight"),
                                               G("xatt.layer_norm.bias"))
            d_qb, d_kb = bf(d_q.view(M, -1)), bf(d_k.view(B * N, -1))
            ops.wgrad(d_qb, bf(fh), G("xatt.q.weight"))
            ops.colsum(d_q.view(M, -1), G("xatt.q.bias"))
            ops.wgrad(d_kb, bf(phn.view(B * N, -1)), G("xatt.k.weight"))
            ops.colsum(d_k.view(B * N, -1), G("xatt.k.bias"))
            d_fh, _ = ops.linear(d_qb, f(xa.q.weight).t().contiguous().to(torch.bfloat16), None, want_f32=True,
                                 want_bf16=False)
            if p_f > 0:
                ops.dropout(d_fh, p_f, s_f, out_f32=d_fh)
            ops.wgrad(bf(d_fh), bf(h2), G("frame_lin.weight"))
            ops.colsum(d_fh, G("frame_lin.bias"))
            d_phn, _ = ops.linear(d_kb, f(xa.k.weight).t().contiguous().to(torch.bfloat16), None, want_f32=True,
                                  want_bf16=False)
            if p_pe > 0:
                ops.dropout(d_phn, p_pe, s_pe, out_f32=d_phn)
            d_emb = G("phn_emb_layer.weight")
            keep = (ids.view(-1) != 0)                                      # padding_idx = 0 receives no gradient
            d_emb.index_add_(0, ids.view(-1).long()[keep], d_phn[keep])
            dp = getattr(self, "_dp", None)
            if dp is not None:
                gb.allreduce(group=dp[1], average=True)

        align_out = torch.max(att, axis=2)[1]
        frame_phn = torch.gather(ids.long(), 1, align_out).cpu().numpy()
        pred_frame_phns = [[int(x) for x in frame_phn[b, : frame_seq_lens[b]]] for b in range(B)]
        object.__setattr__(self, "_last_train", dict(step=self._drop_step, seeds=(s_f, s_pe, s_r)))
        return loss_val, run_backward, {"loss": None, "tv_loss": tv_loss, "align_loss": align_loss, "tvs_pred": tvs_out,
                                        "pred_frame_phns": pred_frame_phns, "pred_ctc_phn_seq": phn_pred_list}

    def get_config(self):
        return {"pr_model_path": self.pr_model_path, "w2v2_pr_cfg": self.w2v2_pr_cfg, "device": self.device,
                "vocab": self.vocab}

    def _single(self, wav):
        dev = next(self.w2v2_pr.parameters()).device
        if type(wav) is torch.Tensor:
            wav = wav[0]
        wav_input = torch.as_tensor(np.asarray(wav), dtype=torch.float32).reshape(1, -1).to(dev)
        wav_len = torch.tensor([wav_input.shape[1]], dtype=torch.int64, device=dev)
        return wav_input, wav_len

    def get_alignment(self, wav, phn_seq=None):
        """models/force_aptai.py:188-236: (N, T) log-softmax alignment matrix."""
        self.eval()
        wav_input, wav_len = self._single(wav)
        t = self._trunk(wav_input, wav_len, None if phn_seq is None else [phn_seq])
        att = t["att"][0]
        res = att[0: t["frame_seq_lens"][0], 0: t["phn_seq_lens"][0]].permute(1, 0)
        return {"alignment": res.detach().cpu().numpy()}

    def get_faptai_output(self, wav, phn_seq=None):
        """models/force_aptai.py:238-322."""
        self.eval()
        wav_input, wav_len = self._single(wav)
        t = self._trunk(wav_input, wav_len, None if phn_seq is None else [phn_seq])
        with torch.no_grad():
            rnn_out = self.rnn(t["att_out"], t["frame_seq_lens"])
            tvs = self.tv_lowpass(rnn_out[0].contiguous())[0].cpu().numpy()
        tvs_pred = {n: list(tvs[:, i]) for i, n in enumerate(TV_NAMES)}
        align_out = torch.max(t["att"][0], axis=1)[1]
        pred_frame_phns = [int(x) for x in t["phn_pred_seq"][0].long()[align_out].cpu().numpy()]
        return {"tvs_pred": tvs_pred, "pred_frame_phns": pred_frame_phns, "pred_ctc_phn_seq": t["phn_pred_list"],
                "hidden_alignment": t["att_out"], "hidden_tvs": rnn_out[1]}

    # ---------------------------------------------------------------------------------------------- additive API
    @torch.no_grad()
    def forced_align(self, audio_inputs, audio_lengths, phn_seqs, log_probs=None):
        """CTC-Viterbi forced alignment of known phoneme sequences against the frozen recogniser's log-probs
        (bit-exact with torchaudio.functional.forced_align on identical log-probs).  Returns (paths int32 [B,T]
        with -1 beyond each utterance, scores fp32 [B,T], status int32 [B])."""
        pr = self.w2v2_pr
        dev = next(pr.parameters()).device
        if log_probs is None:
            _, _, logits = pr._logits(audio_inputs, audio_lengths)
            log_probs = ops.softmax_rows(logits.contiguous(), log=True)
        B, T, V = log_probs.shape
        flen = pr.wav2vec2.frame_lengths_i32(audio_lengths)
        Smax = max(1, max(len(s) for s in phn_seqs))
        tg = np.zeros((B, Smax), dtype=np.int32)
        for b, s in enumerate(phn_seqs):
            tg[b, : len(s)] = np.asarray(s, dtype=np.int32)
        tl = torch.tensor([len(s) for s in phn_seqs], dtype=torch.int32, device=dev)
        return ops.ctc_viterbi(log_probs.contiguous(), torch.from_numpy(tg).to(dev), flen.contiguous(), tl,
                               blank=int(pr.wav2vec2.cfg.blank))
