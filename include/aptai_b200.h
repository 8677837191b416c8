/* aptai_b200 — C ABI of the B200-native APTAI hot path.
 *
 * The reference (tobwei/APTAI) has no FFI of its own: its hot path is the Python nn.Module API of
 * models/aptai.py, models/w2v2_pr.py, models/force_aptai.py, models/modules.py, which in turn calls
 * transformers.Wav2Vec2Model and torch ops (SURVEY.md §8b).  Each entry point below replaces one library call
 * the reference makes on that path; the call site it replaces is cited next to it ("HF:n" = transformers 5.5.0
 * models/wav2vec2/modeling_wav2vec2.py line n).  The Python facade in aptai_b200/ binds these with ctypes.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is DEVICE memory unless the name ends in _host
 *  - the caller (PyTorch) owns all buffers; nothing here allocates device memory
 *  - all launches are asynchronous on `stream` (a cudaStream_t passed as void*)
 *  - return 0 on success, negative aptai_status on argument errors, positive cudaError_t on launch errors;
 *    aptai_last_error_string() returns a thread-local message
 *  - there is no CPU fallback: on a device that is not sm_100 every compute call returns APTAI_ERR_ARCH
 */
#ifndef APTAI_B200_H
#define APTAI_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum aptai_status {
  APTAI_OK = 0,
  APTAI_ERR_ARG = -1,       /* bad shape / null pointer / misalignment */
  APTAI_ERR_ARCH = -2,      /* device is not sm_100 */
  APTAI_ERR_WORKSPACE = -3, /* workspace too small */
  APTAI_ERR_DRIVER = -4     /* cuTensorMapEncodeTiled unavailable / failed */
};

int aptai_version(void);
const char* aptai_last_error_string(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
int64_t aptai_launch_count(void);

/* ------------------------------------------------------------------ tcgen05 GEMM family ---------------------
 * One kernel family serves nn.Linear (HF:429-434, 524-547, 566-573), the strided conv layers 1..6 as implicit
 * GEMM (HF:254-323) and the grouped positional conv (HF:329-368).
 *
 *   out[s, r, n] = epilogue( sum_{tap, c} A[s, (r*P + tap), colbase(n) + c] * W[n, tap*kb_per_tap*64 + c] )
 *
 * A is bf16, logically [segs][a_rows][a_cols] with row stride a_row_stride and segment stride a_seg_stride
 * (elements).  W is bf16 [N][K] row-major (K contiguous), K = taps*kb_per_tap*64.
 * Plain GEMM: segs=1, P=1, taps=1.  Conv k/stride 2: P=2, taps=k, kb_per_tap=C_in/64.
 * Grouped pos-conv: taps=128, kb_per_tap=1, block_n = group width, a_col_per_nblk = group width.
 * epilogue: (+bias[n]) -> (LayerNorm over the N=512 row, ln=1) -> (GELU, act=1) -> (+residual) ->
 *           (padded rows written as 0, see seg_valid_rows) -> fp32 and/or bf16 store at row s*out_seg_stride + r.
 */
typedef struct aptai_gemm_args {
  const void* a;          /* bf16 */
  int64_t a_row_stride;   /* elements */
  int64_t a_seg_stride;   /* elements */
  int32_t a_rows;         /* physical rows per segment the TMA may touch */
  int32_t a_cols;         /* channels per physical row */
  int32_t P;              /* row step per output row (conv stride) */
  int32_t taps;
  int32_t kb_per_tap;     /* 64-element K blocks per tap */
  int32_t a_col_per_nblk; /* channel offset per n tile (grouped conv), else 0 */
  const void* w;          /* bf16 [N][K] */
  int32_t N;
  int32_t block_n;        /* 0 = choose; otherwise one of 48, 64, 128, 256.  ln=1: 0 or 256, the half-split row tile
                             (two 256-column accumulator halves, epilogue overlapped with the MMAs) */
  int32_t segs;
  int32_t rows_per_seg;   /* output rows per segment */
  const float* bias;      /* [N] or NULL */
  const float* gamma;     /* [N], ln=1 only */
  const float* beta;      /* [N], ln=1 only */
  const float* residual;  /* fp32, same row mapping and ldo as the outputs, or NULL */
  float* out_f32;         /* or NULL */
  void* out_bf16;         /* or NULL */
  int64_t ldo;            /* output row pitch in elements */
  int64_t out_seg_stride; /* output rows between segments */
  const int32_t* seg_valid_rows; /* [out_rows / mask_seg_rows] or NULL: valid rows per masking segment */
  int32_t mask_seg_rows;  /* output row o = s*out_seg_stride + r is zeroed when o % mask_seg_rows >= seg_valid_rows[o / mask_seg_rows] */
  int32_t act;            /* 0 none, 1 erf-GELU, 2 multiply by gelu'(aux) (backward) */
  int32_t ln;             /* 0/1: LayerNorm over the full row (requires N == 512) */
  float ln_eps;
  int32_t cta_pair;       /* 0 auto, 1 single-CTA tiles (128 x BN), 2 CTA-pair tiles (256 x BN, cta_group::2) */
  int32_t half_fmt;       /* 0: A, W and out_bf16 are bf16; 1: they are IEEE fp16 (conv stack / feature projection) */
  const void* aux;        /* act=2 only: bf16, same row mapping/ldo as the outputs: out = acc * gelu'(aux)  (dgrad of
                             HF:566-573 through the activation) */
  void* out_pre;          /* optional 16-bit copy of the value before the activation (kept for the backward pass) */
} aptai_gemm_args;

int aptai_gemm_bf16(const aptai_gemm_args* args, void* stream);

/* Traversal hint for the calling thread's NEXT launches of aptai_gemm_bf16 / aptai_layernorm / aptai_attention_fwd_v3:
 * reverse != 0 makes them walk their output tiles / rows / utterances from the end.  Results are identical.  A chain of
 * kernels whose activations exceed the 126 MB L2 (LayerNorm -> QKV -> attention -> out-proj -> ...) alternates the
 * direction, so that every kernel STARTS on the rows its producer wrote LAST, which are still in L2. */
void aptai_set_traversal(int reverse);

/* ------------------------------------------------------------------ feature encoder front end ---------------
 * conv layer 0 (1 -> 512 channels, kernel 10, stride 5) + norm + GELU, channels-last bf16 output [B][T0][512].
 * norm=1: LayerNorm over channels per frame (HF:281-299).  norm=2: GroupNorm(512 groups) over time per
 * channel, statistics over all T0 frames of the padded row (HF:308-323).  norm=0: none (HF:260-272).
 * w is fp32 [512][10]; bias may be NULL.  stats_ws: aptai_conv0_workspace_bytes(B, norm) bytes, 256-byte aligned
 * (normalisation statistics — for norm=2 B*65 doubles of waveform moments followed by the [B][512][2] scale / shift
 * array and the [B][512][2] {mean - bias, rstd} array the backward pass re-uses — then the 64 KB split-bf16 weight
 * operand of the tensor-core kernel).
 * flags: bit 0 = the 16-bit output is IEEE fp16 instead of bf16; bit 1 = run the SIMT kernel instead of the
 * tcgen05 one (csrc/conv0_tc.cu: the K = 10 contraction on three-term split bf16 operands, fp32-exact to 2^-24) —
 * for A/B measurements, the results agree to fp32 rounding.
 */
size_t aptai_conv0_workspace_bytes(int B, int norm);
int aptai_conv0_norm_gelu(const float* wav, int B, int64_t L, const float* w, const float* bias,
                          const float* gamma, const float* beta, int norm, float eps, void* out_bf16, int T0,
                          float* stats_ws, int flags, void* stream);

/* LayerNorm over the last dim (HF:431, 600-602, 639, 645, 692, 792): fp32 / bf16 / fp16 in, fp32 and/or 16-bit
 * (bf16, or fp16 when out16_fp16) out. */
int aptai_layernorm(const void* x, int x_fmt /* 0 f32, 1 bf16, 2 fp16 */, int64_t rows, int cols, const float* gamma,
                    const float* beta, float eps, float* out_f32, void* out_bf16, int out16_fp16, void* stream);

/* fp32 [segs][rows][cols] -> bf16 [segs][halo+rows+halo][cols] with zeroed halo rows (HF:371-379 'same' pad). */
int aptai_cast_pad_bf16(const float* x, int segs, int rows, int cols, int halo, void* out_bf16, void* stream);
/* same with the 16-bit format chosen by the caller: half_fmt 0 = bf16, 1 = IEEE fp16 (precision="fp16" inference) */
int aptai_cast_pad_h16(const float* x, int segs, int rows, int cols, int halo, void* out_h16, int half_fmt,
                       void* stream);

/* weight-norm fold of the positional conv (torch parametrizations.weight_norm, dim=2; HF:336-358):
 * w[o][c][j] = g[j] * v[o][c][j] / ||v[:, :, j]||, written bf16 as [H][taps][cpad] (cpad >= cin, zero padded). */
int aptai_posconv_fold(const float* g, const float* v, int H, int cin, int taps, int cpad, void* w_bf16,
                       float* norm_ws, void* stream);
int aptai_posconv_fold_fmt(const float* g, const float* v, int H, int cin, int taps, int cpad, void* w_h16,
                           float* norm_ws, int half_fmt /* 0 bf16, 1 fp16 */, void* stream);

/* Grouped positional conv for 64-channel groups (H % 64 == 0, 128 taps), in place on the fp32 hidden stream:
 * h[b][t][:] += gelu(conv(x_pad)[b][t][:] + bias)  (HF:329-379; x_pad bf16 [B][T+128][H] from aptai_cast_pad_bf16,
 * w_fold bf16 [H][128*64] from aptai_posconv_fold).  Every input row is loaded once per (256-frame block, group): the tap
 * shift is a descriptor offset into a shared-memory slab (csrc/posconv_tc.cu). */
int aptai_posconv_slab(const void* x_pad, const void* w_fold, const float* bias, float* h, int B, int T, int H,
                       void* stream);
/* same on operands in the caller's 16-bit format (x_pad and w_fold both bf16, half_fmt 0, or both fp16, half_fmt 1) */
int aptai_posconv_slab_fmt(const void* x_pad, const void* w_fold, const float* bias, float* h, int B, int T, int H,
                           int half_fmt, void* stream);

/* ------------------------------------------------------------------ attention (HF:500-549, SDPA) ------------
 * qkv: bf16 [B*T][3*H] (q | k | v, q pre-scaled by head_dim^-0.5), ctx: bf16 [B*T][H], head_dim 64.
 * Keys t >= key_len[b] are masked; every query row is computed (padded queries attend to valid keys, HF:438-463).
 */
int aptai_attention_fwd(const void* qkv, void* ctx, const int32_t* key_len, int B, int T, int heads, void* stream);
/* same kernel with the 16-bit format of qkv / ctx chosen by the caller (half_fmt 0 = bf16, 1 = IEEE fp16: q, k, v, the
 * probabilities and the context carry three more mantissa bits at the same tensor-core rate); lse may be NULL */
int aptai_attention_fwd_fmt(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T, int heads,
                            int half_fmt, void* stream);
/* third-generation kernel, same contract (csrc/attention_v3.cu): P stays in TMEM as the A operand of P V, three S
 * buffers per query tile, 3 of every 8 exponential pairs on the FMA pipe, TMA store of the context tile.
 * half_fmt as in aptai_attention_fwd_fmt (0 = bf16, 1 = IEEE fp16); lse may be NULL. */
int aptai_attention_fwd_v3(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T, int heads,
                           int half_fmt, void* stream);

/* ------------------------------------------------------------------ heads and post-processing ---------------
 * APTAI heads (models/aptai.py:43-55,83-86,105-106): tv = tanh(h) W_tv^T + b_tv (9), logits = leaky_relu(h)
 * W_phn^T + b_phn (V), pred = argmax (first maximum).  act_a/act_b: 0 identity, 1 tanh, 2 leaky_relu(0.01).
 * Either head may be absent (n = 0).  h is fp32 [rows][H].
 */
int aptai_heads(const float* h, int64_t rows, int H, const float* wa, const float* ba, int na, int act_a,
                float* out_a, const float* wb, const float* bb, int nb, int act_b, float* out_b,
                int64_t* argmax_b, void* stream);

/* Phoneme-recogniser head wider than aptai_heads' 48 head-B slots (models/w2v2_pr.py:47 pr_head = Linear(H, V)),
 * 1 <= V <= 1024, H a multiple of 64 (csrc/pr_head.cu).  fp32 accuracy on the tensor cores: the split-operand GEMM of
 * the accuracy mode, [h_hi | h_lo | h_hi] . [W_hi | W_hi | W_lo]^T + b (relative error ~2^-17 of |h| |W|).
 * Padding and pitch: W gets zero rows up to Vp = 64 * ceil(V / 64) (a GEMM tile width), and `out` is fp32 [rows][ld_out]
 * with ld_out >= Vp, ld_out % 8 == 0: columns [0, V) hold the logits, [V, Vp) are written with zeros, columns >= Vp
 * are not touched.  b may be NULL.  ws: aptai_pr_head_wide_workspace_bytes(rows, H, V, 0) bytes, 256-byte aligned.
 * Nothing here allocates or synchronises (CUDA-graph capturable): the weight split runs on every call. */
size_t aptai_pr_head_wide_workspace_bytes(int64_t rows, int H, int V, int backward);
int aptai_pr_head_wide(const float* h, int64_t rows, int H, const float* w, const float* b, int V, float* out,
                       int64_t ld_out, void* ws, size_t ws_bytes, void* stream);
/* One pass over fp32 rows x [rows][ldx] (columns [0, V), V <= 1024, one warp per row): any of the compact logits
 * fp32 [rows][V], the first-max argmax int64 [rows], log_softmax and softmax fp32 [rows][V] (each may be NULL). */
int aptai_logits_rows(const float* x, int64_t rows, int V, int64_t ldx, float* logits, int64_t* argmax, float* logp,
                      float* prob, void* stream);
/* Backward of aptai_pr_head_wide: d_logits fp32 [rows][V] with row pitch ld_d >= V;
 * dh = d_logits W (written, fp32 [rows][H]), dw += d_logits^T h (fp32 [V][H]), db += column sums (fp32 [V]); each
 * output may be NULL.  Split-operand GEMMs (K = 3 Vp for dh; three MN-major wgrad products for dw).
 * ws: aptai_pr_head_wide_workspace_bytes(rows, H, V, 1) bytes, 256-byte aligned. */
int aptai_pr_head_wide_bwd(const float* h, int64_t rows, int H, const float* w, int V, const float* d_logits,
                           int64_t ld_d, float* dh, float* dw, float* db, void* ws, size_t ws_bytes, void* stream);

/* LowPassFilterLayer (models/modules.py:46-61): per channel 51-tap FIR, zero 'same' padding along T, fp64
 * accumulation of the fp64 taps, fp32 in/out [B][T][C]. */
int aptai_lowpass_fir(const float* x, int B, int T, int C, const double* taps, int ntaps, float* y, void* stream);

/* softmax (log_out=0) or log_softmax (log_out=1) over the last dim of fp32 [rows][V]
 * (models/aptai.py:105,148 F.softmax; models/force_aptai.py:130 log_softmax). */
int aptai_softmax_rows(const float* x, int64_t rows, int V, int log_out, float* y, void* stream);
/* Tail of the forward in one launch: optional final LayerNorm of the pre-LN encoder (HF:792; ln_gamma/ln_beta NULL = h is
 * already normalised) -> both heads as in aptai_heads -> argmax of head B (may be NULL) -> log_softmax of head B (logp_b,
 * may be NULL: the input of the alignment stage) -> optionally the normalised hidden state (h_norm fp32 [rows][H], may be
 * NULL).  Replaces models/aptai.py:83-86,105-106 + the encoder's last LayerNorm + F.log_softmax.  H % 32 == 0, H <= 1024. */
int aptai_tail(const float* h, int64_t rows, int H, const float* ln_gamma, const float* ln_beta, float eps,
               const float* wa, const float* ba, int na, int act_a, float* out_a, const float* wb, const float* bb,
               int nb, int act_b, float* out_b, int64_t* argmax_b, float* logp_b, float* h_norm, void* stream);
/* frames per utterance after the conv feature encoder (HF:1005-1024 `_get_feat_extract_output_lengths`, called by
 * models/aptai.py:77 through transformers): samples int64 [B] -> out_i64 and/or out_i32 [B]; kernels / strides are HOST
 * arrays of n_layers <= 8 entries. */
int aptai_frame_lengths(const int64_t* samples, int B, const int32_t* kernels, const int32_t* strides, int n_layers,
                        int64_t* out_i64, int32_t* out_i32, void* stream);

/* Force_APTAI cross-attention block (models/force_aptai.py:118-130, models/modules.py:139-153), fp32:
 * phn = emb[phn_ids] + pe; q = Wq frame + bq; k = Wk phn + bk; energy = q k^T - 1000*(ids==0);
 * att_out = LayerNorm(cat[softmax(energy) k, q]) [B][T][256]; att = log_softmax(energy - 1000*(ids==0)) [B][T][60].
 * frame fp32 [B][T][128]; phn_ids int32 [B][60]; emb [vocab][128]; pe [60][128]; Wq/Wk [128][128]. */
int aptai_cross_attention(const float* frame, const int32_t* phn_ids, const float* phn_hidden /* optional [B][60][128]:
                          precomputed phoneme embeddings, then phn_ids is only the 0/non-0 padding mask */,
                          const float* emb, int vocab, const float* pe,
                          const float* wq, const float* bq, const float* wk, const float* bk, const float* ln_w,
                          const float* ln_b, float eps, int B, int T, float* att_out, float* energy, float* att,
                          void* stream);

/* Backward of the block for training (train/train_force_aptai.py: loss.backward() through CrossAttention and the
 * log-softmax alignment matrix).  phn_hidden fp32 [B][60][128] = the phoneme embeddings the forward used (after the
 * positional-encoding dropout).  d_att_out fp32 [B][T][256]; d_att fp32 [B][T][60] or NULL (gradient of att).
 * d_q fp32 [B][T][128]: gradient of the projected queries (dW_q, db_q and d_frame are GEMMs on it); d_k fp32
 * [B][60][128]: gradient of the projected keys, d_ln_w / d_ln_b fp32 [256]: all three ACCUMULATE (atomics). */
int aptai_cross_attention_bwd(const float* frame, const int32_t* phn_ids, const float* phn_hidden, const float* wq,
                              const float* bq, const float* wk, const float* bk, const float* ln_w, float eps, int B,
                              int T, const float* d_att_out, const float* d_att, float* d_q, float* d_k,
                              float* d_ln_w, float* d_ln_b, void* stream);

/* Recurrence of Force_APTAI's bidirectional LSTM (models/modules.py:197-211: nn.LSTM(256, 256, bidirectional,
 * batch_first) over pack_padded_sequence).  gates_in fp32 [B][T][2][1024] = W_ih x_t + b_ih + b_hh per direction
 * (torch gate order i,f,g,o), w_hh_* fp32 [1024][256], lens int32 [B]; out fp32 [B][T][512] (forward | reverse),
 * zero beyond lens[b]. */
int aptai_bilstm_256(const float* gates_in, const float* w_hh_fwd, const float* w_hh_rev, const int32_t* lens, int B,
                     int T, float* out, void* stream);
/* Training (train/train_force_aptai.py: loss.backward() through the nn.LSTM of models/modules.py:197): the same
 * recurrence, also keeping the gate activations gates_act fp32 [B][T][2][1024] (i,f,g,o after sigmoid / tanh) and the
 * cell states cells fp32 [B][T][2][256]; and the backward through time, which turns d_out fp32 [B][T][512] into the
 * gradient of the pre-activation gates d_gates fp32 [2][B][T][1024] (direction-major; padding frames are left
 * untouched: pre-zero it).  dW_ih, dW_hh, the bias gradients and dx are GEMMs on d_gates. */
int aptai_bilstm_256_train(const float* gates_in, const float* w_hh_fwd, const float* w_hh_rev, const int32_t* lens,
                           int B, int T, float* out, float* gates_act, float* cells, void* stream);
int aptai_bilstm_256_bwd(const float* d_out, const float* gates_act, const float* cells, const float* w_hh_fwd,
                         const float* w_hh_rev, const int32_t* lens, int B, int T, float* d_gates, void* stream);

/* masked MSE + cross entropy of APTAI.forward (models/aptai.py:89-102).  out3 = {loss, mse, ce}. */
int aptai_masked_mse_ce(const float* tv_pred, const float* tv_tgt, const float* logits, const int64_t* phn_tgt,
                        int64_t rows, int ntv, int V, float* accum_ws, float* out3, void* stream);

/* ------------------------------------------------------------------ CTC / alignment -------------------------
 * log_softmax over V then CTC loss and gradient w.r.t. the logits (models/w2v2_pr.py:59-81, F.ctc_loss with
 * zero_infinity; models/modules.py:93-116 via per-utterance lengths).  logits fp32 [B][T][V] (ld = V).
 * targets int32 [B][Smax]; entries at s >= target_len[b] are ignored.  log_probs_tbv (optional) fp32 [T][B][V].
 * nll[b] = -log p(target|input) (0 where infeasible and zero_infinity).  grad (optional) fp32 [B][T][V] is
 * d(sum_b scale[b]*nll[b])/d logits, scale may be NULL (= 1).  Workspace: aptai_ctc_workspace_bytes().
 * Smax <= 4095 labels, for this entry and aptai_ctc_viterbi_f32.  Smax selects the kernel:
 *   Smax <= 511: one warp holds the 2 * Smax + 1 DP states in registers (4 / 8 / 16 / 32 per lane);
 *   Smax >  511: the states span one CTA of 32 * ceil((2 * Smax + 1) / 512) threads, 16 per thread (alpha and
 *                beta CTAs per utterance, frame log-sum-exp and gradient as separate warp-per-frame passes).
 * Workspace (bytes, each term rounded up to 256, plus 256), SP = padded state count:
 *   Smax <= 511: 2 * B*T*SP*4 (alpha, beta) + B*T*4 (lse), SP = 32 * (4 | 8 | 16 | 32);
 *   Smax >  511: 2 * B*T*SP*4 (alpha, beta) + B*T*4 (lse) + 2 * B*T*8 (normalisers) + B*8 (nll)
 *                + 2 * B*Smax*4 (same-class chains), SP = 512 * ceil((2 * Smax + 1) / 512).
 * Beyond 4095 labels aptai_ctc_workspace_bytes() returns 0 and the entries return APTAI_ERR_ARG.
 */
size_t aptai_ctc_workspace_bytes(int B, int T, int Smax);
int aptai_logsoftmax_ctc(const float* logits, int B, int T, int V, const int32_t* targets, int Smax,
                         const int32_t* input_len, const int32_t* target_len, int blank, int zero_infinity,
                         float* log_probs_tbv, float* nll, const float* scale, float* grad, void* ws,
                         size_t ws_bytes, void* stream);

/* Extended form used by ForwardSumLoss (models/modules.py:93-116): prepend_blank=1 makes class 0 a virtual column
 * of constant value blank_value (F.pad(..., value=blank_logprob)), class c>=1 is logits column c-1; vocab_len[b]
 * (optional) restricts the log-softmax of utterance b to its first vocab_len[b] classes; loss_sum (optional)
 * receives sum_b scale[b]*nll[b].  grad is always w.r.t. the physical logits columns. */
int aptai_logsoftmax_ctc_ex(const float* logits, int B, int T, int V, int prepend_blank, float blank_value,
                            const int32_t* vocab_len, const int32_t* targets, int Smax, const int32_t* input_len,
                            const int32_t* target_len, int blank, int zero_infinity, float* log_probs_tbv,
                            float* nll, const float* scale, float* loss_sum, float* grad, void* ws,
                            size_t ws_bytes, void* stream);

/* CTC Viterbi forced alignment, bit-exact with torchaudio.functional.forced_align (SURVEY.md Appendix E).
 * log_probs fp32 [B][T][C]; paths int32 [B][T] (frames t >= input_len[b] get -1); scores fp32 [B][T].
 * Smax <= 511: one warp per utterance, back-pointers in shared memory (in the workspace beyond 200 KB);
 * Smax <= 4095: one CTA per utterance, back-pointers (2 bits per state) always in the workspace,
 * B*T*128*ceil((2*Smax+1)/512) bytes; beyond 4095 aptai_viterbi_workspace_bytes() returns 0, the entry
 * APTAI_ERR_ARG. */
size_t aptai_viterbi_workspace_bytes(int B, int T, int Smax);
int aptai_ctc_viterbi_f32(const float* log_probs, const int32_t* targets, const int32_t* input_len,
                          const int32_t* target_len, int B, int T, int C, int Smax, int blank, int32_t* paths,
                          float* scores, int32_t* status, void* ws, size_t ws_bytes, void* stream);

/* greedy CTC collapse on device (argmax -> merge repeats -> drop blank); models/w2v2_pr.py:143-159 next-row. */
int aptai_ctc_greedy(const float* logits, int B, int T, int V, const int32_t* input_len, int blank,
                     int32_t* tokens, int32_t* token_frames, int32_t* ntokens, int maxtok, void* stream);

/* The reference's lexicon-free CTC decode on device: replaces torchaudio.models.decoder.ctc_decoder(lexicon=None,
 * lm=None, nbest=1, beam_size=10, beam_threshold=50, blank_token, sil_token)(logits)[b][0].{tokens, timesteps}
 * (models/w2v2_pr.py:143-159, 209-229, 257-272; utility.py:448-471).  With no LM and max-merge the best beam is the
 * frame-wise argmax path; flashlight's raw path carries a leading and a trailing `sil` entry (T + 2 entries), which
 * torchaudio's _get_tokens / _get_timesteps (_ctc_decoder.py:248-262) collapse together with the frame labels:
 * tokens int32 [B][maxtok] start / end with `sil`, timesteps int32 [B][maxtok] = frame + 1.  maxtok >= T + 2.
 * input_len NULL = decode all T frames, as the reference does (it passes no lengths). */
int aptai_ctc_decode_ref(const float* logits, int B, int T, int V, const int32_t* input_len, int blank, int sil,
                         int32_t* tokens, int32_t* timesteps, int32_t* ntokens, int maxtok, void* stream);


/* ================================================================== accuracy mode ("f32x3") ==================
 * Every contraction of the path as THREE bf16 tensor-core products on hi/lo operand pairs (x = x_hi + x_lo,
 * w = w_hi + w_lo; x.w ~= x_hi.w_hi + x_lo.w_hi + x_hi.w_lo, ~2^-17 relative), fp32 everywhere else: the mode in
 * which the north-star tolerances (phoneme argmax >= 99.9 %, CTC-type losses 1e-3) hold against the fp32
 * reference.  The GEMMs are aptai_gemm_bf16 on operands laid out A' = [hi | lo | hi] (K tripled),
 * W' = [hi | hi | lo]; these entry points are the streaming kernels around them (csrc/accurate.cu). */

/* fp32 [rows][cols] (row stride ld_in) * scale -> bf16 [rows][3*cols]: [hi|lo|hi] (weight_layout 0) or [hi|hi|lo] */
int aptai_split3_bf16(const float* x, int64_t rows, int cols, int64_t ld_in, int weight_layout, float scale,
                      void* out_bf16, void* stream);
/* per row: (LayerNorm, exact two-pass fp32 statistics; HF:431,600-602,639,645,692,792 and the conv LayerNorms
 * HF:288-299) -> (erf-GELU) -> fp32 [rows][cols] and / or split bf16 [rows][3*cols].  cols in {256, 512, 768, 1024}. */
int aptai_rowop_split3(const float* x, int64_t rows, int cols, const float* gamma, const float* beta, float eps,
                       int norm, int gelu, float* out_f32, void* out_split3, void* stream);
/* conv layer 0 + norm + GELU (HF:281-323) in fp32 with split bf16 output [B][T0][3*512]; norm as in
 * aptai_conv0_norm_gelu, stats_ws likewise (GroupNorm only). */
int aptai_conv0_accurate(const float* wav, int B, int64_t L, const float* w, const float* bias, const float* gamma,
                         const float* beta, int norm, float eps, void* out_split3, int T0, float* stats_ws,
                         void* stream);
/* out = res + gelu(x): tail of the positional conv embedding (HF:360-368 + residual add) */
int aptai_gelu_add_f32(const float* x, const float* res, int64_t n, float* out, void* stream);
/* fp32 [segs][rows][cols] -> zero-haloed bf16 hi and lo copies [segs][rows + 2*halo][cols] */
int aptai_cast_pad_split(const float* x, int segs, int rows, int cols, int halo, void* hi_bf16, void* lo_bf16,
                         void* stream);
/* weight-norm fold of the positional conv (HF:336-358) with hi / lo bf16 outputs [H][taps*cpad] */
int aptai_posconv_fold_split(const float* g, const float* v, int H, int cin, int taps, int cpad, void* w_hi, void* w_lo,
                             float* norm_ws, void* stream);
/* softmax(q k^T + key-length mask) v on fp32 operands (HF:500-549): qkv fp32 [B*T][3*heads*64] (q pre-scaled),
 * ctx fp32 [B*T][heads*64] */
int aptai_attention_fwd_f32(const float* qkv, float* ctx, const int32_t* key_len, int B, int T, int heads,
                            void* stream);

/* ================================================================== training step (backward + optimizer) =====
 * The reference trains with torch autograd (train/train_aptai.py:431-443: zero_grad / loss.backward() /
 * optimizer.step()); these entry points are the kernels that autograd would otherwise dispatch for the hot path.
 * dgrad of a Linear is aptai_gemm_bf16 on the transposed weight (act=2 multiplies by gelu'(aux)).
 */

/* attention forward that also stores the log2-domain log-sum-exp per query row, lse fp32 [B][heads][T] */
int aptai_attention_fwd_lse(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T, int heads,
                            void* stream);
/* D[b][h][t] = sum_d d_ctx * ctx  (bf16 [B*T][heads*64] inputs), the softmax-backward row term */
int aptai_attention_bwd_dot(const void* d_ctx, const void* ctx, int B, int T, int heads, float* D, void* stream);
/* same, and zero_f32 (fp32 [B*T][heads*64], may be NULL) is cleared in the same pass: the dQ accumulator of the
 * aptai_attention_bwd launch that follows, without a memset launch of its own */
int aptai_attention_bwd_dot_zero(const void* d_ctx, const void* ctx, int B, int T, int heads, float* D, float* zero_f32,
                                 void* stream);
/* attention backward (autograd of HF:500-549).  qkv bf16 [B*T][3H] (q pre-scaled), d_ctx bf16 [B*T][H];
 * writes dk, dv into the k / v blocks of dqkv (bf16 [B*T][3H]) and ACCUMULATES dq (w.r.t. the pre-scaled q) into
 * dq32 fp32 [B*T][H], which the caller zeroes before and converts with aptai_scale_cast_bf16 afterwards. */
int aptai_attention_bwd(const void* qkv, const void* d_ctx, const float* lse, const float* dvec,
                        const int32_t* key_len, int B, int T, int heads, float* dq32, void* dqkv, void* stream);
/* Training-mode variants with dropout on the attention probabilities (HF:461): P is masked and rescaled by 1/(1-p)
 * where it multiplies V, with a counter-based mask of (seed, utterance, head, query, key) that the backward regenerates;
 * aptai_attention_dropout_mask materialises keep/(1-p) as fp32 [B][heads][T][T] (test replay). */
int aptai_attention_fwd_dropout(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T, int heads,
                                float drop_p, uint64_t drop_seed, void* stream);
int aptai_attention_bwd_dropout(const void* qkv, const void* d_ctx, const float* lse, const float* dvec,
                                const int32_t* key_len, int B, int T, int heads, float* dq32, void* dqkv, float drop_p,
                                uint64_t drop_seed, void* stream);
int aptai_attention_dropout_mask(int B, int T, int heads, float drop_p, uint64_t drop_seed, float* out, void* stream);
/* out_bf16[r][0..cols) (row pitch ldo) = scale * x[r][0..cols) */
int aptai_scale_cast_bf16(const float* x, int64_t rows, int cols, float scale, void* out_bf16, int64_t ldo,
                          void* stream);

/* weight gradient of a Linear: dw[n][k] += scale * sum_m dy[m][n] * x[m][k]  (dy bf16 [M][N] pitch dy_ld,
 * x bf16 [M][K] pitch x_ld, dw fp32 pitch dw_ld; split over frames, fp32 reductions) */
int aptai_gemm_wgrad_bf16(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, int64_t M, int N, int K,
                          float scale, float* dw, int64_t dw_ld, void* stream);
/* weight gradient of the grouped positional conv (HF:329-368) in the folded layout of aptai_posconv_fold:
 * dw_folded[o][tap*64 + c] += sum_{b,t} dy[b][t][o] * x_pad[b][t + tap][g(o)*gw + c]
 * dy bf16 [B][T][H], x_pad bf16 [B][T + taps][H] (the forward's aptai_cast_pad_bf16 output). */
int aptai_posconv_wgrad_bf16(const void* dy, const void* x_pad, int B, int T, int H, int groups, int taps,
                             float* dw_folded, void* stream);
/* weight gradient of a strided conv layer of the feature encoder (HF:254-323) in the forward GEMM's tap-major layout:
 * dw[o][tap*C + c] += sum_{b,t} dz[b][t][o] * x[b][t*stride + tap][c];  dz bf16 [B][T_out][C], x bf16 [B][T_in][C]
 * (row T_in of the last utterance may be touched by the strided TMA view: keep the forward's slack rows). */
int aptai_conv_wgrad_bf16(const void* dz, const void* x, int B, int T_out, int T_in, int C, int ktaps, int stride,
                          float* dw_tapmajor, void* stream);
/* conv feature encoder, 'layer' norm variant, training path: y = GELU(LayerNorm_512(z)) as a separate streaming kernel
 * (forward), and its backward dz = LN'(dy * GELU'(LN(z))) with dgamma/dbeta accumulated.  dy fp32 with a row map
 * (logical row r of segment s at physical row s*dy_seg_pitch + r).  For conv layer 0 pass z = NULL and wav / w0t
 * ([10][512] transposed weight) / bias0: z is recomputed from the waveform (frame t reads samples 5t .. 5t+9; wav_ld,
 * the row pitch, is also the samples per utterance: 5*(dy_rows_per_seg-1)+10 <= wav_ld, else APTAI_ERR_ARG). */
int aptai_ln_gelu_fwd_512(const void* z_bf16, int64_t rows, const float* gamma, const float* beta, float eps,
                          void* y_bf16, void* stream);
int aptai_ln_gelu_bwd_512(const float* dy, int64_t dy_rows_per_seg, int64_t dy_seg_pitch, const void* z_bf16,
                          const float* wav, int64_t wav_ld, const float* w0t, const float* bias0, int64_t rows,
                          const float* gamma, const float* beta, float eps, void* dz_bf16, float* dgamma, float* dbeta,
                          void* stream);
/* 'group' norm variant (base models, HF:308-323).  Layers 1..6 (no norm, no bias): dz = dy * GELU'(z).  Conv layer 0 with
 * GroupNorm over time: affine fp32 [B][512][2] = {gamma*rstd, (bias-mean)*gamma*rstd + beta} and norm_stats fp32
 * [B][512][2] = {mean - bias, rstd} as produced by the forward (aptai_conv0_norm_gelu's stats_ws), sums fp32
 * [B][512][2] receives {sum_t g, sum_t g*xhat} (dbeta / dgamma per utterance), dz bf16 [B*T0][512]. */
int aptai_gelu_bwd_rows_512(const float* dy, int64_t dy_rows_per_seg, int64_t dy_seg_pitch, const void* z_bf16,
                            int64_t rows, void* dz_bf16, void* stream);
int aptai_conv0_groupnorm_bwd(const float* dy, int64_t dy_seg_pitch, const float* wav, int B, int64_t L, int T0,
                              const float* w0, const float* affine, const float* norm_stats, float* sums, void* dz_bf16,
                              void* stream);
/* X[b*T0 + t][0..63] = wav[b][5t .. 5t+9], 0-padded, bf16: B operand of conv-0's weight-gradient GEMM */
int aptai_conv0_im2col_bf16(const float* wav, int B, int64_t L, int64_t T0, void* x_bf16, void* stream);
/* weight-norm backward (torch parametrizations.weight_norm, dim=2): dg[taps] += , dv[H][cin][taps] += from the
 * folded dW.  ws: 2*taps doubles. */
int aptai_posconv_weightnorm_bwd(const float* dw_folded, const float* g, const float* v, int H, int cin, int taps,
                                 int cpad, float* dg, float* dv, void* ws, void* stream);

/* out[i] = dy[i] * gelu'(pre[i]) (backward of the positional conv's GELU, HF:366); pre bf16, n % 4 == 0 */
int aptai_gelu_bwd(const float* dy, const void* pre_bf16, int64_t n, float* out, void* stream);

/* out[n] += scale * sum_m x[m][n]  (bias gradients); x bf16 (x_bf16=1) or fp32, row pitch ld */
int aptai_colsum(const void* x, int x_bf16, int64_t M, int N, int64_t ld, float scale, float* out, void* stream);

/* LayerNorm backward (HF:431,600-602,639,645,692,792).  x = the forward's input (fp32), dy fp32; dx = dres + LN'(dy)
 * written fp32 and/or bf16; dgamma/dbeta (optional, both or none) are accumulated (+=). */
int aptai_layernorm_bwd(const float* dy, const float* x, int64_t rows, int cols, const float* gamma, float eps,
                        const float* dres, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta, void* stream);
/* same, and dcolsum[c] += sum over rows of the output gradient dx[row][c] (fp32, before the 16-bit rounding): the bias
 * gradient of the Linear that wrote the residual stream this LayerNorm reads (out-proj / FFN2), without the colsum
 * launch that would re-read dx */
int aptai_layernorm_bwd_colsum(const float* dy, const float* x, int64_t rows, int cols, const float* gamma, float eps,
                               const float* dres, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta,
                               float* dcolsum, void* stream);

/* backward of aptai_heads: dh = act_a'(h) (dA Wa) + act_b'(h) (dB Wb) (optional), dW += dOut^T act(h), db += colsum */
int aptai_heads_bwd(const float* h, int64_t rows, int H, const float* da, int na, const float* wa, int act_a,
                    float* dwa, float* dba, const float* db, int nb, const float* wb, int act_b, float* dwb,
                    float* dbb, float* dh, void* stream);

/* backward of aptai_masked_mse_ce w.r.t. tv_pred and logits; accum_ws is the forward's workspace (counts),
 * grad_scale (optional device scalar) multiplies both. */
int aptai_masked_mse_ce_bwd(const float* tv_pred, const float* tv_tgt, const float* logits, const int64_t* phn_tgt,
                            int64_t rows, int ntv, int V, const float* accum_ws, const float* grad_scale, float* d_tv,
                            float* d_logits, void* stream);

/* Kernel-operand copies of the fp32 master weights in one launch (after load_state_dict / every optimizer step):
 * per table entry dst[r][c] = bf16(scale*src[r][c]) (row pitch dst_ld), dst_t[c][r] = bf16(scale_t*src[r][c]) (row
 * pitch dst_t_ld), dst_f32 = scale*src; any destination may be NULL.  tile0 = index of the entry's first 64x64
 * tile, tiles_x = ceil(cols/64); total_tiles = sum over entries of tiles_x * ceil(rows/64).  The table lives in device memory. */
typedef struct aptai_prep_entry {
  const float* src;
  void* dst;
  void* dst_t;
  float* dst_f32;
  int32_t rows, cols, dst_ld, dst_t_ld;
  float scale, scale_t;
  int32_t tile0, tiles_x;
} aptai_prep_entry;
int aptai_prepare_weights(const void* entries_dev, int n_entries, int total_tiles, void* stream);
/* same with every 16-bit destination of the launch written as IEEE fp16 (half_fmt 1) instead of bf16 (0) */
int aptai_prepare_weights_fmt(const void* entries_dev, int n_entries, int total_tiles, int half_fmt, void* stream);

/* Inverted dropout, counter-based (HF:434,546,570,603-607,647-653,694,766; models/aptai.py:44,52; w2v2_pr.py:56):
 * out[i] = residual[i] + keep(seed, i) * x[i] / (1 - p), keep = hash(seed, i) >= p.  x fp32 or bf16 (x_bf16), residual
 * optional fp32, outputs fp32 and/or bf16 (may alias x).  The backward of a site is the same call on the gradient
 * with the same (p, seed). */
int aptai_dropout(const void* x, int x_bf16, const float* residual, int64_t n, float p, uint64_t seed, float* out_f32,
                  void* out_bf16, void* stream);

/* torch.optim.Adam step (train/train_aptai.py:350-356) over a table of parameter tensors in one launch.
 * params_dev: device array of fp32 pointers; grad_offsets / state_offsets / numel: element offset of each tensor in
 * the flat grad buffer, in the flat exp_avg / exp_avg_sq buffers, and its size;
 * chunks_dev: {int32 tensor, int32 pad, int64 start}[n_chunks]. */
int aptai_adam_step(void* const* params_dev, const int64_t* grad_offsets_dev, const int64_t* state_offsets_dev,
                    const int64_t* numel_dev, const void* chunks_dev, int n_chunks, int chunk_elems, const float* grad, float* exp_avg,
                    float* exp_avg_sq, float lr, float beta1, float beta2, float eps, float weight_decay, int step,
                    float grad_scale, void* stream);

/* ================================================================== callers' data formats (SURVEY.md 8f rows 3, 4) ==
 * Input side. */
/* ragged -> padded batch (torch.nn.utils.rnn.pad_sequence(batch_first=True) of train/train_aptai.py:268-332):
 * flat = the B sequences back to back (4- or 8-byte elements), offsets int64 [B+1]; out [B][Lmax], tail = pad value */
int aptai_collate_pad(const void* flat, int elem_bytes, const int64_t* offsets, int B, int64_t Lmax,
                      const void* pad_value_host, void* out, void* stream);
/* polyphase FIR of torchaudio.functional.resample (data/dataset_hprc.py:68-72): kernel fp32 [nw][2*width+orig] from
 * _get_sinc_resample_kernel (orig, nw already divided by their gcd); y[b][j] for j < ceil(nw*in_len[b]/orig), 0 after */
int aptai_resample_fir(const float* x, const int64_t* in_len, int B, int64_t in_ld, const float* kernel, int orig,
                       int nw, int width, float* y, int64_t out_ld, void* stream);
/* interpolate_signal (data/dataset_hprc.py:2307-2313): scipy interp1d(arange(n), sig, 'linear', axis=0) evaluated at
 * linspace(0, n-1, m); sig fp64 [n][C] -> out fp64 [m][C], bit-exact.  per_channel=1: each column as a 1-D call (the
 * reference's pattern, dataset_hprc.py:2370: scipy then uses numpy.interp's formula); 0: scipy's N-D formula */
int aptai_interp_linear_f64(const double* sig, int n, int C, int m, int per_channel, double* out, void* stream);
/* Output side. */
/* phn_frames2dur / phn_frame_id2phn (utility.py:539-566): run-length segments of frame labels int64 [B][T] over the
 * first lens[b] frames: seg_start/seg_end (frames, end exclusive), seg_phn, nseg[b] (may exceed max_seg: truncated) */
int aptai_frames_to_segments(const int64_t* frames, const int32_t* lens, int B, int T, int32_t* seg_start,
                             int32_t* seg_end, int64_t* seg_phn, int32_t* nseg, int max_seg, void* stream);
/* tvs_metric_rmse / tvs_metric_ppc (utility.py:393-444) per utterance and channel over the first lens[b] frames:
 * gt, pred fp32 [B][T][C] -> rmse, pcc fp64 [B][C] (RMSE bit-exact with the reference's sequential fp64 sum) */
int aptai_tv_metrics(const float* gt, const float* pred, const int32_t* lens, int B, int T, int C, double* rmse,
                     double* pcc, void* stream);
/* get_stats counters (utility.py:589-611): boundaries fp64 [B][maxn] (seconds) with counts ny/nyhat;
 * counters int32 [B][4] = {precision_counter, recall_counter, len(yhat), len(y)} */
int aptai_boundary_stats(const double* y, const int32_t* ny, const double* yhat, const int32_t* nyhat, int B, int maxn,
                         double tolerance, int32_t* counters, void* stream);
/* evaluate_overlap (utility.py:614-622): hits_counts uint64 [2] = {#equal frames, #frames} over the valid frames */
int aptai_frame_overlap(const int64_t* a, const int64_t* b, const int32_t* lens, int B, int T, uint64_t* hits_counts,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* APTAI_B200_H */
