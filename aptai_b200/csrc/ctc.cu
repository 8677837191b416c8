// Alignment stage: fused log-softmax + CTC loss/gradient, CTC Viterbi forced alignment, greedy CTC collapse.
// One utterance per CTA; the 2S+1 CTC states live in registers, NI consecutive states per lane, so the s-1 / s-2
// neighbours are in-thread except at the lane boundary (two warp shuffles per time step).  Transcripts of more than
// 511 labels take the CTA-wide kernels below ("long transcripts"), up to 4095 labels.
//
// Reference call sites: models/w2v2_pr.py:59-81 (log_softmax + F.ctc_loss, zero_infinity, blank 0),
// models/modules.py:93-116 (ForwardSumLoss: per-utterance vocabulary width, prepended blank column),
// SURVEY.md Appendix E (Viterbi rule of torchaudio.functional.forced_align).
#include "common.h"
#include "ptx.cuh"

#include <math.h>

#include <algorithm>

namespace aptai {

constexpr float NEG_INF = -INFINITY;
constexpr int CTC_THREADS = 128;

struct CtcArgs {
  const float* logits;   // [B][T][V]
  int B, T, V;           // V = physical columns
  int prepend_blank;     // 1: class 0 is a virtual column of value blank_value, class c>=1 is column c-1
  float blank_value;
  const int* targets;    // [B][Smax]
  int Smax;
  const int* input_len;
  const int* target_len;
  const int* vocab_len;  // optional per-utterance number of classes (<= Veff)
  int blank;
  int zero_infinity;
  float* log_probs_tbv;  // optional [T][B][Veff]
  float* nll;            // [B]
  const float* scale;    // optional [B]
  float* grad;           // optional [B][T][V]
  float* alpha;          // ws [B][T][SP]
  float* beta;           // ws [B][T][SP]
  float* lse;            // ws [B][T]
  int SP;                // padded state count = 32*NI
};

__device__ __forceinline__ float logit_at(const CtcArgs& a, const float* row, int c) {
  if (a.prepend_blank) return c == 0 ? a.blank_value : row[c - 1];
  return row[c];
}

__device__ __forceinline__ float lse3(float x, float y, float z) {
  float m = fmaxf(x, fmaxf(y, z));
  if (m == NEG_INF) m = 0.f;
  return logf(expf(x - m) + expf(y - m) + expf(z - m)) + m;
}

template <int NI>
__global__ void __launch_bounds__(CTC_THREADS)
ctc_kernel(const CtcArgs a) {
  extern __shared__ float sm[];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Veff = a.V + (a.prepend_blank ? 1 : 0);
  const int Vb = a.vocab_len ? min(a.vocab_len[b], Veff) : Veff;
  int Tb = min(a.input_len[b], a.T);
  int S = min(a.target_len[b], a.Smax);
  const int NS = 2 * S + 1;
  const int SP = 32 * NI;
  const float* lg = a.logits + static_cast<long long>(b) * a.T * a.V;
  float* lse = a.lse + static_cast<long long>(b) * a.T;
  float* alpha = a.alpha + static_cast<long long>(b) * a.T * SP;
  float* beta = a.beta + static_cast<long long>(b) * a.T * SP;
  const int* tg = a.targets + static_cast<long long>(b) * a.Smax;

  // smem: labels per state [SP] | next-same-label chain [SP/2] | per-warp scratch (4 x (SP + Veff))
  int* s_lab = reinterpret_cast<int*>(sm);
  int* s_nxt = s_lab + SP;
  int* s_first = s_nxt + SP / 2;
  float* s_scr = reinterpret_cast<float*>(s_first + SP / 2);

  // ---- phase 0: log-sum-exp per frame (all T frames: the reference returns log_softmax for padded frames too)
  for (int t = tid; t < a.T; t += CTC_THREADS) {
    const float* row = lg + static_cast<long long>(t) * a.V;
    float m = NEG_INF;
    for (int c = 0; c < Vb; ++c) m = fmaxf(m, logit_at(a, row, c));
    float s = 0.f;
    for (int c = 0; c < Vb; ++c) s += expf(logit_at(a, row, c) - m);
    const float l = logf(s) + m;
    lse[t] = l;
    if (a.log_probs_tbv) {
      float* o = a.log_probs_tbv + (static_cast<long long>(t) * a.B + b) * Veff;
      for (int c = 0; c < Veff; ++c) o[c] = c < Vb ? logit_at(a, row, c) - l : NEG_INF;
    }
  }
  for (int s = tid; s < SP; s += CTC_THREADS) s_lab[s] = (s & 1) ? (s / 2 < S ? tg[s / 2] : a.blank) : a.blank;
  for (int j = tid; j < SP / 2; j += CTC_THREADS) {
    int nx = -1, first = 1;
    if (j < S) {
      const int l = tg[j];
      for (int k = j + 1; k < S; ++k)
        if (tg[k] == l) { nx = k; break; }
      for (int k = 0; k < j; ++k)
        if (tg[k] == l) { first = 0; break; }
    }
    s_nxt[j] = nx;
    s_first[j] = first;
  }
  __syncthreads();

  // degenerate: no frames -> loss is inf (or 0 with zero_infinity), gradient 0
  const bool empty = Tb <= 0;

  // ---- phase 1: alpha (warp 0) and beta (warp 1) recursions
  if (!empty && warp < 2) {
    int lab[NI];
    bool skip_ok[NI];   // alpha: may come from s-2 ; beta: may go to s+2 (same condition shifted)
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int s = lane * NI + i;
      lab[i] = s_lab[s];
      if (warp == 0)
        skip_ok[i] = (s & 1) && s >= 3 && s < NS && s_lab[s] != s_lab[s - 2];
      else
        skip_ok[i] = (s & 1) && s + 2 < NS && s_lab[s] != s_lab[s + 2];
    }
    float cur[NI];
    if (warp == 0) {
      const float* row = lg;
      const float l0 = lse[0];
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int s = lane * NI + i;
        cur[i] = (s < 2 && s < NS) ? logit_at(a, row, lab[i]) - l0 : NEG_INF;
      }
#pragma unroll
      for (int i = 0; i < NI; ++i) alpha[lane * NI + i] = cur[i];
      for (int t = 1; t < Tb; ++t) {
        const float* rw = lg + static_cast<long long>(t) * a.V;
        const float lt = lse[t];
        float lp[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) lp[i] = logit_at(a, rw, lab[i]) - lt;
        float p1 = __shfl_up_sync(0xffffffffu, cur[NI - 1], 1);
        float p2 = __shfl_up_sync(0xffffffffu, cur[NI - 2], 1);
        if (lane == 0) { p1 = NEG_INF; p2 = NEG_INF; }
        float nw[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          const float x1 = i >= 1 ? cur[i - 1] : p1;
          const float x2r = i >= 2 ? cur[i - 2] : (i == 1 ? p1 : p2);
          const float x2 = skip_ok[i] ? x2r : NEG_INF;
          const int s = lane * NI + i;
          nw[i] = s < NS ? lse3(cur[i], x1, x2) + lp[i] : NEG_INF;
        }
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          cur[i] = nw[i];
          alpha[static_cast<long long>(t) * SP + lane * NI + i] = nw[i];
        }
      }
    } else {
      const int t1 = Tb - 1;
      const float* row = lg + static_cast<long long>(t1) * a.V;
      const float l0 = lse[t1];
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int s = lane * NI + i;
        cur[i] = (s < NS && s >= NS - 2) ? logit_at(a, row, lab[i]) - l0 : NEG_INF;
      }
#pragma unroll
      for (int i = 0; i < NI; ++i) beta[static_cast<long long>(t1) * SP + lane * NI + i] = cur[i];
      for (int t = t1 - 1; t >= 0; --t) {
        const float* rw = lg + static_cast<long long>(t) * a.V;
        const float lt = lse[t];
        float lp[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) lp[i] = logit_at(a, rw, lab[i]) - lt;
        float n1 = __shfl_down_sync(0xffffffffu, cur[0], 1);
        float n2 = __shfl_down_sync(0xffffffffu, cur[1], 1);
        if (lane == 31) { n1 = NEG_INF; n2 = NEG_INF; }
        float nw[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          const float x1 = i + 1 < NI ? cur[i + 1] : n1;
          const float x2r = i + 2 < NI ? cur[i + 2] : (i + 2 == NI ? n1 : n2);
          const float x2 = skip_ok[i] ? x2r : NEG_INF;
          const int s = lane * NI + i;
          nw[i] = s < NS ? lse3(cur[i], x1, x2) + lp[i] : NEG_INF;
        }
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          cur[i] = nw[i];
          beta[static_cast<long long>(t) * SP + lane * NI + i] = nw[i];
        }
      }
    }
  }
  __syncthreads();

  // ---- loss
  float nll = INFINITY;
  if (!empty) {
    const float* al = alpha + static_cast<long long>(Tb - 1) * SP;
    const float a1 = al[NS - 1];
    const float a2 = NS >= 2 ? al[NS - 2] : NEG_INF;
    float m = fmaxf(a1, a2);
    if (m == NEG_INF) m = 0.f;
    nll = -(logf(expf(a1 - m) + expf(a2 - m)) + m);
  }
  const bool infeasible = !(nll < INFINITY);   // inf or NaN
  if (tid == 0) a.nll[b] = (infeasible && a.zero_infinity) ? 0.f : nll;
  if (!a.grad) return;

  // ---- phase 2: gradient w.r.t. the logits, one warp per frame
  const float sc = a.scale ? a.scale[b] : 1.f;
  float* scr_ab = s_scr + warp * (SP + Veff);
  float* scr_cls = scr_ab + SP;
  float* gb = a.grad + static_cast<long long>(b) * a.T * a.V;
  for (int t = warp; t < a.T; t += CTC_THREADS / 32) {
    float* grow = gb + static_cast<long long>(t) * a.V;
    if (t >= Tb || (infeasible && a.zero_infinity)) {
      for (int c = lane; c < a.V; c += 32) grow[c] = 0.f;
      continue;
    }
    const float* al = alpha + static_cast<long long>(t) * SP;
    const float* be = beta + static_cast<long long>(t) * SP;
    float m = NEG_INF;
    for (int s = lane; s < SP; s += 32) {
      const float v = s < NS ? al[s] + be[s] : NEG_INF;
      scr_ab[s] = v;
      m = fmaxf(m, v);
    }
    for (int c = lane; c < Veff; c += 32) scr_cls[c] = 0.f;
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (m == NEG_INF) m = 0.f;
    __syncwarp();
    // blank states (even s): lane-strided sum + warp reduction
    float bs = 0.f;
    for (int s = 2 * lane; s < NS; s += 64) bs += expf(scr_ab[s] - m);
    for (int o = 16; o; o >>= 1) bs += __shfl_xor_sync(0xffffffffu, bs, o);
    // label states (odd s): the first occurrence of each label walks its chain (deterministic order)
    for (int j = lane; j < S; j += 32) {
      if (!s_first[j]) continue;
      float acc = 0.f;
      for (int k = j; k >= 0; k = s_nxt[k]) acc += expf(scr_ab[2 * k + 1] - m);
      const int cls = tg[j];
      if (cls == a.blank) continue;     // a blank inside the targets is folded into bs below via class check
      scr_cls[cls] = acc;
    }
    __syncwarp();
    const float* rw = lg + static_cast<long long>(t) * a.V;
    const float lt = lse[t];
    for (int c = lane; c < Veff; c += 32) {
      const int col = a.prepend_blank ? c - 1 : c;
      if (col < 0) continue;
      float g = 0.f;
      if (c < Vb) {
        const float lp = logit_at(a, rw, c) - lt;
        const float occ = (c == a.blank) ? bs : scr_cls[c];
        // (exp(lp) - exp(log(occ) + m + nll - lp)) : ATen ctc_loss_backward formula
        const float post = occ > 0.f ? expf(logf(occ) + m + nll - lp) : 0.f;
        g = (expf(lp) - post) * sc;
      }
      grow[col] = g;
    }
    __syncwarp();
  }
}

__global__ void ctc_reduce_kernel(const float* __restrict__ nll, const float* __restrict__ scale, int B,
                                  float* __restrict__ out) {
  // deterministic serial sum: out[0] = sum_b scale[b] * nll[b]
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += (scale ? scale[b] : 1.f) * nll[b];
    out[0] = s;
  }
}

// ------------------------------------------------------------------------------------------------ Viterbi
struct VitArgs {
  const float* lp;      // [B][T][C]
  const int* targets;   // [B][Smax]
  const int* input_len;
  const int* target_len;
  int B, T, C, Smax, blank;
  int* paths;           // [B][T]
  float* scores;        // [B][T]
  int* status;          // [B] 0 ok, 1 infeasible (T < L + R)
  void* bp_global;      // ws [B][T][32] back-pointer words (used when they do not fit in shared memory)
  int bp_in_smem;
};

// back-pointer word of one lane and one frame: 2 bits per state, NI states
template <int NI> struct BpWord { typedef uint16_t type; };
template <> struct BpWord<16> { typedef uint32_t type; };
template <> struct BpWord<32> { typedef uint64_t type; };

template <int NI>
__global__ void __launch_bounds__(32)
viterbi_kernel(const VitArgs a) {
  typedef typename BpWord<NI>::type bp_t;
  extern __shared__ __align__(8) unsigned char bp_sm_raw[];
  bp_t* bp_sm = reinterpret_cast<bp_t*>(bp_sm_raw);
  __shared__ int s_lab[32 * NI];
  const int b = blockIdx.x;
  const int lane = threadIdx.x;
  const int Tb = min(a.input_len[b], a.T);
  const int L = min(a.target_len[b], a.Smax);
  const int NS = 2 * L + 1;
  const int* tg = a.targets + static_cast<long long>(b) * a.Smax;
  const float* lp = a.lp + static_cast<long long>(b) * a.T * a.C;
  int* path = a.paths + static_cast<long long>(b) * a.T;
  float* score = a.scores ? a.scores + static_cast<long long>(b) * a.T : nullptr;
  bp_t* bp = a.bp_in_smem ? bp_sm : reinterpret_cast<bp_t*>(a.bp_global) + static_cast<long long>(b) * a.T * 32;

  for (int t = Tb + lane; t < a.T; t += 32) {
    path[t] = -1;
    if (score) score[t] = 0.f;
  }
  int R = 0;
  for (int j = 1 + lane; j < L; j += 32) R += (tg[j] == tg[j - 1]);
  for (int o = 16; o; o >>= 1) R += __shfl_xor_sync(0xffffffffu, R, o);
  if (Tb <= 0 || Tb < L + R) {
    if (lane == 0 && a.status) a.status[b] = 1;
    for (int t = lane; t < Tb; t += 32) {
      path[t] = -1;
      if (score) score[t] = 0.f;
    }
    return;
  }
  if (lane == 0 && a.status) a.status[b] = 0;
  for (int s = lane; s < 32 * NI; s += 32) s_lab[s] = (s & 1) ? (s / 2 < L ? tg[s / 2] : a.blank) : a.blank;
  __syncwarp();

  int lab[NI];
  bool skip_ok[NI];
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int s = lane * NI + i;
    lab[i] = s_lab[s];
    skip_ok[i] = (s & 1) && s >= 2 && s < NS && s_lab[s] != s_lab[s - 2];
  }
  const int start = (Tb - (L + R) > 0) ? 0 : 1;
  const int end = NS == 1 ? 1 : 2;
  float cur[NI];
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int s = lane * NI + i;
    cur[i] = (s >= start && s < end) ? lp[lab[i]] : NEG_INF;
  }
  for (int t = 1; t < Tb; ++t) {
    const float* row = lp + static_cast<long long>(t) * a.C;
    float e[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) e[i] = row[lab[i]];
    float p1 = __shfl_up_sync(0xffffffffu, cur[NI - 1], 1);
    float p2 = __shfl_up_sync(0xffffffffu, cur[NI - 2], 1);
    if (lane == 0) { p1 = NEG_INF; p2 = NEG_INF; }
    float nw[NI];
    bp_t code = 0;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const float x0 = cur[i];
      const float x1 = i >= 1 ? cur[i - 1] : p1;
      const float x2r = i >= 2 ? cur[i - 2] : (i == 1 ? p1 : p2);
      const float x2 = skip_ok[i] ? x2r : NEG_INF;
      float best;
      uint32_t c;
      if (x2 > x1 && x2 > x0) { best = x2; c = 2; }
      else if (x1 > x0 && x1 > x2) { best = x1; c = 1; }
      else { best = x0; c = 0; }
      const int s = lane * NI + i;
      nw[i] = (s < NS && best != NEG_INF) ? __fadd_rn(best, e[i]) : NEG_INF;
      code |= static_cast<bp_t>(c) << (2 * i);
    }
#pragma unroll
    for (int i = 0; i < NI; ++i) cur[i] = nw[i];
    bp[static_cast<long long>(t) * 32 + lane] = code;
  }
  // final state: S-1 if alpha[S-1] > alpha[S-2] (strict) else S-2 ; S == 1 -> 0
  int s_fin = 0;
  {
    const int sA = NS - 1, sB = NS - 2;
    float vA = NEG_INF, vB = NEG_INF;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int s = lane * NI + i;
      if (s == sA) vA = cur[i];
      if (s == sB) vB = cur[i];
    }
    vA = __shfl_sync(0xffffffffu, vA, sA / NI);
    if (NS >= 2) vB = __shfl_sync(0xffffffffu, vB, sB / NI);
    s_fin = NS == 1 ? 0 : (vA > vB ? sA : sB);
  }
  __syncwarp();
  if (lane == 0) {
    int s = s_fin;
    for (int t = Tb - 1; t >= 0; --t) {
      const int l = s_lab[s];
      path[t] = l;
      if (score) score[t] = lp[static_cast<long long>(t) * a.C + l];
      if (t > 0) {
        const bp_t code = bp[static_cast<long long>(t) * 32 + s / NI];
        s -= static_cast<int>((code >> (2 * (s % NI))) & 3);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ greedy CTC
// sil < 0: plain greedy collapse (argmax -> merge repeats -> drop blanks), token_frames = first frame of each token.
// sil >= 0: the reference's decoder output (models/w2v2_pr.py:143-159 -> torchaudio _ctc_decoder.py:248-262 over
// flashlight's raw path): the raw path is [sil] + per-frame argmax + [sil] (T+2 entries: the root hypothesis of
// decodeBegin and the closing one of decodeEnd), merged / blank-filtered over those T+2 entries, and `timesteps`
// index into the raw path (frame + 1).
__global__ void __launch_bounds__(32)
ctc_greedy_kernel(const float* __restrict__ logits, int T, int V, const int* __restrict__ input_len, int blank, int sil,
                  int* __restrict__ tokens, int* __restrict__ token_frames, int* __restrict__ ntokens, int maxtok) {
  const int b = blockIdx.x, lane = threadIdx.x;
  const int Tb = input_len ? min(input_len[b], T) : T;
  const float* lg = logits + static_cast<long long>(b) * T * V;
  int* tk = tokens + static_cast<long long>(b) * maxtok;
  int* tf = token_frames ? token_frames + static_cast<long long>(b) * maxtok : nullptr;
  const int off = sil >= 0 ? 1 : 0;
  int prev = sil >= 0 ? sil : -1, count = 0;
  if (sil >= 0 && sil != blank) {
    if (lane == 0) { tk[0] = sil; if (tf) tf[0] = 0; }
    count = 1;
  }
  for (int t0 = 0; t0 < Tb; t0 += 32) {
    const int t = t0 + lane;
    int tok = -1;
    if (t < Tb) {
      const float* row = lg + static_cast<long long>(t) * V;
      float bv = row[0];
      tok = 0;
      for (int c = 1; c < V; ++c) {
        const float v = row[c];
        if (v > bv) { bv = v; tok = c; }
      }
    }
    int left = __shfl_up_sync(0xffffffffu, tok, 1);
    if (lane == 0) left = prev;
    const bool keep = t < Tb && tok != left && tok != blank;
    const uint32_t mask = __ballot_sync(0xffffffffu, keep);
    const int pos = count + __popc(mask & ((1u << lane) - 1));
    if (keep && pos < maxtok) {
      tk[pos] = tok;
      if (tf) tf[pos] = t + off;
    }
    count += __popc(mask);
    prev = __shfl_sync(0xffffffffu, tok, min(31, Tb - 1 - t0));      // label of the last valid frame so far
  }
  if (sil >= 0 && sil != blank && prev != sil) {
    if (lane == 0 && count < maxtok) { tk[count] = sil; if (tf) tf[count] = Tb + 1; }
    count += 1;
  }
  if (lane == 0) ntokens[b] = count;
}

// states per lane: 2 * Smax + 1 states over 32 lanes (up to 511 labels; 0 selects the long-transcript kernels)
static int ni_for_states(int Smax) {
  const int ns = 2 * Smax + 1;
  return ns <= 128 ? 4 : (ns <= 256 ? 8 : (ns <= 512 ? 16 : (ns <= 1024 ? 32 : 0)));
}
static size_t bp_word_bytes(int ni) { return ni <= 8 ? 2 : (ni == 16 ? 4 : 8); }

// ------------------------------------------------------------------------------------------------ long transcripts
// Smax > 511 (more than 1024 states): the state vector spans a whole CTA, LONG_NI consecutive states per thread.
// The two neighbours of a thread's first state (alpha / Viterbi) or last state (beta) come from the adjacent thread
// through a double-buffered shared-memory array, so there is one barrier per frame.  Up to 512 threads: 8192 states.
constexpr int LONG_NI = 16;
constexpr int LONG_MAX_THREADS = 512;
constexpr int CTC_LONG_MAX_LABELS = 4095;      // 2 * 4095 + 1 = 8191 states <= LONG_MAX_THREADS * LONG_NI
constexpr int LONG_GRAD_WARPS = 4;

// threads of the recursion CTA: whole warps covering 2 * Smax + 1 states, LONG_NI per thread
static int long_threads(int Smax) { return 32 * ((2 * Smax + 1 + 32 * LONG_NI - 1) / (32 * LONG_NI)); }

struct CtcLongArgs {
  CtcArgs c;          // alpha / beta hold the NORMALISED recursions (see ctc_long_ab_kernel), SP = LONG_NI * threads
  double* norm_a;     // ws [B][T]: log of the factor alpha[t] was divided by (sum of the per-frame normalisers)
  double* norm_b;     // ws [B][T]: the same for beta
  double* nll_raw;    // ws [B]: -log p before zero_infinity
  int* nxt;           // ws [B][Smax]: next label index with the same class, -1 at the end of the chain
  int* first;         // ws [B][Smax]: 1 at the first occurrence of a class
};

// log-sum-exp of one frame and the optional log_probs output: one warp per (utterance, frame)
__global__ void __launch_bounds__(256) ctc_long_lse_kernel(const CtcArgs a) {
  const int lane = threadIdx.x & 31;
  const long long w = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (w >= static_cast<long long>(a.B) * a.T) return;
  const int b = static_cast<int>(w / a.T), t = static_cast<int>(w % a.T);
  const int Veff = a.V + (a.prepend_blank ? 1 : 0);
  const int Vb = a.vocab_len ? min(a.vocab_len[b], Veff) : Veff;
  const float* row = a.logits + w * a.V;
  float m = NEG_INF;
  for (int c = lane; c < Vb; c += 32) m = fmaxf(m, logit_at(a, row, c));
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float s = 0.f;
  for (int c = lane; c < Vb; c += 32) s += expf(logit_at(a, row, c) - m);
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float l = logf(s) + m;
  if (lane == 0) a.lse[w] = l;
  if (a.log_probs_tbv) {
    float* o = a.log_probs_tbv + (static_cast<long long>(t) * a.B + b) * Veff;
    for (int c = lane; c < Veff; c += 32) o[c] = c < Vb ? logit_at(a, row, c) - l : NEG_INF;
  }
}

// same-class chains of the labels (for the deterministic per-class occupancy sums): grid (ceil(Smax / 256), B)
__global__ void __launch_bounds__(256) ctc_long_chain_kernel(const int* __restrict__ targets, int Smax,
                                                             const int* __restrict__ target_len, int* __restrict__ nxt,
                                                             int* __restrict__ first) {
  extern __shared__ int s_tg[];
  const int b = blockIdx.y;
  const int S = min(target_len[b], Smax);
  const int* tg = targets + static_cast<long long>(b) * Smax;
  for (int k = threadIdx.x; k < S; k += blockDim.x) s_tg[k] = tg[k];
  __syncthreads();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= Smax) return;
  int nx = -1, fs = 1;
  if (j < S) {
    const int l = s_tg[j];
    for (int k = j + 1; k < S; ++k)
      if (s_tg[k] == l) { nx = k; break; }
    for (int k = j - 1; k >= 0; --k)
      if (s_tg[k] == l) { fs = 0; break; }
  }
  nxt[static_cast<long long>(b) * Smax + j] = nx;
  first[static_cast<long long>(b) * Smax + j] = fs;
}

// alpha (blockIdx.y == 0) and beta (blockIdx.y == 1) of one utterance, LONG_NI states per thread.
// At T ~ 9000 the unnormalised log-space values reach ~1e4 and fp32 rounding accumulates, so every frame is divided
// by the previous frame's maximum: alpha'[t] = alpha[t] - norm_a[t], norm_a[t] = sum of those maxima (fp64).  The
// maximum of each frame travels with the neighbour exchange (per-warp maxima in shared memory), so the normaliser
// costs no extra barrier.  The alpha CTA writes nll.
__global__ void __launch_bounds__(LONG_MAX_THREADS, 1) ctc_long_ab_kernel(const CtcLongArgs la) {
  const CtcArgs& a = la.c;
  __shared__ float2 s_edge[2][LONG_MAX_THREADS];
  __shared__ float s_wmax[2][LONG_MAX_THREADS / 32];
  const int b = blockIdx.x;
  const bool fwd = blockIdx.y == 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nthr = blockDim.x, nwarp = nthr >> 5;
  const int Tb = min(a.input_len[b], a.T);
  const int S = min(a.target_len[b], a.Smax);
  const int NS = 2 * S + 1;
  const int SP = a.SP;
  const float* lg = a.logits + static_cast<long long>(b) * a.T * a.V;
  const float* lse = a.lse + static_cast<long long>(b) * a.T;
  float* out = (fwd ? a.alpha : a.beta) + static_cast<long long>(b) * a.T * SP;
  double* norm = (fwd ? la.norm_a : la.norm_b) + static_cast<long long>(b) * a.T;
  const int* tg = a.targets + static_cast<long long>(b) * a.Smax;

  if (Tb <= 0) {      // no frames: loss inf (0 with zero_infinity), gradient 0
    if (fwd && tid == 0) {
      la.nll_raw[b] = INFINITY;
      a.nll[b] = a.zero_infinity ? 0.f : INFINITY;
    }
    return;
  }
  int lab[LONG_NI];
  uint32_t skip = 0;   // bit i: alpha may come from s-2 / beta may go to s+2
#pragma unroll
  for (int i = 0; i < LONG_NI; ++i) {
    const int s = tid * LONG_NI + i;
    const bool odd = (s & 1) && s < NS;
    lab[i] = odd ? tg[s / 2] : a.blank;
    const bool ok = fwd ? (odd && s >= 3 && tg[s / 2] != tg[s / 2 - 1]) : (odd && s + 2 < NS && tg[s / 2] != tg[s / 2 + 1]);
    skip |= static_cast<uint32_t>(ok) << i;
  }
  const int t0 = fwd ? 0 : Tb - 1;
  const int dir = fwd ? 1 : -1;
  float cur[LONG_NI];
  {
    const float* row = lg + static_cast<long long>(t0) * a.V;
    const float l0 = lse[t0];
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) {
      const int s = tid * LONG_NI + i;
      const bool init = fwd ? (s < 2 && s < NS) : (s < NS && s >= NS - 2);
      cur[i] = init ? logit_at(a, row, lab[i]) - l0 : NEG_INF;
      out[static_cast<long long>(t0) * SP + s] = cur[i];
    }
  }
  if (tid == 0) norm[t0] = 0.0;
  auto publish = [&](int p) {
    float mx = cur[0];
#pragma unroll
    for (int i = 1; i < LONG_NI; ++i) mx = fmaxf(mx, cur[i]);
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    s_edge[p][tid] = fwd ? make_float2(cur[LONG_NI - 1], cur[LONG_NI - 2]) : make_float2(cur[0], cur[1]);
    if (lane == 0) s_wmax[p][warp] = mx;
  };
  auto gather = [&](int t, float* lp) {
    const float* row = lg + static_cast<long long>(t) * a.V;
    const float lt = lse[t];
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) lp[i] = logit_at(a, row, lab[i]) - lt;
  };
  publish(0);
  double C = 0.0;
  float lpn[LONG_NI];
  if (Tb > 1) gather(t0 + dir, lpn);
  for (int step = 1; step < Tb; ++step) {
    const int t = t0 + dir * step;
    float lp[LONG_NI];
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) lp[i] = lpn[i];
    if (step + 1 < Tb) gather(t + dir, lpn);       // next frame's log-probs in flight during this one
    __syncthreads();
    const int p = (step - 1) & 1;
    const int nb_tid = fwd ? tid - 1 : tid + 1;
    const float2 nb = (nb_tid >= 0 && nb_tid < nthr) ? s_edge[p][nb_tid] : make_float2(NEG_INF, NEG_INF);
    float c = NEG_INF;
    for (int w = 0; w < nwarp; ++w) c = fmaxf(c, s_wmax[p][w]);
    if (c == NEG_INF) c = 0.f;
    C += c;
    float nw[LONG_NI];
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) {
      float x1, x2r;
      if (fwd) {
        x1 = i >= 1 ? cur[i - 1] : nb.x;
        x2r = i >= 2 ? cur[i - 2] : (i == 1 ? nb.x : nb.y);
      } else {
        x1 = i + 1 < LONG_NI ? cur[i + 1] : nb.x;
        x2r = i + 2 < LONG_NI ? cur[i + 2] : (i + 2 == LONG_NI ? nb.x : nb.y);
      }
      const float x2 = (skip >> i) & 1 ? x2r : NEG_INF;
      const int s = tid * LONG_NI + i;
      nw[i] = s < NS ? lse3(cur[i], x1, x2) - c + lp[i] : NEG_INF;
    }
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) {
      cur[i] = nw[i];
      out[static_cast<long long>(t) * SP + tid * LONG_NI + i] = nw[i];
    }
    if (tid == 0) norm[t] = C;
    publish(step & 1);
  }
  if (!fwd) return;
  __syncthreads();    // alpha of the last frame, written by other threads, is visible after the barrier
  if (tid == 0) {
    const float* al = out + static_cast<long long>(Tb - 1) * SP;
    const float a1 = al[NS - 1];
    const float a2 = NS >= 2 ? al[NS - 2] : NEG_INF;
    float m = fmaxf(a1, a2);
    if (m == NEG_INF) m = 0.f;
    const double nll = -(static_cast<double>(logf(expf(a1 - m) + expf(a2 - m)) + m) + C);
    la.nll_raw[b] = nll;
    const float nf = static_cast<float>(nll);
    a.nll[b] = (!(nf < INFINITY) && a.zero_infinity) ? 0.f : nf;
  }
}

// gradient w.r.t. the logits, one warp per (utterance, frame); per-class occupancies are summed along the
// same-class chains in a fixed order (no atomics: bit-identical from run to run)
__global__ void __launch_bounds__(32 * LONG_GRAD_WARPS) ctc_long_grad_kernel(const CtcLongArgs la) {
  extern __shared__ float sm[];
  const CtcArgs& a = la.c;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long w = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp;
  if (w >= static_cast<long long>(a.B) * a.T) return;
  const int b = static_cast<int>(w / a.T), t = static_cast<int>(w % a.T);
  const int Veff = a.V + (a.prepend_blank ? 1 : 0);
  const int Vb = a.vocab_len ? min(a.vocab_len[b], Veff) : Veff;
  const int Tb = min(a.input_len[b], a.T);
  const int S = min(a.target_len[b], a.Smax);
  const int NS = 2 * S + 1;
  const int SP = a.SP;
  float* grow = a.grad + w * a.V;
  const double nll = la.nll_raw[b];
  const bool infeasible = !(static_cast<float>(nll) < INFINITY);
  if (t >= Tb || (infeasible && a.zero_infinity)) {
    for (int c = lane; c < a.V; c += 32) grow[c] = 0.f;
    return;
  }
  const float sc = a.scale ? a.scale[b] : 1.f;
  const int* tg = a.targets + static_cast<long long>(b) * a.Smax;
  const int* nxt = la.nxt + static_cast<long long>(b) * a.Smax;
  const int* first = la.first + static_cast<long long>(b) * a.Smax;
  float* scr_ab = sm + warp * (SP + Veff);
  float* scr_cls = scr_ab + SP;
  const float* al = a.alpha + w * SP;
  const float* be = a.beta + w * SP;
  float m = NEG_INF;
  for (int s = lane; s < SP; s += 32) {
    const float v = s < NS ? al[s] + be[s] : NEG_INF;
    scr_ab[s] = v;
    m = fmaxf(m, v);
  }
  for (int c = lane; c < Veff; c += 32) scr_cls[c] = 0.f;
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (m == NEG_INF) m = 0.f;
  __syncwarp();
  float bs = 0.f;
  for (int s = 2 * lane; s < NS; s += 64) bs += expf(scr_ab[s] - m);
  for (int o = 16; o; o >>= 1) bs += __shfl_xor_sync(0xffffffffu, bs, o);
  for (int j = lane; j < S; j += 32) {
    if (!first[j]) continue;
    float acc = 0.f;
    for (int k = j; k >= 0; k = nxt[k]) acc += expf(scr_ab[2 * k + 1] - m);
    const int cls = tg[j];
    if (cls == a.blank) continue;
    scr_cls[cls] = acc;
  }
  __syncwarp();
  // log posterior = alpha' + beta' + (norm_a + norm_b + nll): the fp64 sum cancels to O(1)
  const float K = static_cast<float>(la.norm_a[w] + la.norm_b[w] + nll);
  const float* rw = a.logits + w * a.V;
  const float lt = a.lse[w];
  for (int c = lane; c < Veff; c += 32) {
    const int col = a.prepend_blank ? c - 1 : c;
    if (col < 0) continue;
    float g = 0.f;
    if (c < Vb) {
      const float lp = logit_at(a, rw, c) - lt;
      const float occ = (c == a.blank) ? bs : scr_cls[c];
      const float post = occ > 0.f ? expf(logf(occ) + m + K - lp) : 0.f;
      g = (expf(lp) - post) * sc;
    }
    grow[col] = g;
  }
}

// Viterbi over LONG_NI states per thread; back-pointers as one 32-bit word per (frame, thread) in global memory
__global__ void __launch_bounds__(LONG_MAX_THREADS, 1) viterbi_long_kernel(const VitArgs a) {
  __shared__ float2 s_edge[2][LONG_MAX_THREADS];
  __shared__ int s_red[LONG_MAX_THREADS / 32];
  __shared__ float s_fin[2];
  __shared__ uint32_t s_bp[32][5];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nthr = blockDim.x, nwarp = nthr >> 5;
  const int Tb = min(a.input_len[b], a.T);
  const int L = min(a.target_len[b], a.Smax);
  const int NS = 2 * L + 1;
  const int* tg = a.targets + static_cast<long long>(b) * a.Smax;
  const float* lp = a.lp + static_cast<long long>(b) * a.T * a.C;
  int* path = a.paths + static_cast<long long>(b) * a.T;
  float* score = a.scores ? a.scores + static_cast<long long>(b) * a.T : nullptr;
  uint32_t* bp = reinterpret_cast<uint32_t*>(a.bp_global) + static_cast<long long>(b) * a.T * nthr;

  for (int t = Tb + tid; t < a.T; t += nthr) {
    path[t] = -1;
    if (score) score[t] = 0.f;
  }
  int R = 0;
  for (int j = 1 + tid; j < L; j += nthr) R += (tg[j] == tg[j - 1]);
  for (int o = 16; o; o >>= 1) R += __shfl_xor_sync(0xffffffffu, R, o);
  if (lane == 0) s_red[warp] = R;
  __syncthreads();
  R = 0;
  for (int w = 0; w < nwarp; ++w) R += s_red[w];
  if (Tb <= 0 || Tb < L + R) {
    if (tid == 0 && a.status) a.status[b] = 1;
    for (int t = tid; t < Tb; t += nthr) {
      path[t] = -1;
      if (score) score[t] = 0.f;
    }
    return;
  }
  if (tid == 0 && a.status) a.status[b] = 0;
  int lab[LONG_NI];
  uint32_t skip = 0;
#pragma unroll
  for (int i = 0; i < LONG_NI; ++i) {
    const int s = tid * LONG_NI + i;
    const bool odd = (s & 1) && s < NS;
    lab[i] = odd ? tg[s / 2] : a.blank;
    skip |= static_cast<uint32_t>(odd && s >= 3 && tg[s / 2] != tg[s / 2 - 1]) << i;
  }
  const int start = (Tb - (L + R) > 0) ? 0 : 1;
  const int end = NS == 1 ? 1 : 2;
  float cur[LONG_NI];
#pragma unroll
  for (int i = 0; i < LONG_NI; ++i) {
    const int s = tid * LONG_NI + i;
    cur[i] = (s >= start && s < end) ? lp[lab[i]] : NEG_INF;
  }
  s_edge[0][tid] = make_float2(cur[LONG_NI - 1], cur[LONG_NI - 2]);
  float en[LONG_NI];
  if (Tb > 1) {
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) en[i] = lp[static_cast<long long>(a.C) + lab[i]];
  }
  for (int t = 1; t < Tb; ++t) {
    float e[LONG_NI];
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) e[i] = en[i];
    if (t + 1 < Tb) {
      const float* row = lp + static_cast<long long>(t + 1) * a.C;
#pragma unroll
      for (int i = 0; i < LONG_NI; ++i) en[i] = row[lab[i]];
    }
    __syncthreads();
    const float2 nb = tid > 0 ? s_edge[(t - 1) & 1][tid - 1] : make_float2(NEG_INF, NEG_INF);
    float nw[LONG_NI];
    uint32_t code = 0;
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) {
      const float x0 = cur[i];
      const float x1 = i >= 1 ? cur[i - 1] : nb.x;
      const float x2r = i >= 2 ? cur[i - 2] : (i == 1 ? nb.x : nb.y);
      const float x2 = (skip >> i) & 1 ? x2r : NEG_INF;
      float best;
      uint32_t c;
      if (x2 > x1 && x2 > x0) { best = x2; c = 2; }
      else if (x1 > x0 && x1 > x2) { best = x1; c = 1; }
      else { best = x0; c = 0; }
      const int s = tid * LONG_NI + i;
      nw[i] = (s < NS && best != NEG_INF) ? __fadd_rn(best, e[i]) : NEG_INF;
      code |= c << (2 * i);
    }
#pragma unroll
    for (int i = 0; i < LONG_NI; ++i) cur[i] = nw[i];
    bp[static_cast<long long>(t) * nthr + tid] = code;
    s_edge[t & 1][tid] = make_float2(cur[LONG_NI - 1], cur[LONG_NI - 2]);
  }
#pragma unroll
  for (int i = 0; i < LONG_NI; ++i) {
    const int s = tid * LONG_NI + i;
    if (s == NS - 1) s_fin[0] = cur[i];
    if (s == NS - 2) s_fin[1] = cur[i];
  }
  __syncthreads();    // also makes the back-pointer words of all threads visible
  if (warp == 0) {
    // final state: NS-1 if alpha[NS-1] > alpha[NS-2] (strict) else NS-2 ; NS == 1 -> 0
    int s = NS == 1 ? 0 : (s_fin[0] > s_fin[1] ? NS - 1 : NS - 2);
    // 32 frames at a time: from state s at frame hi the path stays within s - 62 .. s, i.e. within the five words
    // w0-4 .. w0 of each frame; the warp stages those words, then lane 0 walks them
    for (int hi = Tb - 1; hi >= 0; hi -= 32) {
      const int w0 = s / LONG_NI;
      const int t = hi - lane;
      if (t >= 1) {
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          const int wi = w0 - 4 + k;
          s_bp[lane][k] = wi >= 0 ? bp[static_cast<long long>(t) * nthr + wi] : 0u;
        }
      }
      __syncwarp();
      if (lane == 0) {
        for (int k = 0; k < 32 && hi - k >= 0; ++k) {
          const int tt = hi - k;
          path[tt] = (s & 1) ? tg[s / 2] : a.blank;
          if (tt > 0) {
            const uint32_t code = s_bp[k][s / LONG_NI - (w0 - 4)];
            s -= static_cast<int>((code >> (2 * (s % LONG_NI))) & 3u);
          }
        }
      }
      s = __shfl_sync(0xffffffffu, s, 0);
      __syncwarp();
    }
  }
  if (!score) return;
  __syncthreads();
  for (int t = tid; t < Tb; t += nthr) score[t] = lp[static_cast<long long>(t) * a.C + path[t]];
}

}  // namespace aptai

using namespace aptai;

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// long-transcript workspace: alpha, beta [B][T][SP] fp32 | lse [B][T] fp32 | norm_a, norm_b [B][T] fp64 |
// nll_raw [B] fp64 | nxt, first [B][Smax] int32
static size_t ctc_long_workspace_bytes(int B, int T, int Smax) {
  const size_t bt = static_cast<size_t>(B) * T;
  const size_t sp = static_cast<size_t>(LONG_NI) * long_threads(Smax);
  return 2 * align_up(sizeof(float) * bt * sp, 256) + align_up(sizeof(float) * bt, 256) +
         2 * align_up(sizeof(double) * bt, 256) + align_up(sizeof(double) * B, 256) +
         2 * align_up(sizeof(int) * static_cast<size_t>(B) * Smax, 256) + 256;
}

extern "C" size_t aptai_ctc_workspace_bytes(int B, int T, int Smax) {
  const int ni = ni_for_states(Smax);
  if (ni == 0) return Smax <= CTC_LONG_MAX_LABELS ? ctc_long_workspace_bytes(B, T, Smax) : 0;
  const size_t sp = 32 * ni;
  return 2 * align_up(sizeof(float) * B * T * sp, 256) + align_up(sizeof(float) * B * T, 256) + 256;
}

// Smax > 511: lse pass, same-class chains (gradient only), alpha / beta CTAs, gradient pass
static int launch_ctc_long(const CtcArgs& c, void* ws, cudaStream_t st) {
  CtcLongArgs la;
  la.c = c;
  const int B = c.B, T = c.T, Smax = c.Smax;
  const int nthr = long_threads(Smax);
  const size_t bt = static_cast<size_t>(B) * T;
  la.c.SP = LONG_NI * nthr;
  char* w = reinterpret_cast<char*>(ws);
  la.c.alpha = reinterpret_cast<float*>(w);
  w += align_up(sizeof(float) * bt * la.c.SP, 256);
  la.c.beta = reinterpret_cast<float*>(w);
  w += align_up(sizeof(float) * bt * la.c.SP, 256);
  la.c.lse = reinterpret_cast<float*>(w);
  w += align_up(sizeof(float) * bt, 256);
  la.norm_a = reinterpret_cast<double*>(w);
  w += align_up(sizeof(double) * bt, 256);
  la.norm_b = reinterpret_cast<double*>(w);
  w += align_up(sizeof(double) * bt, 256);
  la.nll_raw = reinterpret_cast<double*>(w);
  w += align_up(sizeof(double) * B, 256);
  la.nxt = reinterpret_cast<int*>(w);
  w += align_up(sizeof(int) * static_cast<size_t>(B) * Smax, 256);
  la.first = reinterpret_cast<int*>(w);

  const int Veff = c.V + (c.prepend_blank ? 1 : 0);
  const size_t warp_bytes = sizeof(float) * (static_cast<size_t>(la.c.SP) + Veff);
  const int gwarps = static_cast<int>(std::min<size_t>(LONG_GRAD_WARPS, (200 * 1024) / warp_bytes));
  APTAI_REQUIRE(!c.grad || gwarps >= 1, "ctc: %d classes are too many for the long-transcript gradient", Veff);

  ctc_long_lse_kernel<<<static_cast<unsigned>((bt + 7) / 8), 256, 0, st>>>(la.c);
  if (int rc = after_launch("ctc_long_lse")) return rc;
  if (c.grad) {
    ctc_long_chain_kernel<<<dim3((Smax + 255) / 256, B), 256, sizeof(int) * Smax, st>>>(c.targets, Smax, c.target_len,
                                                                                         la.nxt, la.first);
    if (int rc = after_launch("ctc_long_chain")) return rc;
  }
  ctc_long_ab_kernel<<<dim3(B, c.grad ? 2 : 1), nthr, 0, st>>>(la);
  if (int rc = after_launch("ctc_long_ab")) return rc;
  if (c.grad) {
    const size_t smem = warp_bytes * gwarps;
    if (smem > 48 * 1024) {
      const cudaError_t e = cudaFuncSetAttribute(ctc_long_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(smem));
      if (e != cudaSuccess) {
        set_error("ctc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return static_cast<int>(e);
      }
    }
    ctc_long_grad_kernel<<<static_cast<unsigned>((bt + gwarps - 1) / gwarps), 32 * gwarps, smem, st>>>(la);
    if (int rc = after_launch("ctc_long_grad")) return rc;
  }
  return APTAI_OK;
}

extern "C" int aptai_logsoftmax_ctc(const float* logits, int B, int T, int V, const int32_t* targets, int Smax,
                                    const int32_t* input_len, const int32_t* target_len, int blank,
                                    int zero_infinity, float* log_probs_tbv, float* nll, const float* scale,
                                    float* grad, void* ws, size_t ws_bytes, void* stream);

// Extended entry (ForwardSumLoss): virtual blank column and per-utterance class count.
extern "C" int aptai_logsoftmax_ctc_ex(const float* logits, int B, int T, int V, int prepend_blank,
                                       float blank_value, const int32_t* vocab_len, const int32_t* targets,
                                       int Smax, const int32_t* input_len, const int32_t* target_len, int blank,
                                       int zero_infinity, float* log_probs_tbv, float* nll, const float* scale,
                                       float* loss_sum, float* grad, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(logits && targets && input_len && target_len && nll && ws, "ctc: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && V >= 1 && Smax >= 1, "ctc: bad shape");
  const int ni = ni_for_states(Smax);
  APTAI_REQUIRE(ni != 0 || Smax <= CTC_LONG_MAX_LABELS, "ctc: Smax=%d exceeds the limit of %d labels per utterance",
                Smax, CTC_LONG_MAX_LABELS);
  const int Veff = V + (prepend_blank ? 1 : 0);
  APTAI_REQUIRE(blank >= 0 && blank < Veff, "ctc: blank index out of range");
  const size_t need = aptai_ctc_workspace_bytes(B, T, Smax);
  if (ws_bytes < need) {
    set_error("ctc: workspace %zu < %zu bytes", ws_bytes, need);
    return APTAI_ERR_WORKSPACE;
  }
  CtcArgs a;
  a.logits = logits; a.B = B; a.T = T; a.V = V;
  a.prepend_blank = prepend_blank; a.blank_value = blank_value;
  a.targets = targets; a.Smax = Smax; a.input_len = input_len; a.target_len = target_len; a.vocab_len = vocab_len;
  a.blank = blank; a.zero_infinity = zero_infinity;
  a.log_probs_tbv = log_probs_tbv; a.nll = nll; a.scale = scale; a.grad = grad;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (ni == 0) {
    if (int rc = launch_ctc_long(a, ws, st)) return rc;
    if (loss_sum) {
      ctc_reduce_kernel<<<1, 32, 0, st>>>(nll, scale, B, loss_sum);
      if (int rc = after_launch("ctc_reduce")) return rc;
    }
    return APTAI_OK;
  }
  const size_t sp = 32 * ni;
  char* w = reinterpret_cast<char*>(ws);
  a.alpha = reinterpret_cast<float*>(w);
  w += align_up(sizeof(float) * B * T * sp, 256);
  a.beta = reinterpret_cast<float*>(w);
  w += align_up(sizeof(float) * B * T * sp, 256);
  a.lse = reinterpret_cast<float*>(w);
  a.SP = static_cast<int>(sp);
  const size_t smem = sizeof(int) * (sp + sp) + sizeof(float) * (CTC_THREADS / 32) * (sp + Veff);
  if (ni == 4) ctc_kernel<4><<<B, CTC_THREADS, smem, st>>>(a);
  else if (ni == 8) ctc_kernel<8><<<B, CTC_THREADS, smem, st>>>(a);
  else if (ni == 16) ctc_kernel<16><<<B, CTC_THREADS, smem, st>>>(a);
  else ctc_kernel<32><<<B, CTC_THREADS, smem, st>>>(a);
  if (int rc = after_launch("logsoftmax_ctc")) return rc;
  if (loss_sum) {
    ctc_reduce_kernel<<<1, 32, 0, st>>>(nll, scale, B, loss_sum);
    if (int rc = after_launch("ctc_reduce")) return rc;
  }
  return APTAI_OK;
}

extern "C" int aptai_logsoftmax_ctc(const float* logits, int B, int T, int V, const int32_t* targets, int Smax,
                                    const int32_t* input_len, const int32_t* target_len, int blank,
                                    int zero_infinity, float* log_probs_tbv, float* nll, const float* scale,
                                    float* grad, void* ws, size_t ws_bytes, void* stream) {
  return aptai_logsoftmax_ctc_ex(logits, B, T, V, 0, 0.f, nullptr, targets, Smax, input_len, target_len, blank,
                                 zero_infinity, log_probs_tbv, nll, scale, nullptr, grad, ws, ws_bytes, stream);
}

extern "C" size_t aptai_viterbi_workspace_bytes(int B, int T, int Smax) {
  const int ni = ni_for_states(Smax);
  if (ni == 0)
    return Smax <= CTC_LONG_MAX_LABELS ? align_up(sizeof(uint32_t) * static_cast<size_t>(B) * T * long_threads(Smax), 256)
                                       : 0;
  return align_up(bp_word_bytes(ni ? ni : 32) * static_cast<size_t>(B) * T * 32, 256);
}

extern "C" int aptai_ctc_viterbi_f32(const float* log_probs, const int32_t* targets, const int32_t* input_len,
                                     const int32_t* target_len, int B, int T, int C, int Smax, int blank,
                                     int32_t* paths, float* scores, int32_t* status, void* ws, size_t ws_bytes,
                                     void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(log_probs && targets && input_len && target_len && paths, "viterbi: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && C >= 1 && Smax >= 1, "viterbi: bad shape");
  APTAI_REQUIRE(blank >= 0 && blank < C, "viterbi: blank index out of range");
  const int ni = ni_for_states(Smax);
  APTAI_REQUIRE(ni != 0 || Smax <= CTC_LONG_MAX_LABELS, "viterbi: Smax=%d exceeds the limit of %d labels per utterance",
                Smax, CTC_LONG_MAX_LABELS);
  VitArgs a;
  a.lp = log_probs; a.targets = targets; a.input_len = input_len; a.target_len = target_len;
  a.B = B; a.T = T; a.C = C; a.Smax = Smax; a.blank = blank;
  a.paths = paths; a.scores = scores; a.status = status;
  if (ni == 0) {      // Smax > 511: CTA-wide state vector, back-pointers in the workspace
    const size_t need = aptai_viterbi_workspace_bytes(B, T, Smax);
    if (!ws || ws_bytes < need) {
      set_error("viterbi: workspace %zu < %zu bytes", ws_bytes, need);
      return APTAI_ERR_WORKSPACE;
    }
    a.bp_global = ws;
    a.bp_in_smem = 0;
    viterbi_long_kernel<<<B, long_threads(Smax), 0, reinterpret_cast<cudaStream_t>(stream)>>>(a);
    return after_launch("ctc_viterbi_long");
  }
  const size_t bp_bytes = bp_word_bytes(ni) * static_cast<size_t>(T) * 32;
  a.bp_in_smem = bp_bytes <= 200 * 1024;
  a.bp_global = ws;
  if (!a.bp_in_smem) {
    const size_t need = aptai_viterbi_workspace_bytes(B, T, Smax);
    if (!ws || ws_bytes < need) {
      set_error("viterbi: workspace %zu < %zu bytes", ws_bytes, need);
      return APTAI_ERR_WORKSPACE;
    }
  }
  const size_t smem = a.bp_in_smem ? bp_bytes : 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaError_t e = cudaSuccess;
#define APTAI_VIT_LAUNCH(N)                                                                                          \
  do {                                                                                                              \
    if (smem > 32 * 1024)                                                                                           \
      e = cudaFuncSetAttribute(viterbi_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);         \
    if (e == cudaSuccess) viterbi_kernel<N><<<B, 32, smem, st>>>(a);                                                \
  } while (0)
  if (ni == 4) APTAI_VIT_LAUNCH(4);
  else if (ni == 8) APTAI_VIT_LAUNCH(8);
  else if (ni == 16) APTAI_VIT_LAUNCH(16);
  else APTAI_VIT_LAUNCH(32);
#undef APTAI_VIT_LAUNCH
  if (e != cudaSuccess) {
    set_error("viterbi: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return static_cast<int>(e);
  }
  return after_launch("ctc_viterbi");
}

extern "C" int aptai_ctc_greedy(const float* logits, int B, int T, int V, const int32_t* input_len, int blank,
                                int32_t* tokens, int32_t* token_frames, int32_t* ntokens, int maxtok, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(logits && tokens && ntokens, "ctc_greedy: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && V >= 1 && maxtok >= 1, "ctc_greedy: bad shape");
  ctc_greedy_kernel<<<B, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(logits, T, V, input_len, blank, -1, tokens,
                                                                         token_frames, ntokens, maxtok);
  return after_launch("ctc_greedy");
}

extern "C" int aptai_ctc_decode_ref(const float* logits, int B, int T, int V, const int32_t* input_len, int blank,
                                    int sil, int32_t* tokens, int32_t* timesteps, int32_t* ntokens, int maxtok,
                                    void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(logits && tokens && ntokens, "ctc_decode_ref: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && V >= 1 && maxtok >= T + 2, "ctc_decode_ref: bad shape (maxtok >= T + 2)");
  APTAI_REQUIRE(sil >= 0 && sil < V && blank >= 0 && blank < V, "ctc_decode_ref: bad blank / sil id");
  ctc_greedy_kernel<<<B, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(logits, T, V, input_len, blank, sil, tokens,
                                                                         timesteps, ntokens, maxtok);
  return after_launch("ctc_decode_ref");
}
