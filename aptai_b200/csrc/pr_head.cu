// Phoneme-recogniser head for vocabularies of 49..1024 symbols (models/w2v2_pr.py:47 `pr_head = nn.Linear(H, V)`).
//
// The fused `aptai_heads` kernel keeps its weights in 48 head-B slots; wider heads run here on the tensor cores, at
// the fp32 level of the accuracy mode (csrc/accurate.cu):
//     logits = [h_hi | h_lo | h_hi] . [W_hi | W_hi | W_lo]^T + b          (K = 3H)
// The GEMM's N must be one of its tile widths, so W is padded with zero rows to Vp = 64 * ceil(V / 64) and the raw
// logits are written with a row pitch >= Vp.  `logits_rows_kernel` then reads each row once (one warp, up to 32
// values per lane in registers) and writes any of: the compact [rows][V] logits, the first-max argmax, the log-softmax
// and the softmax.
//
// Backward (d_logits fp32 [rows][V], row pitch ld_d):
//     dh  = [dY_hi | dY_lo | dY_hi] . [Wt_hi | Wt_hi | Wt_lo]^T            (K = 3Vp, Wt = W^T zero-padded to Vp)
//     dW += dY_hi^T h_hi + dY_lo^T h_hi + dY_hi^T h_lo                     (three MN-major wgrad launches)
//     db += column sums of d_logits
#include "common.h"
#include "ptx.cuh"

#include <math.h>
#include <string.h>

namespace aptai {

constexpr int PH_MAX_V = 1024;
constexpr int PH_ALIGN = 256;

static inline int64_t ph_pad_v(int V) { return (static_cast<int64_t>(V) + 63) / 64 * 64; }
static inline size_t ph_round(size_t n) { return (n + PH_ALIGN - 1) / PH_ALIGN * PH_ALIGN; }

// out[r][0..3*cols_pad) = split of x(r, c) = x[r*ld_r + c*ld_c] for r < rows, c < cols, else 0:
// [hi | lo | hi] (mode 0, activations) or [hi | hi | lo] (mode 1, weights), rows_pad output rows
__global__ void split3_pad_kernel(const float* __restrict__ x, long long rows, int cols, long long ld_r, long long ld_c,
                                  long long rows_pad, int cols_pad, int mode, __nv_bfloat16* __restrict__ out) {
  const long long total = rows_pad * cols_pad;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols_pad;
    const int c = static_cast<int>(i - r * cols_pad);
    const float v = (r < rows && c < cols) ? x[r * ld_r + c * ld_c] : 0.f;
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    __nv_bfloat16* o = out + r * 3 * cols_pad + c;
    o[0] = hi;
    o[cols_pad] = mode ? hi : lo;
    o[2 * cols_pad] = mode ? lo : hi;
  }
}

// One warp per row, NPL values per lane (column j*32 + lane).  Argmax: first maximum (strict > along a lane's
// increasing columns, smaller index on equal values across lanes), as heads_kernel and ctc_greedy.  The log-softmax /
// softmax use softmax_rows_kernel's formulas and summation order.
template <int NPL>
__global__ void __launch_bounds__(256)
logits_rows_kernel(const float* __restrict__ x, long long rows, int V, long long ldx, float* __restrict__ logits,
                   long long* __restrict__ argmax, float* __restrict__ logp, float* __restrict__ prob) {
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows;
       row += warps) {
    const float* xr = x + row * ldx;
    float v[NPL];
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const int c = j * 32 + lane;
      v[j] = c < V ? xr[c] : -INFINITY;
    }
    float bv = -INFINITY;
    int bi = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const int c = j * 32 + lane;
      if (c < V && (bi == 0x7fffffff || v[j] > bv)) {
        bv = v[j];
        bi = c;
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) {
        bv = ov;
        bi = oi;
      }
    }
    const long long ro = row * V;
    if (logits) {
#pragma unroll
      for (int j = 0; j < NPL; ++j) {
        const int c = j * 32 + lane;
        if (c < V) logits[ro + c] = v[j];
      }
    }
    if (argmax && lane == 0) argmax[row] = bi;
    if (logp || prob) {
      const float m = bv;
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < NPL; ++j)
        if (j * 32 + lane < V) s += expf(v[j] - m);
#pragma unroll
      for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float ls = logf(s);
#pragma unroll
      for (int j = 0; j < NPL; ++j) {
        const int c = j * 32 + lane;
        if (c < V) {
          const float d = v[j] - m;
          if (logp) logp[ro + c] = d - ls;
          if (prob) prob[ro + c] = expf(d) / s;
        }
      }
    }
  }
}

// db[c] += sum over rows of d[r*ld + c]: 32 columns per CTA (one per lane), the 8 warps stride a slab of rows, fp32
// partial sums combined in shared memory, one atomic per column and CTA (any row pitch, unlike aptai_colsum)
__global__ void __launch_bounds__(256)
colsum_pitch_kernel(const float* __restrict__ d, long long rows, int V, long long ld, long long rows_per_slab,
                    float* __restrict__ db) {
  __shared__ float part[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  const long long r0 = static_cast<long long>(blockIdx.y) * rows_per_slab;
  const long long r1 = r0 + rows_per_slab < rows ? r0 + rows_per_slab : rows;
  float s = 0.f;
  if (c < V)
    for (long long r = r0 + warp; r < r1; r += 8) s += d[r * ld + c];
  part[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && c < V) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += part[k][lane];
    atomicAdd(db + c, t);
  }
}

static int ph_grid(long long work, int per_block, int cap) {
  const long long g = (work + per_block - 1) / per_block;
  return static_cast<int>(g < cap ? (g < 1 ? 1 : g) : cap);
}

static int launch_split3_pad(const float* x, long long rows, int cols, long long ld_r, long long ld_c,
                             long long rows_pad, int cols_pad, int mode, void* out, cudaStream_t st) {
  split3_pad_kernel<<<ph_grid(rows_pad * cols_pad, 256, 8192), 256, 0, st>>>(
      x, rows, cols, ld_r, ld_c, rows_pad, cols_pad, mode, reinterpret_cast<__nv_bfloat16*>(out));
  return after_launch("pr_head_split3_pad");
}

// Workspace carve-up (each part 256-byte aligned).  Forward: h split [rows][3H], W split [Vp][3H], bias [Vp].
// Backward: d_logits split [rows][3Vp], W^T split [H][3Vp], h split [rows][3H].
struct PhWs {
  size_t a, b, c;
  size_t total() const { return a + b + c; }
};

static PhWs ph_ws(int64_t rows, int H, int V, int backward) {
  const int64_t Vp = ph_pad_v(V);
  PhWs w;
  if (backward) {
    w.a = ph_round(static_cast<size_t>(rows) * 3 * Vp * 2);
    w.b = ph_round(static_cast<size_t>(H) * 3 * Vp * 2);
    w.c = ph_round(static_cast<size_t>(rows) * 3 * H * 2);
  } else {
    w.a = ph_round(static_cast<size_t>(rows) * 3 * H * 2);
    w.b = ph_round(static_cast<size_t>(Vp) * 3 * H * 2);
    w.c = ph_round(static_cast<size_t>(Vp) * 4);
  }
  return w;
}

static void ph_gemm_args(aptai_gemm_args* g, const void* a, int64_t M, int K, const void* w, int N, const float* bias,
                         float* out, int64_t ldo) {
  memset(g, 0, sizeof(*g));
  g->a = a; g->a_row_stride = K; g->a_seg_stride = 0; g->a_rows = static_cast<int32_t>(M); g->a_cols = K;
  g->P = 1; g->taps = 1; g->kb_per_tap = K / 64; g->a_col_per_nblk = 0;
  g->w = w; g->N = N; g->block_n = 0; g->segs = 1; g->rows_per_seg = static_cast<int32_t>(M);
  g->bias = bias; g->out_f32 = out; g->ldo = ldo; g->out_seg_stride = 0;
}

}  // namespace aptai

using namespace aptai;

extern "C" size_t aptai_pr_head_wide_workspace_bytes(int64_t rows, int H, int V, int backward) {
  if (rows < 1 || H < 64 || V < 1 || V > PH_MAX_V) return 0;
  return ph_ws(rows, H, V, backward).total();
}

extern "C" int aptai_pr_head_wide(const float* h, int64_t rows, int H, const float* w, const float* b, int V,
                                  float* out, int64_t ld_out, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(h && w && out && ws, "pr_head_wide: null pointer");
  APTAI_REQUIRE(V >= 1 && V <= PH_MAX_V, "pr_head_wide: V=%d outside 1..%d (the wide head's limit of %d symbols)", V,
                PH_MAX_V, PH_MAX_V);
  APTAI_REQUIRE(rows >= 1 && rows <= 0x7fffffff, "pr_head_wide: rows=%lld", static_cast<long long>(rows));
  APTAI_REQUIRE(H >= 64 && H % 64 == 0, "pr_head_wide: H=%d must be a positive multiple of 64", H);
  const int64_t Vp = ph_pad_v(V);
  APTAI_REQUIRE(ld_out >= Vp && ld_out % 8 == 0,
                "pr_head_wide: ld_out=%lld must cover the padded width %lld and be a multiple of 8",
                static_cast<long long>(ld_out), static_cast<long long>(Vp));
  const PhWs L = ph_ws(rows, H, V, 0);
  APTAI_REQUIRE(ws_bytes >= L.total() && (reinterpret_cast<uintptr_t>(ws) & (PH_ALIGN - 1)) == 0,
                "pr_head_wide: workspace of %zu bytes (256-byte aligned) needed, got %zu", L.total(), ws_bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* p = static_cast<uint8_t*>(ws);
  void* h3 = p;
  void* w3 = p + L.a;
  float* bp = reinterpret_cast<float*>(p + L.a + L.b);
  if (int rc = launch_split3_pad(h, rows, H, H, 1, rows, H, 0, h3, st)) return rc;
  if (int rc = launch_split3_pad(w, V, H, H, 1, Vp, H, 1, w3, st)) return rc;
  if (b) {
    if (cudaError_t e = cudaMemsetAsync(bp + V, 0, (Vp - V) * sizeof(float), st)) return static_cast<int>(e);
    if (cudaError_t e = cudaMemcpyAsync(bp, b, V * sizeof(float), cudaMemcpyDeviceToDevice, st))
      return static_cast<int>(e);
  }
  aptai_gemm_args g;
  ph_gemm_args(&g, h3, rows, 3 * H, w3, static_cast<int>(Vp), b ? bp : nullptr, out, ld_out);
  return aptai_gemm_bf16(&g, stream);
}

extern "C" int aptai_logits_rows(const float* x, int64_t rows, int V, int64_t ldx, float* logits, int64_t* argmax,
                                 float* logp, float* prob, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(x && (logits || argmax || logp || prob), "logits_rows: null input or no output");
  APTAI_REQUIRE(V >= 1 && V <= PH_MAX_V, "logits_rows: V=%d outside 1..%d (32 values per lane, limit %d)", V, PH_MAX_V,
                PH_MAX_V);
  APTAI_REQUIRE(rows >= 1 && ldx >= V, "logits_rows: rows=%lld, ldx=%lld < V", static_cast<long long>(rows),
                static_cast<long long>(ldx));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int grid = ph_grid(rows, 8, num_sms() * 8);
  long long* am = reinterpret_cast<long long*>(argmax);
  if (V <= 64)
    logits_rows_kernel<2><<<grid, 256, 0, st>>>(x, rows, V, ldx, logits, am, logp, prob);
  else if (V <= 128)
    logits_rows_kernel<4><<<grid, 256, 0, st>>>(x, rows, V, ldx, logits, am, logp, prob);
  else if (V <= 256)
    logits_rows_kernel<8><<<grid, 256, 0, st>>>(x, rows, V, ldx, logits, am, logp, prob);
  else if (V <= 512)
    logits_rows_kernel<16><<<grid, 256, 0, st>>>(x, rows, V, ldx, logits, am, logp, prob);
  else
    logits_rows_kernel<32><<<grid, 256, 0, st>>>(x, rows, V, ldx, logits, am, logp, prob);
  return after_launch("logits_rows");
}

extern "C" int aptai_pr_head_wide_bwd(const float* h, int64_t rows, int H, const float* w, int V, const float* d_logits,
                                      int64_t ld_d, float* dh, float* dw, float* db, void* ws, size_t ws_bytes,
                                      void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(h && w && d_logits && ws && (dh || dw || db), "pr_head_wide_bwd: null pointer or no output");
  APTAI_REQUIRE(V >= 1 && V <= PH_MAX_V, "pr_head_wide_bwd: V=%d outside 1..%d (the wide head's limit of %d symbols)",
                V, PH_MAX_V, PH_MAX_V);
  APTAI_REQUIRE(rows >= 1 && rows <= 0x7fffffff && ld_d >= V, "pr_head_wide_bwd: rows=%lld, ld_d=%lld < V",
                static_cast<long long>(rows), static_cast<long long>(ld_d));
  APTAI_REQUIRE(H >= 64 && H % 64 == 0, "pr_head_wide_bwd: H=%d must be a positive multiple of 64", H);
  const int64_t Vp = ph_pad_v(V);
  const PhWs L = ph_ws(rows, H, V, 1);
  APTAI_REQUIRE(ws_bytes >= L.total() && (reinterpret_cast<uintptr_t>(ws) & (PH_ALIGN - 1)) == 0,
                "pr_head_wide_bwd: workspace of %zu bytes (256-byte aligned) needed, got %zu", L.total(), ws_bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* p = static_cast<uint8_t*>(ws);
  void* dy3 = p;
  void* wt3 = p + L.a;
  void* h3 = p + L.a + L.b;
  if (dh || dw)
    if (int rc = launch_split3_pad(d_logits, rows, V, ld_d, 1, rows, static_cast<int>(Vp), 0, dy3, st)) return rc;
  if (dh) {
    if (int rc = launch_split3_pad(w, H, V, 1, H, H, static_cast<int>(Vp), 1, wt3, st)) return rc;
    aptai_gemm_args g;
    ph_gemm_args(&g, dy3, rows, static_cast<int>(3 * Vp), wt3, H, nullptr, dh, H);
    if (int rc = aptai_gemm_bf16(&g, stream)) return rc;
  }
  if (dw) {
    if (int rc = launch_split3_pad(h, rows, H, H, 1, rows, H, 0, h3, st)) return rc;
    const __nv_bfloat16* y = static_cast<const __nv_bfloat16*>(dy3);
    const __nv_bfloat16* x = static_cast<const __nv_bfloat16*>(h3);
    const int64_t ly = 3 * Vp, lx = 3 * H;
    // (dY_hi, h_hi), (dY_lo, h_hi), (dY_hi, h_lo): column blocks of the [hi | lo | hi] splits
    const int64_t yo[3] = {0, Vp, 0}, xo[3] = {0, 2 * H, H};
    for (int t = 0; t < 3; ++t)
      if (int rc = wgrad_bf16_rows(y + yo[t], ly, x + xo[t], lx, rows, static_cast<int>(Vp), H, 1.f, dw, H, V, stream))
        return rc;
  }
  if (db) {
    const int cb = (V + 31) / 32;
    long long slabs = (4LL * num_sms() + cb - 1) / cb;
    if (slabs > (rows + 255) / 256) slabs = (rows + 255) / 256;
    const long long rps = (rows + slabs - 1) / slabs;
    colsum_pitch_kernel<<<dim3(cb, static_cast<unsigned>((rows + rps - 1) / rps)), 256, 0, st>>>(d_logits, rows, V,
                                                                                              ld_d, rps, db);
    return after_launch("pr_head_colsum");
  }
  return 0;
}
