// Accuracy mode ("f32x3") support kernels.
//
// The default path feeds the tensor cores bf16 / fp16 operands (2^-9 / 2^-12 relative rounding per operand), which
// keeps the articulatory trajectories inside the north-star tolerance but flips the phoneme argmax on near-tie frames
// of an untrained head (SURVEY.md Appendix D).  The accuracy mode keeps every activation in fp32 and runs every
// contraction on the SAME tcgen05 GEMM kernels as three bf16 products:
//     x = x_hi + x_lo,  w = w_hi + w_lo   (bf16 pairs, 16 mantissa bits together)
//     x . w  ~=  x_hi.w_hi + x_lo.w_hi + x_hi.w_lo            (dropped x_lo.w_lo ~ 2^-18 relative)
// by laying the operands out as  A' = [x_hi | x_lo | x_hi]  (K tripled) and  W' = [w_hi | w_hi | w_lo].
// This file holds the streaming kernels around those GEMMs: the hi/lo split, LayerNorm / GELU with split output,
// the fp32 attention (SIMT: the softmax(QK^T)V chain on fp32 operands), and the positional-conv tail.
// Replaces the same reference lines as their default-path twins (HF:254-323 conv norms, HF:429-434, HF:500-549,
// HF:566-573, HF:600-655 LayerNorms).
#include "common.h"
#include "ptx.cuh"

namespace aptai {

// out[r] = [hi | lo | hi] (mode 0, activations) or [hi | hi | lo] (mode 1, weights); x may be strided by ld_in.
__global__ void split3_kernel(const float* __restrict__ x, long long rows, int cols, long long ld_in, int mode,
                              float scale, __nv_bfloat16* __restrict__ out) {
  const long long total = rows * cols;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i - r * cols);
    __nv_bfloat16 hi, lo;
    split_bf16(x[r * ld_in + c] * scale, hi, lo);
    __nv_bfloat16* o = out + r * 3 * cols + c;
    o[0] = hi;
    o[cols] = mode ? hi : lo;
    o[2 * cols] = mode ? lo : hi;
  }
}

// Row operator, warp per row, row in registers: (optional LayerNorm, exact two-pass statistics) -> (optional erf-GELU)
// -> fp32 and / or split-bf16 outputs.  cols <= 1024, multiple of 32.
template <int NV>
__global__ void __launch_bounds__(256)
rowop_split3_kernel(const float* __restrict__ x, long long rows, const float* __restrict__ gamma,
                    const float* __restrict__ beta, float eps, int norm, int gelu, float* __restrict__ out_f32,
                    __nv_bfloat16* __restrict__ out3) {
  constexpr int COLS = NV * 32;
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * COLS;
  float v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = xr[i * 32 + lane];
  if (norm) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) s += v[i];
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.0f / COLS);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float d = v[i] - mean;
      q = fmaf(d, d, q);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = 1.0f / sqrtf(q * (1.0f / COLS) + eps);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = fmaf((v[i] - mean) * rstd, gamma[i * 32 + lane], beta[i * 32 + lane]);
  }
  if (gelu) {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = gelu_erf(v[i]);
  }
  if (out_f32) {
#pragma unroll
    for (int i = 0; i < NV; ++i) out_f32[row * COLS + i * 32 + lane] = v[i];
  }
  if (out3) {
    __nv_bfloat16* o = out3 + row * 3 * COLS;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      __nv_bfloat16 hi, lo;
      split_bf16(v[i], hi, lo);
      const int c = i * 32 + lane;
      o[c] = hi;
      o[COLS + c] = lo;
      o[2 * COLS + c] = hi;
    }
  }
}

// out = res + gelu(x)   (positional conv tail, HF:360-368 + the residual add of HF:690|764)
__global__ void gelu_add_kernel(const float* __restrict__ x, const float* __restrict__ res, long long n,
                                float* __restrict__ out) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    out[i] = res[i] + gelu_erf(x[i]);
}

// fp32 -> two zero-haloed bf16 copies (hi, lo) for the positional conv's shifted-window operand
__global__ void cast_pad_split_kernel(const float* __restrict__ x, int rows, int cols, int halo,
                                      __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int seg = blockIdx.y;
  const long long prow = rows + 2 * halo;
  const long long total = prow * cols;
  const float* in = x + static_cast<long long>(seg) * rows * cols;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols - halo;
    __nv_bfloat16 h = __float2bfloat16_rn(0.f), l = h;
    if (r >= 0 && r < rows) split_bf16(in[r * cols + (i % cols)], h, l);
    hi[seg * total + i] = h;
    lo[seg * total + i] = l;
  }
}

// Folded weight-norm of the positional conv, split: w[o][j][c] = g[j] * v[o][c][j] / ||v[:, :, j]||  (HF:336-358)
__global__ void posconv_fold_split_kernel(const float* __restrict__ g, const float* __restrict__ v,
                                          const float* __restrict__ norm, int H, int cin, int taps, int cpad,
                                          __nv_bfloat16* __restrict__ w_hi, __nv_bfloat16* __restrict__ w_lo) {
  const long long total = static_cast<long long>(H) * taps * cpad;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % cpad);
    const int j = static_cast<int>((i / cpad) % taps);
    const long long o = i / (static_cast<long long>(cpad) * taps);
    float val = 0.f;
    if (c < cin) val = g[j] * v[(o * cin + c) * taps + j] / norm[j];
    split_bf16(val, w_hi[i], w_lo[i]);
  }
}

__global__ void posconv_norm64_kernel(const float* __restrict__ v, int n_oc, int taps, float* __restrict__ norm) {
  const int j = blockIdx.x;
  double s = 0;
  for (int i = threadIdx.x; i < n_oc; i += blockDim.x) {
    const double a = v[static_cast<long long>(i) * taps + j];
    s += a * a;
  }
  __shared__ double red[256];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) norm[j] = static_cast<float>(sqrt(red[0]));
}

// ------------------------------------------------------------------------------------------------ fp32 attention
// softmax(q k^T + key mask) v on fp32 operands (HF:500-549; q pre-scaled by head_dim^-0.5 through its weights).
// CTA = 128 queries of one (utterance, head); thread = query row (q, the output accumulator and one tile of scores
// in registers); keys / values stream through shared memory in tiles of 32 and are read as broadcasts.
constexpr int AF_Q = 128, AF_K = 32, AF_D = 64;

__global__ void __launch_bounds__(AF_Q)
attention_f32_kernel(const float* __restrict__ qkv, const int* __restrict__ key_len, int T, int heads,
                     float* __restrict__ ctx) {
  __shared__ __align__(16) float ks[AF_K][AF_D];
  __shared__ __align__(16) float vs[AF_K][AF_D];
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * AF_Q;
  const int H = heads * AF_D;
  const long long ld = 3LL * H;
  const int tq = q0 + threadIdx.x;
  const bool active = tq < T;
  const int nk = min(key_len[b], T);
  const float* base = qkv + static_cast<long long>(b) * T * ld + h * AF_D;
  float q[AF_D], o[AF_D];
#pragma unroll
  for (int d = 0; d < AF_D; d += 4) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active) t = *reinterpret_cast<const float4*>(base + tq * ld + d);
    const float L2E = 1.4426950408889634f;
    q[d] = t.x * L2E; q[d + 1] = t.y * L2E; q[d + 2] = t.z * L2E; q[d + 3] = t.w * L2E;
    o[d] = o[d + 1] = o[d + 2] = o[d + 3] = 0.f;
  }
  float m = -INFINITY, l = 0.f;
  for (int k0 = 0; k0 < nk; k0 += AF_K) {
    __syncthreads();
    for (int i = threadIdx.x; i < AF_K * AF_D / 4; i += AF_Q) {
      const int kr = i / (AF_D / 4), c4 = i % (AF_D / 4);
      float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
      if (k0 + kr < nk) {
        const float* rowp = base + static_cast<long long>(k0 + kr) * ld + c4 * 4;
        kk = *reinterpret_cast<const float4*>(rowp + H);
        vv = *reinterpret_cast<const float4*>(rowp + 2 * H);
      }
      *reinterpret_cast<float4*>(&ks[kr][c4 * 4]) = kk;
      *reinterpret_cast<float4*>(&vs[kr][c4 * 4]) = vv;
    }
    __syncthreads();
    const int kn = min(AF_K, nk - k0);
    float s[AF_K];
    float tmax = -INFINITY;
#pragma unroll
    for (int j = 0; j < AF_K; ++j) {
      float a0 = 0.f, a1 = 0.f;
#pragma unroll
      for (int d = 0; d < AF_D; d += 4) {
        const float4 kk = *reinterpret_cast<const float4*>(&ks[j][d]);
        a0 = fmaf(q[d], kk.x, a0); a1 = fmaf(q[d + 1], kk.y, a1);
        a0 = fmaf(q[d + 2], kk.z, a0); a1 = fmaf(q[d + 3], kk.w, a1);
      }
      s[j] = j < kn ? a0 + a1 : -INFINITY;
      tmax = fmaxf(tmax, s[j]);
    }
    const float mn = fmaxf(m, tmax);
    const float corr = exp2f(m - mn);          // m = -inf on the first tile: exp2(-inf) = 0
    l *= corr;
#pragma unroll
    for (int d = 0; d < AF_D; ++d) o[d] *= corr;
    m = mn;
#pragma unroll
    for (int j = 0; j < AF_K; ++j) {
      const float p = exp2f(s[j] - m);         // masked keys: exp2(-inf) = 0
      l += p;
#pragma unroll
      for (int d = 0; d < AF_D; d += 4) {
        const float4 vv = *reinterpret_cast<const float4*>(&vs[j][d]);
        o[d] = fmaf(p, vv.x, o[d]); o[d + 1] = fmaf(p, vv.y, o[d + 1]);
        o[d + 2] = fmaf(p, vv.z, o[d + 2]); o[d + 3] = fmaf(p, vv.w, o[d + 3]);
      }
    }
  }
  if (active) {
    const float inv = l > 0.f ? 1.0f / l : 0.f;
    float* op = ctx + (static_cast<long long>(b) * T + tq) * H + h * AF_D;
#pragma unroll
    for (int d = 0; d < AF_D; d += 4)
      *reinterpret_cast<float4*>(op + d) = make_float4(o[d] * inv, o[d + 1] * inv, o[d + 2] * inv, o[d + 3] * inv);
  }
}

}  // namespace aptai

using namespace aptai;

static int grid_for(long long total, int cap = 8192) {
  long long g = (total + 255) / 256;
  return static_cast<int>(g > cap ? cap : (g < 1 ? 1 : g));
}

extern "C" int aptai_split3_bf16(const float* x, int64_t rows, int cols, int64_t ld_in, int weight_layout, float scale,
                                 void* out_bf16, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(x && out_bf16 && rows >= 1 && cols >= 1 && ld_in >= cols, "split3: bad arguments");
  split3_kernel<<<grid_for(rows * cols), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, rows, cols, ld_in, weight_layout, scale, reinterpret_cast<__nv_bfloat16*>(out_bf16));
  return after_launch("split3_bf16");
}

extern "C" int aptai_rowop_split3(const float* x, int64_t rows, int cols, const float* gamma, const float* beta,
                                  float eps, int norm, int gelu, float* out_f32, void* out_split3, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(x && rows >= 1 && (out_f32 || out_split3), "rowop_split3: bad arguments");
  APTAI_REQUIRE(!norm || (gamma && beta), "rowop_split3: LayerNorm needs gamma / beta");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
  __nv_bfloat16* o3 = reinterpret_cast<__nv_bfloat16*>(out_split3);
  switch (cols) {
    case 256: rowop_split3_kernel<8><<<grid, 256, 0, st>>>(x, rows, gamma, beta, eps, norm, gelu, out_f32, o3); break;
    case 512: rowop_split3_kernel<16><<<grid, 256, 0, st>>>(x, rows, gamma, beta, eps, norm, gelu, out_f32, o3); break;
    case 768: rowop_split3_kernel<24><<<grid, 256, 0, st>>>(x, rows, gamma, beta, eps, norm, gelu, out_f32, o3); break;
    case 1024: rowop_split3_kernel<32><<<grid, 256, 0, st>>>(x, rows, gamma, beta, eps, norm, gelu, out_f32, o3); break;
    default:
      set_error("rowop_split3: cols=%d unsupported (256, 512, 768, 1024)", cols);
      return APTAI_ERR_ARG;
  }
  return after_launch("rowop_split3");
}

extern "C" int aptai_gelu_add_f32(const float* x, const float* res, int64_t n, float* out, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(x && res && out && n >= 1, "gelu_add: bad arguments");
  gelu_add_kernel<<<grid_for(n), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, res, n, out);
  return after_launch("gelu_add_f32");
}

extern "C" int aptai_cast_pad_split(const float* x, int segs, int rows, int cols, int halo, void* hi_bf16, void* lo_bf16,
                                    void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(x && hi_bf16 && lo_bf16 && segs >= 1 && rows >= 1 && cols >= 1 && halo >= 0, "cast_pad_split: bad arguments");
  const long long total = static_cast<long long>(rows + 2 * halo) * cols;
  cast_pad_split_kernel<<<dim3(grid_for(total, 4096), segs), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, rows, cols, halo, reinterpret_cast<__nv_bfloat16*>(hi_bf16), reinterpret_cast<__nv_bfloat16*>(lo_bf16));
  return after_launch("cast_pad_split");
}

extern "C" int aptai_posconv_fold_split(const float* g, const float* v, int H, int cin, int taps, int cpad, void* w_hi,
                                        void* w_lo, float* norm_ws, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(g && v && w_hi && w_lo && norm_ws, "posconv_fold_split: null pointer");
  APTAI_REQUIRE(cpad >= cin && H >= 1 && taps >= 1, "posconv_fold_split: bad shape");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  posconv_norm64_kernel<<<taps, 256, 0, st>>>(v, H * cin, taps, norm_ws);
  if (int rc = after_launch("posconv_norm")) return rc;
  const long long total = static_cast<long long>(H) * taps * cpad;
  posconv_fold_split_kernel<<<grid_for(total), 256, 0, st>>>(g, v, norm_ws, H, cin, taps, cpad,
                                                              reinterpret_cast<__nv_bfloat16*>(w_hi),
                                                              reinterpret_cast<__nv_bfloat16*>(w_lo));
  return after_launch("posconv_fold_split");
}

extern "C" int aptai_attention_fwd_f32(const float* qkv, float* ctx, const int32_t* key_len, int B, int T, int heads,
                                       void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(qkv && ctx && key_len && B >= 1 && T >= 1 && heads >= 1, "attention_fwd_f32: bad arguments");
  dim3 grid((T + AF_Q - 1) / AF_Q, heads, B);
  attention_f32_kernel<<<grid, AF_Q, 0, reinterpret_cast<cudaStream_t>(stream)>>>(qkv, key_len, T, heads, ctx);
  return after_launch("attention_fwd_f32");
}
