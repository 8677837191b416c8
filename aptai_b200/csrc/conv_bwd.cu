// Training of the conv feature encoder ('layer' norm variant: HF:275-299, conv -> LayerNorm over channels -> GELU).
// When the feature encoder is NOT frozen (the reference's default for recogniser training,
// train/train_phoneme_recognizer.py:170) the training forward keeps the conv outputs z_i (16-bit) un-normalised and
// applies LayerNorm + GELU in a separate streaming kernel, so that the backward can recompute everything it needs:
//
//   ln_gelu_fwd        y = GELU(LN(z))                                  z, y bf16 [rows][512]
//   ln_gelu_bwd        dz = LN'( dy * GELU'(LN(z)) ), dgamma, dbeta      z from memory, or recomputed from the waveform
//                                                                       for conv layer 0 (10 taps, stride 5: cheaper than
//                                                                       keeping the largest activation of the model)
//   conv0_im2col       waveform -> bf16 [frames][64] (10 taps, zero padded): conv-0's weight gradient is then the
//                      tcgen05 wgrad GEMM dW0 = dz0^T X
// The conv weight gradients of layers 1..6 are aptai_conv_wgrad_bf16 (gemm_tn.cu), the input gradients plain GEMMs on
// per-tap transposed weights with strided output rows (gemm_tc.cu).
#include "common.h"
#include "ptx.cuh"

#include <math.h>

namespace aptai {

constexpr int CB_C = 512;          // channels of every conv layer (validated by the host)

struct RowMap {                    // logical row r of segment s lives at physical row s * seg_pitch + r
  long long rows_per_seg, seg_pitch;
};

__device__ __forceinline__ long long phys_row(long long row, const RowMap& m) {
  const long long s = row / m.rows_per_seg;
  return s * m.seg_pitch + (row - s * m.rows_per_seg);
}

// one warp per row; lane l owns channels {i*128 + l*4 .. +4}, i = 0..3
__device__ __forceinline__ void load_row16(const __nv_bfloat16* p, int lane, float4 (&v)[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p) + i * 32 + lane);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    v[i] = make_float4(a.x, a.y, b.x, b.y);
  }
}

__device__ __forceinline__ void row_stats(float4 (&v)[4], float eps, float& rstd) {   // v <- v - mean
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * (1.0f / CB_C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  rstd = rsqrtf(q * (1.0f / CB_C) + eps);
}

__global__ void __launch_bounds__(256)
ln_gelu_fwd_kernel(const __nv_bfloat16* __restrict__ z, long long rows, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  float4 v[4];
  load_row16(z + row * CB_C, lane, v);
  float rstd;
  row_stats(v, eps, rstd);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i * 32 + lane);
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i * 32 + lane);
    const float a0 = gelu_erf(fmaf(v[i].x * rstd, g.x, b.x)), a1 = gelu_erf(fmaf(v[i].y * rstd, g.y, b.y));
    const float a2 = gelu_erf(fmaf(v[i].z * rstd, g.z, b.z)), a3 = gelu_erf(fmaf(v[i].w * rstd, g.w, b.w));
    reinterpret_cast<uint2*>(y + row * CB_C)[i * 32 + lane] = make_uint2(pack_bf16(a0, a1), pack_bf16(a2, a3));
  }
}

// dz = LN'(dy * GELU'(LN(z))) (bf16), dgamma += sum g * xhat, dbeta += sum g   with g = dy * GELU'(LN(z)).
// FROM_WAV: z[c] = bias[c] + sum_k w0[c][k] * wav[5 t + k] is recomputed (conv layer 0); w0t is [10][512].
template <bool FROM_WAV>
__global__ void __launch_bounds__(256)
ln_gelu_bwd_kernel(const float* __restrict__ dy, RowMap dy_map, const __nv_bfloat16* __restrict__ z,
                   const float* __restrict__ wav, long long wav_ld, const float* __restrict__ w0t,
                   const float* __restrict__ bias0, long long rows, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ dz,
                   float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 ag[4], ab[4], gm[4], bt[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    ag[i] = ab[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    gm[i] = __ldg(reinterpret_cast<const float4*>(gamma) + i * 32 + lane);
    bt[i] = __ldg(reinterpret_cast<const float4*>(beta) + i * 32 + lane);
  }
  for (long long row = static_cast<long long>(blockIdx.x) * 8 + warp; row < rows;
       row += static_cast<long long>(gridDim.x) * 8) {
    float4 v[4], d[4];
    if (FROM_WAV) {
      const long long b = row / dy_map.rows_per_seg, t = row - b * dy_map.rows_per_seg;
      const float* x = wav + b * wav_ld + 5 * t;
      float xs[10];
#pragma unroll
      for (int k = 0; k < 10; ++k) xs[k] = __ldg(x + k);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        v[i] = bias0 ? __ldg(reinterpret_cast<const float4*>(bias0) + i * 32 + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 10; ++k) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(w0t + k * CB_C) + i * 32 + lane);
          v[i].x = fmaf(w.x, xs[k], v[i].x); v[i].y = fmaf(w.y, xs[k], v[i].y);
          v[i].z = fmaf(w.z, xs[k], v[i].z); v[i].w = fmaf(w.w, xs[k], v[i].w);
        }
      }
    } else {
      load_row16(z + row * CB_C, lane, v);
    }
    const float4* dp = reinterpret_cast<const float4*>(dy + phys_row(row, dy_map) * CB_C);
#pragma unroll
    for (int i = 0; i < 4; ++i) d[i] = __ldg(dp + i * 32 + lane);
    float rstd;
    row_stats(v, eps, rstd);
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;                        // xhat
      d[i].x *= gelu_erf_grad(fmaf(v[i].x, gm[i].x, bt[i].x)); d[i].y *= gelu_erf_grad(fmaf(v[i].y, gm[i].y, bt[i].y));
      d[i].z *= gelu_erf_grad(fmaf(v[i].z, gm[i].z, bt[i].z)); d[i].w *= gelu_erf_grad(fmaf(v[i].w, gm[i].w, bt[i].w));
      ag[i].x = fmaf(d[i].x, v[i].x, ag[i].x); ag[i].y = fmaf(d[i].y, v[i].y, ag[i].y);
      ag[i].z = fmaf(d[i].z, v[i].z, ag[i].z); ag[i].w = fmaf(d[i].w, v[i].w, ag[i].w);
      ab[i].x += d[i].x; ab[i].y += d[i].y; ab[i].z += d[i].z; ab[i].w += d[i].w;
      d[i].x *= gm[i].x; d[i].y *= gm[i].y; d[i].z *= gm[i].z; d[i].w *= gm[i].w;
      sg += (d[i].x + d[i].y) + (d[i].z + d[i].w);
      sgx += (d[i].x * v[i].x + d[i].y * v[i].y) + (d[i].z * v[i].z + d[i].w * v[i].w);
    }
    for (int o = 16; o; o >>= 1) {
      sg += __shfl_xor_sync(0xffffffffu, sg, o);
      sgx += __shfl_xor_sync(0xffffffffu, sgx, o);
    }
    const float mg = sg * (1.0f / CB_C), mgx = sgx * (1.0f / CB_C);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float o0 = rstd * (d[i].x - mg - v[i].x * mgx), o1 = rstd * (d[i].y - mg - v[i].y * mgx);
      const float o2 = rstd * (d[i].z - mg - v[i].z * mgx), o3 = rstd * (d[i].w - mg - v[i].w * mgx);
      reinterpret_cast<uint2*>(dz + row * CB_C)[i * 32 + lane] = make_uint2(pack_bf16(o0, o1), pack_bf16(o2, o3));
    }
  }
  __shared__ float sgm[CB_C], sbt[CB_C];
  for (int w = 0; w < 8; ++w) {
    if (warp == w) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4* pg = reinterpret_cast<float4*>(sgm) + i * 32 + lane;
        float4* pb = reinterpret_cast<float4*>(sbt) + i * 32 + lane;
        if (w == 0) {
          *pg = ag[i];
          *pb = ab[i];
        } else {
          float4 a = *pg, b = *pb;
          a.x += ag[i].x; a.y += ag[i].y; a.z += ag[i].z; a.w += ag[i].w;
          b.x += ab[i].x; b.y += ab[i].y; b.z += ab[i].z; b.w += ab[i].w;
          *pg = a;
          *pb = b;
        }
      }
    }
    __syncthreads();
  }
  for (int c = threadIdx.x; c < CB_C; c += 256) {
    atomicAdd(dgamma + c, sgm[c]);
    atomicAdd(dbeta + c, sbt[c]);
  }
}

// X[b*T0 + t][k] = wav[b][5 t + k] (k < 10), 0 (k < 64): the bf16 B operand of conv-0's weight-gradient GEMM
// (64 columns = one TMA box of the wgrad kernel)
__global__ void conv0_im2col_kernel(const float* __restrict__ wav, long long wav_ld, long long T0, long long rows,
                                    __nv_bfloat16* __restrict__ X) {
  for (long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
       r += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = r / T0, t = r - b * T0;
    const float* x = wav + b * wav_ld + 5 * t;
    uint32_t w[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) w[k] = pack_bf16(__ldg(x + 2 * k), __ldg(x + 2 * k + 1));
    uint4* o = reinterpret_cast<uint4*>(X + r * 64);
    o[0] = make_uint4(w[0], w[1], w[2], w[3]);
    o[1] = make_uint4(w[4], 0u, 0u, 0u);
#pragma unroll
    for (int q = 2; q < 8; ++q) o[q] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// ---- 'group' norm variant (base models, HF:308-323: GroupNorm with one group per channel = statistics over time) ----
// layers 1..6 have neither norm nor bias: dz = dy * GELU'(z)
__global__ void gelu_bwd_rows_kernel(const float* __restrict__ dy, RowMap dy_map, const __nv_bfloat16* __restrict__ z,
                                     long long rows, __nv_bfloat16* __restrict__ dz) {
  const long long total = rows * (CB_C / 4);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / (CB_C / 4);
    const int c4 = static_cast<int>(i - row * (CB_C / 4));
    const float4 d = __ldg(reinterpret_cast<const float4*>(dy + phys_row(row, dy_map) * CB_C) + c4);
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(z) + i);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    reinterpret_cast<uint2*>(dz)[i] = make_uint2(pack_bf16(d.x * gelu_erf_grad(a.x), d.y * gelu_erf_grad(a.y)),
                                                 pack_bf16(d.z * gelu_erf_grad(b.x), d.w * gelu_erf_grad(b.y)));
  }
}

// conv layer 0 with GroupNorm: y = GELU(a * zraw + e), a = gamma * rstd, e = (bias - mean) * a + beta per (utterance,
// channel) (the forward's `affine` array), zraw recomputed from the waveform.  xhat = (zraw - mean0) * rstd with
// {mean0, rstd} from the forward's `norm_stats` (mean0 = mean - bias): (ln - beta) / gamma would lose xhat where gamma
// is 0 and cancel where |gamma| << |beta|.  With g = dy * GELU'(ln):
//   PASS 1: sums[b][c] = {sum_t g, sum_t g * xhat}         PASS 2: dz = a * (g - S1/T0 - xhat * S2/T0)   (bf16)
// grid = (frame chunks, B), 256 threads, thread = channels c and c + 256.
template <int PASS>
__global__ void __launch_bounds__(256)
conv0_gn_bwd_kernel(const float* __restrict__ dy, RowMap dy_map, const float* __restrict__ wav, long long wav_ld,
                    const float* __restrict__ w0, const float* __restrict__ affine,
                    const float* __restrict__ norm_stats, int T0, int frames_per_block, float* __restrict__ sums,
                    __nv_bfloat16* __restrict__ dz) {
  const int b = blockIdx.y;
  const int t_begin = blockIdx.x * frames_per_block, t_end = min(T0, t_begin + frames_per_block);
  float w[2][10], a[2], e[2], mu[2], rs[2], s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f}, m1[2], m2[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int c = threadIdx.x + h * 256;
#pragma unroll
    for (int k = 0; k < 10; ++k) w[h][k] = __ldg(w0 + c * 10 + k);
    a[h] = affine[(static_cast<long long>(b) * CB_C + c) * 2];
    e[h] = affine[(static_cast<long long>(b) * CB_C + c) * 2 + 1];
    mu[h] = norm_stats[(static_cast<long long>(b) * CB_C + c) * 2];
    rs[h] = norm_stats[(static_cast<long long>(b) * CB_C + c) * 2 + 1];
    if (PASS == 2) {
      m1[h] = sums[(static_cast<long long>(b) * CB_C + c) * 2] / T0;
      m2[h] = sums[(static_cast<long long>(b) * CB_C + c) * 2 + 1] / T0;
    }
  }
  __shared__ float xs[16];
  for (int t = t_begin; t < t_end; ++t) {
    __syncthreads();
    if (threadIdx.x < 10) xs[threadIdx.x] = __ldg(wav + b * wav_ld + 5LL * t + threadIdx.x);
    __syncthreads();
    const long long prow = phys_row(static_cast<long long>(b) * T0 + t, dy_map);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = threadIdx.x + h * 256;
      float zr = 0.f;
#pragma unroll
      for (int k = 0; k < 10; ++k) zr = fmaf(w[h][k], xs[k], zr);
      const float ln = fmaf(a[h], zr, e[h]);
      const float xhat = (zr - mu[h]) * rs[h];
      const float g = __ldg(dy + prow * CB_C + c) * gelu_erf_grad(ln);
      if (PASS == 1) {
        s1[h] += g;
        s2[h] = fmaf(g, xhat, s2[h]);
      } else {
        dz[(static_cast<long long>(b) * T0 + t) * CB_C + c] = __float2bfloat16(a[h] * (g - m1[h] - xhat * m2[h]));
      }
    }
  }
  if (PASS == 1) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = threadIdx.x + h * 256;
      atomicAdd(sums + (static_cast<long long>(b) * CB_C + c) * 2, s1[h]);
      atomicAdd(sums + (static_cast<long long>(b) * CB_C + c) * 2 + 1, s2[h]);
    }
  }
}

}  // namespace aptai

using namespace aptai;

extern "C" int aptai_gelu_bwd_rows_512(const float* dy, int64_t dy_rows_per_seg, int64_t dy_seg_pitch, const void* z_bf16,
                                       int64_t rows, void* dz_bf16, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(dy && z_bf16 && dz_bf16 && rows >= 1 && dy_rows_per_seg >= 1 && dy_seg_pitch >= dy_rows_per_seg,
                "gelu_bwd_rows: bad arguments");
  RowMap m{dy_rows_per_seg, dy_seg_pitch};
  const long long total = rows * (CB_C / 4);
  int gx = static_cast<int>((total + 255) / 256);
  if (gx > 16384) gx = 16384;
  gelu_bwd_rows_kernel<<<gx, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      dy, m, reinterpret_cast<const __nv_bfloat16*>(z_bf16), rows, reinterpret_cast<__nv_bfloat16*>(dz_bf16));
  return after_launch("gelu_bwd_rows");
}

extern "C" int aptai_conv0_groupnorm_bwd(const float* dy, int64_t dy_seg_pitch, const float* wav, int B, int64_t L,
                                         int T0, const float* w0, const float* affine, const float* norm_stats,
                                         float* sums, void* dz_bf16, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(dy && wav && w0 && affine && norm_stats && sums && dz_bf16, "conv0_groupnorm_bwd: null pointer");
  APTAI_REQUIRE(B >= 1 && T0 >= 1 && dy_seg_pitch >= T0 && 5LL * (T0 - 1) + 10 <= L, "conv0_groupnorm_bwd: bad shape");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(sums, 0, static_cast<size_t>(B) * CB_C * 2 * sizeof(float), st);
  if (e != cudaSuccess) {
    set_error("conv0_groupnorm_bwd: memset: %s", cudaGetErrorString(e));
    return static_cast<int>(e);
  }
  RowMap m{T0, dy_seg_pitch};
  const int fpb = 128;
  dim3 grid((T0 + fpb - 1) / fpb, B);
  __nv_bfloat16* dz = reinterpret_cast<__nv_bfloat16*>(dz_bf16);
  conv0_gn_bwd_kernel<1><<<grid, 256, 0, st>>>(dy, m, wav, L, w0, affine, norm_stats, T0, fpb, sums, dz);
  if (int rc = after_launch("conv0_gn_bwd_sums")) return rc;
  conv0_gn_bwd_kernel<2><<<grid, 256, 0, st>>>(dy, m, wav, L, w0, affine, norm_stats, T0, fpb, sums, dz);
  return after_launch("conv0_gn_bwd");
}

extern "C" int aptai_ln_gelu_fwd_512(const void* z_bf16, int64_t rows, const float* gamma, const float* beta, float eps,
                                     void* y_bf16, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(z_bf16 && gamma && beta && y_bf16 && rows >= 1, "ln_gelu_fwd: bad arguments");
  ln_gelu_fwd_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(z_bf16), rows, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(y_bf16));
  return after_launch("ln_gelu_fwd");
}

extern "C" int aptai_ln_gelu_bwd_512(const float* dy, int64_t dy_rows_per_seg, int64_t dy_seg_pitch, const void* z_bf16,
                                     const float* wav, int64_t wav_ld, const float* w0t, const float* bias0,
                                     int64_t rows, const float* gamma, const float* beta, float eps, void* dz_bf16,
                                     float* dgamma, float* dbeta, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(dy && gamma && beta && dz_bf16 && dgamma && dbeta && rows >= 1, "ln_gelu_bwd: null pointer");
  APTAI_REQUIRE((z_bf16 != nullptr) != (wav != nullptr && w0t != nullptr), "ln_gelu_bwd: give z, or wav + w0t (conv 0)");
  APTAI_REQUIRE(dy_rows_per_seg >= 1 && dy_seg_pitch >= dy_rows_per_seg, "ln_gelu_bwd: bad row map");
  APTAI_REQUIRE(z_bf16 || 5 * (dy_rows_per_seg - 1) + 10 <= wav_ld,
                "ln_gelu_bwd: %lld frames need %lld samples per utterance, the waveform has %lld",
                (long long)dy_rows_per_seg, 5LL * (dy_rows_per_seg - 1) + 10, (long long)wav_ld);
  RowMap m{dy_rows_per_seg, dy_seg_pitch};
  long long blocks = (rows + 7) / 8;
  const long long cap = 8LL * num_sms();
  if (blocks > cap) blocks = cap;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  __nv_bfloat16* dz = reinterpret_cast<__nv_bfloat16*>(dz_bf16);
  if (z_bf16)
    ln_gelu_bwd_kernel<false><<<static_cast<unsigned>(blocks), 256, 0, st>>>(
        dy, m, reinterpret_cast<const __nv_bfloat16*>(z_bf16), nullptr, 0, nullptr, nullptr, rows, gamma, beta, eps, dz,
        dgamma, dbeta);
  else
    ln_gelu_bwd_kernel<true><<<static_cast<unsigned>(blocks), 256, 0, st>>>(dy, m, nullptr, wav, wav_ld, w0t, bias0, rows,
                                                                         gamma, beta, eps, dz, dgamma, dbeta);
  return after_launch("ln_gelu_bwd");
}

extern "C" int aptai_conv0_im2col_bf16(const float* wav, int B, int64_t L, int64_t T0, void* x_bf16, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(wav && x_bf16 && B >= 1 && T0 >= 1 && 5 * (T0 - 1) + 10 <= L, "conv0_im2col: bad arguments");
  const long long rows = static_cast<long long>(B) * T0;
  int gx = static_cast<int>((rows + 255) / 256);
  if (gx > 8192) gx = 8192;
  conv0_im2col_kernel<<<gx, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(wav, L, T0, rows,
                                                                               reinterpret_cast<__nv_bfloat16*>(x_bf16));
  return after_launch("conv0_im2col");
}
