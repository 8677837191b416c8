// Feature-encoder front end: conv layer 0 (1 -> 512 channels, k=10, s=5) fused with its normalisation and GELU,
// writing channels-last bf16 [B][T0][512] so that conv layers 1..6 can run as implicit GEMM on the tensor cores.
//
// HBM-bound by design (K=10 is not a tensor-core shape): 2 B written per output element, the waveform is read
// once through shared memory.  Normalisation statistics never touch the conv output:
//   * LayerNorm over channels (HF:281-299, 'layer' variant): mean/var over the 512 channels of one frame are a
//     linear / quadratic form of the frame's 10 samples:  mean = wbar.x + bbar,
//     var = x' Gc x + 2 gc.x + vb  with Gc the (centred) 10x10 channel-covariance of the weights.
//   * GroupNorm(512 groups of 1 channel) over time (HF:308-323, 'group' variant): mean/var over the T0 frames of
//     one channel are a linear / quadratic form of that channel's 10 weights in the strided autocorrelation of
//     the waveform, accumulated in fp64.  Statistics run over the whole padded row, as in the reference.
#include "common.h"
#include "ptx.cuh"

namespace aptai {

constexpr int C0 = 512;      // conv_dim[0]
constexpr int K0 = 10;       // conv_kernel[0]
constexpr int S0 = 5;        // conv_stride[0]
constexpr int FT = 64;       // frames per block
constexpr int NQ = K0 * (K0 + 1) / 2;   // 55 unique entries of a symmetric 10x10

// consts layout (floats): [0,10) wbar | [10] bbar | [11,21) gc | [21] vb | [32, 32+100) Gc row-major
__global__ void conv0_ln_consts_kernel(const float* __restrict__ w, const float* __restrict__ bias,
                                       float* __restrict__ consts) {
  __shared__ double wbar[K0];
  __shared__ double bbar;
  const int tid = threadIdx.x;
  if (tid < K0) {
    double s = 0;
    for (int c = 0; c < C0; ++c) s += w[c * K0 + tid];
    wbar[tid] = s / C0;
  }
  if (tid == K0) {
    double s = 0;
    if (bias)
      for (int c = 0; c < C0; ++c) s += bias[c];
    bbar = s / C0;
  }
  __syncthreads();
  if (tid < K0 * K0) {
    const int j = tid / K0, k = tid % K0;
    double s = 0;
    for (int c = 0; c < C0; ++c) s += (w[c * K0 + j] - wbar[j]) * (w[c * K0 + k] - wbar[k]);
    consts[32 + tid] = static_cast<float>(s / C0);
  } else if (tid < K0 * K0 + K0) {
    const int j = tid - K0 * K0;
    double s = 0;
    if (bias)
      for (int c = 0; c < C0; ++c) s += (w[c * K0 + j] - wbar[j]) * (bias[c] - bbar);
    consts[11 + j] = static_cast<float>(s / C0);
    consts[j] = static_cast<float>(wbar[j]);
  } else if (tid == K0 * K0 + K0) {
    double s = 0;
    if (bias)
      for (int c = 0; c < C0; ++c) s += (bias[c] - bbar) * (bias[c] - bbar);
    consts[21] = static_cast<float>(s / C0);
    consts[10] = static_cast<float>(bbar);
  }
}

// GroupNorm pass A: per utterance sums of x[5t+j] and x[5t+j]*x[5t+k] over the T0 frames (fp64 atomics).
__global__ void conv0_gn_moments_kernel(const float* __restrict__ wav, long long L, int T0, double* __restrict__ mom) {
  const int b = blockIdx.y;
  const float* x = wav + static_cast<long long>(b) * L;
  double s1[K0], s2[NQ];
#pragma unroll
  for (int j = 0; j < K0; ++j) s1[j] = 0;
#pragma unroll
  for (int q = 0; q < NQ; ++q) s2[q] = 0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T0; t += gridDim.x * blockDim.x) {
    float v[K0];
#pragma unroll
    for (int j = 0; j < K0; ++j) v[j] = x[static_cast<long long>(t) * S0 + j];
    int q = 0;
#pragma unroll
    for (int j = 0; j < K0; ++j) {
      s1[j] += v[j];
#pragma unroll
      for (int k = j; k < K0; ++k) s2[q++] += static_cast<double>(v[j]) * v[k];
    }
  }
  __shared__ double red[K0 + NQ];
  if (threadIdx.x < K0 + NQ) red[threadIdx.x] = 0;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < K0; ++j) {
    double v = s1[j];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red[j], v);
  }
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    double v = s2[q];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red[K0 + q], v);
  }
  __syncthreads();
  if (threadIdx.x < K0 + NQ) atomicAdd(&mom[b * (K0 + NQ) + threadIdx.x], red[threadIdx.x]);
}

// GroupNorm pass B: per (utterance, channel) scale/shift so that out = gelu(conv * a + s).  norm_stats (may be NULL)
// receives {mean of the bias-free conv output, rstd}: the backward's xhat = (conv - mean) * rstd, which it cannot
// recover from the scale/shift when gamma is 0 or small.
__global__ void conv0_gn_affine_kernel(const double* __restrict__ mom, const float* __restrict__ w,
                                       const float* __restrict__ bias, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, int T0, float eps, float* __restrict__ affine,
                                       float* __restrict__ norm_stats) {
  const int b = blockIdx.x;
  const int c = threadIdx.x;
  const double* m = mom + b * (K0 + NQ);
  double mu[K0], wc[K0];
#pragma unroll
  for (int j = 0; j < K0; ++j) {
    mu[j] = m[j] / T0;
    wc[j] = w[c * K0 + j];
  }
  double mean = bias ? static_cast<double>(bias[c]) : 0.0;
  double var = 0;
  int q = 0;
#pragma unroll
  for (int j = 0; j < K0; ++j) {
    mean += wc[j] * mu[j];
#pragma unroll
    for (int k = j; k < K0; ++k) {
      const double cov = m[K0 + q] / T0 - mu[j] * mu[k];
      var += (j == k ? 1.0 : 2.0) * wc[j] * wc[k] * cov;
      ++q;
    }
  }
  if (var < 0) var = 0;
  const double rstd = 1.0 / sqrt(var + static_cast<double>(eps));
  const double a = rstd * gamma[c];
  const double conv_bias = bias ? static_cast<double>(bias[c]) : 0.0;
  // y = (conv_nobias + conv_bias - mean) * a + beta
  affine[(b * C0 + c) * 2 + 0] = static_cast<float>(a);
  affine[(b * C0 + c) * 2 + 1] = static_cast<float>((conv_bias - mean) * a + beta[c]);
  if (norm_stats) {
    norm_stats[(b * C0 + c) * 2 + 0] = static_cast<float>(mean - conv_bias);
    norm_stats[(b * C0 + c) * 2 + 1] = static_cast<float>(rstd);
  }
}

// NORM: 0 none, 1 LayerNorm over channels per frame, 2 GroupNorm affine per (utterance, channel)
template <int NORM>
__global__ void __launch_bounds__(256)
conv0_kernel(const float* __restrict__ wav, long long L, int T0, const float* __restrict__ w,
             const float* __restrict__ bias, const float* __restrict__ gamma, const float* __restrict__ beta,
             const float* __restrict__ consts, const float* __restrict__ affine, float eps,
             __nv_bfloat16* __restrict__ out, int out_fp16) {
  // every sample is kept twice, {x, x}: one 8-byte shared load feeds a packed fp32x2 FMA that advances the thread's
  // two channels at once (the kernel is instruction-bound, profiles/r01_launches_b120x8s.md)
  __shared__ __align__(16) float2 xs2[FT * S0 + K0];
  __shared__ __align__(16) float4 fstat[FT];          // {-mean, -mean, rstd, rstd}
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * FT;
  const int nf = min(FT, T0 - t0);
  const float* x = wav + static_cast<long long>(b) * L + static_cast<long long>(t0) * S0;
  const int ns = (nf - 1) * S0 + K0;
  for (int i = threadIdx.x; i < FT * S0 + K0; i += blockDim.x) {
    const float v = i < ns ? x[i] : 0.f;
    xs2[i] = make_float2(v, v);
  }
  __syncthreads();
  if (NORM == 1) {
    if (threadIdx.x < FT) {
      float f[K0];
#pragma unroll
      for (int j = 0; j < K0; ++j) f[j] = xs2[threadIdx.x * S0 + j].x;
      float mean = consts[10];
      float var = consts[21];
#pragma unroll
      for (int j = 0; j < K0; ++j) {
        mean = fmaf(consts[j], f[j], mean);
        float acc = 2.f * consts[11 + j];
#pragma unroll
        for (int k = 0; k < K0; ++k) acc = fmaf(consts[32 + j * K0 + k], f[k], acc);
        var = fmaf(acc, f[j], var);
      }
      const float rstd = rsqrtf(fmaxf(var, 0.f) + eps);
      fstat[threadIdx.x] = make_float4(-mean, -mean, rstd, rstd);
    }
    __syncthreads();
  }
  const int c = threadIdx.x * 2;
  uint64_t w01[K0];
#pragma unroll
  for (int j = 0; j < K0; ++j) w01[j] = f32x2_pack(w[c * K0 + j], w[(c + 1) * K0 + j]);
  float b0 = bias ? bias[c] : 0.f, b1 = bias ? bias[c + 1] : 0.f;
  float g0 = 1.f, g1 = 1.f, e0 = 0.f, e1 = 0.f;
  if (NORM == 1) {
    g0 = gamma[c]; g1 = gamma[c + 1]; e0 = beta[c]; e1 = beta[c + 1];
  } else if (NORM == 2) {
    g0 = affine[(b * C0 + c) * 2]; e0 = affine[(b * C0 + c) * 2 + 1];
    g1 = affine[(b * C0 + c + 1) * 2]; e1 = affine[(b * C0 + c + 1) * 2 + 1];
    b0 = 0.f; b1 = 0.f;   // folded into the shift
  }
  const uint64_t b01 = f32x2_pack(b0, b1), g01 = f32x2_pack(g0, g1), e01 = f32x2_pack(e0, e1);
  uint32_t* o = reinterpret_cast<uint32_t*>(out + (static_cast<long long>(b) * T0 + t0) * C0 + c);
  const uint64_t* xp = reinterpret_cast<const uint64_t*>(xs2);
  for (int f = 0; f < nf; ++f) {
    const uint64_t* xf = xp + f * S0;
    uint64_t y = b01;
#pragma unroll
    for (int j = 0; j < K0; ++j) y = f32x2_fma(w01[j], xf[j], y);
    if (NORM == 1) {
      const ulonglong2 st = *reinterpret_cast<const ulonglong2*>(&fstat[f]);      // {-mean, -mean}, {rstd, rstd}
      y = f32x2_fma(f32x2_mul(f32x2_add(y, st.x), st.y), g01, e01);
    } else if (NORM == 2) {
      y = f32x2_fma(y, g01, e01);
    }
    float y0, y1;
    f32x2_unpack(y, y0, y1);
    gelu_fast2(y0, y1);                  // 16-bit output: see gelu_fast2 (ptx.cuh)
    o[static_cast<long long>(f) * (C0 / 2)] = pack_h16(y0, y1, out_fp16);
  }
}

// Accuracy mode (csrc/accurate.cu): the same layer with plain fp32 arithmetic (two-pass LayerNorm statistics over
// the 512 channels of a frame, warp per frame) and a split-bf16 output [B][T0][hi 512 | lo 512 | hi 512] that feeds
// conv layer 1 as a three-product implicit GEMM.  NORM as above.
template <int NORM>
__global__ void __launch_bounds__(256)
conv0_accurate_kernel(const float* __restrict__ wav, long long L, int T0, const float* __restrict__ w,
                      const float* __restrict__ bias, const float* __restrict__ gamma, const float* __restrict__ beta,
                      const float* __restrict__ affine, float eps, __nv_bfloat16* __restrict__ out3) {
  __shared__ float ws[K0][C0];                 // tap-major copy of the weights
  for (int i = threadIdx.x; i < K0 * C0; i += blockDim.x) ws[i % K0][i / K0] = w[i];
  __syncthreads();
  const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = blockIdx.x * 64 + warp; t < min(T0, blockIdx.x * 64 + 64); t += 8) {
    const float* x = wav + static_cast<long long>(b) * L + static_cast<long long>(t) * S0;
    float xs[K0];
#pragma unroll
    for (int j = 0; j < K0; ++j) xs[j] = __ldg(x + j);
    float y[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = 2 * lane + 64 * i + e;
        float a = 0.f;
#pragma unroll
        for (int j = 0; j < K0; ++j) a = fmaf(ws[j][c], xs[j], a);
        if (NORM == 2) a = fmaf(a, affine[(b * C0 + c) * 2], affine[(b * C0 + c) * 2 + 1]);
        else if (bias) a += bias[c];
        y[2 * i + e] = a;
      }
    }
    if (NORM == 1) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) s += y[i];
#pragma unroll
      for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float mean = s * (1.0f / C0);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float d = y[i] - mean;
        q = fmaf(d, d, q);
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
      const float rstd = 1.0f / sqrtf(q * (1.0f / C0) + eps);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int c = 2 * lane + 64 * i + e;
          y[2 * i + e] = fmaf((y[2 * i + e] - mean) * rstd, gamma[c], beta[c]);
        }
    }
    uint32_t* o = reinterpret_cast<uint32_t*>(out3 + (static_cast<long long>(b) * T0 + t) * 3 * C0);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float g0 = gelu_erf(y[2 * i]), g1 = gelu_erf(y[2 * i + 1]);
      const __nv_bfloat16 h0 = __float2bfloat16_rn(g0), h1 = __float2bfloat16_rn(g1);
      const uint32_t hi = pack_bf16(g0, g1);
      const uint32_t lo = pack_bf16(g0 - __bfloat162float(h0), g1 - __bfloat162float(h1));
      const int cp = lane + 32 * i;            // pair index
      o[cp] = hi;
      o[C0 / 2 + cp] = lo;
      o[C0 + cp] = hi;
    }
  }
}

}  // namespace aptai

using namespace aptai;

extern "C" int aptai_conv0_accurate(const float* wav, int B, int64_t L, const float* w, const float* bias,
                                    const float* gamma, const float* beta, int norm, float eps, void* out_split3,
                                    int T0, float* stats_ws, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(wav && w && out_split3, "conv0_accurate: null pointer");
  APTAI_REQUIRE(B >= 1 && L >= K0 && T0 == (L - K0) / S0 + 1, "conv0_accurate: bad shape B=%d L=%lld T0=%d", B,
                (long long)L, T0);
  APTAI_REQUIRE(norm >= 0 && norm <= 2, "conv0_accurate: norm must be 0, 1 or 2");
  APTAI_REQUIRE(norm == 0 || (gamma && beta), "conv0_accurate: norm needs gamma and beta");
  APTAI_REQUIRE(norm != 2 || stats_ws, "conv0_accurate: GroupNorm needs stats_ws");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 grid((T0 + 63) / 64, B);
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(out_split3);
  if (norm == 2) {
    double* mom = reinterpret_cast<double*>(stats_ws);
    float* affine = reinterpret_cast<float*>(mom + static_cast<size_t>(B) * (K0 + NQ));
    cudaError_t e = cudaMemsetAsync(mom, 0, sizeof(double) * B * (K0 + NQ), st);
    if (e != cudaSuccess) {
      set_error("conv0_accurate: memset: %s", cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    int chunks = (T0 + 256 * 8 - 1) / (256 * 8);
    if (chunks > 64) chunks = 64;
    conv0_gn_moments_kernel<<<dim3(chunks, B), 256, 0, st>>>(wav, L, T0, mom);
    if (int rc = after_launch("conv0_gn_moments")) return rc;
    conv0_gn_affine_kernel<<<B, C0, 0, st>>>(mom, w, bias, gamma, beta, T0, eps, affine, nullptr);
    if (int rc = after_launch("conv0_gn_affine")) return rc;
    conv0_accurate_kernel<2><<<grid, 256, 0, st>>>(wav, L, T0, w, bias, gamma, beta, affine, eps, out);
  } else if (norm == 1) {
    conv0_accurate_kernel<1><<<grid, 256, 0, st>>>(wav, L, T0, w, bias, gamma, beta, nullptr, eps, out);
  } else {
    conv0_accurate_kernel<0><<<grid, 256, 0, st>>>(wav, L, T0, w, bias, gamma, beta, nullptr, eps, out);
  }
  return after_launch("conv0_accurate");
}

namespace aptai {
int conv0_tc_launch(const float* wav, int B, int64_t L, int T0, const float* w, const float* bias, const float* gamma,
                    const float* beta, int norm, float eps, const float* consts, const float* affine, void* ws_b,
                    void* out16, int out_fp16, cudaStream_t st);       // conv0_tc.cu
}

// stats_ws layout: [statistics: norm 1 -> 1 KB of closed-form constants; norm 2 -> B*65 doubles of moments +
// B*512*2 floats of scale/shift + B*512*2 floats of {mean, rstd}; norm 0 -> nothing] then, 256-byte aligned, the
// 64 KB split weight operand of the tensor-core kernel
static size_t conv0_stats_bytes(int B, int norm) {
  const size_t s = norm == 1 ? 1024 : (norm == 2 ? sizeof(double) * B * (K0 + NQ) + sizeof(float) * B * C0 * 4 : 0);
  return (s + 255) / 256 * 256;
}
extern "C" size_t aptai_conv0_workspace_bytes(int B, int norm) { return conv0_stats_bytes(B, norm) + C0 * 64 * 2; }

extern "C" int aptai_conv0_norm_gelu(const float* wav, int B, int64_t L, const float* w, const float* bias,
                                     const float* gamma, const float* beta, int norm, float eps, void* out_bf16,
                                     int T0, float* stats_ws, int flags, void* stream) {
  if (int rc = check_arch()) return rc;
  const int out_fp16 = flags & 1;
  const bool simt = (flags & 2) != 0;
  APTAI_REQUIRE(wav && w && out_bf16 && stats_ws, "conv0: null pointer");
  APTAI_REQUIRE(B >= 1 && L >= K0, "conv0: bad shape B=%d L=%lld", B, (long long)L);
  APTAI_REQUIRE(T0 == (L - K0) / S0 + 1, "conv0: T0=%d does not match L=%lld", T0, (long long)L);
  APTAI_REQUIRE(norm >= 0 && norm <= 2, "conv0: norm must be 0, 1 or 2");
  APTAI_REQUIRE(norm == 0 || (gamma && beta), "conv0: norm needs gamma and beta");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 grid((T0 + FT - 1) / FT, B);
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(out_bf16);
  void* ws_b = reinterpret_cast<char*>(stats_ws) + conv0_stats_bytes(B, norm);
  if (norm == 1) {
    conv0_ln_consts_kernel<<<1, 128, 0, st>>>(w, bias, stats_ws);
    if (int rc = after_launch("conv0_ln_consts")) return rc;
    if (!simt) return conv0_tc_launch(wav, B, L, T0, w, bias, gamma, beta, 1, eps, stats_ws, nullptr, ws_b, out, out_fp16, st);
    conv0_kernel<1><<<grid, 256, 0, st>>>(wav, L, T0, w, bias, gamma, beta, stats_ws, nullptr, eps, out, out_fp16);
  } else if (norm == 2) {
    // stats_ws: [B*65] doubles of moments, then [B*512*2] floats of scale/shift, then [B*512*2] floats of {mean, rstd}
    double* mom = reinterpret_cast<double*>(stats_ws);
    float* affine = reinterpret_cast<float*>(mom + static_cast<size_t>(B) * (K0 + NQ));
    float* norm_stats = affine + static_cast<size_t>(B) * C0 * 2;
    cudaError_t e = cudaMemsetAsync(mom, 0, sizeof(double) * B * (K0 + NQ), st);
    if (e != cudaSuccess) {
      set_error("conv0: memset: %s", cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    int chunks = (T0 + 256 * 8 - 1) / (256 * 8);
    if (chunks > 64) chunks = 64;
    conv0_gn_moments_kernel<<<dim3(chunks, B), 256, 0, st>>>(wav, L, T0, mom);
    if (int rc = after_launch("conv0_gn_moments")) return rc;
    conv0_gn_affine_kernel<<<B, C0, 0, st>>>(mom, w, bias, gamma, beta, T0, eps, affine, norm_stats);
    if (int rc = after_launch("conv0_gn_affine")) return rc;
    if (!simt) return conv0_tc_launch(wav, B, L, T0, w, bias, gamma, beta, 2, eps, nullptr, affine, ws_b, out, out_fp16, st);
    conv0_kernel<2><<<grid, 256, 0, st>>>(wav, L, T0, w, bias, gamma, beta, nullptr, affine, eps, out, out_fp16);
  } else {
    if (!simt) return conv0_tc_launch(wav, B, L, T0, w, bias, gamma, beta, 0, eps, nullptr, nullptr, ws_b, out, out_fp16, st);
    conv0_kernel<0><<<grid, 256, 0, st>>>(wav, L, T0, w, bias, gamma, beta, nullptr, nullptr, eps, out, out_fp16);
  }
  return after_launch("conv0_norm_gelu");
}
