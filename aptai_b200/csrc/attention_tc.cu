// tcgen05 / TMEM fused attention forward (HF:500-549 with SDPA semantics: non-causal, key-padding mask).
//
// Persistent, warp-specialised, one work item = 128 query rows of one (utterance, head); two CTAs are resident
// per SM (256 TMEM columns and 96 KB of shared memory each) so that the softmax warps of both keep the MUFU busy:
//   warp 8      TMA producer   Q tile once per item; (K_j, V_j) tiles of 64 keys through a 3-stage ring
//   warp 9      MMA issuer 1   S_j = Q K_j^T  (M=128, N=n_j<=64, K=64) -> TMEM S buffer j%2 (double buffered)
//   warp 10     MMA issuer 2   O  += P_j V_j  (M=128, N=64, K=n_j)     -> TMEM O; P_j (bf16) from shared memory,
//                                                                         V_j as an MN-major B operand
//   warps 0..7  softmax        two threads per query row (32 of the tile's 64 keys each): tcgen05.ld, key-length mask, running max
//                              with lazy rescaling of O (only when the max grows by more than 2^8), exp2, row sum,
//                              P_j -> shared memory in the UMMA K-major SWIZZLE_128B layout; final O / l -> bf16
// S_{j+2} is issued as soon as P_j is written (S buffer j%2 free), so S_{j+1} is always ready when the softmax
// warps finish tile j: they never wait on the tensor core in steady state.
// q must be pre-scaled by head_dim^-0.5 (folded into the q projection at plan time); head_dim is 64.
// Every query row is computed (padded queries attend to valid keys, HF:438-463); keys >= key_len[b] are masked.
#include "common.h"
#include "ptx.cuh"

namespace aptai {

constexpr int AQ = 128;                 // query rows per work item
constexpr int AK = 64;                  // keys per KV tile
constexpr int AD = 64;                  // head dim
constexpr int ATC_THREADS = 384;        // warps 0..7 softmax (2 per 32-row quadrant), 8 TMA, 9 S-MMA, 10 PV-MMA, 11 TMEM alloc
constexpr int W_TMA = 8, W_MMA = 9, W_MMA2 = 10, W_ALLOC = 11;   // single-thread roles in the highest warp ids
constexpr int Q_BYTES = AQ * AD * 2;    // 16 KB
constexpr int KV_BYTES = AK * AD * 2;   // 8 KB per K or V tile
constexpr int P_BYTES = AQ * AK * 2;    // 16 KB
constexpr int KV_STAGES = 3;
constexpr int ATC_DATA = Q_BYTES + KV_STAGES * 2 * KV_BYTES + 2 * P_BYTES;   // 96 KB
constexpr int ATC_XCH = 2 * 2 * AQ * 4;                                     // row-max / row-sum exchange between half-row threads
constexpr int ATC_SMEM = ATC_DATA + 256 + ATC_XCH;                           // + barriers; two CTAs fit one SM
constexpr uint32_t TM_S = 0, TM_O = 128, TM_COLS = 256;   // S double buffered (2 x 64 columns), O 64 columns
constexpr float ATC_LOG2E = 1.4426950408889634f;
constexpr float RESCALE_THRESHOLD = 8.0f;   // log2 units

struct AttnParams {
  const int* key_len;
  __nv_bfloat16* ctx;
  float* lse;   // optional [B][heads][T]: log2-domain log-sum-exp per query row (kept for the backward pass)
  int B, T, heads, H, n_qt, items;
};

__device__ __forceinline__ float ex2_approx(float x) {   // single MUFU.EX2 (flushes denormal results to 0)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// MN-major SWIZZLE_128B descriptor for a B operand stored [k rows][64 mn-elements] (128 B per k row):
// 8-row groups along K are 1024 B apart (SBO); a single 64-element MN block, so LBO is unused.
__device__ __forceinline__ uint64_t umma_desc_sw128_mn(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1024 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// FP16: q / k / v, P and the context are IEEE fp16 instead of bf16 (precision="fp16")
template <bool FP16>
__global__ void __launch_bounds__(ATC_THREADS, 2)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                    const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sKV = smem + Q_BYTES;                               // [stage][K | V]
  uint8_t* sP = smem + Q_BYTES + KV_STAGES * 2 * KV_BYTES;     // [2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ATC_DATA);
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("aptai attention: dynamic shared memory base is not 1024-byte aligned\n");
    __trap();
  }
  uint64_t* q_full = bars + 0;
  uint64_t* q_empty = bars + 1;
  uint64_t* o_full = bars + 2;
  uint64_t* o_empty = bars + 3;
  uint64_t* kv_full = bars + 4;    // [3]
  uint64_t* kv_empty = bars + 7;   // [3]  P_j V_j complete
  uint64_t* s_full = bars + 10;    // [2]
  uint64_t* p_full = bars + 12;    // [2]  P_j written (and S_j consumed)
  uint64_t* p_empty = bars + 14;   // [2]  P_j V_j complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  float* xch = reinterpret_cast<float*>(smem + ATC_DATA + 256);   // [2 parity][2 halves][128 rows]

  // warp index through a shuffle: provably warp-uniform (single-issuer roles: whole warp converged, elect.sync
  // around the issue, loop state in uniform registers — see gemm_tc.cu)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
  }
  if (warp == W_MMA && lane == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    mbar_init(o_full, 1);
    mbar_init(o_empty, 8);
    for (int i = 0; i < KV_STAGES; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 8);
      mbar_init(&p_empty[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == W_ALLOC) tmem_alloc(tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == W_TMA) {
    // ---------------------------------------------------------------- TMA producer
    {
      uint32_t g = 0, it = 0;
      for (int w = blockIdx.x; w < p.items; w += gridDim.x, ++it) {
        const int qt = w % p.n_qt;
        const int bh = w / p.n_qt;
        const int h = bh % p.heads, b = bh / p.heads;
        const int klen = __shfl_sync(0xffffffffu, max(1, min(__ldg(p.key_len + b), p.T)), 0);
        const int n = (klen + AK - 1) / AK;
        const int row0 = b * p.T;
        mbar_wait_backoff(q_empty, (it & 1) ^ 1, 100);
        if (elect_one()) {
          mbar_expect_tx(q_full, Q_BYTES);
          tma_load_2d(&tmQ, q_full, sQ, h * AD, row0 + qt * AQ);
        }
        __syncwarp();
        for (int j = 0; j < n; ++j, ++g) {
          const uint32_t st = g % KV_STAGES, u = g / KV_STAGES;
          mbar_wait_backoff(&kv_empty[st], (u & 1) ^ 1, 100);
          if (elect_one()) {
            mbar_expect_tx(&kv_full[st], 2 * KV_BYTES);
            tma_load_2d(&tmKV, &kv_full[st], sKV + st * 2 * KV_BYTES, p.H + h * AD, row0 + j * AK);
            tma_load_2d(&tmKV, &kv_full[st], sKV + st * 2 * KV_BYTES + KV_BYTES, 2 * p.H + h * AD, row0 + j * AK);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == W_MMA) {
    // ---------------------------------------------------------------- MMA issuer 1: S_j = Q K_j^T
    // (two issuing threads per CTA: a tcgen05.mma issue costs the thread ~100 cycles but these N=64 MMAs are
    //  only 32 cycles of tensor work, so a single issuer for S and PV was the bottleneck of the tile period)
    {
      constexpr uint32_t FMT_AB = FP16 ? 0u : ((1u << 7) | (1u << 10));      // a_format / b_format: 0 = f16, 1 = bf16
      constexpr uint32_t IDESC_BASE = (1u << 4) | FMT_AB | (static_cast<uint32_t>(AQ >> 4) << 24);
      uint32_t g = 0, it = 0;
      for (int w = blockIdx.x; w < p.items; w += gridDim.x, ++it) {
        const int bh = w / p.n_qt;
        const int b = bh / p.heads;
        const int klen = __shfl_sync(0xffffffffu, max(1, min(__ldg(p.key_len + b), p.T)), 0);
        const int n = (klen + AK - 1) / AK;
        mbar_wait(q_full, it & 1);
        const uint32_t q_addr = smem_u32(sQ);
        for (int j = 0; j < n; ++j, ++g) {
          const uint32_t st = g % KV_STAGES, u = g / KV_STAGES;
          const int nj = min(AK, ((klen - j * AK) + 15) & ~15);
          // S buffer g&1 was last used by tile g-2: the softmax warps have consumed it once P_{g-2} is written
          if (g >= 2) mbar_wait_backoff(&p_full[g & 1], ((g - 2) >> 1) & 1, 32);
          mbar_wait(&kv_full[st], u & 1);
          tc_fence_after();
          const uint32_t k_addr = smem_u32(sKV + st * 2 * KV_BYTES);
          const uint32_t idesc = IDESC_BASE | (static_cast<uint32_t>(nj >> 3) << 17);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < AD / 16; ++k)
              umma_bf16(tmem_base + TM_S + (g & 1) * AK, umma_desc_sw128(q_addr + k * 32),
                        umma_desc_sw128(k_addr + k * 32), idesc, k != 0 ? 1u : 0u);
            umma_commit(&s_full[g & 1]);
            if (j == n - 1) umma_commit(q_empty);           // Q tile no longer needed once the last S is done
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == W_MMA2) {
    // ---------------------------------------------------------------- MMA issuer 2: O += P_j V_j
    {
      constexpr uint32_t FMT_AB = FP16 ? 0u : ((1u << 7) | (1u << 10));
      constexpr uint32_t IDESC_PV = (1u << 4) | FMT_AB | (static_cast<uint32_t>(AQ >> 4) << 24) |
                                    (1u << 16) | (static_cast<uint32_t>(AD >> 3) << 17);   // B MN-major, N=64
      uint32_t g = 0, it = 0;
      for (int w = blockIdx.x; w < p.items; w += gridDim.x, ++it) {
        const int bh = w / p.n_qt;
        const int b = bh / p.heads;
        const int klen = __shfl_sync(0xffffffffu, max(1, min(__ldg(p.key_len + b), p.T)), 0);
        const int n = (klen + AK - 1) / AK;
        for (int j = 0; j < n; ++j, ++g) {
          const uint32_t sb = g & 1, st = g % KV_STAGES;
          const int nj = min(AK, ((klen - j * AK) + 15) & ~15);
          mbar_wait_backoff(&p_full[sb], (g >> 1) & 1, 32);    // P_j in shared memory (S_j done long before)
          mbar_wait(&kv_full[st], (g / KV_STAGES) & 1);        // V_j (already landed: S_j needed the same stage)
          if (j == 0) mbar_wait(o_empty, (it & 1) ^ 1);        // previous item's O has been read out
          tc_fence_after();
          const uint32_t p_addr = smem_u32(sP + sb * P_BYTES);
          const uint32_t v_addr = smem_u32(sKV + st * 2 * KV_BYTES + KV_BYTES);
          if (elect_one()) {
            for (int k = 0; k < nj / 16; ++k)
              umma_bf16(tmem_base + TM_O, umma_desc_sw128(p_addr + k * 32), umma_desc_sw128_mn(v_addr + k * 2048),
                        IDESC_PV, (j | k) != 0 ? 1u : 0u);
            umma_commit(&kv_empty[st]);        // K_j was consumed by S_j, which completed before P_j existed
            umma_commit(&p_empty[sb]);
            if (j == n - 1) umma_commit(o_full);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp < 8) {
    // ---------------------------------------------------------------- softmax + output
    // two threads per query row: warp w and warp w+4 share TMEM quadrant w%4; `half` selects 32 of the 64 keys of
    // a tile (and 32 of the 64 output columns).  The row maximum is exchanged through shared memory.
    const int q = warp & 3;
    const int half = warp >> 2;
    const int row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t pair_bar = 1 + q;                       // named barrier of the two warps of this quadrant
    uint32_t g = 0, it = 0;
    for (int w = blockIdx.x; w < p.items; w += gridDim.x, ++it) {
      const int qt = w % p.n_qt;
      const int bh = w / p.n_qt;
      const int h = bh % p.heads, b = bh / p.heads;
      const int klen = max(1, min(__ldg(p.key_len + b), p.T));
      const int n = (klen + AK - 1) / AK;
      float m_used = -INFINITY, l = 0.f;
      for (int j = 0; j < n; ++j, ++g) {
        const uint32_t sb = g & 1, u = g >> 1;
        const int valid = min(AK, klen - j * AK) - half * 32;      // keys of MY 32-key half that exist (may be <= 0)
        const bool full_half = valid >= 32;
        mbar_wait(&s_full[sb], u & 1);
        tc_fence_after();
        uint32_t r0[32];
        tmem_ld32(t_lane + TM_S + sb * AK + half * 32, r0);
        tmem_ld_wait();
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
        if (full_half) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            mx0 = fmaxf(mx0, __uint_as_float(r0[i]));
            mx1 = fmaxf(mx1, __uint_as_float(r0[i + 1]));
            mx2 = fmaxf(mx2, __uint_as_float(r0[i + 2]));
            mx3 = fmaxf(mx3, __uint_as_float(r0[i + 3]));
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < valid) mx0 = fmaxf(mx0, __uint_as_float(r0[i]));
        }
        float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        float* xm = xch + (g & 1) * 2 * AQ;
        xm[half * AQ + row] = mx;
        named_bar_sync(pair_bar, 64);
        mx = fmaxf(mx, xm[(half ^ 1) * AQ + row]) * ATC_LOG2E;
        // lazy rescale: keep the stale max unless the new one exceeds it by more than 2^8 (both halves decide alike)
        float factor = 1.f;
        if (mx > m_used + RESCALE_THRESHOLD) {
          factor = exp2f(m_used - mx);          // 0 on the first tile (m_used = -inf)
          m_used = mx;
        }
        const bool need = (factor != 1.f) && (j > 0);
        if (__any_sync(0xffffffffu, need)) {
          // O must be complete (P_{j-1} V_{j-1} done) before it is rescaled in place; each half owns 32 columns
          const uint32_t gp = g - 1;
          mbar_wait(&p_empty[gp & 1], (gp >> 1) & 1);
          tc_fence_after();
          uint32_t r[32];
          tmem_ld32(t_lane + TM_O + half * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * factor);
          asm volatile(
              "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
              "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
              "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
              ::"r"(t_lane + TM_O + half * 32), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]),
              "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]),
              "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]),
              "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
              "r"(r[30]), "r"(r[31])
              : "memory");
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        l *= factor;
        // p = exp2(s*log2e - m_used); my 32 keys -> 4 of the 8 sixteen-byte units of the row (K-major SWIZZLE_128B)
        mbar_wait(&p_empty[sb], (u & 1) ^ 1);      // P_{j-2} V_{j-2} has consumed this P buffer
        uint8_t* prow = sP + sb * P_BYTES + row * 128;
        float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
        const int ncol16 = (min(AK, klen - j * AK) + 15) >> 4;      // 16-key groups the P V MMA will read
#pragma unroll
        for (int u8 = 0; u8 < 4; ++u8) {             // 8 keys = one 16-byte unit at a time (short live ranges)
          float pv[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            pv[i] = ex2_approx(fmaf(__uint_as_float(r0[u8 * 8 + i]), ATC_LOG2E, -m_used));
            if (!full_half && u8 * 8 + i >= valid) pv[i] = 0.f;
          }
          rs0 += pv[0] + pv[4]; rs1 += pv[1] + pv[5]; rs2 += pv[2] + pv[6]; rs3 += pv[3] + pv[7];
          const int unit = half * 4 + u8;
          if ((unit >> 1) < ncol16) {
            uint4 v4 = make_uint4(pack_h16c<FP16>(pv[0], pv[1]), pack_h16c<FP16>(pv[2], pv[3]), pack_h16c<FP16>(pv[4], pv[5]),
                                  pack_h16c<FP16>(pv[6], pv[7]));
            *reinterpret_cast<uint4*>(prow + ((unit ^ (row & 7)) << 4)) = v4;
          }
        }
        l += (rs0 + rs1) + (rs2 + rs3);
        // S consumed; P visible to the async proxy (tensor core)
        tc_fence_before();
        fence_async_proxy();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[sb]);
      }
      // ---- output: O / l -> bf16 (each half owns 32 of the 64 columns; the row sum is exchanged first)
      float* xl = xch + (it & 1) * 2 * AQ;
      named_bar_sync(pair_bar, 64);                 // the max-exchange slots of this parity are free again
      xl[half * AQ + row] = l;
      named_bar_sync(pair_bar, 64);
      const float l_tot = l + xl[(half ^ 1) * AQ + row];
      const float inv = 1.f / l_tot;
      mbar_wait(o_full, it & 1);
      tc_fence_after();
      const int qrow = qt * AQ + row;
      if (p.lse != nullptr && half == 0 && qrow < p.T)
        p.lse[(static_cast<long long>(b) * p.heads + h) * p.T + qrow] = m_used + log2f(l_tot);
      __nv_bfloat16* out = p.ctx + (static_cast<long long>(b) * p.T + qrow) * p.H + h * AD + half * 32;
      {
        uint32_t r[32];
        tmem_ld32(t_lane + TM_O + half * 32, r);
        tmem_ld_wait();
        if (qrow < p.T) {
#pragma unroll
          for (int i = 0; i < 32; i += 8)
            *reinterpret_cast<uint4*>(out + i) =
                make_uint4(pack_h16c<FP16>(__uint_as_float(r[i]) * inv, __uint_as_float(r[i + 1]) * inv),
                           pack_h16c<FP16>(__uint_as_float(r[i + 2]) * inv, __uint_as_float(r[i + 3]) * inv),
                           pack_h16c<FP16>(__uint_as_float(r[i + 4]) * inv, __uint_as_float(r[i + 5]) * inv),
                           pack_h16c<FP16>(__uint_as_float(r[i + 6]) * inv, __uint_as_float(r[i + 7]) * inv));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_ALLOC) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TM_COLS);
  }
}

}  // namespace aptai

using namespace aptai;

template <bool FP16>
static int attention_fwd_impl(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T, int heads,
                              void* stream) {
  auto kern = attention_tc_kernel<FP16>;
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(qkv && ctx && key_len, "attention: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && heads >= 1, "attention: bad shape");
  APTAI_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(ctx) & 15) == 0,
                "attention: buffers must be 16-byte aligned");
  const int H = heads * AD;
  CUtensorMap tmq, tmkv;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(3) * H, static_cast<uint64_t>(B) * T};
    uint64_t strides[1] = {static_cast<uint64_t>(3) * H * 2};
    uint32_t boxq[2] = {AD, AQ};
    uint32_t boxkv[2] = {AD, AK};
    if (int rc = encode_tmap_bf16(&tmq, qkv, 2, dims, strides, boxq, 1)) return rc;
    if (int rc = encode_tmap_bf16(&tmkv, qkv, 2, dims, strides, boxkv, 1)) return rc;
  }
  AttnParams p;
  p.key_len = key_len;
  p.ctx = reinterpret_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  p.B = B; p.T = T; p.heads = heads; p.H = H;
  p.n_qt = (T + AQ - 1) / AQ;
  p.items = B * heads * p.n_qt;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ATC_SMEM);
    if (e != cudaSuccess) {
      set_error("attention: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  const int ctas_per_sm = 2;      // two CTAs per SM are intended (80 KB smem, 256 TMEM columns, <= 128 registers each)
  const int grid = p.items < ctas_per_sm * num_sms() ? p.items : ctas_per_sm * num_sms();
  kern<<<grid, ATC_THREADS, ATC_SMEM, reinterpret_cast<cudaStream_t>(stream)>>>(tmq, tmkv, p);
  return after_launch("attention_tc");
}

extern "C" int aptai_attention_fwd(const void* qkv, void* ctx, const int32_t* key_len, int B, int T, int heads,
                                   void* stream) {
  return attention_fwd_impl<false>(qkv, ctx, nullptr, key_len, B, T, heads, stream);
}

extern "C" int aptai_attention_fwd_fmt(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T,
                                       int heads, int half_fmt, void* stream) {
  return half_fmt ? attention_fwd_impl<true>(qkv, ctx, lse, key_len, B, T, heads, stream)
                  : attention_fwd_impl<false>(qkv, ctx, lse, key_len, B, T, heads, stream);
}

extern "C" int aptai_attention_fwd_lse(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T,
                                       int heads, void* stream) {
  APTAI_REQUIRE(lse != nullptr, "attention_fwd_lse: null lse");
  return attention_fwd_impl<false>(qkv, ctx, lse, key_len, B, T, heads, stream);
}
