// tcgen05 / TMEM fused attention forward, second generation: TWO 128-query tiles per CTA ping-pong on one K/V stream.
//
// The first-generation kernel (attention_tc.cu) is latency-bound per key tile: its eight softmax warps walk the chain
// tcgen05.ld -> row max -> exp2 -> P store -> proxy fence -> mbarrier in lock step, so an SM only ever has two such
// chains (two CTAs) in flight and the tensor pipe idles ~75 % of the time (DESIGN.md section 8).  Here a work item is
// 256 query rows of one (utterance, head):
//   warp 8       TMA producer    Q0, Q1 once per item; (K_j, V_j) tiles of 64 keys through a 2-stage ring, shared by
//                                both query tiles (half the K/V traffic per query)
//   warp 9       MMA issuer 1    S_t = Q_t K_j^T for t = 0, 1      (TMEM: one 64-column S buffer per query tile)
//   warp 10      MMA issuer 2    O_t += P_t V_j                    (TMEM: one 64-column O accumulator per query tile)
//                (a single issuer per query tile doing both S_t and O_t measured 5 % slower: the ~100-cycle issue
//                 cost of each tcgen05.mma makes two parallel issuing threads worth more than decoupled tiles)
//   warps 0..3   softmax group 0 one thread per query row of tile 0 (all 64 keys of the key tile: no cross-thread max)
//   warps 4..7   softmax group 1 the same for tile 1
// The two groups run independent chains, so with two CTAs per SM four chains overlap: while one group waits for its
// next S tile, the others keep the MUFU and the tensor pipe busy.  S is read from TMEM twice (max pass, exp pass)
// instead of being held in 64 registers, which keeps the kernel at two CTAs per SM.
// Same contract as aptai_attention_fwd: q pre-scaled by head_dim^-0.5, every query row computed, keys >= key_len[b]
// masked, lazy rescaling of O (threshold 2^8), optional log2-domain lse output for the backward pass.
// It serves the training forward with dropout on the attention probabilities (aptai_attention_fwd_dropout; at p = 0
// the mask keeps every element and the scale is 1).
#include "common.h"
#include "ptx.cuh"

namespace aptai {

constexpr int A2_Q = 128;                 // rows per query tile
constexpr int A2_K = 64;                  // keys per key tile
constexpr int A2_D = 64;
constexpr int A2_THREADS = 384;           // warps 0..3 / 4..7 softmax groups, 8 TMA, 9 S-MMA, 10 PV-MMA, 11 TMEM alloc
constexpr int A2_W_TMA = 8, A2_W_S = 9, A2_W_PV = 10, A2_W_ALLOC = 11;
constexpr int A2_QB = A2_Q * A2_D * 2;    // 16 KB per Q tile
constexpr int A2_KVB = A2_K * A2_D * 2;   // 8 KB per K or V tile
constexpr int A2_PB = A2_Q * A2_K * 2;    // 16 KB per P tile
constexpr int A2_STAGES = 2;
constexpr int A2_DATA = 2 * A2_QB + A2_STAGES * 2 * A2_KVB + 2 * A2_PB;   // 96 KB
constexpr int A2_SMEM = A2_DATA + 256;
constexpr uint32_t A2_TS = 0, A2_TO = 128, A2_TCOLS = 256;   // S_t at t*64, O_t at 128 + t*64
constexpr float A2_LOG2E = 1.4426950408889634f;
constexpr float A2_RESCALE = 8.0f;

struct Attn2Params {
  const int* key_len;
  __nv_bfloat16* ctx;
  float* lse;
  int B, T, heads, H, n_qp, items;
  // attention-probability dropout (training): P is masked and rescaled where it feeds P V; the row sum is not
  uint32_t drop_thresh24;
  float drop_inv_keep;
  unsigned long long drop_seed;
};

struct A2Drop {          // per-thread dropout context of one (item, query row)
  uint32_t seed_bh, q, T, thresh24;
  float inv_keep;
};

__device__ __forceinline__ float a2_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint64_t a2_desc_mn(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1024 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__device__ __forceinline__ void a2_tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
      "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
      "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// exp pass over one FULL 64-key tile of one query row: p = exp2(s*log2e - m_used) -> bf16 -> shared memory (K-major
// SWIZZLE_128B), row sum, optionally the raw row maximum.  TMEM is read in four 16-column chunks, the load of chunk
// c+1 in flight while chunk c is processed; packed fp32x2 math (FFMA2 / FADD2) for the exponent argument and the sum.
template <bool TRACK_MAX>
__device__ __forceinline__ void a2_exp_tile_full(uint32_t ts, float m_used, uint8_t* prow, int row, float& rowsum,
                                                 float& rawmax, const A2Drop& dc, int key0) {
  const uint64_t l2e = f32x2_pack(A2_LOG2E, A2_LOG2E), nm = f32x2_pack(-m_used, -m_used);
  uint64_t acc0 = f32x2_pack(0.f, 0.f), acc1 = acc0;
  float m0 = -INFINITY, m1 = -INFINITY;
  uint32_t ra[16], rb[16];
  auto process = [&](const uint32_t (&r)[16], int chunk) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      uint32_t wv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float s0 = __uint_as_float(r[u * 8 + 2 * i]), s1 = __uint_as_float(r[u * 8 + 2 * i + 1]);
        if (TRACK_MAX) {
          if (i & 1) m1 = fmaxf(fmaxf(m1, s0), s1);
          else m0 = fmaxf(fmaxf(m0, s0), s1);
        }
        float a0, a1;
        f32x2_unpack(f32x2_fma(f32x2_pack(s0, s1), l2e, nm), a0, a1);
        const float p0 = a2_ex2(a0), p1 = a2_ex2(a1);
        if (i & 1) acc1 = f32x2_add(acc1, f32x2_pack(p0, p1));
        else acc0 = f32x2_add(acc0, f32x2_pack(p0, p1));
        const uint32_t kk = key0 + chunk * 16 + u * 8 + 2 * i;
        const float d0 = attn_drop_keep(dc.seed_bh, dc.q, kk, dc.T, dc.thresh24) ? p0 * dc.inv_keep : 0.f;
        const float d1 = attn_drop_keep(dc.seed_bh, dc.q, kk + 1, dc.T, dc.thresh24) ? p1 * dc.inv_keep : 0.f;
        wv[i] = pack_bf16(d0, d1);
      }
      *reinterpret_cast<uint4*>(prow + (((chunk * 2 + u) ^ (row & 7)) << 4)) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
    }
  };
  tmem_ld16(ts, ra);
  tmem_ld_wait();
  tmem_ld16(ts + 16, rb);
  process(ra, 0);
  tmem_ld_wait();
  tmem_ld16(ts + 32, ra);
  process(rb, 1);
  tmem_ld_wait();
  tmem_ld16(ts + 48, rb);
  process(ra, 2);
  tmem_ld_wait();
  process(rb, 3);
  float r0, r1;
  f32x2_unpack(f32x2_add(acc0, acc1), r0, r1);
  rowsum = r0 + r1;
  rawmax = fmaxf(m0, m1);
}

__global__ void __launch_bounds__(A2_THREADS, 2)
attention_tc2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                     const Attn2Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                                   // [2 tiles]
  uint8_t* sKV = smem + 2 * A2_QB;                      // [stage][K | V]
  uint8_t* sP = sKV + A2_STAGES * 2 * A2_KVB;           // [2 tiles]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + A2_DATA);
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("aptai attention v2: dynamic shared memory base is not 1024-byte aligned\n");
    __trap();
  }
  uint64_t* q_full = bars + 0;
  uint64_t* q_empty = bars + 1;
  uint64_t* kv_full = bars + 2;     // [2]
  uint64_t* kv_empty = bars + 4;    // [2]
  uint64_t* s_full = bars + 6;      // [2] per query tile
  uint64_t* p_full = bars + 8;      // [2] P_t written (and S_t consumed)
  uint64_t* p_empty = bars + 10;    // [2] P_t V_j complete
  uint64_t* o_full = bars + 12;     // [2]
  uint64_t* o_empty = bars + 14;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == A2_W_TMA && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
  }
  if (warp == A2_W_S && lane == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&p_empty[i], 1);
      mbar_init(&o_full[i], 1);
      mbar_init(&o_empty[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == A2_W_ALLOC) tmem_alloc(tmem_slot, A2_TCOLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == A2_W_TMA) {
    // ---------------------------------------------------------------- TMA producer
    if (lane == 0) {
      uint32_t g = 0, it = 0;
      for (int w = blockIdx.x; w < p.items; w += gridDim.x, ++it) {
        const int qp = w % p.n_qp;
        const int bh = w / p.n_qp;
        const int h = bh % p.heads, b = bh / p.heads;
        const int klen = max(1, min(__ldg(p.key_len + b), p.T));
        const int n = (klen + A2_K - 1) / A2_K;
        const int row0 = b * p.T;
        const bool two = qp * 2 * A2_Q + A2_Q < p.T;
        mbar_wait_backoff(q_empty, (it & 1) ^ 1, 100);
        mbar_expect_tx(q_full, two ? 2 * A2_QB : A2_QB);
        tma_load_2d(&tmQ, q_full, sQ, h * A2_D, row0 + qp * 2 * A2_Q);
        if (two) tma_load_2d(&tmQ, q_full, sQ + A2_QB, h * A2_D, row0 + qp * 2 * A2_Q + A2_Q);
        for (int j = 0; j < n; ++j, ++g) {
          const uint32_t st = g % A2_STAGES, u = g / A2_STAGES;
          mbar_wait_backoff(&kv_empty[st], (u & 1) ^ 1, 100);
          mbar_expect_tx(&kv_full[st], 2 * A2_KVB);
          tma_load_2d(&tmKV, &kv_full[st], sKV + st * 2 * A2_KVB, p.H + h * A2_D, row0 + j * A2_K);
          tma_load_2d(&tmKV, &kv_full[st], sKV + st * 2 * A2_KVB + A2_KVB, 2 * p.H + h * A2_D, row0 + j * A2_K);
        }
      }
    }
  } else if (warp == A2_W_S) {
    // ---------------------------------------------------------------- MMA issuer 1: S_t = Q_t K_j^T
    if (lane == 0) {
      constexpr uint32_t IDESC_BASE = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(A2_Q >> 4) << 24);
      uint32_t g = 0, it = 0;
      uint32_t gt[2] = {0, 0};         // key tiles processed so far by each query tile (barrier phases)
      for (int w = blockIdx.x; w < p.items; w += gridDim.x, ++it) {
        const int qp = w % p.n_qp;
        const int b = (w / p.n_qp) / p.heads;
        const int klen = max(1, min(__ldg(p.key_len + b), p.T));
        const int n = (klen + A2_K - 1) / A2_K;
        const int nt = (qp * 2 * A2_Q + A2_Q < p.T) ? 2 : 1;
        mbar_wait(q_full, it & 1);
        for (int j = 0; j < n; ++j, ++g) {
          const uint32_t st = g % A2_STAGES;
          const int nj = min(A2_K, ((klen - j * A2_K) + 15) & ~15);
          const uint32_t idesc = IDESC_BASE | (static_cast<uint32_t>(nj >> 3) << 17);
          mbar_wait(&kv_full[st], (g / A2_STAGES) & 1);
          const uint32_t k_addr = smem_u32(sKV + st * 2 * A2_KVB);
          // serve whichever query tile is ready first: S_t is free once its softmax group has consumed the previous
          // key tile (P_t written); the two groups drift apart, a fixed order would make one wait for the other
          uint32_t pending = nt == 2 ? 3u : 1u, spins = 0;
          while (pending) {
            for (int t = 0; t < nt; ++t) {
              if (!(pending & (1u << t))) continue;
              if (gt[t] >= 1 && !mbar_try_wait(&p_full[t], (gt[t] - 1) & 1)) continue;
              tc_fence_after();
              const uint32_t q_addr = smem_u32(sQ + t * A2_QB);
#pragma unroll
              for (int k = 0; k < A2_D / 16; ++k)
                umma_bf16(tmem_base + A2_TS + t * A2_K, umma_desc_sw128(q_addr + k * 32),
                          umma_desc_sw128(k_addr + k * 32), idesc, k != 0 ? 1u : 0u);
              umma_commit(&s_full[t]);
              ++gt[t];
              pending &= ~(1u << t);
            }
            if (++spins > APTAI_SPIN_LIMIT) {
              printf("aptai attention v2: S issuer timed out (block %d)\n", (int)blockIdx.x);
              __trap();
            }
          }
          if (j == n - 1) umma_commit(q_empty);
        }
      }
    }
  } else if (warp == A2_W_PV) {
    // ---------------------------------------------------------------- MMA issuer 2: O_t += P_t V_j
    if (lane == 0) {
      constexpr uint32_t IDESC_PV = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(A2_Q >> 4) << 24) |
                                    (1u << 16) | (static_cast<uint32_t>(A2_D >> 3) << 17);   // B MN-major, N=64
      uint32_t g = 0;
      uint32_t gt[2] = {0, 0}, itt[2] = {0, 0};
      for (int w = blockIdx.x; w < p.items; w += gridDim.x) {
        const int qp = w % p.n_qp;
        const int b = (w / p.n_qp) / p.heads;
        const int klen = max(1, min(__ldg(p.key_len + b), p.T));
        const int n = (klen + A2_K - 1) / A2_K;
        const int nt = (qp * 2 * A2_Q + A2_Q < p.T) ? 2 : 1;
        for (int j = 0; j < n; ++j, ++g) {
          const uint32_t st = g % A2_STAGES;
          const int nj = min(A2_K, ((klen - j * A2_K) + 15) & ~15);
          mbar_wait(&kv_full[st], (g / A2_STAGES) & 1);
          const uint32_t v_addr = smem_u32(sKV + st * 2 * A2_KVB + A2_KVB);
          uint32_t pending = nt == 2 ? 3u : 1u, spins = 0;
          while (pending) {
            for (int t = 0; t < nt; ++t) {
              if (!(pending & (1u << t))) continue;
              if (!mbar_try_wait(&p_full[t], gt[t] & 1)) continue;
              if (j == 0) mbar_wait(&o_empty[t], (itt[t] & 1) ^ 1);      // previous item's O_t has been read out
              tc_fence_after();
              const uint32_t p_addr = smem_u32(sP + t * A2_PB);
              for (int k = 0; k < nj / 16; ++k)
                umma_bf16(tmem_base + A2_TO + t * A2_D, umma_desc_sw128(p_addr + k * 32),
                          a2_desc_mn(v_addr + k * 2048), IDESC_PV, (j | k) != 0 ? 1u : 0u);
              umma_commit(&p_empty[t]);
              if (j == n - 1) {
                umma_commit(&o_full[t]);
                ++itt[t];
              }
              ++gt[t];
              pending &= ~(1u << t);
            }
            if (++spins > APTAI_SPIN_LIMIT) {
              printf("aptai attention v2: PV issuer timed out (block %d)\n", (int)blockIdx.x);
              __trap();
            }
          }
          umma_commit(&kv_empty[st]);      // K_j: both S_t(j) completed before their P_t(j) existed
        }
      }
    }
  } else if (warp < 8) {
    // ---------------------------------------------------------------- softmax groups: thread = one query row
    const int t = warp >> 2;                       // query tile of this group
    const int q4 = warp & 3;
    const int row = q4 * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const uint32_t ts = t_lane + A2_TS + t * A2_K, to = t_lane + A2_TO + t * A2_D;
    uint8_t* prow = sP + t * A2_PB + row * 128;
    uint32_t g = 0, it = 0;                         // this tile's own counters
    for (int w = blockIdx.x; w < p.items; w += gridDim.x) {
      const int qp = w % p.n_qp;
      const int bh = w / p.n_qp;
      const int h = bh % p.heads, b = bh / p.heads;
      if (t == 1 && !(qp * 2 * A2_Q + A2_Q < p.T)) continue;      // second tile lies beyond the utterance
      const int klen = max(1, min(__ldg(p.key_len + b), p.T));
      const int n = (klen + A2_K - 1) / A2_K;
      float m_used = -INFINITY, l = 0.f;
      A2Drop dc;
      dc.seed_bh = attn_drop_seed_bh(p.drop_seed, static_cast<uint32_t>(bh));
      dc.q = static_cast<uint32_t>(qp * 2 * A2_Q + t * A2_Q + row);
      dc.T = static_cast<uint32_t>(p.T);
      dc.thresh24 = p.drop_thresh24;
      dc.inv_keep = p.drop_inv_keep;
      // a warp whose 32 query rows all lie beyond the utterance only keeps the barrier protocol going: its P rows stay
      // stale, the matching O rows are never written
      const bool warp_live = qp * 2 * A2_Q + t * A2_Q + q4 * 32 < p.T;
      for (int j = 0; j < n; ++j, ++g) {
        const int valid = min(A2_K, klen - j * A2_K);            // keys of this tile that exist (>= 1)
        mbar_wait(&s_full[t], g & 1);
        if (!warp_live) {
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_full[t]);
          continue;
        }
        tc_fence_after();
        // Steady state (full key tile, not the first of the item): ONE pass with the stale maximum — exp, P store and
        // row sum while tracking the true maximum; it stands unless some row of the warp outgrew the lazy-rescale
        // threshold (rare), in which case the tile is redone below with the new maximum.
        bool done = false;
        if (valid >= A2_K && j > 0) {
          mbar_wait(&p_empty[t], (g - 1) & 1);           // P_t free: P_t(j-1) V_(j-1) has completed
          float rsum, rmax;
          a2_exp_tile_full<true>(ts, m_used, prow, row, rsum, rmax, dc, j * A2_K);
          if (!__any_sync(0xffffffffu, rmax * A2_LOG2E > m_used + A2_RESCALE)) {
            l += rsum;
            done = true;
          }
        }
        if (!done) {
        // pass 1: row maximum over the valid keys
        float mx;
        {
          uint32_t r[32];
          float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
          if (valid >= A2_K) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              tmem_ld32(ts + c * 32, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                m0 = fmaxf(m0, __uint_as_float(r[i]));     m1 = fmaxf(m1, __uint_as_float(r[i + 1]));
                m2 = fmaxf(m2, __uint_as_float(r[i + 2])); m3 = fmaxf(m3, __uint_as_float(r[i + 3]));
              }
            }
          } else {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              if (c * 32 < valid) {
                tmem_ld32(ts + c * 32, r);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i)
                  if (c * 32 + i < valid) m0 = fmaxf(m0, __uint_as_float(r[i]));
              }
            }
          }
          mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) * A2_LOG2E;
        }
        float factor = 1.f;
        if (mx > m_used + A2_RESCALE) {
          factor = exp2f(m_used - mx);            // 0 on the first tile (m_used = -inf)
          m_used = mx;
        }
        // P_t (and O_t for a rescale) are free once P_t(j-1) V_(j-1) has completed
        if (g >= 1) mbar_wait(&p_empty[t], (g - 1) & 1);
        const bool need = (factor != 1.f) && (j > 0);
        if (__any_sync(0xffffffffu, need)) {
          tc_fence_after();
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t r[32];
            tmem_ld32(to + c * 32, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * factor);
            a2_tmem_st32(to + c * 32, r);
          }
        }
        l *= factor;
        // pass 2: p = exp2(s*log2e - m_used) -> bf16 -> shared memory (K-major SWIZZLE_128B), row sum.
        // Full key tiles (all but the last of an utterance) take the path without per-element masking.
        float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
        if (valid >= A2_K) {
          float rmax_unused;
          a2_exp_tile_full<false>(ts, m_used, prow, row, rs0, rmax_unused, dc, j * A2_K);
        } else {
          const int ncol16 = (valid + 15) >> 4;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (c * 32 < valid) {
              uint32_t r[32];
              tmem_ld32(ts + c * 32, r);
              tmem_ld_wait();
#pragma unroll
              for (int u8 = 0; u8 < 4; ++u8) {
                float pv[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  pv[i] = a2_ex2(fmaf(__uint_as_float(r[u8 * 8 + i]), A2_LOG2E, -m_used));
                  if (c * 32 + u8 * 8 + i >= valid) pv[i] = 0.f;
                }
                rs0 += pv[0] + pv[4]; rs1 += pv[1] + pv[5]; rs2 += pv[2] + pv[6]; rs3 += pv[3] + pv[7];
#pragma unroll
                for (int i = 0; i < 8; ++i)
                  pv[i] = attn_drop_keep(dc.seed_bh, dc.q, j * A2_K + c * 32 + u8 * 8 + i, dc.T, dc.thresh24)
                              ? pv[i] * dc.inv_keep : 0.f;
                const int unit = c * 4 + u8;
                if ((unit >> 1) < ncol16)
                  *reinterpret_cast<uint4*>(prow + ((unit ^ (row & 7)) << 4)) =
                      make_uint4(pack_bf16(pv[0], pv[1]), pack_bf16(pv[2], pv[3]), pack_bf16(pv[4], pv[5]),
                                 pack_bf16(pv[6], pv[7]));
              }
            }
          }
        }
        l += (rs0 + rs1) + (rs2 + rs3);
        }   // !done
        tc_fence_before();
        fence_async_proxy();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[t]);
      }
      // ---- output: O_t / l -> bf16, lse
      mbar_wait(&o_full[t], it & 1);
      tc_fence_after();
      const int qrow = qp * 2 * A2_Q + t * A2_Q + row;
      const float inv = 1.f / l;
      if (p.lse != nullptr && qrow < p.T)
        p.lse[(static_cast<long long>(b) * p.heads + h) * p.T + qrow] = m_used + log2f(l);
      __nv_bfloat16* out = p.ctx + (static_cast<long long>(b) * p.T + qrow) * p.H + h * A2_D;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        tmem_ld32(to + c * 32, r);
        tmem_ld_wait();
        if (qrow < p.T) {
#pragma unroll
          for (int i = 0; i < 32; i += 8)
            *reinterpret_cast<uint4*>(out + c * 32 + i) =
                make_uint4(pack_bf16(__uint_as_float(r[i]) * inv, __uint_as_float(r[i + 1]) * inv),
                           pack_bf16(__uint_as_float(r[i + 2]) * inv, __uint_as_float(r[i + 3]) * inv),
                           pack_bf16(__uint_as_float(r[i + 4]) * inv, __uint_as_float(r[i + 5]) * inv),
                           pack_bf16(__uint_as_float(r[i + 6]) * inv, __uint_as_float(r[i + 7]) * inv));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[t]);
      ++it;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == A2_W_ALLOC) {
    tc_fence_after();
    tmem_dealloc(tmem_base, A2_TCOLS);
  }
}

}  // namespace aptai

using namespace aptai;

extern "C" int aptai_attention_fwd_dropout(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T,
                                           int heads, float drop_p, uint64_t drop_seed, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(qkv && ctx && key_len, "attention_v2: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && heads >= 1, "attention_v2: bad shape");
  APTAI_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "attention_v2: dropout p must be in [0, 1)");
  APTAI_REQUIRE(drop_p == 0.f || static_cast<long long>(T) * T < (1LL << 32), "attention_v2: T too large for dropout");
  APTAI_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(ctx) & 15) == 0,
                "attention_v2: buffers must be 16-byte aligned");
  const int H = heads * A2_D;
  CUtensorMap tmq, tmkv;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(3) * H, static_cast<uint64_t>(B) * T};
    uint64_t strides[1] = {static_cast<uint64_t>(3) * H * 2};
    uint32_t boxq[2] = {A2_D, A2_Q};
    uint32_t boxkv[2] = {A2_D, A2_K};
    if (int rc = encode_tmap_bf16(&tmq, qkv, 2, dims, strides, boxq, 1)) return rc;
    if (int rc = encode_tmap_bf16(&tmkv, qkv, 2, dims, strides, boxkv, 1)) return rc;
  }
  Attn2Params p;
  p.key_len = key_len;
  p.ctx = reinterpret_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  p.B = B; p.T = T; p.heads = heads; p.H = H;
  p.n_qp = (T + 2 * A2_Q - 1) / (2 * A2_Q);
  p.items = B * heads * p.n_qp;
  p.drop_thresh24 = static_cast<uint32_t>(static_cast<double>(drop_p) * 16777216.0);
  p.drop_inv_keep = 1.0f / (1.0f - drop_p);
  p.drop_seed = drop_seed;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(attention_tc2_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaError_t e = cudaFuncSetAttribute(attention_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, A2_SMEM);
    if (e != cudaSuccess) {
      set_error("attention_v2: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  const int slots = 2 * num_sms();
  const int grid = p.items < slots ? p.items : slots;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  attention_tc2_kernel<<<grid, A2_THREADS, A2_SMEM, st>>>(tmq, tmkv, p);
  return after_launch("attention_tc2");
}

namespace aptai {
// keep/(1-p) of every (b, h, q, k): what a training step's attention dropout used (tests replay it)
__global__ void attn_dropout_mask_kernel(int T, uint32_t thresh24, float inv_keep, unsigned long long seed,
                                         float* __restrict__ out, long long total) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t k = static_cast<uint32_t>(i % T);
    const uint32_t q = static_cast<uint32_t>((i / T) % T);
    const uint32_t bh = static_cast<uint32_t>(i / (static_cast<long long>(T) * T));
    out[i] = attn_drop_keep(attn_drop_seed_bh(seed, bh), q, k, static_cast<uint32_t>(T), thresh24) ? inv_keep : 0.f;
  }
}
}  // namespace aptai

extern "C" int aptai_attention_dropout_mask(int B, int T, int heads, float drop_p, uint64_t drop_seed, float* out,
                                            void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(out && B >= 1 && T >= 1 && heads >= 1 && drop_p >= 0.f && drop_p < 1.f, "attention_dropout_mask: bad arguments");
  const long long total = static_cast<long long>(B) * heads * T * T;
  int gx = static_cast<int>((total + 255) / 256);
  if (gx > 16384) gx = 16384;
  attn_dropout_mask_kernel<<<gx, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      T, static_cast<uint32_t>(static_cast<double>(drop_p) * 16777216.0), 1.0f / (1.0f - drop_p), drop_seed, out, total);
  return after_launch("attention_dropout_mask");
}
