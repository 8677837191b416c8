// tcgen05 / TMEM fused attention forward, third generation (HF:500-549, SDPA with the key-length mask).
//
// What the second generation (attention_tc2.cu) left on the table (profiles/r01_attention_tc2_b120x399.md: tensor
// pipe 22 %, MUFU 39 %): P made a round trip registers -> shared memory -> UMMA with a proxy fence per key tile, every
// query tile had ONE S buffer (its softmax chain waited for the next Q K^T after every key tile) and every exponential
// went through the MUFU, which at head_dim 64 needs twice the cycles of the two MMAs it sits between.  Here:
//   * P never leaves TMEM: the softmax threads overwrite the first 32 columns of the S buffer they have just read
//     with P in bf16 (tcgen05.st) and O += P V takes its A operand from TMEM (tcgen05.mma [d], [a_tmem], b_desc);
//   * every query tile owns THREE 64-column S buffers, so Q K^T of key tiles j+1 and j+2 are complete before the
//     softmax of tile j ends; one CTA per SM, 512 TMEM columns: S[2 tiles][3] at 0..383, O[2 tiles] at 384..511;
//   * one issuing thread per query tile: on "P(j) written" it issues O += P(j) V(j) and then S(j+3) = Q K(j+3)^T —
//     tcgen05.mma of one thread execute in order, so the Q K^T that overwrites the buffer P(j) lives in needs no
//     barrier behind the P V that reads it;
//   * the whole stream of (work item, key tile) pairs is software-pipelined ACROSS work items (double-buffered Q,
//     6-stage K/V ring shared by the two query tiles), so item boundaries cost no bubble;
//   * 3 of every 8 exponentials are evaluated on the FMA pipe (Cody-Waite split by a round-down magic add, degree-3
//     minimax polynomial, exponent inserted with one shift-add; 8.6e-5 relative error, 45x below the bf16 rounding of
//     P), which balances MUFU and issue slots;
//   * the scores of a row-tile (64 fp32) are held in registers between the max pass and the exp pass (one CTA per SM
//     leaves 168 registers per thread), so TMEM is read once and there is no stale-maximum redo path;
//   * O leaves through shared memory and one TMA store per softmax WARP (3-D tensor map (channel, frame, utterance),
//     box 64 x 32 rows: clipped at the utterance's last frame, no per-row predicate, no barrier between warps); the
//     read-out of an item's O is deferred into the first key tile of the next item, where the wait for the item's
//     last P V hides behind that tile's softmax.
// Same contract as aptai_attention_fwd: q pre-scaled by head_dim^-0.5, keys >= key_len[b] masked, lazy rescaling
// of O (threshold 2^8), optional log2-domain lse output for the backward pass.
#include "common.h"
#include "ptx.cuh"

namespace aptai {

constexpr int A3_Q = 128;                  // rows per query tile
constexpr int A3_K = 64;                   // keys per key tile
constexpr int A3_D = 64;
constexpr int A3_THREADS = 352;            // warps 0..3 / 4..7 softmax groups, 8 TMEM alloc + TMA, 9 / 10 MMA issuers
constexpr int A3_W_TMA = 8, A3_W_MMA0 = 9, A3_W_ALLOC = 8;   // 11 warps: 184 registers per thread
constexpr int A3_NBUF = 3;                 // S buffers per query tile
constexpr int A3_STAGES = 6;               // K/V ring
constexpr int A3_QB = A3_Q * A3_D * 2;     // 16 KB per Q tile
constexpr int A3_KVB = A3_K * A3_D * 2;    // 8 KB per K or V tile
constexpr int A3_OB = A3_Q * A3_D * 2;     // 16 KB output staging per query tile
constexpr int A3_DATA = 4 * A3_QB + A3_STAGES * 2 * A3_KVB + 2 * A3_OB;   // 192 KB
constexpr int A3_SMEM = A3_DATA + 512;
constexpr uint32_t A3_TO = 2 * A3_NBUF * A3_K;   // O_t at 384 + t*64
constexpr uint32_t A3_TCOLS = 512;
constexpr float A3_LOG2E = 1.4426950408889634f;
constexpr float A3_RESCALE = 8.0f;
constexpr int A3_POLY8 = 3;                // of every 8 exponential pairs, this many are evaluated on the FMA pipe

struct Attn3Params {
  const int* key_len;
  float* lse;
  int B, T, heads, n_qp, items, per_cta;
  int reverse;              // aptai_set_traversal: utterances from the last to the first
};

// Work items (utterance b, head h, query-tile pair qp) in the order w = (b * heads + h) * n_qp + qp.  CTA c owns the
// contiguous range [c * per_cta, (c + 1) * per_cta): every role walks it with increments only (no division in the
// single-thread roles' loops), and consecutive items of a CTA re-use the same K/V out of L2.
struct A3Iter {
  int w, w_end, qp, h, b, klen, n;
  int bp;                   // physical utterance index (B - 1 - b when the traversal is reversed)
  bool two;                 // the second 128-query tile of the pair exists
};
__device__ __forceinline__ void a3_iter_lengths(A3Iter& it, const Attn3Params& p) {
  // the shuffle makes the loaded length provably warp-uniform for the compiler (every role calls this with the whole
  // warp converged): loop bounds derived from it stay in uniform registers
  it.bp = p.reverse ? p.B - 1 - it.b : it.b;
  it.klen = __shfl_sync(0xffffffffu, max(1, min(__ldg(p.key_len + it.bp), p.T)), 0);
  it.n = (it.klen + A3_K - 1) / A3_K;
}
__device__ __forceinline__ bool a3_iter_init(A3Iter& it, const Attn3Params& p) {
  it.w = static_cast<int>(blockIdx.x) * p.per_cta;
  it.w_end = min(p.items, it.w + p.per_cta);
  if (it.w >= it.w_end) return false;
  it.qp = it.w % p.n_qp;
  const int bh = it.w / p.n_qp;
  it.h = bh % p.heads;
  it.b = bh / p.heads;
  a3_iter_lengths(it, p);
  it.two = it.qp * 2 * A3_Q + A3_Q < p.T;
  return true;
}
__device__ __forceinline__ bool a3_iter_next(A3Iter& it, const Attn3Params& p) {
  if (++it.w >= it.w_end) return false;
  if (++it.qp == p.n_qp) {
    it.qp = 0;
    if (++it.h == p.heads) {
      it.h = 0;
      ++it.b;
      a3_iter_lengths(it, p);
    }
  }
  it.two = it.qp * 2 * A3_Q + A3_Q < p.T;
  return true;
}

// position of one MMA issuer in the flattened stream of (work item, key tile) pairs of its query tile
struct A3Cursor {
  A3Iter it;
  int j;
  uint32_t buf, par;        // S buffer of this position and the parity of its use
  uint32_t qi;              // items of this query tile so far, minus one (Q buffer = qi & 1)
  uint32_t kst, kph;        // K/V ring stage of this position and the parity of its use
  bool valid, skip;         // skip: an item WITHOUT this (second) query tile; only its K/V-ring phases are observed
};
// with_skipped (the Q K^T cursor of tile 1's issuer): the cursor also stops at the positions of items that have no
// second query tile, where the issuer only observes the kv_full phases one by one — an mbarrier parity wait is
// ambiguous once the barrier is more than one phase ahead of what the thread has seen
__device__ __forceinline__ void a3_enter_item(A3Cursor& c, const Attn3Params& p, int t, bool with_skipped) {
  while (c.valid) {
    c.skip = (t == 1 && !c.it.two);
    c.j = 0;
    if (!c.skip) {
      ++c.qi;
      return;
    }
    if (with_skipped) return;
    c.kst = (c.kst + c.it.n) % A3_STAGES;       // a cursor that never waits on the ring only needs the stage index
    c.valid = a3_iter_next(c.it, p);
  }
}
__device__ __forceinline__ void a3_init(A3Cursor& c, const Attn3Params& p, int t, bool with_skipped) {
  c.buf = 0; c.par = 0; c.qi = 0xffffffffu; c.kst = 0; c.kph = 0; c.j = 0; c.skip = false;
  c.valid = a3_iter_init(c.it, p);
  a3_enter_item(c, p, t, with_skipped);
}
__device__ __forceinline__ void a3_advance(A3Cursor& c, const Attn3Params& p, int t, bool with_skipped) {
  if (!c.skip && ++c.buf == A3_NBUF) {
    c.buf = 0;
    c.par ^= 1;
  }
  if (++c.kst == A3_STAGES) {
    c.kst = 0;
    c.kph ^= 1;
  }
  if (++c.j == c.it.n) {
    c.valid = a3_iter_next(c.it, p);
    a3_enter_item(c, p, t, with_skipped);
  }
}

__device__ __forceinline__ uint64_t a3_desc_mn(uint32_t saddr) {      // V tile [keys][64 d] as MN-major B operand
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1024 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__device__ __forceinline__ float a3_max3(float a, float b, float c) {
  float m;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(m) : "f"(a), "f"(b), "f"(c));
  return m;
}
__device__ __forceinline__ float a3_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// two fp32 -> one packed 16-bit pair in the kernel's operand format (bf16, or IEEE fp16 for precision="fp16")
template <bool FP16>
__device__ __forceinline__ uint32_t a3_pack16(float lo, float hi) {
  uint32_t r;
  if (FP16) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 2^x for two arguments on the FMA pipe.  x = n + f with n = floor(x) taken from the low mantissa bits of
// x + 1.5 * 2^23 (round-down add); 2^f = 1 + f (c1 + f (c2 + f c3)) on [0, 1) (minimax, 8.6e-5 relative);
// the result's exponent field is advanced by n with one shift-add.  x is clamped at -126 (2^x flushes to the
// smallest normal instead of wrapping the exponent field).
__device__ __forceinline__ void a3_ex2_poly2(float x0, float x1, float& p0, float& p1) {
  const uint64_t x = f32x2_pack(fmaxf(x0, -126.f), fmaxf(x1, -126.f));
  uint64_t r;
  asm("add.rm.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(f32x2_pack(12582912.f, 12582912.f)));
  const uint64_t fl = f32x2_add(r, f32x2_pack(-12582912.f, -12582912.f));          // floor(x)
  const uint64_t f = f32x2_fma(fl, f32x2_pack(-1.f, -1.f), x);                      // x - floor(x)
  uint64_t q = f32x2_fma(f, f32x2_pack(0.0770656615f, 0.0770656615f), f32x2_pack(0.2276464999f, 0.2276464999f));
  q = f32x2_fma(q, f, f32x2_pack(0.6951164603f, 0.6951164603f));
  q = f32x2_fma(q, f, f32x2_pack(1.f, 1.f));
  float q0, q1, r0, r1;
  f32x2_unpack(q, q0, q1);
  f32x2_unpack(r, r0, r1);
  p0 = __uint_as_float(__float_as_uint(q0) + (__float_as_uint(r0) << 23));
  p1 = __uint_as_float(__float_as_uint(q1) + (__float_as_uint(r1) << 23));
}

// FP16: q / k / v, P and the context are IEEE fp16 instead of bf16 (same tensor-core rate, three more mantissa bits;
// P <= 1 and the 2^8 lazy-rescale window keep the unnormalised P far inside fp16's range)
template <bool FP16>
__global__ void __launch_bounds__(A3_THREADS, 1)
attention_v3_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                    const __grid_constant__ CUtensorMap tmO, const Attn3Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                                   // [tile][2 buffers]
  uint8_t* sKV = smem + 4 * A3_QB;                      // [stage][K | V]
  uint8_t* sO = sKV + A3_STAGES * 2 * A3_KVB;           // [tile]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + A3_DATA);
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("aptai attention v3: dynamic shared memory base is not 1024-byte aligned\n");
    __trap();
  }
  uint64_t* q_full = bars + 0;                    // [tile][2]
  uint64_t* q_empty = bars + 4;                   // [tile][2]
  uint64_t* kv_full = bars + 8;                   // [STAGES]
  uint64_t* kv_empty = bars + 8 + A3_STAGES;      // [STAGES]
  uint64_t* s_full = bars + 8 + 2 * A3_STAGES;    // [tile][NBUF]
  uint64_t* p_full = s_full + 2 * A3_NBUF;        // [tile][NBUF]
  uint64_t* pv_done = p_full + 2 * A3_NBUF;       // [tile][NBUF]: P(j) V(j) of the position in that buffer completed
  uint64_t* o_full = pv_done + 2 * A3_NBUF;       // [tile]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  if (warp == A3_W_TMA && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmO);
  }
  if (warp == A3_W_MMA0 && lane == 0) {
    for (int i = 0; i < 4; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    for (int i = 0; i < A3_STAGES; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 2);              // one commit per query tile's issuer
    }
    for (int i = 0; i < 2 * A3_NBUF; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);                // the four warps of the tile's softmax group
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < 2; ++i) mbar_init(&o_full[i], 1);
    fence_mbar_init();
  }
  if (warp == A3_W_ALLOC) tmem_alloc(tmem_slot, A3_TCOLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == A3_W_TMA) {
    // ---------------------------------------------------------------- TMA producer (whole warp converged, one
    // elected lane issues: the loop state stays warp-uniform)
    {
      uint32_t kst = 0, kph = 0, qi0 = 0, qi1 = 0;
      A3Iter it;
      for (bool ok = a3_iter_init(it, p); ok; ok = a3_iter_next(it, p)) {
        {
          const uint32_t qb = qi0 & 1;
          mbar_wait_backoff(&q_empty[qb], ((qi0 >> 1) & 1) ^ 1, 100);
          if (elect_one()) {
            mbar_expect_tx(&q_full[qb], A3_QB);
            tma_load_3d(&tmQ, &q_full[qb], sQ + qb * A3_QB, it.h * A3_D, it.qp * 2 * A3_Q, it.bp);
          }
          ++qi0;
        }
        if (it.two) {
          const uint32_t qb = qi1 & 1;
          mbar_wait_backoff(&q_empty[2 + qb], ((qi1 >> 1) & 1) ^ 1, 100);
          if (elect_one()) {
            mbar_expect_tx(&q_full[2 + qb], A3_QB);
            tma_load_3d(&tmQ, &q_full[2 + qb], sQ + (2 + qb) * A3_QB, it.h * A3_D, it.qp * 2 * A3_Q + A3_Q, it.bp);
          }
          ++qi1;
        }
        for (int j = 0; j < it.n; ++j) {
          mbar_wait_backoff(&kv_empty[kst], kph ^ 1, 100);
          if (elect_one()) {
            mbar_expect_tx(&kv_full[kst], 2 * A3_KVB);
            uint8_t* dst = sKV + kst * 2 * A3_KVB;
            tma_load_3d(&tmKV, &kv_full[kst], dst, p.heads * A3_D + it.h * A3_D, j * A3_K, it.bp);
            tma_load_3d(&tmKV, &kv_full[kst], dst + A3_KVB, 2 * p.heads * A3_D + it.h * A3_D, j * A3_K, it.bp);
          }
          if (++kst == A3_STAGES) {
            kst = 0;
            kph ^= 1;
          }
        }
      }
    }
  } else if (warp == A3_W_MMA0 || warp == A3_W_MMA0 + 1) {
    // ---------------------------------------------------------------- MMA issuer of query tile t: the whole warp walks
    // the loop converged (barrier tests made warp-uniform by a vote), one elected lane issues — so cursors,
    // descriptors and TMEM addresses live in uniform registers and a tcgen05.mma costs a handful of instructions
    // instead of a register->uniform-register broadcast loop each
    {
      const int t = warp - A3_W_MMA0;
      constexpr uint32_t FMT_AB = FP16 ? 0u : ((1u << 7) | (1u << 10));      // a_format / b_format: 0 = f16, 1 = bf16
      constexpr uint32_t IDESC_S = (1u << 4) | FMT_AB | (static_cast<uint32_t>(A3_Q >> 4) << 24);
      constexpr uint32_t IDESC_PV = (1u << 4) | FMT_AB | (static_cast<uint32_t>(A3_Q >> 4) << 24) |
                                    (1u << 16) | (static_cast<uint32_t>(A3_D >> 3) << 17);   // B MN-major, N = 64
      const uint32_t ts0 = tmem_base + t * A3_NBUF * A3_K;
      const uint32_t to = tmem_base + A3_TO + t * A3_D;
      const uint64_t qd0 = umma_desc_sw128(smem_u32(sQ + t * 2 * A3_QB));
      const uint64_t kd0 = umma_desc_sw128(smem_u32(sKV));
      const uint64_t vd0 = a3_desc_mn(smem_u32(sKV) + A3_KVB);
      uint64_t* s_full_t = s_full + t * A3_NBUF;
      uint64_t* p_full_t = p_full + t * A3_NBUF;
      uint64_t* pv_done_t = pv_done + t * A3_NBUF;
      A3Cursor qk, pv;
      a3_init(pv, p, t, false);
      a3_init(qk, p, t, true);
      // Event loop on non-blocking barrier tests: a blocking wait for the next Q K^T's operands would hold back the
      // P V whose commit releases the very K/V stage the producer needs (deadlock across items without a second
      // query tile).  S(e + NBUF) reuses the buffer of P(e), so it is issued only after P(e) V(e) — same thread,
      // and tcgen05.mma execute in issue order.  The loop body is kept to a few dozen instructions (stage / buffer
      // indices advance by increments, descriptors by additions): a single thread feeds half of the tensor pipe.
      uint32_t idle = 0;
      int ahead = 0;                                    // Q K^T issued whose P V has not been issued yet
      while (pv.valid | qk.valid) {
        bool progress = false;
        if (pv.valid && ahead > 0 && __all_sync(0xffffffffu, mbar_test_wait(&p_full_t[pv.buf], pv.par))) {
          tc_fence_after();
          const int rem = pv.it.klen - pv.j * A3_K;
          const int nk = rem >= A3_K ? A3_K / 16 : (rem + 15) >> 4;
          const uint64_t vd = vd0 + pv.kst * (2 * A3_KVB >> 4);
          const uint32_t tp = ts0 + pv.buf * A3_K;
          const uint32_t first = pv.j != 0 ? 1u : 0u;
          if (elect_one()) {
            umma_bf16_ts(to, tp, vd, IDESC_PV, first);
            if (nk > 1) umma_bf16_ts(to, tp + 8, vd + 128, IDESC_PV, 1u);
            if (nk > 2) umma_bf16_ts(to, tp + 16, vd + 256, IDESC_PV, 1u);
            if (nk > 3) umma_bf16_ts(to, tp + 24, vd + 384, IDESC_PV, 1u);
            umma_commit(&kv_empty[pv.kst]);                   // this tile's Q K_j^T was issued earlier by this thread
            if (!pv.it.two) umma_commit(&kv_empty[pv.kst]);   // no second query tile: its share of the release
            umma_commit(&pv_done_t[pv.buf]);
            if (pv.j == pv.it.n - 1) umma_commit(&o_full[t]);
          }
          __syncwarp();
          a3_advance(pv, p, t, false);
          --ahead;
          progress = true;
        }
        if (qk.valid) {
          if (qk.skip) {
            if (__all_sync(0xffffffffu, mbar_test_wait(&kv_full[qk.kst], qk.kph))) {
              a3_advance(qk, p, t, true);
              progress = true;
            }
          } else if (ahead < A3_NBUF) {
            const uint32_t qb = qk.qi & 1;
            if (__all_sync(0xffffffffu, (qk.j != 0 || mbar_test_wait(&q_full[t * 2 + qb], (qk.qi >> 1) & 1)) &&
                                            mbar_test_wait(&kv_full[qk.kst], qk.kph))) {
              tc_fence_after();
              const int rem = qk.it.klen - qk.j * A3_K;
              const int nj = rem >= A3_K ? A3_K : (rem + 15) & ~15;
              const uint32_t idesc = IDESC_S | (static_cast<uint32_t>(nj >> 3) << 17);
              const uint64_t qd = qd0 + qb * (A3_QB >> 4);
              const uint64_t kd = kd0 + qk.kst * (2 * A3_KVB >> 4);
              const uint32_t ts = ts0 + qk.buf * A3_K;
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < A3_D / 16; ++k) umma_bf16(ts, qd + 2 * k, kd + 2 * k, idesc, k != 0 ? 1u : 0u);
                umma_commit(&s_full_t[qk.buf]);
                if (qk.j == qk.it.n - 1) umma_commit(&q_empty[t * 2 + qb]);
              }
              __syncwarp();
              a3_advance(qk, p, t, true);
              ++ahead;
              progress = true;
            }
          }
        }
        if (progress) idle = 0;
        else ++idle;
        if (idle > (APTAI_SPIN_LIMIT >> 4)) {
          if (lane == 0) printf("aptai attention v3: MMA issuer %d timed out (block %d)\n", t, (int)blockIdx.x);
          __trap();
        }
      }
    }
  } else if (warp < 8) {
    // ---------------------------------------------------------------- softmax groups: thread = one query row
    const int t = warp >> 2;
    const int q4 = warp & 3;
    const int row = q4 * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const uint32_t ts0 = t_lane + t * A3_NBUF * A3_K, to = t_lane + A3_TO + t * A3_D;
    uint8_t* so_tile = sO + t * A3_OB;
    uint8_t* so_row = so_tile + row * 128;
    uint32_t buf = 0, par = 0, it_n = 0;
    const uint64_t l2e = f32x2_pack(A3_LOG2E, A3_LOG2E);

    // Output of a finished item: O_t / l -> bf16 -> shared memory (SWIZZLE_128B rows) -> one TMA store per query tile;
    // lse.  It runs DEFERRED, inside the first key tile of the group's next item (after that tile's P is stored,
    // before the arrival that lets P V overwrite O_t): the wait for the item's last P V hides behind that softmax.
    bool pending = false;
    int e_b = 0, e_h = 0, e_q0 = 0;
    float e_m = 0.f, e_l = 1.f;
    bool e_live = false;
    auto epilogue = [&]() {
      // per WARP: its 32 rows go out with its own TMA store (box 64 x 32), so the four warps of a group never wait
      // for one another here — a group-wide barrier cost 12 % of the softmax warps' time (profiles/r02_attention_v3.md)
      mbar_wait(&o_full[t], it_n & 1);                  // every warp observes every phase (parity stays unambiguous)
      ++it_n;
      if (e_live) {
        if (lane == 0) tma_store_wait_read<0>();        // this warp's previous store has finished reading its slab
        __syncwarp();
        tc_fence_after();
        const int qrow = e_q0 + row;
        const float inv = 1.f / e_l;
        if (p.lse != nullptr && qrow < p.T)
          p.lse[(static_cast<long long>(e_b) * p.heads + e_h) * p.T + qrow] = e_m + log2f(e_l);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t r[32];
          tmem_ld32(to + c * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 4; ++u)
            *reinterpret_cast<uint4*>(so_row + (((c * 4 + u) ^ (row & 7)) << 4)) = make_uint4(
                a3_pack16<FP16>(__uint_as_float(r[8 * u]) * inv, __uint_as_float(r[8 * u + 1]) * inv),
                a3_pack16<FP16>(__uint_as_float(r[8 * u + 2]) * inv, __uint_as_float(r[8 * u + 3]) * inv),
                a3_pack16<FP16>(__uint_as_float(r[8 * u + 4]) * inv, __uint_as_float(r[8 * u + 5]) * inv),
                a3_pack16<FP16>(__uint_as_float(r[8 * u + 6]) * inv, __uint_as_float(r[8 * u + 7]) * inv));
        }
        tc_fence_before();
        fence_async_proxy();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tmO, so_tile + q4 * 32 * 128, e_h * A3_D, e_q0 + q4 * 32, e_b);
          tma_store_commit();
        }
      }
      pending = false;
    };

    A3Iter it;
    for (bool ok = a3_iter_init(it, p); ok; ok = a3_iter_next(it, p)) {
      if (t == 1 && !it.two) continue;
      float m_used = -INFINITY, l = 0.f;
      const int q0 = it.qp * 2 * A3_Q + t * A3_Q;
      const bool warp_live = q0 + q4 * 32 < p.T;
      for (int j = 0; j < it.n; ++j) {
        const uint32_t ts = ts0 + buf * A3_K;
        uint64_t* pf = &p_full[t * A3_NBUF + buf];
        // P(j-1) V(j-1) done: the barrier of the PREVIOUS position's buffer.  Its next commit belongs to position
        // j+2, which cannot be issued before this warp has arrived for j, and the commit before (position j-4)
        // completed before S(j) existed — so waiting on this parity is unambiguous even though most phases of these
        // barriers are never observed.
        uint64_t* prev_done = &pv_done[t * A3_NBUF + (buf == 0 ? A3_NBUF - 1 : buf - 1)];
        const uint32_t prev_par = buf == 0 ? par ^ 1 : par;
        mbar_wait(&s_full[t * A3_NBUF + buf], par);
        if (++buf == A3_NBUF) {
          buf = 0;
          par ^= 1;
        }
        if (!warp_live) {        // all 32 rows lie beyond the utterance: keep the protocol going, rows are never stored
          if (pending) epilogue();
          __syncwarp();
          if (lane == 0) mbar_arrive(pf);
          continue;
        }
        tc_fence_after();
        uint32_t s[64];
        uint32_t (&s_lo)[32] = *reinterpret_cast<uint32_t (*)[32]>(&s[0]);
        uint32_t (&s_hi)[32] = *reinterpret_cast<uint32_t (*)[32]>(&s[32]);
        tmem_ld32(ts, s_lo);
        tmem_ld32(ts + 32, s_hi);
        float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
        auto max_pass = [&](int i0, int i1) {
#pragma unroll
          for (int i = i0; i < i1; i += 8) {
            m0 = a3_max3(m0, __uint_as_float(s[i]), __uint_as_float(s[i + 1]));
            m1 = a3_max3(m1, __uint_as_float(s[i + 2]), __uint_as_float(s[i + 3]));
            m2 = a3_max3(m2, __uint_as_float(s[i + 4]), __uint_as_float(s[i + 5]));
            m3 = a3_max3(m3, __uint_as_float(s[i + 6]), __uint_as_float(s[i + 7]));
          }
        };
        const int valid = it.klen - j * A3_K;          // >= 1
        tmem_ld_wait();
        if (valid >= A3_K) {
          max_pass(0, 64);
        } else {
#pragma unroll
          for (int i = 0; i < 64; ++i)
            if (i >= valid) s[i] = 0xff800000u;        // -inf
          max_pass(0, 64);
        }
        const float mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) * A3_LOG2E;
        float factor = 1.f;
        if (mx > m_used + A3_RESCALE) {
          factor = exp2f(m_used - mx);                 // 0 on the first tile (m_used = -inf)
          m_used = mx;
        }
        if (__any_sync(0xffffffffu, factor != 1.f && j > 0)) {
          // rare after the first tiles: rescale the O rows once P(j-1) V(j-1) has completed
          mbar_wait(prev_done, prev_par);
          tc_fence_after();
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t r[32];
            tmem_ld32(to + c * 32, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * factor);
            tmem_st32(to + c * 32, r);
          }
        }
        l *= factor;
        const uint64_t nm = f32x2_pack(-m_used, -m_used);
        uint64_t acc0 = f32x2_pack(0.f, 0.f), acc1 = acc0;
        uint32_t pk[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float a0, a1, p0, p1;
          f32x2_unpack(f32x2_fma(f32x2_pack(__uint_as_float(s[2 * i]), __uint_as_float(s[2 * i + 1])), l2e, nm), a0, a1);
          if ((i & 7) < A3_POLY8) {
            a3_ex2_poly2(a0, a1, p0, p1);
          } else {
            p0 = a3_ex2(a0);
            p1 = a3_ex2(a1);
          }
          if (i & 1) acc1 = f32x2_add(acc1, f32x2_pack(p0, p1));
          else acc0 = f32x2_add(acc0, f32x2_pack(p0, p1));
          pk[i] = a3_pack16<FP16>(p0, p1);
        }
        float r0, r1;
        f32x2_unpack(f32x2_add(acc0, acc1), r0, r1);
        l += r0 + r1;
        tmem_st32(ts, pk);                             // P(j) over the first 32 columns of the S buffer just read
        if (pending) epilogue();                       // previous item's O_t (j == 0 only), before P V may overwrite it
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pf);
      }
      pending = true;
      e_b = it.bp; e_h = it.h; e_q0 = q0; e_m = m_used; e_l = l; e_live = warp_live;
    }
    if (pending) epilogue();
    if (lane == 0) tma_store_wait_all<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == A3_W_ALLOC) {
    tc_fence_after();
    tmem_dealloc(tmem_base, A3_TCOLS);
  }
}

}  // namespace aptai

using namespace aptai;

template <bool FP16>
static int launch_attention_v3(const CUtensorMap& tq, const CUtensorMap& tkv, const CUtensorMap& to,
                               const Attn3Params& p, cudaStream_t st) {
  auto kern = attention_v3_kernel<FP16>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, A3_SMEM);
    if (e != cudaSuccess) {
      set_error("attention_v3: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  const int grid = (p.items + p.per_cta - 1) / p.per_cta;
  kern<<<grid, A3_THREADS, A3_SMEM, st>>>(tq, tkv, to, p);
  return after_launch("attention_v3");
}

extern "C" int aptai_attention_fwd_v3(const void* qkv, void* ctx, float* lse, const int32_t* key_len, int B, int T,
                                      int heads, int half_fmt, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(qkv && ctx && key_len, "attention_v3: null pointer");
  APTAI_REQUIRE(B >= 1 && T >= 1 && heads >= 1, "attention_v3: bad shape");
  APTAI_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(ctx) & 15) == 0,
                "attention_v3: buffers must be 16-byte aligned");
  const int H = heads * A3_D;
  CUtensorMap tmq, tmkv, tmo;
  {
    uint64_t dims[3] = {static_cast<uint64_t>(3) * H, static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
    uint64_t strides[2] = {static_cast<uint64_t>(3) * H * 2, static_cast<uint64_t>(3) * H * 2 * T};
    uint32_t boxq[3] = {A3_D, A3_Q, 1};
    uint32_t boxkv[3] = {A3_D, A3_K, 1};
    if (int rc = encode_tmap_bf16(&tmq, qkv, 3, dims, strides, boxq, 1)) return rc;
    if (int rc = encode_tmap_bf16(&tmkv, qkv, 3, dims, strides, boxkv, 1)) return rc;
    uint64_t odims[3] = {static_cast<uint64_t>(H), static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
    uint64_t ostrides[2] = {static_cast<uint64_t>(H) * 2, static_cast<uint64_t>(H) * 2 * T};
    uint32_t boxo[3] = {A3_D, 32, 1};          // one store per softmax warp (32 query rows)
    if (int rc = encode_tmap_bf16(&tmo, ctx, 3, odims, ostrides, boxo, 1)) return rc;
  }
  Attn3Params p;
  p.key_len = key_len;
  p.lse = lse;
  p.B = B; p.T = T; p.heads = heads;
  p.n_qp = (T + 2 * A3_Q - 1) / (2 * A3_Q);
  p.items = B * heads * p.n_qp;
  p.per_cta = (p.items + num_sms() - 1) / num_sms();
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  p.reverse = traversal_reverse();
  return half_fmt ? launch_attention_v3<true>(tmq, tmkv, tmo, p, st) : launch_attention_v3<false>(tmq, tmkv, tmo, p, st);
}
