// tcgen05 / TMEM / TMA bf16 GEMM family for sm_100a.
//
// One persistent, warp-specialised kernel (TMA producer warp, single-thread MMA issuer, 8 epilogue warps) serves
//   * nn.Linear projections of the wav2vec2 encoder            (HF:429-434, 524-547, 566-573)
//   * the strided conv layers 1..6 as implicit GEMM            (HF:254-323)  [A rows = overlapping frame windows]
//   * the grouped positional conv (k=128, 16 groups)           (HF:329-368)  [A rows = shifted frame windows]
// by describing the A operand with a 4-D tensor map (channel, row parity, row/P, segment) so that the k-block
// `kb` of output row r reads physical row r*P + tap, tap = kb / kb_per_tap.
//
// Tile: 128 x BN x 64 per pipeline stage, accumulators in TMEM (double buffered when 2*BN <= 512 columns),
// epilogue straight from TMEM: bias / LayerNorm(512) / erf-GELU / fp32 residual / padded-row zeroing / fp32+bf16 stores.
#include "common.h"
#include "ptx.cuh"

namespace aptai {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int UMMA_K = 16;
// warps 0..7: epilogue, warp 8: TMA producer, warp 9: MMA issuer, warp 10: TMEM alloc, warp 11: idle.
// The single-thread producer / MMA roles sit in the HIGHEST warp ids: the scheduler arbitrates highest-warp-id first
// (B300_MICROARCH.md), so the thread that feeds the tensor core is never starved by the epilogue warps sharing its
// scheduler.
// Epilogue warps first, then the TMA producer, the MMA issuer and the TMEM allocator (see GemmCfg: EPI_W / W_TMA /
// W_MMA / W_ALLOC / THREADS).

struct GemmParams {
  int num_kb, kb_per_tap, P, a_col_per_nblk;
  int rows_per_seg, m_tiles_per_seg, n_tiles, num_tiles;
  const float* bias;
  const float* gamma;
  const float* beta;
  const float* residual;
  float* out_f32;
  __nv_bfloat16* out_bf16;
  long long ldo, out_seg_stride;
  const int* seg_valid_rows;
  int mask_seg_rows;
  int act;
  float ln_eps;
  int fp16;   // operands and the 16-bit output are IEEE fp16 instead of bf16
  const __nv_bfloat16* aux;   // act == 2: pre-activation u saved by the forward pass; out = acc * gelu'(u)
  __nv_bfloat16* out_pre;     // optional second 16-bit output: the value BEFORE the activation (training forward)
  int tma16;                  // the single 16-bit output leaves through shared memory + TMA stores (tensor map tmC)
  int reverse;                // walk the tiles from the last to the first (aptai_set_traversal)
  int red32;                  // in-place fp32 residual update h += acc + bias as TMA reduce-add stores (tmC, fp32)
  const float* l2_hint;       // red32: the rows the reduction will touch, prefetched into L2 one tile ahead
};

constexpr int LN_N = 512;     // row width of the fused-LayerNorm tiles (conv_dim)

template <int BN, bool CTA2, bool LN = false>
struct GemmCfg {
  // Epilogue warps (the LN code below is written for EPI_W / 4 column parts).  16 were measured against 8 on the
  // fused-LayerNorm conv tile and bought nothing (0.577 vs 0.578 ms on the conv-1 shape, profiles/conv_ln_one.py): the
  // two-pass epilogue is bound by the MUFU / packed-FMA work of the GELU and the normalisation, not by per-warp latency.
  static constexpr int EPI_W = 8;
  static constexpr int EPI_T = EPI_W * 32;
  static constexpr int W_TMA = EPI_W, W_MMA = EPI_W + 1, W_ALLOC = EPI_W + 2;
  static constexpr int THREADS = LN ? (EPI_W + 3) * 32 : 384;
  static constexpr int NPAIR = CTA2 ? 2 : 1;                     // CTAs cooperating on one tile (cta_group)
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;          // per CTA: its own 128 rows of A
  static constexpr int B_ROWS = BN / NPAIR;                      // rows of the B tile held by this CTA
  static constexpr int B_BYTES = (BN / NPAIR) * BLOCK_K * 2;     // per CTA: its share of the B columns
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // narrow tiles (grouped pos-conv, N = 48/64): the tensor core is fed by ~100-cycle tcgen05.mma issues of only
  // 32 cycles of work each, so two CTAs per SM (two issuing threads) are worth more than a deep ring
  static constexpr int CTAS_PER_SM = (BN <= 64 && !CTA2) ? 2 : 1;
  // the half-split LayerNorm tile (LN, BN = 256: see gemm_body) fits five 32 KB stages (pair) / three 48 KB stages
  // next to its staging, statistics and vector buffers
  static constexpr int STAGES = CTAS_PER_SM == 2 ? 3
                                : LN ? (CTA2 ? 5 : 3)
                                : (STAGE_BYTES > 64 * 1024 ? 2 : (STAGE_BYTES > 40 * 1024 ? 4 : 6));
  static constexpr int ACC_STRIDE = BN < 64 ? 64 : BN;
  static constexpr int ACC_STAGES = (2 * ACC_STRIDE <= 512) ? 2 : 1;
  static constexpr int TMEM_COLS = ACC_STAGES * ACC_STRIDE <= 128 ? 128 : (ACC_STAGES * ACC_STRIDE <= 256 ? 256 : 512);
  static constexpr int CHUNK = (BN % 64 == 0) ? 32 : 8;          // columns per tcgen05.ld in the epilogue
  static constexpr int BAR_BYTES = 256;
  static constexpr int LN_BYTES = LN ? 2 * 4 * BLOCK_M * sizeof(float2) : 0;   // LN statistics exchange
  static constexpr int STG_BYTES = EPI_W * 4096;                 // 4 KB staging buffer per epilogue warp
  // fused-LayerNorm tile: bias | gamma | beta of the whole 512-wide row live in shared memory, loaded once per CTA
  // (their per-element global loads were the top long-scoreboard stall of that epilogue: 27 % of the stall samples,
  // profiles/r01_gemm_convln.md).  The other tiles have no shared memory left for it (4 stages + 32 KB staging).
  static constexpr int VEC_BYTES = LN ? 3 * LN_N * 4 : 0;
  // bias of the current N tile, double buffered by tile parity (the per-chunk __ldg of the bias was the top
  // long-scoreboard stall of the FFN1 epilogue: 18 % of the epilogue warps' samples, profiles/r02_gemm_ffn.md)
  static constexpr int BIAS_BYTES = (BN % 64 == 0 && !LN) ? 2 * BN * 4 : 0;
  // layout: [stages | staging (1024-aligned: it is the source of SWIZZLE_128B TMA stores) | barriers | LN | vectors]
  static constexpr int OFF_STG = STAGES * STAGE_BYTES;
  static constexpr int OFF_BAR = OFF_STG + STG_BYTES;
  static constexpr int OFF_LN = OFF_BAR + BAR_BYTES;
  static constexpr int OFF_VEC = OFF_LN + LN_BYTES;
  static constexpr int OFF_BIAS = OFF_VEC + VEC_BYTES;
  static constexpr int SMEM_BYTES = OFF_BIAS + BIAS_BYTES;
};

template <int CH>
__device__ __forceinline__ void tmem_ld_chunk(uint32_t taddr, uint32_t (&r)[CH]);
template <>
__device__ __forceinline__ void tmem_ld_chunk<32>(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld32(taddr, r); }
template <>
__device__ __forceinline__ void tmem_ld_chunk<8>(uint32_t taddr, uint32_t (&r)[8]) { tmem_ld8(taddr, r); }

template <int BN, bool LN, bool CTA2>
__device__ __forceinline__ void gemm_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                                          const GemmParams& p) {
  using C = GemmCfg<BN, CTA2, LN>;
  // Half-split fused-LayerNorm tile (LN with BN = 256): the 512-wide row is produced as TWO 256-column accumulator
  // halves, each over the whole K loop (the A k-blocks are fetched twice, from L2), so that the epilogue's statistics
  // pass over half 0 runs under the MMAs of half 1 and its normalise / GELU / store pass over half 1 under the next
  // tile's MMAs of half 0.  One 512-column accumulator would fill the TMEM and make MMA and epilogue alternate:
  // measured in profiles/r02_gemm_convln.md (tensor pipe 58 % against 69 %, profiles/r02_gemm_convln_halfsplit.md).
  static_assert(!LN || BN == 256, "the fused-LayerNorm tile is the half-split 256-column tile");
  constexpr int NSUB = LN ? 2 : 1;             // accumulator halves per tile
  // the dynamic shared memory window starts 1024-byte aligned (no static shared memory in this kernel); checked, not
  // padded: the CTA-pair tile uses all but 768 bytes of the 227 KB
  extern __shared__ __align__(1024) uint8_t smem[];
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("aptai gemm: dynamic shared memory base is not 1024-byte aligned\n");
    __trap();
  }
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float2* ln_part = reinterpret_cast<float2*>(smem + C::OFF_LN);
  float* vecs = reinterpret_cast<float*>(smem + C::OFF_VEC);
  float* bias_s = reinterpret_cast<float*>(smem + C::OFF_BIAS);

  // warp index and cluster rank through a shuffle: provably warp-uniform for the compiler, so the single-issuer roles
  // below keep their loop state, descriptors and addresses in uniform registers (see the MMA role)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  // CTA pair (cta_group::2): rank 0 is the leader and issues every MMA; each CTA owns 128 rows of the 256-row
  // tile (its own TMEM lanes) and stages its own A rows plus half of the B columns.
  const uint32_t rank = CTA2 ? __shfl_sync(0xffffffffu, cluster_ctarank(), 0) : 0u;
  const int tile0 = CTA2 ? (blockIdx.x >> 1) : blockIdx.x;
  const int tile_step = CTA2 ? (gridDim.x >> 1) : gridDim.x;
  constexpr int TILE_M = BLOCK_M * C::NPAIR;

  constexpr int W_TMA = C::W_TMA, W_MMA = C::W_MMA, W_ALLOC = C::W_ALLOC, EPI_WARPS = C::EPI_W, EPI_THREADS = C::EPI_T;
  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.tma16 | p.red32) tma_prefetch_desc(&tmC);
  }
  if (warp == W_MMA && lane == 0) {
    for (int i = 0; i < C::STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], EPI_WARPS * C::NPAIR);
    }
    fence_mbar_init();
  }
  if (warp == W_ALLOC) {
    if (CTA2) tmem_alloc_cg2(tmem_slot, C::TMEM_COLS);
    else tmem_alloc(tmem_slot, C::TMEM_COLS);
  }
  tc_fence_before();
  if (CTA2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == W_TMA) {
    // ------------------------------------------------------------------ TMA producer: the whole warp walks the loop
    // converged, one elected lane issues
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile_i = tile0; tile_i < p.num_tiles; tile_i += tile_step) {
        const int tile = p.reverse ? p.num_tiles - 1 - tile_i : tile_i;
        for (int sub = 0; sub < NSUB; ++sub) {
        const int n_blk = LN ? sub : tile % p.n_tiles;
        const int mt = LN ? tile : tile / p.n_tiles;
        const int seg = mt / p.m_tiles_per_seg;
        const int r0 = (mt - seg * p.m_tiles_per_seg) * TILE_M + static_cast<int>(rank) * BLOCK_M;
        const int a_col0 = n_blk * p.a_col_per_nblk;
        int tap = 0, kc = 0;                       // k-block kb = tap * kb_per_tap + kc, advanced by increments
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait_backoff(&empty_bar[stage], phase ^ 1, 64);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          const int tq = p.P == 1 ? tap : tap / p.P;
          if (elect_one()) {
            if (CTA2) {
              // both CTAs' bytes are counted on the LEADER's barrier; only the leader arms it
              if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
              const uint32_t fb = map_to_cta(&full_bar[stage], 0);
              tma_load_4d_cg2(&tmA, fb, sa, kc * BLOCK_K + a_col0, tap - tq * p.P, r0 + tq, seg);
              tma_load_2d_cg2(&tmB, fb, sb, kb * BLOCK_K, n_blk * BN + static_cast<int>(rank) * C::B_ROWS);
            } else {
              mbar_expect_tx(&full_bar[stage], C::STAGE_BYTES);
              tma_load_4d(&tmA, &full_bar[stage], sa, kc * BLOCK_K + a_col0, tap - tq * p.P, r0 + tq, seg);
              tma_load_2d(&tmB, &full_bar[stage], sb, kb * BLOCK_K, n_blk * BN);
            }
          }
          __syncwarp();
          if (++kc == p.kb_per_tap) {
            kc = 0;
            ++tap;
          }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        }   // sub
      }
    }
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer: whole warp converged, one
    // elected lane issues.  Under `if (lane == 0)` every tcgen05.mma cost ~21 SASS instructions (operands moved from
    // per-thread to uniform registers through an R2UR.BROADCAST + ELECT + BRA.U.ANY loop): ~500 issue cycles per
    // k-block against 512 cycles of tensor work for the 256x256x64 pair tile — the issuing thread was co-critical
    // with the tensor pipe.  With warp-uniform control flow the loop state lives in uniform registers.
    if (rank == 0) {
      const uint32_t IDESC = p.fp16 ? umma_idesc_f16(TILE_M, BN) : umma_idesc_bf16(TILE_M, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t smem_base = smem_u32(smem);
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step) {
        for (int sub = 0; sub < NSUB; ++sub) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::ACC_STRIDE;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_base + stage * C::STAGE_BYTES;
          const uint32_t b_base = a_base + C::A_BYTES;
          if (elect_one()) {
            const uint64_t adesc0 = umma_desc_sw128(a_base);
            const uint64_t bdesc0 = umma_desc_sw128(b_base);
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
              const uint64_t adesc = adesc0 + (k * UMMA_K * 2 >> 4);
              const uint64_t bdesc = bdesc0 + (k * UMMA_K * 2 >> 4);
              if (CTA2) umma_bf16_cg2(d_tmem, adesc, bdesc, IDESC, (kb | k) != 0 ? 1u : 0u);
              else umma_bf16(d_tmem, adesc, bdesc, IDESC, (kb | k) != 0 ? 1u : 0u);
            }
            // smem slot reusable (in both CTAs of the pair) once these MMAs have read it
            if (CTA2) umma_commit_cg2(&empty_bar[stage], 0x3);
            else umma_commit(&empty_bar[stage]);
            if (kb == p.num_kb - 1) {              // accumulator complete -> epilogue warps (of both CTAs)
              if (CTA2) umma_commit_cg2(&tfull_bar[acc], 0x3);
              else umma_commit(&tfull_bar[acc]);
            }
          }
          __syncwarp();
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (C::ACC_STAGES == 2) {
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
        } else {
          acc_phase ^= 1;
        }
        }   // sub
      }
    }
  } else if (warp < EPI_WARPS) {
    // ------------------------------------------------------------------ epilogue: TMEM -> registers -> global
    constexpr int CH = C::CHUNK;
    const int q = warp & 3;                  // TMEM lane quadrant this warp may read
    const int half = warp >> 2;
    constexpr int HALF_N = BN / 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    int ln_buf = 0;
    uint32_t ln2_phase = 0;                 // half-split LayerNorm tile: parity of tfull[0] / tfull[1] (one use per tile)
    (void)ln2_phase;
    const uint32_t tempty_leader0 = CTA2 ? map_to_cta(&tempty_bar[0], 0) : 0u;
    if constexpr (LN) {
      for (int i = threadIdx.x; i < LN_N; i += EPI_THREADS) {
        vecs[i] = p.bias ? __ldg(p.bias + i) : 0.f;
        vecs[LN_N + i] = __ldg(p.gamma + i);
        vecs[2 * LN_N + i] = __ldg(p.beta + i);
      }
      named_bar_sync(1, EPI_THREADS);
    }

    uint32_t tpar = 0;                       // tile parity: bias buffer of this tile
    for (int tile_i = tile0; tile_i < p.num_tiles; tile_i += tile_step, tpar ^= 1) {
      const int tile = p.reverse ? p.num_tiles - 1 - tile_i : tile_i;
      const int n_blk = LN ? 0 : tile % p.n_tiles;
      const int mt = LN ? tile : tile / p.n_tiles;
      const int seg = mt / p.m_tiles_per_seg;
      const int row_in_tile = q * 32 + lane;
      const float* bias_t = bias_s + tpar * BN;
      if constexpr (C::BIAS_BYTES > 0) {
        // this tile's bias -> shared memory, before the accumulator is awaited.  Double buffered: the barrier below
        // keeps the eight warps within one tile of each other, so nobody still reads the buffer being refilled.
        if (p.bias != nullptr) {
          if (static_cast<int>(threadIdx.x) < BN) bias_s[tpar * BN + threadIdx.x] = __ldg(p.bias + n_blk * BN + threadIdx.x);
          named_bar_sync(1, EPI_THREADS);
        }
      }
      const int r = (mt - seg * p.m_tiles_per_seg) * TILE_M + static_cast<int>(rank) * BLOCK_M + row_in_tile;
      const bool valid_row = r < p.rows_per_seg;
      const long long out_row = static_cast<long long>(seg) * p.out_seg_stride + r;
      bool zero_row = false;
      if (p.seg_valid_rows != nullptr && valid_row) {
        const long long ms = out_row / p.mask_seg_rows;
        zero_row = (out_row - ms * p.mask_seg_rows) >= __ldg(p.seg_valid_rows + ms);
      }
      const long long out_off = out_row * p.ldo;
      const int n_tile0 = n_blk * BN;

      const float* resid_hint = p.residual != nullptr ? p.residual : p.l2_hint;
      if (resid_hint != nullptr) {
        // pull the NEXT tile's residual rows towards L2 while this tile is processed: the fp32 residual stream
        // makes the K=1024 projections memory-bound, and two epilogue warps per scheduler cannot keep enough
        // HBM requests in flight on their own
        const int nt_i = tile_i + tile_step;
        const int nt = p.reverse ? p.num_tiles - 1 - nt_i : nt_i;
        if (nt_i < p.num_tiles) {
          const int nmt = nt / p.n_tiles;
          const int nseg = nmt / p.m_tiles_per_seg;
          const int nr = (nmt - nseg * p.m_tiles_per_seg) * TILE_M + static_cast<int>(rank) * BLOCK_M + row_in_tile;
          if (nr < p.rows_per_seg) {
            const float* np_ = resid_hint + (static_cast<long long>(nseg) * p.out_seg_stride + nr) * p.ldo +
                               (nt % p.n_tiles) * BN + half * HALF_N;
#pragma unroll
            for (int i = 0; i < HALF_N * 4 / 128; ++i)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(np_ + i * 32));
          }
        }
      }
      if constexpr (!LN) {
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
      }
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (LN ? 0 : acc * C::ACC_STRIDE);

      if constexpr (LN) {
        // ---- half-split fused LayerNorm(512) + GELU tile: thread = one row x 128 columns of EACH 256-column
        // accumulator half.  Pass 1 (shifted single-pass statistics of acc + bias) runs on half 0 while the tensor
        // core still works on half 1; pass 2 (normalise, GELU, 16-bit slabs, TMA stores) releases half 0 to the next
        // tile's MMAs before it turns to half 1.
        constexpr int HN = 256;                               // columns per accumulator half
        constexpr int NPART = EPI_WARPS / 4;                  // threads per row (2)
        constexpr int PART_N = HN / NPART;                    // columns per thread and half (128)
        const int part = warp >> 2;
        const int cb = part * PART_N;
        float pivot = 0.f;
        uint64_t s1a = f32x2_pack(0.f, 0.f), s1b = s1a, s2a = s1a, s2b = s1a, npiv = s1a;
        uint32_t nx[32];
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
          mbar_wait(&tfull_bar[hh], ln2_phase);
          tc_fence_after();
          const uint32_t t_h = t_row + hh * HN + cb;
          const float* bias_h = vecs + hh * HN + cb;
          tmem_ld32(t_h, nx);
          for (int c = 0; c < PART_N; c += 32) {
            tmem_ld_wait();
            uint32_t rr[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) rr[i] = nx[i];
            if (c + 32 < PART_N) tmem_ld32(t_h + c + 32, nx);
            if (hh == 0 && c == 0) {
              pivot = __uint_as_float(rr[0]) + bias_h[0];
              npiv = f32x2_pack(-pivot, -pivot);
            }
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias_h + c + i);
              const uint64_t d0 = f32x2_add(f32x2_add(f32x2_pack(__uint_as_float(rr[i]), __uint_as_float(rr[i + 1])),
                                                      f32x2_pack(b4.x, b4.y)), npiv);
              const uint64_t d1 = f32x2_add(f32x2_add(f32x2_pack(__uint_as_float(rr[i + 2]), __uint_as_float(rr[i + 3])),
                                                      f32x2_pack(b4.z, b4.w)), npiv);
              s1a = f32x2_add(s1a, d0);
              s1b = f32x2_add(s1b, d1);
              s2a = f32x2_fma(d0, d0, s2a);
              s2b = f32x2_fma(d1, d1, s2b);
            }
          }
        }
        float s1x, s1y, s2x, s2y;
        f32x2_unpack(f32x2_add(s1a, s1b), s1x, s1y);
        f32x2_unpack(f32x2_add(s2a, s2b), s2x, s2y);
        const float s1 = s1x + s1y, s2 = s2x + s2y;
        constexpr float inv_n = 1.0f / (2 * PART_N);
        const float mean_p = pivot + s1 * inv_n;
        const float m2_p = fmaxf(s2 - s1 * s1 * inv_n, 0.f);
        float2* buf = ln_part + ln_buf * NPART * BLOCK_M;
        buf[part * BLOCK_M + row_in_tile] = make_float2(mean_p, m2_p);
        tmem_ld32(t_row + cb, nx);                     // first chunk of pass 2, in flight across the exchange
        named_bar_sync(1, EPI_THREADS);
        ln_buf ^= 1;
        float msum = 0.f, m2sum = 0.f;
        float2 st[NPART];
#pragma unroll
        for (int k = 0; k < NPART; ++k) {
          st[k] = buf[k * BLOCK_M + row_in_tile];
          msum += st[k].x;
          m2sum += st[k].y;
        }
        const float mean = msum * (1.0f / NPART);
#pragma unroll
        for (int k = 0; k < NPART; ++k)
          m2sum = fmaf((st[k].x - mean) * (st[k].x - mean), static_cast<float>(2 * PART_N), m2sum);
        const float var = m2sum * (1.0f / LN_N);
        const float rstd = rsqrtf(var + p.ln_eps);
        const uint64_t rs2 = f32x2_pack(rstd, rstd), nm2 = f32x2_pack(-mean * rstd, -mean * rstd);
        uint4* sb = reinterpret_cast<uint4*>(smem + C::OFF_STG + warp * 4096);
        const int r_first = r - lane;
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t t_h = t_row + hh * HN + cb;
          const int col_h = hh * HN + cb;                  // first of this thread's 128 columns in the 512-wide row
          if (hh == 1) tmem_ld32(t_h, nx);
          for (int c = 0; c < PART_N; c += 32) {
            tmem_ld_wait();
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(nx[i]);
            if (c + 32 < PART_N) {
              tmem_ld32(t_h + c + 32, nx);
            } else {
              // this half is in registers: hand it back to the MMA issuer (of the pair's leader)
              tc_fence_before();
              __syncwarp();
              if (lane == 0) {
                if (CTA2) mbar_arrive_cluster_relaxed(tempty_leader0 + hh * 8);
                else mbar_arrive(&tempty_bar[hh]);
              }
            }
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(vecs + col_h + c + i);
              const float4 g4 = *reinterpret_cast<const float4*>(vecs + LN_N + col_h + c + i);
              const float4 e4 = *reinterpret_cast<const float4*>(vecs + 2 * LN_N + col_h + c + i);
              uint64_t t0 = f32x2_add(f32x2_pack(v[i], v[i + 1]), f32x2_pack(b4.x, b4.y));
              uint64_t t1 = f32x2_add(f32x2_pack(v[i + 2], v[i + 3]), f32x2_pack(b4.z, b4.w));
              t0 = f32x2_fma(f32x2_fma(t0, rs2, nm2), f32x2_pack(g4.x, g4.y), f32x2_pack(e4.x, e4.y));
              t1 = f32x2_fma(f32x2_fma(t1, rs2, nm2), f32x2_pack(g4.z, g4.w), f32x2_pack(e4.z, e4.w));
              f32x2_unpack(t0, v[i], v[i + 1]);
              f32x2_unpack(t1, v[i + 2], v[i + 3]);
            }
            if (p.act == 1) {
#pragma unroll
              for (int i = 0; i < 32; i += 2) gelu_fast2(v[i], v[i + 1]);
            }
            if (zero_row) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = 0.f;
            }
            const int hsel = (c >> 5) & 1;
            if (hsel == 0) {
              if (lane == 0) tma_store_wait_read<0>();
              __syncwarp();
            }
            {
              uint4 pk[4];
              pack32_h16(v, pk, p.fp16);     // one format branch per 32 values (a per-pair select costs two F2FP issue slots)
#pragma unroll
              for (int u = 0; u < 4; ++u) sb[lane * 8 + ((hsel * 4 + u) ^ (lane & 7))] = pk[u];
            }
            if (hsel == 1) {
              fence_async_proxy();
              __syncwarp();
              if (lane == 0) {
                tma_store_3d(&tmC, sb, col_h + c - 32, r_first, seg);
                tma_store_commit();
              }
            }
          }
        }
        ln2_phase ^= 1;
      } else {
      // residual block of the first chunk, requested before the accumulator is even complete (coalesced path)
      float4 res_next[8];
      if constexpr (CH == 32) {
        if (p.residual) {
          const int lrow0 = lane >> 3, lunit0 = lane & 7;
          const long long offr = out_off - static_cast<long long>(lane) * p.ldo + n_tile0 + half * HALF_N;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = i * 4 + lrow0;
            res_next[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r - lane + rr < p.rows_per_seg)
              res_next[i] = __ldg(reinterpret_cast<const float4*>(p.residual + offr + rr * p.ldo + lunit0 * 4));
          }
        }
      }
      // software pipeline: the tcgen05.ld of chunk c+1 is in flight while chunk c is processed
      uint32_t nxt[CH];
      tmem_ld_chunk<CH>(t_row + half * HALF_N, nxt);
      for (int c = half * HALF_N; c < (half + 1) * HALF_N; c += CH) {
        tmem_ld_wait();
        float v[CH];
        const int n0 = n_tile0 + c;
#pragma unroll
        for (int i = 0; i < CH; ++i) v[i] = __uint_as_float(nxt[i]);
        if (c + CH < (half + 1) * HALF_N) tmem_ld_chunk<CH>(t_row + c + CH, nxt);
        if (p.bias) {
          if constexpr (C::BIAS_BYTES > 0) {
#pragma unroll
            for (int i = 0; i < CH; i += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias_t + c + i);
              v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < CH; i += 4) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + i));
              v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
            }
          }
        }
        if constexpr (CH == 32) {
          // ---- coalesced path: transpose through a warp-private, XOR-swizzled 4 KB buffer so that every global
          // access covers whole 128-byte (fp32) / 64-byte (bf16) row segments instead of 32 different rows
          float* stg = reinterpret_cast<float*>(smem + C::OFF_STG) + warp * 1024;
          const int r_first = r - lane;                                  // first row of this warp's 32-row group
          const long long off0 = out_off - static_cast<long long>(lane) * p.ldo + n0;
          const int lrow = lane >> 3, lunit = lane & 7;
          // 16-bit store of v[] (thread = row) as whole 64-byte row segments
          auto store16 = [&](__nv_bfloat16* dst) {
            uint4* sb = reinterpret_cast<uint4*>(stg);                    // 128-byte row pitch, units 0..3 used
            {
              uint4 pk[4];
              pack32_h16(v, pk, p.fp16);     // one format branch per 32 values (a per-pair select costs two F2FP issue slots)
#pragma unroll
              for (int u = 0; u < 4; ++u) sb[lane * 8 + (u ^ (lane & 7))] = pk[u];
            }
            __syncwarp();
            const int bu = lane & 3;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = i * 8 + ((lane >> 2) & 1) * 4 + (lane >> 3);
              const uint4 x = sb[rr * 8 + (bu ^ (rr & 7))];
              if (r_first + rr < p.rows_per_seg)
                *reinterpret_cast<uint4*>(dst + off0 + rr * p.ldo + bu * 8) = x;
            }
            __syncwarp();
          };
          if (p.red32) {
            // ---- in-place residual update h += acc + bias: the 32-row x 128-byte fp32 slab goes to the staging buffer
            // and ONE TMA reduce-add store applies it at the L2 — the residual is never loaded into the SM
            if (lane == 0) tma_store_wait_read<0>();       // the slab's previous store has been read out
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 8; ++u)
              *reinterpret_cast<float4*>(stg + lane * 32 + ((u ^ (lane & 7)) << 2)) =
                  make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
            fence_async_proxy();
            __syncwarp();
            if (lane == 0) {
              tma_reduce_add_3d(&tmC, stg, n0, r_first, seg);
              tma_store_commit();
            }
            continue;
          }
          if (p.tma16) {
            // ---- single 16-bit output (QKV, FFN1, conv-free projections): two 32-column chunks fill one 32-row x
            // 128-byte slab of the warp's staging buffer in the SWIZZLE_128B pattern, then ONE TMA store writes it
            // (clipped at the segment's last row by the tensor map: no per-row predicate, no LDS / STG round trip)
            if (p.act == 1) {
#pragma unroll
              for (int i = 0; i < CH; i += 2) gelu_fast2(v[i], v[i + 1]);
            }
            if (zero_row) {
#pragma unroll
              for (int i = 0; i < CH; ++i) v[i] = 0.f;
            }
            const int hsel = (c >> 5) & 1;                 // which half of the 128-byte row this chunk fills
            if (hsel == 0) {
              if (lane == 0) tma_store_wait_read<0>();     // the slab's previous store has been read out
              __syncwarp();
            }
            uint4* sb = reinterpret_cast<uint4*>(stg);
            {
              uint4 pk[4];
              pack32_h16(v, pk, p.fp16);     // one format branch per 32 values (a per-pair select costs two F2FP issue slots)
#pragma unroll
              for (int u = 0; u < 4; ++u) sb[lane * 8 + ((hsel * 4 + u) ^ (lane & 7))] = pk[u];
            }
            if (hsel == 1) {
              fence_async_proxy();
              __syncwarp();
              if (lane == 0) {
                tma_store_3d(&tmC, stg, n0 - 32, r_first, seg);
                tma_store_commit();
              }
            }
            continue;
          }
          if (p.out_pre) store16(p.out_pre);
          if (p.act == 1) {
            if (p.out_f32 == nullptr) {            // result only leaves in 16 bits: the cheap form (see gelu_fast2)
#pragma unroll
              for (int i = 0; i < CH; i += 2) gelu_fast2(v[i], v[i + 1]);
            } else {
#pragma unroll
              for (int i = 0; i < CH; i += 2) gelu_erf2(v[i], v[i + 1]);
            }
          } else if (p.act == 2) {
            // dgrad through the GELU: v *= gelu'(u), u = the forward's pre-activation (bf16).  The 32x32 block of u is
            // fetched as whole 64-byte row segments (4 lanes per row, 8 rows per instruction) and transposed through
            // the warp's staging buffer, mirroring store16
            uint4* sb = reinterpret_cast<uint4*>(stg);
            const int bu = lane & 3;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = i * 8 + ((lane >> 2) & 1) * 4 + (lane >> 3);
              uint4 x = make_uint4(0u, 0u, 0u, 0u);
              if (r_first + rr < p.rows_per_seg)
                x = __ldg(reinterpret_cast<const uint4*>(p.aux + off0 + rr * p.ldo + bu * 8));
              sb[rr * 8 + (bu ^ (rr & 7))] = x;
            }
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const uint4 u4 = sb[lane * 8 + (u ^ (lane & 7))];
              const uint32_t uw[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 uf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&uw[j]));
                gelu_erf_grad2_mul(v[8 * u + 2 * j], v[8 * u + 2 * j + 1], uf.x, uf.y);
              }
            }
            __syncwarp();
          }
          if (p.residual) {
            // the residual block of THIS chunk was requested one chunk ago (res_next): its global latency is hidden
            // behind the previous chunk's work instead of being exposed four times per tile
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int rr = i * 4 + lrow;
              *reinterpret_cast<float4*>(stg + rr * 32 + ((lunit ^ (rr & 7)) << 2)) = res_next[i];
            }
            __syncwarp();
            if (c + CH < (half + 1) * HALF_N) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int rr = i * 4 + lrow;
                res_next[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r_first + rr < p.rows_per_seg)
                  res_next[i] = __ldg(reinterpret_cast<const float4*>(p.residual + off0 + CH + rr * p.ldo + lunit * 4));
              }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float4 r4 = *reinterpret_cast<const float4*>(stg + lane * 32 + ((u ^ (lane & 7)) << 2));
              v[4 * u] += r4.x; v[4 * u + 1] += r4.y; v[4 * u + 2] += r4.z; v[4 * u + 3] += r4.w;
            }
            __syncwarp();
          }
          if (zero_row) {
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] = 0.f;
          }
          if (p.out_f32) {
#pragma unroll
            for (int u = 0; u < 8; ++u)
              *reinterpret_cast<float4*>(stg + lane * 32 + ((u ^ (lane & 7)) << 2)) =
                  make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int rr = i * 4 + lrow;
              const float4 x = *reinterpret_cast<const float4*>(stg + rr * 32 + ((lunit ^ (rr & 7)) << 2));
              if (r_first + rr < p.rows_per_seg)
                *reinterpret_cast<float4*>(p.out_f32 + off0 + rr * p.ldo + lunit * 4) = x;
            }
            __syncwarp();
          }
          if (p.out_bf16) store16(p.out_bf16);
        } else {
        if (p.out_pre && valid_row) {      // narrow tiles (48-wide groups): row-per-thread 16-byte stores
          uint4* op = reinterpret_cast<uint4*>(p.out_pre + out_off + n0);
#pragma unroll
          for (int i = 0; i < CH; i += 8)
            op[i / 8] = make_uint4(pack_h16(v[i], v[i + 1], p.fp16), pack_h16(v[i + 2], v[i + 3], p.fp16),
                                   pack_h16(v[i + 4], v[i + 5], p.fp16), pack_h16(v[i + 6], v[i + 7], p.fp16));
        }
        if (p.act == 1) {
          if (p.out_f32 == nullptr) {
#pragma unroll
            for (int i = 0; i < CH; i += 2) gelu_fast2(v[i], v[i + 1]);
          } else {
#pragma unroll
            for (int i = 0; i < CH; i += 2) gelu_erf2(v[i], v[i + 1]);
          }
        }
        if (valid_row) {
          if (p.residual) {
            const float4* rp = reinterpret_cast<const float4*>(p.residual + out_off + n0);
#pragma unroll
            for (int i = 0; i < CH; i += 4) {
              const float4 r4 = __ldg(rp + i / 4);
              v[i] += r4.x; v[i + 1] += r4.y; v[i + 2] += r4.z; v[i + 3] += r4.w;
            }
          }
          if (zero_row) {
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] = 0.f;
          }
          if (p.out_f32) {
            float4* op = reinterpret_cast<float4*>(p.out_f32 + out_off + n0);
#pragma unroll
            for (int i = 0; i < CH; i += 4) op[i / 4] = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
          }
          if (p.out_bf16) {
            uint4* op = reinterpret_cast<uint4*>(p.out_bf16 + out_off + n0);
#pragma unroll
            for (int i = 0; i < CH; i += 8)
              op[i / 8] = make_uint4(pack_h16(v[i], v[i + 1], p.fp16), pack_h16(v[i + 2], v[i + 3], p.fp16),
                                     pack_h16(v[i + 4], v[i + 5], p.fp16), pack_h16(v[i + 6], v[i + 7], p.fp16));
          }
        }
        }
      }
      }   // !LN
      if constexpr (!LN) {
      // all tcgen05.ld of this warp have completed (wait::ld above) -> hand the accumulator back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CTA2) mbar_arrive_cluster_relaxed(tempty_leader0 + acc * 8);
        else mbar_arrive(&tempty_bar[acc]);
      }
      if (C::ACC_STAGES == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      } else {
        acc_phase ^= 1;
      }
      }
    }
  }

  if (warp < EPI_WARPS && lane == 0 && (p.tma16 | p.red32)) tma_store_wait_all<0>();   // shared memory stays valid until read
  tc_fence_before();
  if (CTA2) cluster_sync_all();
  else __syncthreads();
  if (warp == W_ALLOC) {
    tc_fence_after();
    if (CTA2) tmem_dealloc_cg2(tmem_base, C::TMEM_COLS);
    else tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

template <int BN, bool LN>
__global__ void __launch_bounds__((GemmCfg<BN, false, LN>::THREADS), (GemmCfg<BN, false, LN>::CTAS_PER_SM))
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  gemm_body<BN, LN, false>(tmA, tmB, tmC, p);
}

// CTA-pair variant: cluster of 2, tcgen05.mma.cta_group::2 (M = 256), half of B per CTA
template <int BN, bool LN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__((GemmCfg<BN, true, LN>::THREADS), 1)
gemm_bf16_tcgen05_2cta_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                              const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  gemm_body<BN, LN, true>(tmA, tmB, tmC, p);
}

template <int BN, bool LN>
static int launch_gemm_2cta(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p,
                            cudaStream_t st) {
  using C = GemmCfg<BN, true, LN>;
  auto kern = gemm_bf16_tcgen05_2cta_kernel<BN, LN>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("gemm(2cta): cudaFuncSetAttribute(%d bytes): %s", C::SMEM_BYTES, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  int clusters = num_sms() / 2;
  if (p.num_tiles < clusters) clusters = p.num_tiles;
  kern<<<2 * clusters, C::THREADS, C::SMEM_BYTES, st>>>(ta, tb, tc, p);
  return after_launch("gemm_bf16_tcgen05_2cta");
}

template <int BN, bool LN>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p,
                       cudaStream_t st) {
  using C = GemmCfg<BN, false, LN>;
  auto kern = gemm_bf16_tcgen05_kernel<BN, LN>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("gemm: cudaFuncSetAttribute(%d bytes): %s", C::SMEM_BYTES, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  const int slots = num_sms() * C::CTAS_PER_SM;
  int grid = p.num_tiles < slots ? p.num_tiles : slots;
  kern<<<grid, C::THREADS, C::SMEM_BYTES, st>>>(ta, tb, tc, p);
  return after_launch("gemm_bf16_tcgen05");
}

}  // namespace aptai

using namespace aptai;

extern "C" int aptai_gemm_bf16(const aptai_gemm_args* g, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(g != nullptr, "gemm: null args");
  APTAI_REQUIRE(g->a && g->w, "gemm: null operand");
  APTAI_REQUIRE(g->out_f32 || g->out_bf16, "gemm: no output pointer");
  APTAI_REQUIRE(g->P >= 1 && g->taps >= 1 && g->kb_per_tap >= 1, "gemm: bad tap geometry");
  APTAI_REQUIRE(g->segs >= 1 && g->rows_per_seg >= 1 && g->a_rows >= 1, "gemm: bad row geometry");
  APTAI_REQUIRE(g->a_row_stride % 8 == 0 && g->a_seg_stride % 8 == 0, "gemm: A strides must be multiples of 8");
  APTAI_REQUIRE((reinterpret_cast<uintptr_t>(g->a) & 15) == 0 && (reinterpret_cast<uintptr_t>(g->w) & 15) == 0,
                "gemm: operands must be 16-byte aligned");
  APTAI_REQUIRE(g->ldo % 8 == 0, "gemm: ldo must be a multiple of 8");
  APTAI_REQUIRE(g->seg_valid_rows == nullptr || g->mask_seg_rows >= 1, "gemm: mask_seg_rows must be >= 1");
  int bn = g->block_n;
  if (g->ln) {
    APTAI_REQUIRE(g->N == 512 && (bn == 0 || bn == 256), "gemm: fused LayerNorm needs N == 512 and block_n 0 or 256");
    APTAI_REQUIRE(g->gamma && g->beta, "gemm: fused LayerNorm needs gamma/beta");
    // the half-split tile: two 256-column accumulator halves per 512-wide row, epilogue overlapped with the MMAs
    bn = 256;
  } else if (bn == 0) {
    bn = (g->N % 256 == 0) ? 256 : (g->N % 128 == 0) ? 128 : (g->N % 64 == 0) ? 64 : (g->N % 48 == 0) ? 48 : 0;
  }
  APTAI_REQUIRE(bn == 48 || bn == 64 || bn == 128 || bn == 256, "gemm: unsupported block_n for N=%d", g->N);
  APTAI_REQUIRE(g->N % bn == 0, "gemm: N=%d not a multiple of block_n=%d", g->N, bn);
  const int n_tiles = g->ln ? 1 : g->N / bn;     // the half-split tile owns the whole row: its two halves are sub-tiles
  APTAI_REQUIRE(g->act != 2 || (g->aux != nullptr && !g->ln && bn % 64 == 0),
                "gemm: act=2 (GELU dgrad) needs aux and a 64-multiple tile without LayerNorm");
  APTAI_REQUIRE(g->out_pre == nullptr || !g->ln, "gemm: out_pre is not available with the fused LayerNorm");
  APTAI_REQUIRE(!g->ln || (g->out_bf16 != nullptr && g->out_f32 == nullptr && g->residual == nullptr &&
                           (reinterpret_cast<uintptr_t>(g->out_bf16) & 15) == 0),
                "gemm: the fused-LayerNorm tile writes one 16-byte-aligned 16-bit output (TMA stores) and takes no residual");
  const long long K = static_cast<long long>(g->taps) * g->kb_per_tap * BLOCK_K;

  // CTA-pair (cta_group::2) tiles halve the B traffic per SM; they need a wide N tile and enough 256-row tiles
  bool pair = false;
  if (bn >= 256) {
    const long long tiles2 = static_cast<long long>(g->segs) * ((g->rows_per_seg + 2 * BLOCK_M - 1) / (2 * BLOCK_M)) *
                             n_tiles;
    pair = g->cta_pair == 2 || (g->cta_pair == 0 && tiles2 >= 2LL * (num_sms() / 2));
  }
  CUtensorMap ta, tb;
  {
    const uint64_t r2 = (static_cast<uint64_t>(g->a_rows) + g->P - 1) / g->P;
    uint64_t dims[4] = {static_cast<uint64_t>(g->a_cols), static_cast<uint64_t>(g->P), r2,
                        static_cast<uint64_t>(g->segs)};
    uint64_t seg_stride = g->a_seg_stride > 0 ? static_cast<uint64_t>(g->a_seg_stride)
                                              : static_cast<uint64_t>(g->a_row_stride) * g->a_rows;
    uint64_t strides[3] = {static_cast<uint64_t>(g->a_row_stride) * 2,
                           static_cast<uint64_t>(g->a_row_stride) * 2 * g->P, seg_stride * 2};
    uint32_t box[4] = {BLOCK_K, 1, BLOCK_M, 1};
    if (int rc = encode_tmap_bf16(&ta, g->a, 4, dims, strides, box, 1)) return rc;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(g->N)};
    uint64_t strides[1] = {static_cast<uint64_t>(K) * 2};
    uint32_t box[2] = {BLOCK_K, static_cast<uint32_t>(bn / (pair ? 2 : 1))};
    if (int rc = encode_tmap_bf16(&tb, g->w, 2, dims, strides, box, 1)) return rc;
  }
  // single 16-bit output without residual / second output: staged in shared memory and written by TMA stores
  const bool tma16 = !g->ln && bn >= 128 && g->out_bf16 != nullptr && g->out_f32 == nullptr && g->out_pre == nullptr &&
                     g->residual == nullptr && g->act != 2 && (reinterpret_cast<uintptr_t>(g->out_bf16) & 15) == 0;
  CUtensorMap tc = ta;
  if (tma16 || g->ln) {
    uint64_t dims[3] = {static_cast<uint64_t>(g->N), static_cast<uint64_t>(g->rows_per_seg),
                        static_cast<uint64_t>(g->segs)};
    uint64_t strides[2] = {static_cast<uint64_t>(g->ldo) * 2,
                           static_cast<uint64_t>(g->segs > 1 ? g->out_seg_stride : g->rows_per_seg) * g->ldo * 2};
    uint32_t box[3] = {64, 32, 1};
    if (int rc = encode_tmap_bf16(&tc, g->out_bf16, 3, dims, strides, box, 1)) return rc;
  }
  // in-place fp32 residual update (out_f32 == residual, nothing else written): TMA reduce-add stores
  const bool red32 = !g->ln && bn >= 64 && bn % 64 == 0 && g->out_f32 != nullptr && g->residual == g->out_f32 &&
                     g->out_bf16 == nullptr && g->out_pre == nullptr && g->act == 0 && g->seg_valid_rows == nullptr &&
                     (reinterpret_cast<uintptr_t>(g->out_f32) & 15) == 0 && g->ldo % 4 == 0;
  if (red32) {
    uint64_t dims[3] = {static_cast<uint64_t>(g->N), static_cast<uint64_t>(g->rows_per_seg),
                        static_cast<uint64_t>(g->segs)};
    uint64_t strides[2] = {static_cast<uint64_t>(g->ldo) * 4,
                           static_cast<uint64_t>(g->segs > 1 ? g->out_seg_stride : g->rows_per_seg) * g->ldo * 4};
    uint32_t box[3] = {32, 32, 1};
    if (int rc = encode_tmap_f32(&tc, g->out_f32, 3, dims, strides, box, 1)) return rc;
  }
  GemmParams p;
  p.tma16 = (tma16 || g->ln) ? 1 : 0;
  p.reverse = traversal_reverse();
  p.red32 = red32 ? 1 : 0;
  p.l2_hint = red32 ? g->out_f32 : nullptr;
  p.num_kb = g->taps * g->kb_per_tap;
  p.kb_per_tap = g->kb_per_tap;
  p.P = g->P;
  p.a_col_per_nblk = g->a_col_per_nblk;
  p.rows_per_seg = g->rows_per_seg;
  const int tile_m = pair ? 2 * BLOCK_M : BLOCK_M;
  p.m_tiles_per_seg = (g->rows_per_seg + tile_m - 1) / tile_m;
  p.n_tiles = n_tiles;
  p.num_tiles = g->segs * p.m_tiles_per_seg * p.n_tiles;
  p.bias = g->bias;
  p.gamma = g->gamma;
  p.beta = g->beta;
  p.residual = red32 ? nullptr : g->residual;
  p.out_f32 = g->out_f32;
  p.out_bf16 = reinterpret_cast<__nv_bfloat16*>(g->out_bf16);
  p.ldo = g->ldo;
  p.out_seg_stride = g->out_seg_stride;
  p.seg_valid_rows = g->seg_valid_rows;
  p.mask_seg_rows = g->mask_seg_rows;
  p.act = g->act;
  p.ln_eps = g->ln_eps;
  p.fp16 = g->half_fmt ? 1 : 0;
  p.aux = reinterpret_cast<const __nv_bfloat16*>(g->aux);
  p.out_pre = reinterpret_cast<__nv_bfloat16*>(g->out_pre);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (g->ln) return pair ? launch_gemm_2cta<256, true>(ta, tb, tc, p, st) : launch_gemm<256, true>(ta, tb, tc, p, st);
  switch (bn) {
    case 256: return pair ? launch_gemm_2cta<256, false>(ta, tb, tc, p, st) : launch_gemm<256, false>(ta, tb, tc, p, st);
    case 128: return launch_gemm<128, false>(ta, tb, tc, p, st);
    case 64: return launch_gemm<64, false>(ta, tb, tc, p, st);
    case 48: return launch_gemm<48, false>(ta, tb, tc, p, st);
  }
  set_error("gemm: unreachable block_n %d", bn);
  return APTAI_ERR_ARG;
}
