// Weight-gradient GEMM on tcgen05 for sm_100a:  dW[n][k] += sum_m dY[m][n] * X[m][k]
//
// Backward of every nn.Linear of the encoder (HF:524-547, 566-573, 429-434: torch autograd's `grad_output.t() @ input`)
// and of the grouped positional conv (HF:329-368: conv1d weight gradient).  Both operands are activations stored
// row-major with the CONTRACTION index (the frame m) as the slow dimension, i.e. they are "MN-major" UMMA operands:
// TMA loads plain 64-row x 64-column boxes (SWIZZLE_128B) and the shared-memory descriptors carry the transposition
// (a_major = b_major = 1), so no transposed copy of any activation is ever written to HBM.
//
// Tile: 128 (dY columns) x 256 (X columns), accumulators in TMEM (2 x 256 columns: the epilogue of one work item
// overlaps the MMAs of the next), contraction in 64-frame blocks through a 4-stage TMA/mbarrier ring.
// The output has only (N/128)*(K/256) tiles (32..128 for the encoder's matrices), so the frame dimension is split
// across CTAs (split-K) and partial tiles are combined with fp32 vector reductions (red.global.add.v4.f32) into the
// gradient buffer — which is also what gradient accumulation wants (+=).
//
// Grouped positional conv: work item = (group g, block of 4 taps); A = dY columns of two adjacent groups (only the
// first 64 accumulator lanes are kept), B = the same 64 input channels of X at 4 consecutive frame shifts.
#include "common.h"
#include "ptx.cuh"

namespace aptai {

constexpr int TN_BM = 128;       // dY columns per tile  (UMMA M)
constexpr int TN_BN = 256;       // X columns per tile   (UMMA N)
constexpr int TN_BK = 64;        // frames per pipeline stage
constexpr int TN_STAGES = 4;
constexpr int TN_A_BYTES = TN_BK * TN_BM * 2;     // 16 KB: two 64x64 boxes
constexpr int TN_B_BYTES = TN_BK * TN_BN * 2;     // 32 KB: four 64x64 boxes
constexpr int TN_STAGE_BYTES = TN_A_BYTES + TN_B_BYTES;
constexpr int TN_SMEM = 1024 + TN_STAGES * TN_STAGE_BYTES + 256;
constexpr int TN_THREADS = 384;  // warps 0..7 epilogue, 8 TMA, 9 MMA, 10 TMEM alloc
constexpr int TN_W_TMA = 8, TN_W_MMA = 9, TN_W_ALLOC = 10;

struct TnParams {
  int n_tiles, k_tiles, splits, items;
  int segs, mblk_per_seg, total_kb;     // contraction blocks = segs * mblk_per_seg, divided among `splits`
  int a_col_step;                       // A column origin = nt * a_col_step
  int b_col_kt, b_col_nt, b_col_box;    // B box j column  = kt*b_col_kt + nt*b_col_nt + j*b_col_box
  int b_row_kt, b_row_box;              // B box j row     = m0 + kt*b_row_kt + j*b_row_box
  int out_rows_per_tile;                // accumulator lanes kept per tile (128, or 64 for the grouped conv)
  int out_rows, out_cols;               // bounds of the output matrix
  long long ldo;
  float* out;
  float scale;
  int conv_P, conv_cblks;               // strided conv (4-D B map: channel, row parity, row / P, utterance): P = stride,
                                        // conv_cblks = 256-channel blocks per tap; 0 = plain 3-D B map
};

// MN-major SWIZZLE_128B operand: 64-element (128 B) rows along MN, 8-row groups along K 1024 B apart (SBO),
// consecutive 64-element MN blocks 8192 B apart (LBO) — i.e. a stack of 64x64 TMA boxes.
__device__ __forceinline__ uint64_t umma_desc_sw128_mn_blocks(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(8192 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tn_wgrad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const TnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + TN_STAGES * TN_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + TN_STAGES;
  uint64_t* tfull_bar = empty_bar + TN_STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  // warp index through a shuffle: provably warp-uniform, so the single-issuer roles keep their loop state in
  // uniform registers (whole warp converged, elect.sync around the issue: see gemm_tc.cu)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;

  if (warp == TN_W_TMA && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == TN_W_MMA && lane == 0) {
    for (int i = 0; i < TN_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 8);
    }
    fence_mbar_init();
  }
  if (warp == TN_W_ALLOC) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles = p.n_tiles * p.k_tiles;

  if (warp == TN_W_TMA) {
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
        const int tile = item % tiles, sp = item / tiles;
        const int nt = tile / p.k_tiles, kt = tile - nt * p.k_tiles;
        const int kb0 = static_cast<int>((static_cast<long long>(p.total_kb) * sp) / p.splits);
        const int kb1 = static_cast<int>((static_cast<long long>(p.total_kb) * (sp + 1)) / p.splits);
        const int a_col = nt * p.a_col_step;
        const int b_col = kt * p.b_col_kt + nt * p.b_col_nt;
        const int b_row = kt * p.b_row_kt;
        for (int kb = kb0; kb < kb1; ++kb) {
          const int seg = kb / p.mblk_per_seg;
          const int m0 = (kb - seg * p.mblk_per_seg) * TN_BK;
          mbar_wait_backoff(&empty_bar[stage], phase ^ 1, 64);
          uint8_t* sa = smem + stage * TN_STAGE_BYTES;
          uint8_t* sb = sa + TN_A_BYTES;
          if (elect_one()) {
            mbar_expect_tx(&full_bar[stage], TN_STAGE_BYTES);
#pragma unroll
            for (int j = 0; j < TN_BM / 64; ++j) tma_load_3d(&tmA, &full_bar[stage], sa + j * 8192, a_col + j * 64, m0, seg);
            if (p.conv_P > 0) {
              // output frame m of the conv reads input row m * P + tap: parity = tap % P, row / P = m + tap / P
              const int tap = kt / p.conv_cblks, cb = (kt - tap * p.conv_cblks) * TN_BN;
#pragma unroll
              for (int j = 0; j < TN_BN / 64; ++j)
                tma_load_4d(&tmB, &full_bar[stage], sb + j * 8192, cb + j * 64, tap % p.conv_P, m0 + tap / p.conv_P, seg);
            } else {
#pragma unroll
              for (int j = 0; j < TN_BN / 64; ++j)
                tma_load_3d(&tmB, &full_bar[stage], sb + j * 8192, b_col + j * p.b_col_box,
                            m0 + b_row + j * p.b_row_box, seg);
            }
          }
          __syncwarp();
          if (++stage == TN_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == TN_W_MMA) {
    {
      // D = f32, A = B = bf16, both MN-major (bits 15, 16), N = 256, M = 128
      constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                                 (static_cast<uint32_t>(TN_BN >> 3) << 17) | (static_cast<uint32_t>(TN_BM >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
        const int sp = item / tiles;
        const int kb0 = static_cast<int>((static_cast<long long>(p.total_kb) * sp) / p.splits);
        const int kb1 = static_cast<int>((static_cast<long long>(p.total_kb) * (sp + 1)) / p.splits);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * TN_BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_u32(smem + stage * TN_STAGE_BYTES);
          const uint32_t b_base = a_base + TN_A_BYTES;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < TN_BK / 16; ++k)
              umma_bf16(d_tmem, umma_desc_sw128_mn_blocks(a_base + k * 2048),
                        umma_desc_sw128_mn_blocks(b_base + k * 2048), IDESC, (kb > kb0 || k > 0) ? 1u : 0u);
            umma_commit(&empty_bar[stage]);
            if (kb == kb1 - 1) umma_commit(&tfull_bar[acc]);
          }
          __syncwarp();
          if (++stage == TN_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (kb1 <= kb0 && elect_one()) umma_commit(&tfull_bar[acc]);     // empty split: nothing issued, release anyway
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp < 8) {
    const int q = warp & 3, half = warp >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
      const int tile = item % tiles, sp = item / tiles;
      const int nt = tile / p.k_tiles, kt = tile - nt * p.k_tiles;
      const int kb0 = static_cast<int>((static_cast<long long>(p.total_kb) * sp) / p.splits);
      const int kb1 = static_cast<int>((static_cast<long long>(p.total_kb) * (sp + 1)) / p.splits);
      const int lrow = q * 32 + lane;
      const int orow = nt * p.out_rows_per_tile + lrow;
      const bool row_ok = lrow < p.out_rows_per_tile && orow < p.out_rows;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (kb1 > kb0) {     // an empty split issued no MMA: its accumulator is undefined and contributes nothing
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * TN_BN;
        float* orp = p.out + static_cast<long long>(orow) * p.ldo + static_cast<long long>(kt) * TN_BN;
        const int col_lim = p.out_cols - kt * TN_BN;
        uint32_t nxt[32];
        tmem_ld32(t_row + half * 128, nxt);
#pragma unroll 1
        for (int c = half * 128; c < (half + 1) * 128; c += 32) {
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(nxt[i]) * p.scale;
          if (c + 32 < (half + 1) * 128) tmem_ld32(t_row + c + 32, nxt);
          if (row_ok) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              if (c + i < col_lim) red_add_v4(orp + c + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == TN_W_ALLOC) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// CTA-pair variant (cluster of 2, tcgen05.mma.cta_group::2): 256 dY columns x 256 X columns per tile.  Each CTA stages
// only ITS 128 dY columns (A half) and ITS 128 X columns (B half) per 64-frame block — 32 KB per stage instead of the
// 48 KB of the single-CTA tile for the same tensor work per SM — which is what the single-CTA kernel is bound by
// (L2 -> SM crossbar at ~12 TB/s, tensor pipe 53 %: profiles/r01_wgrad_tn_train_c4.md).  The leader CTA issues every
// MMA; each CTA owns the 128 accumulator lanes of its dY columns and reduces them into the gradient itself.
constexpr int TP_STAGES = 6;
constexpr int TP_HALF_BYTES = TN_BK * 128 * 2;               // 16 KB: two 64x64 boxes
constexpr int TP_STAGE_BYTES = 2 * TP_HALF_BYTES;            // A half + B half
constexpr int TP_SMEM = 1024 + TP_STAGES * TP_STAGE_BYTES + 256;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TN_THREADS, 1)
gemm_tn_wgrad_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                          const TnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + TP_STAGES * TP_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + TP_STAGES;
  uint64_t* tfull_bar = empty_bar + TP_STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const int item0 = blockIdx.x >> 1, item_step = gridDim.x >> 1;

  if (warp == TN_W_TMA && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == TN_W_MMA && lane == 0) {
    for (int i = 0; i < TP_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 16);        // 8 epilogue warps in each CTA of the pair
    }
    fence_mbar_init();
  }
  if (warp == TN_W_ALLOC) tmem_alloc_cg2(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles = p.n_tiles * p.k_tiles;

  if (warp == TN_W_TMA) {
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = item0; item < p.items; item += item_step) {
        const int tile = item % tiles, sp = item / tiles;
        const int nt = tile / p.k_tiles, kt = tile - nt * p.k_tiles;
        const int kb0 = static_cast<int>((static_cast<long long>(p.total_kb) * sp) / p.splits);
        const int kb1 = static_cast<int>((static_cast<long long>(p.total_kb) * (sp + 1)) / p.splits);
        const int a_col = nt * 256 + static_cast<int>(rank) * 128;
        const int b_col = kt * 256 + static_cast<int>(rank) * 128;
        for (int kb = kb0; kb < kb1; ++kb) {
          const int m0 = kb * TN_BK;
          mbar_wait_backoff(&empty_bar[stage], phase ^ 1, 64);
          uint8_t* sa = smem + stage * TP_STAGE_BYTES;
          uint8_t* sb = sa + TP_HALF_BYTES;
          if (elect_one()) {
            // both CTAs' bytes are counted on the LEADER's barrier; only the leader arms it
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * TP_STAGE_BYTES);
            const uint32_t fb = map_to_cta(&full_bar[stage], 0);
#pragma unroll
            for (int j = 0; j < 2; ++j) tma_load_3d_cg2(&tmA, fb, sa + j * 8192, a_col + j * 64, m0, 0);
#pragma unroll
            for (int j = 0; j < 2; ++j) tma_load_3d_cg2(&tmB, fb, sb + j * 8192, b_col + j * 64, m0, 0);
          }
          __syncwarp();
          if (++stage == TP_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == TN_W_MMA) {
    if (rank == 0) {
      // D = f32, A = B = bf16, both MN-major, M = 256 (128 per CTA), N = 256 (128 per CTA)
      constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                                 (static_cast<uint32_t>(256 >> 3) << 17) | (static_cast<uint32_t>(256 >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = item0; item < p.items; item += item_step) {
        const int sp = item / tiles;
        const int kb0 = static_cast<int>((static_cast<long long>(p.total_kb) * sp) / p.splits);
        const int kb1 = static_cast<int>((static_cast<long long>(p.total_kb) * (sp + 1)) / p.splits);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_u32(smem + stage * TP_STAGE_BYTES);
          const uint32_t b_base = a_base + TP_HALF_BYTES;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < TN_BK / 16; ++k)
              umma_bf16_cg2(d_tmem, umma_desc_sw128_mn_blocks(a_base + k * 2048),
                            umma_desc_sw128_mn_blocks(b_base + k * 2048), IDESC, (kb > kb0 || k > 0) ? 1u : 0u);
            umma_commit_cg2(&empty_bar[stage], 0x3);
            if (kb == kb1 - 1) umma_commit_cg2(&tfull_bar[acc], 0x3);
          }
          __syncwarp();
          if (++stage == TP_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (kb1 <= kb0 && elect_one()) umma_commit_cg2(&tfull_bar[acc], 0x3);   // empty split: release anyway
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp < 8) {
    const int q = warp & 3, half = warp >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t tempty_leader0 = map_to_cta(&tempty_bar[0], 0);
    for (int item = item0; item < p.items; item += item_step) {
      const int tile = item % tiles, sp = item / tiles;
      const int nt = tile / p.k_tiles, kt = tile - nt * p.k_tiles;
      const int kb0 = static_cast<int>((static_cast<long long>(p.total_kb) * sp) / p.splits);
      const int kb1 = static_cast<int>((static_cast<long long>(p.total_kb) * (sp + 1)) / p.splits);
      const int orow = nt * 256 + static_cast<int>(rank) * 128 + q * 32 + lane;
      const bool row_ok = orow < p.out_rows;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (kb1 > kb0) {
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * 256;
        float* orp = p.out + static_cast<long long>(orow) * p.ldo + static_cast<long long>(kt) * 256;
        const int col_lim = p.out_cols - kt * 256;
        uint32_t nxt[32];
        tmem_ld32(t_row + half * 128, nxt);
#pragma unroll 1
        for (int c = half * 128; c < (half + 1) * 128; c += 32) {
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(nxt[i]) * p.scale;
          if (c + 32 < (half + 1) * 128) tmem_ld32(t_row + c + 32, nxt);
          if (row_ok) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              if (c + i < col_lim) red_add_v4(orp + c + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader0 + acc * 8);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == TN_W_ALLOC) {
    tc_fence_after();
    tmem_dealloc_cg2(tmem_base, 512);
  }
}

// frame-dimension splits so that the work items fill `slots` concurrent workers in whole waves
static int choose_splits(int tiles, int slots, int total_kb) {
  int best = 1;
  double best_eff = 0.0;
  for (int s = 1; s <= 16; ++s) {
    if (total_kb / s < 8 && s > 1) break;
    const int items = tiles * s;
    const int waves = (items + slots - 1) / slots;
    const double eff = static_cast<double>(items) / (static_cast<double>(waves) * slots);
    if (eff > best_eff + 0.02) {
      best_eff = eff;
      best = s;
    }
  }
  return best;
}

static int launch_tn_pair(const CUtensorMap& ta, const CUtensorMap& tb, TnParams& p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tn_wgrad_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM);
    if (e != cudaSuccess) {
      set_error("gemm_wgrad(pair): cudaFuncSetAttribute(%d bytes): %s", TP_SMEM, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  const int tiles = p.n_tiles * p.k_tiles;
  const int clusters = num_sms() / 2;
  p.splits = choose_splits(tiles, clusters, p.total_kb);
  p.items = tiles * p.splits;
  const int grid = 2 * (p.items < clusters ? p.items : clusters);
  gemm_tn_wgrad_pair_kernel<<<grid, TN_THREADS, TP_SMEM, st>>>(ta, tb, p);
  return after_launch("gemm_tn_wgrad_pair");
}

static int launch_tn(const CUtensorMap& ta, const CUtensorMap& tb, TnParams& p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tn_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TN_SMEM);
    if (e != cudaSuccess) {
      set_error("gemm_wgrad: cudaFuncSetAttribute(%d bytes): %s", TN_SMEM, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    attr_set = true;
  }
  const int tiles = p.n_tiles * p.k_tiles;
  const int sms = num_sms();
  // split the frame dimension so that the work items fill the SMs in whole waves, at least 8 blocks per split
  int splits = 1;
  if (tiles < 2 * sms) {
    int best = 1;
    double best_eff = 0.0;
    for (int s = 1; s <= 16; ++s) {
      if (p.total_kb / s < 8 && s > 1) break;
      const int items = tiles * s;
      const int waves = (items + sms - 1) / sms;
      const double eff = static_cast<double>(items) / (static_cast<double>(waves) * sms);
      if (eff > best_eff + 0.02) {
        best_eff = eff;
        best = s;
      }
    }
    splits = best;
  }
  p.splits = splits;
  p.items = tiles * splits;
  const int grid = p.items < sms ? p.items : sms;
  gemm_tn_wgrad_kernel<<<grid, TN_THREADS, TN_SMEM, st>>>(ta, tb, p);
  return after_launch("gemm_tn_wgrad");
}

int wgrad_bf16_rows(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, int64_t M, int N, int K, float scale,
                    float* dw, int64_t dw_ld, int out_rows, void* stream) {
  APTAI_REQUIRE(dy && x && dw, "gemm_wgrad: null pointer");
  APTAI_REQUIRE(M >= 1 && N >= 1 && K >= 1 && out_rows >= 1 && out_rows <= N, "gemm_wgrad: bad shape");
  APTAI_REQUIRE(N % 8 == 0 && K % 8 == 0 && dy_ld % 8 == 0 && x_ld % 8 == 0 && dw_ld % 4 == 0,
                "gemm_wgrad: N, K and the row pitches must be multiples of 8 (dw_ld of 4)");
  APTAI_REQUIRE(((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dw)) & 15) == 0,
                "gemm_wgrad: buffers must be 16-byte aligned");
  CUtensorMap ta, tb;
  uint32_t box[3] = {64, 64, 1};
  {
    uint64_t dims[3] = {static_cast<uint64_t>(N), static_cast<uint64_t>(M), 1};
    uint64_t strides[2] = {static_cast<uint64_t>(dy_ld) * 2, static_cast<uint64_t>(dy_ld) * 2 * M};
    if (int rc = encode_tmap_bf16(&ta, dy, 3, dims, strides, box, 1)) return rc;
  }
  {
    uint64_t dims[3] = {static_cast<uint64_t>(K), static_cast<uint64_t>(M), 1};
    uint64_t strides[2] = {static_cast<uint64_t>(x_ld) * 2, static_cast<uint64_t>(x_ld) * 2 * M};
    if (int rc = encode_tmap_bf16(&tb, x, 3, dims, strides, box, 1)) return rc;
  }
  TnParams p;
  p.n_tiles = (N + TN_BM - 1) / TN_BM;
  p.k_tiles = (K + TN_BN - 1) / TN_BN;
  p.segs = 1;
  p.mblk_per_seg = static_cast<int>((M + TN_BK - 1) / TN_BK);
  p.total_kb = p.mblk_per_seg;
  p.a_col_step = TN_BM;
  p.b_col_kt = TN_BN; p.b_col_nt = 0; p.b_col_box = 64;
  p.b_row_kt = 0; p.b_row_box = 0;
  p.out_rows_per_tile = TN_BM;
  p.out_rows = out_rows; p.out_cols = K;
  p.ldo = dw_ld;
  p.out = dw;
  p.scale = scale;
  p.conv_P = 0; p.conv_cblks = 0;
  if (N >= 256 && K >= 256) {
    p.n_tiles = (N + 255) / 256;
    p.k_tiles = (K + 255) / 256;
    return launch_tn_pair(ta, tb, p, reinterpret_cast<cudaStream_t>(stream));
  }
  return launch_tn(ta, tb, p, reinterpret_cast<cudaStream_t>(stream));
}

}  // namespace aptai

using namespace aptai;

extern "C" int aptai_gemm_wgrad_bf16(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, int64_t M, int N,
                                     int K, float scale, float* dw, int64_t dw_ld, void* stream) {
  if (int rc = check_arch()) return rc;
  return wgrad_bf16_rows(dy, dy_ld, x, x_ld, M, N, K, scale, dw, dw_ld, N, stream);
}

extern "C" int aptai_posconv_wgrad_bf16(const void* dy, const void* x_pad, int B, int T, int H, int groups, int taps,
                                        float* dw_folded, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(dy && x_pad && dw_folded, "posconv_wgrad: null pointer");
  APTAI_REQUIRE(groups >= 1 && H % groups == 0 && H / groups <= 64 && (H / groups) % 8 == 0,
                "posconv_wgrad: group width must be a multiple of 8, at most 64");
  const int gw = H / groups;
  APTAI_REQUIRE(taps % 4 == 0, "posconv_wgrad: taps must be a multiple of 4");
  const int Tp = T + taps;
  CUtensorMap ta, tb;
  uint32_t box[3] = {64, 64, 1};
  {
    uint64_t dims[3] = {static_cast<uint64_t>(H), static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
    uint64_t strides[2] = {static_cast<uint64_t>(H) * 2, static_cast<uint64_t>(H) * 2 * T};
    if (int rc = encode_tmap_bf16(&ta, dy, 3, dims, strides, box, 1)) return rc;
  }
  {
    uint64_t dims[3] = {static_cast<uint64_t>(H), static_cast<uint64_t>(Tp), static_cast<uint64_t>(B)};
    uint64_t strides[2] = {static_cast<uint64_t>(H) * 2, static_cast<uint64_t>(H) * 2 * Tp};
    if (int rc = encode_tmap_bf16(&tb, x_pad, 3, dims, strides, box, 1)) return rc;
  }
  TnParams p;
  p.n_tiles = groups;
  p.k_tiles = taps / 4;
  p.segs = B;
  p.mblk_per_seg = (T + TN_BK - 1) / TN_BK;
  p.total_kb = p.segs * p.mblk_per_seg;
  // group width gw < 64 (base model: 48): the 64-wide boxes also cover channels of the next group; those accumulator
  // lanes / columns land in the padding of the folded layout (c >= gw) or are dropped (lanes >= gw)
  p.a_col_step = gw;
  p.b_col_kt = 0; p.b_col_nt = gw; p.b_col_box = 0;
  p.b_row_kt = 4; p.b_row_box = 1;
  p.out_rows_per_tile = gw;
  p.out_rows = H; p.out_cols = taps * 64;
  p.ldo = static_cast<long long>(taps) * 64;
  p.out = dw_folded;
  p.scale = 1.0f;
  p.conv_P = 0; p.conv_cblks = 0;
  return launch_tn(ta, tb, p, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int aptai_conv_wgrad_bf16(const void* dz, const void* x, int B, int T_out, int T_in, int C, int ktaps,
                                     int stride, float* dw_tapmajor, void* stream) {
  if (int rc = check_arch()) return rc;
  APTAI_REQUIRE(dz && x && dw_tapmajor, "conv_wgrad: null pointer");
  APTAI_REQUIRE(B >= 1 && T_out >= 1 && ktaps >= 1 && stride >= 1 && C % 256 == 0, "conv_wgrad: bad shape (C % 256)");
  APTAI_REQUIRE(static_cast<long long>(T_out - 1) * stride + ktaps <= T_in, "conv_wgrad: T_in too short");
  CUtensorMap ta, tb;
  {
    uint32_t box[3] = {64, 64, 1};
    uint64_t dims[3] = {static_cast<uint64_t>(C), static_cast<uint64_t>(T_out), static_cast<uint64_t>(B)};
    uint64_t strides[2] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(C) * 2 * T_out};
    if (int rc = encode_tmap_bf16(&ta, dz, 3, dims, strides, box, 1)) return rc;
  }
  {
    // the forward GEMM's A view of the conv input: (channel, row parity, row / P, utterance)
    uint32_t box[4] = {64, 1, 64, 1};
    const uint64_t r2 = (static_cast<uint64_t>(T_in) + stride - 1) / stride;
    uint64_t dims[4] = {static_cast<uint64_t>(C), static_cast<uint64_t>(stride), r2, static_cast<uint64_t>(B)};
    uint64_t strides[3] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(C) * 2 * stride,
                           static_cast<uint64_t>(C) * 2 * T_in};
    if (int rc = encode_tmap_bf16(&tb, x, 4, dims, strides, box, 1)) return rc;
  }
  TnParams p;
  p.n_tiles = (C + TN_BM - 1) / TN_BM;
  p.conv_cblks = C / TN_BN;
  p.k_tiles = ktaps * p.conv_cblks;
  p.segs = B;
  p.mblk_per_seg = (T_out + TN_BK - 1) / TN_BK;
  p.total_kb = p.segs * p.mblk_per_seg;
  p.a_col_step = TN_BM;
  p.b_col_kt = 0; p.b_col_nt = 0; p.b_col_box = 0; p.b_row_kt = 0; p.b_row_box = 0;
  p.out_rows_per_tile = TN_BM;
  p.out_rows = C; p.out_cols = ktaps * C;
  p.ldo = static_cast<long long>(ktaps) * C;
  p.out = dw_tapmajor;
  p.scale = 1.0f;
  p.conv_P = stride;
  return launch_tn(ta, tb, p, reinterpret_cast<cudaStream_t>(stream));
}
