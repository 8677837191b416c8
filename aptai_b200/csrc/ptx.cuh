// Thin inline-PTX wrappers for the sm_100a features the kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / ld / commit / fences).
// Everything here is device-only and header-only.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

namespace aptai {

#ifndef APTAI_SPIN_LIMIT
#define APTAI_SPIN_LIMIT (1u << 27)   // bounded mbarrier waits: a protocol bug traps instead of hanging the box
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking test (try_wait may put the thread to sleep for a while): for event loops that poll several barriers
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > APTAI_SPIN_LIMIT) {
      printf("aptai: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

// wait with back-off for single-thread roles whose wake-up latency is not critical (TMA producers): the spin loop
// would otherwise steal issue slots from the compute warps that share its scheduler
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(ns);
    if (++spins > (APTAI_SPIN_LIMIT >> 4)) {
      printf("aptai: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_async_proxy() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// orders this thread's completed async-proxy (TMA) accesses, global memory included, with generic-proxy accesses
__device__ __forceinline__ void fence_proxy_async_all() {
  asm volatile("fence.proxy.async;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// TMA stores (shared -> global, bulk async-group completion): the box is clipped at the tensor bounds, so ragged
// last tiles need no per-row predicate
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// TMA reduction store: global[box] += shared[box] (fp32 add performed at the L2), same completion rules as a store
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the source shared memory of all committed store groups but the newest `N` has been read (it may be overwritten)
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// 2-CTA (cta_group::2) variants: the mbarrier operand is a shared::cluster address (the leader CTA's barrier)
__device__ __forceinline__ void tma_load_2d_cg2(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0,
                                                int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0,
                                                int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_cg2(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0,
                                                int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}

// ---------------------------------------------------------------- clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared::cta pointer of this CTA) as seen in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}
// Relaxed variant for "accumulator drained" signals: the only accesses that must be ordered before the arrival are
// this warp's tcgen05.ld (ordered by tcgen05.fence::before_thread_sync + wait::ld), not its global stores — the
// release form makes the arriving thread wait for every outstanding global store of the epilogue first.
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

// ---------------------------------------------------------------- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {   // whole warp, .sync.aligned
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* dst_smem, uint32_t ncols) {   // one warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// 32 lanes x 32 consecutive columns: thread i of the warp receives lane (base_lane + i), columns [c, c+32)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
// tcgen05.wait::ld that also names the 32 destination registers of the load it waits for: the compiler cannot schedule a
// use of them above the wait, and needs no copies to keep two loads in flight in alternating register arrays
__device__ __forceinline__ void tmem_ld_wait_regs(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor for a K-major bf16 tile whose rows are 128 B (64 elements) wide and were
// written by TMA with CU_TENSOR_MAP_SWIZZLE_128B: 8-row groups are 1024 B apart (SBO), LBO unused.
// bits [0,14) addr>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base offset | [61,64) layout=2
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;                 // LBO (ignored for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;         // SBO
  d |= static_cast<uint64_t>(1) << 46;                 // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                 // SWIZZLE_128B
  return d;
}

// Instruction descriptor, kind::f16: D=f32, A=B=bf16, both K-major, dense.
// bits [4,6) c_format=1 | [7,10) a_format=1 | [10,13) b_format=1 | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// same with IEEE fp16 operands (a_format = b_format = 0): used by the conv stack, whose activations are O(1)
// after LayerNorm/GELU and profit from fp16's three extra mantissa bits (TV parity margin, DESIGN.md section 5)
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; one thread issues for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// cta_group::2: issued by the leader CTA only; A rows / B columns are split across the CTA pair, M = 256.
__device__ __forceinline__ void umma_bf16_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from TMEM (M x K bf16, two elements per 32-bit column, lane = row): D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive columns, registers -> TMEM (thread i writes lane base_lane + i)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
      "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
      "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// commit of the pair's MMAs: one arrival on the barrier at the same offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}
// All previously issued MMAs complete -> one arrival on the mbarrier (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------- math helpers
// HF ACT2FN['gelu'] == exact erf GELU: x * Phi(x).  erfc via Abramowitz-Stegun 7.1.26 (|erf error| <= 1.5e-7)
// on the MUFU pipe (one rcp, one ex2) instead of erff(): ~14 instructions per element, max abs error 4.2e-7 over
// [-8, 8] against the fp64 definition (tests/test_kernels_gpu.py::test_gelu_accuracy) — far inside the bf16
// rounding of every consumer.  The GEMM epilogues (FFN1: 4096 GELUs per row) are issue-bound on erff().
__device__ __forceinline__ float gelu_erf(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * z * -1.4426950408889634f));
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(t, p, 1.421413741f);
  p = fmaf(t, p, -0.284496736f);
  p = fmaf(t, p, 0.254829592f);
  const float h = 0.5f * t * p * e;           // 0.5 * erfc(|x| / sqrt(2))
  return x * (x > 0.f ? 1.0f - h : h);
}
// d/dx [x * Phi(x)] = Phi(x) + x * phi(x); same erfc approximation as gelu_erf (backward of HF ACT2FN['gelu'])
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * z * -1.4426950408889634f));   // exp(-x^2/2)
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(t, p, 1.421413741f);
  p = fmaf(t, p, -0.284496736f);
  p = fmaf(t, p, 0.254829592f);
  const float h = 0.5f * t * p * e;           // 0.5 * erfc(|x| / sqrt(2)) = 1 - Phi(|x|)
  const float cdf = x > 0.f ? 1.0f - h : h;
  return fmaf(x * e, 0.3989422804014327f, cdf);
}
// Two GELUs at once on the packed fp32x2 FMA path of sm_100 (FFMA2 / FMUL2): the polynomial part costs half the
// FMA-pipe issue slots of the scalar version; the MUFU ops stay scalar.  Same formula, same accuracy.
__device__ __forceinline__ uint64_t f32x2_pack(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void f32x2_unpack(uint64_t v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t f32x2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f32x2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f32x2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ void gelu_erf2(float& x0, float& x1) {
  const uint64_t x = f32x2_pack(x0, x1);
  const uint64_t ax = f32x2_pack(fabsf(x0), fabsf(x1));
  float d0, d1, t0, t1, e0, e1, a0, a1;
  f32x2_unpack(f32x2_fma(ax, f32x2_pack(0.3275911f * 0.70710678118654752440f, 0.3275911f * 0.70710678118654752440f),
                         f32x2_pack(1.0f, 1.0f)), d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
  f32x2_unpack(f32x2_mul(f32x2_mul(x, x), f32x2_pack(-0.5f * 1.4426950408889634f, -0.5f * 1.4426950408889634f)), a0, a1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(a0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(a1));
  const uint64_t t = f32x2_pack(t0, t1);
  uint64_t p = f32x2_fma(t, f32x2_pack(0.5f * 1.061405429f, 0.5f * 1.061405429f),
                         f32x2_pack(0.5f * -1.453152027f, 0.5f * -1.453152027f));
  p = f32x2_fma(t, p, f32x2_pack(0.5f * 1.421413741f, 0.5f * 1.421413741f));
  p = f32x2_fma(t, p, f32x2_pack(0.5f * -0.284496736f, 0.5f * -0.284496736f));
  p = f32x2_fma(t, p, f32x2_pack(0.5f * 0.254829592f, 0.5f * 0.254829592f));
  const uint64_t h = f32x2_mul(f32x2_mul(t, p), f32x2_pack(e0, e1));    // 0.5 * erfc(|x| / sqrt(2))
  float r0, r1;
  f32x2_unpack(f32x2_mul(x, h), r0, r1);
  x0 = x0 > 0.f ? x0 - r0 : r0;
  x1 = x1 > 0.f ? x1 - r1 : r1;
}

// erf-GELU for consumers that round the result to 16 bits: x * Phi(x) with Phi(x) = 1 / (1 + 2^(x q(min(x^2, 64)))),
// q(t) = -log2(e) (c0 + c1 t + c2 t^2) the minimax fit of logit(Phi(x)) / x (max abs error 2.6e-5 against the fp64
// definition over all x: a hundred times below the bf16 / fp16 rounding of any value that matters; x^2 is clamped so
// that the fitted polynomial is never used beyond |x| = 8, where Phi is 0 or 1 to 1e-15).  Evaluated through ONE
// MUFU per element: 1 / (1 + e^-z) = 0.5 + 0.5 tanh(z / 2), so x Phi(x) = hx + hx tanh(-ln2/2 * x q), hx = x / 2.
// MUFU.TANH on sm_100 is far better than its 2^-11 specification on this argument range: measured on B200 against
// fp64 (profiles/scripts/mufu_accuracy.cu) the tanh form has max abs error 3.0e-5 / rms 1.23e-5, the ex2 + rcp form
// it replaces 2.5e-5 / 1.23e-5 (both are the fit's error).  5 packed + 4 scalar instructions per pair, 1 MUFU per
// element instead of 2 — the conv-0 kernel and the FFN1 / conv epilogues are MUFU- and issue-bound on it.
// fp32 outputs (and the accuracy mode) keep gelu_erf / gelu_erf2.
__device__ __forceinline__ void gelu_fast2(float& x0, float& x1) {
  const uint64_t x = f32x2_pack(x0, x1);
  float t0, t1, a0, a1, h0, h1;
  f32x2_unpack(f32x2_mul(x, x), t0, t1);
  const uint64_t t = f32x2_pack(fminf(t0, 64.f), fminf(t1, 64.f));
  constexpr float K = -0.34657359027997264f;                       // -ln(2) / 2
  uint64_t q = f32x2_fma(t, f32x2_pack(0.0010148165747523308f * K, 0.0010148165747523308f * K),
                         f32x2_pack(-0.10677912831306458f * K, -0.10677912831306458f * K));
  q = f32x2_fma(q, t, f32x2_pack(-2.3011176586151123f * K, -2.3011176586151123f * K));
  f32x2_unpack(f32x2_mul(q, x), a0, a1);
  asm("tanh.approx.f32 %0, %1;" : "=f"(h0) : "f"(a0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(h1) : "f"(a1));
  const uint64_t hx = f32x2_mul(x, f32x2_pack(0.5f, 0.5f));
  f32x2_unpack(f32x2_fma(hx, f32x2_pack(h0, h1), hx), x0, x1);
}

// gelu_fast2 for callers that can produce HALF the argument for free (a normalisation whose scale / shift vectors are
// pre-halved): h = x / 2 in, x Phi(x) = h + h tanh(h q'(h^2)) out, q' = gelu_fast2's polynomial re-scaled to t' = x^2 / 4.
// One packed multiply fewer than gelu_fast2 (4 packed + 2 scalar + 2 MUFU per pair).
__device__ __forceinline__ void gelu_fast2_half(float& h0, float& h1) {
  const uint64_t h = f32x2_pack(h0, h1);
  float t0, t1, a0, a1, th0, th1;
  f32x2_unpack(f32x2_mul(h, h), t0, t1);
  const uint64_t t = f32x2_pack(fminf(t0, 16.f), fminf(t1, 16.f));
  constexpr float K = -0.34657359027997264f;                       // -ln(2) / 2
  constexpr float C2 = 32.f * 0.0010148165747523308f * K, C1 = 8.f * -0.10677912831306458f * K,
                  C0 = 2.f * -2.3011176586151123f * K;
  uint64_t q = f32x2_fma(t, f32x2_pack(C2, C2), f32x2_pack(C1, C1));
  q = f32x2_fma(q, t, f32x2_pack(C0, C0));
  f32x2_unpack(f32x2_mul(q, h), a0, a1);
  asm("tanh.approx.f32 %0, %1;" : "=f"(th0) : "f"(a0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(th1) : "f"(a1));
  f32x2_unpack(f32x2_fma(h, f32x2_pack(th0, th1), h), h0, h1);
}

// Two GELU derivatives at once on the packed fp32x2 pipe: g0 *= gelu'(u0), g1 *= gelu'(u1)
__device__ __forceinline__ void gelu_erf_grad2_mul(float& g0, float& g1, float u0, float u1) {
  const uint64_t x = f32x2_pack(u0, u1);
  const uint64_t ax = f32x2_pack(fabsf(u0), fabsf(u1));
  float d0, d1, t0, t1, e0, e1, a0, a1;
  f32x2_unpack(f32x2_fma(ax, f32x2_pack(0.3275911f * 0.70710678118654752440f, 0.3275911f * 0.70710678118654752440f),
                         f32x2_pack(1.0f, 1.0f)), d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
  f32x2_unpack(f32x2_mul(f32x2_mul(x, x), f32x2_pack(-0.5f * 1.4426950408889634f, -0.5f * 1.4426950408889634f)), a0, a1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(a0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(a1));
  const uint64_t t = f32x2_pack(t0, t1);
  const uint64_t e = f32x2_pack(e0, e1);
  uint64_t p = f32x2_fma(t, f32x2_pack(0.5f * 1.061405429f, 0.5f * 1.061405429f),
                         f32x2_pack(0.5f * -1.453152027f, 0.5f * -1.453152027f));
  p = f32x2_fma(t, p, f32x2_pack(0.5f * 1.421413741f, 0.5f * 1.421413741f));
  p = f32x2_fma(t, p, f32x2_pack(0.5f * -0.284496736f, 0.5f * -0.284496736f));
  p = f32x2_fma(t, p, f32x2_pack(0.5f * 0.254829592f, 0.5f * 0.254829592f));
  float h0, h1;
  f32x2_unpack(f32x2_mul(f32x2_mul(t, p), e), h0, h1);      // 0.5 * erfc(|x| / sqrt(2)) = 1 - Phi(|x|)
  const uint64_t cdf = f32x2_pack(u0 > 0.f ? 1.0f - h0 : h0, u1 > 0.f ? 1.0f - h1 : h1);
  const uint64_t d = f32x2_fma(f32x2_mul(x, e), f32x2_pack(0.3989422804014327f, 0.3989422804014327f), cdf);
  f32x2_unpack(f32x2_mul(f32x2_pack(g0, g1), d), g0, g1);
}

// Attention-probability dropout (HF:461 `nn.functional.dropout(attn_weights, p)`): counter-based keep decision for
// element (query q, key k) of one (utterance, head).  32-bit "lowbias32" mix: cheap enough for the softmax inner loop.
__device__ __forceinline__ uint32_t attn_drop_mix(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ uint32_t attn_drop_seed_bh(uint64_t seed, uint32_t bh) {
  return attn_drop_mix(static_cast<uint32_t>(seed) ^ (bh * 0x9E3779B9U)) ^ static_cast<uint32_t>(seed >> 32);
}
__device__ __forceinline__ bool attn_drop_keep(uint32_t seed_bh, uint32_t q, uint32_t k, uint32_t T, uint32_t thresh24) {
  return (attn_drop_mix((q * T + k) ^ seed_bh) >> 8) >= thresh24;
}

__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
  __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

template <bool FP16>
__device__ __forceinline__ uint32_t pack_h16c(float a, float b) {      // format fixed at compile time
  return FP16 ? pack_f16(a, b) : pack_bf16(a, b);
}
__device__ __forceinline__ uint32_t pack_h16(float a, float b, int fp16) {
  return fp16 ? pack_f16(a, b) : pack_bf16(a, b);
}
// 32 floats -> four 16-byte units of 16-bit values under ONE (warp-uniform) format branch: the per-pair select of
// pack_h16 compiles to a predicated F2FP.F16 AND a predicated F2FP.BF16 per pair — two issue slots where one does work
__device__ __forceinline__ void pack32_h16(const float (&v)[32], uint4 (&o)[4], int fp16) {
  if (fp16) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
      o[u] = make_uint4(pack_f16(v[8 * u], v[8 * u + 1]), pack_f16(v[8 * u + 2], v[8 * u + 3]),
                        pack_f16(v[8 * u + 4], v[8 * u + 5]), pack_f16(v[8 * u + 6], v[8 * u + 7]));
  } else {
#pragma unroll
    for (int u = 0; u < 4; ++u)
      o[u] = make_uint4(pack_bf16(v[8 * u], v[8 * u + 1]), pack_bf16(v[8 * u + 2], v[8 * u + 3]),
                        pack_bf16(v[8 * u + 4], v[8 * u + 5]), pack_bf16(v[8 * u + 6], v[8 * u + 7]));
  }
}

// hi/lo bf16 pair of an fp32 value (accuracy-mode operands, csrc/accurate.cu): x = hi + lo to ~2^-17 relative
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

}  // namespace aptai
