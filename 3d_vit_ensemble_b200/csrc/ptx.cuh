// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA, TMEM
// alloc/ld/commit/fences).  Descriptor bit layouts follow the PTX ISA "tcgen05 matrix / instruction
// descriptor" tables (same fields CUTLASS's cute/arch/mma_sm100_desc.hpp encodes).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace vit3d {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Waits are bounded: a pipeline bug traps (-> CUDA error at the next API call) after ~2 s instead of
// hanging the GPU.  The clock is only read on the slow path.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  // try_wait itself suspends the thread for a hardware-defined interval; the poll loop is two instructions
  // and the deadline is only looked at every 1024 polls
  const long long t0 = clock64();
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 1024; ++i)
      if (mbar_try_wait(bar, parity)) return;
    if (clock64() - t0 > 4000000000ll) {
      printf("vit3d: mbarrier wait timed out (block %d thread %d parity %u)\n", blockIdx.x, threadIdx.x, parity);
      __trap();
    }
  }
}

// same, acquiring at cluster scope: the arrival came from another CTA of the cluster (mbar_arrive_cluster)
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 1024; ++i)
      if (mbar_try_wait_cluster(bar, parity)) return;
    if (clock64() - t0 > 4000000000ll) {
      printf("vit3d: cluster mbarrier wait timed out (block %d thread %d parity %u)\n", blockIdx.x, threadIdx.x, parity);
      __trap();
    }
  }
}

// One elected lane of a fully active warp.  The MMA-issuing warp elects ONCE and the elected thread runs the
// whole schedule (barrier waits, tcgen05.mma, commits) on its own: `if (elect_one()) { for (...) {...} }`.
// Electing inside the loop - all lanes walking it, `if (elect_one())` + `__syncwarp()` around every stage's
// MMAs - puts a warp-wide election / reconvergence between the last MMA of one stage and the first of the next
// and costs 60 cycles per MMA at four MMAs per stage (tools/mma_pipe_bench.cu); issuing from an
// `if (lane == 0)` region is worse still (the compiler then broadcasts every operand back with R2UR).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// ------------------------------------------------------------------ TMEM
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// 32 lanes x 32 columns of 32-bit: thread t of the warp gets lane (base_lane + t), columns c..c+31
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM, same lane / column mapping as tmem_ld_32x32b_x32 (used to park finished rows in the
// accumulator columns they came from instead of keeping them live in registers)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ UMMA descriptors
// Shared-memory matrix descriptor (64-bit):
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4   [46,48) version (1 on sm_100)
//   [49,52) base offset               [52]    LBO mode          [61,64) swizzle: 0 none, 2 128B, 4 64B, 6 32B
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout & 7) << 61;
  return d;
}
constexpr uint32_t UMMA_LAYOUT_SW128 = 2;

// Instruction descriptor (32-bit) for kind::f16 / kind::tf32:
//   [4,6) D format (1 = F32)  [7,10) A format  [10,13) B format (0 F16, 1 BF16, 2 TF32)
//   [15] A major (0 K, 1 MN)  [16] B major     [17,23) N >> 3     [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc(uint32_t fmt, uint32_t m, uint32_t n, uint32_t a_mn, uint32_t b_mn) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn << 15) | (b_mn << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// kind::f16 with different 16-bit formats for A and B (e.g. fp16 activations x bf16 weights)
__host__ __device__ constexpr uint32_t make_idesc_ab(uint32_t afmt, uint32_t bfmt, uint32_t m, uint32_t n) {
  return (1u << 4) | (afmt << 7) | (bfmt << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
constexpr uint32_t UMMA_FMT_F16 = 0;
constexpr uint32_t UMMA_FMT_BF16 = 1, UMMA_FMT_TF32 = 2;

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
template <bool TF32>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if (TF32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------ cluster multicast (cta_group::1 kernels)
// One bulk tensor load whose box lands at the same shared-memory offset in every CTA of `mask`, each of which
// gets the bytes counted on ITS mbarrier at the same offset: CTAs that consume the same operand (weights)
// share one L2 read.
__device__ __forceinline__ void tma_load_2d_mcast(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                                  uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_mcast(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                                  uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5}], "
      "[%2], %6;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(mask)
      : "memory");
}
// completion of this thread's MMAs -> one arrival on the mbarrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ------------------------------------------------------------------ CTA pairs (cta_group::2)
// Two CTAs of a cluster (ranks 0 / 1, one TPC) run ONE tcgen05.mma of M = 256: each CTA supplies its own 128 rows of A
// and HALF of B (N/2 rows) from the same shared-memory offsets, each CTA's TMEM receives its 128 accumulator rows.
// Only the leader (rank 0) issues MMAs and commits; both CTAs issue TMA loads, which signal the LEADER's mbarrier.
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_result) {        // one warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// shared::cluster address of `p` (a shared::cta pointer of THIS CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t map_to_rank(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// TMA load into THIS CTA's shared memory whose bytes are counted on the mbarrier at shared::cluster address `bar_cluster`
// (the leader's barrier)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
// D[tmem, both CTAs] (+)= A * B with M = 256 over the pair; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the leader's MMAs -> one arrival on the mbarrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma2_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
// one arrival on a mbarrier of another CTA of the cluster (address from map_to_rank)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}

// ------------------------------------------------------------------ clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

}  // namespace ptx
}  // namespace vit3d
