// tcgen05 GEMM for sm_100a:  D[M,N] = A[M,K] * B[N,K]^T  (both operands K-major), fp32 accumulation
// in TMEM, operands staged by TMA (128B swizzle) through a multi-stage mbarrier ring.
//
//   * persistent, warp-specialised CTA of 192 threads (1 CTA / SM):
//       warp 0   TMA producer (one lane)        warp 1   TMEM allocator + tcgen05.mma issuer (one lane)
//       warps 2-9 epilogue: tcgen05.ld (32 lanes x 32 columns per warp) -> bias / GELU / residual /
//                 position-embedding add, transposed through swizzled smem -> 128-byte-line global stores
//   * tile 128 x BLOCK_N, BLOCK_K = 128 bytes of K (64 bf16 / 32 tf32); the accumulator is double
//     buffered in TMEM (2 x BLOCK_N columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
//   * kind::f16 (bf16 operands) or kind::tf32 (fp32 operands read directly, no conversion pass).
//   * optional split-K (work item = tile x K-slice, fp32 atomics) for deep-K / small-output products.
#include <stdlib.h>

#include <mutex>
#include <unordered_map>

#include "ptx.cuh"
#include "tc.cuh"
#include "tc_epilogue.cuh"

namespace vit3d {

using namespace ptx;

constexpr int TC_BLOCK_M = 128;
// warp 0 TMA, warp 1 MMA, then the epilogue warps (4 per TMEM lane quarter for BN >= 128, 2 for BN = 64)
constexpr int tc_epi_warps(int bn) { return bn >= 128 ? 16 : 8; }
constexpr int tc_threads(int bn) { return 64 + 32 * tc_epi_warps(bn); }

// Two operand schedules share the kernel:
//   streaming   : ring of STAGES x (A k-block 16 KB + B k-block BN*128 B); any K, optional split-K.
//   B-stationary: when the whole [BN x K] weight slab fits in 128 KB (K <= 256 bf16 at BN = 256) a CTA
//                 keeps ONE n-tile for its lifetime, loads that slab once and streams only A k-blocks
//                 (ring of 4 x 16 KB).  L2->SM operand traffic per tile drops from 192 KB to 64 KB, which
//                 is what bounds the K = 256 GEMMs (qkv, out-proj, fc1) at ~42 B/clk/SM of L2 bandwidth.
constexpr int TC_SLAB_BYTES = 128 * 1024;
constexpr int TC_STAT_STAGES = 4;
template <int BN> struct TcCfg {
  static constexpr int STAGES = BN == 256 ? 4 : (BN == 128 ? 6 : 8);
  static constexpr int A_BYTES = TC_BLOCK_M * 128;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int OPER_BYTES = STAGES * STAGE_BYTES;     // == TC_SLAB_BYTES + TC_STAT_STAGES * A_BYTES
  static constexpr int TMEM_COLS = 2 * BN;
  static constexpr int EPI_WARPS = tc_epi_warps(BN);
  static constexpr int THREADS = tc_threads(BN);
  static constexpr int EPI_WARP_BYTES = 2048;          // one 32-row x 64-byte transpose tile per epilogue warp
  static constexpr int EPI_BYTES = EPI_WARPS * EPI_WARP_BYTES;
  static constexpr int BIAS_BYTES = BN * 6;            // the n-tile's bias: fp32 copy + packed-half copy
  static constexpr int SMEM_BYTES = OPER_BYTES + EPI_BYTES + BIAS_BYTES + 256 /*barriers*/;
  static_assert(OPER_BYTES >= TC_SLAB_BYTES + TC_STAT_STAGES * A_BYTES, "operand region too small for the stationary schedule");
  static_assert(SMEM_BYTES <= 232448, "over the 227 KB shared-memory limit");
};

// work-item sequence of a CTA (identical in the producer, MMA and epilogue roles)
struct TileIter {
  int tiles_m, tiles_n, splits, total, w, tm, tn, split;
  bool stat;
  int cpn, g;
  __device__ TileIter(bool stationary, int tiles_m_, int tiles_n_, int splits_)
      : tiles_m(tiles_m_), tiles_n(tiles_n_), splits(splits_), stat(stationary) {
    total = tiles_m * tiles_n * splits;
    if (stat) {
      tn = blockIdx.x % tiles_n;
      g = blockIdx.x / tiles_n;
      cpn = gridDim.x / tiles_n;
      tm = g - cpn;
      split = 0;
    } else {
      w = (int)blockIdx.x - (int)gridDim.x;
    }
  }
  // the tile after the current one, without advancing (false: this was the last one)
  __device__ bool peek(int& tm2, int& tn2) const {
    if (stat) {
      tm2 = tm + cpn;
      tn2 = tn;
      return tm2 < tiles_m;
    }
    const int w2 = w + (int)gridDim.x;
    if (w2 >= total) return false;
    const int tile = w2 / splits;
    tn2 = tile % tiles_n;
    tm2 = tile / tiles_n;
    return true;
  }
  __device__ bool next() {
    if (stat) {
      tm += cpn;
      return tm < tiles_m;
    }
    w += gridDim.x;
    if (w >= total) return false;
    split = w % splits;
    const int tile = w / splits;
    tn = tile % tiles_n;
    tm = tile / tiles_n;
    return true;
  }
};

// EPI: EPI_GENERIC (run-time epilogue flags) or the compile-time mode of epilogue_bf16_lean.
// 18 warps = 5 on one scheduler: 16384 / (5 * 32) -> at most 96 registers per thread (ptxas derives this).
template <bool TF32, int BN, int EPI = EPI_GENERIC>
__global__ void __launch_bounds__(tc_threads(BN), 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmPre,
               const __grid_constant__ CUtensorMap tmX, TcEpilogue ep, int M, int N, int K, int tiles_m, int tiles_n,
               int splits, int stationary, int patch_blocks, int mn_major) {
  using Cfg = TcCfg<BN>;
  constexpr int BLOCK_K = TF32 ? 32 : 64;   // 128 bytes of K per stage row
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;                    // 128B-swizzled operand tiles need 1024-byte alignment
  if (smem_u32(smem) & 1023u) __trap();
  uint8_t* epi_stage = smem + Cfg::OPER_BYTES;
  uint8_t* bias_stage = epi_stage + Cfg::EPI_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias_stage + Cfg::BIAS_BYTES);
  constexpr int MAXST = 8;
  uint64_t* full_bar = bars;                 // [MAXST]
  uint64_t* empty_bar = bars + MAXST;        // [MAXST]
  uint64_t* tmem_full = bars + 2 * MAXST;    // [2]
  uint64_t* tmem_empty = bars + 2 * MAXST + 2;
  uint64_t* slab_full = bars + 2 * MAXST + 4;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * MAXST + 5);

  const bool stat = stationary != 0;
  const bool tall = (mn_major & 2) != 0;   // 256 x BN tile: the A stage doubles, both TMEM buffers form ONE accumulator pair
  const bool mnm = (mn_major & 1) != 0;    // both operands MN-major (weight gradients)
  const int STAGES = stat ? TC_STAT_STAGES : (tall ? Cfg::OPER_BYTES / (Cfg::STAGE_BYTES + Cfg::A_BYTES) : Cfg::STAGES);
  const int stage_bytes = stat ? Cfg::A_BYTES : (tall ? Cfg::STAGE_BYTES + Cfg::A_BYTES : Cfg::STAGE_BYTES);
  uint8_t* ring = stat ? smem + TC_SLAB_BYTES : smem;

  // warp index through a shuffle: warp-uniform for the compiler, so the role branches are uniform control flow
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  // patch mode passes the k-block count as K; MN-major stages hold 64 reduction rows
  const int nkb = patch_blocks > 0 ? K : ((mn_major & 1) ? (K + 63) / 64 : (K + BLOCK_K - 1) / BLOCK_K);
  const int kb_per = (nkb + splits - 1) / splits;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < MAXST; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], ep.cluster);     // the commit of every CTA of the cluster frees a multicast slot
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], Cfg::EPI_WARPS);     // one elected arrival per epilogue warp
    }
    mbar_init(slab_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const int cl = ep.cluster;
  const uint32_t crank = cl > 1 ? cluster_ctarank() : 0u;
  if (cl > 1) cluster_sync_all();   // every CTA's barriers exist before any multicast signal
  pdl_trigger();     // the next kernel may begin its own prologue on SMs this grid frees
  pdl_wait();        // everything above overlapped the previous kernel's tail; global memory from here on

  if (warp == 0) {
    // ===================================================== TMA producer
    if (lane == 0) {
      TileIter ti(stat, tiles_m, tiles_n, splits);
      if (stat && ti.g < tiles_m) {
        mbar_arrive_expect_tx(slab_full, nkb * Cfg::B_BYTES);
        for (int kb = 0; kb < nkb; ++kb) tma_load_2d(smem + kb * Cfg::B_BYTES, &tmB, slab_full, kb * BLOCK_K, ti.tn * BN);
      }
      int stage = 0;
      uint32_t phase = 0;
      const int a_bytes = tall ? 2 * Cfg::A_BYTES : Cfg::A_BYTES;
      while (ti.next()) {
        const int kb0 = ti.split * kb_per, kb1 = min(nkb, kb0 + kb_per);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = ring + stage * stage_bytes;
          mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
          if (patch_blocks > 0) {
            // patch-embedding mode (a1): the A tile is gathered straight from the (B,1,X,Y,Z) volume by a 5-D
            // box {32 floats of a patch row, ny patches, 1 row, nx patches, 128/P volumes}; k-block kb covers
            // patch row i = kb / patch_blocks, floats [32*(kb % patch_blocks), +32) of that row (zero-filled
            // past the row end in both operands).
            const int i = kb / patch_blocks, c0 = (kb % patch_blocks) * 32;
            if (tall) {       // 256 token rows: two boxes of 128 / P volumes each
              tma_load_5d(sa, &tmA, &full_bar[stage], c0, 0, i, 0, 2 * ti.tm * ep.vols_per_tile);
              tma_load_5d(sa + Cfg::A_BYTES, &tmA, &full_bar[stage], c0, 0, i, 0, (2 * ti.tm + 1) * ep.vols_per_tile);
            } else {
              tma_load_5d(sa, &tmA, &full_bar[stage], c0, 0, i, 0, ti.tm * ep.vols_per_tile);
            }
            if (cl > 1)       // this CTA's share of the filters, into the same slot of every CTA of the cluster
              tma_load_3d_mcast(sa + a_bytes + (int)crank * (Cfg::B_BYTES / cl), &tmB, &full_bar[stage], c0, i,
                                ti.tn * BN + (int)crank * (BN / cl), (uint16_t)((1u << cl) - 1u));
            else
              tma_load_3d(sa + a_bytes, &tmB, &full_bar[stage], c0, i, ti.tn * BN);
          } else if (mnm) {
            // both operands MN-major (weight gradients: dW = dY^T X reduces over the token rows): a stage
            // holds 64 reduction rows; each 64-column block is one {64 cols x 64 rows} box = 8 KB
            // (mn_major == 2: the tile spans 256 output rows = two accumulators sharing the B operand)
            const int a_blocks = tall ? 2 * TC_BLOCK_M / 64 : TC_BLOCK_M / 64;
            for (int j = 0; j < a_blocks; ++j)
              tma_load_2d(sa + j * 8192, &tmA, &full_bar[stage], ti.tm * (a_blocks * 64) + 64 * j, kb * 64);
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_2d(sa + a_blocks * 8192 + j * 8192, &tmB, &full_bar[stage], ti.tn * BN + 64 * j, kb * 64);
          } else {
            tma_load_2d(sa, &tmA, &full_bar[stage], kb * BLOCK_K, ti.tm * TC_BLOCK_M);
            if (!stat) tma_load_2d(sa + Cfg::A_BYTES, &tmB, &full_bar[stage], kb * BLOCK_K, ti.tn * BN);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer: ONE thread, elected once, walks the whole
    // schedule - waits, tcgen05.mma, commits (an election + __syncwarp per k-block costs ~60 cycles per MMA:
    // tools/mma_pipe_bench.cu, k_tc_mlp2.cu)
    if (elect_one()) {
      const uint32_t idesc = make_idesc(TF32 ? UMMA_FMT_TF32 : UMMA_FMT_BF16, TC_BLOCK_M, BN, mnm ? 1 : 0, mnm ? 1 : 0);
      // K-major SW128: 8-row groups 1024 B apart, K advances 32 B inside the 128 B swizzle row.
      // MN-major SW128: 64-element MN blocks 8192 B apart (LBO), 8-row K groups 1024 B apart (SBO),
      //                 one MMA (K = 16) consumes two K groups -> advance 2048 B.
      const uint32_t lbo = mnm ? 8192u : 16u;
      const uint64_t kstep = mnm ? (2048u >> 4) : (32u >> 4);            // descriptor address units of 16 B
      const uint64_t ring_desc = make_smem_desc(smem_u32(ring), lbo, 1024, UMMA_LAYOUT_SW128);
      const uint64_t slab_desc = make_smem_desc(smem_u32(smem), lbo, 1024, UMMA_LAYOUT_SW128);
      TileIter ti(stat, tiles_m, tiles_n, splits);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      bool slab_ready = !stat;
      for (; ti.next(); ++it) {
        const int kb0 = ti.split * kb_per, kb1 = min(nkb, kb0 + kb_per);
        const int buf = tall ? 0 : (it & 1);
        mbar_wait(&tmem_empty[buf], (tall ? (it & 1) : ((it >> 1) & 1)) ^ 1);
        if (!slab_ready) { mbar_wait(slab_full, 0); slab_ready = true; }
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * BN;
        // no tcgen05 fence after an operand k-block has landed: the mbarrier's complete_tx orders the TMA writes
        // before the MMAs' reads
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          const uint64_t ad = ring_desc + (uint64_t)((stage * stage_bytes) >> 4);
          const uint64_t bd = stat ? slab_desc + (uint64_t)((kb * Cfg::B_BYTES) >> 4)
                                   : ad + (uint64_t)(((tall ? 2 : 1) * Cfg::A_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)     // 4 x 32 bytes of K per stage
            umma<TF32>(d_tmem, ad + k * kstep, bd + k * kstep, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          if (tall) {
#pragma unroll
            for (int k = 0; k < 4; ++k)   // rows 128..255 of the tile: second accumulator, same B k-block
              umma<TF32>(d_tmem + BN, ad + (uint64_t)(Cfg::A_BYTES >> 4) + k * kstep, bd + k * kstep, idesc,
                         (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if (cl > 1) umma_commit_mcast(&empty_bar[stage], (uint16_t)((1u << cl) - 1u));
          else umma_commit(&empty_bar[stage]);   // frees the smem slot when these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[buf]);       // accumulator ready for the epilogue
      }
    }
    __syncwarp();
  } else {
    // ===================================================== epilogue warps
    const int q = warp & 3;                 // TMEM lane quarter this warp may read
    const int part = (warp - 2) >> 2;       // which slice of the tile's columns
    constexpr int CW = BN / (Cfg::EPI_WARPS / 4);
    const uint32_t stage = smem_u32(epi_stage + (warp - 2) * Cfg::EPI_WARP_BYTES);
    TileIter ti(stat, tiles_m, tiles_n, splits);
    int it = 0;
    int cur_tn = -1;
    // training fc1: a thread's keep bits (CW columns of its row) are fetched one tile AHEAD - the epilogue is the
    // bottleneck of that GEMM (accumulators are ready long before), so a load issued at the top of the tile would
    // expose its whole global-memory latency
    constexpr bool KEEP = EPI >= 0 && (EPI & 8) != 0;
    uint32_t keep_nx[CW / 32];
    auto load_keep = [&](int tm2, int tn2) {
#pragma unroll
      for (int j = 0; j < CW / 32; ++j) keep_nx[j] = ep.drop_bits == nullptr ? 0xffffffffu : 0u;
      const int m = tm2 * TC_BLOCK_M + q * 32 + lane;
      if (ep.drop_bits != nullptr && m < M) {
        const uint32_t* drop_row = ep.drop_bits + (((long long)m * N + tn2 * BN + part * CW) >> 5);
#pragma unroll
        for (int j = 0; j < CW / 32; ++j) keep_nx[j] = __ldg(drop_row + j);
      }
    };
    for (; ti.next(); ++it) {
      uint32_t keep[CW / 32];
      if constexpr (KEEP) {
        if (it == 0) load_keep(ti.tm, ti.tn);
#pragma unroll
        for (int j = 0; j < CW / 32; ++j) keep[j] = keep_nx[j];
        int tm2, tn2;
        if (ti.peek(tm2, tn2)) load_keep(tm2, tn2);
      }
      const int buf = tall ? 0 : (it & 1);
      if constexpr (EPI >= 0 && (EPI & 1) != 0) {
        if (ti.tn != cur_tn) {
          // stage this n-tile's bias (fp32 + packed half) for all epilogue warps; once per CTA under the
          // stationary schedule.  First barrier: everyone is done reading the previous n-tile's copy.
          constexpr int ETH = Cfg::EPI_WARPS * 32;
          asm volatile("bar.sync 1, %0;" ::"n"(ETH) : "memory");
          const int t = (int)threadIdx.x - 64;
          if (t < BN / 4) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + ti.tn * BN + 4 * t));
            *reinterpret_cast<float4*>(bias_stage + 16 * t) = b;
            const __half2 h0 = __floats2half2_rn(b.x, b.y), h1 = __floats2half2_rn(b.z, b.w);
            *reinterpret_cast<uint2*>(bias_stage + BN * 4 + 8 * t) =
                make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
          }
          asm volatile("bar.sync 1, %0;" ::"n"(ETH) : "memory");
          cur_tn = ti.tn;
        }
      }
      if constexpr (EPI >= 0) {
        const int m_base = ti.tm * TC_BLOCK_M + q * 32, n_base = ti.tn * BN + part * CW;
        mbar_wait(&tmem_full[buf], (it >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN + part * CW;
        epilogue_bf16_lean<CW, EPI>(&tmC, &tmPre, taddr, stage, smem_u32(bias_stage) + part * CW * 4,
                                    smem_u32(bias_stage) + BN * 4 + part * CW * 2, lane, m_base, n_base, keep,
                                    ep.drop_scale);
      } else {
        // generic epilogues: ONE call site per kernel variant (every inlined copy of epilogue_rows costs registers at
        // the 96-register cap: two extra copies spilled ~440 bytes and slowed the patch embedding from 117 to 160 us).
        // A tall tile (256 rows) is two passes over the accumulator pair: h = rows [128 h, 128 h + 128).
        mbar_wait(&tmem_full[buf], tall ? (it & 1) : ((it >> 1) & 1));
        tc_fence_after();
        const int n_base = ti.tn * BN + part * CW;
#pragma unroll 1
        for (int h = 0; h < (tall ? 2 : 1); ++h) {
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (tall ? h : buf) * BN + part * CW;
          const int m_base = tall ? ti.tm * (2 * TC_BLOCK_M) + h * TC_BLOCK_M + q * 32 : ti.tm * TC_BLOCK_M + q * 32;
          if constexpr (EPI == EPI_WGRAD) {
            if (ep.atomic == 2) {
              // weight gradients: boxes added into the output by the TMA unit; one tensor map per output segment
              const int seg = ep.seg_rows > 0 ? m_base / ep.seg_rows : 0;
              const CUtensorMap* tr = seg == 0 ? &tmC : (seg == 1 ? &tmPre : &tmX);
              epilogue_reduce_f32<CW>(tr, taddr, stage, lane, m_base - seg * ep.seg_rows, n_base, N);
            } else {
              // fp32 atomics into the (segmented) output, or this work item's dense partial tile
              const bool part_ws = ep.partial_ws != nullptr;
              epilogue_rows<CW, !TF32, false>(ep, &tmC, &tmPre, taddr, stage, lane, part_ws ? q * 32 : m_base,
                                              part_ws ? part * CW : n_base, part_ws ? TC_BLOCK_M : M, part_ws ? BN : N,
                                              part_ws ? (void*)(ep.partial_ws + (size_t)ti.w * (TC_BLOCK_M * BN)) : ep.out,
                                              part_ws ? 0 : ep.atomic, part_ws ? 0 : ep.seg_rows);
            }
          } else {
            epilogue_rows<CW, !TF32, EPI == EPI_GENERIC_DACT>(ep, &tmC, &tmPre, taddr, stage, lane, m_base, n_base, M, N, ep.out,
                                                              ep.atomic, 0);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
    }
    if (lane == 0) bulk_store_wait_all();   // bulk tensor stores must complete before the CTA exits
  }
  tc_fence_before();
  __syncthreads();
  if (cl > 1) cluster_sync_all();   // nobody leaves while a partner may still multicast into this CTA
  if (warp == 1) tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// ----------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 2-D row-major [rows, cols] tensor map; box = [box_rows, box_cols]; swizzle 128B (operands, box_cols*elem
// = 128 B) or 64B (bf16 output tiles, 64 B); out-of-bounds reads give 0, out-of-bounds writes are dropped.
int make_tmap_2d(CUtensorMap* out, const void* ptr, int elem_bytes, long long rows, long long cols, long long ld_elems,
                 int box_rows, int box_cols, int swizzle_bytes) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return VIT3D_ERR_CUDA; }
  struct Key { const void* p; long long r, c, ld; int e, br, bc, sw; };
  struct Hash { size_t operator()(const Key& k) const {
    size_t h = (size_t)k.p; h = h * 1000003u ^ (size_t)k.r; h = h * 1000003u ^ (size_t)k.c;
    h = h * 1000003u ^ (size_t)k.ld; h = h * 1000003u ^ (size_t)(((k.e * 512 + k.br) * 512 + k.bc) * 4 + k.sw / 64); return h; } };
  struct Eq { bool operator()(const Key& a, const Key& b) const {
    return a.p == b.p && a.r == b.r && a.c == b.c && a.ld == b.ld && a.e == b.e && a.br == b.br && a.bc == b.bc && a.sw == b.sw; } };
  static thread_local std::unordered_map<Key, CUtensorMap, Hash, Eq> cache;
  const Key key{ptr, rows, cols, ld_elems, elem_bytes, box_rows, box_cols, swizzle_bytes};
  auto itc = cache.find(key);
  if (itc != cache.end()) { *out = itc->second; return VIT3D_OK; }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld_elems * elem_bytes) & 15)) {
    set_error("TMA operand must be 16-byte aligned (ptr %p, row stride %lld bytes)", ptr, ld_elems * elem_bytes);
    return VIT3D_ERR_INVALID;
  }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)(ld_elems * elem_bytes)};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = enc(out, dt, 2, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return VIT3D_ERR_CUDA; }
  if (cache.size() > 2048) cache.clear();
  cache.emplace(key, *out);
  return VIT3D_OK;
}

template <bool TF32, int BN, int EPI = EPI_GENERIC>
static int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tp,
                     const TcEpilogue& ep, int M, int N, int K, int splits, bool stationary, cudaStream_t st,
                     int patch_blocks = 0, int mn_major = 0, const CUtensorMap* tx = nullptr) {
  using Cfg = TcCfg<BN>;
  auto kern = tc_gemm_kernel<TF32, BN, EPI>;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V3_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    configured_dev = dev;
  }
  const int tiles_m = ceil_div(M, (mn_major & 2) ? 2 * TC_BLOCK_M : TC_BLOCK_M), tiles_n = ceil_div(N, BN);
  const int total = tiles_m * tiles_n * splits;
  const int sms = sm_count();
  int grid = total < sms ? total : sms;
  if (stationary) {
    int cpn = sms / tiles_n;            // CTAs per n-tile
    if (cpn > tiles_m) cpn = tiles_m;
    grid = cpn * tiles_n;
  }
  if (ep.grid_limit > 0 && grid > ep.grid_limit) grid = ep.grid_limit;
  if (ep.cluster > 1) {
    // the cluster's CTAs walk the tile list in lock step (shared ring slots): equal tile counts within every cluster
    if (grid % ep.cluster || (total > grid && (total % grid) % ep.cluster) || stationary || splits != 1) {
      set_error("tc_gemm: cluster multicast needs grid and tail tile counts that are multiples of the cluster size");
      return VIT3D_ERR_INVALID;
    }
    V3_CUDA(launch_pdl_cluster(kern, dim3(grid), dim3(Cfg::THREADS), (size_t)Cfg::SMEM_BYTES, st, ep.cluster, ta, tb, tc, tp,
                               tx ? *tx : tp, ep, M, N, K, tiles_m, tiles_n, splits, stationary ? 1 : 0, patch_blocks, mn_major));
    V3_LAUNCH_CHECK();
    return VIT3D_OK;
  }
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(Cfg::THREADS), (size_t)Cfg::SMEM_BYTES, st, ta, tb, tc, tp, tx ? *tx : tp, ep, M, N, K, tiles_m,
                     tiles_n, splits, stationary ? 1 : 0, patch_blocks, mn_major));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// D[M,N] = A[M,K] B[N,K]^T with both operands dense row-major K-major; elem = 2 (bf16) or 4 (tf32)
int tc_gemm(bool tf32, const void* A, const void* B, int M, int N, int K, const TcEpilogue& ep, int splits,
            cudaStream_t st) {
  const int eb = tf32 ? 4 : 2;
  const int sms = sm_count();
  const int tm = ceil_div(M, TC_BLOCK_M);
  const int nkb = ceil_div(K, 128 / eb);
  // widest N tile that still gives every SM work
  int bn = 256;
  if (N <= 64 || (long long)tm * ceil_div(N, 256) * splits < sms) bn = 128;
  if (N <= 64 || (bn == 128 && (long long)tm * ceil_div(N, 128) * splits < sms)) bn = 64;
  // stationary-B schedule when the [bn x K] weight slab fits (shrink the tile once if that makes it fit)
  auto fits = [&](int b) { return splits == 1 && (long long)nkb * b * 128 <= TC_SLAB_BYTES && ceil_div(N, b) <= sms; };
  bool stationary = fits(bn);
  if (!stationary && bn == 256 && fits(128)) { bn = 128; stationary = true; }
  CUtensorMap ta, tb, tc, tp;
  int rc = make_tmap_2d(&ta, A, eb, M, K, K, TC_BLOCK_M, 128 / eb, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&tb, B, eb, N, K, K, bn, 128 / eb, 128);
  if (rc != VIT3D_OK) return rc;
  tc = ta;
  tp = ta;
  if (!ep.out_f32) {   // bf16 outputs leave through bulk tensor stores
    if (ep.row_group > 0 || ep.atomic) { set_error("tc_gemm: bf16 output with row remap / atomics is not supported"); return VIT3D_ERR_INVALID; }
    rc = make_tmap_2d(&tc, ep.out, 2, M, N, N, 32, 32, 64);
    if (rc != VIT3D_OK) return rc;
    if (ep.pre) {
      rc = make_tmap_2d(&tp, ep.pre, 2, M, N, N, 32, 32, 64);
      if (rc != VIT3D_OK) return rc;
    }
  }
  if (tf32) {
    if (bn == 256) return launch_tc<true, 256>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
    if (bn == 128) return launch_tc<true, 128>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
    return launch_tc<true, 64>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
  }
  // compile-time specialised epilogue for the hot bf16-output products (full column tiles)
  if (!ep.out_f32 && bn >= 128 && N % bn == 0 &&
      (!ep.pre || ep.act == VIT3D_ACT_GELU) && (ep.act == VIT3D_ACT_NONE || ep.bias) &&
      (!ep.drop_bits || ep.store_dact) && (!ep.store_dact || (ep.pre && ep.bias && ep.act == VIT3D_ACT_GELU))) {
    const int mode = (ep.bias ? 1 : 0) | (ep.act == VIT3D_ACT_GELU ? 2 : 0) | (ep.pre ? 4 : 0) | (ep.store_dact ? 8 : 0);
#define V3_LEAN(BN_, MODE_) \
  if (bn == BN_ && mode == MODE_) return launch_tc<false, BN_, MODE_>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
    V3_LEAN(256, 0) V3_LEAN(256, 1) V3_LEAN(256, 3) V3_LEAN(256, 7) V3_LEAN(256, 15)
    V3_LEAN(128, 0) V3_LEAN(128, 1) V3_LEAN(128, 3) V3_LEAN(128, 7) V3_LEAN(128, 15)
#undef V3_LEAN
  }
  if (ep.store_dact) {
    if (bn == 256) return launch_tc<false, 256, EPI_GENERIC_DACT>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
    if (bn == 128) return launch_tc<false, 128, EPI_GENERIC_DACT>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
    return launch_tc<false, 64, EPI_GENERIC_DACT>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
  }
  if (bn == 256) return launch_tc<false, 256>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
  if (bn == 128) return launch_tc<false, 128>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
  return launch_tc<false, 64>(ta, tb, tc, tp, ep, M, N, K, splits, stationary, st);
}

// D[Mo,No] += A^T B with A = [Kred, Mo] and B = [Kred, No] row-major bf16 (both operands MN-major):
// the weight-gradient product dW[N,K] += dY[M,N]^T X[M,K].  Split over the reduction (token rows) so that
// every SM has work; partial tiles are accumulated with fp32 atomics into `out`.
int tc_gemm_wgrad(const void* A, const void* B, float* out, int Mo, int No, int Kred, cudaStream_t st) {
  return tc_gemm_wgrad_seg(A, B, out, nullptr, nullptr, 0, Mo, No, Kred, st);
}

// same, output rows [i*seg_rows, (i+1)*seg_rows) accumulated into out0 / out1 / out2 (seg_rows % 128 == 0; 0 = one buffer)
// the tile width / split count tc_gemm_wgrad_seg uses for a product (also sizes the partial-tile workspace)
void tc_wgrad_plan(int Mo, int No, int Kred, int* bn_out, int* splits_out, int* tiles_out) {
  const int sms = sm_count();
  int bn = 256;
  if (No % 256) bn = 128;
  if (No % 128) bn = 64;
  const int tiles = ceil_div(Mo, TC_BLOCK_M) * ceil_div(No, bn);
  const int nkb = ceil_div(Kred, 64);
  int splits = sms / tiles;
  if (splits > nkb) splits = nkb;
  if (splits < 1) splits = 1;
  for (;;) {
    const int kp = ceil_div(nkb, splits), s2 = ceil_div(nkb, kp);
    if (s2 == splits) break;
    splits = s2;
  }
  if (bn_out) *bn_out = bn;
  if (splits_out) *splits_out = splits;
  if (tiles_out) *tiles_out = tiles;
}

// partial-tile variant: every work item stores its tile to `ws` (tiles * splits * 128 * bn floats), no atomics
int tc_gemm_wgrad_partial(const void* A, const void* B, float* ws, int Mo, int No, int Kred, cudaStream_t st) {
  int bn, splits, tiles;
  tc_wgrad_plan(Mo, No, Kred, &bn, &splits, &tiles);
  CUtensorMap ta, tb;
  int rc = make_tmap_2d(&ta, A, 2, Kred, Mo, Mo, 64, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&tb, B, 2, Kred, No, No, 64, 64, 128);
  if (rc != VIT3D_OK) return rc;
  TcEpilogue ep;
  ep.out = ws; ep.out_f32 = 1; ep.partial_ws = ws;
  if (bn == 256) return launch_tc<false, 256, EPI_WGRAD>(ta, tb, ta, ta, ep, Mo, No, Kred, splits, false, st, 0, 1);
  if (bn == 128) return launch_tc<false, 128, EPI_WGRAD>(ta, tb, ta, ta, ep, Mo, No, Kred, splits, false, st, 0, 1);
  return launch_tc<false, 64, EPI_WGRAD>(ta, tb, ta, ta, ep, Mo, No, Kred, splits, false, st, 0, 1);
}

int tc_gemm_wgrad_seg(const void* A, const void* B, float* out, float* out1, float* out2, int seg_rows, int Mo, int No,
                      int Kred, cudaStream_t st) {
  const int sms = sm_count();
  int bn = 256;
  if (No % 256) bn = 128;
  if (No % 128) bn = 64;
  int tiles = ceil_div(Mo, TC_BLOCK_M) * ceil_div(No, bn);
  const int nkb = ceil_div(Kred, 64);
  // Tall tiles (256 x 256, two accumulators sharing the B k-block): 64 KB of operands per 1024 MMA cycles instead
  // of 48 KB per 512 - the streamed products are bound by operand delivery (~40 B/clk/SM), so the large products
  // (fc1 / fc2: 12 tall tiles) take them; small outputs keep 128-row tiles (less reduce volume per work item).
  const bool red = tuning(VIT3D_TUNE_WGRAD_RED) != 0 && No % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                   (!out1 || (reinterpret_cast<uintptr_t>(out1) & 15) == 0) && (!out2 || (reinterpret_cast<uintptr_t>(out2) & 15) == 0);
  const int tall_tiles = (Mo / 256) * ceil_div(No, 256);
  const bool tall = red && tuning(VIT3D_TUNE_WGRAD_RED) == 2 && bn == 256 && Mo % 256 == 0 && (seg_rows == 0 || seg_rows % 256 == 0) &&
                    tall_tiles >= 8 && tall_tiles <= sms && nkb / (sms / tall_tiles) >= 8;
  if (tall) tiles = tall_tiles;
  // Every work item ends in a tile of fp32 adds into the SAME few output tiles, so the reduce volume - work items x
  // tile size - is what the small products (out-projection: 2 output tiles) pay for.  One work item per SM, not two.
  int splits = sms / tiles;              // floor: 24 tiles x 6 slices = 144 items are one wave, 24 x 7 = 168 would be two
  if (splits > nkb) splits = nkb;
  if (splits < 1) splits = 1;
  // no K-slice may be empty (an empty slice would publish an unwritten accumulator): iterate to the
  // fixpoint splits == ceil(nkb / ceil(nkb / splits)), which is what the kernel derives from `splits`
  for (;;) {
    const int kp = ceil_div(nkb, splits), s2 = ceil_div(nkb, kp);
    if (s2 == splits) break;
    splits = s2;
  }
  CUtensorMap ta, tb;
  int rc = make_tmap_2d(&ta, A, 2, Kred, Mo, Mo, 64, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&tb, B, 2, Kred, No, No, 64, 64, 128);
  if (rc != VIT3D_OK) return rc;
  TcEpilogue ep;
  ep.out = out; ep.out_f32 = 1; ep.atomic = 1;
  if (seg_rows > 0) {
    if (seg_rows % TC_BLOCK_M || !out1 || Mo > 3 * seg_rows || (Mo > 2 * seg_rows && !out2)) {
      set_error("wgrad: bad output segmentation (seg_rows %d, rows %d)", seg_rows, Mo);
      return VIT3D_ERR_INVALID;
    }
    ep.seg_rows = seg_rows; ep.out_seg[0] = out1; ep.out_seg[1] = out2;
  }
  CUtensorMap tc = ta, tp = ta, tx = ta;
  if (red) {
    // partial tiles leave as [32 x 16] fp32 boxes the TMA unit adds into the output (one map per segment)
    const int rows0 = seg_rows > 0 ? (Mo < seg_rows ? Mo : seg_rows) : Mo;
    rc = make_tmap_2d(&tc, out, 4, rows0, No, No, 32, 16, 64);
    if (rc != VIT3D_OK) return rc;
    if (seg_rows > 0 && Mo > seg_rows) {
      rc = make_tmap_2d(&tp, out1, 4, Mo - seg_rows < seg_rows ? Mo - seg_rows : seg_rows, No, No, 32, 16, 64);
      if (rc != VIT3D_OK) return rc;
    }
    if (seg_rows > 0 && Mo > 2 * seg_rows) {
      rc = make_tmap_2d(&tx, out2, 4, Mo - 2 * seg_rows, No, No, 32, 16, 64);
      if (rc != VIT3D_OK) return rc;
    }
    ep.atomic = 2;
  }
  if (tall) return launch_tc<false, 256, EPI_WGRAD>(ta, tb, tc, tp, ep, Mo, No, Kred, splits, false, st, 0, 3, &tx);
  if (bn == 256) return launch_tc<false, 256, EPI_WGRAD>(ta, tb, tc, tp, ep, Mo, No, Kred, splits, false, st, 0, 1, &tx);
  if (bn == 128) return launch_tc<false, 128, EPI_WGRAD>(ta, tb, tc, tp, ep, Mo, No, Kred, splits, false, st, 0, 1, &tx);
  return launch_tc<false, 64, EPI_WGRAD>(ta, tb, tc, tp, ep, Mo, No, Kred, splits, false, st, 0, 1, &tx);
}

bool tc_wgrad_supported(int prec, int M, int N, int K) {
  return prec == VIT3D_PREC_BF16 && M >= 64 && N % 64 == 0 && K % 64 == 0;
}

bool tc_linear_supported(int prec, int M, int N, int K) {
  if (M <= 0) return false;
  if (prec == VIT3D_PREC_BF16) return K % 8 == 0 && N % 8 == 0 && K >= 64 && N >= 64;
  if (prec == VIT3D_PREC_TF32) return K % 4 == 0 && N % 4 == 0 && K >= 32 && N >= 64;
  return false;
}

// fused Linear + residual + LayerNorm (k_tc_gemm_res.cu): a CTA's 128 x 256 tile must span whole rows
bool tc_linear_ln_supported(int prec, int M, int N, int K) {
  return prec == VIT3D_PREC_BF16 && tc_res_supported(M, N, K, true);
}

int tc_linear_fwd(const TcLinear& t, cudaStream_t st) {
  // fp32 residual-stream outputs (out-projection, fc2, fp32 data gradients): TMA panel epilogue
  const bool aligned = ((reinterpret_cast<uintptr_t>(t.y) | reinterpret_cast<uintptr_t>(t.residual) |
                         reinterpret_cast<uintptr_t>(t.ln_out)) & 15) == 0;
  if (t.prec == VIT3D_PREC_BF16 && t.y_f32 && t.act == VIT3D_ACT_NONE && !t.pre && aligned &&
      tc_res_supported(t.M, t.N, t.K, t.ln_out != nullptr))
    return tc_gemm_res(t, st);
  if (t.ln_out) V3_UNSUPPORTED("linear + LayerNorm: unsupported shape / alignment (M=%d N=%d K=%d)", t.M, t.N, t.K);
  TcEpilogue ep;
  ep.bias = t.bias; ep.residual = t.residual; ep.out = t.y; ep.pre = t.pre; ep.out_f32 = t.y_f32; ep.act = t.act;
  ep.round_tf32 = (t.prec == VIT3D_PREC_TF32 && t.act == VIT3D_ACT_GELU && !t.residual) ? 1 : 0;
  if (t.drop_bits) {
    if (t.y_f32 || t.N % 32) { set_error("linear + dropout: generic path needs bf16 output and N %% 32 == 0"); return VIT3D_ERR_UNSUPPORTED; }
    ep.drop_bits = t.drop_bits; ep.drop_scale = t.drop_scale;
  }
  if (t.store_dact) {
    if (!t.pre || !t.bias || t.act != VIT3D_ACT_GELU || t.y_f32 || t.N % 32) {
      set_error("linear: store_dact needs bias, GELU, a `pre` buffer, bf16 output and N %% 32 == 0");
      return VIT3D_ERR_UNSUPPORTED;
    }
    ep.store_dact = 1;
  }
  return tc_gemm(t.prec == VIT3D_PREC_TF32, t.x, t.w, t.M, t.N, t.K, ep, 1, st);
}

// ----------------------------------------------------------------------------- a1: patch embedding
// Conv3d(kernel = stride = patch) as an im2col-by-TMA GEMM in TF32: the fp32 volume is read exactly once,
// straight into the swizzled A tiles (no gather pass, no conversion pass); bias, position rows and the
// "skip the cls row" output remap are fused in the epilogue.
int make_tmap_nd(CUtensorMap* out, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                 const cuuint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return VIT3D_ERR_CUDA; }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank, const_cast<void*>(ptr), dims, strides_bytes, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(rank %d) failed (%d)", rank, (int)r); return VIT3D_ERR_CUDA; }
  return VIT3D_OK;
}

bool tc_patch_embed_supported(int B, int X, int Y, int Z, int p0, int p1, int p2, int H) {
  if (B <= 0 || p2 != Z || X % p0 || Y % p1) return false;
  const int nx = X / p0, ny = Y / p1, P = nx * ny;
  const int inner = p1 * p2;                       // contiguous floats of one patch row
  if (P > 128 || 128 % P) return false;            // whole volumes per 128-row tile
  if (ny > 256 || nx > 256 || 128 / P > 256) return false;
  if ((inner * 4) % 16 || (Y * Z * 4) % 16) return false;
  return H % 64 == 0 && H >= 64;
}

int tc_patch_embed_fwd(const float* x, const float* w, const float* bias, const float* pos, float* tokens, int B, int X,
                       int Y, int Z, int p0, int p1, int p2, int H, cudaStream_t st) {
  if (!tc_patch_embed_supported(B, X, Y, Z, p0, p1, p2, H)) V3_UNSUPPORTED("tc patch embedding: unsupported geometry");
  const int nx = X / p0, ny = Y / p1, P = nx * ny, inner = p1 * p2;
  const int vpt = 128 / P;
  const int pblocks = ceil_div(inner, 32);
  const int nkb = p0 * pblocks;
  const int M = B * P, N = H;
  const int sms = sm_count();
  const int tm = ceil_div(M, TC_BLOCK_M);
  int bn = 256;
  if (N % 256 || (long long)tm * (N / 256) < sms) bn = 128;
  if (N % 128 || (bn == 128 && (long long)tm * (N / 128) < sms)) bn = 64;
  CUtensorMap ta, tb;
  {
    // x viewed (innermost first): [inner floats][ny patches][p0 rows][nx patches][B volumes]
    cuuint64_t dims[5] = {(cuuint64_t)inner, (cuuint64_t)ny, (cuuint64_t)p0, (cuuint64_t)nx, (cuuint64_t)B};
    cuuint64_t str[4] = {(cuuint64_t)inner * 4, (cuuint64_t)Y * Z * 4, (cuuint64_t)p0 * Y * Z * 4, (cuuint64_t)X * Y * Z * 4};
    cuuint32_t box[5] = {32, (cuuint32_t)ny, 1, (cuuint32_t)nx, (cuuint32_t)vpt};
    int rc = make_tmap_nd(&ta, x, 5, dims, str, box);
    if (rc != VIT3D_OK) return rc;
    // w viewed: [inner floats][p0 rows][H filters]
    cuuint64_t wd[3] = {(cuuint64_t)inner, (cuuint64_t)p0, (cuuint64_t)H};
    cuuint64_t ws[2] = {(cuuint64_t)inner * 4, (cuuint64_t)p0 * inner * 4};
    cuuint32_t wb[3] = {32, 1, (cuuint32_t)bn};
    rc = make_tmap_nd(&tb, w, 3, wd, ws, wb);
    if (rc != VIT3D_OK) return rc;
  }
  TcEpilogue ep;
  ep.bias = bias; ep.rowadd = pos; ep.row_group = P; ep.out = tokens; ep.out_f32 = 1; ep.vols_per_tile = vpt;
  // Optional (VIT3D_TUNE_PATCH_CLUSTER, off): the filter bank (1.3 MB, re-streamed for every row tile: 32 KB per k-block
  // beside 16 KB of volume data) fetched ONCE per cluster - each CTA loads 1/cl of the filters and multicasts them.
  // The cluster's CTAs share ring slots, so they must walk equally many tiles: the grid is cut to whole co-resident
  // clusters whose tail (total % grid) is a multiple of the cluster size (B200: 74 pairs, but only 33 clusters of 4).
  // Measured at batch 1024: 117.7-119 us with pairs, 116.7-119.5 us without - not bound by L2 operand delivery
  // (ncu: the MMA thread waits for operands 31 % of its time, TF32 tensor pipe 51 % busy, 80 of 148 CTAs idle during
  // the fourth tile round of 512 tiles).
  if (bn == 256 && N == 256 && tuning(VIT3D_TUNE_PATCH_CLUSTER) != 0 && tm >= 2 * sms) {
    for (int cl = tuning(VIT3D_TUNE_PATCH_CLUSTER) >= 4 ? 4 : 2; cl >= 2 && ep.cluster == 1; cl -= 2) {
      int nmax = 0;
      {
        using Cfg = TcCfg<256>;
        auto kern = tc_gemm_kernel<true, 256, EPI_GENERIC>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(sms - sms % cl);
        cfg.blockDim = dim3(Cfg::THREADS);
        cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (cudaOccupancyMaxActiveClusters(&nmax, kern, &cfg) != cudaSuccess) { cudaGetLastError(); nmax = 0; }
      }
      int g = nmax * cl < sms ? nmax * cl : sms - sms % cl;
      for (int tries = 0; tries < 8 && g >= cl; ++tries, g -= cl)
        if (tm <= g || (tm % g) % cl == 0) break;
      if (g >= cl && g * 10 >= sms * 9 && (tm <= g || (tm % g) % cl == 0)) {      // keep >= 90 % of the SMs busy
        ep.cluster = cl;
        ep.grid_limit = g;
        cuuint64_t wd[3] = {(cuuint64_t)inner, (cuuint64_t)p0, (cuuint64_t)H};
        cuuint64_t ws[2] = {(cuuint64_t)inner * 4, (cuuint64_t)p0 * inner * 4};
        cuuint32_t wb[3] = {32, 1, (cuuint32_t)(bn / cl)};
        int rc = make_tmap_nd(&tb, w, 3, wd, ws, wb);
        if (rc != VIT3D_OK) return rc;
      }
    }
  }
  // optional 256-row tiles (two accumulators over one weight k-block, 64 KB stages of 1024 MMA cycles): measured
  // 124 us against 117 us for 128-row tiles at batch 1024 (the single accumulator pair cannot overlap a tile's
  // epilogue with the next tile's MMAs) - off by default
  if (bn == 256 && ep.cluster == 1 && tuning(VIT3D_TUNE_PATCH_TALL) != 0 && M >= 4 * TC_BLOCK_M * sm_count() / 2)
    return launch_tc<true, 256>(ta, tb, ta, ta, ep, M, N, nkb, 1, false, st, pblocks, 2);
  if (bn == 256) return launch_tc<true, 256>(ta, tb, ta, ta, ep, M, N, nkb, 1, false, st, pblocks);
  if (bn == 128) return launch_tc<true, 128>(ta, tb, ta, ta, ep, M, N, nkb, 1, false, st, pblocks);
  return launch_tc<true, 64>(ta, tb, ta, ta, ep, M, N, nkb, 1, false, st, pblocks);
}

}  // namespace vit3d
