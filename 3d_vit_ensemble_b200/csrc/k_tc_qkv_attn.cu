// Inference attention with the q|k|v projection fused in (BF16 mode, 65-token volumes, hidden 256, D = 16 or 32):
// reads the LayerNorm output yn and writes only the context and the probabilities - the packed [M, 768] q|k|v matrix of
// the two-kernel path (tc_gemm_kernel, then attn_fwd_tc_kernel) never reaches global memory.
//
// Work split.  A CTA owns one HEAD GROUP: the 32 q, 32 k and 32 v columns of 32 / D heads, whose [96 x 256] slice of
// the packed weight (48 KB) stays in shared memory for the CTA's lifetime.  The eight groups' CTAs of one range of
// whole volumes sit next to each other in the grid, so yn comes from HBM about once and the other reads hit L2.
//   warp 0      TMA producer: the weight slice once, then the CTA's rows of yn in 128-row tiles (4 k-blocks of 64)
//               through a 4-stage ring.  Tiles start at the range's first row and follow each other without gaps,
//               so a volume can straddle two tiles; no row is computed twice.
//   warp 1      TMEM allocator + tcgen05.mma issuer: M = 128, N = 96, K = 256 as 16 steps of 16 - the same K order
//               as tc_gemm_kernel's stationary schedule, so the q|k|v values are the two-kernel path's bit for bit.
//               Double-buffered accumulator (2 x 96 of 256 columns).
//   warps 2-5   epilogue, one per TMEM lane quarter: + bias, round to bf16 (epilogue_bf16_lean<.., 1>'s arithmetic)
//               into a circular buffer of 320 q|k|v rows, then `rows_full` for the tile.
//   warps 6-    attention: the (volume, head, 16-row tile) tasks of the range, dealt round-robin over the warps, run
//               attn_fwd_task (tc_attn_task.cuh) on the volumes each tile completed; `rows_free` after each tile.
// 320 rows = the 128 rows the epilogue writes + up to 64 tail rows of an unfinished volume + the 128 rows of the tile
// the attention warps are still reading, so the epilogue of tile u + 1 overlaps the attention of tile u (with 64-column
// groups the 96 KB slice leaves room for 192 rows only, and epilogue and attention ran one after the other: 79.6 against
// 65.7 us at batch 1024, DESIGN.md §3).
// Shared memory: weight slice 48 KB + yn ring 4 x 16 KB + row buffer 320 x 208 B (65 KB) + bias 384 B + barriers.
#include "ptx.cuh"
#include "tc.cuh"
#include "tc_attn_task.cuh"
#include "tc_epilogue.cuh"

namespace vit3d {

using namespace ptx;

constexpr int QA_GC = 32;                      // q (and k, v) columns of a head group
constexpr int QA_N = 3 * QA_GC;                // 96: accumulator columns per tile
constexpr int QA_TMEM_BUF = 128;               // TMEM column stride of the two accumulator buffers
constexpr int QA_GROUPS = AT_A / QA_GC;        // 8
constexpr int QA_K = 256;                      // hidden size: the reduction
constexpr int QA_KB = QA_K / 64;               // k-blocks of 128 bytes
constexpr int QA_STAGES = 4;
constexpr int QA_A_BYTES = 128 * 128;          // one 128-row x 64-column yn k-block
constexpr int QA_W_KB_BYTES = QA_N * 128;      // one 96-row k-block of the weight slice
constexpr int QA_ROWS = 320;                   // circular q|k|v row buffer
constexpr int QA_PITCH = QA_N * 2 + 16;        // 208 B: 8 consecutive rows fall on distinct 16-byte bank groups (ldmatrix)
constexpr int QA_EPI_WARPS = 4;
constexpr int QA_ATT_WARPS = 16;
constexpr int QA_THREADS = 32 * (2 + QA_EPI_WARPS + QA_ATT_WARPS);
constexpr int QA_OFF_RING = QA_KB * QA_W_KB_BYTES;
constexpr int QA_OFF_ROWS = QA_OFF_RING + QA_STAGES * QA_A_BYTES;
constexpr int QA_OFF_BIAS = QA_OFF_ROWS + QA_ROWS * QA_PITCH;
constexpr int QA_OFF_BARS = QA_OFF_BIAS + QA_N * 4;
constexpr int QA_NBARS = 2 * QA_STAGES + 2 + 2 + 1 + 2 + 2;   // full, empty, tmem_full, tmem_empty, slab, rows_full, rows_free
constexpr int QA_SMEM = QA_OFF_BARS + QA_NBARS * 8 + 16;        // + the TMEM base address word
static_assert(QA_SMEM <= 232448, "over the 227 KB shared-memory limit");
static_assert(QA_W_KB_BYTES % 1024 == 0 && QA_OFF_RING % 1024 == 0, "128B-swizzled tiles need 1024-byte alignment");

template <int D, int VIS>
__global__ void __launch_bounds__(QA_THREADS, 1)
qkv_attn_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmW, const float* __restrict__ bias,
                __nv_bfloat16* __restrict__ ctx, float* __restrict__ probs, int B, int ranges, float scale_log2e, int pld) {
  constexpr int G = QA_GC / D;                 // heads per group
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023u) __trap();        // 128B-swizzled operand tiles
  uint8_t* ring = smem + QA_OFF_RING;
  const uint32_t rows_s = smem_u32(smem + QA_OFF_ROWS);
  float* bias_s = reinterpret_cast<float*>(smem + QA_OFF_BIAS);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + QA_OFF_BARS);
  uint64_t* full_bar = bars;                                  // [QA_STAGES]
  uint64_t* empty_bar = bars + QA_STAGES;                     // [QA_STAGES]
  uint64_t* tmem_full = bars + 2 * QA_STAGES;                 // [2]
  uint64_t* tmem_empty = tmem_full + 2;                       // [2]
  uint64_t* slab_full = tmem_empty + 2;
  uint64_t* rows_full = slab_full + 1;                        // [2] the epilogue wrote tile u's rows
  uint64_t* rows_free = rows_full + 2;                        // [2] the attention warps are done with tile u's volumes
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(rows_free + 2);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int grp = (int)blockIdx.x % QA_GROUPS, range = (int)blockIdx.x / QA_GROUPS;
  const int v0 = (int)((long long)B * range / ranges), v1 = (int)((long long)B * (range + 1) / ranges);
  const int row_base = v0 * AT_S, nrows = (v1 - v0) * AT_S;
  const int ntiles = (nrows + 127) / 128;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmY);
    prefetch_tmap(&tmW);
    for (int s = 0; s < QA_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], QA_EPI_WARPS);
      mbar_init(&rows_full[b], QA_EPI_WARPS);
      mbar_init(&rows_free[b], QA_ATT_WARPS);
    }
    mbar_init(slab_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<256>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ===================================================== TMA producer
    if (lane == 0 && ntiles > 0) {
      mbar_arrive_expect_tx(slab_full, QA_KB * QA_W_KB_BYTES);
      for (int kb = 0; kb < QA_KB; ++kb)
        for (int p = 0; p < 3; ++p)       // q, k, v rows of the group: 32-row boxes stacked into one 96-row k-block
          tma_load_2d(smem + kb * QA_W_KB_BYTES + p * (QA_W_KB_BYTES / 3), &tmW, slab_full, kb * 64, p * AT_A + grp * QA_GC);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t)
        for (int kb = 0; kb < QA_KB; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], QA_A_BYTES);
          tma_load_2d(ring + stage * QA_A_BYTES, &tmY, &full_bar[stage], kb * 64, row_base + t * 128);
          if (++stage == QA_STAGES) { stage = 0; phase ^= 1; }
        }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer (one thread)
    if (elect_one() && ntiles > 0) {
      const uint32_t idesc = make_idesc(UMMA_FMT_BF16, 128, QA_N, 0, 0);
      const uint64_t ring_desc = make_smem_desc(smem_u32(ring), 16, 1024, UMMA_LAYOUT_SW128);
      const uint64_t slab_desc = make_smem_desc(smem_u32(smem), 16, 1024, UMMA_LAYOUT_SW128);
      mbar_wait(slab_full, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        mbar_wait(&tmem_empty[buf], ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * QA_TMEM_BUF;
        for (int kb = 0; kb < QA_KB; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          const uint64_t ad = ring_desc + (uint64_t)((stage * QA_A_BYTES) >> 4);
          const uint64_t bd = slab_desc + (uint64_t)((kb * QA_W_KB_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma<false>(d_tmem, ad + k * 2, bd + k * 2, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (++stage == QA_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[buf]);
      }
    }
    __syncwarp();
  } else if (warp < 2 + QA_EPI_WARPS) {
    // ===================================================== epilogue warps: TMEM lane quarter warp % 4, all 96 columns
    const int q = warp & 3;
    for (int i = (warp - 2) * 32 + lane; i < QA_N; i += QA_EPI_WARPS * 32)
      bias_s[i] = __ldg(bias + (i / QA_GC) * AT_A + grp * QA_GC + i % QA_GC);
    asm volatile("bar.sync 1, %0;" ::"n"(QA_EPI_WARPS * 32) : "memory");
    for (int u = 0; u < ntiles; ++u) {
      const int buf = u & 1;
      const uint32_t dst = rows_s + ((u * 128 + q * 32 + lane) % QA_ROWS) * QA_PITCH;
      mbar_wait(&tmem_full[buf], (u >> 1) & 1);
      if (u >= 2) mbar_wait(&rows_free[buf], ((u >> 1) - 1) & 1);   // the slots this tile overwrites are read no more
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t r[3][16];
#pragma unroll
        for (int i = 0; i < 3; ++i) tmem_ld_32x32b_x16(tmem_base + ((uint32_t)(q * 32) << 16) + buf * QA_TMEM_BUF + 48 * h + 16 * i, r[i]);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c = 48 * h + 16 * i;
          uint32_t w[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            w[j] = pack2_bf16(__uint_as_float(r[i][2 * j]) + bias_s[c + 2 * j], __uint_as_float(r[i][2 * j + 1]) + bias_s[c + 2 * j + 1]);
          st_shared_v4(dst + c * 2, w[0], w[1], w[2], w[3]);
          st_shared_v4(dst + c * 2 + 16, w[4], w[5], w[6], w[7]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&tmem_empty[buf]);
        mbar_arrive(&rows_full[buf]);
      }
    }
  } else {
    // ===================================================== attention warps
    const int aw = warp - 2 - QA_EPI_WARPS;
    int task = aw;                            // this warp's next task: (volume, head, row tile) = task / (5G), ...
    for (int u = 0; u < ntiles; ++u) {
      const int buf = u & 1;
      const int task_end = min(u * 128 + 128, nrows) / AT_S * (G * 5);     // tasks of the volumes tile u completed
      mbar_wait(&rows_full[buf], (u >> 1) & 1);
      for (; task < task_end; task += QA_ATT_WARPS) {
        const int j = task / (G * 5), hg = task % (G * 5) / 5;
        const int s0 = (j * AT_S) % QA_ROWS;
        attn_fwd_task<D, VIS, QA_GC>(
            [rows_s, s0](int r) {
              const int s = s0 + r;
              return rows_s + (uint32_t)((s >= QA_ROWS ? s - QA_ROWS : s) * QA_PITCH);
            },
            hg * D, grp * G + hg, task % 5, v0 + j, lane, ctx, probs, scale_log2e, pld);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&rows_free[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<256>(tmem_base);
}

bool tc_qkv_attn_supported(int S, int heads, int D) { return tc_attn_supported(S, heads, D) && D <= QA_GC; }

template <int D, int VIS>
static int launch_qkv_attn(const CUtensorMap& ty, const CUtensorMap& tw, const float* bias, void* ctx, float* probs, int pld,
                           int B, cudaStream_t st) {
  auto kern = qkv_attn_kernel<D, VIS>;
  V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, QA_SMEM));
  // one range of whole volumes per QA_GROUPS SMs; no range is empty
  const int ranges = B < sm_count() / QA_GROUPS ? B : sm_count() / QA_GROUPS;
  const float scale_log2e = 1.4426950408889634f / sqrtf((float)D);
  V3_CUDA(launch_pdl(kern, dim3(ranges * QA_GROUPS), dim3(QA_THREADS), (size_t)QA_SMEM, st, ty, tw, bias,
                     reinterpret_cast<__nv_bfloat16*>(ctx), probs, B, ranges, scale_log2e, pld));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
template <int D>
static int launch_qkv_attn_d(const CUtensorMap& ty, const CUtensorMap& tw, const float* bias, void* ctx, float* probs, int pld,
                             int B, cudaStream_t st) {
  if (!probs) return launch_qkv_attn<D, 0>(ty, tw, bias, ctx, probs, pld, B, st);
  return launch_qkv_attn<D, 2>(ty, tw, bias, ctx, probs, pld, B, st);
}

int tc_qkv_attn_fwd(const void* yn, const void* w_qkv, const float* b_qkv, void* ctx, float* probs, int probs_ld, int B,
                    int S, int heads, int D, cudaStream_t st) {
  if (!tc_qkv_attn_supported(S, heads, D)) V3_UNSUPPORTED("qkv attention: unsupported shape S=%d heads=%d D=%d", S, heads, D);
  if (B <= 0) return VIT3D_OK;
  if (probs && (probs_ld != 72 || (reinterpret_cast<uintptr_t>(probs) & 31))) {
    set_error("qkv attention: probability rows are 72 floats (9 whole sectors) in a 32-byte aligned buffer");
    return VIT3D_ERR_INVALID;
  }
  if (reinterpret_cast<uintptr_t>(ctx) & 15) {
    set_error("qkv attention: ctx must be 16-byte aligned");
    return VIT3D_ERR_INVALID;
  }
  CUtensorMap ty, tw;
  int rc = make_tmap_2d(&ty, yn, 2, (long long)B * S, QA_K, QA_K, 128, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&tw, w_qkv, 2, 3 * AT_A, QA_K, QA_K, QA_GC, 64, 128);
  if (rc != VIT3D_OK) return rc;
  if (D == 16) return launch_qkv_attn_d<16>(ty, tw, b_qkv, ctx, probs, probs_ld, B, st);
  return launch_qkv_attn_d<32>(ty, tw, b_qkv, ctx, probs, probs_ld, B, st);
}

}  // namespace vit3d
