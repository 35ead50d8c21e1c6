// Fused softmax attention for the 65-token sequences of the 3D ViT (a2, modeling.py:83-96), bf16.
//
// One persistent CTA per SM walks over volumes.  The packed qkv rows of a volume (65 x 768 bf16,
// contiguous in HBM) are pulled into shared memory with bulk async copies (UBLKCP, mbarrier
// completion), double buffered so the next volume streams in while this one is computed.  Each warp
// takes (head, 16-row tile) tasks: S = Q K^T with mma.sync.m16n8k16 (bf16, fp32 accumulate), the
// softmax runs in registers with quad shuffles, P (bf16) feeds the P V mma straight from the
// accumulator registers, the context tile overwrites the Q tile it came from in shared memory and the
// whole [65 x 256] context block leaves with bulk async stores.  With vis=True the fp32 probabilities
// (B,k,65,65) are written from registers.  HBM traffic per volume: 99.8 KB in, 33.3 KB out
// (+ k*65*65*4 B of probabilities) - the kernel is bandwidth bound.
#include <stdlib.h>

#include "ptx.cuh"
#include "tc.cuh"
#include "tc_attn_task.cuh"

namespace vit3d {

using namespace ptx;

constexpr int AT_ROWB = 3 * AT_A * 2;       // 1536 bytes of qkv per token
constexpr int AT_PITCH = AT_ROWB + 16;      // padded smem row pitch: conflict-free ldmatrix
constexpr int AT_BUF = AT_S * AT_PITCH;     // 100,880 bytes per volume buffer
constexpr int AT_THREADS = 512;          // backward kernel: 16 warps
constexpr int AT_SMEM = 2 * AT_BUF + 64 + 128;

__device__ __forceinline__ void bulk_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(sdst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(gdst)),
               "r"(smem_u32(ssrc)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// THREADS compute threads: 512 (16 warps) or 640 (20 warps), plus one producer warp.  A volume is HEADS * 5
// (head, 16-row tile) tasks: 40 tasks take 3 rounds of 16 warps but 2 rounds of 20 (80 tasks: 5 vs 4).
// The warps are only coupled through data: the producer warp refills a volume buffer when all compute warps
// have released it (mbarrier with one arrival per warp), and every warp ships its own context tile, so a fast
// warp walks on into the next volume instead of waiting at a block-wide barrier (15 % of the samples before).
// VIS: the probability layout (attn_fwd_task, tc_attn_task.cuh).
template <int D, int THREADS, int VIS>
__global__ void __launch_bounds__(THREADS + 32, 1)
attn_fwd_tc_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ ctx, float* __restrict__ probs,
                   int B, float scale_log2e, int pld) {
  constexpr int HEADS = AT_A / D;
  constexpr int NW = THREADS / 32;    // compute warps
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 2 * AT_BUF);     // [2] volume landed
  uint64_t* freeb = full + 2;                                          // [2] every compute warp is done with it

  // warp index through a shuffle: warp-uniform for the compiler, so the role branches are uniform control flow
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    mbar_init(&freeb[0], NW);
    mbar_init(&freeb[1], NW);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();
  pdl_wait();

  if (warp == NW) {
    // ===================================================== producer warp: one bulk copy per token row
    int it = 0;
    for (int b = blockIdx.x; b < B; b += gridDim.x, ++it) {
      const int buf = it & 1;
      if (it >= 2) mbar_wait(&freeb[buf], ((it >> 1) - 1) & 1);       // volume it-2 has been consumed
      if (lane == 0) mbar_arrive_expect_tx(&full[buf], AT_S * AT_ROWB);
      __syncwarp();
      const uint8_t* src = reinterpret_cast<const uint8_t*>(qkv) + (size_t)b * AT_S * AT_ROWB;
      uint8_t* dst = smem + buf * AT_BUF;
      for (int r = lane; r < AT_S; r += 32) bulk_g2s(dst + r * AT_PITCH, src + (size_t)r * AT_ROWB, AT_ROWB, &full[buf]);
    }
    return;
  }

  int it = 0;
  for (int b = blockIdx.x; b < B; b += gridDim.x, ++it) {
    const int buf = it & 1;
    mbar_wait(&full[buf], (it >> 1) & 1);
    const uint32_t sb = smem_u32(smem + buf * AT_BUF);

    // HEADS * 5 tasks over NW warps: 40 over 16 is 2.5 per warp.  The warps are only coupled through the
    // double-buffered volume images, so the half with three tasks in this volume takes two in the next one
    // (the assignment rotates by NW / 2 per volume) and every warp does five tasks per two volumes.
    for (int task = (warp + (it & 1) * (NW / 2)) % NW; task < HEADS * 5; task += NW) {
      const int h = task / 5;
      attn_fwd_task<D, VIS, AT_A>([sb](int r) { return sb + (uint32_t)(r * AT_PITCH); }, h * D, h, task % 5, b, lane, ctx, probs,
                                  scale_log2e, pld);
    }
    // this warp no longer reads the volume buffer
    __syncwarp();
    if (lane == 0) mbar_arrive(&freeb[buf]);
  }
}

bool tc_attn_supported(int S, int heads, int D) {
  return S == AT_S && heads * D == AT_A && (D == 16 || D == 32 || D == 64);
}

template <int D, int THREADS, int VIS>
static int launch_attn_v(const void* qkv, void* ctx, float* probs, int pld, int B, cudaStream_t st) {
  auto kern = attn_fwd_tc_kernel<D, THREADS, VIS>;
  V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM));
  const int grid = B < sm_count() ? B : sm_count();
  const float scale_log2e = 1.4426950408889634f / sqrtf((float)D);
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS + 32), (size_t)AT_SMEM, st, reinterpret_cast<const __nv_bfloat16*>(qkv),
                     reinterpret_cast<__nv_bfloat16*>(ctx), probs, B, scale_log2e, pld));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
template <int D, int THREADS>
static int launch_attn(const void* qkv, void* ctx, float* probs, int pld, int B, cudaStream_t st) {
  if (!probs) return launch_attn_v<D, THREADS, 0>(qkv, ctx, probs, pld, B, st);
  return pld == AT_S ? launch_attn_v<D, THREADS, 1>(qkv, ctx, probs, pld, B, st) : launch_attn_v<D, THREADS, 2>(qkv, ctx, probs, pld, B, st);
}
// 0 = automatic.  20 warps make a volume of 8 heads exactly two rounds of (head, row-tile) tasks and are the
// faster choice without the probabilities; with them (vis=True) the kernel is bound by its store path and 16
// warps measured faster for 8 and 16 heads (63.5 vs 67.6 us, 110.9 vs 111.3 us at batch 1024), 20 for 4 heads
// (45.7 vs 49.9 us).
static int attn_threads(int D, bool vis) {
  const int v = tuning(VIT3D_TUNE_ATTN_THREADS);
  if (v == 512 || v == 640) return v;
  return (D <= 32 && vis) ? 512 : 640;
}

int tc_attn_fwd_unit(const void* qkv, void* ctx, float* probs, int probs_ld, int B, int D, cudaStream_t st);
int tc_attn_fwd(const void* qkv, void* ctx, float* probs, int probs_ld, int B, int S, int heads, int D, cudaStream_t st) {
  if (!tc_attn_supported(S, heads, D)) V3_UNSUPPORTED("tc attention: unsupported shape S=%d heads=%d D=%d", S, heads, D);
  if (B <= 0) return VIT3D_OK;
  if (probs && probs_ld != S && (probs_ld != 72 || (reinterpret_cast<uintptr_t>(probs) & 31))) {
    set_error("tc attention: padded probability rows are 72 floats (9 whole sectors) in a 32-byte aligned buffer");
    return VIT3D_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(ctx) & 15) ||
      (reinterpret_cast<uintptr_t>(probs) & 7)) {
    set_error("tc attention: qkv/ctx must be 16-byte aligned, probs 8-byte aligned");
    return VIT3D_ERR_INVALID;
  }
  {
    const int mode = tuning(VIT3D_TUNE_ATTN_FWD_UNIT);      // 0: one volume per CTA; 1: units when no probabilities; 2: always
    if (mode == 2 || (mode == 1 && probs == nullptr)) return tc_attn_fwd_unit(qkv, ctx, probs, probs_ld, B, D, st);
  }
  if (attn_threads(D, probs != nullptr) == 640) {
    if (D == 16) return launch_attn<16, 640>(qkv, ctx, probs, probs_ld, B, st);
    if (D == 32) return launch_attn<32, 640>(qkv, ctx, probs, probs_ld, B, st);
    return launch_attn<64, 640>(qkv, ctx, probs, probs_ld, B, st);
  }
  if (D == 16) return launch_attn<16, 512>(qkv, ctx, probs, probs_ld, B, st);
  if (D == 32) return launch_attn<32, 512>(qkv, ctx, probs, probs_ld, B, st);
  return launch_attn<64, 512>(qkv, ctx, probs, probs_ld, B, st);
}

// ============================================================================ backward
// dqkv from dctx, probabilities recomputed (nothing but qkv is saved by the forward).  One CTA per SM,
// one volume at a time: qkv (65 x 768) and dctx (65 x 256) are staged in shared memory by bulk copies.
//   pass 1, task = (head, 16-query tile):  S = Q K^T, P = softmax, dP = dO V^T, delta = rowsum(P dP),
//           dS = P (dP - delta) / sqrt(D), dQ = dS K  -> dQ staging tile; row statistics (max, 1/sum,
//           delta) go to shared memory.
//   pass 2, task = (head, 16-key tile):    S^T = K Q^T, P^T from the saved statistics, dP^T = V dO^T,
//           dS^T, dV = P^T dO, dK = dS^T Q -> written over the K / V tile they came from (dead by then).
// All seven products run on mma.sync.m16n8k16 (bf16 in, fp32 accumulate); softmax math is fp32.
constexpr int AB_DOP = AT_A * 2 + 16;                 // padded row pitch of the dctx / dQ images (528 B)
constexpr int AB_QKV = AT_S * AT_PITCH;               // 100,880
constexpr int AB_DO = AT_S * AB_DOP;                  // 34,320
constexpr int AB_STATS = 16 * 80 * 3 * 4;             // (max, 1/sum, delta) x 80 rows x <=16 heads
constexpr int AB_SMEM = AB_QKV + 2 * AB_DO + AB_STATS + 64 + 128;

template <int D>
__global__ void __launch_bounds__(AT_THREADS, 1)
attn_bwd_tc_kernel(const __nv_bfloat16* __restrict__ dctx, const __nv_bfloat16* __restrict__ qkv,
                   __nv_bfloat16* __restrict__ dqkv, float* __restrict__ db_q, float* __restrict__ db_k,
                   float* __restrict__ db_v, int B, float scale, float scale_log2e) {
  constexpr int HEADS = AT_A / D;
  constexpr int KSTEPS = D / 16;
  constexpr int NT = 10;
  constexpr int DT = D / 8;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  uint8_t* s_qkv = smem;
  uint8_t* s_do = smem + AB_QKV;
  uint8_t* s_dq = s_do + AB_DO;
  float* s_stat = reinterpret_cast<float*>(s_dq + AB_DO);        // [HEADS][3][80]
  uint64_t* full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_stat) + AB_STATS);

  // warp index through a shuffle: warp-uniform for the compiler, so the role branches are uniform control flow
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  if (threadIdx.x == 0) {
    mbar_init(full, 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();
  pdl_wait();
  const uint32_t sb = smem_u32(s_qkv), dob = smem_u32(s_do);
  // q / k / v bias gradients = column sums of dq | dk | dv over all tokens: thread t keeps the partial sums of
  // columns t and 512 + t of the [65 x 768] gradient image over this CTA's volumes, one atomic each at the end
  float bsum0 = 0.f, bsum1 = 0.f;

  int it = 0;
  for (int b = blockIdx.x; b < B; b += gridDim.x, ++it) {
    if (warp == 0) {
      bulk_wait_read0();     // previous volume's stores have finished reading shared memory
      if (lane == 0) mbar_arrive_expect_tx(full, AT_S * (AT_ROWB + AT_A * 2));
      __syncwarp();
      const uint8_t* src = reinterpret_cast<const uint8_t*>(qkv) + (size_t)b * AT_S * AT_ROWB;
      const uint8_t* dsrc = reinterpret_cast<const uint8_t*>(dctx) + (size_t)b * AT_S * AT_A * 2;
      for (int r = lane; r < AT_S; r += 32) {
        bulk_g2s(s_qkv + r * AT_PITCH, src + (size_t)r * AT_ROWB, AT_ROWB, full);
        bulk_g2s(s_do + r * AB_DOP, dsrc + (size_t)r * AT_A * 2, AT_A * 2, full);
      }
    }
    mbar_wait(full, it & 1);

    // ------------------------------------------------------------------ pass 1: query tiles
    for (int task = warp; task < HEADS * 5; task += AT_THREADS / 32) {
      const int h = task / 5, rt = task % 5;
      const int r0 = rt * 16;
      uint32_t qa[KSTEPS][4], da[KSTEPS][4];
      {
        const int row = min(r0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          ldsm_x4(sb + row * AT_PITCH + (h * D + ks * 16 + (lane >> 4) * 8) * 2, qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
          ldsm_x4(dob + row * AB_DOP + (h * D + ks * 16 + (lane >> 4) * 8) * 2, da[ks][0], da[ks][1], da[ks][2], da[ks][3]);
        }
      }
      float s[NT][4], dp[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
        if (nt < 9) {
          const int key = min(nt * 8 + (lane & 7), AT_S - 1);
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            uint32_t b0, b1;
            ldsm_x2(sb + key * AT_PITCH + (AT_A + h * D + ks * 16 + ((lane >> 3) & 1) * 8) * 2, b0, b1);
            mma_bf16(s[nt], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b0, b1);
            ldsm_x2(sb + key * AT_PITCH + (2 * AT_A + h * D + ks * 16 + ((lane >> 3) & 1) * 8) * 2, b0, b1);
            mma_bf16(dp[nt], da[ks][0], da[ks][1], da[ks][2], da[ks][3], b0, b1);
          }
        }
      }
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 9; ++nt) {
        const int c = nt * 8 + 2 * t;
        if (c < AT_S) { mx0 = fmaxf(mx0, s[nt][0]); mx1 = fmaxf(mx1, s[nt][2]); }
        if (c + 1 < AT_S) { mx0 = fmaxf(mx0, s[nt][1]); mx1 = fmaxf(mx1, s[nt][3]); }
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const int c = nt * 8 + 2 * t;
        const bool v0 = c < AT_S, v1 = c + 1 < AT_S;
        s[nt][0] = v0 ? ex2_approx((s[nt][0] - mx0) * scale_log2e) : 0.f;
        s[nt][1] = v1 ? ex2_approx((s[nt][1] - mx0) * scale_log2e) : 0.f;
        s[nt][2] = v0 ? ex2_approx((s[nt][2] - mx1) * scale_log2e) : 0.f;
        s[nt][3] = v1 ? ex2_approx((s[nt][3] - mx1) * scale_log2e) : 0.f;
        sum0 += s[nt][0] + s[nt][1];
        sum1 += s[nt][2] + s[nt][3];
      }
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
      const float inv0 = 1.f / sum0, inv1 = 1.f / sum1;
      float dl0 = 0.f, dl1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] *= inv0; s[nt][1] *= inv0; s[nt][2] *= inv1; s[nt][3] *= inv1;       // P
        dl0 += s[nt][0] * dp[nt][0] + s[nt][1] * dp[nt][1];
        dl1 += s[nt][2] * dp[nt][2] + s[nt][3] * dp[nt][3];
      }
      dl0 += __shfl_xor_sync(0xffffffffu, dl0, 1);
      dl0 += __shfl_xor_sync(0xffffffffu, dl0, 2);
      dl1 += __shfl_xor_sync(0xffffffffu, dl1, 1);
      dl1 += __shfl_xor_sync(0xffffffffu, dl1, 2);
      const int row0 = r0 + g, row1 = r0 + g + 8;
      if (t == 0) {
        float* st = s_stat + h * 240;
        st[row0] = mx0; st[80 + row0] = inv0; st[160 + row0] = dl0;
        st[row1] = mx1; st[80 + row1] = inv1; st[160 + row1] = dl1;
      }
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {                                              // dS (P is 0 on padding)
        s[nt][0] *= (dp[nt][0] - dl0) * scale; s[nt][1] *= (dp[nt][1] - dl0) * scale;
        s[nt][2] *= (dp[nt][2] - dl1) * scale; s[nt][3] *= (dp[nt][3] - dl1) * scale;
      }
      float o[DT][4];
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 5; ++kk) {
        const uint32_t a0 = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
        const uint32_t a1 = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        const uint32_t a2 = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        const uint32_t a3 = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        const int key = min(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          uint32_t b0, b1;
          ldsm_x2_t(sb + key * AT_PITCH + (AT_A + h * D + dt * 8) * 2, b0, b1);      // K rows, transposed
          mma_bf16(o[dt], a0, a1, a2, a3, b0, b1);
        }
      }
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const int col = h * D + dt * 8 + 2 * t;
        if (row0 < AT_S) *reinterpret_cast<uint32_t*>(s_dq + row0 * AB_DOP + col * 2) = pack_bf16(o[dt][0], o[dt][1]);
        if (row1 < AT_S) *reinterpret_cast<uint32_t*>(s_dq + row1 * AB_DOP + col * 2) = pack_bf16(o[dt][2], o[dt][3]);
      }
    }
    __syncthreads();

    // ------------------------------------------------------------------ pass 2: key tiles
    for (int task = warp; task < HEADS * 5; task += AT_THREADS / 32) {
      const int h = task / 5, kt = task % 5;
      const int k0 = kt * 16;
      const float* st = s_stat + h * 240;
      uint32_t ka[KSTEPS][4], va[KSTEPS][4];
      {
        const int row = min(k0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          ldsm_x4(sb + row * AT_PITCH + (AT_A + h * D + ks * 16 + (lane >> 4) * 8) * 2, ka[ks][0], ka[ks][1], ka[ks][2], ka[ks][3]);
          ldsm_x4(sb + row * AT_PITCH + (2 * AT_A + h * D + ks * 16 + (lane >> 4) * 8) * 2, va[ks][0], va[ks][1], va[ks][2], va[ks][3]);
        }
      }
      float s[NT][4], dp[NT][4];     // rows = keys (g, g+8), columns = queries
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
        if (nt < 9) {
          const int qrow = min(nt * 8 + (lane & 7), AT_S - 1);
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            uint32_t b0, b1;
            ldsm_x2(sb + qrow * AT_PITCH + (h * D + ks * 16 + ((lane >> 3) & 1) * 8) * 2, b0, b1);      // Q rows
            mma_bf16(s[nt], ka[ks][0], ka[ks][1], ka[ks][2], ka[ks][3], b0, b1);
            ldsm_x2(dob + qrow * AB_DOP + (h * D + ks * 16 + ((lane >> 3) & 1) * 8) * 2, b0, b1);       // dO rows
            mma_bf16(dp[nt], va[ks][0], va[ks][1], va[ks][2], va[ks][3], b0, b1);
          }
        }
      }
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const int c = nt * 8 + 2 * t;
        const bool v0 = c < AT_S, v1 = c + 1 < AT_S;
        const float m0 = v0 ? st[c] : 0.f, i0 = v0 ? st[80 + c] : 0.f, d0 = v0 ? st[160 + c] : 0.f;
        const float m1 = v1 ? st[c + 1] : 0.f, i1 = v1 ? st[80 + c + 1] : 0.f, d1 = v1 ? st[160 + c + 1] : 0.f;
        const float p00 = v0 ? ex2_approx((s[nt][0] - m0) * scale_log2e) * i0 : 0.f;       // P^T
        const float p01 = v1 ? ex2_approx((s[nt][1] - m1) * scale_log2e) * i1 : 0.f;
        const float p10 = v0 ? ex2_approx((s[nt][2] - m0) * scale_log2e) * i0 : 0.f;
        const float p11 = v1 ? ex2_approx((s[nt][3] - m1) * scale_log2e) * i1 : 0.f;
        s[nt][0] = p00; s[nt][1] = p01; s[nt][2] = p10; s[nt][3] = p11;
        dp[nt][0] = p00 * (dp[nt][0] - d0) * scale; dp[nt][1] = p01 * (dp[nt][1] - d1) * scale;   // dS^T
        dp[nt][2] = p10 * (dp[nt][2] - d0) * scale; dp[nt][3] = p11 * (dp[nt][3] - d1) * scale;
      }
      float ov[DT][4], ok[DT][4];
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        ov[dt][0] = ov[dt][1] = ov[dt][2] = ov[dt][3] = 0.f;
        ok[dt][0] = ok[dt][1] = ok[dt][2] = ok[dt][3] = 0.f;
      }
#pragma unroll
      for (int kk = 0; kk < 5; ++kk) {
        const uint32_t p0 = pack_bf16(s[2 * kk][0], s[2 * kk][1]), p1 = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        const uint32_t p2 = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]), p3 = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        const uint32_t e0 = pack_bf16(dp[2 * kk][0], dp[2 * kk][1]), e1 = pack_bf16(dp[2 * kk][2], dp[2 * kk][3]);
        const uint32_t e2 = pack_bf16(dp[2 * kk + 1][0], dp[2 * kk + 1][1]), e3 = pack_bf16(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
        const int qrow = min(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          uint32_t b0, b1;
          ldsm_x2_t(dob + qrow * AB_DOP + (h * D + dt * 8) * 2, b0, b1);              // dO rows, transposed
          mma_bf16(ov[dt], p0, p1, p2, p3, b0, b1);
          ldsm_x2_t(sb + qrow * AT_PITCH + (h * D + dt * 8) * 2, b0, b1);             // Q rows, transposed
          mma_bf16(ok[dt], e0, e1, e2, e3, b0, b1);
        }
      }
      __syncwarp();
      const int row0 = k0 + g, row1 = k0 + g + 8;
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const int col = h * D + dt * 8 + 2 * t;
        if (row0 < AT_S) {
          *reinterpret_cast<uint32_t*>(s_qkv + row0 * AT_PITCH + (AT_A + col) * 2) = pack_bf16(ok[dt][0], ok[dt][1]);
          *reinterpret_cast<uint32_t*>(s_qkv + row0 * AT_PITCH + (2 * AT_A + col) * 2) = pack_bf16(ov[dt][0], ov[dt][1]);
        }
        if (row1 < AT_S) {
          *reinterpret_cast<uint32_t*>(s_qkv + row1 * AT_PITCH + (AT_A + col) * 2) = pack_bf16(ok[dt][2], ok[dt][3]);
          *reinterpret_cast<uint32_t*>(s_qkv + row1 * AT_PITCH + (2 * AT_A + col) * 2) = pack_bf16(ov[dt][2], ov[dt][3]);
        }
      }
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (warp == 0) {
      uint8_t* dst = reinterpret_cast<uint8_t*>(dqkv) + (size_t)b * AT_S * AT_ROWB;
      for (int r = lane; r < AT_S; r += 32) {
        bulk_s2g(dst + (size_t)r * AT_ROWB, s_dq + r * AB_DOP, AT_A * 2);                            // dQ
        bulk_s2g(dst + (size_t)r * AT_ROWB + AT_A * 2, s_qkv + r * AT_PITCH + AT_A * 2, 2 * AT_A * 2);  // dK | dV
      }
      bulk_commit();
    }
    if (db_q) {
      const int c0 = threadIdx.x;                 // 0..511: dQ columns 0..255, dK columns 256..511
      {
        const uint8_t* base = c0 < AT_A ? s_dq + c0 * 2 : s_qkv + c0 * 2;
        const int pitch = c0 < AT_A ? AB_DOP : AT_PITCH;
        float a = 0.f;
#pragma unroll 5
        for (int r = 0; r < AT_S; ++r) a += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(base + r * pitch));
        bsum0 += a;
      }
      if (c0 < AT_A) {                            // dV columns 512..767
        const uint8_t* base = s_qkv + (2 * AT_A + c0) * 2;
        float a = 0.f;
#pragma unroll 5
        for (int r = 0; r < AT_S; ++r) a += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(base + r * AT_PITCH));
        bsum1 += a;
      }
      __syncthreads();       // the next volume's loads overwrite the images these sums read
    }
  }
  if (db_q) {
    const int c0 = threadIdx.x;
    if (blockIdx.x < B) {
      atomicAdd(c0 < AT_A ? db_q + c0 : db_k + (c0 - AT_A), bsum0);
      if (c0 < AT_A) atomicAdd(db_v + c0, bsum1);
    }
  }
  if (warp == 0) bulk_wait0();
}

// ---------------------------------------------------------------------------- backward, unit kernel
// Same math as attn_bwd_tc_kernel, re-cut for the SM: a work unit is (volume, group of 4 heads), a CTA is 4 warps
// and ONE WARP OWNS ONE HEAD for both passes (its row statistics never leave the warp, no CTA barrier between the
// passes).  The unit's q | k | v | dO column blocks arrive as 65-row x 128-byte boxes (TMA, SWIZZLE_128B: 4 * NB
// tensor copies instead of 130 per-row bulk copies, ~46 cycles of TMA service each), dQ / dK / dV leave the same
// way.  ~50 KB of shared memory and 128 registers per thread: four CTAs per SM at D = 16, so one CTA's loads and
// stores hide behind the other three's math, and a batch of 256 volumes is 1024 units over 592 CTA slots
// (7 units on the busiest SM = 1.75 volumes, where one-volume-per-CTA needs 2).
constexpr int AU_TILE = 72 * 128;          // one column block: 65 rows (padded to a multiple of 8) of 128 bytes
template <int D> struct AuCfg {
  static constexpr int UC = 4 * D;                    // columns of a unit (4 heads)
  static constexpr int NB = UC / 64;                  // 128-byte column blocks per matrix
  static constexpr int MAT = NB * AU_TILE;
  static constexpr int STATS = 4 * 240 * 4;           // (max, 1/sum, delta) x 80 rows per warp
  static constexpr int SMEM = 5 * MAT + STATS + 64 + 1024;
  static constexpr int CTAS = D == 16 ? 4 : (D == 32 ? 2 : 1);
  static constexpr int NC = (3 * UC + 127) / 128;     // bias-gradient columns per thread
};
// byte address of (row, byte column colb) inside a matrix of swizzled column blocks
__device__ __forceinline__ uint32_t au_addr(uint32_t base, int row, int colb) {
  return base + (colb >> 7) * AU_TILE + row * 128 + ((((colb >> 4) ^ row) & 7) << 4) + (colb & 15);
}
__device__ __forceinline__ void st_shared_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void au_store_box(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}

template <int D>
__global__ void __launch_bounds__(128, AuCfg<D>::CTAS)
attn_bwd_unit_kernel(const __grid_constant__ CUtensorMap tmQkv, const __grid_constant__ CUtensorMap tmDo,
                     const __grid_constant__ CUtensorMap tmDqkv, float* __restrict__ db_q, float* __restrict__ db_k,
                     float* __restrict__ db_v, int units, int groups, float scale, float scale_log2e) {
  using Cfg = AuCfg<D>;
  constexpr int KSTEPS = D / 16;
  constexpr int NT = 10;
  constexpr int DT = D / 8;
  constexpr int MAT = Cfg::MAT, NB = Cfg::NB, UC = Cfg::UC;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sq = smem_u32(smem), sk = sq + MAT, sv = sk + MAT, sdo = sv + MAT, sdq = sdo + MAT;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  float* st = reinterpret_cast<float*>(smem + 5 * MAT) + warp * 240;       // [0,80): max c + log2 sum, [80,160): delta
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 5 * MAT + Cfg::STATS);
  const int g = lane >> 2, t = lane & 3;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQkv);
    prefetch_tmap(&tmDo);
    prefetch_tmap(&tmDqkv);
    mbar_init(full, 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();
  pdl_wait();
  const int hq = blockIdx.x % groups;      // the grid is a multiple of `groups`: a CTA keeps its head group
  const int c0 = hq * UC;
  const int hc = warp * D * 2;             // byte column of this warp's head inside the unit
  float bs[Cfg::NC];
#pragma unroll
  for (int i = 0; i < Cfg::NC; ++i) bs[i] = 0.f;

  int it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int row_g = (u / groups) * AT_S;
    if (threadIdx.x == 0) {
      bulk_wait_read0();                   // the previous unit's stores have finished reading shared memory
      mbar_arrive_expect_tx(full, 4 * NB * AT_S * 128);
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        tma_load_2d(smem + j * AU_TILE, &tmQkv, full, c0 + 64 * j, row_g);
        tma_load_2d(smem + MAT + j * AU_TILE, &tmQkv, full, AT_A + c0 + 64 * j, row_g);
        tma_load_2d(smem + 2 * MAT + j * AU_TILE, &tmQkv, full, 2 * AT_A + c0 + 64 * j, row_g);
        tma_load_2d(smem + 3 * MAT + j * AU_TILE, &tmDo, full, c0 + 64 * j, row_g);
      }
    }
    mbar_wait(full, it & 1);

    // ------------------------------------------------------------------ pass 1: query tiles of this warp's head
#pragma unroll 1
    for (int rt = 0; rt < 5; ++rt) {
      const int r0 = rt * 16;
      uint32_t qa[KSTEPS][4], da[KSTEPS][4];
      {
        const int row = min(r0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          ldsm_x4(au_addr(sq, row, hc + ks * 32 + (lane >> 4) * 16), qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
          ldsm_x4(au_addr(sdo, row, hc + ks * 32 + (lane >> 4) * 16), da[ks][0], da[ks][1], da[ks][2], da[ks][3]);
        }
      }
      float s[NT][4], dp[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
        if (nt < 9) {
          const int key = min(nt * 8 + (lane & 7), AT_S - 1);
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            uint32_t b0, b1;
            ldsm_x2(au_addr(sk, key, hc + ks * 32 + ((lane >> 3) & 1) * 16), b0, b1);
            mma_bf16(s[nt], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b0, b1);
            ldsm_x2(au_addr(sv, key, hc + ks * 32 + ((lane >> 3) & 1) * 16), b0, b1);
            mma_bf16(dp[nt], da[ks][0], da[ks][1], da[ks][2], da[ks][3], b0, b1);
          }
        }
      }
      // softmax statistics over the 65 valid keys: columns 0..63 (nt < 8) are always valid, nt = 8 holds only
      // key 64 (quad lane 0, first element), nt = 9 is padding for the K = 80 reduction of dQ = dS K
      const bool tail = t == 0;
      float mx0 = tail ? s[8][0] : -INFINITY, mx1 = tail ? s[8][2] : -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mc0 = mx0 * scale_log2e, mc1 = mx1 * scale_log2e;
      // e = exp(s - max) (unnormalised P), sum = rowsum(e), dl = rowsum(e dP): one FFMA + MUFU + FADD + FFMA per element
      float sum0 = 0.f, sum1 = 0.f, dl0 = 0.f, dl1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = ex2_approx(fmaf(s[nt][0], scale_log2e, -mc0));
        s[nt][1] = ex2_approx(fmaf(s[nt][1], scale_log2e, -mc0));
        s[nt][2] = ex2_approx(fmaf(s[nt][2], scale_log2e, -mc1));
        s[nt][3] = ex2_approx(fmaf(s[nt][3], scale_log2e, -mc1));
        sum0 += s[nt][0] + s[nt][1];
        sum1 += s[nt][2] + s[nt][3];
        dl0 = fmaf(s[nt][0], dp[nt][0], fmaf(s[nt][1], dp[nt][1], dl0));
        dl1 = fmaf(s[nt][2], dp[nt][2], fmaf(s[nt][3], dp[nt][3], dl1));
      }
      s[8][0] = tail ? ex2_approx(fmaf(s[8][0], scale_log2e, -mc0)) : 0.f;
      s[8][2] = tail ? ex2_approx(fmaf(s[8][2], scale_log2e, -mc1)) : 0.f;
      s[8][1] = s[8][3] = 0.f;
      sum0 += s[8][0]; sum1 += s[8][2];
      dl0 = fmaf(s[8][0], dp[8][0], dl0);
      dl1 = fmaf(s[8][2], dp[8][2], dl1);
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
      dl0 += __shfl_xor_sync(0xffffffffu, dl0, 1);
      dl0 += __shfl_xor_sync(0xffffffffu, dl0, 2);
      dl1 += __shfl_xor_sync(0xffffffffu, dl1, 1);
      dl1 += __shfl_xor_sync(0xffffffffu, dl1, 2);
      const float inv0 = 1.f / sum0, inv1 = 1.f / sum1;
      dl0 *= inv0; dl1 *= inv1;                        // delta = rowsum(P dP)
      const int row0 = r0 + g, row1 = r0 + g + 8;
      if (tail) {
        // pass 2 rebuilds P = exp2(s c - (max c + log2 sum)) with one FFMA + MUFU per element
        st[row0] = mc0 + __log2f(sum0); st[80 + row0] = dl0;
        st[row1] = mc1 + __log2f(sum1); st[80 + row1] = dl1;
      }
      // dS / (scale / sum) = e (dP - delta); the per-row factor scale / sum is applied to the dQ tile instead
#pragma unroll
      for (int nt = 0; nt < 9; ++nt) {
        s[nt][0] *= dp[nt][0] - dl0; s[nt][1] *= dp[nt][1] - dl0;
        s[nt][2] *= dp[nt][2] - dl1; s[nt][3] *= dp[nt][3] - dl1;
      }
      s[9][0] = s[9][1] = s[9][2] = s[9][3] = 0.f;
      const float ks0 = inv0 * scale, ks1 = inv1 * scale;
      float o[DT][4];
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 5; ++kk) {
        const uint32_t a0 = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
        const uint32_t a1 = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        const uint32_t a2 = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        const uint32_t a3 = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        const int key = min(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          uint32_t b0, b1;
          ldsm_x2_t(au_addr(sk, key, hc + dt * 16), b0, b1);                          // K rows, transposed
          mma_bf16(o[dt], a0, a1, a2, a3, b0, b1);
        }
      }
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const int colb = hc + (dt * 8 + 2 * t) * 2;
        if (row0 < AT_S) st_shared_u32(au_addr(sdq, row0, colb), pack_bf16(o[dt][0] * ks0, o[dt][1] * ks0));
        if (row1 < AT_S) st_shared_u32(au_addr(sdq, row1, colb), pack_bf16(o[dt][2] * ks1, o[dt][3] * ks1));
      }
    }
    __syncwarp();

    // ------------------------------------------------------------------ pass 2: key tiles of the same head
#pragma unroll 1
    for (int kt = 0; kt < 5; ++kt) {
      const int k0 = kt * 16;
      uint32_t ka[KSTEPS][4], va[KSTEPS][4];
      {
        const int row = min(k0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          ldsm_x4(au_addr(sk, row, hc + ks * 32 + (lane >> 4) * 16), ka[ks][0], ka[ks][1], ka[ks][2], ka[ks][3]);
          ldsm_x4(au_addr(sv, row, hc + ks * 32 + (lane >> 4) * 16), va[ks][0], va[ks][1], va[ks][2], va[ks][3]);
        }
      }
      float s[NT][4], dp[NT][4];     // rows = keys (g, g+8), columns = queries
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
        if (nt < 9) {
          const int qrow = min(nt * 8 + (lane & 7), AT_S - 1);
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            uint32_t b0, b1;
            ldsm_x2(au_addr(sq, qrow, hc + ks * 32 + ((lane >> 3) & 1) * 16), b0, b1);      // Q rows
            mma_bf16(s[nt], ka[ks][0], ka[ks][1], ka[ks][2], ka[ks][3], b0, b1);
            ldsm_x2(au_addr(sdo, qrow, hc + ks * 32 + ((lane >> 3) & 1) * 16), b0, b1);     // dO rows
            mma_bf16(dp[nt], va[ks][0], va[ks][1], va[ks][2], va[ks][3], b0, b1);
          }
        }
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {                 // query columns 0..63: always valid
        const int c = nt * 8 + 2 * t;
        const float2 ml = *reinterpret_cast<const float2*>(st + c), dl = *reinterpret_cast<const float2*>(st + 80 + c);
        s[nt][0] = ex2_approx(fmaf(s[nt][0], scale_log2e, -ml.x));       // P^T
        s[nt][1] = ex2_approx(fmaf(s[nt][1], scale_log2e, -ml.y));
        s[nt][2] = ex2_approx(fmaf(s[nt][2], scale_log2e, -ml.x));
        s[nt][3] = ex2_approx(fmaf(s[nt][3], scale_log2e, -ml.y));
        dp[nt][0] = s[nt][0] * (dp[nt][0] - dl.x); dp[nt][1] = s[nt][1] * (dp[nt][1] - dl.y);   // dS^T / scale
        dp[nt][2] = s[nt][2] * (dp[nt][2] - dl.x); dp[nt][3] = s[nt][3] * (dp[nt][3] - dl.y);
      }
      {                                                // query 64 (quad lane 0, first element); the rest is padding
        const bool tail = t == 0;
        const float ml = st[64], dl = st[80 + 64];
        s[8][0] = tail ? ex2_approx(fmaf(s[8][0], scale_log2e, -ml)) : 0.f;
        s[8][2] = tail ? ex2_approx(fmaf(s[8][2], scale_log2e, -ml)) : 0.f;
        s[8][1] = s[8][3] = 0.f;
        dp[8][0] = s[8][0] * (dp[8][0] - dl); dp[8][2] = s[8][2] * (dp[8][2] - dl);
        dp[8][1] = dp[8][3] = 0.f;
        s[9][0] = s[9][1] = s[9][2] = s[9][3] = 0.f;
        dp[9][0] = dp[9][1] = dp[9][2] = dp[9][3] = 0.f;
      }
      float ov[DT][4], ok[DT][4];
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        ov[dt][0] = ov[dt][1] = ov[dt][2] = ov[dt][3] = 0.f;
        ok[dt][0] = ok[dt][1] = ok[dt][2] = ok[dt][3] = 0.f;
      }
#pragma unroll
      for (int kk = 0; kk < 5; ++kk) {
        const uint32_t p0 = pack_bf16(s[2 * kk][0], s[2 * kk][1]), p1 = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        const uint32_t p2 = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]), p3 = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        const uint32_t e0 = pack_bf16(dp[2 * kk][0], dp[2 * kk][1]), e1 = pack_bf16(dp[2 * kk][2], dp[2 * kk][3]);
        const uint32_t e2 = pack_bf16(dp[2 * kk + 1][0], dp[2 * kk + 1][1]), e3 = pack_bf16(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
        const int qrow = min(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          uint32_t b0, b1;
          ldsm_x2_t(au_addr(sdo, qrow, hc + dt * 16), b0, b1);              // dO rows, transposed
          mma_bf16(ov[dt], p0, p1, p2, p3, b0, b1);
          ldsm_x2_t(au_addr(sq, qrow, hc + dt * 16), b0, b1);               // Q rows, transposed
          mma_bf16(ok[dt], e0, e1, e2, e3, b0, b1);
        }
      }
      __syncwarp();
      const int row0 = k0 + g, row1 = k0 + g + 8;
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const int colb = hc + (dt * 8 + 2 * t) * 2;
        if (row0 < AT_S) {
          st_shared_u32(au_addr(sk, row0, colb), pack_bf16(ok[dt][0] * scale, ok[dt][1] * scale));
          st_shared_u32(au_addr(sv, row0, colb), pack_bf16(ov[dt][0], ov[dt][1]));
        }
        if (row1 < AT_S) {
          st_shared_u32(au_addr(sk, row1, colb), pack_bf16(ok[dt][2] * scale, ok[dt][3] * scale));
          st_shared_u32(au_addr(sv, row1, colb), pack_bf16(ov[dt][2], ov[dt][3]));
        }
      }
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        au_store_box(&tmDqkv, sdq + j * AU_TILE, c0 + 64 * j, row_g);                   // dQ
        au_store_box(&tmDqkv, sk + j * AU_TILE, AT_A + c0 + 64 * j, row_g);             // dK
        au_store_box(&tmDqkv, sv + j * AU_TILE, 2 * AT_A + c0 + 64 * j, row_g);         // dV
      }
      bulk_commit();
    }
    if (db_q) {
      // q / k / v bias gradients: column sums of the unit's dQ | dK | dV images, kept in registers across units
#pragma unroll
      for (int i = 0; i < Cfg::NC; ++i) {
        const int c = (int)threadIdx.x + 128 * i;
        if (c < 3 * UC) {
          const int m = c / UC, col = c - m * UC;
          const uint32_t base = m == 0 ? sdq : (m == 1 ? sk : sv);
          float a = 0.f;
#pragma unroll 5
          for (int r = 0; r < AT_S; ++r)
            a += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(smem + (au_addr(base, r, col * 2) - sq)));
          bs[i] += a;
        }
      }
    }
    __syncthreads();         // every warp is done with the images before the next unit's loads overwrite them
  }
  if (db_q && (int)blockIdx.x < units) {
#pragma unroll
    for (int i = 0; i < Cfg::NC; ++i) {
      const int c = (int)threadIdx.x + 128 * i;
      if (c < 3 * UC) {
        const int m = c / UC, col = c - m * UC;
        atomicAdd((m == 0 ? db_q : (m == 1 ? db_k : db_v)) + c0 + col, bs[i]);
      }
    }
  }
  if (threadIdx.x == 0) bulk_wait0();
}

int make_tmap_2d(CUtensorMap* out, const void* ptr, int elem_bytes, long long rows, long long cols, long long ld_elems,
                 int box_rows, int box_cols, int swizzle_bytes);

template <int D>
static int launch_attn_bwd_unit(const void* dctx, const void* qkv, void* dqkv, float* db_q, float* db_k, float* db_v, int B,
                                cudaStream_t st) {
  using Cfg = AuCfg<D>;
  auto kern = attn_bwd_unit_kernel<D>;
  V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
  CUtensorMap tq, td, to;
  int rc = make_tmap_2d(&tq, qkv, 2, (long long)B * AT_S, 3 * AT_A, 3 * AT_A, AT_S, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&td, dctx, 2, (long long)B * AT_S, AT_A, AT_A, AT_S, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&to, dqkv, 2, (long long)B * AT_S, 3 * AT_A, 3 * AT_A, AT_S, 64, 128);
  if (rc != VIT3D_OK) return rc;
  const int groups = AT_A / Cfg::UC;                // head groups (units) per volume
  const int units = B * groups;
  int grid = sm_count() * Cfg::CTAS;
  if (grid > units) grid = units;
  grid -= grid % groups;
  const float scale = 1.0f / sqrtf((float)D);
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(128), (size_t)Cfg::SMEM, st, tq, td, to, db_q, db_k, db_v, units, groups, scale,
                     1.4426950408889634f * scale));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}


// ---------------------------------------------------------------------------- forward, unit kernel (bf16)
// The forward in the backward's unit form: a CTA of 4 warps takes (volume, 4 heads), q | k | v column blocks arrive as
// 65-row x 128-byte TMA boxes (SWIZZLE_128B), one warp owns one head, the context tile overwrites the Q tile and
// leaves as boxes.  18-55 KB of shared memory: 4 CTAs per SM at D <= 32.  Compute body = attn_fwd_tc_kernel's.
template <int D> struct AvCfg {
  static constexpr int UC = 4 * D;                    // bf16 columns per unit row and matrix (4 heads)
  static constexpr int NB = UC / 64;
  static constexpr int MAT = NB * AU_TILE;
  static constexpr int SMEM = 3 * MAT + 64 + 1024;
  static constexpr int CTAS = D == 64 ? 2 : 4;
};

template <int D, int VIS>
__global__ void __launch_bounds__(128, AvCfg<D>::CTAS)
attn_fwd_unit_kernel(const __grid_constant__ CUtensorMap tmQkv, const __grid_constant__ CUtensorMap tmCtx,
                     float* __restrict__ probs, int units, int groups, float scale_log2e, int pld) {
  using Cfg = AvCfg<D>;
  constexpr int HEADS = AT_A / D;
  constexpr int KSTEPS = D / 16;
  constexpr int NT = 10;
  constexpr int DT = D / 8;
  constexpr int MAT = Cfg::MAT, NB = Cfg::NB, UC = Cfg::UC;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sq = smem_u32(smem), sk = sq + MAT, sv = sk + MAT;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 3 * MAT);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQkv);
    prefetch_tmap(&tmCtx);
    mbar_init(full, 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();
  pdl_wait();
  const int hq = blockIdx.x % groups;
  const int c0 = hq * UC;
  const int hc = warp * D * 2;
  const int h = hq * 4 + warp;

  int it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int b = u / groups;
    const int row_g = b * AT_S;
    if (threadIdx.x == 0) {
      bulk_wait_read0();
      mbar_arrive_expect_tx(full, 3 * NB * AT_S * 128);
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        tma_load_2d(smem + j * AU_TILE, &tmQkv, full, c0 + 64 * j, row_g);
        tma_load_2d(smem + MAT + j * AU_TILE, &tmQkv, full, AT_A + c0 + 64 * j, row_g);
        tma_load_2d(smem + 2 * MAT + j * AU_TILE, &tmQkv, full, 2 * AT_A + c0 + 64 * j, row_g);
      }
    }
    mbar_wait(full, it & 1);

#pragma unroll 1
    for (int rt = 0; rt < 5; ++rt) {
      const int r0 = rt * 16;
      uint32_t qa[KSTEPS][4];
      {
        const int row = min(r0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks)
          ldsm_x4(au_addr(sq, row, hc + ks * 32 + (lane >> 4) * 16), qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
      }
      float s[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        if (nt < 9) {
          const int key = min(nt * 8 + (lane & 7), AT_S - 1);
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            uint32_t b0, b1;
            ldsm_x2(au_addr(sk, key, hc + ks * 32 + ((lane >> 3) & 1) * 16), b0, b1);
            mma_bf16(s[nt], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b0, b1);
          }
        }
      }
      const bool tail = t == 0;
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
      }
      if (tail) { mx0 = fmaxf(mx0, s[8][0]); mx1 = fmaxf(mx1, s[8][2]); }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float m0 = mx0 * scale_log2e, m1 = mx1 * scale_log2e;
      float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = ex2_approx(fmaf(s[nt][0], scale_log2e, -m0));
        s[nt][1] = ex2_approx(fmaf(s[nt][1], scale_log2e, -m0));
        s[nt][2] = ex2_approx(fmaf(s[nt][2], scale_log2e, -m1));
        s[nt][3] = ex2_approx(fmaf(s[nt][3], scale_log2e, -m1));
        sum0 += s[nt][0] + s[nt][1];
        sum1 += s[nt][2] + s[nt][3];
      }
      s[8][0] = tail ? ex2_approx(fmaf(s[8][0], scale_log2e, -m0)) : 0.f;
      s[8][2] = tail ? ex2_approx(fmaf(s[8][2], scale_log2e, -m1)) : 0.f;
      s[8][1] = s[8][3] = 0.f;
      sum0 += s[8][0];
      sum1 += s[8][2];
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
      const float inv0 = 1.f / sum0, inv1 = 1.f / sum1;
      const int row0 = r0 + g, row1 = r0 + g + 8;
      const bool fullt = rt < 4;
      const bool w0 = fullt || g == 0, w1 = fullt;
      if constexpr (VIS != 0) {
#pragma unroll
        for (int nt = 0; nt < 9; ++nt) {
          s[nt][0] *= inv0; s[nt][1] *= inv0;
          s[nt][2] *= inv1; s[nt][3] *= inv1;
        }
      }
      if constexpr (VIS == 2) {
        float* p0 = probs + ((size_t)(b * HEADS + h) * AT_S + row0) * pld + 2 * t;
        float* p1 = p0 + 8 * (size_t)pld;
#pragma unroll
        for (int nt = 0; nt < 9; ++nt) {
          st_global_f2_if(w0, p0 + nt * 8, s[nt][0], s[nt][1]);
          st_global_f2_if(w1, p1 + nt * 8, s[nt][2], s[nt][3]);
        }
      }
      if constexpr (VIS == 1) {
        const int bh = b * HEADS + h;
        const bool odd = ((bh + row0) & 1) != 0;
        float* p0 = probs + ((size_t)bh * AT_S + row0) * AT_S + 2 * t + (odd ? 1 : 0);
        float* p1 = p0 + 8 * AT_S;
        const int src = (lane & ~3) | ((t + 1) & 3);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const float n0 = __shfl_sync(0xffffffffu, tail ? s[nt + 1][0] : s[nt][0], src);
          const float n1 = __shfl_sync(0xffffffffu, tail ? s[nt + 1][2] : s[nt][2], src);
          const float2 v0 = make_float2(odd ? s[nt][1] : s[nt][0], odd ? n0 : s[nt][1]);
          const float2 v1 = make_float2(odd ? s[nt][3] : s[nt][2], odd ? n1 : s[nt][3]);
          st_global_f2_if(w0, p0 + nt * 8, v0.x, v0.y);
          st_global_f2_if(w1, p1 + nt * 8, v1.x, v1.y);
        }
        const int off = odd ? -1 : 64;
        st_global_f1_if(tail && w0, p0 + off, odd ? s[0][0] : s[8][0]);
        st_global_f1_if(tail && w1, p1 + off, odd ? s[0][2] : s[8][2]);
      }
      float o[DT][4];
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 5; ++kk) {
        const uint32_t a0 = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
        const uint32_t a1 = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        const uint32_t a2 = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        const uint32_t a3 = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        const int key = min(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          uint32_t b0, b1;
          ldsm_x2_t(au_addr(sv, key, hc + dt * 16), b0, b1);
          mma_bf16(o[dt], a0, a1, a2, a3, b0, b1);
        }
      }
      __syncwarp();
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const int colb = hc + (dt * 8 + 2 * t) * 2;
        const float c0f = VIS != 0 ? 1.f : inv0, c1f = VIS != 0 ? 1.f : inv1;
        if (w0) st_shared_u32(au_addr(sq, row0, colb), pack_bf16(o[dt][0] * c0f, o[dt][1] * c0f));
        if (w1) st_shared_u32(au_addr(sq, row1, colb), pack_bf16(o[dt][2] * c1f, o[dt][3] * c1f));
      }
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
      for (int j = 0; j < NB; ++j) au_store_box(&tmCtx, sq + j * AU_TILE, c0 + 64 * j, row_g);
      bulk_commit();
    }
  }
  if (threadIdx.x == 0) bulk_wait0();
}

template <int D, int VIS>
static int launch_attn_unit_v(const void* qkv, void* ctx, float* probs, int pld, int B, cudaStream_t st) {
  using Cfg = AvCfg<D>;
  auto kern = attn_fwd_unit_kernel<D, VIS>;
  V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
  CUtensorMap tq, tc;
  int rc = make_tmap_2d(&tq, qkv, 2, (long long)B * AT_S, 3 * AT_A, 3 * AT_A, AT_S, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&tc, ctx, 2, (long long)B * AT_S, AT_A, AT_A, AT_S, 64, 128);
  if (rc != VIT3D_OK) return rc;
  const int groups = AT_A / Cfg::UC;
  const int units = B * groups;
  int grid = sm_count() * Cfg::CTAS;
  if (grid > units) grid = units;
  grid -= grid % groups;
  const float scale_log2e = 1.4426950408889634f / sqrtf((float)D);
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(128), (size_t)Cfg::SMEM, st, tq, tc, probs, units, groups, scale_log2e, pld));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
template <int D>
static int launch_attn_unit(const void* qkv, void* ctx, float* probs, int pld, int B, cudaStream_t st) {
  if (!probs) return launch_attn_unit_v<D, 0>(qkv, ctx, probs, pld, B, st);
  if (pld == AT_S) return launch_attn_unit_v<D, 1>(qkv, ctx, probs, pld, B, st);
  return launch_attn_unit_v<D, 2>(qkv, ctx, probs, pld, B, st);
}
int tc_attn_fwd_unit(const void* qkv, void* ctx, float* probs, int probs_ld, int B, int D, cudaStream_t st) {
  if (D == 16) return launch_attn_unit<16>(qkv, ctx, probs, probs_ld, B, st);
  if (D == 32) return launch_attn_unit<32>(qkv, ctx, probs, probs_ld, B, st);
  return launch_attn_unit<64>(qkv, ctx, probs, probs_ld, B, st);
}

// ---------------------------------------------------------------------------- forward, TF32 mode (fp32 activations)
// The 1e-3 accuracy mode keeps q | k | v, the probabilities and the context in fp32; its attention ran on a generic
// SIMT kernel (one block per head, 4.5 ms per layer at batch 1024 - 79 % of the TF32-mode step).  Same unit design as
// the backward kernel above: a CTA of 4 warps takes (volume, 4 heads), the unit's q | k | v column blocks arrive as
// 65-row x 128-byte boxes (32 floats = one head of D = 32), one warp owns one head.  Products on mma.sync.m16n8k8
// (tf32 in, fp32 accumulate): Q K^T as a 3xTF32 split product (fp32-grade scores), P V with P and V rounded to tf32
// (round to nearest, cvt.rna - the tensor core would truncate).  softmax in fp32, probabilities (packed or padded
// rows) leave from the accumulator registers, the context tile overwrites the Q tile and leaves as TMA boxes.
template <int D> struct AfCfg {
  static constexpr int UC = 4 * D;                    // floats per unit row and matrix (4 heads)
  static constexpr int NB = UC / 32;                  // 128-byte column blocks per matrix
  static constexpr int MAT = NB * AU_TILE;
  static constexpr int SMEM = 3 * MAT + 64 + 1024;
  static constexpr int CTAS = D == 16 ? 4 : (D == 32 ? 2 : 1);
};
__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ uint32_t ld_shared_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// VIS: 0 = no probabilities, 1 = packed rows of 65 floats, 2 = rows padded to `pld` floats (pld % 8 == 0)
template <int D, int VIS>
__global__ void __launch_bounds__(128, AfCfg<D>::CTAS)
attn_fwd_tf32_kernel(const __grid_constant__ CUtensorMap tmQkv, const __grid_constant__ CUtensorMap tmCtx,
                     float* __restrict__ probs, int units, int groups, float scale_log2e, int pld, int round_out) {
  using Cfg = AfCfg<D>;
  constexpr int HEADS = AT_A / D;
  constexpr int KSTEPS = D / 8;
  constexpr int NT = 9;
  constexpr int DT = D / 8;
  constexpr int MAT = Cfg::MAT, NB = Cfg::NB, UC = Cfg::UC;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sq = smem_u32(smem), sk = sq + MAT, sv = sk + MAT;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 3 * MAT);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQkv);
    prefetch_tmap(&tmCtx);
    mbar_init(full, 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();
  pdl_wait();
  const int hq = blockIdx.x % groups;      // the grid is a multiple of `groups`: a CTA keeps its head group
  const int c0 = hq * UC;                  // first float column of the unit inside q (and k, v, ctx)
  const int hc = warp * D * 4;             // byte column of this warp's head inside the unit
  const int h = hq * 4 + warp;             // head index

  int it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int b = u / groups;
    const int row_g = b * AT_S;
    if (threadIdx.x == 0) {
      bulk_wait_read0();                   // the previous unit's context boxes have left shared memory
      mbar_arrive_expect_tx(full, 3 * NB * AT_S * 128);
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        tma_load_2d(smem + j * AU_TILE, &tmQkv, full, c0 + 32 * j, row_g);
        tma_load_2d(smem + MAT + j * AU_TILE, &tmQkv, full, AT_A + c0 + 32 * j, row_g);
        tma_load_2d(smem + 2 * MAT + j * AU_TILE, &tmQkv, full, 2 * AT_A + c0 + 32 * j, row_g);
      }
    }
    mbar_wait(full, it & 1);
    // round V to tf32 in place, once (every V element feeds five query tiles); Q and K stay fp32 - their products are
    // split below
    for (int i = threadIdx.x; i < NB * AT_S * 8; i += 128) {
      const int tile = 2 * NB + i / (AT_S * 8), rem = i % (AT_S * 8);
      float4* p4 = reinterpret_cast<float4*>(smem + tile * AU_TILE + rem * 16);
      float4 v = *p4;
      v.x = __uint_as_float(to_tf32(v.x)); v.y = __uint_as_float(to_tf32(v.y));
      v.z = __uint_as_float(to_tf32(v.z)); v.w = __uint_as_float(to_tf32(v.w));
      *p4 = v;
    }
    __syncthreads();

#pragma unroll 1
    for (int rt = 0; rt < 5; ++rt) {
      const int r0 = rt * 16;
      // S = Q K^T as a 3xTF32 product (x = hi + lo, hi = tf32(x), lo = tf32(x - hi); q_lo k_hi + q_hi k_lo + q_hi k_hi):
      // the scores go through exp, where a plain tf32 product (2^-11 relative on both operands) costs ~1e-2 relative
      // on the probabilities of sharp rows.  The arithmetic is tiny next to the memory traffic.
      uint32_t qh[KSTEPS][4], ql[KSTEPS][4];
      {
        const int row = min(r0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          uint32_t f[4];
          ldsm_x4(au_addr(sq, row, hc + ks * 32 + (lane >> 4) * 16), f[0], f[1], f[2], f[3]);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            qh[ks][i] = to_tf32(__uint_as_float(f[i]));
            ql[ks][i] = to_tf32(__uint_as_float(f[i]) - __uint_as_float(qh[ks][i]));
          }
        }
      }
      float s[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        const int key = min(nt * 8 + (lane & 7), AT_S - 1);
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          uint32_t f0, f1;
          ldsm_x2(au_addr(sk, key, hc + ks * 32 + ((lane >> 3) & 1) * 16), f0, f1);
          const uint32_t h0 = to_tf32(__uint_as_float(f0)), h1 = to_tf32(__uint_as_float(f1));
          const uint32_t l0 = to_tf32(__uint_as_float(f0) - __uint_as_float(h0)), l1 = to_tf32(__uint_as_float(f1) - __uint_as_float(h1));
          mma_tf32(s[nt], ql[ks][0], ql[ks][1], ql[ks][2], ql[ks][3], h0, h1);
          mma_tf32(s[nt], qh[ks][0], qh[ks][1], qh[ks][2], qh[ks][3], l0, l1);
          mma_tf32(s[nt], qh[ks][0], qh[ks][1], qh[ks][2], qh[ks][3], h0, h1);
        }
      }
      // softmax over the 65 valid keys: n-tiles 0..7 are valid in every lane, key 64 is element [0] / [2] of n-tile 8
      // in the lanes with t == 0
      const bool tail = t == 0;
      float mx0 = tail ? s[8][0] : -INFINITY, mx1 = tail ? s[8][2] : -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float m0 = mx0 * scale_log2e, m1 = mx1 * scale_log2e;
      float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = exp2f(fmaf(s[nt][0], scale_log2e, -m0));
        s[nt][1] = exp2f(fmaf(s[nt][1], scale_log2e, -m0));
        s[nt][2] = exp2f(fmaf(s[nt][2], scale_log2e, -m1));
        s[nt][3] = exp2f(fmaf(s[nt][3], scale_log2e, -m1));
        sum0 += s[nt][0] + s[nt][1];
        sum1 += s[nt][2] + s[nt][3];
      }
      s[8][0] = tail ? exp2f(fmaf(s[8][0], scale_log2e, -m0)) : 0.f;
      s[8][2] = tail ? exp2f(fmaf(s[8][2], scale_log2e, -m1)) : 0.f;
      s[8][1] = s[8][3] = 0.f;
      sum0 += s[8][0];
      sum1 += s[8][2];
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
      sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
      sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
      const float inv0 = 1.f / sum0, inv1 = 1.f / sum1;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        s[nt][0] *= inv0; s[nt][1] *= inv0;
        s[nt][2] *= inv1; s[nt][3] *= inv1;
      }
      const int row0 = r0 + g, row1 = r0 + g + 8;
      const bool fullt = rt < 4;
      const bool w0 = fullt || g == 0, w1 = fullt;
      if constexpr (VIS == 2) {
        float* p0 = probs + ((size_t)(b * HEADS + h) * AT_S + row0) * pld + 2 * t;
        float* p1 = p0 + 8 * (size_t)pld;
#pragma unroll
        for (int nt = 0; nt < 9; ++nt) {
          st_global_f2_if(w0, p0 + nt * 8, s[nt][0], s[nt][1]);
          st_global_f2_if(w1, p1 + nt * 8, s[nt][2], s[nt][3]);
        }
      }
      if constexpr (VIS == 1) {
        // packed rows of 65 floats start at alternating 8-byte phases: see attn_fwd_tc_kernel
        const int bh = b * HEADS + h;
        const bool odd = ((bh + row0) & 1) != 0;
        float* p0 = probs + ((size_t)bh * AT_S + row0) * AT_S + 2 * t + (odd ? 1 : 0);
        float* p1 = p0 + 8 * AT_S;
        const int src = (lane & ~3) | ((t + 1) & 3);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const float n0 = __shfl_sync(0xffffffffu, tail ? s[nt + 1][0] : s[nt][0], src);
          const float n1 = __shfl_sync(0xffffffffu, tail ? s[nt + 1][2] : s[nt][2], src);
          const float2 v0 = make_float2(odd ? s[nt][1] : s[nt][0], odd ? n0 : s[nt][1]);
          const float2 v1 = make_float2(odd ? s[nt][3] : s[nt][2], odd ? n1 : s[nt][3]);
          st_global_f2_if(w0, p0 + nt * 8, v0.x, v0.y);
          st_global_f2_if(w1, p1 + nt * 8, v1.x, v1.y);
        }
        const int off = odd ? -1 : 64;
        st_global_f1_if(tail && w0, p0 + off, odd ? s[0][0] : s[8][0]);
        st_global_f1_if(tail && w1, p1 + off, odd ? s[0][2] : s[8][2]);
      }
      // O = P V.  An accumulator tile holds columns (2t, 2t+1) where the A fragment wants (t, t+4): the reduction runs
      // over keys in the order (2t | 2t+1) - k-slot t is key 8 kk + 2t, slot t+4 is key 8 kk + 2t + 1 - and V is read
      // in the same order
      float o[DT][4];
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < NT; ++kk) {
        const uint32_t a0 = to_tf32(s[kk][0]), a1 = to_tf32(s[kk][2]), a2 = to_tf32(s[kk][1]), a3 = to_tf32(s[kk][3]);
        const int key0 = min(kk * 8 + 2 * t, AT_S - 1), key1 = min(kk * 8 + 2 * t + 1, AT_S - 1);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          const uint32_t b0 = ld_shared_u32(au_addr(sv, key0, hc + (dt * 8 + g) * 4));
          const uint32_t b1 = ld_shared_u32(au_addr(sv, key1, hc + (dt * 8 + g) * 4));
          mma_tf32(o[dt], a0, a1, a2, a3, b0, b1);
        }
      }
      // the context tile overwrites the Q tile it came from (only this warp reads that head's columns)
      __syncwarp();
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const int colb = hc + (dt * 8 + 2 * t) * 4;
        float x0 = o[dt][0], x1 = o[dt][1], x2 = o[dt][2], x3 = o[dt][3];
        if (round_out) {
          x0 = __uint_as_float(to_tf32(x0)); x1 = __uint_as_float(to_tf32(x1));
          x2 = __uint_as_float(to_tf32(x2)); x3 = __uint_as_float(to_tf32(x3));
        }
        if (w0) { st_shared_u32(au_addr(sq, row0, colb), __float_as_uint(x0)); st_shared_u32(au_addr(sq, row0, colb + 4), __float_as_uint(x1)); }
        if (w1) { st_shared_u32(au_addr(sq, row1, colb), __float_as_uint(x2)); st_shared_u32(au_addr(sq, row1, colb + 4), __float_as_uint(x3)); }
      }
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
      for (int j = 0; j < NB; ++j) au_store_box(&tmCtx, sq + j * AU_TILE, c0 + 32 * j, row_g);
      bulk_commit();
    }
  }
  if (threadIdx.x == 0) bulk_wait0();
}

template <int D, int VIS>
static int launch_attn_tf32_v(const CUtensorMap& tq, const CUtensorMap& tc, float* probs, int pld, int B, int round_out,
                              cudaStream_t st) {
  using Cfg = AfCfg<D>;
  auto kern = attn_fwd_tf32_kernel<D, VIS>;
  V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
  const int groups = AT_A / Cfg::UC;
  const int units = B * groups;
  int grid = sm_count() * Cfg::CTAS;
  if (grid > units) grid = units;
  grid -= grid % groups;
  const float scale_log2e = 1.4426950408889634f / sqrtf((float)D);
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(128), (size_t)Cfg::SMEM, st, tq, tc, probs, units, groups, scale_log2e, pld, round_out));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
template <int D>
static int launch_attn_tf32(const CUtensorMap& tq, const CUtensorMap& tc, float* probs, int pld, int B, int round_out,
                            cudaStream_t st) {
  if (!probs) return launch_attn_tf32_v<D, 0>(tq, tc, probs, pld, B, round_out, st);
  if (pld == AT_S) return launch_attn_tf32_v<D, 1>(tq, tc, probs, pld, B, round_out, st);
  return launch_attn_tf32_v<D, 2>(tq, tc, probs, pld, B, round_out, st);
}

// fp32 q | k | v [B*65, 768] -> fp32 context [B*65, 256] (+ fp32 probabilities, rows of probs_ld floats)
int tc_attn_fwd_tf32(const float* qkv, float* ctx, float* probs, int probs_ld, int B, int S, int heads, int D, int round_out,
                     cudaStream_t st) {
  if (!tc_attn_supported(S, heads, D)) V3_UNSUPPORTED("tf32 attention: unsupported shape S=%d heads=%d D=%d", S, heads, D);
  if (B <= 0) return VIT3D_OK;
  if (probs && probs_ld != S && (probs_ld % 8 || probs_ld < S + 7 || (reinterpret_cast<uintptr_t>(probs) & 31))) {
    set_error("tf32 attention: padded probability rows are a multiple of 8 floats >= 72 in a 32-byte aligned buffer");
    return VIT3D_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(ctx) & 15) || (reinterpret_cast<uintptr_t>(probs) & 7)) {
    set_error("tf32 attention: qkv/ctx must be 16-byte aligned, probs 8-byte aligned");
    return VIT3D_ERR_INVALID;
  }
  CUtensorMap tq, tc;
  int rc = make_tmap_2d(&tq, qkv, 4, (long long)B * AT_S, 3 * AT_A, 3 * AT_A, AT_S, 32, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&tc, ctx, 4, (long long)B * AT_S, AT_A, AT_A, AT_S, 32, 128);
  if (rc != VIT3D_OK) return rc;
  if (D == 16) return launch_attn_tf32<16>(tq, tc, probs, probs_ld, B, round_out, st);
  if (D == 32) return launch_attn_tf32<32>(tq, tc, probs, probs_ld, B, round_out, st);
  return launch_attn_tf32<64>(tq, tc, probs, probs_ld, B, round_out, st);
}

template <int D>
static int launch_attn_bwd(const void* dctx, const void* qkv, void* dqkv, float* db_q, float* db_k, float* db_v, int B,
                           cudaStream_t st) {
  auto kern = attn_bwd_tc_kernel<D>;
  V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, AB_SMEM));
  const int grid = B < sm_count() ? B : sm_count();
  const float scale = 1.0f / sqrtf((float)D);
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(AT_THREADS), (size_t)AB_SMEM, st, reinterpret_cast<const __nv_bfloat16*>(dctx),
                     reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(dqkv), db_q, db_k, db_v, B,
                     scale, 1.4426950408889634f * scale));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

int tc_attn_bwd(const void* dctx, const void* qkv, void* dqkv, float* db_q, float* db_k, float* db_v, int B, int S,
                int heads, int D, cudaStream_t st) {
  if (!tc_attn_supported(S, heads, D)) V3_UNSUPPORTED("tc attention bwd: unsupported shape S=%d heads=%d D=%d", S, heads, D);
  if (B <= 0) return VIT3D_OK;
  if ((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(dctx) & 15) ||
      (reinterpret_cast<uintptr_t>(dqkv) & 15)) {
    set_error("tc attention bwd: buffers must be 16-byte aligned");
    return VIT3D_ERR_INVALID;
  }
  if ((db_q != nullptr) != (db_k != nullptr) || (db_q != nullptr) != (db_v != nullptr)) {
    set_error("tc attention bwd: pass all three bias-gradient buffers or none");
    return VIT3D_ERR_INVALID;
  }
  if (tuning(VIT3D_TUNE_ATTN_BWD) != 0) {
    if (D == 16) return launch_attn_bwd_unit<16>(dctx, qkv, dqkv, db_q, db_k, db_v, B, st);
    if (D == 32) return launch_attn_bwd_unit<32>(dctx, qkv, dqkv, db_q, db_k, db_v, B, st);
    return launch_attn_bwd_unit<64>(dctx, qkv, dqkv, db_q, db_k, db_v, B, st);
  }
  if (D == 16) return launch_attn_bwd<16>(dctx, qkv, dqkv, db_q, db_k, db_v, B, st);
  if (D == 32) return launch_attn_bwd<32>(dctx, qkv, dqkv, db_q, db_k, db_v, B, st);
  return launch_attn_bwd<64>(dctx, qkv, dqkv, db_q, db_k, db_v, B, st);
}

}  // namespace vit3d
