// tcgen05 GEMM with an fp32 "residual stream" epilogue (sm_100a):
//
//     y[M,N]  = A[M,K] * B[N,K]^T + bias + residual          (fp32, y may alias residual)
//     yn[M,N] = LayerNorm(y) * gamma + beta                   (bf16, optional, N == 256)
//
// the out-projection and fc2 of a Block (modeling.py:97,122 with the `x + h` adds of :191,:196) and - fused -
// the LayerNorm that consumes the sum (ffn_norm / the next Block's attention_norm, :189,:194).  These
// products write and read fp32 rows, so they are bound by HBM, not by the tensor pipe: what matters is
// that every global byte moves through the TMA unit with many transfers in flight, and that no thread
// waits on a global load.
//
//   * warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (128 x 256 tile, accumulator double
//     buffered in TMEM), 16 epilogue warps; operands stream through a 3-stage ring (48 KB per stage).
//   * every epilogue warp owns 32 rows x 64 columns of the tile = two [32 x 32] fp32 panels (128-byte
//     rows, 128B swizzle) and one 4 KB shared-memory panel buffer.  The RESIDUAL panel is fetched into
//     that buffer by a bulk tensor load that is issued as soon as the buffer is free - for the first panel
//     of a tile that is while the MMAs of the tile are still running - the thread adds its accumulator row
//     (tcgen05.ld 32x32b: one row per thread) and the bias in place, and the same buffer leaves by a bulk
//     tensor store.  Rows >= M are clipped / zero-filled by the TMA unit: no predicates.
//   * fused LayerNorm: the finished row values are parked back in the TMEM columns they came from
//     (tcgen05.st), the four column slices of a row exchange (sum, sum of squares) through their panel
//     buffers, then every thread re-reads its slice from TMEM, normalises it and the bf16 panel leaves by
//     one more bulk tensor store.  No register array of row values, no second pass over HBM.
#include "ptx.cuh"
#include "tc.cuh"
#include "tc_epilogue.cuh"

namespace vit3d {

using namespace ptx;

constexpr int RS_BM = 128, RS_BN = 256, RS_STAGES = 3;
constexpr int RS_A_BYTES = RS_BM * 128, RS_B_BYTES = RS_BN * 128, RS_STAGE_BYTES = RS_A_BYTES + RS_B_BYTES;
constexpr int RS_OPER_BYTES = RS_STAGES * RS_STAGE_BYTES;               // 147,456
constexpr int RS_EPI_WARPS = 16, RS_THREADS = 64 + 32 * RS_EPI_WARPS;
constexpr int RS_PANEL_BYTES = 4096;                                    // 32 rows x 32 fp32
constexpr int RS_PARAM_BYTES = 3 * RS_BN * 4;                           // bias, gamma, beta of the n-tile
constexpr int RS_SMEM_BYTES = RS_OPER_BYTES + RS_EPI_WARPS * RS_PANEL_BYTES + RS_PARAM_BYTES + 512;

struct ResEpilogue {
  const float* bias = nullptr;     // [N]
  const float* gamma = nullptr;    // [N]  (LN)
  const float* beta = nullptr;     // [N]  (LN)
  float* mean = nullptr;           // [M] optional (LN)
  float* rstd = nullptr;           // [M] optional (LN)
  float eps = 1e-6f;
  const uint32_t* drop_bits = nullptr;   // keep bits over [M,N] (MODE bit 3): (A B^T + bias) * keep * drop_scale + residual
  float drop_scale = 1.f;
};

// MODE bit 0: bias, bit 1: residual, bit 2: fused LayerNorm output, bit 3: Dropout before the residual add (training)
// CL = 2: clusters of two CTAs that stay independent (own row tile, own tensor core, own barriers) except for the B
// operand: the [256 x 64] weight k-block is fetched ONCE per cluster - each CTA loads half of its rows and multicasts
// them into both CTAs' ring slots.  A streamed 128 x 256 tile needs 48 KB of operands per 512 MMA cycles (96 B/clk,
// above what the L2 delivers to one SM); sharing B makes it 32 KB.  Needs tiles_n == 1 and an even tile count.
template <int MODE, int CL = 1>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(RS_THREADS, 1)
tc_gemm_res_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmRes,
                   const __grid_constant__ CUtensorMap tmLn, ResEpilogue ep, int M, int N, int K, int tiles_m,
                   int tiles_n) {
  constexpr bool BIAS = (MODE & 1) != 0, RES = (MODE & 2) != 0, LN = (MODE & 4) != 0, DROP = (MODE & 8) != 0;
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023u) __trap();
  uint8_t* panels = smem + RS_OPER_BYTES;
  float* param = reinterpret_cast<float*>(panels + RS_EPI_WARPS * RS_PANEL_BYTES);   // [bias | gamma | beta]
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(param) + RS_PARAM_BYTES);
  uint64_t* full_bar = bars;                    // [RS_STAGES]
  uint64_t* empty_bar = bars + 4;               // [RS_STAGES]
  uint64_t* tmem_full = bars + 8;               // [2]
  uint64_t* tmem_empty = bars + 10;             // [2]
  uint64_t* res_bar = bars + 12;                // [RS_EPI_WARPS] residual panel landed
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 12 + RS_EPI_WARPS);

  // warp index through a shuffle: warp-uniform for the compiler, so the role branches are uniform control flow
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int nkb = (K + 63) / 64;
  const int total = tiles_m * tiles_n;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmY);
    for (int s = 0; s < RS_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], CL);      // the commit of every CTA of the cluster frees the slot
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], RS_EPI_WARPS);
    }
    for (int w = 0; w < RS_EPI_WARPS; ++w) mbar_init(&res_bar[w], 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<2 * RS_BN>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t rank = CL > 1 ? cluster_ctarank() : 0u;
  if constexpr (CL > 1) cluster_sync_all();       // every CTA's barriers exist before any multicast signal
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ===================================================== TMA producer (operands)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int tn = w % tiles_n, tm = w / tiles_n;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * RS_STAGE_BYTES;
          mbar_arrive_expect_tx(&full_bar[stage], RS_STAGE_BYTES);
          tma_load_2d(sa, &tmA, &full_bar[stage], kb * 64, tm * RS_BM);
          if constexpr (CL > 1)     // this CTA's share of the B rows, into the same slot of every CTA of the cluster
            tma_load_2d_mcast(sa + RS_A_BYTES + (int)rank * (RS_B_BYTES / CL), &tmB, &full_bar[stage], kb * 64,
                              tn * RS_BN + (int)rank * (RS_BN / CL), (uint16_t)((1u << CL) - 1u));
          else
            tma_load_2d(sa + RS_A_BYTES, &tmB, &full_bar[stage], kb * 64, tn * RS_BN);
          if (++stage == RS_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer: ONE thread, elected once, walks the whole
    // schedule (tools/mma_pipe_bench.cu, k_tc_mlp2.cu: an election per k-block costs ~60 cycles per MMA)
    if (elect_one()) {
      const uint32_t idesc = make_idesc(UMMA_FMT_BF16, RS_BM, RS_BN, 0, 0);
      const uint64_t ring_desc = make_smem_desc(smem_u32(smem), 16, 1024, UMMA_LAYOUT_SW128);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
        const int buf = it & 1;
        mbar_wait(&tmem_empty[buf], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * RS_BN;
        // no tcgen05 fence after an operand k-block has landed (the mbarrier's complete_tx orders the TMA writes)
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          const uint64_t ad = ring_desc + (uint64_t)((stage * RS_STAGE_BYTES) >> 4);
          const uint64_t bd = ad + (uint64_t)(RS_A_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma<false>(d_tmem, ad + 2 * k, bd + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          if constexpr (CL > 1) umma_commit_mcast(&empty_bar[stage], (uint16_t)((1u << CL) - 1u));
          else umma_commit(&empty_bar[stage]);
          if (++stage == RS_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[buf]);
      }
    }
    __syncwarp();
  } else {
    // ===================================================== epilogue warps
    const int ew = warp - 2;                // 0..15
    const int q = warp & 3;                 // TMEM lane quarter
    const int part = ew >> 2;               // 64-column slice of the tile
    const int sib0 = (q + 2) & 3;           // epilogue-warp index of the part-0 warp of this quarter (warps 2..5)
    uint8_t* buf_ptr = panels + ew * RS_PANEL_BYTES;
    const uint32_t buf_s = smem_u32(buf_ptr);
    uint64_t* rbar = &res_bar[ew];
    uint32_t rphase = 0;
    const uint32_t my_row = buf_s + lane * 128;
    const int sw7 = lane & 7;
    const uint32_t bias_s = smem_u32(param) + part * 64 * 4;
    int cur_tn = -1;
    int it = 0;
    if constexpr (RES) {
      if ((int)blockIdx.x < total && lane == 0) {
        const int tn = blockIdx.x % tiles_n, tm = blockIdx.x / tiles_n;
        mbar_arrive_expect_tx(rbar, RS_PANEL_BYTES);
        tma_load_2d(buf_ptr, &tmRes, rbar, tn * RS_BN + part * 64, tm * RS_BM + q * 32);
      }
    }
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      const int tn = w % tiles_n, tm = w / tiles_n;
      const int buf = it & 1;
      const int m_base = tm * RS_BM + q * 32, n_base = tn * RS_BN + part * 64;
      if constexpr (BIAS || LN) {
        if (tn != cur_tn) {
          // the n-tile's bias / gamma / beta for all epilogue warps (once per CTA when tiles_n == 1)
          asm volatile("bar.sync 1, %0;" ::"n"(RS_EPI_WARPS * 32) : "memory");
          const int t = (int)threadIdx.x - 64;
          if (t < RS_BN / 4) {
            if constexpr (BIAS)
              reinterpret_cast<float4*>(param)[t] = __ldg(reinterpret_cast<const float4*>(ep.bias + tn * RS_BN) + t);
            if constexpr (LN) {
              reinterpret_cast<float4*>(param + RS_BN)[t] = __ldg(reinterpret_cast<const float4*>(ep.gamma + tn * RS_BN) + t);
              reinterpret_cast<float4*>(param + 2 * RS_BN)[t] = __ldg(reinterpret_cast<const float4*>(ep.beta + tn * RS_BN) + t);
            }
          }
          asm volatile("bar.sync 1, %0;" ::"n"(RS_EPI_WARPS * 32) : "memory");
          cur_tn = tn;
        }
      }
      mbar_wait(&tmem_full[buf], (it >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * RS_BN + part * 64;
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + p * 32, r);
        uint32_t mw = 0u;
        if constexpr (DROP) {
          if (m_base + lane < M) mw = __ldg(ep.drop_bits + (((long long)(m_base + lane) * N + n_base + p * 32) >> 5));
        }
        if constexpr (RES) {
          mbar_wait(rbar, rphase);        // this panel of the residual has landed in the buffer
          rphase ^= 1;
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t a = my_row + ((j ^ sw7) << 4);
          float v0 = __uint_as_float(r[4 * j]), v1 = __uint_as_float(r[4 * j + 1]);
          float v2 = __uint_as_float(r[4 * j + 2]), v3 = __uint_as_float(r[4 * j + 3]);
          if constexpr (BIAS) {
            const uint4 b = ld_shared_v4(bias_s + (p * 32 + 4 * j) * 4);
            v0 += __uint_as_float(b.x); v1 += __uint_as_float(b.y); v2 += __uint_as_float(b.z); v3 += __uint_as_float(b.w);
          }
          if constexpr (DROP) {
            v0 = ((mw >> (4 * j)) & 1u) ? v0 * ep.drop_scale : 0.f;
            v1 = ((mw >> (4 * j + 1)) & 1u) ? v1 * ep.drop_scale : 0.f;
            v2 = ((mw >> (4 * j + 2)) & 1u) ? v2 * ep.drop_scale : 0.f;
            v3 = ((mw >> (4 * j + 3)) & 1u) ? v3 * ep.drop_scale : 0.f;
          }
          if constexpr (RES) {
            const uint4 x = ld_shared_v4(a);
            v0 += __uint_as_float(x.x); v1 += __uint_as_float(x.y); v2 += __uint_as_float(x.z); v3 += __uint_as_float(x.w);
          }
          st_shared_v4(a, __float_as_uint(v0), __float_as_uint(v1), __float_as_uint(v2), __float_as_uint(v3));
          if constexpr (LN) {
            s1 += (v0 + v1) + (v2 + v3);
            s2 = fmaf(v0, v0, fmaf(v1, v1, fmaf(v2, v2, fmaf(v3, v3, s2))));
            r[4 * j] = __float_as_uint(v0); r[4 * j + 1] = __float_as_uint(v1);
            r[4 * j + 2] = __float_as_uint(v2); r[4 * j + 3] = __float_as_uint(v3);
          }
        }
        if constexpr (LN) tmem_st_32x32b_x32(taddr + p * 32, r);      // park the finished values
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmY, buf_s, n_base + p * 32, m_base);
          bulk_store_commit();
          bulk_store_wait_read();           // the store has read the buffer: it is free again
          if constexpr (RES) {
            if (p == 0) {
              mbar_arrive_expect_tx(rbar, RS_PANEL_BYTES);
              tma_load_2d(buf_ptr, &tmRes, rbar, n_base + 32, m_base);
            }
          }
        }
        __syncwarp();
      }
      if constexpr (LN) {
        // (sum, sum of squares) of the four 64-column slices of row (q*32 + lane) meet in the panel buffers
        tmem_st_wait();
        *reinterpret_cast<float2*>(buf_ptr + lane * 8) = make_float2(s1, s2);
        asm volatile("bar.sync %0, %1;" ::"r"(2 + q), "n"(128) : "memory");
        float t1 = 0.f, t2 = 0.f;
#pragma unroll
        for (int pp = 0; pp < 4; ++pp) {
          const float2 s = *reinterpret_cast<const float2*>(panels + (sib0 + 4 * pp) * RS_PANEL_BYTES + lane * 8);
          t1 += s.x; t2 += s.y;
        }
        asm volatile("bar.sync %0, %1;" ::"r"(2 + q), "n"(128) : "memory");   // all four have read: buffers reusable
        const float inv_n = 1.0f / (float)N;
        const float mean = t1 * inv_n;
        const float rstd = rsqrtf(fmaxf(t2 * inv_n - mean * mean, 0.f) + ep.eps);
        if (part == 0 && m_base + lane < M) {
          if (ep.mean) ep.mean[m_base + lane] = mean;
          if (ep.rstd) ep.rstd[m_base + lane] = rstd;
        }
        const float shift = -mean * rstd;
        const uint32_t g_s = smem_u32(param + RS_BN) + part * 64 * 4, b_s = smem_u32(param + 2 * RS_BN) + part * 64 * 4;
        const int sw3 = (lane >> 1) & 3;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(taddr + p * 32, r);
          tmem_ld_wait();
          const uint32_t row = buf_s + p * 2048 + lane * 64;      // bf16 [32 x 32] panel, 64B swizzle
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint32_t wv[4];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint4 g = ld_shared_v4(g_s + (p * 32 + 8 * j + 4 * h) * 4);
              const uint4 b = ld_shared_v4(b_s + (p * 32 + 8 * j + 4 * h) * 4);
              const float y0 = fmaf(fmaf(__uint_as_float(r[8 * j + 4 * h]), rstd, shift), __uint_as_float(g.x), __uint_as_float(b.x));
              const float y1 = fmaf(fmaf(__uint_as_float(r[8 * j + 4 * h + 1]), rstd, shift), __uint_as_float(g.y), __uint_as_float(b.y));
              const float y2 = fmaf(fmaf(__uint_as_float(r[8 * j + 4 * h + 2]), rstd, shift), __uint_as_float(g.z), __uint_as_float(b.z));
              const float y3 = fmaf(fmaf(__uint_as_float(r[8 * j + 4 * h + 3]), rstd, shift), __uint_as_float(g.w), __uint_as_float(b.w));
              wv[2 * h] = pack2_bf16(y0, y1);
              wv[2 * h + 1] = pack2_bf16(y2, y3);
            }
            st_shared_v4(row + ((j ^ sw3) << 4), wv[0], wv[1], wv[2], wv[3]);
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmLn, buf_s, n_base, m_base);
          tma_store_2d(&tmLn, buf_s + 2048, n_base + 32, m_base);
          bulk_store_commit();
          bulk_store_wait_read();
        }
        __syncwarp();
      }
      // accumulator buffer drained
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&tmem_empty[buf]);
        if constexpr (RES) {
          const int wn = w + gridDim.x;       // residual of the next tile's first panel: overlaps its MMAs
          if (wn < total) {
            const int tn2 = wn % tiles_n, tm2 = wn / tiles_n;
            mbar_arrive_expect_tx(rbar, RS_PANEL_BYTES);
            tma_load_2d(buf_ptr, &tmRes, rbar, tn2 * RS_BN + part * 64, tm2 * RS_BM + q * 32);
          }
        }
      }
      __syncwarp();
    }
    if (lane == 0) bulk_store_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CL > 1) cluster_sync_all();       // nobody leaves while a partner may still multicast into this CTA
  if (warp == 1) tmem_dealloc<2 * RS_BN>(tmem_base);
}

bool tc_res_supported(int M, int N, int K, bool ln) {
  if (M <= 0 || N % RS_BN || K % 8 || K < 64) return false;
  return !ln || N == RS_BN;
}

template <int MODE, int CL = 1>
static int launch_res(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ty, const CUtensorMap& tr,
                      const CUtensorMap& tl, const ResEpilogue& ep, int M, int N, int K, cudaStream_t st) {
  auto kern = tc_gemm_res_kernel<MODE, CL>;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V3_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_SMEM_BYTES));
    configured_dev = dev;
  }
  const int tiles_m = ceil_div(M, RS_BM), tiles_n = N / RS_BN;
  const int total = tiles_m * tiles_n;
  const int sms = sm_count();
  int grid = total < sms ? total : sms;
  grid -= grid % CL;       // whole clusters; res_pair_ok() made sure every CTA of a cluster walks equally many tiles
  V3_CUDA(launch_pdl(kern, dim3(grid), dim3(RS_THREADS), (size_t)RS_SMEM_BYTES, st, ta, tb, ty, tr, tl, ep, M, N, K, tiles_m,
                     tiles_n));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// y = A B^T (+ bias) (+ residual) in fp32, optionally yn = LayerNorm(y) in bf16.  A [M,K], B [N,K] bf16.
int tc_gemm_res(const TcLinear& t, cudaStream_t st) {
  const bool ln = t.ln_out != nullptr;
  if (!tc_res_supported(t.M, t.N, t.K, ln)) V3_UNSUPPORTED("tc_gemm_res: unsupported shape M=%d N=%d K=%d", t.M, t.N, t.K);
  if (ln && (!t.ln_gamma || !t.ln_beta)) { set_error("tc_gemm_res: LayerNorm needs gamma and beta"); return VIT3D_ERR_INVALID; }
  CUtensorMap ta, tb, ty, tr, tl;
  int rc = make_tmap_2d(&ta, t.x, 2, t.M, t.K, t.K, RS_BM, 64, 128);
  if (rc != VIT3D_OK) return rc;
  // CTA pairs sharing the weight k-blocks by multicast: one n-tile, an even number of row tiles, a deep reduction
  // (K = 256 products are bound by their output traffic, not by operand delivery).  Measured at conf 18 / batch 256
  // (fc2: M = 16640, K = 3072, one tile per CTA): 39.6 us paired vs 39.7 us single - the product is not bound by L2
  // operand delivery; an in-tile L2 look-ahead of 4-16 k-blocks made it 2-3 us SLOWER.  ncu: the tensor pipe is
  // busy 41 % of the CTA's life, the LayerNorm epilogue of the CTA's only tile (~9 us) is fully exposed.
  const int tiles_total = ceil_div(t.M, RS_BM) * (t.N / RS_BN);
  const bool pair = tuning(VIT3D_TUNE_RES_PAIR) != 0 && t.N == RS_BN && tiles_total % 2 == 0 && t.K >= 1024 &&
                    (tiles_total <= sm_count() || (sm_count() % 2 == 0 && tiles_total % sm_count() % 2 == 0));
  rc = make_tmap_2d(&tb, t.w, 2, t.N, t.K, t.K, pair ? RS_BN / 2 : RS_BN, 64, 128);
  if (rc != VIT3D_OK) return rc;
  rc = make_tmap_2d(&ty, t.y, 4, t.M, t.N, t.N, 32, 32, 128);
  if (rc != VIT3D_OK) return rc;
  tr = ty;
  tl = ty;
  if (t.residual) {
    rc = make_tmap_2d(&tr, t.residual, 4, t.M, t.N, t.N, 32, 32, 128);
    if (rc != VIT3D_OK) return rc;
  }
  if (ln) {
    rc = make_tmap_2d(&tl, t.ln_out, 2, t.M, t.N, t.N, 32, 32, 64);
    if (rc != VIT3D_OK) return rc;
  }
  ResEpilogue ep;
  ep.bias = t.bias; ep.gamma = t.ln_gamma; ep.beta = t.ln_beta; ep.mean = t.ln_mean; ep.rstd = t.ln_rstd; ep.eps = t.ln_eps;
  ep.drop_bits = t.drop_bits; ep.drop_scale = t.drop_scale;
  const int mode = (t.bias ? 1 : 0) | (t.residual ? 2 : 0) | (ln ? 4 : 0);
  if (t.drop_bits) {
    // training fc2: Dropout between the Linear and the residual add (modeling.py:123, :196)
    if (!t.bias || !t.residual) { set_error("tc_gemm_res: the dropout variant needs bias and residual"); return VIT3D_ERR_UNSUPPORTED; }
    if (ln && pair) return launch_res<15, 2>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    return ln ? launch_res<15>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st) : launch_res<11>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
  }
  switch (mode) {
    case 0: return launch_res<0>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    case 1: return launch_res<1>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    case 2: return launch_res<2>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    case 3: return launch_res<3>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    case 4: return launch_res<4>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    case 5: return launch_res<5>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    case 6: return launch_res<6>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
    default: return pair ? launch_res<7, 2>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st)
                         : launch_res<7>(ta, tb, ty, tr, tl, ep, t.M, t.N, t.K, st);
  }
}

}  // namespace vit3d
