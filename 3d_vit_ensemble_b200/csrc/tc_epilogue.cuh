// Shared epilogue machinery of the tcgen05 kernels (GEMM, fused MLP): TMEM -> registers -> swizzled
// shared-memory transpose -> coalesced global / bulk tensor stores, with bias / GELU / residual / position
// rows fused.
#pragma once
#include <cuda_fp16.h>

#include "ptx.cuh"
#include "tc.cuh"

namespace vit3d {

using namespace ptx;

struct TcEpilogue {
  const float* bias = nullptr;      // [N]
  const float* residual = nullptr;  // [M,N] fp32
  const float* rowadd = nullptr;    // [(row_group+1), N] position table
  void* out = nullptr;              // [rows, N] fp32 or bf16
  void* pre = nullptr;              // pre-activation copy (type of out)
  int out_f32 = 1;
  int act = 0;
  int row_group = 0;                // >0: out row = m + m / row_group + 1
  int cluster = 1;                  // patch mode: CTAs of a cluster share every filter-bank k-block by TMA multicast
  int grid_limit = 0;               // > 0: launch at most this many CTAs (cluster launches: whole co-resident clusters)
  int atomic = 0;                   // accumulate (split-K): 1 = fp32 vector atomics, 2 = TMA reduce-add boxes (tmC / tmPre / tmX per segment)
  int vols_per_tile = 0;            // patch-embedding mode: volumes per 128-row tile
  int round_tf32 = 0;               // fp32 output is the operand of a TF32 GEMM: round to nearest tf32
  // training: Dropout after the activation (modeling.py:121) applied from a keep-bit array (bit i = element i of
  // the [M,N] output, k_train.cu dropout_bits); bf16 outputs, N % 32 == 0
  const uint32_t* drop_bits = nullptr;
  float drop_scale = 1.f;
  // training fc1: the `pre` output receives d act / d pre = gelu'(pre) * keep * drop_scale - the factor the backward
  // multiplies the incoming gradient by - instead of the pre-activation itself (the backward then needs neither the
  // GELU derivative nor the keep bits; computed here it hides under this kernel's store-bound time)
  int store_dact = 0;
  // atomic (weight-gradient) outputs split by rows over up to three buffers: rows [i*seg_rows, (i+1)*seg_rows)
  // go to out / out_seg[0] / out_seg[1] (the packed q|k|v weight gradient lands in three parameters' .grad)
  float* out_seg[2] = {nullptr, nullptr};
  int seg_rows = 0;
  // split-K weight gradients WITHOUT atomics: work item w stores its 128 x BN fp32 tile densely at partial_ws + w*128*BN
  // (plain 16-byte stores); vit3d_wgrad_reduce sums the slices of a tile afterwards.  (Measured: not faster than the
  // atomics for the training step - the extra HBM traffic outweighs them; kept as an option.)
  float* partial_ws = nullptr;
};


// 2-D row-major tensor map (defined in k_tc_gemm.cu, cached per thread)
int make_tmap_2d(CUtensorMap* out, const void* ptr, int elem_bytes, long long rows, long long cols, long long ld_elems,
                 int box_rows, int box_cols, int swizzle_bytes);
// rank-N fp32 tensor map with 128-byte swizzle (defined in k_tc_gemm.cu, not cached)
int make_tmap_nd(CUtensorMap* out, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                 const cuuint32_t* box);

// ----------------------------------------------------------------------------- epilogue
// fast GELU (bf16 outputs, and the fp32 outputs of TF32 mode): x * sigmoid(2u), u = x (c0 + c1 x^2 + c2 x^4) fitted to the exact erf
// GELU (max abs error 3e-5, far below the bf16 rounding of the result): 7 FMA-pipe ops + 2 MUFU.
__device__ __forceinline__ float gelu_fast(float x) {
  const float x2 = fminf(x * x, 100.f);                // the fitted polynomial is monotone up to |x| = 10
  // -2*log2(e) * {0.797458471, 0.0370503451, -3.58732362e-4}
  float p = fmaf(x2, 1.03506367e-3f, -0.106903009f);
  p = fmaf(x2, p, -2.30099750f);
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * p));          // exp(-2u)
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return x * r;
}

__device__ __forceinline__ uint32_t pack2_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

// GELU of two values at once in packed half precision, result packed bf16x2.  Same fitted form as
// gelu_fast written with tanh: y = hx + hx * tanh(x (c0 + c1 x^2 + c2 x^4)), hx = x/2.  Seven HFMA2-pipe
// ops and ONE MUFU (tanh.approx.f16x2) per PAIR - the scalar fp32 form costs 7 + 2 MUFU per ELEMENT and
// made the fc1 epilogue MUFU/issue bound.  f16 carries 11 significant bits against the 8 of the bf16
// result: measured mean |error| after the bf16 rounding is 1.38e-3 vs 1.30e-3 for a correctly rounded GELU
// (|x| <= 4).  Pre-activations beyond +-65504 would overflow to inf (never the case for LayerNorm'd inputs).
// same, result left as packed f16x2: the fused MLP feeds it to tcgen05 as an fp16 A operand (11 significant
// bits instead of bf16's 8, and no f16 -> f32 -> bf16 repacking in the epilogue)
__device__ __forceinline__ uint32_t gelu_pair_f16(float a, float b) {
  const __half2 x = __floats2half2_rn(a, b);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.58732362e-4f), __float2half2_rn(0.0370503451f));
  p = __hfma2(x2, p, __float2half2_rn(0.797458471f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 th = *reinterpret_cast<const __half2*>(&ti);
  const __half2 hx = __hmul2(x, __float2half2_rn(0.5f));
  const __half2 y = __hfma2(hx, th, hx);
  return *reinterpret_cast<const uint32_t*>(&y);
}
__device__ __forceinline__ uint32_t gelu_pair_bf16(float a, float b) {
  const __half2 x = __floats2half2_rn(a, b);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.58732362e-4f), __float2half2_rn(0.0370503451f));
  p = __hfma2(x2, p, __float2half2_rn(0.797458471f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 th = *reinterpret_cast<const __half2*>(&ti);
  const __half2 hx = __hmul2(x, __float2half2_rn(0.5f));
  const float2 f = __half22float2(__hfma2(hx, th, hx));
  return pack2_bf16(f.x, f.y);
}
// same fitted GELU, result left as two floats (the dropout variants scale before packing)
__device__ __forceinline__ float2 gelu_pair_f2(float a, float b) {
  const __half2 x = __floats2half2_rn(a, b);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.58732362e-4f), __float2half2_rn(0.0370503451f));
  p = __hfma2(x2, p, __float2half2_rn(0.797458471f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 th = *reinterpret_cast<const __half2*>(&ti);
  const __half2 hx = __hmul2(x, __float2half2_rn(0.5f));
  return __half22float2(__hfma2(hx, th, hx));
}
// fitted GELU and its derivative for a pair, sharing the tanh (packed half):
//   y = hx (1 + t), y' = 0.5 (1 + t) + hx (1 - t^2) (c0 + 3 c1 x^2 + 5 c2 x^4),  t = tanh(x (c0 + c1 x^2 + c2 x^4)), hx = x / 2
__device__ __forceinline__ void gelu_and_grad_pair(float a, float b, float2& y, float2& dy) {
  const __half2 x = __floats2half2_rn(a, b);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.58732362e-4f), __float2half2_rn(0.0370503451f));
  p = __hfma2(x2, p, __float2half2_rn(0.797458471f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 t = *reinterpret_cast<const __half2*>(&ti);
  const __half2 half = __float2half2_rn(0.5f);
  const __half2 hx = __hmul2(x, half);
  y = __half22float2(__hfma2(hx, t, hx));
  __half2 q = __hfma2(x2, __float2half2_rn(5.f * -3.58732362e-4f), __float2half2_rn(3.f * 0.0370503451f));
  q = __hfma2(x2, q, __float2half2_rn(0.797458471f));
  const __half2 a1 = __hfma2(t, half, half);                              // 0.5 (1 + t)
  const __half2 s = __hfma2(__hneg2(t), t, __float2half2_rn(1.f));        // 1 - t^2
  dy = __half22float2(__hfma2(__hmul2(hx, s), q, a1));
}
// Training fc1 epilogue for one column pair, all in packed half: x = acc + bias; the dropout scale is folded into
// the constants (hs = 0.5 * scale), the keep bits arrive as a 32-bit AND mask (0xffff per kept column):
//   w = bf16x2(gelu(x) * keep * scale),  dq = bf16x2(gelu'(x) * keep * scale)
__device__ __forceinline__ void gelu_grad_drop_pair(float a, float b, uint32_t bias_h2, __half2 hs, uint32_t mask, uint32_t& w,
                                                    uint32_t& dq) {
  const __half2 x = __hadd2(__floats2half2_rn(a, b), *reinterpret_cast<const __half2*>(&bias_h2));
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.58732362e-4f), __float2half2_rn(0.0370503451f));
  p = __hfma2(x2, p, __float2half2_rn(0.797458471f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 t = *reinterpret_cast<const __half2*>(&ti);
  const __half2 hx = __hmul2(x, hs);                                       // scale x / 2
  __half2 y = __hfma2(hx, t, hx);
  __half2 q = __hfma2(x2, __float2half2_rn(5.f * -3.58732362e-4f), __float2half2_rn(3.f * 0.0370503451f));
  q = __hfma2(x2, q, __float2half2_rn(0.797458471f));
  const __half2 a1 = __hfma2(t, hs, hs);                                   // scale (1 + t) / 2
  const __half2 sm = __hfma2(__hneg2(t), t, __float2half2_rn(1.f));        // 1 - t^2
  __half2 dy = __hfma2(__hmul2(hx, sm), q, a1);
  const uint32_t yb = *reinterpret_cast<const uint32_t*>(&y) & mask, db = *reinterpret_cast<const uint32_t*>(&dy) & mask;
  y = *reinterpret_cast<const __half2*>(&yb);
  dy = *reinterpret_cast<const __half2*>(&db);
  w = pack2_bf16(__low2float(y), __high2float(y));
  dq = pack2_bf16(__low2float(dy), __high2float(dy));
}
// keep bits (2j, 2j+1) of `mw` -> AND mask for the half pair: A = mw << s0 puts bit 2j at the top of byte j/4,
// B = mw << (s0 - 1) puts bit 2j+1 there; prmt in sign-replication mode spreads the two byte signs over a half each
template <int J>
__device__ __forceinline__ uint32_t keep_mask_pair(const uint32_t (&sh)[8]) {
  constexpr int s0 = 7 - ((2 * J) & 7), k = J >> 2;
  constexpr uint32_t lo = 8u | k, hi = 8u | (4u + k);
  constexpr uint32_t sel = (hi << 12) | (hi << 8) | (lo << 4) | lo;
  uint32_t m;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(m) : "r"(sh[s0]), "r"(sh[s0 - 1]), "n"(sel));
  return m;
}
template <int J>
__device__ __forceinline__ void gelu_grad_drop_unroll(const uint32_t (&r)[32], const uint32_t (&bh)[16], __half2 hs,
                                                      const uint32_t (&sh)[8], uint32_t (&w)[16], uint32_t (&dq)[16]) {
  if constexpr (J < 16) {
    gelu_grad_drop_pair(__uint_as_float(r[2 * J]), __uint_as_float(r[2 * J + 1]), bh[J], hs, keep_mask_pair<J>(sh), w[J], dq[J]);
    gelu_grad_drop_unroll<J + 1>(r, bh, hs, sh, w, dq);
  }
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

// Each epilogue warp owns 32 accumulator rows (one TMEM lane quarter) x CW columns.  TMEM hands every
// thread one ROW (tcgen05.ld 32x32b); rows are transposed through a 2 KB swizzled shared-memory tile
// (32 rows x 64 bytes) so that global loads/stores are whole 32-byte sectors, 64 contiguous bytes per row.
//   fp32 output : 16 columns per round; raw accumulators are staged, bias / position rows / GELU /
//                 residual are applied in the coalesced phase (element-wise, layout does not matter).
//   bf16 output : 32 columns per round; bias (+GELU) are applied in the row-owner phase, packed to bf16
//                 and staged; the coalesced phase is a pure copy.
// staging position of 16-byte chunk j of row r: r*64 + ((j ^ ((r >> 1) & 3)) << 4)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
// fp32 reduce-add of a staged box into global memory, executed by the TMA unit at the L2 (split-K weight gradients:
// no REDG instructions through the SM's load/store path, which retires ~1 element per clock and SM)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// split-K weight-gradient epilogue: the warp's 32 x CW fp32 slice leaves as [32 x 16] boxes (SWIZZLE_64B staging)
// that the TMA unit adds into `tm` at (row0, n_base + c); rows / columns past the map's extent are clipped.
template <int CW>
__device__ __forceinline__ void epilogue_reduce_f32(const CUtensorMap* tm, uint32_t taddr, uint32_t stage, int lane,
                                                    int row0, int n_base, int N) {
  const uint32_t my_row = stage + lane * 64;
  const int sw = (lane >> 1) & 3;
#pragma unroll 1
  for (int c = 0; c < CW; c += 16) {
    if (n_base + c >= N) break;
    uint32_t r[16];
    tmem_ld_32x32b_x16(taddr + c, r);
    if (lane == 0) bulk_store_wait_read();      // the previous box has left the staging tile
    __syncwarp();
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 4; ++j) st_shared_v4(my_row + ((j ^ sw) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_reduce_add_2d(tm, stage, n_base + c, row0);
      bulk_store_commit();
    }
  }
}

// `out_ptr` / `atomic` / `seg_rows` are passed beside `ep` so that a caller can redirect the output (split-K partial
// tiles) without building a modified copy of the struct - a copy lives in local memory and drags every ep.* read of
// the epilogue there with it (measured: +43 us on the patch-embedding GEMM)
template <int CW, bool FAST_GELU, bool DACT = false>
__device__ __forceinline__ void epilogue_rows(const TcEpilogue& ep, const CUtensorMap* tmC, const CUtensorMap* tmPre,
                                              uint32_t taddr, uint32_t stage, int lane, int m_base, int n_base, int M,
                                              int N, void* out_ptr, int atomic, int seg_rows) {
  const uint32_t my_row = stage + lane * 64;
  const int sw = (lane >> 1) & 3;
  const int chunk = lane & 3, rsub = lane >> 2;       // coalesced phase: 4 lanes per row, 8 rows per instruction
  if (ep.out_f32) {
#pragma unroll 1
    for (int c = 0; c < CW; c += 16) {
      if (n_base + c >= N) break;
      uint32_t r[16];
      tmem_ld_32x32b_x16(taddr + c, r);
      const int col = n_base + c + chunk * 4;
      const bool colok = col < N;
      // issue every global read of this round before the TMEM wait / the stores (out may alias residual)
      float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 res[4], radd[4];
      if (colok) {
        if (ep.bias) bias = __ldg(reinterpret_cast<const float4*>(ep.bias + col));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m_base + i * 8 + rsub;
          res[i] = radd[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m < M) {
            if (ep.residual) res[i] = __ldg(reinterpret_cast<const float4*>(ep.residual + (long long)m * N + col));
            if (ep.rowadd)
              radd[i] = __ldg(reinterpret_cast<const float4*>(ep.rowadd + (long long)((m % ep.row_group) + 1) * N + col));
          }
        }
      }
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 4; ++j) st_shared_v4(my_row + ((j ^ sw) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
      __syncwarp();
      if (colok) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = i * 8 + rsub;
          const int m = m_base + row;
          if (m < M) {
            const uint4 u = ld_shared_v4(stage + row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4));
            float4 v = make_float4(__uint_as_float(u.x) + bias.x + radd[i].x, __uint_as_float(u.y) + bias.y + radd[i].y,
                                   __uint_as_float(u.z) + bias.z + radd[i].z, __uint_as_float(u.w) + bias.w + radd[i].w);
            long long orow = ep.row_group > 0 ? (long long)m + m / ep.row_group + 1 : (long long)m;
            float* obase = reinterpret_cast<float*>(out_ptr);
            if (seg_rows > 0) {
              const int seg = m / seg_rows;
              if (seg > 0) obase = seg == 1 ? ep.out_seg[0] : ep.out_seg[1];
              orow = m - seg * seg_rows;
            }
            // the output address is formed at each store, not once above: at the 96-register cap that leaves ptxas less to spill
            if (atomic) {
              // one 16-byte vector reduction instead of four scalar ones (split-K weight gradients)
              float* o = obase + orow * N + col;
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                           : "memory");
            } else {
              if (ep.pre) *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.pre) + orow * N + col) = v;
              // fitted GELU (max abs error 2.9e-5 in fp32, 9 instructions): the erff form made the TF32-mode fc1 - 136 M
              // outputs per layer at batch 1024 - epilogue-bound at 333 us; the exact FP32 mode never comes through here
              if (ep.act == VIT3D_ACT_GELU) { v.x = gelu_fast(v.x); v.y = gelu_fast(v.y); v.z = gelu_fast(v.z); v.w = gelu_fast(v.w); }
              v.x += res[i].x; v.y += res[i].y; v.z += res[i].z; v.w += res[i].w;
              if (ep.round_tf32) { v.x = round_tf32(v.x); v.y = round_tf32(v.y); v.z = round_tf32(v.z); v.w = round_tf32(v.w); }
              *reinterpret_cast<float4*>(obase + orow * N + col) = v;
            }
          }
        }
      }
      __syncwarp();
    }
  } else {
    // bf16 output: 32 columns (64 B per row) per round, staged in the TMA SWIZZLE_64B layout and written
    // with one bulk tensor store per round (rows >= M / columns >= N are clipped by the TMA unit).
#pragma unroll 1
    for (int c = 0; c < CW; c += 32) {
      if (n_base + c >= N) break;
      float v[32];
      {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + c, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      }
      if (ep.bias) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          if (n_base + c + j < N) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + n_base + c + j));
            v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
          }
        }
      }
      // DACT (the training fc1 outside the lean epilogue's shapes) is a compile-time variant: its second 32-value
      // array must not cost the other generic kernels registers (they sit at the 96-register cap)
      float dq[DACT ? 32 : 1];
      if constexpr (DACT) {
        // training fc1: (gelu, gelu') per element, both multiplied by keep * scale; `pre` receives the derivative
        const int m = m_base + lane;
        uint32_t mw = 0xffffffffu;
        if (ep.drop_bits) mw = m < M ? __ldg(ep.drop_bits + (((long long)m * N + n_base + c) >> 5)) : 0u;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float2 y, g;
          gelu_and_grad_pair(v[2 * j], v[2 * j + 1], y, g);
          const float k0 = ((mw >> (2 * j)) & 1u) ? ep.drop_scale : 0.f, k1 = ((mw >> (2 * j + 1)) & 1u) ? ep.drop_scale : 0.f;
          v[2 * j] = y.x * k0; v[2 * j + 1] = y.y * k1;
          dq[2 * j] = g.x * k0; dq[2 * j + 1] = g.y * k1;
        }
      }
#pragma unroll 1
      for (int pass = 0; pass < 2; ++pass) {
        // pass 0: pre-activation copy (training), pass 1: output
        if (pass == 0 && ep.pre == nullptr) continue;
        if constexpr (DACT) {
          if (lane == 0) bulk_store_wait_read();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (pass == 0)
              st_shared_v4(my_row + ((j ^ sw) << 4), pack2_bf16(dq[8 * j], dq[8 * j + 1]), pack2_bf16(dq[8 * j + 2], dq[8 * j + 3]),
                           pack2_bf16(dq[8 * j + 4], dq[8 * j + 5]), pack2_bf16(dq[8 * j + 6], dq[8 * j + 7]));
            else
              st_shared_v4(my_row + ((j ^ sw) << 4), pack2_bf16(v[8 * j], v[8 * j + 1]), pack2_bf16(v[8 * j + 2], v[8 * j + 3]),
                           pack2_bf16(v[8 * j + 4], v[8 * j + 5]), pack2_bf16(v[8 * j + 6], v[8 * j + 7]));
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(pass == 0 ? tmPre : tmC, stage, n_base + c, m_base);
            bulk_store_commit();
          }
          continue;
        }
        const bool gelu = pass == 1 && ep.act == VIT3D_ACT_GELU;
        if (gelu && !FAST_GELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_f(v[j]);
        }
        const bool drop = pass == 1 && ep.drop_bits != nullptr;
        if (drop) {
          if (gelu && FAST_GELU) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float2 f = gelu_pair_f2(v[2 * j], v[2 * j + 1]);
              v[2 * j] = f.x; v[2 * j + 1] = f.y;
            }
          }
          const int m = m_base + lane;
          const uint32_t mw = m < M ? __ldg(ep.drop_bits + (((long long)m * N + n_base + c) >> 5)) : 0u;
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = ((mw >> j) & 1u) ? v[j] * ep.drop_scale : 0.f;
        }
        if (lane == 0) bulk_store_wait_read();      // the previous round's store has finished reading the tile
        __syncwarp();
        if (gelu && FAST_GELU && !drop) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            st_shared_v4(my_row + ((j ^ sw) << 4), gelu_pair_bf16(v[8 * j], v[8 * j + 1]), gelu_pair_bf16(v[8 * j + 2], v[8 * j + 3]),
                         gelu_pair_bf16(v[8 * j + 4], v[8 * j + 5]), gelu_pair_bf16(v[8 * j + 6], v[8 * j + 7]));
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            st_shared_v4(my_row + ((j ^ sw) << 4), pack2_bf16(v[8 * j], v[8 * j + 1]), pack2_bf16(v[8 * j + 2], v[8 * j + 3]),
                         pack2_bf16(v[8 * j + 4], v[8 * j + 5]), pack2_bf16(v[8 * j + 6], v[8 * j + 7]));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(pass == 0 ? tmPre : tmC, stage, n_base + c, m_base);
          bulk_store_commit();
        }
      }
    }
  }
}


// ----------------------------------------------------------------------------- lean bf16 epilogue
// The hot bf16-output GEMMs (qkv, fc1 + GELU, the data-gradient products) are bound by the instruction
// issue rate of their epilogue warps, not by the tensor pipe: at K = 256 a 128 x 256 tile is 2048 MMA
// cycles, i.e. each scheduler has 2048 issue slots for 8192 output elements x (4 warps).  This variant is
// specialised at compile time (no run-time flags, no column predicates: N % BN == 0; rows >= M are clipped
// by the bulk tensor store), reads the bias from shared memory (staged once per n-tile by the CTA; fp32
// and packed-half copies) instead of the global loads + scoreboard waits of the generic path, and with
// GELU and no pre-activation output adds the bias in packed half precision after the conversion.
//   MODE bit 0: bias, bit 1: GELU, bit 2: also store the pre-activation (training)
constexpr int EPI_GENERIC = -1;
constexpr int EPI_WGRAD = -3;            // weight gradients: TMA reduce boxes / fp32 atomics over row segments / partial tiles
constexpr int EPI_GENERIC_DACT = -2;     // generic epilogue with the training fc1's (gelu, gelu') outputs compiled in
__device__ __forceinline__ uint32_t gelu_pair_bf16_h2(__half2 x) {
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.58732362e-4f), __float2half2_rn(0.0370503451f));
  p = __hfma2(x2, p, __float2half2_rn(0.797458471f));
  const __half2 u = __hmul2(x, p);
  uint32_t ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 th = *reinterpret_cast<const __half2*>(&ti);
  const __half2 hx = __hmul2(x, __float2half2_rn(0.5f));
  const float2 f = __half22float2(__hfma2(hx, th, hx));
  return pack2_bf16(f.x, f.y);
}

//   MODE bit 3: the training fc1 (needs bits 0-2): output = gelu(v) * keep * scale, and the `pre` output receives
//               d act / d pre = gelu'(v) * keep * scale (TcEpilogue::store_dact).  `keep` = the CW / 32 words of keep
//               bits of this thread's row (fetched by the caller before the accumulator wait; 0 for rows >= M, all
//               ones when the call has no dropout)
template <int CW, int MODE>
__device__ __forceinline__ void epilogue_bf16_lean(const CUtensorMap* tmC, const CUtensorMap* tmPre, uint32_t taddr,
                                                   uint32_t stage, uint32_t bias_f32, uint32_t bias_h2, int lane,
                                                   int m_base, int n_base, const uint32_t* keep = nullptr,
                                                   float drop_scale = 1.f) {
  constexpr bool BIAS = (MODE & 1) != 0, GELU = (MODE & 2) != 0, PRE = (MODE & 4) != 0, DROP = (MODE & 8) != 0;
  static_assert(!DROP || (GELU && PRE), "dropout variant = training fc1 (bias + GELU + pre-activation)");
  const uint32_t my_row = stage + lane * 64;
  const int sw = (lane >> 1) & 3;
#pragma unroll
  for (int c = 0; c < CW; c += 32) {
    uint32_t r[32];
    tmem_ld_32x32b_x32(taddr + c, r);
    tmem_ld_wait();
    uint32_t w[16];
    if constexpr (GELU && !PRE) {
      // packed-half path: convert, add the half bias, GELU, repack as bf16
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        uint4 b = make_uint4(0u, 0u, 0u, 0u);
        if constexpr (BIAS) b = ld_shared_v4(bias_h2 + (c + 2 * j) * 2);
        const uint32_t bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          __half2 x = __floats2half2_rn(__uint_as_float(r[2 * (j + i)]), __uint_as_float(r[2 * (j + i) + 1]));
          if constexpr (BIAS) x = __hadd2(x, *reinterpret_cast<const __half2*>(&bb[i]));
          w[j + i] = gelu_pair_bf16_h2(x);
        }
      }
    } else if constexpr (DROP) {
      // training fc1: packed-half GELU and derivative, dropout scale folded in, keep bits as AND masks
      uint32_t dq[16], bh[16];
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const uint4 b = ld_shared_v4(bias_h2 + (c + 2 * j) * 2);
        bh[j] = b.x; bh[j + 1] = b.y; bh[j + 2] = b.z; bh[j + 3] = b.w;
      }
      const uint32_t mw = keep[c >> 5];
      uint32_t sh[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) sh[i] = mw << i;
      gelu_grad_drop_unroll<0>(r, bh, __float2half2_rn(0.5f * drop_scale), sh, w, dq);
      if (lane == 0) bulk_store_wait_read();
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) st_shared_v4(my_row + ((j ^ sw) << 4), dq[4 * j], dq[4 * j + 1], dq[4 * j + 2], dq[4 * j + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(tmPre, stage, n_base + c, m_base);
        bulk_store_commit();
      }
    } else {
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      if constexpr (BIAS) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const uint4 b = ld_shared_v4(bias_f32 + (c + j) * 4);
          v[j] += __uint_as_float(b.x); v[j + 1] += __uint_as_float(b.y);
          v[j + 2] += __uint_as_float(b.z); v[j + 3] += __uint_as_float(b.w);
        }
      }
      if constexpr (PRE) {
        if (lane == 0) bulk_store_wait_read();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j)
          st_shared_v4(my_row + ((j ^ sw) << 4), pack2_bf16(v[8 * j], v[8 * j + 1]), pack2_bf16(v[8 * j + 2], v[8 * j + 3]),
                       pack2_bf16(v[8 * j + 4], v[8 * j + 5]), pack2_bf16(v[8 * j + 6], v[8 * j + 7]));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(tmPre, stage, n_base + c, m_base);
          bulk_store_commit();
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) w[j] = GELU ? gelu_pair_bf16(v[2 * j], v[2 * j + 1]) : pack2_bf16(v[2 * j], v[2 * j + 1]);
    }
    if (lane == 0) bulk_store_wait_read();      // the previous store has finished reading the staging tile
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) st_shared_v4(my_row + ((j ^ sw) << 4), w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(tmC, stage, n_base + c, m_base);
      bulk_store_commit();
    }
  }
}

}  // namespace vit3d
