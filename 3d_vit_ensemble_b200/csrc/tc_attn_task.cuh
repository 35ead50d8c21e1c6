// The (head, 16-row tile) task of the bf16 attention forward on a volume image in shared memory, shared by
// attn_fwd_tc_kernel (k_tc_attn.cu: images of the packed qkv rows) and qkv_attn_kernel (k_tc_qkv_attn.cu: images of
// one head group's q | k | v columns, written by its own projection epilogue), plus the mma.sync helpers it uses.
#pragma once
#include "ptx.cuh"

namespace vit3d {

constexpr int AT_S = 65;           // tokens per volume
constexpr int AT_A = 256;          // all-head size (heads * D)

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

// Predicated stores as single instructions (the compiler turns `if (lane_predicate) *p = v;` into a divergent
// branch with a BSSY/BSYNC pair and re-materialised descriptor registers around every store).
__device__ __forceinline__ void st_global_f2_if(bool pred, float* p, float x, float y) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q st.global.v2.f32 [%0], {%1, %2};\n\t}" ::"l"(p), "f"(x), "f"(y),
               "r"((uint32_t)pred)
               : "memory");
}
__device__ __forceinline__ void st_global_f1_if(bool pred, float* p, float x) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.global.f32 [%0], %1;\n\t}" ::"l"(p), "f"(x), "r"((uint32_t)pred)
               : "memory");
}
__device__ __forceinline__ void st_shared_u32_if(bool pred, uint32_t addr, uint32_t v) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.shared.b32 [%0], %1;\n\t}" ::"r"(addr), "r"(v), "r"((uint32_t)pred)
               : "memory");
}

// One task of volume b: rows [16 rt, 16 rt + 16) of head h.  S = Q K^T with mma.sync.m16n8k16 (bf16, fp32 accumulate),
// the softmax runs in registers with quad shuffles, P (bf16) feeds the P V mma straight from the accumulator registers,
// the context tile overwrites the Q tile it came from in the image and the warp ships it to ctx itself.
//   row(r): shared address of token row r < 80 of the volume image (rows >= 65 are never dereferenced);  qc: element column of the head's q block in the image,
//   its k and v blocks start at qc + KOFF and qc + 2 KOFF;  h: the head's index among all AT_A / D heads.
// VIS: 0 = no probabilities; 1 = probabilities in the reference's packed layout (rows of 65 floats); 2 = rows padded to
// `pld` floats with pld % 8 == 0 (288-byte rows at pld = 72): every row starts on a 32-byte sector, so each 8-byte
// column pair a lane stores is sector-aligned - the packed layout's rows start at 4-byte phases, its 32-byte row
// segments straddle sectors and the L1 -> L2 write traffic was 1.58x the payload (ncu, profiles/r01_attn_fwd_vis_*).
template <int D, int VIS, int KOFF, typename RowAddr>
__device__ __forceinline__ void attn_fwd_task(const RowAddr& row, int qc, int h, int rt, int b, int lane,
                                              __nv_bfloat16* __restrict__ ctx, float* __restrict__ probs,
                                              float scale_log2e, int pld) {
  constexpr int HEADS = AT_A / D;
  constexpr int KSTEPS = D / 16;      // k-steps of the Q K^T product
  constexpr int NT = 10;              // key n-tiles of 8 (80 >= 65; tiles 8.. are partly / fully padding)
  constexpr int DT = D / 8;           // output n-tiles of the P V product
  const int g = lane >> 2, t = lane & 3;
  const int r0 = rt * 16;
  // ---- Q fragments (A operand), rows clamped to the last token
  uint32_t qa[KSTEPS][4];
  {
    const uint32_t ra = row(min(r0 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1));
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
      const uint32_t addr = ra + (qc + ks * 16 + (lane >> 4) * 8) * 2;
      ldsm_x4(addr, qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
    }
  }
  // ---- S = Q K^T
  float s[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    if (nt < 9) {
      const uint32_t ra = row(min(nt * 8 + (lane & 7), AT_S - 1));
#pragma unroll
      for (int ks = 0; ks < KSTEPS; ++ks) {
        uint32_t b0, b1;
        const uint32_t addr = ra + (KOFF + qc + ks * 16 + ((lane >> 3) & 1) * 8) * 2;
        ldsm_x2(addr, b0, b1);
        mma_bf16(s[nt], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b0, b1);
      }
    }
  }
  // ---- softmax over the 65 valid keys (rows g and g+8 of the tile).  Columns 0..63 (n-tiles 0..7) are
  //      valid in every lane; column 64 is element [0] / [2] of n-tile 8 in the lanes with t == 0.
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
  // which of this lane's two rows exist: both in the row tiles 0..3, only row 64 (g == 0) in tile 4.
  // `full` is warp-uniform, so the stores below are predicated instructions, not divergent branches.
  const bool full = rt < 4;
  const bool w0 = full || g == 0, w1 = full;
  if constexpr (VIS == 2) {
#pragma unroll
    for (int nt = 0; nt < 9; ++nt) {
      s[nt][0] *= inv0; s[nt][1] *= inv0;
      s[nt][2] *= inv1; s[nt][3] *= inv1;
    }
    float* p0 = probs + ((size_t)(b * HEADS + h) * AT_S + row0) * pld + 2 * t;
    float* p1 = p0 + 8 * (size_t)pld;
    // n-tile 8 = column 64 and the 7 padding floats (zeros): EVERY sector of a row is written completely - a row
    // whose last sector carried 4 valid bytes made the L2 read-modify-write it (measured slower than the packed rows)
#pragma unroll
    for (int nt = 0; nt < 9; ++nt) {
      st_global_f2_if(w0, p0 + nt * 8, s[nt][0], s[nt][1]);
      st_global_f2_if(w1, p1 + nt * 8, s[nt][2], s[nt][3]);
    }
  }
  if constexpr (VIS == 1) {
    // The probabilities leave from the accumulator registers, normalised in place (the P V product below
    // then needs no rescaling).  What bounds this kernel with vis=True is the L1 store path and the issue
    // slots around it, so every store carries a PAIR of columns as one 8-byte word and the code is
    // branch-free.  Rows of 65 floats start at alternating 8-byte phases: where (head block + row) is
    // even the pair is this thread's own (c, c+1); where it is odd the aligned pair is (c+1, c+2) and
    // column c+2 comes from the neighbour lane of the quad by one shuffle.  The pairs of n-tiles 0..7
    // cover columns 0..63 (even rows) or 1..64 (odd rows); the remaining column - 64 or 0 - lives in the
    // lane with t == 0 either way.
#pragma unroll
    for (int nt = 0; nt < 9; ++nt) {
      s[nt][0] *= inv0; s[nt][1] *= inv0;
      s[nt][2] *= inv1; s[nt][3] *= inv1;
    }
    const int bh = b * HEADS + h;
    const bool odd = ((bh + row0) & 1) != 0;          // row1 = row0 + 8 has the same parity
    float* p0 = probs + ((size_t)bh * AT_S + row0) * AT_S + 2 * t + (odd ? 1 : 0);
    float* p1 = p0 + 8 * AT_S;
    const int src = (lane & ~3) | ((t + 1) & 3);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      // what this lane hands to its left neighbour: its column c, or (t == 0) the first column of the next tile
      const float n0 = __shfl_sync(0xffffffffu, tail ? s[nt + 1][0] : s[nt][0], src);
      const float n1 = __shfl_sync(0xffffffffu, tail ? s[nt + 1][2] : s[nt][2], src);
      const float2 v0 = make_float2(odd ? s[nt][1] : s[nt][0], odd ? n0 : s[nt][1]);
      const float2 v1 = make_float2(odd ? s[nt][3] : s[nt][2], odd ? n1 : s[nt][3]);
      st_global_f2_if(w0, p0 + nt * 8, v0.x, v0.y);
      st_global_f2_if(w1, p1 + nt * 8, v1.x, v1.y);
    }
    {
      // in the lanes with t == 0, p0 points at column (odd ? 1 : 0)
      const int off = odd ? -1 : 64;
      st_global_f1_if(tail && w0, p0 + off, odd ? s[0][0] : s[8][0]);
      st_global_f1_if(tail && w1, p1 + off, odd ? s[0][2] : s[8][2]);
    }
  }
  // ---- O = P V  (P from the accumulator registers; keys 65..79 carry p = 0)
  float o[DT][4];
#pragma unroll
  for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
#pragma unroll
  for (int kk = 0; kk < 5; ++kk) {
    const uint32_t a0 = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
    const uint32_t a1 = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
    const uint32_t a2 = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
    const uint32_t a3 = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
    const uint32_t ra = row(min(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, AT_S - 1));
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) {
      uint32_t b0, b1;
      const uint32_t addr = ra + (2 * KOFF + qc + dt * 8) * 2;
      ldsm_x2_t(addr, b0, b1);
      mma_bf16(o[dt], a0, a1, a2, a3, b0, b1);
    }
  }
  // ---- the context tile overwrites the Q tile it came from (only this task reads that block) and the warp
  //      ships it itself: 16-byte chunks, a store instruction covers whole 32/64/128-byte row segments
  __syncwarp();
  {
    const uint32_t ra0 = row(row0), ra1 = row(row1);     // row1 < 80: an address only where w1 is false
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) {
      const int col = qc + dt * 8 + 2 * t;
      const float c0 = VIS != 0 ? 1.f : inv0, c1 = VIS != 0 ? 1.f : inv1;      // VIS: P was normalised before the product
      st_shared_u32_if(w0, ra0 + col * 2, pack_bf16(o[dt][0] * c0, o[dt][1] * c0));
      st_shared_u32_if(w1, ra1 + col * 2, pack_bf16(o[dt][2] * c1, o[dt][3] * c1));
    }
  }
  __syncwarp();
  {
    constexpr int CPR = D / 8;                  // 16-byte chunks per row of the tile
    uint8_t* gdst = reinterpret_cast<uint8_t*>(ctx) + ((size_t)b * AT_S * AT_A + h * D) * 2;
#pragma unroll
    for (int i = lane; i < 16 * CPR; i += 32) {
      const int r = r0 + i / CPR, ch = i % CPR;
      if (r < AT_S) {
        uint4 v;
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                     : "r"(row(r) + qc * 2 + ch * 16));
        *reinterpret_cast<uint4*>(gdst + (size_t)r * AT_A * 2 + ch * 16) = v;
      }
    }
  }
}

}  // namespace vit3d
