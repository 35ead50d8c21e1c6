// Shape-generic fp32 kernels: the exact path (VIT3D_PREC_FP32) and the fallback for shapes
// the tcgen05 kernels do not serve (e.g. the as-shipped hidden-16 / head-dim-1 models).
// All arithmetic is fp32 FMA; operands may be stored fp32 or bf16 (runtime flag).
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.cuh"

namespace vit3d {

__device__ __forceinline__ float ld_any(const void* p, long long i, int f32) {
  return f32 ? reinterpret_cast<const float*>(p)[i] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
}
__device__ __forceinline__ void st_any(void* p, long long i, int f32, float v) {
  if (f32) reinterpret_cast<float*>(p)[i] = v;
  else reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16(v);
}

// ============================================================================ GEMM (SIMT)
// C[m,n] (+)= sum_k A(m,k) * B(k,n), A(m,k)=A[m*sa_m+k*sa_k], B(k,n)=B[k*sb_k+n*sb_n].
// 64x64 tile, BK=16, 256 threads, 4x4 micro-tile.  gridDim.z > 1 => split-K with atomics.
constexpr int GBM = 64, GBN = 64, GBK = 16;

__global__ void __launch_bounds__(256) sgemm_generic_kernel(SgemmArgs g) {
  __shared__ float As[GBK][GBM + 4];
  __shared__ float Bs[GBK][GBN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * GBM, n0 = blockIdx.x * GBN;
  const int tx = tid % 16, ty = tid / 16;  // tx -> n, ty -> m
  const int kchunk = (g.K + gridDim.z - 1) / gridDim.z;
  const int kbeg = blockIdx.z * kchunk;
  const int kend = min(g.K, kbeg + kchunk);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool a_kc = (g.sa_k == 1), b_nc = (g.sb_n == 1);
  for (int k0 = kbeg; k0 < kend; k0 += GBK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      int mm, kk;
      if (a_kc) { kk = idx % GBK; mm = idx / GBK; } else { mm = idx % GBM; kk = idx / GBM; }
      const int gm = m0 + mm, gk = k0 + kk;
      float v = 0.f;
      if (gm < g.M && gk < kend) v = ld_any(g.A, (long long)gm * g.sa_m + (long long)gk * g.sa_k, g.a_f32);
      As[kk][mm] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      int nn, kk;
      if (b_nc) { nn = idx % GBN; kk = idx / GBN; } else { kk = idx % GBK; nn = idx / GBK; }
      const int gn = n0 + nn, gk = k0 + kk;
      float v = 0.f;
      if (gn < g.N && gk < kend) v = ld_any(g.B, (long long)gk * g.sb_k + (long long)gn * g.sb_n, g.b_f32);
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GBK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
    long long orow = m;
    if (g.row_group > 0) orow = (long long)m + m / g.row_group + 1;   // skip one cls row per volume
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j];
      const long long ci = orow * g.ldc + n;
      if (gridDim.z > 1) {  // split-K: accumulate only
        atomicAdd(reinterpret_cast<float*>(g.C) + ci, v);
        continue;
      }
      if (g.bias) v += g.bias[n];
      if (g.rowadd) v += g.rowadd[(long long)((m % g.row_group) + 1) * g.N + n];  // position embedding
      if (g.pre) st_any(g.pre, ci, g.c_f32, v);
      if (g.act == VIT3D_ACT_GELU) v = gelu_f(v);
      if (g.residual) v += g.residual[(long long)m * g.ldr + n];
      if (g.accumulate) v += ld_any(g.C, ci, g.c_f32);
      st_any(g.C, ci, g.c_f32, v);
    }
  }
}

int launch_sgemm(const SgemmArgs& a, cudaStream_t st) {
  if (a.M <= 0 || a.N <= 0) return VIT3D_OK;
  dim3 grid(ceil_div(a.N, GBN), ceil_div(a.M, GBM), 1);
  if (a.splitk > 1) {
    if (!(a.accumulate && a.c_f32 && !a.bias && !a.residual && !a.pre && a.act == 0 && a.row_group == 0)) {
      set_error("sgemm split-K needs a pure fp32 accumulate epilogue");
      return VIT3D_ERR_INVALID;
    }
    grid.z = a.splitk;
  }
  sgemm_generic_kernel<<<grid, 256, 0, st>>>(a);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ---------------------------------------------------------------------------- skinny-N Linear (the head)
// y[m, n] = x[m, :] . w[n, :] + bias[n] for N <= 8 (num_classes = 1 in the reference scripts): one warp per
// output row, fp32 FMA, strided x rows (the head reads token 0 of every volume).  The tiled GEMM spends
// 28 us on this [1024 x 1 x 256] product (one CTA column); this takes a few microseconds.
__global__ void __launch_bounds__(256) rowdot_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ w,
                                                     const float* __restrict__ bias, float* __restrict__ y, int M, int N,
                                                     int K) {
  const int m = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (m >= M) return;
  const float* xr = x + (long long)m * ldx;
  for (int n = 0; n < N; ++n) {
    const float* wr = w + (long long)n * K;
    float acc = 0.f;
    for (int k = lane; k < K; k += 32) acc = fmaf(__ldg(xr + k), __ldg(wr + k), acc);
    acc = warp_sum(acc);
    if (lane == 0) y[(long long)m * N + n] = acc + (bias ? bias[n] : 0.f);
  }
}
int launch_rowdot(const float* x, long long ldx, const float* w, const float* bias, float* y, int M, int N, int K,
                  cudaStream_t st) {
  if (M <= 0) return VIT3D_OK;
  rowdot_kernel<<<ceil_div(M, 8), 256, 0, st>>>(x, ldx, w, bias, y, M, N, K);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// pick a split so that a skinny-output / deep-K product (weight gradients) fills the GPU
int pick_splitk(int M, int N, int K) {
  const int tiles = ceil_div(M, GBM) * ceil_div(N, GBN);
  const int target = 4 * sm_count();
  int s = target / (tiles > 0 ? tiles : 1);
  const int maxs = K / 256;
  if (s > maxs) s = maxs;
  if (s < 1) s = 1;
  if (s > 512) s = 512;
  return s;
}

// ============================================================================ patch gather (a1)
// Pure permutation (bit-exact): patches[(b*P+p)*Kp + (i*p1+j)*p2+z] = x[b,0,px*p0+i,py*p1+j,pz*p2+z]
__global__ void patch_gather_kernel(const float* __restrict__ x, void* __restrict__ out, int out_f32, int B, int X, int Y,
                                    int Z, int p0, int p1, int p2, int nx, int ny, int nz) {
  const long long Kp = (long long)p0 * p1 * p2;
  const long long P = (long long)nx * ny * nz;
  const long long total = (long long)B * P * Kp;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long kk = t % Kp;
    const long long rp = t / Kp;
    const int p = (int)(rp % P), b = (int)(rp / P);
    const int z = (int)(kk % p2), j = (int)((kk / p2) % p1), i = (int)(kk / ((long long)p2 * p1));
    const int pz = p % nz, py = (p / nz) % ny, px = p / (nz * ny);
    const long long src = (((long long)b * X + (px * p0 + i)) * Y + (py * p1 + j)) * Z + (pz * p2 + z);
    st_any(out, t, out_f32, x[src]);
  }
}
// Fast path (the reference geometry: the patch spans all Z slices, so a patch row of p1*p2 floats is contiguous in the
// volume AND in the patch matrix): four elements per thread, 32-bit index arithmetic, one 16-byte load and one
// 16 / 8-byte store.  Same permutation, bit for bit.
template <bool F32>
__global__ void __launch_bounds__(256) patch_gather_rows_kernel(const float* __restrict__ x, void* __restrict__ out, unsigned total4,
                                                                int X, int Y, int Z, int p0, int p1, int nx, int ny) {
  const unsigned inner4 = (unsigned)(p1 * Z) >> 2;          // float4 per patch row
  const unsigned P = (unsigned)(nx * ny);
  for (unsigned u = blockIdx.x * blockDim.x + threadIdx.x; u < total4; u += gridDim.x * blockDim.x) {
    const unsigned r = u / inner4, v = u - r * inner4;       // r = (b*P + p)*p0 + i
    const unsigned bp = r / (unsigned)p0, i = r - bp * (unsigned)p0;
    const unsigned b = bp / P, p = bp - b * P;
    const unsigned px = p / (unsigned)ny, py = p - px * (unsigned)ny;
    const size_t src = (((size_t)b * X + (px * p0 + i)) * Y + (size_t)py * p1) * Z + 4u * v;
    const float4 val = *reinterpret_cast<const float4*>(x + src);
    if (F32) {
      reinterpret_cast<float4*>(out)[u] = val;
    } else {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(val.x, val.y), hi = __floats2bfloat162_rn(val.z, val.w);
      reinterpret_cast<uint2*>(out)[u] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
    }
  }
}

int launch_patch_gather(const float* x, void* out, int out_f32, int B, int X, int Y, int Z, int p0, int p1, int p2,
                        cudaStream_t st) {
  const int nx = X / p0, ny = Y / p1, nz = Z / p2;
  const long long total = (long long)B * nx * ny * nz * p0 * p1 * p2;
  if (total == 0) return VIT3D_OK;
  if (nz == 1 && p2 == Z && (p1 * Z) % 4 == 0 && (Y * Z) % 4 == 0 && total < (1ll << 33) &&
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0) {
    const unsigned total4 = (unsigned)(total / 4);
    unsigned blocks = (total4 + 255) / 256;
    const unsigned cap = (unsigned)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (out_f32) patch_gather_rows_kernel<true><<<blocks, 256, 0, st>>>(x, out, total4, X, Y, Z, p0, p1, nx, ny);
    else patch_gather_rows_kernel<false><<<blocks, 256, 0, st>>>(x, out, total4, X, Y, Z, p0, p1, nx, ny);
    V3_LAUNCH_CHECK();
    return VIT3D_OK;
  }
  int blocks = (int)((total + 255) / 256);
  const int cap = sm_count() * 16;
  if (blocks > cap) blocks = cap;
  patch_gather_kernel<<<blocks, 256, 0, st>>>(x, out, out_f32, B, X, Y, Z, p0, p1, p2, nx, ny, nz);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// Inverse permutation (bit-exact): x[b,0,px*p0+i,py*p1+j,pz*p2+z] = patches[(b*P+p)*Kp + (i*p1+j)*p2+z]; EVERY voxel of x
// is written, 0 where no patch covers it (the X % p0, Y % p1, Z % p2 remainders Conv3d drops).
__global__ void patch_scatter_kernel(const float* __restrict__ patches, float* __restrict__ x, long long total, int X, int Y,
                                     int Z, int p0, int p1, int p2, int nx, int ny, int nz) {
  const long long Kp = (long long)p0 * p1 * p2;
  const long long P = (long long)nx * ny * nz;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int zi = (int)(t % Z), yi = (int)((t / Z) % Y), xi = (int)((t / ((long long)Z * Y)) % X);
    const long long b = t / ((long long)Z * Y * X);
    float v = 0.f;
    if (xi < nx * p0 && yi < ny * p1 && zi < nz * p2) {
      const int px = xi / p0, i = xi - px * p0, py = yi / p1, j = yi - py * p1, pz = zi / p2, z = zi - pz * p2;
      const long long p = ((long long)px * ny + py) * nz + pz;
      v = patches[(b * P + p) * Kp + (i * p1 + j) * p2 + z];
    }
    x[t] = v;
  }
}
// Fast path (the patch spans all Z slices, so a patch row of p1*Z floats is contiguous in the volume AND in the patch
// matrix): four voxels per thread, one 16-byte load and one 16-byte store.  Same permutation, bit for bit.
__global__ void __launch_bounds__(256) patch_scatter_rows_kernel(const float* __restrict__ patches, float* __restrict__ x,
                                                                 unsigned total4, int X, int Y, int Z, int p0, int p1, int nx,
                                                                 int ny) {
  const unsigned inner = (unsigned)(p1 * Z), yz = (unsigned)(Y * Z), Kp = (unsigned)p0 * inner;
  const unsigned P = (unsigned)(nx * ny);
  for (unsigned u = blockIdx.x * blockDim.x + threadIdx.x; u < total4; u += gridDim.x * blockDim.x) {
    const unsigned e = 4u * u;
    const unsigned bx = e / yz, rem = e - bx * yz;            // bx = b*X + xi, rem = yi*Z + z
    const unsigned b = bx / (unsigned)X, xi = bx - b * (unsigned)X;
    const unsigned py = rem / inner, off = rem - py * inner;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (xi < (unsigned)(nx * p0) && py < (unsigned)ny) {
      const unsigned px = xi / (unsigned)p0, i = xi - px * (unsigned)p0;
      const size_t src = ((size_t)b * P + px * (unsigned)ny + py) * Kp + i * inner + off;
      v = *reinterpret_cast<const float4*>(patches + src);
    }
    reinterpret_cast<float4*>(x)[u] = v;
  }
}

int launch_patch_scatter(const float* patches, float* x, int B, int X, int Y, int Z, int p0, int p1, int p2, cudaStream_t st) {
  const int nx = X / p0, ny = Y / p1, nz = Z / p2;
  const long long total = (long long)B * X * Y * Z;
  if (total == 0) return VIT3D_OK;
  if (nz == 1 && p2 == Z && (p1 * Z) % 4 == 0 && (Y * Z) % 4 == 0 && total < (1ll << 33) &&
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(patches)) & 15) == 0) {
    const unsigned total4 = (unsigned)(total / 4);
    unsigned blocks = (total4 + 255) / 256;
    const unsigned cap = (unsigned)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    patch_scatter_rows_kernel<<<blocks, 256, 0, st>>>(patches, x, total4, X, Y, Z, p0, p1, nx, ny);
    V3_LAUNCH_CHECK();
    return VIT3D_OK;
  }
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  patch_scatter_kernel<<<(int)blocks, 256, 0, st>>>(patches, x, total, X, Y, Z, p0, p1, p2, nx, ny, nz);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// tokens[b,0,:] = cls + pos[0]  (the patch rows are written by the GEMM epilogue)
__global__ void cls_rows_kernel(const float* __restrict__ cls, const float* __restrict__ pos, float* __restrict__ tokens,
                                int B, int S, int H) {
  const long long total = (long long)B * H;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int h = (int)(t % H), b = (int)(t / H);
    tokens[(long long)b * S * H + h] = cls[h] + pos[h];
  }
}
int launch_cls_rows(const float* cls, const float* pos, float* tokens, int B, int S, int H, cudaStream_t st) {
  const long long total = (long long)B * H;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 4096) blocks = 4096;
  cls_rows_kernel<<<blocks, 256, 0, st>>>(cls, pos, tokens, B, S, H);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// dpos[s,h] += sum_b dtok[b,s,h];  dcls[h] += sum_b dtok[b,0,h]
__global__ void embed_param_grads_kernel(const float* __restrict__ dtok, float* __restrict__ dpos, float* __restrict__ dcls,
                                         int B, int S, int H, int bchunk) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;  // over S*H
  if (col >= S * H) return;
  const int b0 = blockIdx.y * bchunk, b1 = min(B, b0 + bchunk);
  float acc = 0.f;
  for (int b = b0; b < b1; ++b) acc += dtok[(long long)b * S * H + col];
  atomicAdd(dpos + col, acc);
  if (col < H) atomicAdd(dcls + col, acc);
}
int launch_embed_param_grads(const float* dtok, float* dpos, float* dcls, int B, int S, int H, cudaStream_t st) {
  const int cols = S * H;
  int by = ceil_div(B, 32);
  if (by > 64) by = 64;
  const int bchunk = ceil_div(B, by);
  by = ceil_div(B, bchunk);
  dim3 grid(ceil_div(cols, 256), by);
  embed_param_grads_kernel<<<grid, 256, 0, st>>>(dtok, dpos, dcls, B, S, H, bchunk);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// out[(b*P+p), :] = dtok[(b*(P+1)+1+p), :]   (drop the cls rows)
__global__ void gather_patch_rows_kernel(const float* __restrict__ dtok, void* __restrict__ out, int out_f32, long long total,
                                         int P, int H) {
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long m = t / H;
    const int h = (int)(t % H);
    st_any(out, t, out_f32, dtok[(m + m / P + 1) * H + h]);
  }
}
int launch_gather_patch_rows(const float* dtok, void* out, int out_f32, int B, int P, int H, cudaStream_t st) {
  const long long total = (long long)B * P * H;
  if (total == 0) return VIT3D_OK;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  gather_patch_rows_kernel<<<(int)blocks, 256, 0, st>>>(dtok, out, out_f32, total, P, H);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ LayerNorm
// One warp per row.  Rows with H <= 32*LN_MAXV live in registers, wider rows are re-read.
constexpr int LN_MAXV = 8;

template <int OUT_MODE>   // 0 fp32, 1 bf16, 2 fp32 rounded to tf32
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, void* __restrict__ y,
                                                     float* __restrict__ mean, float* __restrict__ rstd, int M, int H,
                                                     float eps) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  pdl_trigger();
  pdl_wait();
  if (row >= M) return;
  const float* xr = x + (long long)row * H;
  float v[LN_MAXV];
  const bool in_regs = H <= 32 * LN_MAXV;
  float s = 0.f;
  if (in_regs) {
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      v[i] = c < H ? xr[c] : 0.f;
      s += v[i];
    }
  } else {
    for (int c = lane; c < H; c += 32) s += xr[c];
  }
  const float mu = warp_sum(s) / (float)H;
  float q = 0.f;
  if (in_regs) {
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      const float d = c < H ? v[i] - mu : 0.f;
      q += d * d;
    }
  } else {
    for (int c = lane; c < H; c += 32) { const float d = xr[c] - mu; q += d * d; }
  }
  const float rs = rsqrtf(warp_sum(q) / (float)H + eps);
  if (lane == 0) {
    if (mean) mean[row] = mu;
    if (rstd) rstd[row] = rs;
  }
  if (in_regs) {
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < H) {
        const float o = (v[i] - mu) * rs * gamma[c] + beta[c];
        if (OUT_MODE == 1) reinterpret_cast<__nv_bfloat16*>(y)[(long long)row * H + c] = __float2bfloat16(o);
        else reinterpret_cast<float*>(y)[(long long)row * H + c] = OUT_MODE == 2 ? round_tf32(o) : o;
      }
    }
  } else {
    for (int c = lane; c < H; c += 32) {
      const float o = (xr[c] - mu) * rs * gamma[c] + beta[c];
      if (OUT_MODE == 1) reinterpret_cast<__nv_bfloat16*>(y)[(long long)row * H + c] = __float2bfloat16(o);
      else reinterpret_cast<float*>(y)[(long long)row * H + c] = OUT_MODE == 2 ? round_tf32(o) : o;
    }
  }
}
int launch_ln_fwd(const float* x, const float* g, const float* b, void* y, int y_bf16, float* mean, float* rstd, int M,
                  int H, float eps, cudaStream_t st) {
  if (M <= 0) return VIT3D_OK;
  const int rows_per_block = 8;
  const int blocks = ceil_div(M, rows_per_block);
  if (y_bf16 == 1) V3_CUDA(launch_pdl(ln_fwd_kernel<1>, dim3(blocks), dim3(256), (size_t)0, st, x, g, b, y, mean, rstd, M, H, eps));
  else if (y_bf16 == 2) V3_CUDA(launch_pdl(ln_fwd_kernel<2>, dim3(blocks), dim3(256), (size_t)0, st, x, g, b, y, mean, rstd, M, H, eps));
  else V3_CUDA(launch_pdl(ln_fwd_kernel<0>, dim3(blocks), dim3(256), (size_t)0, st, x, g, b, y, mean, rstd, M, H, eps));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// dx = dres + rstd * (g*dy - mean_h(g*dy) - xhat * mean_h(g*dy*xhat));  dgamma += sum dy*xhat; dbeta += sum dy.
// Each block owns `rows_per_block` rows; column partials are reduced in shared memory, one atomic per column per block.
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                     const float* __restrict__ mean, const float* __restrict__ rstd,
                                                     const float* __restrict__ gamma, const float* __restrict__ dres,
                                                     float* __restrict__ dx, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta, int M, int H, int rows_per_block) {
  extern __shared__ float sm[];  // [2][H] column partials
  float* s_dg = sm;
  float* s_db = sm + H;
  for (int c = threadIdx.x; c < 2 * H; c += blockDim.x) sm[c] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  for (int row = r0 + warp; row < r1; row += nwarps) {
    const float mu = mean[row], rs = rstd[row];
    const float* xr = x + (long long)row * H;
    const float* dyr = dy + (long long)row * H;
    float s1 = 0.f, s2 = 0.f;
    for (int c = lane; c < H; c += 32) {
      const float xh = (xr[c] - mu) * rs;
      const float gd = gamma[c] * dyr[c];
      s1 += gd;
      s2 += gd * xh;
    }
    s1 = warp_sum(s1) / (float)H;
    s2 = warp_sum(s2) / (float)H;
    for (int c = lane; c < H; c += 32) {
      const float xh = (xr[c] - mu) * rs;
      const float d = dyr[c];
      float o = rs * (gamma[c] * d - s1 - xh * s2);
      if (dres) o += dres[(long long)row * H + c];
      dx[(long long)row * H + c] = o;
      atomicAdd(&s_dg[c], d * xh);
      atomicAdd(&s_db[c], d);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    atomicAdd(dgamma + c, s_dg[c]);
    atomicAdd(dbeta + c, s_db[c]);
  }
}
int launch_ln_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                  const float* dres, float* dx, float* dgamma, float* dbeta, int M, int H, cudaStream_t st) {
  if (M <= 0) return VIT3D_OK;
  int rpb = ceil_div(M, 2 * sm_count());
  if (rpb < 8) rpb = 8;
  const int blocks = ceil_div(M, rpb);
  ln_bwd_kernel<<<blocks, 256, 2 * H * sizeof(float), st>>>(dy, x, mean, rstd, gamma, dres, dx, dgamma, dbeta, M, H, rpb);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ column sums (bias grads)
// db[n] += sum_m dy[m,n]
__global__ void __launch_bounds__(256) colsum_kernel(const void* __restrict__ dy, int f32, float* __restrict__ db, int M,
                                                     int N, int rows_per_block) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  float acc = 0.f;
  if (n < N)
    for (int m = r0 + (threadIdx.x >> 5); m < r1; m += 8) acc += ld_any(dy, (long long)m * N + n, f32);
  __shared__ float red[8][33];
  red[threadIdx.x >> 5][threadIdx.x & 31] = acc;
  __syncthreads();
  if (threadIdx.x < 32 && n < N) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    atomicAdd(db + n, s);
  }
}
// vectorised version: a thread owns V consecutive columns (one 16-byte load per row: 8 bf16 / 4 fp32), a warp
// reads 512 contiguous bytes of a row, the 8 warps of a block stride over the rows (4 loads in flight each)
template <bool F32>
__global__ void __launch_bounds__(256) colsum_vec_kernel(const void* __restrict__ dy, float* __restrict__ db, int M, int N,
                                                         int rows_per_block) {
  constexpr int V = F32 ? 4 : 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = (blockIdx.x * 32 + lane) * V;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  float acc[V];
#pragma unroll
  for (int j = 0; j < V; ++j) acc[j] = 0.f;
  if (col < N) {
    const uint4* base = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(dy) + (size_t)col * (F32 ? 4 : 2));
    const size_t pitch = (size_t)N * (F32 ? 4 : 2) / 16;      // row pitch in uint4
    auto add = [&](const uint4& v) {
      if (F32) {
        acc[0] += __uint_as_float(v.x); acc[1] += __uint_as_float(v.y); acc[2] += __uint_as_float(v.z); acc[3] += __uint_as_float(v.w);
      } else {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[2 * j] += __uint_as_float(w[j] << 16);
          acc[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
        }
      }
    };
    int m = r0 + warp;
    for (; m + 24 < r1; m += 32) {
      const uint4 a = __ldg(base + (size_t)m * pitch), b = __ldg(base + (size_t)(m + 8) * pitch);
      const uint4 c = __ldg(base + (size_t)(m + 16) * pitch), d = __ldg(base + (size_t)(m + 24) * pitch);
      add(a); add(b); add(c); add(d);
    }
    for (; m < r1; m += 8) add(__ldg(base + (size_t)m * pitch));
  }
  __shared__ float red[8][32][V + 1];
#pragma unroll
  for (int j = 0; j < V; ++j) red[warp][lane][j] = acc[j];
  __syncthreads();
  if (warp == 0 && col < N) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) sum += red[w][lane][j];
      atomicAdd(db + col + j, sum);
    }
  }
}

int launch_colsum(const void* dy, int f32, float* db, int M, int N, cudaStream_t st) {
  if (M <= 0 || N <= 0) return VIT3D_OK;
  const int V = f32 ? 4 : 8;
  if (N % V == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0) {
    const int gx = ceil_div(N, 32 * V);
    // two blocks per SM: every block ends in one atomic per column, and the L2 serialises the atomics of a column
    // (512 blocks on 256 columns - the patch-embedding bias gradient - spent most of their 43 us there)
    int gy = (2 * sm_count()) / gx;
    if (gy < 1) gy = 1;
    int rpb = ceil_div(M, gy);
    if (rpb < 32) rpb = 32;
    gy = ceil_div(M, rpb);
    if (f32) colsum_vec_kernel<true><<<dim3(gx, gy), 256, 0, st>>>(dy, db, M, N, rpb);
    else colsum_vec_kernel<false><<<dim3(gx, gy), 256, 0, st>>>(dy, db, M, N, rpb);
    V3_LAUNCH_CHECK();
    return VIT3D_OK;
  }
  const int gx = ceil_div(N, 32);
  int gy = (4 * sm_count()) / gx;
  if (gy < 1) gy = 1;
  int rpb = ceil_div(M, gy);
  if (rpb < 64) rpb = 64;
  gy = ceil_div(M, rpb);
  colsum_kernel<<<dim3(gx, gy), 256, 0, st>>>(dy, f32, db, M, N, rpb);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ attention core (generic)
// One block per (volume, head): K and V of that head are staged in shared memory (fp32), one
// warp per query row; any S <= 32*ATT_MAXJ, any D.
constexpr int ATT_MAXJ = 9;  // S <= 288 (the as-shipped patch-8 models have S = 257)

__global__ void __launch_bounds__(256) attn_fwd_generic_kernel(const void* __restrict__ qkv, int f32,
                                                               void* __restrict__ ctx, float* __restrict__ probs, int B,
                                                               int S, int heads, int D, float scale, int round_out) {
  extern __shared__ float sm[];
  const int A = heads * D;
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  float* Ks = sm;                 // [S][D]
  float* Vs = Ks + S * D;         // [S][D]
  float* Ps = Vs + S * D;         // [nwarps][S]
  float* Qs = Ps + (blockDim.x >> 5) * S;  // [nwarps][D]
  const long long base = (long long)b * S * 3 * A;
  for (int t = threadIdx.x; t < S * D; t += blockDim.x) {
    const int j = t / D, d = t % D;
    Ks[t] = ld_any(qkv, base + (long long)j * 3 * A + A + h * D + d, f32);
    Vs[t] = ld_any(qkv, base + (long long)j * 3 * A + 2 * A + h * D + d, f32);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  float* p = Ps + warp * S;
  float* q = Qs + warp * D;
  for (int i = warp; i < S; i += nwarps) {
    for (int d = lane; d < D; d += 32) q[d] = ld_any(qkv, base + (long long)i * 3 * A + h * D + d, f32);
    __syncwarp();
    float sc[ATT_MAXJ];
    float mx = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      float s = -INFINITY;
      if (j < S) {
        s = 0.f;
        for (int d = 0; d < D; ++d) s = fmaf(q[d], Ks[j * D + d], s);
        s *= scale;   // (q k^T) / sqrt(D), modeling.py:87-88
      }
      sc[jj] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      const float e = j < S ? expf(sc[jj] - mx) : 0.f;
      sc[jj] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      if (j < S) {
        const float pr = sc[jj] * inv;
        p[j] = pr;
        if (probs) probs[(((long long)b * heads + h) * S + i) * S + j] = pr;
      }
    }
    __syncwarp();
    for (int d = lane; d < D; d += 32) {
      float acc = 0.f;
      for (int j = 0; j < S; ++j) acc = fmaf(p[j], Vs[j * D + d], acc);
      st_any(ctx, ((long long)b * S + i) * A + h * D + d, f32, round_out ? round_tf32(acc) : acc);
    }
    __syncwarp();
  }
}
size_t attn_generic_smem(int S, int D, int nwarps, bool bwd) {
  if (!bwd) return sizeof(float) * ((size_t)2 * S * D + (size_t)nwarps * S + (size_t)nwarps * D);
  return sizeof(float) * ((size_t)6 * S * D + (size_t)2 * nwarps * S);
}
int launch_attn_fwd_generic(const void* qkv, int f32, void* ctx, float* probs, int B, int S, int heads, int D,
                            int round_out, cudaStream_t st) {
  if (B <= 0) return VIT3D_OK;
  if (S > 32 * ATT_MAXJ) V3_UNSUPPORTED("generic attention supports S <= %d (got %d)", 32 * ATT_MAXJ, S);
  const int threads = 256;
  const size_t smem = attn_generic_smem(S, D, threads / 32, false);
  if (smem > 200 * 1024) V3_UNSUPPORTED("generic attention: S*D too large for shared memory (S=%d D=%d)", S, D);
  if (smem > 48 * 1024)
    V3_CUDA(cudaFuncSetAttribute(attn_fwd_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  attn_fwd_generic_kernel<<<B * heads, threads, smem, st>>>(qkv, f32, ctx, probs, B, S, heads, D, 1.0f / sqrtf((float)D),
                                                            round_out);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// backward: recompute P row by row; dV[j]+=P[i,j] dO[i]; dP=dO V^T; dS=P*(dP-rowsum(P*dP));
// dQ[i]=scale*dS K; dK[j]+=scale*dS[i,j] Q[i].  dK/dV accumulate in shared memory.
__global__ void __launch_bounds__(256) attn_bwd_generic_kernel(const void* __restrict__ dctx, const void* __restrict__ qkv,
                                                               int f32, void* __restrict__ dqkv, int B, int S, int heads,
                                                               int D, float scale) {
  extern __shared__ float sm[];
  const int A = heads * D;
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int nwarps = blockDim.x >> 5;
  float* Qs = sm;
  float* Ks = Qs + S * D;
  float* Vs = Ks + S * D;
  float* dOs = Vs + S * D;
  float* dKs = dOs + S * D;
  float* dVs = dKs + S * D;
  float* Ps = dVs + S * D;          // [nwarps][S]
  float* dSs = Ps + nwarps * S;     // [nwarps][S]
  const long long base = (long long)b * S * 3 * A;
  for (int t = threadIdx.x; t < S * D; t += blockDim.x) {
    const int j = t / D, d = t % D;
    Qs[t] = ld_any(qkv, base + (long long)j * 3 * A + h * D + d, f32);
    Ks[t] = ld_any(qkv, base + (long long)j * 3 * A + A + h * D + d, f32);
    Vs[t] = ld_any(qkv, base + (long long)j * 3 * A + 2 * A + h * D + d, f32);
    dOs[t] = ld_any(dctx, ((long long)b * S + j) * A + h * D + d, f32);
    dKs[t] = 0.f;
    dVs[t] = 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* p = Ps + warp * S;
  float* ds = dSs + warp * S;
  for (int i = warp; i < S; i += nwarps) {
    const float* q = Qs + i * D;
    const float* dO = dOs + i * D;
    float sc[ATT_MAXJ], dp[ATT_MAXJ];
    float mx = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      float s = -INFINITY, g = 0.f;
      if (j < S) {
        s = 0.f;
        for (int d = 0; d < D; ++d) {
          s = fmaf(q[d], Ks[j * D + d], s);
          g = fmaf(dO[d], Vs[j * D + d], g);
        }
        s *= scale;
      }
      sc[jj] = s;
      dp[jj] = g;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      const float e = j < S ? expf(sc[jj] - mx) : 0.f;
      sc[jj] = e;
      sum += e;
    }
    const float inv = 1.f / warp_sum(sum);
    float delta = 0.f;
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      sc[jj] *= inv;
      delta += sc[jj] * dp[jj];
    }
    delta = warp_sum(delta);
#pragma unroll
    for (int jj = 0; jj < ATT_MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      if (j < S) {
        p[j] = sc[jj];
        ds[j] = sc[jj] * (dp[jj] - delta) * scale;
      }
    }
    __syncwarp();
    // dQ[i,:]
    for (int d = lane; d < D; d += 32) {
      float acc = 0.f;
      for (int j = 0; j < S; ++j) acc = fmaf(ds[j], Ks[j * D + d], acc);
      st_any(dqkv, base + (long long)i * 3 * A + h * D + d, f32, acc);
    }
    // dK, dV contributions of row i
    for (int t = lane; t < S * D; t += 32) {
      const int j = t / D, d = t % D;
      atomicAdd(&dKs[t], ds[j] * q[d]);
      atomicAdd(&dVs[t], p[j] * dO[d]);
    }
    __syncwarp();
  }
  __syncthreads();
  for (int t = threadIdx.x; t < S * D; t += blockDim.x) {
    const int j = t / D, d = t % D;
    st_any(dqkv, base + (long long)j * 3 * A + A + h * D + d, f32, dKs[t]);
    st_any(dqkv, base + (long long)j * 3 * A + 2 * A + h * D + d, f32, dVs[t]);
  }
}
int launch_attn_bwd_generic(const void* dctx, const void* qkv, int f32, void* dqkv, int B, int S, int heads, int D,
                            cudaStream_t st) {
  if (B <= 0) return VIT3D_OK;
  if (S > 32 * ATT_MAXJ) V3_UNSUPPORTED("generic attention supports S <= %d (got %d)", 32 * ATT_MAXJ, S);
  const int threads = 256;
  const size_t smem = attn_generic_smem(S, D, threads / 32, true);
  if (smem > 200 * 1024) V3_UNSUPPORTED("generic attention bwd: S*D too large for shared memory (S=%d D=%d)", S, D);
  if (smem > 48 * 1024)
    V3_CUDA(cudaFuncSetAttribute(attn_bwd_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  attn_bwd_generic_kernel<<<B * heads, threads, smem, st>>>(dctx, qkv, f32, dqkv, B, S, heads, D, 1.0f / sqrtf((float)D));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ elementwise
template <typename F>
__global__ void ew_kernel(long long n, F f) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) f(i);
}
static int ew_blocks(long long n) {
  long long b = (n + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

int launch_gelu_fwd(const void* h, void* a, long long n, int f32, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) { st_any(a, i, f32, gelu_f(ld_any(h, i, f32))); });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
// bf16 fast path: 8 elements per thread (16-byte accesses); gelu_grad_fast (common.cuh) is the derivative of the
// fitted tanh-form GELU the BF16 forward evaluates
// DROP: the Dropout between GELU and fc2 (modeling.py:121) is undone here too - dh = keep * da / (1-p) * gelu'(h)
// with the mask regenerated from (seed, site, step, element index), so training needs no separate dropout
// backward pass over the [M, mlp_dim] gradient.
template <bool DROP>
__global__ void __launch_bounds__(256) gelu_bwd_bf16_kernel(const uint4* __restrict__ da, const uint4* __restrict__ h,
                                                            uint4* __restrict__ dh, long long n8, uint32_t th, float sc,
                                                            unsigned long long seed, unsigned site, unsigned step,
                                                            const unsigned* __restrict__ step_dev) {
  if (DROP && step_dev) step += *step_dev;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n8; q += (long long)gridDim.x * blockDim.x) {
    const uint4 a = da[q], b = h[q];
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
    float keep[8];
    if (DROP) {
      // elements 8q .. 8q+7 = the eight 16-bit lanes of Philox block q (common.cuh dropout_keep)
      const unsigned long long b0 = (unsigned long long)q;
      const Philox4 r0 = philox4x32_10((uint32_t)b0, (uint32_t)(b0 >> 32), site, step, (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
      for (int j = 0; j < 8; ++j) keep[j] = dropout_lane16(r0, j) >= th ? sc : 0.f;
    }
    uint32_t ow[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 av = *reinterpret_cast<const __nv_bfloat162*>(&aw[j]);
      const __nv_bfloat162 hv = *reinterpret_cast<const __nv_bfloat162*>(&bw[j]);
      float g0 = __low2float(av) * gelu_grad_fast(__low2float(hv));
      float g1 = __high2float(av) * gelu_grad_fast(__high2float(hv));
      if (DROP) { g0 *= keep[2 * j]; g1 *= keep[2 * j + 1]; }
      const __nv_bfloat162 o = __floats2bfloat162_rn(g0, g1);
      ow[j] = *reinterpret_cast<const uint32_t*>(&o);
    }
    dh[q] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
  }
}
bool gelu_dropout_bwd_supported(const void* da, const void* h, void* dh, long long n, int f32) {
  const bool aligned = ((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(dh)) & 15) == 0;
  return !f32 && aligned && n % 8 == 0;
}
int launch_gelu_dropout_bwd(const void* da, const void* h, void* dh, long long n, float p, unsigned long long seed,
                            unsigned site, unsigned step, const unsigned* step_dev, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  gelu_bwd_bf16_kernel<true><<<ew_blocks(n / 8), 256, 0, st>>>(
      reinterpret_cast<const uint4*>(da), reinterpret_cast<const uint4*>(h), reinterpret_cast<uint4*>(dh), n / 8,
      dropout_thresh(p), 1.0f / (1.0f - p), seed, site, step, step_dev);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_gelu_bwd(const void* da, const void* h, void* dh, long long n, int f32, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  if (gelu_dropout_bwd_supported(da, h, dh, n, f32)) {
    gelu_bwd_bf16_kernel<false><<<ew_blocks(n / 8), 256, 0, st>>>(reinterpret_cast<const uint4*>(da),
                                                                  reinterpret_cast<const uint4*>(h),
                                                                  reinterpret_cast<uint4*>(dh), n / 8, 0u, 1.f, 0ull, 0u, 0u, nullptr);
    V3_LAUNCH_CHECK();
    return VIT3D_OK;
  }
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(
      n, [=] __device__(long long i) { st_any(dh, i, f32, ld_any(da, i, f32) * gelu_grad_f(ld_any(h, i, f32))); });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
// 4 elements per thread: one Philox block serves 4 consecutive elements; 8/16-byte vector accesses.
template <bool F32>
__global__ void __launch_bounds__(256) dropout4_kernel(const void* __restrict__ x, const void* __restrict__ residual,
                                                       void* __restrict__ y, long long n4, long long n, uint32_t th,
                                                       float sc, unsigned long long seed, unsigned site, unsigned step,
                                                       const unsigned* __restrict__ step_dev) {
  if (step_dev) step += *step_dev;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n4; q += (long long)gridDim.x * blockDim.x) {
    // elements 4q .. 4q+3 = 16-bit lanes 4 (q & 1) .. of Philox block q >> 1 (common.cuh dropout_keep)
    const long long qb = q >> 1;
    const Philox4 r = philox4x32_10((uint32_t)qb, (uint32_t)(qb >> 32), site, step, (uint32_t)seed, (uint32_t)(seed >> 32));
    const int l0 = (int)(q & 1) * 4;
    const long long i = q * 4;
    float v[4], res[4] = {0.f, 0.f, 0.f, 0.f};
    if (i + 3 < n) {
      if (F32) {
        const float4 a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + i);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        if (residual) {
          const float4 b = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(residual) + i);
          res[0] = b.x; res[1] = b.y; res[2] = b.z; res[3] = b.w;
        }
      } else {
        const uint2 a = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(x) + i);
        const __nv_bfloat162 a0 = *reinterpret_cast<const __nv_bfloat162*>(&a.x), a1 = *reinterpret_cast<const __nv_bfloat162*>(&a.y);
        v[0] = __low2float(a0); v[1] = __high2float(a0); v[2] = __low2float(a1); v[3] = __high2float(a1);
        if (residual) {
          const uint2 b = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(residual) + i);
          const __nv_bfloat162 b0 = *reinterpret_cast<const __nv_bfloat162*>(&b.x), b1 = *reinterpret_cast<const __nv_bfloat162*>(&b.y);
          res[0] = __low2float(b0); res[1] = __high2float(b0); res[2] = __low2float(b1); res[3] = __high2float(b1);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = (dropout_lane16(r, l0 + j) >= th ? v[j] * sc : 0.f) + res[j];
      if (F32) {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + i) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
        __nv_bfloat162 o0 = __floats2bfloat162_rn(v[0], v[1]), o1 = __floats2bfloat162_rn(v[2], v[3]);
        uint2 o;
        o.x = *reinterpret_cast<uint32_t*>(&o0); o.y = *reinterpret_cast<uint32_t*>(&o1);
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + i) = o;
      }
    } else {
      for (int j = 0; j < 4 && i + j < n; ++j) {
        float o = dropout_lane16(r, l0 + j) >= th ? ld_any(x, i + j, F32) * sc : 0.f;
        if (residual) o += ld_any(residual, i + j, F32);
        st_any(y, i + j, F32, o);
      }
    }
  }
}
int launch_dropout(const void* x, const void* residual, void* y, long long n, int f32, float p,
                   unsigned long long seed, unsigned site, unsigned step, const unsigned* step_dev, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  const uint32_t th = dropout_thresh(p);
  const float sc = 1.0f / (1.0f - p);
  const long long n4 = (n + 3) / 4;
  const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) |
                         reinterpret_cast<uintptr_t>(residual)) & 15) == 0;
  if (!aligned) { set_error("dropout: buffers must be 16-byte aligned"); return VIT3D_ERR_INVALID; }
  if (f32) dropout4_kernel<true><<<ew_blocks(n4), 256, 0, st>>>(x, residual, y, n4, n, th, sc, seed, site, step, step_dev);
  else dropout4_kernel<false><<<ew_blocks(n4), 256, 0, st>>>(x, residual, y, n4, n, th, sc, seed, site, step, step_dev);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_dropout_mask(unsigned char* mask, long long n, float p, unsigned long long seed, unsigned site, unsigned step,
                        cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  const uint32_t th = dropout_thresh(p);
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(
      n, [=] __device__(long long i) { mask[i] = dropout_keep(seed, site, step, (unsigned long long)i, th) ? 1 : 0; });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_dropout_masked(const void* x, const unsigned char* mask, const void* residual, void* y, long long n,
                          int f32, float p, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  const float sc = 1.0f / (1.0f - p);
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) {
    float o = mask[i] ? ld_any(x, i, f32) * sc : 0.f;
    if (residual) o += ld_any(residual, i, f32);
    st_any(y, i, f32, o);
  });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_cast(const void* x, int x_f32, void* y, int y_f32, long long n, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) { st_any(y, i, y_f32, ld_any(x, i, x_f32)); });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
// y[cols, rows] (bf16) = x[rows, cols]^T (fp32): transposed bf16 shadow of a weight for the dgrad GEMM
__global__ void transpose_cast_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int rows, int cols) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? x[(long long)r * cols + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) y[(long long)c * rows + r] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}
int launch_transpose_cast(const float* x, void* y, int rows, int cols, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return VIT3D_OK;
  dim3 grid(ceil_div(cols, 32), ceil_div(rows, 32));
  transpose_cast_kernel<<<grid, dim3(32, 8), 0, st>>>(x, reinterpret_cast<__nv_bfloat16*>(y), rows, cols);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
// N2: y = float(x_u8) - mean, 16 elements per thread (one 16-byte load, four 16-byte stores)
__global__ void __launch_bounds__(256) u8_to_f32_kernel(const uint8_t* __restrict__ x, float* __restrict__ y, long long n16,
                                                        long long n, float mean) {
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n16; q += (long long)gridDim.x * blockDim.x) {
    const long long i = q * 16;
    if (i + 15 < n) {
      const uint4 v = *reinterpret_cast<const uint4*>(x + i);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<float4*>(y + i + 4 * j) =
            make_float4((float)(w[j] & 255u) - mean, (float)((w[j] >> 8) & 255u) - mean, (float)((w[j] >> 16) & 255u) - mean,
                        (float)(w[j] >> 24) - mean);
    } else {
      for (long long k = i; k < n; ++k) y[k] = (float)x[k] - mean;
    }
  }
}
int launch_u8_to_f32(const uint8_t* x, float* y, long long n, float mean, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) { set_error("u8_to_f32: buffers must be 16-byte aligned"); return VIT3D_ERR_INVALID; }
  const long long n16 = (n + 15) / 16;
  u8_to_f32_kernel<<<ew_blocks(n16), 256, 0, st>>>(x, y, n16, n, mean);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_cast_f16(const float* x, void* y, long long n, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  __half* o = reinterpret_cast<__half*>(y);
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) { o[i] = __float2half_rn(x[i]); });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_round_tf32(const float* x, float* y, long long n, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) { y[i] = round_tf32(x[i]); });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_add_inplace(float* y, const float* x, long long n, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) { y[i] += x[i]; });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ BCE-with-logits (a7)
// loss_i = -(pw*y*logsigmoid(z) + (1-y)*logsigmoid(-z)); mean over n.  Single block (n = batch size).
__device__ __forceinline__ float log_sigmoid(float z) { return fminf(z, 0.f) - log1pf(expf(-fabsf(z))); }

__global__ void __launch_bounds__(256) bce_fwd_kernel(const float* __restrict__ z, const float* __restrict__ y, float pw,
                                                      const float* __restrict__ pw_dev, float* __restrict__ loss, int n) {
  if (pw_dev) pw = *pw_dev;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float w = pw < 0.f ? 1.f : pw;
    acc -= w * y[i] * log_sigmoid(z[i]) + (1.f - y[i]) * log_sigmoid(-z[i]);
  }
  __shared__ float red[8];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w];
    *loss = s / (float)n;
  }
}
__global__ void bce_bwd_kernel(const float* __restrict__ z, const float* __restrict__ y, float pw,
                               const float* __restrict__ pw_dev, const float* __restrict__ dloss, float* __restrict__ dz,
                               int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (pw_dev) pw = *pw_dev;
  const float w = pw < 0.f ? 1.f : pw;
  const float s = 1.f / (1.f + expf(-z[i]));
  // d/dz of -(w y log s + (1-y) log(1-s)) = -(w y (1-s)) + (1-y) s
  const float g = (1.f - y[i]) * s - w * y[i] * (1.f - s);
  dz[i] = g * (dloss ? *dloss : 1.f) / (float)n;
}
int launch_bce_fwd(const float* z, const float* y, float pw, const float* pw_dev, float* loss, int n, cudaStream_t st) {
  bce_fwd_kernel<<<1, 256, 0, st>>>(z, y, pw, pw_dev, loss, n);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_bce_bwd(const float* z, const float* y, float pw, const float* pw_dev, const float* dloss, float* dz, int n,
                   cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  bce_bwd_kernel<<<ceil_div(n, 256), 256, 0, st>>>(z, y, pw, pw_dev, dloss, dz, n);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ meta-classifier (a9)
__global__ void meta_fwd_kernel(const float* __restrict__ f, const float* __restrict__ w, const float* __restrict__ b,
                                float* __restrict__ out, int B, int F, int C) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * C) return;
  const int c = t % C, r = t / C;
  float acc = b[c];
  for (int k = 0; k < F; ++k) acc = fmaf(f[r * F + k], w[c * F + k], acc);
  out[t] = 1.f / (1.f + expf(-acc));
}
// one block: tiny problem (F = members, C = 1)
__global__ void __launch_bounds__(256) meta_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ out,
                                                       const float* __restrict__ f, const float* __restrict__ w,
                                                       float* __restrict__ df, float* __restrict__ dw,
                                                       float* __restrict__ db, int B, int F, int C) {
  // dz = dout * out * (1-out)
  for (int t = threadIdx.x; t < B * F; t += blockDim.x) {
    const int k = t % F, r = t / F;
    float acc = 0.f;
    for (int c = 0; c < C; ++c) {
      const float o = out[r * C + c];
      acc = fmaf(dout[r * C + c] * o * (1.f - o), w[c * F + k], acc);
    }
    df[t] = acc;
  }
  for (int t = threadIdx.x; t < C * F; t += blockDim.x) {
    const int k = t % F, c = t / F;
    float acc = 0.f;
    for (int r = 0; r < B; ++r) {
      const float o = out[r * C + c];
      acc = fmaf(dout[r * C + c] * o * (1.f - o), f[r * F + k], acc);
    }
    dw[t] += acc;
  }
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = 0.f;
    for (int r = 0; r < B; ++r) {
      const float o = out[r * C + c];
      acc += dout[r * C + c] * o * (1.f - o);
    }
    db[c] += acc;
  }
}
int launch_meta_fwd(const float* f, const float* w, const float* b, float* out, int B, int F, int C, cudaStream_t st) {
  if (B * C <= 0) return VIT3D_OK;
  meta_fwd_kernel<<<ceil_div(B * C, 256), 256, 0, st>>>(f, w, b, out, B, F, C);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_meta_bwd(const float* dout, const float* out, const float* f, const float* w, float* df, float* dw, float* db,
                    int B, int F, int C, cudaStream_t st) {
  meta_bwd_kernel<<<1, 256, 0, st>>>(dout, out, f, w, df, dw, db, B, F, C);
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

// ============================================================================ optimizers (N1)
// lr_dev / step_dev (device scalars, may be NULL) override the host values: a captured CUDA graph can
// follow an LR schedule and Adam's bias correction without re-capture.
int launch_sgd(float* p, const float* g, float* mom, long long n, float lr, float momentum, float wd, int first,
               float gscale, const float* lr_dev, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) {
    const float lr_ = lr_dev ? *lr_dev : lr;
    float d = g[i] * gscale + wd * p[i];
    if (momentum != 0.f) {
      const float b = first ? d : momentum * mom[i] + d;
      mom[i] = b;
      d = b;
    }
    p[i] -= lr_ * d;
  });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}
int launch_adam(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps,
                float wd, int step, float gscale, const float* lr_dev, const int* step_dev, cudaStream_t st) {
  if (n <= 0) return VIT3D_OK;
  ew_kernel<<<ew_blocks(n), 256, 0, st>>>(n, [=] __device__(long long i) {
    const float lr_ = lr_dev ? *lr_dev : lr;
    const float t = (float)(step_dev ? *step_dev : step);
    const float bc1 = 1.f - powf(b1, t), bc2 = 1.f - powf(b2, t);
    const float step_size = lr_ / bc1;
    const float inv_sqrt_bc2 = rsqrtf(bc2);
    const float gr = g[i] * gscale + wd * p[i];
    const float mi = b1 * m[i] + (1.f - b1) * gr;
    const float vi = b2 * v[i] + (1.f - b2) * gr * gr;
    m[i] = mi;
    v[i] = vi;
    p[i] -= step_size * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
  });
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

}  // namespace vit3d
