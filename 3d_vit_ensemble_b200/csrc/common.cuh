// Shared device/host helpers for libvit3d_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/vit3d.h"

namespace vit3d {

// ----------------------------------------------------------------------------- errors
// Thread-local last-error text; every extern "C" entry returns an int code and never throws.
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define V3_CUDA(call)                                                         \
  do {                                                                        \
    cudaError_t e__ = (call);                                                 \
    if (e__ != cudaSuccess) return ::vit3d::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

void count_launch();
#define V3_LAUNCH_CHECK()                                                     \
  do {                                                                        \
    ::vit3d::count_launch();                                                  \
    cudaError_t e__ = cudaPeekAtLastError();                                  \
    if (e__ != cudaSuccess) return ::vit3d::cuda_fail(e__, "kernel launch", __FILE__, __LINE__); \
  } while (0)

#define V3_REQUIRE(cond, ...)                                                 \
  do {                                                                        \
    if (!(cond)) {                                                            \
      ::vit3d::set_error(__VA_ARGS__);                                        \
      return VIT3D_ERR_INVALID;                                               \
    }                                                                         \
  } while (0)

#define V3_UNSUPPORTED(...)                                                   \
  do {                                                                        \
    ::vit3d::set_error(__VA_ARGS__);                                          \
    return VIT3D_ERR_UNSUPPORTED;                                             \
  } while (0)

static inline cudaStream_t as_stream(vit3d_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }
int sm_count();
// run-time tuning switches (test and probe hooks set by vit3d_set_tuning, see include/vit3d.h)
int tuning(int key);

// ----------------------------------------------------------------------------- programmatic dependent launch
// Kernels launched with launch_pdl() may start while the previous kernel in the stream is still draining:
// everything before pdl_wait() (barrier init, TMEM allocation, descriptor prefetch, smem carve-up) overlaps
// the predecessor's tail; pdl_wait() returns once the predecessor has completed and its writes are visible.
// No global memory may be read OR written before pdl_wait().  pdl_trigger() lets the NEXT kernel's CTAs be
// scheduled as soon as this kernel's CTAs free their SMs.  Captured into CUDA graphs as programmatic edges.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// same, as thread-block clusters of `cluster` CTAs along x (grid.x must be a multiple of it)
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                             int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  attr[1].id = cudaLaunchAttributeClusterDimension;
  attr[1].val.clusterDim.x = (unsigned)cluster;
  attr[1].val.clusterDim.y = 1;
  attr[1].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cluster > 1 ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ----------------------------------------------------------------------------- device math
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// round-to-nearest fp32 -> tf32 (10-bit mantissa) kept in an fp32 container.  tcgen05 kind::tf32 ignores
// the low 13 mantissa bits (truncation); pre-rounding GEMM operands halves the error and removes its bias.
__device__ __forceinline__ float round_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// exact (erf) GELU, as torch.nn.functional.gelu default (modeling.py:52,107)
__device__ __forceinline__ float gelu_f(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_grad_f(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// derivative of the fitted tanh-form GELU the BF16 forward evaluates, y = 0.5 x (1 + tanh(u)),
// u = x (c0 + c1 x^2 + c2 x^4):   y' = 0.5 (1 + t) + 0.5 x (1 - t^2) (c0 + 3 c1 x^2 + 5 c2 x^4)
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float x2 = fminf(x * x, 100.f);
  const float u = x * fmaf(x2, fmaf(x2, -3.58732362e-4f, 0.0370503451f), 0.797458471f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float du = fmaf(x2, fmaf(x2, 5.f * -3.58732362e-4f, 3.f * 0.0370503451f), 0.797458471f);
  return 0.5f * (1.f + t) + 0.5f * x * (1.f - t * t) * du;
}

// ----------------------------------------------------------------------------- Philox4x32-10
// Counter-based RNG for dropout: the mask of element i at (site, step) is a pure function
// of (seed, site, step, i), so backward regenerates it instead of storing it.
struct Philox4 {
  uint32_t v[4];
};
__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}
__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
    const uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  Philox4 o;
  o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}
// keep-decision for element index i (64-bit) of dropout site `site` at step `step`.  One Philox block serves EIGHT
// consecutive elements: element i reads 16-bit lane (i & 7) of block (i >> 3) - lane 2k = low half of word k, lane
// 2k+1 = its high half - and is kept when the lane is >= thresh16, so P(keep) = 1 - thresh16 / 65536 (p = 0.1 ->
// 0.100006).  Halving the Philox calls per element matters: a conf-18 step at batch 256 draws 4.4e8 decisions.
__host__ __device__ __forceinline__ uint32_t dropout_lane16(const Philox4& r, int lane) {
  const uint32_t w = r.v[lane >> 1];
  return (lane & 1) ? (w >> 16) : (w & 0xffffu);
}
__host__ __device__ __forceinline__ bool dropout_keep(unsigned long long seed, uint32_t site, uint32_t step,
                                                      unsigned long long i, uint32_t thresh16) {
  const unsigned long long blk = i >> 3;
  Philox4 r = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), site, step, (uint32_t)seed, (uint32_t)(seed >> 32));
  return dropout_lane16(r, (int)(i & 7)) >= thresh16;
}
static inline uint32_t dropout_thresh(float p) {
  double t = (double)p * 65536.0 + 0.5;
  if (t < 0) t = 0;
  if (t > 65535.0) t = 65535.0;
  return (uint32_t)t;
}

}  // namespace vit3d
