// extern "C" surface of libvit3d_sm100.so (declared in include/vit3d.h): argument checks and
// dispatch between the tcgen05 kernels and the shape-generic fp32 kernels.
#include <stdarg.h>

#include "common.cuh"
#include "kernels.cuh"
#include "tc.cuh"

namespace vit3d {

static thread_local char g_err[512] = "";
static unsigned long long g_launches = 0;   // kernels launched by this library (bench.py's gpu_launches)
void count_launch() { __atomic_fetch_add(&g_launches, 1ull, __ATOMIC_RELAXED); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  return VIT3D_ERR_CUDA;
}
int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 148;
    cached = p.multiProcessorCount;
    cached_dev = dev;
  }
  return cached;
}

// tuning switches (test and probe hooks, include/vit3d.h), indexed by key; process-wide, read and written with
// relaxed atomics (the entry points are re-entrant).  Retired keys keep their slot but can be neither set nor read.
static int g_tuning[VIT3D_TUNE_COUNT] = {
    0,  //  0 retired
    0,  //  1 ATTN_THREADS
    0,  //  2 retired
    0,  //  3 retired
    0,  //  4 retired
    0,  //  5 MLP_PAIR
    1,  //  6 WGRAD_RED
    1,  //  7 ATTN_BWD
    0,  //  8 RES_PAIR
    1,  //  9 ATTN_TF32
    0,  // 10 retired
    0,  // 11 PATCH_TALL
    0,  // 12 PATCH_CLUSTER
    0,  // 13 retired
    0,  // 14 ATTN_FWD_UNIT
};
constexpr unsigned kLiveTuningKeys =
    1u << VIT3D_TUNE_ATTN_THREADS | 1u << VIT3D_TUNE_MLP_PAIR | 1u << VIT3D_TUNE_WGRAD_RED | 1u << VIT3D_TUNE_ATTN_BWD |
    1u << VIT3D_TUNE_RES_PAIR | 1u << VIT3D_TUNE_ATTN_TF32 | 1u << VIT3D_TUNE_PATCH_TALL | 1u << VIT3D_TUNE_PATCH_CLUSTER |
    1u << VIT3D_TUNE_ATTN_FWD_UNIT;
static bool tuning_key_live(int key) { return key >= 0 && key < VIT3D_TUNE_COUNT && ((kLiveTuningKeys >> key) & 1u); }
int tuning(int key) {
  return (key >= 0 && key < VIT3D_TUNE_COUNT) ? __atomic_load_n(&g_tuning[key], __ATOMIC_RELAXED) : 0;
}

static inline int act_f32(int prec) { return prec != VIT3D_PREC_BF16; }

}  // namespace vit3d

using namespace vit3d;

extern "C" {

int vit3d_version(void) { return VIT3D_VERSION; }
const char* vit3d_last_error(void) { return g_err; }

int vit3d_device_info(int* sms, int* cc) {
  int dev = 0;
  V3_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  V3_CUDA(cudaGetDeviceProperties(&p, dev));
  if (sms) *sms = p.multiProcessorCount;
  if (cc) *cc = p.major * 10 + p.minor;
  return VIT3D_OK;
}
int vit3d_set_tuning(int key, int value) {
  V3_REQUIRE(tuning_key_live(key), "set_tuning: unknown or retired key %d", key);
  __atomic_store_n(&g_tuning[key], value, __ATOMIC_RELAXED);
  return VIT3D_OK;
}
int vit3d_get_tuning(int key) {
  V3_REQUIRE(tuning_key_live(key), "get_tuning: unknown or retired key %d", key);
  return tuning(key);
}
unsigned long long vit3d_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }
int vit3d_act_bytes(int prec) { return prec == VIT3D_PREC_BF16 ? 2 : 4; }
int vit3d_tc_supported(int prec, int M, int N, int K) { return tc_linear_supported(prec, M, N, K) ? 1 : 0; }

// ------------------------------------------------------------------------- a1
int vit3d_patch_gather(const float* x, float* patches, int B, int X, int Y, int Z, int p0, int p1, int p2,
                       vit3d_stream_t stream) {
  V3_REQUIRE(B >= 0 && p0 > 0 && p1 > 0 && p2 > 0 && X >= p0 && Y >= p1 && Z >= p2, "patch_gather: bad shape");
  if (B == 0) return VIT3D_OK;
  V3_REQUIRE(x && patches, "patch_gather: null pointer");
  return launch_patch_gather(x, patches, 1, B, X, Y, Z, p0, p1, p2, as_stream(stream));
}

size_t vit3d_patch_embed_ws_bytes(int B, int X, int Y, int Z, int p0, int p1, int p2, int H, int prec) {
  (void)prec;
  const size_t P = (size_t)(X / p0) * (Y / p1) * (Z / p2);
  const size_t Kp = (size_t)p0 * p1 * p2;
  // patches [B*P,Kp] + compacted dY [B*P,H] (backward), fp32
  return sizeof(float) * ((size_t)B * P * Kp + (size_t)B * P * H) + 256;
}

int vit3d_patch_embed_fwd(const float* x, const float* w, const float* bias, const float* cls, const float* pos,
                          float* tokens, int B, int X, int Y, int Z, int p0, int p1, int p2, int H, int prec, void* ws,
                          size_t ws_bytes, vit3d_stream_t stream) {
  V3_REQUIRE(x && w && bias && cls && pos && tokens, "patch_embed_fwd: null pointer");
  V3_REQUIRE(B >= 0 && p0 > 0 && p1 > 0 && p2 > 0 && X >= p0 && Y >= p1 && Z >= p2 && H > 0, "patch_embed_fwd: bad shape");
  cudaStream_t st = as_stream(stream);
  const int P = (X / p0) * (Y / p1) * (Z / p2), Kp = p0 * p1 * p2, S = P + 1;
  if (B == 0) return VIT3D_OK;
  // BF16 mode: TF32 tensor-core embedding straight from the volume (5e-4 relative error, far inside the
  // bf16 budget).  TF32 mode is the 1e-3-logit accuracy mode: the raw input cannot be pre-rounded (the
  // tensor core truncates it to 10 mantissa bits), so it keeps the exact fp32 gather + FMA embedding.
  if (prec == VIT3D_PREC_BF16 && tc_patch_embed_supported(B, X, Y, Z, p0, p1, p2, H)) {
    int rc = tc_patch_embed_fwd(x, w, bias, pos, tokens, B, X, Y, Z, p0, p1, p2, H, st);
    if (rc != VIT3D_OK) return rc;
    return launch_cls_rows(cls, pos, tokens, B, S, H, st);
  }
  V3_REQUIRE(ws && ws_bytes >= vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, prec), "patch_embed_fwd: workspace too small");
  if (prec == VIT3D_PREC_TF32 && tc_patch_embed_supported(B, X, Y, Z, p0, p1, p2, H) &&
      (size_t)B * X * Y * Z * sizeof(float) <= ws_bytes) {
    // TF32 mode: the volume is rounded to nearest TF32 into the workspace first (the tensor core would truncate the raw
    // input), then takes the same TMA-im2col tensor-core GEMM as BF16 mode: every GEMM operand of this mode is an
    // RN-rounded TF32 value.  (The SIMT fp32 embedding was 1.78 of the 6.3 ms of a conf-5 batch of 1024.)
    float* xr = reinterpret_cast<float*>(ws);
    int rc = launch_round_tf32(x, xr, (long long)B * X * Y * Z, st);
    if (rc != VIT3D_OK) return rc;
    rc = tc_patch_embed_fwd(xr, w, bias, pos, tokens, B, X, Y, Z, p0, p1, p2, H, st);
    if (rc != VIT3D_OK) return rc;
    return launch_cls_rows(cls, pos, tokens, B, S, H, st);
  }
  float* patches = reinterpret_cast<float*>(ws);
  int rc = launch_patch_gather(x, patches, 1, B, X, Y, Z, p0, p1, p2, st);
  if (rc != VIT3D_OK) return rc;
  SgemmArgs g;
  g.A = patches; g.sa_m = Kp; g.sa_k = 1;
  g.B = w; g.sb_k = 1; g.sb_n = Kp;
  g.C = tokens; g.ldc = H;
  g.bias = bias; g.rowadd = pos; g.row_group = P;
  g.M = B * P; g.N = H; g.K = Kp;
  rc = launch_sgemm(g, st);
  if (rc != VIT3D_OK) return rc;
  return launch_cls_rows(cls, pos, tokens, B, S, H, st);
}

int vit3d_patch_embed_bwd(const float* x, const float* dtokens, float* dw, float* dbias, float* dcls, float* dpos, int B,
                          int X, int Y, int Z, int p0, int p1, int p2, int H, int prec, void* ws, size_t ws_bytes,
                          vit3d_stream_t stream) {
  V3_REQUIRE(x && dtokens && dw && dbias && dcls && dpos, "patch_embed_bwd: null pointer");
  V3_REQUIRE(ws && ws_bytes >= vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, prec), "patch_embed_bwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int P = (X / p0) * (Y / p1) * (Z / p2), Kp = p0 * p1 * p2, S = P + 1;
  if (B == 0) return VIT3D_OK;
  int rc;
  if (prec == VIT3D_PREC_BF16 && tc_wgrad_supported(prec, B * P, H, Kp)) {
    // BF16 mode: bf16 im2col + bf16 dY, weight gradient on tcgen05 (both operands MN-major, split over the
    // B*P token rows, fp32 atomics into dw)
    __nv_bfloat16* patches = reinterpret_cast<__nv_bfloat16*>(ws);
    __nv_bfloat16* dYb = patches + (size_t)B * P * Kp;
    rc = launch_patch_gather(x, patches, 0, B, X, Y, Z, p0, p1, p2, st);
    if (rc != VIT3D_OK) return rc;
    rc = launch_gather_patch_rows(dtokens, dYb, 0, B, P, H, st);
    if (rc != VIT3D_OK) return rc;
    rc = tc_gemm_wgrad(dYb, patches, dw, H, Kp, B * P, st);
    if (rc != VIT3D_OK) return rc;
    rc = launch_colsum(dYb, 0, dbias, B * P, H, st);
    if (rc != VIT3D_OK) return rc;
    return launch_embed_param_grads(dtokens, dpos, dcls, B, S, H, st);
  }
  float* patches = reinterpret_cast<float*>(ws);
  float* dY = patches + (size_t)B * P * Kp;
  rc = launch_patch_gather(x, patches, 1, B, X, Y, Z, p0, p1, p2, st);
  if (rc != VIT3D_OK) return rc;
  rc = launch_gather_patch_rows(dtokens, dY, 1, B, P, H, st);
  if (rc != VIT3D_OK) return rc;
  // dw[H,Kp] += dY^T[H, BP] @ patches[BP, Kp]
  SgemmArgs g;
  g.A = dY; g.sa_m = 1; g.sa_k = H;
  g.B = patches; g.sb_k = Kp; g.sb_n = 1;
  g.C = dw; g.ldc = Kp; g.accumulate = 1;
  g.M = H; g.N = Kp; g.K = B * P;
  g.splitk = pick_splitk(g.M, g.N, g.K);
  rc = launch_sgemm(g, st);
  if (rc != VIT3D_OK) return rc;
  rc = launch_colsum(dY, 1, dbias, B * P, H, st);
  if (rc != VIT3D_OK) return rc;
  return launch_embed_param_grads(dtokens, dpos, dcls, B, S, H, st);
}

int vit3d_patch_embed_dgrad(const float* dtokens, const float* w, const void* w_t_lp, float* dx, int B, int X, int Y, int Z,
                            int p0, int p1, int p2, int H, int prec, void* ws, size_t ws_bytes, vit3d_stream_t stream) {
  V3_REQUIRE(B >= 0 && p0 > 0 && p1 > 0 && p2 > 0 && X >= p0 && Y >= p1 && Z >= p2 && H > 0, "patch_embed_dgrad: bad shape");
  if (B == 0) return VIT3D_OK;
  V3_REQUIRE(dtokens && w && dx, "patch_embed_dgrad: null pointer");
  V3_REQUIRE(ws && ws_bytes >= vit3d_patch_embed_ws_bytes(B, X, Y, Z, p0, p1, p2, H, prec), "patch_embed_dgrad: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int P = (X / p0) * (Y / p1) * (Z / p2), Kp = p0 * p1 * p2, S = P + 1;
  int rc;
  const bool aligned = ((reinterpret_cast<uintptr_t>(dtokens) | reinterpret_cast<uintptr_t>(dx) |
                         reinterpret_cast<uintptr_t>(w_t_lp)) & 15) == 0;
  if (prec != VIT3D_PREC_FP32 && w_t_lp && aligned && tc_patch_dgrad_supported(B, X, Y, Z, p0, p1, p2, H)) {
    // BF16 and TF32 modes: one tcgen05 kernel in TF32, stores straight into dx.  BF16 mode reads the fp32 dtokens as they
    // are (the tensor core truncates them to TF32, as it does the volume in the forward); TF32 mode keeps its rule that
    // every GEMM operand is round-to-nearest TF32 and rounds dtokens into the workspace first.
    const float* a = dtokens;
    if (prec == VIT3D_PREC_TF32) {
      V3_REQUIRE((size_t)B * S * H * sizeof(float) <= ws_bytes, "patch_embed_dgrad: workspace too small");
      float* dr = reinterpret_cast<float*>(ws);
      rc = launch_round_tf32(dtokens, dr, (long long)B * S * H, st);
      if (rc != VIT3D_OK) return rc;
      a = dr;
    }
    return tc_patch_dgrad(a, reinterpret_cast<const float*>(w_t_lp), dx, B, X, Y, Z, p0, p1, p2, H, st);
  }
  // exact fp32: compact the patch rows of dtokens, dpatches[B*P, Kp] = dY[B*P, H] @ w[H, Kp], inverse im2col into dx
  float* patches = reinterpret_cast<float*>(ws);
  float* dY = patches + (size_t)B * P * Kp;
  rc = launch_gather_patch_rows(dtokens, dY, 1, B, P, H, st);
  if (rc != VIT3D_OK) return rc;
  SgemmArgs g;
  g.A = dY; g.sa_m = H; g.sa_k = 1;
  g.B = w; g.sb_k = Kp; g.sb_n = 1;
  g.C = patches; g.ldc = Kp;
  g.M = B * P; g.N = Kp; g.K = H;
  rc = launch_sgemm(g, st);
  if (rc != VIT3D_OK) return rc;
  return launch_patch_scatter(patches, dx, B, X, Y, Z, p0, p1, p2, st);
}

// ------------------------------------------------------------------------- LayerNorm
int vit3d_ln_fwd(const float* x, const float* gamma, const float* beta, void* y, int y_bf16, float* mean, float* rstd,
                 int M, int H, float eps, vit3d_stream_t stream) {
  V3_REQUIRE(x && gamma && beta && y, "ln_fwd: null pointer");
  V3_REQUIRE(M >= 0 && H > 0, "ln_fwd: bad shape");
  return launch_ln_fwd(x, gamma, beta, y, y_bf16, mean, rstd, M, H, eps, as_stream(stream));
}
int vit3d_ln_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                 const float* dres, float* dx, float* dgamma, float* dbeta, int M, int H, vit3d_stream_t stream) {
  V3_REQUIRE(dy && x && mean && rstd && gamma && dx && dgamma && dbeta, "ln_bwd: null pointer");
  V3_REQUIRE(M >= 0 && H > 0 && H <= 8192, "ln_bwd: bad shape");
  return launch_ln_bwd(dy, x, mean, rstd, gamma, dres, dx, dgamma, dbeta, M, H, as_stream(stream));
}

// ------------------------------------------------------------------------- Linear
int vit3d_linear_fwd(const void* x, int ldx, int x_f32, const float* w, const void* w_lp, const float* bias,
                     const float* residual, void* y, int y_f32, void* pre, int act, int M, int N, int K, int prec,
                     vit3d_stream_t stream) {
  V3_REQUIRE(x && w && y, "linear_fwd: null pointer");
  V3_REQUIRE(M >= 0 && N > 0 && K > 0 && ldx >= K, "linear_fwd: bad shape M=%d N=%d K=%d ldx=%d", M, N, K, ldx);
  V3_REQUIRE(!(pre && residual), "linear_fwd: pre-activation output and residual are exclusive");
  cudaStream_t st = as_stream(stream);
  if (M == 0) return VIT3D_OK;
  const int xf = x_f32 || act_f32(prec);
  const int yf = y_f32 || residual != nullptr || act_f32(prec);
  if (prec != VIT3D_PREC_FP32 && tc_linear_supported(prec, M, N, K) && (prec == VIT3D_PREC_TF32 ? xf : !xf) &&
      (prec == VIT3D_PREC_TF32 || w_lp) && ldx == K) {
    TcLinear t;
    t.x = x; t.w = w_lp ? w_lp : (const void*)w; t.bias = bias; t.residual = residual;
    t.y = y; t.y_f32 = yf; t.pre = pre; t.act = act; t.M = M; t.N = N; t.K = K; t.prec = prec;
    return tc_linear_fwd(t, st);
  }
  if (N <= 8 && xf && yf && !residual && !pre && act == VIT3D_ACT_NONE)      // the classification head
    return launch_rowdot(reinterpret_cast<const float*>(x), ldx, w, bias, reinterpret_cast<float*>(y), M, N, K, st);
  SgemmArgs g;
  g.A = x; g.sa_m = ldx; g.sa_k = 1; g.a_f32 = xf;
  g.B = w; g.sb_k = 1; g.sb_n = K; g.b_f32 = 1;
  g.C = y; g.ldc = N; g.c_f32 = yf;
  g.bias = bias; g.residual = residual; g.ldr = N; g.pre = pre; g.act = act;
  g.M = M; g.N = N; g.K = K;
  return launch_sgemm(g, st);
}

int vit3d_linear_ln_supported(int M, int N, int K) { return tc_linear_ln_supported(VIT3D_PREC_BF16, M, N, K) ? 1 : 0; }

int vit3d_linear_ln_fwd(const void* x, const void* w_lp, const float* bias, const float* residual, float* y,
                        const float* gamma, const float* beta, float eps, void* ln_out, float* mean, float* rstd, int M,
                        int N, int K, vit3d_stream_t stream) {
  V3_REQUIRE(x && w_lp && y && gamma && beta && ln_out, "linear_ln_fwd: null pointer");
  V3_REQUIRE(M >= 0 && N > 0 && K > 0, "linear_ln_fwd: bad shape M=%d N=%d K=%d", M, N, K);
  if (M == 0) return VIT3D_OK;
  if (!tc_linear_ln_supported(VIT3D_PREC_BF16, M, N, K))
    V3_UNSUPPORTED("linear_ln_fwd: needs BF16 mode shapes with N == 256 (got M=%d N=%d K=%d)", M, N, K);
  TcLinear t;
  t.x = x; t.w = w_lp; t.bias = bias; t.residual = residual; t.y = y; t.y_f32 = 1; t.M = M; t.N = N; t.K = K;
  t.prec = VIT3D_PREC_BF16;
  t.ln_gamma = gamma; t.ln_beta = beta; t.ln_out = ln_out; t.ln_mean = mean; t.ln_rstd = rstd; t.ln_eps = eps;
  return tc_linear_fwd(t, as_stream(stream));
}

int vit3d_linear_bwd(const void* dy, int dy_f32, const void* x, int ldx, int x_f32, const float* w, const void* w_t_lp,
                     void* dx, int lddx, int dx_f32, float* dw, float* db, int M, int N, int K, int prec,
                     vit3d_stream_t stream) {
  V3_REQUIRE(dy && w, "linear_bwd: null pointer");
  V3_REQUIRE(M >= 0 && N > 0 && K > 0, "linear_bwd: bad shape");
  V3_REQUIRE(!dw || x, "linear_bwd: dw needs x");
  cudaStream_t st = as_stream(stream);
  if (M == 0) return VIT3D_OK;
  const int dyf = dy_f32 || act_f32(prec);
  const int xf = x_f32 || act_f32(prec);
  const int dxf = dx_f32 || act_f32(prec);
  int rc;
  if (dx) {
    // dx[M,K] = dy[M,N] @ w[N,K]
    if (prec == VIT3D_PREC_BF16 && !dyf && w_t_lp && (lddx <= 0 || lddx == K) && tc_linear_supported(prec, M, K, N)) {
      TcLinear t;
      t.x = dy; t.w = w_t_lp; t.y = dx; t.y_f32 = dxf; t.M = M; t.N = K; t.K = N; t.prec = prec;
      rc = tc_linear_fwd(t, st);
    } else {
      SgemmArgs g;
      g.A = dy; g.sa_m = N; g.sa_k = 1; g.a_f32 = dyf;
      g.B = w; g.sb_k = K; g.sb_n = 1; g.b_f32 = 1;
      g.C = dx; g.ldc = lddx > 0 ? lddx : K; g.c_f32 = dxf;
      g.M = M; g.N = K; g.K = N;
      rc = launch_sgemm(g, st);
    }
    if (rc != VIT3D_OK) return rc;
  }
  if (dw) {
    // dw[N,K] += dy^T[N,M] @ x[M,K]
    if (!dyf && !xf && ldx == K && tc_wgrad_supported(prec, M, N, K)) {
      rc = tc_gemm_wgrad(dy, x, dw, N, K, M, st);
    } else {
      SgemmArgs g;
      g.A = dy; g.sa_m = 1; g.sa_k = N; g.a_f32 = dyf;
      g.B = x; g.sb_k = ldx; g.sb_n = 1; g.b_f32 = xf;
      g.C = dw; g.ldc = K; g.c_f32 = 1; g.accumulate = 1;
      g.M = N; g.N = K; g.K = M;
      g.splitk = pick_splitk(g.M, g.N, g.K);
      rc = launch_sgemm(g, st);
    }
    if (rc != VIT3D_OK) return rc;
  }
  if (db) {
    rc = launch_colsum(dy, dyf, db, M, N, st);
    if (rc != VIT3D_OK) return rc;
  }
  return VIT3D_OK;
}

// ------------------------------------------------------------------------- fused MLP
int vit3d_mlp_fwd(const void* xn, const void* w1_lp, const float* b1, const void* w2_lp, const float* b2,
                  const float* residual, float* out, int M, int H, int d, vit3d_stream_t stream) {
  V3_REQUIRE(xn && w1_lp && b1 && w2_lp && b2 && residual && out, "mlp_fwd: null pointer");
  V3_REQUIRE(M >= 0 && H > 0 && d > 0, "mlp_fwd: bad shape");
  if (M == 0) return VIT3D_OK;
  return tc_mlp2_fwd(xn, w1_lp, b1, w2_lp, b2, residual, out, nullptr, nullptr, 0.f, nullptr, 0, M, H, d, as_stream(stream));
}
int vit3d_mlp_supported(int M, int H, int d) { return tc_mlp2_supported(M, H, d) ? 1 : 0; }

int vit3d_mlp_ln_supported(int M, int H, int d) { return tc_mlp2_supported(M, H, d) ? 1 : 0; }
int vit3d_mlp_ln_fwd(const void* xn, const void* w1_lp, const float* b1, const void* w2_h, const float* b2,
                     const float* residual, float* out, const float* gamma, const float* beta, float eps, void* ln_out,
                     int M, int H, int d, vit3d_stream_t stream) {
  V3_REQUIRE(xn && w1_lp && b1 && w2_h && b2 && residual && out && gamma && beta && ln_out, "mlp_ln_fwd: null pointer");
  V3_REQUIRE(M >= 0 && H > 0 && d > 0, "mlp_ln_fwd: bad shape");
  if (M == 0) return VIT3D_OK;
  return tc_mlp2_fwd(xn, w1_lp, b1, w2_h, b2, residual, out, gamma, beta, eps, ln_out, 0, M, H, d, as_stream(stream));
}
int vit3d_mlp_lnf_fwd(const void* xn, const void* w1_lp, const float* b1, const void* w2_h, const float* b2,
                      const float* residual, const float* gamma, const float* beta, float eps, float* ln_out, int M, int H,
                      int d, vit3d_stream_t stream) {
  V3_REQUIRE(xn && w1_lp && b1 && w2_h && b2 && residual && gamma && beta && ln_out, "mlp_lnf_fwd: null pointer");
  V3_REQUIRE(M >= 0 && H > 0 && d > 0, "mlp_lnf_fwd: bad shape");
  if (M == 0) return VIT3D_OK;
  return tc_mlp2_fwd(xn, w1_lp, b1, w2_h, b2, residual, nullptr, gamma, beta, eps, ln_out, 1, M, H, d, as_stream(stream));
}

// ------------------------------------------------------------------------- attention core
int vit3d_attn_fwd(const void* qkv, void* ctx, float* probs, int B, int S, int heads, int D, int prec,
                   vit3d_stream_t stream) {
  V3_REQUIRE(qkv && ctx, "attn_fwd: null pointer");
  V3_REQUIRE(B >= 0 && S > 0 && heads > 0 && D > 0, "attn_fwd: bad shape");
  cudaStream_t st = as_stream(stream);
  if (prec == VIT3D_PREC_BF16 && tc_attn_supported(S, heads, D)) return tc_attn_fwd(qkv, ctx, probs, S, B, S, heads, D, st);
  if (prec == VIT3D_PREC_TF32 && tc_attn_supported(S, heads, D) && tuning(VIT3D_TUNE_ATTN_TF32) != 0)
    return tc_attn_fwd_tf32(reinterpret_cast<const float*>(qkv), reinterpret_cast<float*>(ctx), probs, S, B, S, heads, D, 1, st);
  return launch_attn_fwd_generic(qkv, act_f32(prec), ctx, probs, B, S, heads, D, prec == VIT3D_PREC_TF32, st);
}
int vit3d_attn_fwd_padded(const void* qkv, void* ctx, float* probs, int probs_ld, int B, int S, int heads, int D,
                          vit3d_stream_t stream) {
  V3_REQUIRE(qkv && ctx && probs, "attn_fwd_padded: null pointer");
  V3_REQUIRE(B >= 0 && S > 0 && heads > 0 && D > 0 && probs_ld >= S, "attn_fwd_padded: bad shape");
  if (!tc_attn_supported(S, heads, D)) V3_UNSUPPORTED("attn_fwd_padded: unsupported shape S=%d heads=%d D=%d", S, heads, D);
  return tc_attn_fwd(qkv, ctx, probs, probs_ld, B, S, heads, D, as_stream(stream));
}
int vit3d_attn_padded_supported(int S, int heads, int D) { return tc_attn_supported(S, heads, D) ? 1 : 0; }
int vit3d_attn_bwd(const void* dctx, const void* qkv, void* dqkv, int B, int S, int heads, int D, int prec,
                   vit3d_stream_t stream) {
  V3_REQUIRE(dctx && qkv && dqkv, "attn_bwd: null pointer");
  V3_REQUIRE(B >= 0 && S > 0 && heads > 0 && D > 0, "attn_bwd: bad shape");
  if (prec == VIT3D_PREC_BF16 && tc_attn_supported(S, heads, D)) return tc_attn_bwd(dctx, qkv, dqkv, nullptr, nullptr, nullptr, B, S, heads, D, as_stream(stream));
  return launch_attn_bwd_generic(dctx, qkv, act_f32(prec), dqkv, B, S, heads, D, as_stream(stream));
}

// ------------------------------------------------------------------------- elementwise
int vit3d_gelu_fwd(const void* h, void* a, long long n, int prec, vit3d_stream_t stream) {
  V3_REQUIRE(h && a && n >= 0, "gelu_fwd: bad argument");
  return launch_gelu_fwd(h, a, n, act_f32(prec), as_stream(stream));
}
int vit3d_gelu_bwd(const void* da, const void* h, void* dh, long long n, int prec, vit3d_stream_t stream) {
  V3_REQUIRE(da && h && dh && n >= 0, "gelu_bwd: bad argument");
  return launch_gelu_bwd(da, h, dh, n, act_f32(prec), as_stream(stream));
}
int vit3d_gelu_dropout_bwd(const void* da, const void* h, void* dh, long long n, int prec, float p,
                           unsigned long long seed, unsigned site, unsigned step, const unsigned* step_dev,
                           vit3d_stream_t stream) {
  V3_REQUIRE(da && h && dh && n >= 0 && p >= 0.f && p < 1.f, "gelu_dropout_bwd: bad argument");
  if (!gelu_dropout_bwd_supported(da, h, dh, n, act_f32(prec)))
    V3_UNSUPPORTED("gelu_dropout_bwd: needs bf16 activations, 16-byte aligned buffers and n %% 8 == 0");
  return launch_gelu_dropout_bwd(da, h, dh, n, p, seed, site, step, step_dev, as_stream(stream));
}
int vit3d_dropout(const void* x, const void* residual, void* y, long long n, int is_f32, float p,
                  unsigned long long seed, unsigned site, unsigned step, const unsigned* step_dev,
                  vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0 && p >= 0.f && p < 1.f, "dropout: bad argument");
  return launch_dropout(x, residual, y, n, is_f32, p, seed, site, step, step_dev, as_stream(stream));
}
int vit3d_dropout_mask(unsigned char* mask, long long n, float p, unsigned long long seed, unsigned site, unsigned step,
                       vit3d_stream_t stream) {
  V3_REQUIRE(mask && n >= 0 && p >= 0.f && p < 1.f, "dropout_mask: bad argument");
  return launch_dropout_mask(mask, n, p, seed, site, step, as_stream(stream));
}
int vit3d_dropout_masked(const void* x, const unsigned char* mask, const void* residual, void* y, long long n,
                         int is_f32, float p, vit3d_stream_t stream) {
  V3_REQUIRE(x && mask && y && n >= 0 && p >= 0.f && p < 1.f, "dropout_masked: bad argument");
  return launch_dropout_masked(x, mask, residual, y, n, is_f32, p, as_stream(stream));
}
int vit3d_cast_f32_to_bf16(const float* x, void* y, long long n, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0, "cast: bad argument");
  return launch_cast(x, 1, y, 0, n, as_stream(stream));
}
int vit3d_transpose_f32_to_bf16(const float* x, void* y, int rows, int cols, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && rows >= 0 && cols >= 0, "transpose: bad argument");
  return launch_transpose_cast(x, y, rows, cols, as_stream(stream));
}
int vit3d_u8_to_f32(const unsigned char* x, float* y, long long n, float mean, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0, "u8_to_f32: bad argument");
  return launch_u8_to_f32(x, y, n, mean, as_stream(stream));
}
int vit3d_round_tf32(const float* x, float* y, long long n, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0, "round_tf32: bad argument");
  return launch_round_tf32(x, y, n, as_stream(stream));
}
int vit3d_cast_f32_to_f16(const float* x, void* y, long long n, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0, "cast: bad argument");
  return launch_cast_f16(x, y, n, as_stream(stream));
}
int vit3d_cast_bf16_to_f32(const void* x, float* y, long long n, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0, "cast: bad argument");
  return launch_cast(x, 0, y, 1, n, as_stream(stream));
}
int vit3d_add_inplace(float* y, const float* x, long long n, vit3d_stream_t stream) {
  V3_REQUIRE(x && y && n >= 0, "add_inplace: bad argument");
  return launch_add_inplace(y, x, n, as_stream(stream));
}

// ------------------------------------------------------------------------- loss / meta / optimizers
int vit3d_bce_logits_fwd(const float* logits, const float* labels, float pos_weight, const float* pos_weight_dev,
                         float* loss, int n, vit3d_stream_t stream) {
  V3_REQUIRE(logits && labels && loss && n > 0, "bce_fwd: bad argument");
  return launch_bce_fwd(logits, labels, pos_weight, pos_weight_dev, loss, n, as_stream(stream));
}
int vit3d_bce_logits_bwd(const float* logits, const float* labels, float pos_weight, const float* pos_weight_dev,
                         const float* dloss, float* dlogits, int n, vit3d_stream_t stream) {
  V3_REQUIRE(logits && labels && dlogits && n > 0, "bce_bwd: bad argument");
  return launch_bce_bwd(logits, labels, pos_weight, pos_weight_dev, dloss, dlogits, n, as_stream(stream));
}
int vit3d_meta_fwd(const float* feats, const float* w, const float* b, float* out, int B, int F, int C,
                   vit3d_stream_t stream) {
  V3_REQUIRE(feats && w && b && out && B >= 0 && F > 0 && C > 0, "meta_fwd: bad argument");
  return launch_meta_fwd(feats, w, b, out, B, F, C, as_stream(stream));
}
int vit3d_meta_bwd(const float* dout, const float* out, const float* feats, const float* w, float* dfeats, float* dw,
                   float* db, int B, int F, int C, vit3d_stream_t stream) {
  V3_REQUIRE(dout && out && feats && w && dfeats && dw && db && B >= 0 && F > 0 && C > 0, "meta_bwd: bad argument");
  return launch_meta_bwd(dout, out, feats, w, dfeats, dw, db, B, F, C, as_stream(stream));
}
int vit3d_sgd_step(float* p, const float* g, float* mom, long long n, float lr, float momentum, float weight_decay,
                   int first_step, float grad_scale, const float* lr_dev, vit3d_stream_t stream) {
  V3_REQUIRE(p && g && n >= 0 && (momentum == 0.f || mom), "sgd_step: bad argument");
  return launch_sgd(p, g, mom, n, lr, momentum, weight_decay, first_step, grad_scale, lr_dev, as_stream(stream));
}
int vit3d_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, float grad_scale, const float* lr_dev, const int* step_dev,
                    vit3d_stream_t stream) {
  V3_REQUIRE(p && g && m && v && n >= 0 && (step >= 1 || step_dev), "adam_step: bad argument");
  return launch_adam(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale, lr_dev, step_dev,
                     as_stream(stream));
}

// ------------------------------------------------------------------------- fused BF16 training step (a8)
int vit3d_memset_zero(void* p, size_t bytes, vit3d_stream_t stream) {
  V3_REQUIRE(p || bytes == 0, "memset_zero: null pointer");
  if (bytes == 0) return VIT3D_OK;
  V3_CUDA(cudaMemsetAsync(p, 0, bytes, as_stream(stream)));
  return VIT3D_OK;
}
int vit3d_dropout_bits(uint32_t* bits, int nseg, const unsigned* sites, const long long* nelems, float p,
                       unsigned long long seed, unsigned step, const unsigned* step_dev, vit3d_stream_t stream) {
  V3_REQUIRE(bits && sites && nelems && nseg > 0 && nseg <= VIT3D_MAX_DROP_SEGS && p >= 0.f && p < 1.f,
             "dropout_bits: bad argument");
  for (int i = 0; i < nseg; ++i) V3_REQUIRE(nelems[i] >= 0 && nelems[i] % 32 == 0, "dropout_bits: segment %d is not a multiple of 32 elements", i);
  return launch_dropout_bits(bits, nseg, sites, nelems, p, seed, step, step_dev, as_stream(stream));
}
int vit3d_ln256_fwd(const float* x, const void* drop_bits, float drop_scale, float* x_dropped, const float* gamma,
                    const float* beta, void* y_bf16, float* y_f32, float* mean, float* rstd, int M, float eps,
                    vit3d_stream_t stream) {
  V3_REQUIRE(x && gamma && beta && (y_bf16 || y_f32) && M >= 0, "ln256_fwd: bad argument");
  V3_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(x_dropped) | reinterpret_cast<uintptr_t>(y_bf16) |
               reinterpret_cast<uintptr_t>(y_f32) | reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) == 0,
             "ln256_fwd: buffers must be 16-byte aligned");
  return launch_ln256_fwd(x, reinterpret_cast<const uint8_t*>(drop_bits), drop_scale, x_dropped, gamma, beta, y_bf16, y_f32,
                          mean, rstd, M, eps, as_stream(stream));
}
int vit3d_ln256_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                    const float* dres, const void* drop_bits, float drop_scale, int mask_f32, float* dx, void* dx_bf16,
                    float* dgamma, float* dbeta, float* dbias, int M, vit3d_stream_t stream) {
  V3_REQUIRE(dy && x && mean && rstd && gamma && (dx || dx_bf16) && M >= 0, "ln256_bwd: bad argument");
  V3_REQUIRE(((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dres) |
               reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dx_bf16) | reinterpret_cast<uintptr_t>(gamma)) & 15) == 0,
             "ln256_bwd: buffers must be 16-byte aligned");
  return launch_ln256_bwd(dy, x, mean, rstd, gamma, dres, reinterpret_cast<const uint8_t*>(drop_bits), drop_scale, mask_f32, dx,
                          dx_bf16, dgamma, dbeta, dbias, M, as_stream(stream));
}
int vit3d_mul_colsum_bwd(const void* da, const void* dact, void* dh, float* db, int M, int d, vit3d_stream_t stream) {
  V3_REQUIRE(da && dact && dh && M >= 0 && d > 0 && d % 8 == 0, "mul_colsum_bwd: bad argument");
  V3_REQUIRE(((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(dact) | reinterpret_cast<uintptr_t>(dh)) & 15) == 0,
             "mul_colsum_bwd: buffers must be 16-byte aligned");
  return launch_mul_colsum_bwd(da, dact, dh, db, M, d, as_stream(stream));
}
int vit3d_head_bwd(const float* dlogits, const float* encoded, const float* w, float* dencoded, float* dw, float* db, int B,
                   int S, int H, vit3d_stream_t stream) {
  V3_REQUIRE(dlogits && encoded && w && dencoded && dw && db && B >= 0 && S > 0, "head_bwd: bad argument");
  if (H != 256) V3_UNSUPPORTED("head_bwd: hidden size 256 only (got %d)", H);
  return launch_head_bwd(dlogits, encoded, w, dencoded, dw, db, B, S, as_stream(stream));
}
int vit3d_refresh_shadows(const void* jobs, int njobs, int total_tiles, unsigned* step_dev, vit3d_stream_t stream) {
  V3_REQUIRE(jobs && njobs > 0 && total_tiles > 0, "refresh_shadows: bad argument");
  return launch_refresh_shadows(jobs, njobs, total_tiles, step_dev, as_stream(stream));
}
int vit3d_fc1_train_fwd(const void* xn, const void* w1_lp, const float* b1, void* dact, void* act, const void* drop_bits,
                        float drop_scale, int M, int d, int H, vit3d_stream_t stream) {
  V3_REQUIRE(xn && w1_lp && b1 && dact && act && M >= 0 && d > 0 && H > 0, "fc1_train_fwd: bad argument");
  if (M == 0) return VIT3D_OK;
  if (!tc_linear_supported(VIT3D_PREC_BF16, M, d, H) || d % 32) V3_UNSUPPORTED("fc1_train_fwd: unsupported shape M=%d d=%d H=%d", M, d, H);
  TcLinear t;
  t.x = xn; t.w = w1_lp; t.bias = b1; t.y = act; t.y_f32 = 0; t.pre = dact; t.act = VIT3D_ACT_GELU; t.M = M; t.N = d; t.K = H;
  t.prec = VIT3D_PREC_BF16;
  t.drop_bits = reinterpret_cast<const uint32_t*>(drop_bits); t.drop_scale = drop_bits ? drop_scale : 1.f;
  t.store_dact = 1;
  return tc_linear_fwd(t, as_stream(stream));
}
int vit3d_linear_res_train_fwd(const void* x, const void* w_lp, const float* bias, const float* residual, float* y,
                               const void* drop_bits, float drop_scale, const float* gamma, const float* beta, float eps,
                               void* ln_out, float* mean, float* rstd, int M, int N, int K, vit3d_stream_t stream) {
  V3_REQUIRE(x && w_lp && bias && residual && y && M >= 0 && N > 0 && K > 0, "linear_res_train_fwd: bad argument");
  V3_REQUIRE(!ln_out || (gamma && beta), "linear_res_train_fwd: LayerNorm needs gamma and beta");
  if (M == 0) return VIT3D_OK;
  if (!tc_res_supported(M, N, K, ln_out != nullptr))
    V3_UNSUPPORTED("linear_res_train_fwd: unsupported shape M=%d N=%d K=%d", M, N, K);
  TcLinear t;
  t.x = x; t.w = w_lp; t.bias = bias; t.residual = residual; t.y = y; t.y_f32 = 1; t.M = M; t.N = N; t.K = K;
  t.prec = VIT3D_PREC_BF16;
  t.ln_gamma = gamma; t.ln_beta = beta; t.ln_out = ln_out; t.ln_mean = mean; t.ln_rstd = rstd; t.ln_eps = eps;
  t.drop_bits = reinterpret_cast<const uint32_t*>(drop_bits); t.drop_scale = drop_scale;
  return tc_gemm_res(t, as_stream(stream));
}
int vit3d_wgrad(const void* dy, const void* x, float* dw0, float* dw1, float* dw2, int seg_rows, int M, int N, int K,
                vit3d_stream_t stream) {
  V3_REQUIRE(dy && x && dw0 && M >= 0 && N > 0 && K > 0, "wgrad: bad argument");
  if (M == 0) return VIT3D_OK;
  if (!tc_wgrad_supported(VIT3D_PREC_BF16, M, N, K)) V3_UNSUPPORTED("wgrad: unsupported shape M=%d N=%d K=%d", M, N, K);
  return tc_gemm_wgrad_seg(dy, x, dw0, dw1, dw2, seg_rows, N, K, M, as_stream(stream));
}
size_t vit3d_wgrad_ws_bytes(int M, int N, int K) {
  int bn, splits, tiles;
  tc_wgrad_plan(N, K, M, &bn, &splits, &tiles);
  return (size_t)tiles * splits * 128 * bn * sizeof(float);
}
int vit3d_wgrad_partial(const void* dy, const void* x, float* ws, int M, int N, int K, int* bn, int* splits,
                        vit3d_stream_t stream) {
  V3_REQUIRE(dy && x && ws && M > 0 && N > 0 && K > 0, "wgrad_partial: bad argument");
  if (!tc_wgrad_supported(VIT3D_PREC_BF16, M, N, K) || N % 128) V3_UNSUPPORTED("wgrad_partial: unsupported shape M=%d N=%d K=%d", M, N, K);
  tc_wgrad_plan(N, K, M, bn, splits, nullptr);
  return tc_gemm_wgrad_partial(dy, x, ws, N, K, M, as_stream(stream));
}
int vit3d_wgrad_reduce(const void* host_jobs, int njobs, vit3d_stream_t stream) {
  V3_REQUIRE(host_jobs && njobs >= 0 && njobs <= VIT3D_MAX_WGRAD_JOBS, "wgrad_reduce: bad argument");
  return launch_wgrad_reduce(host_jobs, njobs, as_stream(stream));
}
int vit3d_attn_bwd_bias(const void* dctx, const void* qkv, void* dqkv, float* db_q, float* db_k, float* db_v, int B, int S,
                        int heads, int D, vit3d_stream_t stream) {
  V3_REQUIRE(dctx && qkv && dqkv && db_q && db_k && db_v, "attn_bwd_bias: null pointer");
  V3_REQUIRE(B >= 0 && S > 0 && heads > 0 && D > 0, "attn_bwd_bias: bad shape");
  if (!tc_attn_supported(S, heads, D)) V3_UNSUPPORTED("attn_bwd_bias: unsupported shape S=%d heads=%d D=%d", S, heads, D);
  return tc_attn_bwd(dctx, qkv, dqkv, db_q, db_k, db_v, B, S, heads, D, as_stream(stream));
}
int vit3d_mlp_bwd_supported(int M, int H, int d) { return tc_mlp_bwd_supported(M, H, d) ? 1 : 0; }
int vit3d_mlp_bwd(const void* gy, const void* w2_t_lp, const void* w1_t_lp, const void* dact, void* dh, float* dxn, float* db1,
                  int M, int H, int d, vit3d_stream_t stream) {
  V3_REQUIRE(gy && w2_t_lp && w1_t_lp && dact && dh && dxn && M >= 0 && H > 0 && d > 0, "mlp_bwd: bad argument");
  V3_REQUIRE(((reinterpret_cast<uintptr_t>(gy) | reinterpret_cast<uintptr_t>(dh) | reinterpret_cast<uintptr_t>(dxn)) & 15) == 0,
             "mlp_bwd: buffers must be 16-byte aligned");
  if (M == 0) return VIT3D_OK;
  return tc_mlp_bwd(gy, w2_t_lp, w1_t_lp, dact, dh, dxn, db1, M, H, d, as_stream(stream));
}
int vit3d_train_supported(int B, int S, int H, int heads, int d) {
  if (B <= 0 || H != 256 || heads <= 0 || H % heads) return 0;
  const int M = B * S;
  return tc_attn_supported(S, heads, H / heads) && tc_res_supported(M, H, H, true) && tc_res_supported(M, H, d, true) &&
                 tc_linear_supported(VIT3D_PREC_BF16, M, d, H) && d % 64 == 0 && tc_wgrad_supported(VIT3D_PREC_BF16, M, d, H)
             ? 1 : 0;
}

}  // extern "C"
