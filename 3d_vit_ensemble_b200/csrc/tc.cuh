// tcgen05 / TMA / mma.sync tensor-core kernels (sm_100a): internal interface.
#pragma once
#include "common.cuh"

namespace vit3d {

struct TcLinear {
  const void* x = nullptr;       // [M,K] bf16 (BF16) or fp32 (TF32), row-major, dense
  const void* w = nullptr;       // [N,K] same element type as x
  const float* bias = nullptr;   // [N] or null
  const float* residual = nullptr;  // [M,N] fp32 or null
  void* y = nullptr;             // [M,N] fp32 (y_f32) or bf16
  int y_f32 = 0;
  void* pre = nullptr;           // optional pre-activation copy, same type as y
  int act = 0;
  int M = 0, N = 0, K = 0, prec = 0;
  // optional LayerNorm of the finished rows fused into the epilogue (BF16 mode, N == 256, fp32 y):
  const float* ln_gamma = nullptr;
  const float* ln_beta = nullptr;
  void* ln_out = nullptr;        // [M,N] bf16
  float* ln_mean = nullptr;      // [M] optional
  float* ln_rstd = nullptr;      // [M] optional
  float ln_eps = 1e-6f;
  // training: Dropout of (x W^T + b) (fp32 outputs: before the residual add, modeling.py:123,:196) or of the
  // activation (bf16 outputs, modeling.py:121) from a keep-bit array over the [M,N] output
  const uint32_t* drop_bits = nullptr;
  float drop_scale = 1.f;
  int store_dact = 0;            // training fc1: `pre` receives gelu'(pre) * keep * drop_scale (TcEpilogue::store_dact)
};
bool tc_linear_ln_supported(int prec, int M, int N, int K);
// k_tc_gemm_res.cu: fp32 output (+ bias, + residual, + fused LayerNorm) through TMA panels; N % 256 == 0
bool tc_res_supported(int M, int N, int K, bool ln);
int tc_gemm_res(const TcLinear& t, cudaStream_t st);

bool tc_linear_supported(int prec, int M, int N, int K);
int tc_linear_fwd(const TcLinear& t, cudaStream_t st);

// dW[N,K] += dY[M,N]^T X[M,K]  (bf16 operands, fp32 atomics)
bool tc_wgrad_supported(int prec, int M, int N, int K);
int tc_gemm_wgrad(const void* dy, const void* x, float* dw, int N, int K, int M, cudaStream_t st);
void tc_wgrad_plan(int N, int K, int M, int* bn, int* splits, int* tiles);
int tc_gemm_wgrad_partial(const void* dy, const void* x, float* ws, int N, int K, int M, cudaStream_t st);
int tc_gemm_wgrad_seg(const void* dy, const void* x, float* dw0, float* dw1, float* dw2, int seg_rows, int N, int K, int M,
                      cudaStream_t st);

bool tc_patch_embed_supported(int B, int X, int Y, int Z, int p0, int p1, int p2, int H);
int tc_patch_embed_fwd(const float* x, const float* w, const float* bias, const float* pos, float* tokens, int B, int X,
                       int Y, int Z, int p0, int p1, int p2, int H, cudaStream_t st);
// k_tc_patch_dgrad.cu: dx = d tokens / d x on tcgen05 (TF32), straight into the volume by 5-D TMA stores; w_t is the
// TF32-rounded transposed filter bank [Kp, H]
bool tc_patch_dgrad_supported(int B, int X, int Y, int Z, int p0, int p1, int p2, int H);
int tc_patch_dgrad(const float* dtokens, const float* w_t, float* dx, int B, int X, int Y, int Z, int p0, int p1, int p2,
                   int H, cudaStream_t st);

// k_tc_mlp3.cu: the fused MLP block with 128-column chunks, fc1 accumulator and GELU tile double buffered (same contract
// as tc_mlp2_fwd)
bool tc_mlp3_supported(int M, int H, int d);
int tc_mlp3(const void* xn, const void* w1, const float* b1, const void* w2_h, const float* b2, const float* residual,
            float* y, const float* gamma, const float* beta, float eps, void* ln_out, int ln_f32, int M, int H, int d,
            cudaStream_t st);
// k_tc_mlp2.cu: chunked fused MLP (256 fc1 columns per chunk, optional CTA pairs), + residual, + fused LayerNorm
bool tc_mlp2_supported(int M, int H, int d);
int tc_mlp2_fwd(const void* xn, const void* w1, const float* b1, const void* w2_h, const float* b2, const float* residual,
                float* y, const float* gamma, const float* beta, float eps, void* ln_out, int ln_f32, int M, int H, int d,
                cudaStream_t st);

// k_tc_mlp_bwd.cu: fused data-gradient chain of the MLP backward (dgrad fc2 -> GELU' x dropout mask -> dgrad fc1)
bool tc_mlp_bwd_supported(int M, int H, int d);
int tc_mlp_bwd(const void* gy, const void* w2_t, const void* w1_t, const void* dact, void* dh, float* dxn, float* db1, int M,
               int H, int d, cudaStream_t st);

bool tc_attn_supported(int S, int heads, int D);
// probs_ld: floats per probability row (S = the packed layout of the reference tensor; a multiple of 8 = padded rows)
int tc_attn_fwd(const void* qkv, void* ctx, float* probs, int probs_ld, int B, int S, int heads, int D, cudaStream_t st);
// TF32 mode: fp32 q | k | v and context, mma.sync tf32 (k_tc_attn.cu); round_out: context rounded to tf32
int tc_attn_fwd_tf32(const float* qkv, float* ctx, float* probs, int probs_ld, int B, int S, int heads, int D, int round_out,
                     cudaStream_t st);
// db_q / db_k / db_v (each [heads*D] fp32, all or none): += column sums of dq / dk / dv (the q, k, v bias gradients)
int tc_attn_bwd(const void* dctx, const void* qkv, void* dqkv, float* db_q, float* db_k, float* db_v, int B, int S,
                int heads, int D, cudaStream_t st);

}  // namespace vit3d
