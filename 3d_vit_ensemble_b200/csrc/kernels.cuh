// Internal launcher declarations shared by the translation units of libvit3d_sm100.so.
#pragma once
#include "common.cuh"

namespace vit3d {

struct SgemmArgs {
  const void* A = nullptr; long long sa_m = 0, sa_k = 0; int a_f32 = 1;
  const void* B = nullptr; long long sb_k = 0, sb_n = 0; int b_f32 = 1;
  void* C = nullptr; long long ldc = 0; int c_f32 = 1; int accumulate = 0;
  const float* bias = nullptr;       // per output column
  const float* rowadd = nullptr;     // [row_group+1, N] position table (needs row_group > 0)
  const float* residual = nullptr; long long ldr = 0;
  void* pre = nullptr;               // pre-activation copy (same type as C)
  int act = 0;
  int row_group = 0;                 // >0: output row = m + m/row_group + 1 (leave room for the cls rows)
  int splitk = 1;
  int M = 0, N = 0, K = 0;
};

int launch_sgemm(const SgemmArgs& a, cudaStream_t st);
int pick_splitk(int M, int N, int K);
int launch_rowdot(const float* x, long long ldx, const float* w, const float* bias, float* y, int M, int N, int K,
                  cudaStream_t st);
int launch_patch_gather(const float* x, void* out, int out_f32, int B, int X, int Y, int Z, int p0, int p1, int p2,
                        cudaStream_t st);
int launch_patch_scatter(const float* patches, float* x, int B, int X, int Y, int Z, int p0, int p1, int p2, cudaStream_t st);
int launch_cls_rows(const float* cls, const float* pos, float* tokens, int B, int S, int H, cudaStream_t st);
int launch_embed_param_grads(const float* dtok, float* dpos, float* dcls, int B, int S, int H, cudaStream_t st);
int launch_gather_patch_rows(const float* dtok, void* out, int out_f32, int B, int P, int H, cudaStream_t st);
int launch_ln_fwd(const float* x, const float* g, const float* b, void* y, int y_bf16, float* mean, float* rstd, int M,
                  int H, float eps, cudaStream_t st);
int launch_ln_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                  const float* dres, float* dx, float* dgamma, float* dbeta, int M, int H, cudaStream_t st);
int launch_colsum(const void* dy, int f32, float* db, int M, int N, cudaStream_t st);
int launch_attn_fwd_generic(const void* qkv, int f32, void* ctx, float* probs, int B, int S, int heads, int D,
                            int round_out, cudaStream_t st);
int launch_round_tf32(const float* x, float* y, long long n, cudaStream_t st);
int launch_cast_f16(const float* x, void* y, long long n, cudaStream_t st);
int launch_u8_to_f32(const uint8_t* x, float* y, long long n, float mean, cudaStream_t st);
int launch_transpose_cast(const float* x, void* y, int rows, int cols, cudaStream_t st);
int launch_attn_bwd_generic(const void* dctx, const void* qkv, int f32, void* dqkv, int B, int S, int heads, int D,
                            cudaStream_t st);
int launch_gelu_fwd(const void* h, void* a, long long n, int f32, cudaStream_t st);
int launch_gelu_bwd(const void* da, const void* h, void* dh, long long n, int f32, cudaStream_t st);
bool gelu_dropout_bwd_supported(const void* da, const void* h, void* dh, long long n, int f32);
int launch_gelu_dropout_bwd(const void* da, const void* h, void* dh, long long n, float p, unsigned long long seed,
                            unsigned site, unsigned step, const unsigned* step_dev, cudaStream_t st);
int launch_dropout(const void* x, const void* residual, void* y, long long n, int f32, float p,
                   unsigned long long seed, unsigned site, unsigned step, const unsigned* step_dev, cudaStream_t st);
int launch_dropout_mask(unsigned char* mask, long long n, float p, unsigned long long seed, unsigned site, unsigned step,
                        cudaStream_t st);
int launch_dropout_masked(const void* x, const unsigned char* mask, const void* residual, void* y, long long n,
                          int f32, float p, cudaStream_t st);
int launch_cast(const void* x, int x_f32, void* y, int y_f32, long long n, cudaStream_t st);
int launch_add_inplace(float* y, const float* x, long long n, cudaStream_t st);
int launch_bce_fwd(const float* z, const float* y, float pw, const float* pw_dev, float* loss, int n, cudaStream_t st);
int launch_bce_bwd(const float* z, const float* y, float pw, const float* pw_dev, const float* dloss, float* dz, int n,
                   cudaStream_t st);
int launch_meta_fwd(const float* f, const float* w, const float* b, float* out, int B, int F, int C, cudaStream_t st);
int launch_meta_bwd(const float* dout, const float* out, const float* f, const float* w, float* df, float* dw, float* db,
                    int B, int F, int C, cudaStream_t st);
int launch_sgd(float* p, const float* g, float* mom, long long n, float lr, float momentum, float wd, int first,
               float gscale, const float* lr_dev, cudaStream_t st);
int launch_adam(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps,
                float wd, int step, float gscale, const float* lr_dev, const int* step_dev, cudaStream_t st);

// k_train.cu: bandwidth-bound passes of the fused BF16 training step
int launch_dropout_bits(uint32_t* bits, int nseg, const unsigned* sites, const long long* nelems, float p,
                        unsigned long long seed, unsigned step, const unsigned* step_dev, cudaStream_t st);
int launch_ln256_fwd(const float* x, const uint8_t* bits, float sc, float* xd, const float* gamma, const float* beta,
                     void* y_bf16, float* y_f32, float* mean, float* rstd, int M, float eps, cudaStream_t st);
int launch_ln256_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                     const float* dres, const uint8_t* bits, float sc, int mask_f32, float* dx, void* dxb, float* dgamma,
                     float* dbeta, float* dbias, int M, cudaStream_t st);
int launch_mul_colsum_bwd(const void* da, const void* dact, void* dh, float* db, int M, int d, cudaStream_t st);
int launch_head_bwd(const float* dlogit, const float* enc, const float* w, float* denc, float* dw, float* db, int B, int S,
                    cudaStream_t st);
int launch_wgrad_reduce(const void* host_jobs, int njobs, cudaStream_t st);
int launch_refresh_shadows(const void* jobs, int njobs, int total_tiles, unsigned* step_dev, cudaStream_t st);

}  // namespace vit3d
