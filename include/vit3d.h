/* vit3d.h — C ABI of libvit3d_sm100.so
 *
 * B200 (sm_100a) kernels for the 3D-ViT stacking-ensemble forward/backward path of
 * evapachetti/3d_vit_ensemble `models/modeling.py`.  The reference has no FFI for this
 * path (it is pure PyTorch, SURVEY.md §8b): the drop-in boundary is the Python class
 * surface of `models/modeling.py`, and these entry points are what that surface binds
 * underneath (ctypes stub: 3d_vit_ensemble_b200/_lib.py; see INTEGRATION.md).
 * Each function cites the reference code whose arithmetic it replaces.
 *
 * Conventions
 *   - plain pointers + sizes; all pointers are DEVICE pointers unless stated otherwise.
 *   - ownership: the caller allocates every input, output, saved-for-backward buffer and
 *     workspace.  The library owns no device memory.
 *   - every call is asynchronous on `stream` (a cudaStream_t), never synchronises, never
 *     uses the default stream implicitly and is CUDA-graph capturable.
 *   - return 0 on success, negative on error; message via vit3d_last_error() (thread local).
 *   - "token matrix": activations are row-major [M, H] with M = B*S rows (S = patches+1,
 *     row b*S is the cls token of volume b) exactly as the reference's (B,S,H) tensors.
 *   - precision modes (`prec`):
 *        VIT3D_PREC_FP32  every contraction in fp32 FMA (any shape; the exact path)
 *        VIT3D_PREC_TF32  tcgen05 kind::tf32, fp32 storage
 *        VIT3D_PREC_BF16  tcgen05 kind::f16 (bf16 operands, fp32 accumulate in TMEM);
 *                         GEMM operand activations are stored bf16, the residual stream,
 *                         LayerNorm statistics, softmax and every gradient of a parameter fp32.
 *     "act" below means: float for FP32/TF32, __nv_bfloat16 for BF16 (vit3d_act_bytes()).
 *   - parameter gradients are ACCUMULATED (+=) into the buffers passed in.
 */
#ifndef VIT3D_H_
#define VIT3D_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif
#ifdef __cplusplus
extern "C" {
#endif

#define VIT3D_VERSION 100

typedef void* vit3d_stream_t; /* cudaStream_t */

enum { VIT3D_OK = 0, VIT3D_ERR_INVALID = -1, VIT3D_ERR_UNSUPPORTED = -2, VIT3D_ERR_CUDA = -3 };
enum { VIT3D_PREC_FP32 = 0, VIT3D_PREC_TF32 = 1, VIT3D_PREC_BF16 = 2 };
enum { VIT3D_ACT_NONE = 0, VIT3D_ACT_GELU = 1 };

int vit3d_version(void);
const char* vit3d_last_error(void);
/* sm count and compute capability (major*10+minor) of the current device */
int vit3d_device_info(int* sm_count, int* cc);
/* number of kernels this library has launched in this process so far */
unsigned long long vit3d_launch_count(void);
/* Tuning switches: test and probe hooks, not user options.  Each selects between kernel variants that agree to
 * rounding, so that tests can check every variant and probes can time them in one process.  Process-wide; the
 * defaults below are the variants in use, and only vit3d_set_tuning changes them.  Keys 0, 2, 3, 4, 10 and 13 are
 * retired: vit3d_set_tuning and vit3d_get_tuning return VIT3D_ERR_INVALID for them (as for any unknown key).
 *   VIT3D_TUNE_ATTN_THREADS  0 (default: chosen per shape), 640 or 512 threads per attention-forward CTA.
 *   VIT3D_TUNE_MLP_PAIR      0 (default): one CTA per 128-row tile of the fused MLP; 1: clusters of two CTAs that
 *                            share every weight k-block by TMA multicast (half the L2 reads; measured equal -
 *                            the kernel is bound by its GELU / final epilogue, not by L2); 2: cta_group::2 pairs; 3: the
 *                            128-column-chunk kernel with double-buffered fc1 accumulator and GELU tile (k_tc_mlp3.cu,
 *                            measured equal).
 *   VIT3D_TUNE_WGRAD_RED     1 (default): split-K weight-gradient tiles are added into the gradient buffer by the
 *                            TMA unit (cp.reduce.async.bulk.tensor, fp32 add at the L2); 0: red.global.add.v4.f32
 *                            from the epilogue warps (~1 element per clock and SM); 2: as 1 with 256-row tiles for the large
 *                            products (measured equal).
 *   VIT3D_TUNE_RES_PAIR      0 (default): independent CTAs; 1: deep-K Linear + residual + LayerNorm products (fc2) run
 *                            on clusters of two CTAs that share every weight k-block by TMA multicast (measured
 *                            equal: not bound by L2 operand delivery).
 *   VIT3D_TUNE_ATTN_TF32     1 (default): TF32-mode attention forward (65 tokens, 256 channels) on mma.sync tf32 in
 *                            (volume, 4-head) units; 0: the generic fp32 SIMT kernel.
 *   VIT3D_TUNE_PATCH_TALL    0 (default): 128-row tiles; 1: the TF32 patch-embedding GEMM of large batches runs 256-row
 *                            tiles (two TMEM accumulators sharing each weight k-block; measured 124 vs 117 us at
 *                            batch 1024).
 *   VIT3D_TUNE_PATCH_CLUSTER 0 (default): independent CTAs; 2 / 4: the patch-embedding GEMM of large batches runs on
 *                            clusters of 2 / 4 CTAs that fetch every filter-bank k-block once (TMA multicast; measured
 *                            equal).
 *   VIT3D_TUNE_ATTN_FWD_UNIT bf16 attention forward: 0 (default) one volume per CTA (bulk-copy staged); 1 (volume, 4-head)
 *                            units with TMA boxes when no probabilities are written; 2 always.
 *   VIT3D_TUNE_ATTN_BWD      1 (default): attention backward in (volume, 4-head) units, 4-warp CTAs, TMA boxes; 0: one
 *                            16-warp CTA per volume with per-row bulk copies. */
enum { VIT3D_TUNE_ATTN_THREADS = 1, VIT3D_TUNE_MLP_PAIR = 5, VIT3D_TUNE_WGRAD_RED = 6, VIT3D_TUNE_ATTN_BWD = 7,
       VIT3D_TUNE_RES_PAIR = 8, VIT3D_TUNE_ATTN_TF32 = 9, VIT3D_TUNE_PATCH_TALL = 11, VIT3D_TUNE_PATCH_CLUSTER = 12,
       VIT3D_TUNE_ATTN_FWD_UNIT = 14, VIT3D_TUNE_COUNT = 15 };
int vit3d_set_tuning(int key, int value);
int vit3d_get_tuning(int key);
/* bytes per "act" element for a precision mode */
int vit3d_act_bytes(int prec);
/* 1 if the tcgen05 path serves a [M,N,K] linear in this precision, else the fp32 FMA path is used */
int vit3d_tc_supported(int prec, int M, int N, int K);

/* ---------------------------------------------------------------- a1: Embeddings
 * Conv3d(1->H, kernel=stride=(p0,p1,p2)) + flatten(2).transpose + cat(cls) + position add
 * (modeling.py:153-156,162-173).  x is (B,1,X,Y,Z) fp32 contiguous. */

/* bit-exact im2col permutation: patches[(b*P+p), (i*p1+j)*p2+z], p=(px*ny+py)*nz+pz */
int vit3d_patch_gather(const float* x, float* patches, int B, int X, int Y, int Z, int p0, int p1, int p2,
                       vit3d_stream_t stream);
/* tokens[B,S,H] = cat(cls, patches @ w^T + bias) + pos ; w is the Conv3d weight viewed [H, p0*p1*p2].
 * ws: >= vit3d_patch_embed_ws_bytes() scratch. */
size_t vit3d_patch_embed_ws_bytes(int B, int X, int Y, int Z, int p0, int p1, int p2, int H, int prec);
int vit3d_patch_embed_fwd(const float* x, const float* w, const float* bias, const float* cls, const float* pos,
                          float* tokens, int B, int X, int Y, int Z, int p0, int p1, int p2, int H, int prec,
                          void* ws, size_t ws_bytes, vit3d_stream_t stream);
/* grads of a1 w.r.t. w, bias, cls, pos (accumulated) from dtokens[B,S,H] */
int vit3d_patch_embed_bwd(const float* x, const float* dtokens, float* dw, float* dbias, float* dcls, float* dpos,
                          int B, int X, int Y, int Z, int p0, int p1, int p2, int H, int prec,
                          void* ws, size_t ws_bytes, vit3d_stream_t stream);
/* dx[B,1,X,Y,Z] = d tokens / d x  (written, not accumulated; uncovered voxels get 0).
 * w_t_lp: the filter bank TRANSPOSED, [Kp, H]: TF32-rounded fp32 (BF16 / TF32 modes) or NULL (FP32 mode, uses w).
 * ws as for vit3d_patch_embed_fwd (vit3d_patch_embed_ws_bytes).
 * BF16 / TF32 modes with w_t_lp, 16-byte aligned buffers, H <= 256 and a geometry the tensor-core forward serves: one
 * tcgen05 kernel (TF32 mode rounds dtokens to nearest TF32 first: two launches).  Otherwise exact fp32: patch-row
 * compaction, FMA GEMM, inverse im2col (three launches). */
int vit3d_patch_embed_dgrad(const float* dtokens, const float* w, const void* w_t_lp, float* dx,
                            int B, int X, int Y, int Z, int p0, int p1, int p2, int H, int prec,
                            void* ws, size_t ws_bytes, vit3d_stream_t stream);

/* ---------------------------------------------------------------- a4/a5: LayerNorm(eps, biased var, affine)
 * nn.LayerNorm(H, eps=1e-6) at modeling.py:182-183,189,194,242,253.
 * y is [M,H] in fp32 (y_bf16=0), bf16 (y_bf16=1) or fp32 rounded to TF32 (y_bf16=2, operand of a TF32
 * GEMM); mean/rstd [M] may be NULL in inference. */
int vit3d_ln_fwd(const float* x, const float* gamma, const float* beta, void* y, int y_bf16, float* mean,
                 float* rstd, int M, int H, float eps, vit3d_stream_t stream);
/* dx = (dres ? dres : 0) + LN'(dy); dgamma/dbeta accumulated.  dy fp32 [M,H]. */
int vit3d_ln_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                 const float* dres, float* dx, float* dgamma, float* dbeta, int M, int H, vit3d_stream_t stream);

/* ---------------------------------------------------------------- nn.Linear (modeling.py:63-67,105-106,277,351)
 * y[M,N] = act(x[M,K] @ w[N,K]^T + bias) (+ residual).  x/y/pre are "act" typed unless noted.
 *   w        fp32 master weight [N,K];   w_lp  bf16 copy of w (BF16 mode) / TF32-rounded fp32 copy (TF32
 *            mode, optional) / NULL
 *   residual fp32 [M,N] or NULL (then y is "act"); with residual, y is fp32 (residual stream)
 *   pre      optional [M,N] "act": pre-activation saved for backward (act==GELU)
 *   ldx      row stride of x in elements (lets the head read rows b*S of the token matrix)
 *   y_f32    force fp32 output even without residual (logits, dgrad into LayerNorm backward) */
int vit3d_linear_fwd(const void* x, int ldx, int x_f32, const float* w, const void* w_lp, const float* bias,
                     const float* residual, void* y, int y_f32, void* pre, int act, int M, int N, int K, int prec,
                     vit3d_stream_t stream);
/* Linear + residual + the LayerNorm that follows it in the Block (modeling.py:189-196: `x = x + h` then
 * `ffn_norm(x)` / the next Block's `attention_norm(x)` / `encoder_norm(x)`), one kernel, BF16 mode, N == 256:
 *   y[M,N]      = x[M,K] @ w_lp[N,K]^T + bias + residual        (fp32 residual stream; y may alias residual)
 *   ln_out[M,N] = (y - mean) * rstd * gamma + beta                (bf16: the A operand of the next GEMM)
 * mean / rstd [M] optional (saved for vit3d_ln_bwd).  Each thread of the epilogue owns one accumulator row;
 * the row statistics are combined across the four column slices in shared memory, so the fp32 rows are
 * never re-read.  Returns VIT3D_ERR_UNSUPPORTED for other shapes (compose vit3d_linear_fwd + vit3d_ln_fwd). */
int vit3d_linear_ln_fwd(const void* x, const void* w_lp, const float* bias, const float* residual, float* y,
                        const float* gamma, const float* beta, float eps, void* ln_out, float* mean, float* rstd, int M,
                        int N, int K, vit3d_stream_t stream);
int vit3d_linear_ln_supported(int M, int N, int K);
/* dx[M,K] = dy[M,N] @ w[N,K]  (dx_f32: write fp32);  dw[N,K] += dy^T @ x ; db[N] += colsum(dy).
 * Any of dx / dw / db may be NULL.  dy is "act" typed unless dy_f32.
 *   w_t_lp  bf16 TRANSPOSED copy of w, [K,N] (vit3d_transpose_f32_to_bf16): with it, bf16 dy and BF16 mode
 *           the data gradient runs on tcgen05; the weight gradient does when dy and x are bf16 (both
 *           operands are read MN-major, nothing is transposed in memory). */
int vit3d_linear_bwd(const void* dy, int dy_f32, const void* x, int ldx, int x_f32, const float* w, const void* w_t_lp,
                     void* dx, int lddx, int dx_f32, float* dw, float* db, int M, int N, int K, int prec,
                     vit3d_stream_t stream);

/* ---------------------------------------------------------------- a3: Mlp.forward fused (inference)
 * out[M,H] = residual + fc2(gelu(fc1(xn) + b1)) + b2  (modeling.py:118-124 with the x + Mlp(..) add of :196;
 * dropout is the identity in eval mode).  BF16 mode, H = 256, d % 256 == 0: xn bf16 [M,H] (LayerNorm
 * output), w1_lp bf16 [d,H], w2_h FP16 [H,d] (vit3d_cast_f32_to_f16: the GELU output is kept in fp16 -
 * 11 significant bits - and tcgen05 kind::f16 needs both operands of fc2 in the same 16-bit format); the
 * [M,d] intermediate stays on chip.  Returns VIT3D_ERR_UNSUPPORTED for other shapes (compose
 * vit3d_linear_fwd instead). */
int vit3d_mlp_fwd(const void* xn, const void* w1_lp, const float* b1, const void* w2_h, const float* b2,
                  const float* residual, float* out, int M, int H, int d, vit3d_stream_t stream);
int vit3d_mlp_supported(int M, int H, int d);
/* Same block with the LayerNorm that consumes its output (the next Block's attention_norm, modeling.py:189)
 * applied in the final epilogue: ln_out[M,H] = LayerNorm(out) * gamma + beta as bf16.  H = 256, d % 256 == 0.
 * `out` may alias `residual`. */
int vit3d_mlp_ln_fwd(const void* xn, const void* w1_lp, const float* b1, const void* w2_h, const float* b2,
                     const float* residual, float* out, const float* gamma, const float* beta, float eps, void* ln_out,
                     int M, int H, int d, vit3d_stream_t stream);
int vit3d_mlp_ln_supported(int M, int H, int d);
/* The LAST Block's MLP with the encoder's final LayerNorm (Encoder.forward, modeling.py:253) folded in:
 * ln_out[M,H] = LayerNorm(residual + fc2(gelu(fc1(xn) + b1)) + b2) * gamma + beta as FP32 - the `encoded`
 * tensor VisionTransformer.forward returns (modeling.py:280,288).  The un-normalised block output is not
 * written (nothing reads it at inference).  Same shape support as vit3d_mlp_ln_fwd. */
int vit3d_mlp_lnf_fwd(const void* xn, const void* w1_lp, const float* b1, const void* w2_h, const float* b2,
                      const float* residual, const float* gamma, const float* beta, float eps, float* ln_out, int M, int H,
                      int d, vit3d_stream_t stream);

/* ---------------------------------------------------------------- a2: scaled-dot-product attention core
 * scores = q k^T / sqrt(D); probs = softmax(scores); ctx = probs v  (modeling.py:83-96).
 * qkv is the packed [M, 3*k*D] matrix (q | k | v column blocks, head h at columns h*D..),
 * ctx [M, k*D] "act"; probs (optional, vis=True) fp32 [B,k,S,S]. */
int vit3d_attn_fwd(const void* qkv, void* ctx, float* probs, int B, int S, int heads, int D, int prec,
                   vit3d_stream_t stream);
/* Same in BF16 mode with PADDED probability rows: probs is [B,k,S,probs_ld] with probs_ld = 72 (S = 65) and a 32-byte
 * aligned base; the 7 padding floats of a row are written as zeros (whole sectors only).  Every row then starts on a 32-byte sector and the
 * column pairs a lane stores never straddle one (the packed rows of 65 floats start at 4-byte phases: 1.58x write
 * amplification between L1 and L2).  The Python surface hands out `probs[..., :S]` - same shape and values as the
 * reference's attention_probs tensor, non-contiguous. */
int vit3d_attn_fwd_padded(const void* qkv, void* ctx, float* probs, int probs_ld, int B, int S, int heads, int D,
                          vit3d_stream_t stream);
int vit3d_attn_padded_supported(int S, int heads, int D);
/* dqkv from dctx (probabilities are recomputed from qkv) */
int vit3d_attn_bwd(const void* dctx, const void* qkv, void* dqkv, int B, int S, int heads, int D, int prec,
                   vit3d_stream_t stream);

/* ---------------------------------------------------------------- elementwise pieces
 * exact-erf GELU (modeling.py:52,107,120): a = gelu(h); da -> dh */
int vit3d_gelu_fwd(const void* h, void* a, long long n, int prec, vit3d_stream_t stream);
int vit3d_gelu_bwd(const void* da, const void* h, void* dh, long long n, int prec, vit3d_stream_t stream);
/* dh = dropout'(da) * gelu'(h) in one pass (BF16 mode): the backward of Dropout(gelu(h)) at modeling.py:120-121,
 * mask regenerated from (seed, site, step).  VIT3D_ERR_UNSUPPORTED unless bf16 / aligned / n % 8 == 0. */
int vit3d_gelu_dropout_bwd(const void* da, const void* h, void* dh, long long n, int prec, float p,
                           unsigned long long seed, unsigned site, unsigned step, const unsigned* step_dev,
                           vit3d_stream_t stream);
/* Dropout(p) in training (modeling.py:121,123,174): y = x * keep / (1-p) (+ residual, same type, may be
 * NULL: the x + Mlp(..) add of modeling.py:196) with a counter-based Philox mask keyed by
 * (seed, site, step, element index); the same call on dy (residual NULL) gives dx.  One Philox4x32-10 block serves
 * eight consecutive elements (16-bit lanes): P(drop) = round(p * 65536) / 65536. */
/* step_dev (device, may be NULL) is added to `step` on the device: lets a captured CUDA graph draw new
 * masks at every replay. */
int vit3d_dropout(const void* x, const void* residual, void* y, long long n, int is_f32, float p,
                  unsigned long long seed, unsigned site, unsigned step, const unsigned* step_dev,
                  vit3d_stream_t stream);
/* export the keep mask (1 byte per element) for mask-injection parity tests */
int vit3d_dropout_mask(unsigned char* mask, long long n, float p, unsigned long long seed, unsigned site,
                       unsigned step, vit3d_stream_t stream);
/* y = x * mask / (1-p) with an explicit mask (parity mode) */
int vit3d_dropout_masked(const void* x, const unsigned char* mask, const void* residual, void* y, long long n,
                         int is_f32, float p, vit3d_stream_t stream);
int vit3d_cast_f32_to_bf16(const float* x, void* y, long long n, vit3d_stream_t stream);
int vit3d_cast_bf16_to_f32(const void* x, float* y, long long n, vit3d_stream_t stream);
int vit3d_cast_f32_to_f16(const float* x, void* y, long long n, vit3d_stream_t stream);
/* N2 input pipeline (create_dataset.py:31-69 reads 8-bit slices; tools.py:18-26 subtracts the training
 * mean): y = float(x_u8) - mean on the device, so volumes cross PCIe as uint8 (81,920 B instead of
 * 327,680 B per volume). */
int vit3d_u8_to_f32(const unsigned char* x, float* y, long long n, float mean, vit3d_stream_t stream);
/* y[cols,rows] (bf16) = x[rows,cols]^T (fp32) */
int vit3d_transpose_f32_to_bf16(const float* x, void* y, int rows, int cols, vit3d_stream_t stream);
/* y = x rounded to nearest TF32 (fp32 container): shadow weights for the TF32 mode */
int vit3d_round_tf32(const float* x, float* y, long long n, vit3d_stream_t stream);
/* y += x (fp32) */
int vit3d_add_inplace(float* y, const float* x, long long n, vit3d_stream_t stream);

/* ---------------------------------------------------------------- a7: head loss
 * BCEWithLogitsLoss(pos_weight)(logits.view(-1,1), labels.view(-1,1)), mean (modeling.py:283-286).
 * pos_weight < 0 means None; pos_weight_dev (device scalar, may be NULL) overrides it (CUDA-graph replays
 * with a per-batch class weight).  loss: 1 float.  dlogits = dloss * dL/dlogits (dloss: device scalar or
 * NULL = 1). */
int vit3d_bce_logits_fwd(const float* logits, const float* labels, float pos_weight, const float* pos_weight_dev,
                         float* loss, int n, vit3d_stream_t stream);
int vit3d_bce_logits_bwd(const float* logits, const float* labels, float pos_weight, const float* pos_weight_dev,
                         const float* dloss, float* dlogits, int n, vit3d_stream_t stream);

/* ---------------------------------------------------------------- a9: meta-classifier
 * out[B,C] = sigmoid(cat(member logits)[B,F] @ w[C,F]^T + b) (modeling.py:355-356) */
int vit3d_meta_fwd(const float* feats, const float* w, const float* b, float* out, int B, int F, int C,
                   vit3d_stream_t stream);
int vit3d_meta_bwd(const float* dout, const float* out, const float* feats, const float* w, float* dfeats, float* dw,
                   float* db, int B, int F, int C, vit3d_stream_t stream);

/* ---------------------------------------------------------------- N1: optimizer steps on a flat fp32 arena
 * torch.optim.SGD(momentum, weight_decay) (train_baseline_cv.py:111-114) and Adam (train_ensemble_whole_dataset.py:53)
 * semantics of torch 2.x (first momentum step copies the gradient). */
int vit3d_sgd_step(float* p, const float* g, float* mom, long long n, float lr, float momentum, float weight_decay,
                   int first_step, float grad_scale, const float* lr_dev, vit3d_stream_t stream);
int vit3d_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, float grad_scale, const float* lr_dev, const int* step_dev,
                    vit3d_stream_t stream);
/* lr_dev / step_dev: optional DEVICE scalars that override lr / step (CUDA-graph replays under an LR
 * schedule).  first_step may stay 0 when the momentum buffer starts zeroed (same arithmetic). */

/* ---------------------------------------------------------------- a8: fused BF16 training step (hidden 256)
 * The autograd backward of modeling.py:118-124, :187-197 (loss.backward() at train_baseline_cv.py:176) as an
 * explicit kernel sequence, driven by 3d_vit_ensemble_b200/fused_train.py.  The pieces below are the ones the
 * per-operator entry points above do not offer: dropout masks as bit arrays applied inside GEMM epilogues,
 * LayerNorm backward fused with the residual-gradient add / the bf16 operand copy / the bias-gradient column
 * sums, packed q|k|v weight gradients that land in three parameters, one-launch weight-shadow refresh. */
#define VIT3D_MAX_DROP_SEGS 40
#define VIT3D_SHADOW_JOB_BYTES 40
#define VIT3D_SHADOW_TILE 64
/* cudaMemsetAsync(p, 0, bytes) on `stream` (gradient arena zeroing without a framework fill kernel) */
int vit3d_memset_zero(void* p, size_t bytes, vit3d_stream_t stream);
/* 1 if the fused training step serves this model shape (B volumes of S tokens, hidden H, mlp width d) */
int vit3d_train_supported(int B, int S, int H, int heads, int d);
/* Keep bits of ALL Dropout sites of one training step (modeling.py:121,123,174) in one launch.  Segment i
 * covers nelems[i] (% 32 == 0) elements of dropout site sites[i]; segments are laid end to end in `bits`
 * (bit e of 32-bit word w of a segment = element 32 w + e, i.e. byte e/8, bit e%8 in memory).  The decision
 * for an element equals vit3d_dropout / vit3d_dropout_mask for the same (seed, site, step, index).  `sites`
 * and `nelems` are HOST arrays (nseg <= VIT3D_MAX_DROP_SEGS); step_dev as in vit3d_dropout. */
int vit3d_dropout_bits(uint32_t* bits, int nseg, const unsigned* sites, const long long* nelems, float p,
                       unsigned long long seed, unsigned step, const unsigned* step_dev, vit3d_stream_t stream);
/* LayerNorm over rows of 256 with an optional Dropout of its INPUT (Embeddings.dropout, modeling.py:174):
 *   xd = x * keep * drop_scale  (written to x_dropped when drop_bits and x_dropped are given; else xd = x)
 *   y  = LayerNorm(xd) * gamma + beta as bf16 (y_bf16) and/or fp32 (y_f32); mean / rstd [M] optional. */
int vit3d_ln256_fwd(const float* x, const void* drop_bits, float drop_scale, float* x_dropped, const float* gamma,
                    const float* beta, void* y_bf16, float* y_f32, float* mean, float* rstd, int M, float eps,
                    vit3d_stream_t stream);
/* LayerNorm-256 backward fused with what surrounds it in a pre-LN Block (modeling.py:187-197):
 *   o       = (dres ? dres : 0) + LN'(dy)              gradient w.r.t. the LayerNorm input (+ the skip path)
 *   ob      = o * keep * drop_scale (drop_bits given: the Dropout of modeling.py:123 / :174 below this point)
 *   dx      = o, or ob when mask_f32 (fp32, optional, may alias dres)
 *   dx_bf16 = bf16(ob) (optional): the operand of the dgrad / wgrad GEMMs of the Linear that produced this
 *             tensor;  dbias += column sums of ob (that Linear's bias gradient, optional)
 *   dgamma += sum dy * xhat;  dbeta += sum dy. */
int vit3d_ln256_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                    const float* dres, const void* drop_bits, float drop_scale, int mask_f32, float* dx, void* dx_bf16,
                    float* dgamma, float* dbeta, float* dbias, int M, vit3d_stream_t stream);
/* dh = da * dact (bf16 [M,d]): the element-wise stage of the MLP backward (modeling.py:120-121) with dact = gelu'(pre) *
 * keep * drop_scale as written by vit3d_fc1_train_fwd; db[d] += column sums of dh (the fc1 bias gradient, optional).
 * dh may alias da. */
int vit3d_mul_colsum_bwd(const void* da, const void* dact, void* dh, float* db, int M, int d, vit3d_stream_t stream);
/* The data-gradient chain of Mlp.forward's backward (modeling.py:118-124) in ONE kernel (H = 256, d % 256 == 0):
 *   da = gy w2 ; dh = da * dact ; dxn = dh w1 ; db1 += column sums of dh
 * gy [M,H] bf16 (gradient w.r.t. the fc2 output, its Dropout already undone); w2_t_lp = bf16 [d,H] transposed fc2
 * weight, w1_t_lp = bf16 [H,d] transposed fc1 weight; dact [M,d] bf16 from vit3d_fc1_train_fwd; dh [M,d] bf16 is
 * written once (the two weight-gradient GEMMs read it), dxn [M,H] fp32; `da` never reaches memory. */
int vit3d_mlp_bwd(const void* gy, const void* w2_t_lp, const void* w1_t_lp, const void* dact, void* dh, float* dxn, float* db1,
                  int M, int H, int d, vit3d_stream_t stream);
int vit3d_mlp_bwd_supported(int M, int H, int d);
/* head backward (modeling.py:281, num_classes 1): dencoded[B*S,H] = dlogits[b] * w on the cls rows, 0 elsewhere;
 * dw[H] += sum_b dlogits[b] * encoded[b*S,:];  db[1] += sum_b dlogits[b]. */
int vit3d_head_bwd(const float* dlogits, const float* encoded, const float* w, float* dencoded, float* dw, float* db, int B,
                   int S, int H, vit3d_stream_t stream);
/* Rewrites every low-precision weight shadow of a model from its fp32 masters in ONE launch.  `jobs` is a DEVICE
 * array of njobs records of VIT3D_SHADOW_JOB_BYTES bytes, sorted by tile0:
 *   { const float* src; void* dst; int rows, cols, ld, kind, tile0, tiles_c; }
 * src [rows, cols] dense fp32; element (r, c) goes to dst[r*ld + c] as bf16 (kind 0), fp16 (2), fp32 rounded to
 * TF32 (3) or fp32 (4), or to dst[c*ld + r] as bf16 (kind 1, transposed: the dgrad operand).  tile0 = index of the
 * job's first VIT3D_SHADOW_TILE x VIT3D_SHADOW_TILE (64 x 64) tile in the launch, tiles_c = ceil(cols/64); total_tiles = sum
 * over jobs.  step_dev (optional
 * device counter) is incremented by one: the dropout step of a CUDA-graph replay. */
int vit3d_refresh_shadows(const void* jobs, int njobs, int total_tiles, unsigned* step_dev, vit3d_stream_t stream);
/* training fc1 (modeling.py:119-121): act = Dropout(gelu(xn w1^T + b1)) (bf16) and, instead of the pre-activation,
 * dact = gelu'(xn w1^T + b1) * keep * drop_scale (bf16): the factor the backward multiplies the incoming gradient by
 * (vit3d_mlp_bwd / vit3d_mul_colsum_bwd), so the backward needs neither the GELU derivative nor the keep bits.
 * Dropout from keep bits over [M,d] (NULL = none: keep = 1, scale = 1), all in the GEMM epilogue. */
int vit3d_fc1_train_fwd(const void* xn, const void* w1_lp, const float* b1, void* dact, void* act, const void* drop_bits,
                        float drop_scale, int M, int d, int H, vit3d_stream_t stream);
/* training out-projection / fc2 (modeling.py:97,122-123 + the adds of :191,:196 + the next LayerNorm):
 *   y = residual + Dropout(x w^T + bias) (drop_bits NULL = no dropout),  ln_out = LayerNorm(y) bf16 (optional, with
 *   mean / rstd saved for vit3d_ln256_bwd).  N % 256 == 0 (LayerNorm: N == 256). */
int vit3d_linear_res_train_fwd(const void* x, const void* w_lp, const float* bias, const float* residual, float* y,
                               const void* drop_bits, float drop_scale, const float* gamma, const float* beta, float eps,
                               void* ln_out, float* mean, float* rstd, int M, int N, int K, vit3d_stream_t stream);
/* dw[N,K] += dy[M,N]^T x[M,K] (bf16 operands, tcgen05).  seg_rows > 0: rows [i*seg_rows, (i+1)*seg_rows) of the
 * product accumulate into dw0 / dw1 / dw2 (the packed q|k|v projection: three parameters). */
int vit3d_wgrad(const void* dy, const void* x, float* dw0, float* dw1, float* dw2, int seg_rows, int M, int N, int K,
                vit3d_stream_t stream);
/* The same product WITHOUT atomics, in two steps.  vit3d_wgrad_partial: every (output tile, reduction slice) work item
 * stores its 128 x bn fp32 tile densely into `ws` (vit3d_wgrad_ws_bytes(M, N, K) bytes; tile-major, slice-minor) and
 * reports the tile width / slice count it used.  vit3d_wgrad_reduce: ONE launch for all weight-gradient GEMMs of a
 * training step sums the slices of every tile and ADDS the result to the gradient buffers.  `host_jobs` is a HOST
 * array of njobs (<= VIT3D_MAX_WGRAD_JOBS) records of VIT3D_WGRAD_JOB_BYTES bytes:
 *   { const float* ws; float* dst[3]; int seg_rows, rows (= N), cols (= K), bn, splits, tiles_n (= K / bn), block0, pad; }
 * (block0 is filled in by the library).  N % 128 == 0. */
#define VIT3D_MAX_WGRAD_JOBS 48
#define VIT3D_WGRAD_JOB_BYTES 64
size_t vit3d_wgrad_ws_bytes(int M, int N, int K);
int vit3d_wgrad_partial(const void* dy, const void* x, float* ws, int M, int N, int K, int* bn, int* splits,
                        vit3d_stream_t stream);
int vit3d_wgrad_reduce(const void* host_jobs, int njobs, vit3d_stream_t stream);
/* vit3d_attn_bwd (BF16 mode) that also accumulates the q / k / v bias gradients (column sums of dqkv) */
int vit3d_attn_bwd_bias(const void* dctx, const void* qkv, void* dqkv, float* db_q, float* db_k, float* db_v, int B, int S,
                        int heads, int D, vit3d_stream_t stream);

#ifdef __cplusplus
}
#endif
#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#endif /* VIT3D_H_ */
