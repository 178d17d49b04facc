// Launchers of the memory-bound kernels (LayerNorm, embeddings, pooling, loss, Adam, EMA, ...)
// and of the SIMT attention used by the fp32 check mode.
#pragma once
#include "common.cuh"

namespace v2s {

// type tag `at`: 0 = fp32 activations, 1 = bf16, 2 = fp16
int launch_im2col(const float* const* x, void* const* out, int groups, int B, int at, cudaStream_t s);
int launch_cls_rows(const float* const* params, float* const* hidden, int groups, int B, cudaStream_t s);
int launch_assemble_tokens(const float* const* params, const float* const* tok, float* const* hidden, int groups,
                           int B, cudaStream_t s);
int launch_gather_patch_rows(const void* const* src, void* const* dst, int groups, int B, int at, cudaStream_t s);
int launch_ln_fwd(const float* const* x, const float* const* gamma, const float* const* beta,
                  void* const* y, float* const* mean, float* const* rstd, int groups, int M, int at,
                  cudaStream_t s);
// dres (fp32, in/out) += LN-backward(dy); dres_lp (optional, activation type) = updated dres;
// dcolsum (optional) += column sums of the updated dres (bias gradient of the next linear layer)
int launch_ln_bwd(const void* const* dy, const float* const* x, const float* const* mean,
                  const float* const* rstd, const float* const* gamma, float* const* dres,
                  void* const* dres_lp, float* const* dgamma, float* const* dbeta, float* const* dcolsum,
                  int groups, int M, int at, cudaStream_t s, const DetScratch* det = nullptr);
// db[n] += sum_m dy[m,n]; src type tag `t`.  With `det` (deterministic mode) the sum has a fixed order: partial rows in
// det->part, or, when det->part is NULL, one CTA per group
int launch_colsum(const void* const* dy, float* const* db, int groups, int M, int N, int t, cudaStream_t s,
                  const DetScratch* det = nullptr);
int launch_pool_fwd(const float* const* hidden, float* const* feat, const int64_t* feat_stride,
                    int groups, int B, cudaStream_t s);
int launch_pool_bwd(const float* const* dfeat, const int64_t* dfeat_stride, const float* const* dhidden,
                    float* const* dx, void* const* dx_lp, int groups, int B, int at, cudaStream_t s);
int launch_embed_bwd(const float* const* dx, float* const* grads, int groups, int B, cudaStream_t s,
                     const DetScratch* det = nullptr);
// dx (fp32, in/out) += dh; dx_lp (activation type, 16-bit modes only) = updated dx; [B,197,192] per group;
// dcol (optional, per group) += column sums of dh
int launch_residual_grad_add(const float* const* dh, float* const* dx, void* const* dx_lp, float* const* dcol, int groups, int B,
                             int at, cudaStream_t s, const DetScratch* det = nullptr);

// attention over qkv [B,197,576] (q|k|v, head h at columns h*64): ctx [B,197,192], lse [B,3,197]
int launch_attn_fwd_simt(const void* const* qkv, void* const* ctx, float* const* lse, int groups, int B,
                         int at, cudaStream_t s);
int launch_attn_bwd_simt(const void* const* qkv, const void* const* ctx, const float* const* lse,
                         const void* const* dctx, void* const* dqkv, int groups, int B, int at,
                         cudaStream_t s);
// attention probabilities exp(q k^T / 8 - lse) as fp32 probs [B,3,197,197], from qkv and the forward's lse
int launch_attn_probs_simt(const void* const* qkv, const float* const* lse, float* const* probs, int groups, int B,
                           int at, cudaStream_t s);

// tcgen05 versions (bf16, or fp16 with lp_f16 = 1)
int launch_attn_fwd_tc(const void* const* qkv, void* const* ctx, float* const* lse, int groups, int B,
                       cudaStream_t s, int lp_f16 = 0);

int launch_attn_bwd_tc(const void* const* qkv, const void* const* ctx, const float* const* lse,
                       const void* const* dctx, void* const* dqkv, int groups, int B, cudaStream_t s, int lp_f16 = 0);
int launch_attn_probs_tc(const void* const* qkv, const float* const* lse, float* const* probs, int groups, int B,
                         cudaStream_t s, int lp_f16 = 0);

int launch_infonce_loss(const float* p, const float* z_all, float* loss, float* row_loss, float* dp, int B, int n_keys,
                        long long label_offset, float temperature, int accum, float grad_scale, cudaStream_t s,
                        const float* grad_scale_dev = nullptr);
int launch_cosine_loss(const float* p, const float* z, float* loss, float* dp, int B, int accum,
                       float grad_scale, cudaStream_t s, const float* grad_scale_dev = nullptr);
int launch_adam(const v2s_range_t* ranges, int n, int64_t step, double lr, double b1, double b2, double eps,
                double wd, double grad_scale, cudaStream_t s, int lp_f16 = 0);
// device-resident step state (GradScaler-style skipping, CUDA-graph capturable): see v2s_adam_step_amp
int launch_adam_amp(const v2s_range_t* ranges, int n, float* state8, double lr, double b1, double b2, double eps, double wd,
                    double grad_multiplier, const float* grad_scale_dev, const float* found_inf_dev, int lp_f16, int advance,
                    cudaStream_t s);
int launch_ema(float* const* tgt, const float* const* onl, void* const* tgt_lp, int n_pairs,
               int64_t numel, double momentum, cudaStream_t s, int lp_f16 = 0);
int launch_cast_bf16(const float* src, void* dst, int64_t n, cudaStream_t s, int lp_f16 = 0);
int launch_dropout_mask(float* mask, int64_t n, float p, uint64_t seed, uint64_t offset, cudaStream_t s);
int launch_preprocess_u8(const uint8_t* src, float* dst, int B, cudaStream_t s);
int launch_preprocess_u8_patches(const uint8_t* src, void* out, int B, int lp_f16, cudaStream_t s);
int launch_augment_finish(const uint8_t* src, int n, int in_size, const int32_t* bounds, const int32_t* coefs, int ksize,
                          const float* k1d, const int32_t* erase, const float* mean3, const float* std3, float* dst,
                          cudaStream_t s);
int launch_zero(void* p, int64_t bytes, cudaStream_t s);
int launch_splitk_reduce(float* out, const float* part, const float* bias, int M, int N, int splits, cudaStream_t s,
                         bool add = false);

}  // namespace v2s
