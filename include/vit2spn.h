/*
 * vit2spn.h — C ABI of the B200-native ViT-2SPN dual-stream SSP hot path (libvit2spn.so).
 *
 * The reference (mrsaraei/ViT-2SPN) has no FFI layer: its hot path sits behind the
 * torch.nn.Module protocol of ViTBackbone / DualStreamNetwork (ref:ssp_vit2spn_tiny.py:109-166),
 * torch autograd, torch.optim.Adam (ref:173,216) and a Python EMA loop (ref:162-166).  Each entry
 * point below replaces one of those call sites; the Python host mirror (vit-2spn_b200/) binds them
 * with ctypes (see INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - the caller (torch) owns all memory, including one workspace buffer sized by
 *     v2s_workspace_bytes(); the library never allocates or frees device memory and keeps no
 *     reference to caller memory after a call returns (it does cache TMA descriptors keyed by
 *     address, which are re-validated on every call);
 *   - all work is enqueued asynchronously on the cudaStream_t passed as `stream` (void*);
 *   - return value 0 = ok, non-zero = error; message via v2s_last_error(); no C++ exceptions
 *     cross the boundary; there is NO CPU fallback: a non-sm_100 device is an error.
 */
#ifndef VIT2SPN_H_
#define VIT2SPN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define V2S_ABI_VERSION 5 /* 5: the backbone calls added to 4 (image, attention-probability and mask-token gradients,
                             masked forward) are folded into v2s_backbone_forward / _backward: their arguments are
                             fields of v2s_group_outputs, and v2s_backbone_backward takes weight_grads.  Additive to 5:
                             v2s_mim_workspace_bytes, v2s_mim_forward, v2s_mim_backward, v2s_cls_workspace_bytes, v2s_cls_forward,
                             v2s_cls_backward.  Additive to 4:
                             v2s_test_gemm which = 5, v2s_test_attention which = 3.  4: one entry point per operation:
                             v2s_backbone_forward / _backward take the per-group outputs and (backward) the layer range,
                             v2s_heads_loss_fwd_bwd the device loss scale, v2s_adam_step and v2s_ema_update the
                             lp_format; their narrower variants and the bf16-only cast are removed.  3: v2s_infonce_loss,
                             v2s_preprocess_u8_patches, v2s_group.x_format (was a reserved zero field); additive to 3:
                             v2s_group_outputs, v2s_test_attention which = 2 */

/* compute modes */
#define V2S_MODE_FP32 0 /* fp32 activations + fp32 SIMT GEMMs: the "fp32 check mode" of north_star */
#define V2S_MODE_BF16 1 /* bf16 GEMM operands (tcgen05), fp32 accumulate / residual / LN / softmax */
#define V2S_MODE_FP16 2 /* fp16 GEMM operands: the reference's own CUDA precision (torch.autocast default dtype +
                           GradScaler, ref:ssp_vit2spn_tiny.py:175,209-217); needs loss scaling (grad_scale_dev of
                           v2s_heads_loss_fwd_bwd / v2s_infonce_loss, v2s_adam_step_amp) */

/* format of the 16-bit shadow copy of a flat parameter buffer (params_lp) */
#define V2S_LP_BF16 0
#define V2S_LP_FP16 1

/* model constants: ViT-Tiny/16 @224 (ref:ssp_ssl/ssl_vit2spn_scratch.py:100-108) */
#define V2S_HIDDEN 192
#define V2S_LAYERS 12
#define V2S_HEADS 3
#define V2S_HEAD_DIM 64
#define V2S_MLP 768
#define V2S_TOKENS 197
#define V2S_PATCHES 196
#define V2S_PATCH_K 768   /* 3*16*16 */
#define V2S_IMG 224
#define V2S_PROJ_IN 384   /* ref:ssp_vit2spn_tiny.py:134 */
#define V2S_PROJ_HID 1024
#define V2S_PROJ_OUT 128
#define V2S_MAX_GROUPS 4

int v2s_abi_version(void);
const char* v2s_last_error(void);

/* Verifies that `device` is an sm_100 part and selects it.  Replaces nothing in the reference
 * (torch picks the device, ref:ssp_vit2spn_tiny.py:32); exists so that the product fails loudly.  The caller's current
 * device is not changed; every other entry point works on the CURRENT device of the calling thread, which must be
 * the device its pointers live on (the host mirror makes it so around each call). */
int v2s_init(int device);

/* ---- flat parameter layout --------------------------------------------------------------
 * One backbone = one flat fp32 buffer of v2s_backbone_numel() elements.  The 200 HF tensors of
 * transformers.ViTModel (ref:ssp_vit2spn_tiny.py:112) are views at the offsets returned by
 * v2s_backbone_layout(): q/k/v weights (and biases) of a block are adjacent so that they form one
 * fused [576,192] matrix; the final LayerNorm + pooler (never used by the reference's forward,
 * SURVEY D6) sit at the tail, after v2s_backbone_active_numel() elements. */
int64_t v2s_backbone_numel(void);        /* 5 561 472 */
int64_t v2s_backbone_active_numel(void); /* 5 524 032 */
int64_t v2s_heads_numel(void);           /* 558 464 : proj W1,b1,W2,b2, pred W3,b3,W4,b4 */
/* offsets[i] = element offset of the i-th HF parameter (registration order) in the flat buffer */
int v2s_backbone_layout(int64_t* host_offsets200);
int v2s_heads_layout(int64_t* host_offsets8);

/* ---- workspace --------------------------------------------------------------------------- */
/* bytes of workspace for `n_groups` backbones run together at `batch` images each, of which
 * `n_saved` keep their activations for a backward pass. */
int64_t v2s_workspace_bytes(int batch, int mode, int n_groups, int n_saved);

/* One backbone instance in a grouped launch (online_1, online_2, target_1, target_2 are four
 * groups of one call: ref:ssp_vit2spn_tiny.py:146-151). */
typedef struct v2s_group {
  const float* params;    /* flat fp32 parameters (layout above) */
  const void* params_lp;  /* bf16 copy of `params` (same element offsets); NULL in fp32 mode */
  float* grads;           /* flat fp32 gradient buffer, accumulated (+=); NULL if no backward */
  const void* x;          /* x_format 0: images fp32 NCHW [batch,3,224,224];  x_format 1: the patch matrix the patch-embed
                           * GEMM reads, [batch*196, 768] in the mode's 16-bit format, k = c*256 + ky*16 + kx (what
                           * v2s_preprocess_u8_patches writes) - it must stay valid until the backward call, which reads
                           * it again for the patch-embedding weight gradient */
  float* hidden;          /* out (optional): hidden_states[-1], fp32 [batch,197,192] */
  float* feat;            /* out (optional): mean over tokens, row i at feat + i*feat_stride */
  int64_t feat_stride;    /* 192, or 384 when writing straight into the concatenated feature */
  const float* dfeat;     /* backward in: d loss / d feat, row stride dfeat_stride (or NULL) */
  int64_t dfeat_stride;
  const float* dhidden;   /* backward in (optional): d loss / d hidden [batch,197,192]; added */
  int32_t slot;           /* activation-stash slot (0..n_saved-1), or -1: nothing saved */
  int32_t x_format;       /* 0 or 1, see x (1: bf16 / fp16 modes only) */
} v2s_group_t;

/* Per-group optional inputs and outputs of the two calls below: transformers' output_hidden_states / output_attentions,
 * the gradients w.r.t. the pixels and the attention probabilities, and masked patch tokens.  The calls take an array of
 * n_groups of these, or NULL for none.  NULL (or every pointer NULL) requests nothing and costs nothing: the call then
 * launches exactly the kernels of a backbone pass without them.  A saved group's hidden[] and mask must be the same in
 * its forward and its backward call. */
typedef struct v2s_group_outputs {
  float* hidden[V2S_LAYERS + 1];        /* out: hidden_states[l] fp32 [batch,197,192]; all 13 or none. When set, the
                                           group's residual stream lives here; a saved group's backward reads it back */
  float* attn[V2S_LAYERS];              /* out: softmax(QK^T/8) fp32 [batch,3,197,197]; all 12 or none */
  const float* dhidden[V2S_LAYERS + 1]; /* backward in: d loss / d hidden_states[l], added; NULL entries skipped.
                                           dhidden[12] is v2s_group.dhidden (set one of the two).  Without dfeat and
                                           dhidden[12] the backward starts at the highest l with a gradient: the
                                           blocks above it are skipped and get no gradient */
  float* dattn[V2S_LAYERS];             /* backward out: d loss / d attn[l], fp32 [batch,3,197,197], overwritten, 4-byte
                                           aligned: d ctx V^T, what retain_grad() gives on transformers' attentions.
                                           NULL entries skipped; blocks at or above the highest layer the loss reaches
                                           (see dhidden) get nothing written.  Written by the call whose range covers l */
  float* dpixels;                       /* backward out: d loss / d pixel_values (transformers' input gradient), fp32
                                           [batch,3,224,224], overwritten, 16-byte aligned, x_format 0 only; written by
                                           the call whose range ends at layer 0.  The weight gradients are those of the
                                           call without it (same kernels, same bits) */
  const uint8_t* mask;                  /* forward and backward in: uint8 [batch,196] patch mask (NULL: none), transformers'
                                           bool_masked_pos of ViTModel(use_mask_token=True), the input of SimMIM-style
                                           masked image modelling.  The forward replaces the embedding of every patch p of
                                           image b with mask[b*196 + p] != 0 by mask_token, after the patch projection and
                                           its bias and before the position embedding is added.  A saved group's backward
                                           passes the forward's array; a masked backward runs over [0, 12) only.  The
                                           patch weight and bias gradients and the image gradient come from the unmasked
                                           patches only (the image gradient is exactly 0 on masked patches) */
  const float* mask_token;              /* forward in: fp32 [192], 16-byte aligned, required where mask is set */
  float* dmask_token;                   /* backward out (+=): fp32 [192], 4-byte aligned: the sum of the residual-stream
                                           gradient of the masked (image, patch) tokens; only with weight_grads = 1 */
} v2s_group_outputs_t;

/* ViTBackbone.forward for up to 4 backbones (ref:ssp_vit2spn_tiny.py:114-118; HF
 * modeling_vit.py:100-128,328-346): patch-embed, 12 pre-LN blocks, mean over 197 tokens. */
int v2s_backbone_forward(const v2s_group_t* host_groups, const v2s_group_outputs_t* host_outputs /* [n_groups] or NULL */,
                         int n_groups, int batch, int mode, void* workspace, int64_t workspace_bytes, void* stream);
/* Autograd backward of the above for the groups with slot >= 0 (ref:213 loss.backward()), over blocks
 * [layer_lo, layer_hi) only, highest block first: [0, V2S_LAYERS) is the whole backward.  layer_hi == V2S_LAYERS starts
 * from dfeat / dhidden; layer_lo == 0 ends with the embedding gradients; the residual-stream gradient is carried between
 * calls in the workspace.  The flat gradient layout is block-contiguous, so after the call for [lo, hi) the gradients of
 * those blocks are final: a data-parallel host can all-reduce that slice while the next range computes (SURVEY 8e).
 * weight_grads = 1: weight gradients accumulated (+=) into grads; saved groups without grads are skipped.  0: no
 * parameter gradient is computed and grads may be NULL (frozen backbones; no deterministic scratch is used). */
int v2s_backbone_backward(const v2s_group_t* host_groups, const v2s_group_outputs_t* host_outputs /* [n_groups] or NULL */,
                          int n_groups, int batch, int mode, void* workspace, int64_t workspace_bytes, int layer_hi,
                          int layer_lo, int weight_grads, void* stream);

/* projection_head + prediction_head on the concatenated online features and projection_head on
 * the target features (ref:ssp_vit2spn_tiny.py:153-158), fused with the loss
 *   -mean(cos(p, z)) / accumulation_steps   (ref:174,211; eps 1e-8)
 * and its backward through both heads down to d loss / d online features.
 *   head_params / head_grads: flat fp32 (v2s_heads_layout); grads accumulated (+=)
 *   feat_online / feat_target: [batch,384] fp32;  dfeat_online: out [batch,384]
 *   mask_online / mask_target: dropout multipliers [batch,1024] (0 or 1/(1-p)); NULL = no dropout
 *   pred / target_proj: optional outs [batch,128];  loss: out, 1 float (already / accum)
 *   upstream gradient of the loss = grad_scale * *grad_scale_dev; grad_scale_dev may be NULL (= 1).  grad_scale is a
 *   host value (1.0, or a fixed loss scale); grad_scale_dev is read on the device (torch.amp.GradScaler's scale tensor:
 *   scaler.scale(loss).backward() of ref:213 without a host synchronisation) */
int v2s_heads_loss_fwd_bwd(const float* head_params, float* head_grads, const float* feat_online,
                           const float* feat_target, const float* mask_online,
                           const float* mask_target, float* dfeat_online, float* pred,
                           float* target_proj, float* loss, int batch, int accumulation_steps,
                           float grad_scale, const float* grad_scale_dev, int with_backward, void* workspace,
                           int64_t workspace_bytes, void* stream);

/* The same three stages as separate calls, for the autograd-compatible path where the script's
 * own criterion computes the loss between forward and backward (ref:210-213).  The heads'
 * intermediates stay in the first batch*32768 bytes of `workspace` between the two calls. */
int v2s_heads_forward(const float* head_params, const float* feat_online, const float* feat_target,
                      const float* mask_online, const float* mask_target, float* pred,
                      float* target_proj, int batch, void* workspace, int64_t workspace_bytes,
                      void* stream);
int v2s_heads_backward(const float* head_params, float* head_grads, const float* feat_online,
                       const float* mask_online, const float* dpred, float* dfeat_online, int batch,
                       void* workspace, int64_t workspace_bytes, void* stream);
/* SimMIM head of transformers' ViTForMaskedImageModeling (encoder_stride 16) on the CUDA path.  Forward: seq = the final
 * LayerNorm (eps 1e-12) of the 196 patch rows of hidden [batch,197,192] (hidden_states[12]; CLS dropped); reconstruction
 * [batch,3,224,224] fp32 = PixelShuffle(16)(Conv2d(192, 768, 1)(seq)), always written; with mask (uint8 [batch,196],
 * nonzero = masked) also loss (1 float) = sum over masked pixels and the 3 channels of |pixels - reconstruction| /
 * (256 n + 1e-5) / 3, n = masked patches, bit-reproducible (fixed summation order).  pixels: fp32 NCHW [batch,3,224,224],
 * read only with a mask.  ln_gamma / ln_beta / dec_w [768,192] / dec_b [768] are fp32 (the 16-bit modes cast a copy of
 * dec_w into the workspace).  with_backward != 0 keeps in the workspace what v2s_mim_backward reads (the normalised rows,
 * their statistics, the signs sign(r - x) of the masked rows, the W_dec copy, the denominator): pass the same workspace,
 * batch, mode, mask and hidden to the backward.
 * Backward of loss: dloss_dev is the loss's upstream gradient, read on the device (GradScaler's scale included).  dhidden
 * [batch,197,192] is overwritten (CLS rows 0; NULL = not wanted); dpixels (the direct term -c sign, NULL = not wanted),
 * d_ln_gamma / d_ln_beta, d_dec_w / d_dec_b (NULL = frozen) are accumulated (+=).  Deterministic mode
 * (v2s_set_deterministic): fixed-order sums; size the workspace while the switch is on. */
int64_t v2s_mim_workspace_bytes(int batch, int mode);
int v2s_mim_forward(const float* hidden, const float* ln_gamma, const float* ln_beta, const float* dec_w,
                    const float* dec_b, const float* pixels, const uint8_t* mask, float* reconstruction, float* loss,
                    int with_backward, int batch, int mode, void* workspace, int64_t workspace_bytes, void* stream);
int v2s_mim_backward(const float* hidden, const float* ln_gamma, const float* dec_w, const uint8_t* mask,
                     const float* dloss_dev, float* dhidden, float* dpixels, float* d_ln_gamma, float* d_ln_beta,
                     float* d_dec_w, float* d_dec_b, int batch, int mode, void* workspace, int64_t workspace_bytes,
                     void* stream);

/* Classification head of transformers' ViTForImageClassification on the CUDA path.  Forward: xhat = the final LayerNorm
 * (eps 1e-12) of the CLS rows of hidden [batch,197,192] (hidden_states[12]); logits [batch, num_labels] fp32 =
 * xhat cls_w^T + cls_b, always written (cls_w [num_labels,192] and cls_b fp32; the 16-bit modes cast a copy of cls_w,
 * padded with zero rows to a multiple of 8, into the workspace).  loss_kind (V2S_CLS_LOSS_*) != NONE also writes loss (1
 * float), the mean of transformers' loss over its labels, bit-reproducible (fixed summation order):
 *   CE:  labels int64 [batch]; cross-entropy, -100 ignored, mean over the other rows (all ignored: NaN, as torch).  A
 *        label outside [0, num_labels) other than -100 makes the loss NaN; it is never used as an index.
 *   MSE: labels fp32 [batch, num_labels]; mean squared error over all elements.
 *   BCE: labels fp32 [batch, num_labels]; binary cross-entropy with logits, mean over all elements.
 * with_backward != 0 keeps in the workspace what v2s_cls_backward reads (xhat, its statistics, the unscaled loss
 * gradient, the label count, the cls_w copy): pass the same workspace, batch, mode, num_labels, loss_kind and hidden.
 * Backward: G = (*dloss_dev / count) d loss-sum / d logits + dlogits, formed in fp32 and cast to the GEMM operand type.
 * dloss_dev (the loss's upstream gradient, read on the device: GradScaler's scale included; needs a loss) and dlogits
 * (fp32 [batch, num_labels]) may each be NULL, not both.  dhidden [batch,197,192] is overwritten (patch rows 0; NULL =
 * not wanted); d_ln_gamma / d_ln_beta, d_cls_w / d_cls_b (NULL = frozen) are accumulated (+=).  Stages whose outputs are
 * all NULL are skipped.  Deterministic mode (v2s_set_deterministic): fixed-order sums; size the workspace while the
 * switch is on. */
#define V2S_CLS_LOSS_NONE 0
#define V2S_CLS_LOSS_CE 1
#define V2S_CLS_LOSS_MSE 2
#define V2S_CLS_LOSS_BCE 3
int64_t v2s_cls_workspace_bytes(int batch, int num_labels, int mode);
int v2s_cls_forward(const float* hidden, const float* ln_gamma, const float* ln_beta, const float* cls_w, const float* cls_b,
                    int num_labels, int loss_kind, const void* labels, float* logits, float* loss, int with_backward,
                    int batch, int mode, void* workspace, int64_t workspace_bytes, void* stream);
int v2s_cls_backward(const float* hidden, const float* ln_gamma, const float* cls_w, int num_labels, int loss_kind,
                     const void* labels, const float* dlogits, const float* dloss_dev, float* dhidden, float* d_ln_gamma,
                     float* d_ln_beta, float* d_cls_w, float* d_cls_b, int batch, int mode, void* workspace,
                     int64_t workspace_bytes, void* stream);

/* nn.CosineSimilarity(dim=1) loss of ref:174,211 and (optionally, dpred != NULL) its gradient */
int v2s_cosine_loss(const float* pred, const float* target_proj, float* loss, float* dpred, int batch,
                    int accumulation_steps, float grad_scale, void* stream);

/* InfoNCE with global negatives (BASELINE north_star (3) and config 3; the reference itself has no such loss —
 * ref:ssp_vit2spn_tiny.py:174,211 is the negative-free cosine loss above — so this is an opt-in mode, SURVEY D2/D3):
 *   logits[i][j] = cos(pred_i, keys_j) / temperature over ALL n_keys gathered target projections (the host all-gathers
 *   target_proj over the data-parallel ranks: keys = [n_keys,128], this rank's positives are rows label_offset + i),
 *   loss = mean_i CE(logits[i], label_offset + i) / accumulation_steps, dpred = grad_scale * d loss / d pred (keys are
 *   detached like ref:158).  Similarity, temperature scale, row log-sum-exp, cross-entropy and backward are one kernel.
 *   row_loss: scratch [batch]; grad_scale_dev: optional device-resident extra factor (GradScaler), may be NULL. */
int v2s_infonce_loss(const float* pred, const float* keys, float* loss, float* row_loss, float* dpred, int batch,
                     int n_keys, int64_t label_offset, float temperature, int accumulation_steps, float grad_scale,
                     const float* grad_scale_dev, void* stream);

/* dropout multipliers for the projection head: out[i] = keep ? 1/(1-p) : 0, counter-based RNG */
int v2s_dropout_mask(float* mask, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream);

/* torch.optim.Adam.step (ref:173,216) over up to 4 flat ranges: defaults betas (0.9,0.999),
 * eps 1e-8, no weight decay unless weight_decay != 0 (L2, as the fine-tune scripts use).
 * Hyper-parameters are doubles, converted exactly as torch converts its Python floats.
 * `step` is the 1-based step count; grads are multiplied by grad_scale first (1/world, 1/scale).
 * If params_lp != NULL its 16-bit shadow copy, in format lp_format (V2S_LP_BF16 / V2S_LP_FP16), is refreshed in the
 * same pass. */
typedef struct v2s_range {
  float* params;
  const float* grads;
  float* exp_avg;
  float* exp_avg_sq;
  void* params_lp;
  int64_t numel;
} v2s_range_t;
int v2s_adam_step(const v2s_range_t* host_ranges, int n_ranges, int64_t step, double lr, double beta1,
                  double beta2, double eps, double weight_decay, double grad_scale, int lp_format, void* stream);
/* The optimizer step under torch.amp.GradScaler (ref:ssp_vit2spn_tiny.py:175,216-217: scaler.step(optimizer) /
 * scaler.update()), without a host synchronisation: the step count lives on the device and the call is a no-op when
 * the scaler found an inf / nan.  state8 = 8 caller-owned device floats, state8[0] = optimizer steps taken so far
 * (initialise to 0; [1..7] are scratch); gradients are multiplied by grad_multiplier / (*grad_scale_dev)
 * (grad_scale_dev = the scaler's scale tensor, may be NULL = 1); found_inf_dev (may be NULL) != 0 skips the update and
 * leaves the step count unchanged, as torch's fused Adam does.  No host-side value changes from call to call, so the
 * call can be captured in a CUDA graph.  advance_step = 1 starts a new optimizer step (advances state8[0] and derives
 * the step's hyper-parameters into state8[1..4]); 0 applies the step already prepared in state8 to further ranges
 * (more than 4 ranges sharing one step count). */
int v2s_adam_step_amp(const v2s_range_t* host_ranges, int n_ranges, float* state8, double lr, double beta1,
                      double beta2, double eps, double weight_decay, double grad_multiplier,
                      const float* grad_scale_dev, const float* found_inf_dev, int lp_format, int advance_step,
                      void* stream);

/* update_target_network (ref:162-166): target = m*target + (1-m)*online over flat buffers; host_targets_lp (may be
 * NULL): the targets' 16-bit shadow copies, refreshed in the same pass in format lp_format (V2S_LP_BF16 / V2S_LP_FP16) */
int v2s_ema_update(float* const* host_targets, const float* const* host_onlines,
                   void* const* host_targets_lp, int n_pairs, int64_t numel, double momentum, int lp_format,
                   void* stream);

/* fp32 → 16-bit shadow copy of a flat buffer in the given format (V2S_LP_BF16 / V2S_LP_FP16) */
int v2s_cast_lp(const float* src, void* dst, int64_t numel, int lp_format, void* stream);

/* synthetic OCTMNIST-shaped input pipeline (ref:ssp_vit2spn_tiny.py:84-96, deterministic part):
 * uint8 [batch,1,28,28] → bilinear 224x224 → 3 channels → ImageNet normalise → fp32 NCHW */
int v2s_preprocess_u8(const uint8_t* src, float* dst, int batch, void* stream);
/* the same pipeline written straight as the 16-bit patch matrix of v2s_group.x_format = 1 (SURVEY 8f N1: skips the
 * 77 MB fp32 image tensor per view and the im2col pass; bit-identical to v2s_preprocess_u8 + the library's own im2col):
 * uint8 [n_images,1,28,28] -> [n_images*196, 768]; lp_format 0 = bf16, 1 = fp16 */
int v2s_preprocess_u8_patches(const uint8_t* src, void* patch_rows, int n_images, int lp_format, void* stream);

/* GPU half of the reference's augmentation pipeline, from `transforms.Resize((224, 224))` on
 * (ref:ssp_vit2spn_tiny.py:90-95): Pillow-exact BILINEAR resize of the 8-bit view (coefficient tables from the
 * host: bounds [224,2] = first source index and tap count, coefs [224,ksize] in 22-bit fixed point) -> ToTensor
 * -> GaussianBlur 3x3 with per-view taps k1d [n,3] (NULL / taps {0,1,0}: none) -> RandomErasing rectangle
 * erase [n,4] = top, left, height, width set to 0 (NULL / height <= 0: none) -> Normalize with host_mean3 /
 * host_std3, written to all 3 channels.  src: uint8 [n, in_size, in_size] (in_size <= 64), dst: fp32 [n,3,224,224]. */
int v2s_augment_finish_u8(const uint8_t* src, int n, int in_size, const int32_t* bounds, const int32_t* coefs, int ksize,
                          const float* k1d, const int32_t* erase, const float* host_mean3, const float* host_std3,
                          float* dst, void* stream);

/* Persistent kernels (GEMM, MLP, attention forward) size their grids to at most n_sms SMs until reset with 0: leaves
 * SMs to a collective that runs concurrently with the backward pass (gradient all-reduce overlap, SURVEY 8e). */
int v2s_set_sm_limit(int n_sms);

/* Deterministic mode (on != 0; off by default), read when work is enqueued and covering every entry point: the backward
 * passes (backbone and heads) sum every cross-CTA reduction in a fixed order -- split-K weight gradients, bias and
 * LayerNorm parameter gradients, embedding gradients -- so their results are bit-identical from run to run on the same
 * device model, batch, compute mode and inputs.  The split-K split count then follows the device's SM count, not
 * v2s_set_sm_limit.  The partials and arrival counters live at the tail of the workspace: while the switch is on,
 * v2s_workspace_bytes includes them (for n_saved > 0).  A backward fails when the workspace has no room for them beyond
 * the stash and backward regions it uses; they may then overlay the forward-only regions, which a backward does not
 * read, so size the workspace while the switch is on.  With the
 * switch off nothing changes, v2s_workspace_bytes included.  Python sets it from torch.are_deterministic_algorithms_enabled(). */
int v2s_set_deterministic(int on);

/* test hooks: individual operators, used by tests/ to localise a parity failure */
/* GEMM, 16-bit operands: which 0 NT (a [m,k], b [n,k] -> c [m,n] 16-bit), 1 NN (b [k,n]), 2 TN (a [k,m], b [k,n],
 * c [m,n] fp32 +=, split-K), 3 NT with fp32 c, 4 = 2 plus the bias row sums of a (+=) in c[m*n .. m*n + m),
 * 5 the image gradient of the patch embedding (a = patch-row gradient [m = batch*196, 192], b = W_pe [192, 768], c = fp32
 * [batch,3,224,224] written; n = 768, k = 192, tensor-core kernel only).
 * variant bit 0 = SIMT kernel, bit 1 = fp16 instead of bf16.  In deterministic mode (v2s_set_deterministic), which 2 / 4
 * take their scratch from the caller: c continues after its outputs with 1024 + n_sms * (128 * 192 + 128) floats
 * (n_sms = the device's SM count; m a multiple of 8). */
int v2s_test_gemm(int which, const void* a, const void* b, void* c, int m, int n, int k,
                  int variant, void* stream);
/* fused MLP half of a block (mlp_tc.cu), one backbone: mode 0 forward (a = LN2 output [m,192]; writes optional u, h
 * [m,768], out = x_mid + b2 + gelu(a W1^T + b1) W2^T fp32 [m,192], optional LayerNorm of out), mode 1 backward
 * (a = d out [m,192], u in, h = du out [m,768], out = d a [m,192]); 16-bit tensors are bf16 (lp_f16 0) or fp16 (1) */
int v2s_test_mlp(int mode, const void* a, const void* w1, const void* w2, const float* b1, const float* b2, void* u,
                 void* h, const float* resid, void* out, void* ln_out, const float* ln_gamma, const float* ln_beta,
                 float* ln_mean, float* ln_rstd, int m, int lp_f16, void* stream);
/* which 0: forward (qkv -> ctx, lse); 1: backward (qkv, ctx, lse, dctx -> dqkv); 2: attention probabilities
 * (qkv, lse -> fp32 [batch,3,197,197] written to ctx); 3: their gradient dctx V^T (qkv, dctx -> fp32 [batch,3,197,197]
 * written to ctx).  variant bit 0 = SIMT kernels, bit 1 = fp16 instead of bf16 */
int v2s_test_attention(int which, const void* qkv, void* ctx, float* lse, const void* dctx, void* dqkv,
                       int batch, int variant, void* stream);
/* reads and clears the device-side pipeline-protocol error flag of the tcgen05 kernels (0 = ok) */
int v2s_debug_flag(void);
/* per-role stall cycle counters of CTA 0 of the last tcgen05 GEMM (only with V2S_GEMM_DEBUG=1) */
int v2s_debug_counters(int64_t* host32);
int64_t v2s_launch_count(void); /* kernels launched by this library since load (bench: gpu_launches) */
/* device-event timing per kernel class (bench.py roofline); off by default, enabling resets it */
int v2s_prof_enable(int on);
int v2s_prof_report(char* host_buf, int64_t buf_bytes);

#ifdef __cplusplus
}
#endif
#endif /* VIT2SPN_H_ */
