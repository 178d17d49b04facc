// Generic grouped SIMT GEMM with fused epilogues: the fp32 check-mode GEMM and the debugging
// reference for the tcgen05 kernels.  C[M,N] = sum_k A(m,k) * B(k,n), arbitrary strides.
#pragma once
#include "common.cuh"

namespace v2s {

enum GemmEpi : int {
  EPI_STORE = 0,        // out = alpha*acc (+ bias)
  EPI_BIAS_RESID = 1,   // out(fp32) = acc + bias + resid
  EPI_BIAS_GELU = 2,    // u = acc + bias -> out (optional); gelu(u) -> out2
  EPI_PATCH = 3,        // patch-embed: token-row remap, + bias + position embedding (aux)
  EPI_DGELU = 4,        // out = acc * gelu'(aux)
  EPI_ACCUM = 5,        // atomicAdd(out(fp32), alpha*acc)  (wgrad, split-K)
  EPI_BIAS_RELU_MASK = 6,  // a = relu(acc+bias) -> out ; a*mask -> out2
  EPI_DRELU_MASK = 7,      // out = acc * (aux > 0) * mask
  // tensor-core path only (the SIMT kernel refuses it): acc [B*196, 768] of the patch-embedding dgrad is stored fp32
  // straight into the NCHW image gradient out [B,3,224,224]: row (b, py, px), column c*256 + ky*16 + kx
  EPI_PIXELS = 8,
  // tensor-core path only: SimMIM's 1x1-conv decoder, acc [B*196, 768] + bias stored fp32 into the NCHW reconstruction
  // out [B,3,224,224] with EPI_PIXELS' permutation (PixelShuffle(16)); with mim_mask also the masked L1 loss partials
  // (one per output tile) and the sign rows for the backward (see gemm_tc.cu)
  EPI_MIM = 9,
};

struct GemmDesc {
  int M, N, K;
  int64_t a_rs, a_cs;  // A(m,k) = A[m*a_rs + k*a_cs]
  int64_t b_rs, b_cs;  // B(k,n) = B[k*b_rs + n*b_cs]
  int a_remap;         // patch index b*np+p -> token row b*nt+1+p: 1 = on A's m index, 2 = on A's k index
  int b_remap;         // same for the K index of B (wgrad of the patch embedding)
  int split_k;         // number of K splits: EPI_ACCUM (atomic adds), or EPI_STORE with split_stride > 0
  int64_t split_stride; // EPI_STORE + split_k: split s writes its partial result at out + s * split_stride (no bias)
  int groups;
  const void* A[MAXG];
  const void* B[MAXG];
  int epi;
  const float* bias[MAXG];
  const float* resid[MAXG];
  const void* aux[MAXG];
  const float* mask[MAXG];
  void* out[MAXG];
  void* out2[MAXG];
  // EPI_BIAS_RESID, tensor-core path, N == 192 only: LayerNorm of the result row fused into the epilogue
  void* ln_out[MAXG];          // bf16 [M,192] normalised output (NULL: no fusion)
  const float* ln_gamma[MAXG];
  const float* ln_beta[MAXG];
  float* ln_mean[MAXG];        // optional [M]
  float* ln_rstd[MAXG];
  float* rowsum_out[MAXG];  // EPI_ACCUM, tensor-core path only: rowsum_out[m] += sum_k A(m,k) (bias gradient for free)
  int64_t ldc;
  float alpha;
  // tensor-core path, programmatic dependent launch: every input of this GEMM was produced at least two kernels
  // back in the stream and its output is not touched by the kernel launched just before it -> start without
  // draining that kernel, wait for it just before exiting (see gemm_tc.cu)
  int late_wait;
  int lp_f16;       // tensor-core path: the 16-bit operands / outputs are fp16 (1) instead of bf16 (0)
  // tensor-core split-K wgrad launches only: two different problems (same K = token dimension) in one launch.  Groups
  // [0, groups / 2) use M, N and the strides above, groups [groups / 2, groups) use M2, N2 (a_cs = M2, b_rs = N2,
  // ldc = N2: both operands token-major).  One launch ramp and one balanced wave instead of two.
  int M2, N2;
  // deterministic mode, tensor-core split-K wgrad (EPI_ACCUM) only: scratch for the partial tiles and the per-output-tile
  // arrival counters; the split count then ignores v2s_set_sm_limit and the partials are summed in split order
  const DetScratch* det;
  // EPI_MIM with a mask: input images (fp32 NCHW), uint8 [M] patch mask, 16-bit sign rows [M, N] (NULL: none), loss partials
  const float* mim_x;
  const uint8_t* mim_mask;
  void* mim_dsign;
  float* mim_loss_part;
  // the token geometry of EPI_PATCH and the row remaps (patch index b*np+p -> token row b*nt+1+p) and of EPI_PIXELS (image
  // img_h x img_w, patch grid img_gw wide): 196 / 197 / 224 x 224 / 14 unless the image size is set otherwise
  int np, nt, img_h, img_w, img_gw;
};

inline GemmDesc make_gemm_desc() {
  GemmDesc d;
  memset(&d, 0, sizeof(d));
  d.alpha = 1.0f;
  d.split_k = 1;
  d.groups = 1;
  d.np = NP; d.nt = NT; d.img_h = V2S_IMG; d.img_w = V2S_IMG; d.img_gw = V2S_IMG / 16;
  return d;
}

// type tags: 0 = fp32, 1 = bf16, 2 = fp16
int launch_gemm_simt(const GemmDesc& d, int ta, int tb, int to, cudaStream_t stream);

}  // namespace v2s
