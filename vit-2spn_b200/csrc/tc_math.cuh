// Shared device helpers of the tensor-core kernels: the 16-bit operand formats (bf16 / fp16) and the fast erf-GELU
// used by the chained MLP kernel.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "ptx.cuh"

namespace v2s {

// ---- 16-bit operand formats -------------------------------------------------------------------
// The tcgen05 kind::f16 MMA takes bf16 or fp16 operands (format field of the instruction descriptor); everything
// else that differs between the two "low-precision" compute modes is how a pair of floats is packed / unpacked.
//   bf16: torch.autocast(bfloat16) — no loss scaling needed
//   fp16: the reference's actual CUDA precision (torch.autocast default + GradScaler, ref:ssp_vit2spn_tiny.py:175,209-217)
struct LpBf16 {
  static constexpr uint32_t kIdescFmt = 1;      // a_format / b_format = BF16
  static constexpr bool kIsF16 = false;
  static constexpr uint32_t kOnePair = 0x3F803F80u;   // (1.0, 1.0)
  static __device__ __forceinline__ uint32_t pack(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float lo(uint32_t w) { return __uint_as_float(w << 16); }
  static __device__ __forceinline__ float hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
};
struct LpF16 {
  static constexpr uint32_t kIdescFmt = 0;      // a_format / b_format = F16
  static constexpr bool kIsF16 = true;
  static constexpr uint32_t kOnePair = 0x3C003C00u;   // (1.0, 1.0)
  static __device__ __forceinline__ uint32_t pack(float a, float b) {
    __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float lo(uint32_t w) { return __low2float(*reinterpret_cast<const __half2*>(&w)); }
  static __device__ __forceinline__ float hi(uint32_t w) { return __high2float(*reinterpret_cast<const __half2*>(&w)); }
};

// instruction descriptor for kind::f16 with a given operand format: 16-bit x 16-bit -> fp32, M x N tile
__host__ __device__ constexpr uint32_t make_idesc_lp(uint32_t fmt, int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                         // c_format = F32
         | (fmt << 7)                      // a_format: 0 = F16, 1 = BF16
         | (fmt << 10)                     // b_format
         | ((uint32_t)a_mn_major << 15)    // a_major: 0 = K-major, 1 = MN-major
         | ((uint32_t)b_mn_major << 16)    // b_major
         | ((uint32_t)(N >> 3) << 17)      // n_dim
         | ((uint32_t)(M >> 4) << 24);     // m_dim
}

// ---- fast erf-GELU ------------------------------------------------------------------------------
// Forward: gelu(x) = relu(x) - |x| Phi(-|x|) with Phi(-a) = 0.5 exp2(a (c0 + c1 a + .. + c4 a^4)) — log2 of the normal
// tail is smooth, so a degree-5 exponent fitted (minimax on the ABSOLUTE error of a Phi(-a), a in [0, 14]; the fit
// script is tools/fit_gelu.py) gives |gelu error| < 7.1e-7 over all x in fp32 arithmetic: 9 FP + ONE MUFU.EX2 per
// element.  The GELU epilogues are issue / MUFU co-bound, and the Abramowitz-Stegun 7.1.26 form used before (and still
// used by the derivative, which needs exp(-x^2/2) anyway) costs 13 FP + MUFU.RCP + MUFU.EX2.
// The exponent stays <= 0 and tends to -inf with |x| (leading coefficient negative): no clamp needed.
__device__ __forceinline__ float gelu_fast(float x) {
  const float a = fabsf(x);
  float r = fmaf(-4.86990211e-04f, a, 7.19165942e-03f);
  r = fmaf(r, a, -5.21313134e-02f);
  r = fmaf(r, a, -4.59609083e-01f);
  r = fmaf(r, a, -1.15099679e+00f);
  const float e = ptx::ex2_approx(r * a);          // 2 Phi(-|x|)
  return fmaf(-0.5f * a, e, fmaxf(x, 0.0f));
}
// Derivative: gelu'(x) = Phi(x) + x phi(x) satisfies gelu'(x) + gelu'(-x) = 1, so it is m(|x|) for x <= 0 and
// 1 - m(|x|) for x > 0 with m(a) = Phi(-a) - a phi(a) = exp2(q(a)) T(a): the same exponent q as the forward form and a
// degree-5 polynomial T fitted to the absolute error of m (|gelu' error| < 2.6e-6): 15 FP + ONE MUFU.EX2 (the
// Abramowitz-Stegun form used before needed MUFU.RCP + MUFU.EX2; the GELU' epilogue was MUFU co-bound).
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float a = fabsf(x);
  float r = fmaf(-4.86990211e-04f, a, 7.19165942e-03f);
  r = fmaf(r, a, -5.21313134e-02f);
  r = fmaf(r, a, -4.59609083e-01f);
  r = fmaf(r, a, -1.15099679e+00f);
  float t = fmaf(-8.5974e-04f, a, 1.004244e-02f);
  t = fmaf(t, a, -5.430038e-02f);
  t = fmaf(t, a, -3.1854429e-01f);
  t = fmaf(t, a, -3.9889585e-01f);
  t = fmaf(t, a, 4.9999758e-01f);
  const float m = t * ptx::ex2_approx(r * a);
  return x > 0.0f ? 1.0f - m : m;
}

}  // namespace v2s
