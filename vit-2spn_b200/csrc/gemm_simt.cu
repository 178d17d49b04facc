// Generic grouped SIMT GEMM (fp32 accumulate) with fused epilogues.  See gemm_simt.cuh.
#include <string.h>

#include "gemm_simt.cuh"

namespace v2s {

namespace {

constexpr int BK = 16, PAD = 4;   // tile = (16*TM) x (16*TM) x 16, 256 threads, TM x TM outputs per thread

__device__ __forceinline__ int64_t remap_row(int64_t r, int np) { return r + r / np + 1; }

template <typename TA, typename TB, typename TO, int TM>
__global__ void __launch_bounds__(256) gemm_simt_kernel(const GemmDesc d) {
  constexpr int BM = 16 * TM, BN = 16 * TM;
  __shared__ float As[BK][BM + PAD];
  __shared__ float Bs[BK][BN + PAD];
  const int g = blockIdx.z;
  const TA* __restrict__ A = static_cast<const TA*>(d.A[g]);
  const TB* __restrict__ B = static_cast<const TB*>(d.B[g]);
  const int tiles_n = (d.N + BN - 1) / BN;
  const int tile_n = blockIdx.y % tiles_n;
  const int split = blockIdx.y / tiles_n;
  const int m0 = blockIdx.x * BM, n0 = tile_n * BN;
  int k_begin = 0, k_end = d.K;
  if (d.split_k > 1) {
    int chunk = ((d.K + d.split_k - 1) / d.split_k + BK - 1) / BK * BK;
    k_begin = split * chunk;
    k_end = min(d.K, k_begin + chunk);
  }
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  float acc[TM][TM];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TM; ++j) acc[i][j] = 0.f;

  const bool a_kfast = (d.a_cs == 1);
  const bool b_kfast = (d.b_rs == 1);

  // register-prefetch double buffering: the global loads of tile k+1 are in flight while tile k is multiplied
  float ra[TM], rb[TM];
  auto load_tile = [&](int k0) {
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int e = tid + i * 256;
      int kk, mm;
      if (a_kfast) { kk = e % BK; mm = e / BK; } else { mm = e % BM; kk = e / BM; }
      const int m = m0 + mm, k = k0 + kk;
      float v = 0.f;
      if (m < d.M && k < k_end) {
        const int64_t row = d.a_remap == 1 ? remap_row(m, d.np) : (int64_t)m;
        const int64_t col = d.a_remap == 2 ? remap_row(k, d.np) : (int64_t)k;
        v = to_f<TA>(A[row * d.a_rs + col * d.a_cs]);
      }
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int e = tid + i * 256;
      int kk, nn;
      if (b_kfast) { kk = e % BK; nn = e / BK; } else { nn = e % BN; kk = e / BN; }
      const int n = n0 + nn, k = k0 + kk;
      float v = 0.f;
      if (n < d.N && k < k_end) {
        const int64_t krow = d.b_remap ? remap_row(k, d.np) : (int64_t)k;
        v = to_f<TB>(B[krow * d.b_rs + (int64_t)n * d.b_cs]);
      }
      rb[i] = v;
    }
  };
  auto store_tile = [&]() {
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int e = tid + i * 256;
      if (a_kfast) As[e % BK][e / BK] = ra[i]; else As[e / BM][e % BM] = ra[i];
      if (b_kfast) Bs[e % BK][e / BK] = rb[i]; else Bs[e / BN][e % BN] = rb[i];
    }
  };
  if (k_begin < k_end) { load_tile(k_begin); store_tile(); }
  __syncthreads();
  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    const bool has_next = k0 + BK < k_end;
    if (has_next) load_tile(k0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[TM], b[TM];
#pragma unroll
      for (int i = 0; i < TM; ++i) { a[i] = As[kk][ty * TM + i]; b[i] = Bs[kk][tx * TM + i]; }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TM; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
    if (has_next) { store_tile(); __syncthreads(); }
  }

  // ---- epilogue ----
  const float* __restrict__ bias = d.bias[g];
  const float* __restrict__ resid = d.resid[g];
  const float* __restrict__ mask = d.mask[g];
  TO* __restrict__ out = static_cast<TO*>(d.out[g]);
  TO* __restrict__ out2 = static_cast<TO*>(d.out2[g]);
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ty * TM + i;
    if (m >= d.M) continue;
#pragma unroll
    for (int j = 0; j < TM; ++j) {
      const int n = n0 + tx * TM + j;
      if (n >= d.N) continue;
      float v = acc[i][j] * d.alpha;
      const int64_t idx = (int64_t)m * d.ldc + n;
      switch (d.epi) {
        case EPI_STORE:
          if (d.split_k > 1) { out[idx + (int64_t)split * d.split_stride] = from_f<TO>(v); break; }   // partial slab
          if (bias) v += bias[n];
          out[idx] = from_f<TO>(v);
          break;
        case EPI_BIAS_RESID:
          v += bias[n] + resid[idx];
          out[idx] = from_f<TO>(v);
          break;
        case EPI_BIAS_GELU:
          v += bias[n];
          if (out) out[idx] = from_f<TO>(v);
          out2[idx] = from_f<TO>(gelu_f(v));
          break;
        case EPI_PATCH: {
          const int b = m / d.np, p = m % d.np;
          const float* pos = static_cast<const float*>(d.aux[g]);
          v += bias[n] + pos[(int64_t)(1 + p) * D + n];
          out[((int64_t)b * d.nt + 1 + p) * d.ldc + n] = from_f<TO>(v);
        } break;
        case EPI_DGELU: {
          const TO* u = static_cast<const TO*>(d.aux[g]);
          out[idx] = from_f<TO>(v * gelu_grad_f(to_f<TO>(u[idx])));
        } break;
        case EPI_ACCUM:
          atomicAdd(reinterpret_cast<float*>(d.out[g]) + idx, v);
          break;
        case EPI_BIAS_RELU_MASK: {
          v = fmaxf(v + bias[n], 0.f);
          out[idx] = from_f<TO>(v);
          out2[idx] = from_f<TO>(mask ? v * mask[idx] : v);
        } break;
        case EPI_DRELU_MASK: {
          const float* src = static_cast<const float*>(d.aux[g]);
          float t = src[idx] > 0.f ? v : 0.f;
          if (mask) t *= mask[idx];
          out[idx] = from_f<TO>(t);
        } break;
        default: break;
      }
    }
  }
}

template <typename TA, typename TB, typename TO>
int launch_t(const GemmDesc& d, cudaStream_t stream) {
  const int sk = d.split_k > 1 ? d.split_k : 1;
  const int t64 = ((d.M + 63) / 64) * ((d.N + 63) / 64) * sk * d.groups;
  if (t64 < 120) {       // small problem (the heads): 32x32 tiles put 4x more CTAs on the machine
    dim3 grid((d.M + 31) / 32, ((d.N + 31) / 32) * sk, d.groups);
    gemm_simt_kernel<TA, TB, TO, 2><<<grid, 256, 0, stream>>>(d);
  } else {
    dim3 grid((d.M + 63) / 64, ((d.N + 63) / 64) * sk, d.groups);
    gemm_simt_kernel<TA, TB, TO, 4><<<grid, 256, 0, stream>>>(d);
  }
  V2S_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int launch_gemm_simt(const GemmDesc& d, int ta, int tb, int to, cudaStream_t stream) {
  if (d.M <= 0 || d.N <= 0 || d.K <= 0) return 0;
  if (d.epi == EPI_PIXELS || d.epi == EPI_MIM) { set_error("gemm_simt: EPI_PIXELS / EPI_MIM are tensor-core epilogues"); return 1; }
  if (d.split_k > 1 && d.epi != EPI_ACCUM && !(d.epi == EPI_STORE && d.split_stride > 0)) {
    set_error("gemm_simt: split_k requires EPI_ACCUM, or EPI_STORE with a split_stride");
    return 1;
  }
  if (ta == 0 && tb == 0 && to == 0) return launch_t<float, float, float>(d, stream);
  if (ta == 1 && tb == 1 && to == 1) return launch_t<bf16, bf16, bf16>(d, stream);
  if (ta == 1 && tb == 1 && to == 0) return launch_t<bf16, bf16, float>(d, stream);
  if (ta == 2 && tb == 2 && to == 2) return launch_t<f16, f16, f16>(d, stream);
  if (ta == 2 && tb == 2 && to == 0) return launch_t<f16, f16, float>(d, stream);
  set_error("gemm_simt: unsupported type combination %d %d %d", ta, tb, to);
  return 1;
}

}  // namespace v2s
