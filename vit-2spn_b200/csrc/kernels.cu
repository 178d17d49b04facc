// Memory-bound kernels of the SSP step: im2col, LayerNorm fwd/bwd, bias-gradient column sums,
// token mean-pool, embedding backward, cosine loss (+backward), Adam, EMA, casts, dropout mask,
// synthetic input pipeline.  All are coalesced / vectorised HBM kernels with warp-shuffle
// reductions; grouped kernels use blockIdx.y|z as the backbone index.
#include <string.h>

#include "kernels.cuh"

namespace v2s {

namespace {

template <typename T> struct G4 { T p[MAXG]; };
template <typename T, typename S> G4<T> pack4(S const* src, int groups) {
  G4<T> r;
  for (int i = 0; i < MAXG; ++i) r.p[i] = (src && i < groups) ? (T)src[i] : (T) nullptr;
  return r;
}

// ------------------------------------------------------------------------------------------
// im2col: NCHW fp32 image → patch matrix [B*196, 768], k = c*256 + ky*16 + kx
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void im2col_kernel(G4<const float*> x, G4<T*> out, int B) {
  const int g = blockIdx.y;
  const int64_t total = (int64_t)B * NP * (KPE / 4);
  const float* __restrict__ xin = x.p[g];
  T* __restrict__ o = out.p[g];
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int kx4 = idx % 4;
    const int ky = (idx / 4) % 16;
    const int c = (idx / 64) % 3;
    const int p = (idx / 192) % NP;
    const int b = idx / (192 * NP);
    const int py = p / 14, px = p % 14;
    const float4 v = *reinterpret_cast<const float4*>(
        xin + (((int64_t)b * 3 + c) * V2S_IMG + py * 16 + ky) * V2S_IMG + px * 16 + kx4 * 4);
    T* dst = o + ((int64_t)b * NP + p) * KPE + c * 256 + ky * 16 + kx4 * 4;
    dst[0] = from_f<T>(v.x); dst[1] = from_f<T>(v.y); dst[2] = from_f<T>(v.z); dst[3] = from_f<T>(v.w);
  }
}

// Masked patch tokens (transformers' bool_masked_pos): per group a uint8 [B,196] mask (nonzero = masked; NULL = none)
// and the fp32 [192] mask token that replaces a masked patch embedding before the position embedding is added.  The
// kernels below take them as their last argument and read them only in their MASK instantiation.
struct MaskArgs { const uint8_t* mask[MAXG]; const float* token[MAXG]; };
MaskArgs pack_masks(const uint8_t* const* mask, const float* const* token, int groups) {
  MaskArgs m;
  for (int i = 0; i < MAXG; ++i) {
    m.mask[i] = (mask && i < groups) ? mask[i] : nullptr;
    m.token[i] = (token && i < groups) ? token[i] : nullptr;
  }
  return m;
}

// fp32 check mode: the patch GEMM's epilogue wrote hidden[b,1+p,:] = tok + pos[1+p]; this adds the CLS row and, with
// MASK, overwrites each masked patch row with mask_token + pos[1+p]
template <bool MASK>
__global__ void cls_rows_kernel(G4<const float*> params, G4<float*> hidden, MaskArgs mk) {
  const int g = blockIdx.y, b = blockIdx.x, n = threadIdx.x;
  const float* p = params.p[g];
  hidden.p[g][(int64_t)b * NT * D + n] = p[OFF_CLS + n] + p[OFF_POS + n];
  if constexpr (MASK) {
    const uint8_t* m = mk.mask[g];
    if (!m) return;
    const float t = mk.token[g][n];
    for (int q = 0; q < NP; ++q)
      if (m[(int64_t)b * NP + q]) hidden.p[g][((int64_t)b * NT + 1 + q) * D + n] = t + p[OFF_POS + (int64_t)(1 + q) * D + n];
  }
}

// hidden[b,0,:] = cls + pos[0];  hidden[b,1+p,:] = tok[b*196+p,:] + pos[1+p]   (HF:117-124)
// MASK: a masked patch row takes mask_token + pos[1+p] instead (HF:ViTEmbeddings.forward, as a select)
// one float4 per thread; blockIdx.y = image, blockIdx.z = backbone
template <bool MASK>
__global__ void __launch_bounds__(256) assemble_tokens_kernel(G4<const float*> params, G4<const float*> tok,
                                                              G4<float*> hidden, MaskArgs mk) {
  const int g = blockIdx.z, b = blockIdx.y;
  const float* __restrict__ p = params.p[g];
  const float* __restrict__ tk = tok.p[g];
  float* __restrict__ h = hidden.p[g];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < NT * (D / 4); i += gridDim.x * blockDim.x) {
    const int t = i / (D / 4), c = (i % (D / 4)) * 4;
    const float4 pos = *reinterpret_cast<const float4*>(p + OFF_POS + (int64_t)t * D + c);
    float4 v;
    if constexpr (MASK) {
      const float* src = (t == 0) ? p + OFF_CLS + c : tk + ((int64_t)b * NP + t - 1) * D + c;
      if (t > 0 && mk.mask[g] && mk.mask[g][(int64_t)b * NP + t - 1]) src = mk.token[g] + c;
      v = *reinterpret_cast<const float4*>(src);
    } else {
      v = (t == 0) ? *reinterpret_cast<const float4*>(p + OFF_CLS + c)
                   : *reinterpret_cast<const float4*>(tk + ((int64_t)b * NP + t - 1) * D + c);
    }
    *reinterpret_cast<float4*>(h + ((int64_t)b * NT + t) * D + c) =
        make_float4(v.x + pos.x, v.y + pos.y, v.z + pos.z, v.w + pos.w);
  }
}

// compact the patch-token rows of a [B,197,192] tensor into [B*196,192] (drops the CLS rows); 8 bytes per thread
// MASK: the rows of masked patches are written as zeros (no gradient reaches W_pe, b_pe or the pixels through them)
template <typename T, bool MASK>
__global__ void __launch_bounds__(256) gather_patch_rows_kernel(G4<const T*> src, G4<T*> dst, MaskArgs mk) {
  const int g = blockIdx.z, b = blockIdx.y;
  constexpr int V = 8 / sizeof(T);                 // elements per 8-byte access
  const T* __restrict__ s = src.p[g] + ((int64_t)b * NT + 1) * D;
  T* __restrict__ d = dst.p[g] + (int64_t)b * NP * D;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < NP * D / V; i += gridDim.x * blockDim.x) {
    if constexpr (MASK)
      if (mk.mask[g] && mk.mask[g][(int64_t)b * NP + i / (D / V)]) { reinterpret_cast<uint2*>(d)[i] = make_uint2(0u, 0u); continue; }
    reinterpret_cast<uint2*>(d)[i] = reinterpret_cast<const uint2*>(s)[i];
  }
}

// the inverse permutation of im2col (stride = kernel, no overlap-add): patch rows [B*196, 768] fp32 -> NCHW fp32
// [B,3,224,224]; one float4 of the image per thread, so the stores are contiguous (fp32 check mode's image gradient)
__global__ void __launch_bounds__(256) col2im_kernel(G4<const float*> rows, G4<float*> img, int B) {
  const int g = blockIdx.y;
  const float* __restrict__ src = rows.p[g];
  float* __restrict__ dst = img.p[g];
  const int64_t total = (int64_t)B * 3 * V2S_IMG * (V2S_IMG / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int x4 = i % (V2S_IMG / 4), y = (i / (V2S_IMG / 4)) % V2S_IMG;
    const int c = (i / (V2S_IMG * V2S_IMG / 4)) % 3;
    const int64_t b = i / (3 * V2S_IMG * V2S_IMG / 4);
    const int px = x4 / 4, py = y / 16;
    reinterpret_cast<float4*>(dst)[i] = *reinterpret_cast<const float4*>(
        src + (b * NP + py * 14 + px) * KPE + c * 256 + (y % 16) * 16 + (x4 % 4) * 4);
  }
}

// ------------------------------------------------------------------------------------------
// LayerNorm over D=192 (eps 1e-12).  Half a warp per row: 16 lanes x 3 float4 = 192 floats, so a
// warp keeps two rows (6 x 128-bit loads per lane) in flight; reductions are 4 shuffle steps.
// ------------------------------------------------------------------------------------------
struct LnFwdP {
  const float* x[MAXG]; const float* gamma[MAXG]; const float* beta[MAXG];
  void* y[MAXG]; float* mean[MAXG]; float* rstd[MAXG];
  int M;
};

// sum over the 16 lanes of a half-warp; `mask` names exactly those lanes (the two half-warps of a
// warp own different rows and may leave the row loop at different iterations)
__device__ __forceinline__ float hw_sum(float v, unsigned mask) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
  return v;
}

template <typename T> __device__ __forceinline__ void store4(T* dst, float a, float b, float c, float d);
template <> __device__ __forceinline__ void store4<float>(float* dst, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(dst) = make_float4(a, b, c, d);
}
template <> __device__ __forceinline__ void store4<bf16>(bf16* dst, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo); u.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst) = u;
}
template <> __device__ __forceinline__ void store4<f16>(f16* dst, float a, float b, float c, float d) {
  __half2 lo = __floats2half2_rn(a, b), hi = __floats2half2_rn(c, d);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo); u.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst) = u;
}
template <typename T> __device__ __forceinline__ float4 load4(const T* src);
template <> __device__ __forceinline__ float4 load4<float>(const float* src) { return *reinterpret_cast<const float4*>(src); }
template <> __device__ __forceinline__ float4 load4<bf16>(const bf16* src) {
  const uint2 u = *reinterpret_cast<const uint2*>(src);
  const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&u.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
  return make_float4(__low2float(lo), __high2float(lo), __low2float(hi), __high2float(hi));
}

template <> __device__ __forceinline__ float4 load4<f16>(const f16* src) {
  const uint2 u = *reinterpret_cast<const uint2*>(src);
  const __half2 lo = *reinterpret_cast<const __half2*>(&u.x), hi = *reinterpret_cast<const __half2*>(&u.y);
  return make_float4(__low2float(lo), __high2float(lo), __low2float(hi), __high2float(hi));
}

// runs `...` with T = float / bf16 / f16 for the activation type tag 0 / 1 / 2
#define V2S_DISPATCH_AT(at, ...)                            \
  switch (at) {                                             \
    case AT_F32: { using T = float; __VA_ARGS__; } break;   \
    case AT_BF16: { using T = bf16; __VA_ARGS__; } break;   \
    default: { using T = f16; __VA_ARGS__; } break;         \
  }

// packs two floats into the 16-bit shadow format of a flat parameter buffer (bf16, or fp16 when f16 != 0)
__device__ __forceinline__ uint32_t pack_lp(float a, float b, int f16) {
  if (f16) { __half2 v = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

template <typename T>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const __grid_constant__ LnFwdP p) {
  // wait for the predecessor, THEN release the successor: a successor flagged "late wait" (gemm_tc.cu) relies on
  // everything before its predecessor being complete when it starts
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int g = blockIdx.y;
  const int hw = threadIdx.x >> 4, l = threadIdx.x & 15;
  const unsigned hmask = 0xffffu << (16 * (hw & 1));
  const float* __restrict__ x = p.x[g];
  T* __restrict__ y = static_cast<T*>(p.y[g]);
  float4 gm[3], bt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    gm[i] = reinterpret_cast<const float4*>(p.gamma[g])[l + 16 * i];
    bt[i] = reinterpret_cast<const float4*>(p.beta[g])[l + 16 * i];
  }
  for (int row = blockIdx.x * 16 + hw; row < p.M; row += gridDim.x * 16) {
    const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * D);
    float4 v[3];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) { v[i] = xr[l + 16 * i]; s += (v[i].x + v[i].y) + (v[i].z + v[i].w); }
    const float mu = hw_sum(s, hmask) * (1.0f / D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
      q += (a * a + b * b) + (c * c + d * d);
    }
    const float rs = 1.0f / sqrtf(hw_sum(q, hmask) * (1.0f / D) + LN_EPS);
    T* yr = y + (int64_t)row * D;
#pragma unroll
    for (int i = 0; i < 3; ++i)
      store4<T>(yr + 4 * (l + 16 * i), (v[i].x - mu) * rs * gm[i].x + bt[i].x, (v[i].y - mu) * rs * gm[i].y + bt[i].y,
                (v[i].z - mu) * rs * gm[i].z + bt[i].z, (v[i].w - mu) * rs * gm[i].w + bt[i].w);
    if (l == 0 && p.mean[g]) { p.mean[g][row] = mu; p.rstd[g][row] = rs; }
  }
}

// Deterministic mode: fixed-order column reduction across the CTAs of one launch.  Each CTA has written its partial row
// (n floats) to part[blk]; the CTA whose arrival completes the counter sums rows 0..nblk-1 and calls add(c, total) per
// column.  Rows are summed in R contiguous ranges (R threads per float4 column, partials through `red`, capacity
// `red_floats`), then the R range sums in order: the order depends on nblk, n and the block size only, never on which CTA
// came last.  No CTA waits for another.  Called by every thread of the CTA; n a multiple of 4.
template <typename Add>
__device__ __forceinline__ void det_reduce_rows(const float* part, int n, int nblk, unsigned* counter, float* red, int red_floats, Add add) {
  __shared__ unsigned s_last;
  __threadfence();                   // this CTA's partial row is visible device-wide before it is counted
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
    s_last = old == (unsigned)(nblk - 1);
  }
  __syncthreads();
  if (!s_last) return;
  const int n4 = n / 4;
  int R = red_floats / n;
  if (R > 8) R = 8;
  if (R > nblk) R = nblk;
  const int per = (nblk + R - 1) / R;
  for (int it = threadIdx.x; it < R * n4; it += blockDim.x) {
    const int r = it / n4, c4 = it - r * n4;
    const int b1 = min(nblk, (r + 1) * per);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int b = r * per; b < b1; ++b) {
      const float4 v = __ldcg(reinterpret_cast<const float4*>(part + (int64_t)b * n) + c4);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    float* rr = red + r * n + 4 * c4;          // `red` may be only 4-byte aligned
    rr[0] = s.x; rr[1] = s.y; rr[2] = s.z; rr[3] = s.w;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < n; c += blockDim.x) {
    float s = red[c];
    for (int r = 1; r < R; ++r) s += red[r * n + c];
    add(c, s);
  }
  if (threadIdx.x == 0) *counter = 0;      // zero again for the next launch
}

// dres (fp32, in/out) += LN-backward(dy);  dres_lp = updated dres in the activation type;
// PARAMS: dgamma / dbeta / (optional) dcolsum[n] += sum over rows of the UPDATED dres (= bias gradient of the
// linear layer that consumes this residual-stream gradient).  !PARAMS (input-gradient backward of a frozen backbone): the
// row-wise part only, no column sums.
struct LnBwdP {
  const void* dy[MAXG]; const float* x[MAXG]; const float* mean[MAXG]; const float* rstd[MAXG];
  const float* gamma[MAXG]; float* dres[MAXG]; void* dres_lp[MAXG]; float* dgamma[MAXG]; float* dbeta[MAXG];
  float* dcolsum[MAXG];
  int M;
  float* det_part;             // DET: [group][CTA][3 * 192] partial rows
  unsigned* det_counters;      // DET: one per group
};

template <typename T, bool DET, bool PARAMS>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const __grid_constant__ LnBwdP p) {
  __shared__ __align__(16) float red[16][3 * D];          // 36 KB; float4 accesses
  // wait for the predecessor, THEN release the successor: a successor flagged "late wait" (gemm_tc.cu) relies on
  // everything before its predecessor being complete when it starts
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int g = blockIdx.y;
  const int hw = threadIdx.x >> 4, l = threadIdx.x & 15;
  const unsigned hmask = 0xffffu << (16 * (hw & 1));
  const T* __restrict__ dy = static_cast<const T*>(p.dy[g]);
  const float* __restrict__ x = p.x[g];
  float* __restrict__ dres = p.dres[g];
  T* __restrict__ dlp = static_cast<T*>(p.dres_lp[g]);
  float4 gm[3], ag[3], ab[3], ac[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    gm[i] = reinterpret_cast<const float4*>(p.gamma[g])[l + 16 * i];
    ag[i] = ab[i] = ac[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int row = blockIdx.x * 16 + hw; row < p.M; row += gridDim.x * 16) {
    const float mu = p.mean[g][row], rs = p.rstd[g][row];
    const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * D);
    float4 xh[3], gd[3], d[3], o[3];
    float c1 = 0.f, c2 = 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float4 xv = xr[l + 16 * i];
      d[i] = load4<T>(dy + (int64_t)row * D + 4 * (l + 16 * i));
      o[i] = reinterpret_cast<const float4*>(dres + (int64_t)row * D)[l + 16 * i];
      xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
      gd[i] = make_float4(d[i].x * gm[i].x, d[i].y * gm[i].y, d[i].z * gm[i].z, d[i].w * gm[i].w);
      c1 += (gd[i].x + gd[i].y) + (gd[i].z + gd[i].w);
      c2 += (gd[i].x * xh[i].x + gd[i].y * xh[i].y) + (gd[i].z * xh[i].z + gd[i].w * xh[i].w);
      if constexpr (PARAMS) {
        ag[i].x += d[i].x * xh[i].x; ag[i].y += d[i].y * xh[i].y; ag[i].z += d[i].z * xh[i].z; ag[i].w += d[i].w * xh[i].w;
        ab[i].x += d[i].x; ab[i].y += d[i].y; ab[i].z += d[i].z; ab[i].w += d[i].w;
      }
    }
    c1 = hw_sum(c1, hmask) * (1.0f / D);
    c2 = hw_sum(c2, hmask) * (1.0f / D);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      o[i].x += rs * (gd[i].x - c1 - xh[i].x * c2); o[i].y += rs * (gd[i].y - c1 - xh[i].y * c2);
      o[i].z += rs * (gd[i].z - c1 - xh[i].z * c2); o[i].w += rs * (gd[i].w - c1 - xh[i].w * c2);
      reinterpret_cast<float4*>(dres + (int64_t)row * D)[l + 16 * i] = o[i];
      if (dlp) store4<T>(dlp + (int64_t)row * D + 4 * (l + 16 * i), o[i].x, o[i].y, o[i].z, o[i].w);
      if constexpr (PARAMS) { ac[i].x += o[i].x; ac[i].y += o[i].y; ac[i].z += o[i].z; ac[i].w += o[i].w; }
    }
  }
  if constexpr (!PARAMS) return;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int c = 4 * (l + 16 * i);
    *reinterpret_cast<float4*>(&red[hw][c]) = ag[i];
    *reinterpret_cast<float4*>(&red[hw][D + c]) = ab[i];
    *reinterpret_cast<float4*>(&red[hw][2 * D + c]) = ac[i];
  }
  __syncthreads();
  float* part = DET ? p.det_part + ((int64_t)g * gridDim.x + blockIdx.x) * 3 * D : nullptr;
  for (int c = threadIdx.x; c < 3 * D; c += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 16; ++w) s += red[w][c];
    if (DET) part[c] = s;
    else if (c < D) atomicAdd(p.dgamma[g] + c, s);
    else if (c < 2 * D) atomicAdd(p.dbeta[g] + (c - D), s);
    else if (p.dcolsum[g]) atomicAdd(p.dcolsum[g] + (c - 2 * D), s);
  }
  if constexpr (DET) {
    __syncthreads();                 // red is reused by the reduction
    float* dgm = p.dgamma[g]; float* dbt = p.dbeta[g]; float* dcs = p.dcolsum[g];
    det_reduce_rows(p.det_part + (int64_t)g * gridDim.x * 3 * D, 3 * D, gridDim.x, p.det_counters + g, &red[0][0], 16 * 3 * D,
                    [&](int c, float s) {
                      if (c < D) dgm[c] += s;
                      else if (c < 2 * D) dbt[c - D] += s;
                      else if (dcs) dcs[c - 2 * D] += s;
                    });
  }
}

// db[n] += sum_m dy[m,n]   (N a multiple of 8; 8 contiguous columns per thread, 128-bit loads)
struct ColsumP {
  const void* dy[MAXG]; float* db[MAXG];
  int M, N, rows_per_block;
  float* det_part;             // DET with more than one CTA per group: [group][CTA][N] partial rows
  unsigned* det_counters;
};

template <typename T, bool DET>
__global__ void __launch_bounds__(256) colsum_kernel(const __grid_constant__ ColsumP p) {
  __shared__ float red[2048];
  const int g = blockIdx.y;
  const int cols_t = p.N / 8;
  int rows_t = 256 / cols_t;
  if (rows_t * p.N > 2048) rows_t = 2048 / p.N;
  const int ct = threadIdx.x % cols_t, rt = threadIdx.x / cols_t;
  const T* __restrict__ dy = static_cast<const T*>(p.dy[g]);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  const int r0 = blockIdx.x * p.rows_per_block;
  const int r1 = min(p.M, r0 + p.rows_per_block);
  if (rt < rows_t) {
    for (int r = r0 + rt; r < r1; r += rows_t) {
      const T* src = dy + (int64_t)r * p.N + ct * 8;
      const float4 a = load4<T>(src), b = load4<T>(src + 4);
      acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
      acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[rt * p.N + ct * 8 + i] = acc[i];
  }
  __syncthreads();
  float* part = (DET && gridDim.x > 1) ? p.det_part + ((int64_t)g * gridDim.x + blockIdx.x) * p.N : nullptr;
  for (int n = threadIdx.x; n < p.N; n += blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < rows_t; ++w) s += red[w * p.N + n];
    if (!DET) atomicAdd(p.db[g] + n, s);
    else if (part) part[n] = s;
    else p.db[g][n] += s;            // one CTA per group: the only writer
  }
  if constexpr (DET) {
    if (gridDim.x == 1) return;
    __syncthreads();
    float* db = p.db[g];
    det_reduce_rows(p.det_part + (int64_t)g * gridDim.x * p.N, p.N, gridDim.x, p.det_counters + g, red, 2048,
                    [db](int c, float s) { db[c] += s; });
  }
}

__global__ void pool_fwd_kernel(G4<const float*> hidden, G4<float*> feat, G4<int64_t> stride) {
  const int g = blockIdx.y, b = blockIdx.x, n = threadIdx.x;
  const float* h = hidden.p[g] + (int64_t)b * NT * D + n;
  float s = 0.f;
  for (int t = 0; t < NT; ++t) s += h[(int64_t)t * D];
  feat.p[g][(int64_t)b * stride.p[g] + n] = s * (1.0f / NT);
}

// dx[b,t,:] = dfeat[b,:] / 197 (+ dhidden[b,t,:]); also the activation-type copy.  float4 per thread.
template <typename T>
__global__ void __launch_bounds__(256) pool_bwd_kernel(G4<const float*> dfeat, G4<int64_t> stride, G4<const float*> dhidden,
                                                       G4<float*> dx, G4<T*> dx_lp) {
  const int g = blockIdx.z, b = blockIdx.y;
  const float* __restrict__ df = dfeat.p[g];
  const float* __restrict__ dh = dhidden.p[g];
  float* __restrict__ o = dx.p[g];
  T* __restrict__ ol = dx_lp.p[g];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < NT * (D / 4); i += gridDim.x * blockDim.x) {
    const int c = (i % (D / 4)) * 4;
    const int64_t idx = (int64_t)b * NT * D + (int64_t)i * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (df) {
      const float4 f = *reinterpret_cast<const float4*>(df + (int64_t)b * stride.p[g] + c);
      v = make_float4(f.x * (1.0f / NT), f.y * (1.0f / NT), f.z * (1.0f / NT), f.w * (1.0f / NT));
    }
    if (dh) {
      const float4 a = *reinterpret_cast<const float4*>(dh + idx);
      v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    }
    *reinterpret_cast<float4*>(o + idx) = v;
    if (ol) store4<T>(ol + idx, v.x, v.y, v.z, v.w);
  }
}

// d pos / d cls / d patch-bias from the gradient of the embedding output
// DET: the patch-bias sum over the 196 patch tokens goes through det_part [group][196][192] in token order
// MASK (groups with a mask): d patch-bias sums the unmasked (image, patch) rows only; the masked ones are summed into
// d mask_token (dtok; NULL: not wanted).  DET then carries both sums per token, det_part [group][196][384], through the
// same fixed-order reduction with twice the shared rows, so that d patch-bias keeps the unmasked kernel's order and bits.
template <bool DET, bool MASK>
__global__ void embed_bwd_kernel(G4<const float*> dx, G4<float*> grads, int B, float* det_part, unsigned* det_counters,
                                 MaskArgs mk, G4<float*> dtok) {
  const int g = blockIdx.y, t = blockIdx.x, n = threadIdx.x;
  const float* d = dx.p[g] + (int64_t)t * D + n;
  float s = 0.f, sm = 0.f;
  const uint8_t* m = MASK && t > 0 ? mk.mask[g] : nullptr;
  if (MASK && m) {
    for (int b = 0; b < B; ++b) {
      const float v = d[(int64_t)b * NT * D];
      if (m[(int64_t)b * NP + t - 1]) sm += v; else s += v;
    }
  } else {
    for (int b = 0; b < B; ++b) s += d[(int64_t)b * NT * D];
  }
  float* gr = grads.p[g];
  float* dt = MASK ? dtok.p[g] : nullptr;
  gr[OFF_POS + (int64_t)t * D + n] += MASK ? s + sm : s;
  if (t == 0) gr[OFF_CLS + n] += s;
  else if (!DET) {
    atomicAdd(gr + OFF_BPE + n, s);
    if (MASK && m && dt) atomicAdd(dt + n, sm);
  }
  if constexpr (DET) {
    if (t == 0) return;
    constexpr int W = MASK ? 2 * D : D;          // floats per partial row
    __shared__ __align__(16) float red[8 * W];
    float* part = det_part + (int64_t)g * NP * W;
    part[(int64_t)(t - 1) * W + n] = s;
    if constexpr (MASK) part[(int64_t)(t - 1) * W + D + n] = sm;
    det_reduce_rows(part, W, NP, det_counters + g, red, 8 * W, [gr, dt](int c, float v) {
      if (c < D) gr[OFF_BPE + c] += v;
      else if (dt) dt[c - D] += v;
    });
  }
}

// ------------------------------------------------------------------------------------------
// SIMT attention (fp32 check mode / debugging reference).  One CTA per (head, image, group).
// ------------------------------------------------------------------------------------------
constexpr int ASTR = DH + 1;  // odd row stride: conflict-free when lanes walk rows

template <typename T>
__global__ void __launch_bounds__(256) attn_fwd_simt_kernel(G4<const T*> qkv, G4<T*> ctx, G4<float*> lse) {
  extern __shared__ float sm[];
  float* Ks = sm;                    // [197][65]
  float* Vs = Ks + NT * ASTR;        // [197][65]
  float* Ps = Vs + NT * ASTR;        // [8][200]
  float* Qs = Ps + 8 * 200;          // [8][64]
  const int h = blockIdx.x, b = blockIdx.y, g = blockIdx.z;
  const T* base = qkv.p[g] + (int64_t)b * NT * 3 * D;
  for (int i = threadIdx.x; i < NT * DH; i += blockDim.x) {
    const int t = i / DH, d = i % DH;
    Ks[t * ASTR + d] = to_f<T>(base[(int64_t)t * 3 * D + D + h * DH + d]);
    Vs[t * ASTR + d] = to_f<T>(base[(int64_t)t * 3 * D + 2 * D + h * DH + d]);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* P = Ps + warp * 200;
  float* Q = Qs + warp * DH;
  const float scale = 0.125f;  // 64^-0.5
  for (int i = warp; i < NT; i += 8) {
    Q[lane] = to_f<T>(base[(int64_t)i * 3 * D + h * DH + lane]);
    Q[lane + 32] = to_f<T>(base[(int64_t)i * 3 * D + h * DH + lane + 32]);
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < NT; j += 32) {
      float s = 0.f;
#pragma unroll 16
      for (int d = 0; d < DH; ++d) s = fmaf(Q[d], Ks[j * ASTR + d], s);
      s *= scale;
      P[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < NT; j += 32) { const float e = expf(P[j] - mx); P[j] = e; sum += e; }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = 1.0f / sum;
    float o0 = 0.f, o1 = 0.f;
    for (int j = 0; j < NT; ++j) {
      const float p = P[j];
      o0 = fmaf(p, Vs[j * ASTR + lane], o0);
      o1 = fmaf(p, Vs[j * ASTR + lane + 32], o1);
    }
    T* out = ctx.p[g] + ((int64_t)b * NT + i) * D + h * DH;
    out[lane] = from_f<T>(o0 * inv);
    out[lane + 32] = from_f<T>(o1 * inv);
    if (lane == 0 && lse.p[g]) lse.p[g][((int64_t)b * NH + h) * NT + i] = mx + logf(sum);
    __syncwarp();
  }
}

template <typename T>
__global__ void __launch_bounds__(256) attn_bwd_simt_kernel(G4<const T*> qkv, G4<const T*> ctx,
                                                            G4<const float*> lse, G4<const T*> dctx,
                                                            G4<T*> dqkv) {
  extern __shared__ float sm[];
  float* Qs = sm;                     // [197][65]
  float* Ks = Qs + NT * ASTR;
  float* Vs = Ks + NT * ASTR;
  float* dOs = Vs + NT * ASTR;
  float* Ls = dOs + NT * ASTR;        // [197] lse
  float* Ds = Ls + NT;                // [197] rowsum(dO * O)
  float* Ps = Ds + NT;                // [8][200]
  float* dSs = Ps + 8 * 200;          // [8][200]
  const int h = blockIdx.x, b = blockIdx.y, g = blockIdx.z;
  const T* base = qkv.p[g] + (int64_t)b * NT * 3 * D;
  const T* ob = ctx.p[g] + (int64_t)b * NT * D + h * DH;
  const T* dob = dctx.p[g] + (int64_t)b * NT * D + h * DH;
  for (int i = threadIdx.x; i < NT * DH; i += blockDim.x) {
    const int t = i / DH, d = i % DH;
    Qs[t * ASTR + d] = to_f<T>(base[(int64_t)t * 3 * D + h * DH + d]);
    Ks[t * ASTR + d] = to_f<T>(base[(int64_t)t * 3 * D + D + h * DH + d]);
    Vs[t * ASTR + d] = to_f<T>(base[(int64_t)t * 3 * D + 2 * D + h * DH + d]);
    dOs[t * ASTR + d] = to_f<T>(dob[(int64_t)t * D + d]);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = warp; t < NT; t += 8) {
    float s = 0.f;
    for (int d = lane; d < DH; d += 32) s += to_f<T>(ob[(int64_t)t * D + d]) * to_f<T>(dob[(int64_t)t * D + d]);
    s = warp_sum(s);
    if (lane == 0) { Ds[t] = s; Ls[t] = lse.p[g][((int64_t)b * NH + h) * NT + t]; }
  }
  __syncthreads();
  float* P = Ps + warp * 200;
  float* dS = dSs + warp * 200;
  const float scale = 0.125f;
  T* dq_base = dqkv.p[g] + (int64_t)b * NT * 3 * D;
  // phase A: dQ_i = scale * sum_j dS_ij K_j
  for (int i = warp; i < NT; i += 8) {
    const float li = Ls[i], di = Ds[i];
    for (int j = lane; j < NT; j += 32) {
      float s = 0.f, dp = 0.f;
#pragma unroll 16
      for (int d = 0; d < DH; ++d) {
        s = fmaf(Qs[i * ASTR + d], Ks[j * ASTR + d], s);
        dp = fmaf(dOs[i * ASTR + d], Vs[j * ASTR + d], dp);
      }
      const float p = expf(s * scale - li);
      dS[j] = p * (dp - di);
    }
    __syncwarp();
    float a0 = 0.f, a1 = 0.f;
    for (int j = 0; j < NT; ++j) {
      const float w = dS[j];
      a0 = fmaf(w, Ks[j * ASTR + lane], a0);
      a1 = fmaf(w, Ks[j * ASTR + lane + 32], a1);
    }
    T* o = dq_base + (int64_t)i * 3 * D + h * DH;
    o[lane] = from_f<T>(a0 * scale);
    o[lane + 32] = from_f<T>(a1 * scale);
    __syncwarp();
  }
  // phase B: dV_j = sum_i P_ij dO_i ; dK_j = scale * sum_i dS_ij Q_i
  for (int j = warp; j < NT; j += 8) {
    for (int i = lane; i < NT; i += 32) {
      float s = 0.f, dp = 0.f;
#pragma unroll 16
      for (int d = 0; d < DH; ++d) {
        s = fmaf(Qs[i * ASTR + d], Ks[j * ASTR + d], s);
        dp = fmaf(dOs[i * ASTR + d], Vs[j * ASTR + d], dp);
      }
      const float p = expf(s * scale - Ls[i]);
      P[i] = p;
      dS[i] = p * (dp - Ds[i]);
    }
    __syncwarp();
    float v0 = 0.f, v1 = 0.f, k0 = 0.f, k1 = 0.f;
    for (int i = 0; i < NT; ++i) {
      const float p = P[i], w = dS[i];
      v0 = fmaf(p, dOs[i * ASTR + lane], v0);
      v1 = fmaf(p, dOs[i * ASTR + lane + 32], v1);
      k0 = fmaf(w, Qs[i * ASTR + lane], k0);
      k1 = fmaf(w, Qs[i * ASTR + lane + 32], k1);
    }
    T* ok = dq_base + (int64_t)j * 3 * D + D + h * DH;
    T* ov = dq_base + (int64_t)j * 3 * D + 2 * D + h * DH;
    ok[lane] = from_f<T>(k0 * scale); ok[lane + 32] = from_f<T>(k1 * scale);
    ov[lane] = from_f<T>(v0); ov[lane + 32] = from_f<T>(v1);
    __syncwarp();
  }
}

// attention probabilities P = exp(s / 8 - lse) as fp32 [B,3,197,197] (the SIMT twin of attn_probs_tc_kernel): s is
// accumulated in the order attn_fwd_simt_kernel uses, so the rows of the check mode sum to 1 up to fp32 rounding.
// DP = true: dP = dO V^T, the gradient w.r.t. the probabilities, with a = d ctx [B,197,192] (else a = qkv).
template <typename T, bool DP>
__global__ void __launch_bounds__(256) attn_probs_simt_kernel(G4<const T*> qkv, G4<const T*> a, G4<const float*> lse,
                                                              G4<float*> probs) {
  extern __shared__ float sm[];
  float* Ks = sm;                    // [197][65]: K, or V (DP)
  float* Qs = Ks + NT * ASTR;        // [8][64]: rows of Q, or of d ctx (DP)
  const int h = blockIdx.x, b = blockIdx.y, g = blockIdx.z;
  constexpr int A_LD = DP ? D : 3 * D;
  const T* base = qkv.p[g] + (int64_t)b * NT * 3 * D;
  const T* abase = a.p[g] + (int64_t)b * NT * A_LD;
  for (int i = threadIdx.x; i < NT * DH; i += blockDim.x) {
    const int t = i / DH, d = i % DH;
    Ks[t * ASTR + d] = to_f<T>(base[(int64_t)t * 3 * D + (DP ? 2 * D : D) + h * DH + d]);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Q = Qs + warp * DH;
  const float scale = 0.125f;
  for (int i = warp; i < NT; i += 8) {
    Q[lane] = to_f<T>(abase[(int64_t)i * A_LD + h * DH + lane]);
    Q[lane + 32] = to_f<T>(abase[(int64_t)i * A_LD + h * DH + lane + 32]);
    __syncwarp();
    const float li = DP ? 0.f : lse.p[g][((int64_t)b * NH + h) * NT + i];
    float* out = probs.p[g] + (((int64_t)b * NH + h) * NT + i) * NT;
    for (int j = lane; j < NT; j += 32) {
      float s = 0.f;
#pragma unroll 16
      for (int d = 0; d < DH; ++d) s = fmaf(Q[d], Ks[j * ASTR + d], s);
      if (DP) {
        out[j] = s;
      } else {
        s *= scale;
        out[j] = expf(s - li);
      }
    }
    __syncwarp();
  }
}

// dx += dh, dx_lp = dx in the activation type: the gradient w.r.t. an intermediate hidden state joins the residual-stream
// gradient; dcol (optional) += column sums of dh, the part of the producing block's fc2 bias gradient that the fused
// column sums of LN1-backward (taken before dh is added) do not see.  Launched without the dependent-launch attribute,
// so it starts after its predecessor has completed.  Threads: 48 float4 columns x 5 row lanes.
constexpr int RGA_RL = 256 / (D / 4);
template <typename T, bool DET>
__global__ void __launch_bounds__(256) residual_grad_add_kernel(G4<const float*> dh, G4<float*> dx, G4<T*> dx_lp, G4<float*> dcol,
                                                                int rows, float* det_part, unsigned* det_counters) {
  __shared__ float4 part[RGA_RL][D / 4];
  const int g = blockIdx.y;
  const int c4 = threadIdx.x % (D / 4), rl = threadIdx.x / (D / 4);
  const float4* __restrict__ a = reinterpret_cast<const float4*>(dh.p[g]);
  float4* __restrict__ o = reinterpret_cast<float4*>(dx.p[g]);
  T* __restrict__ ol = dx_lp.p[g];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (rl < RGA_RL)
    for (int r = blockIdx.x * RGA_RL + rl; r < rows; r += gridDim.x * RGA_RL) {
      const int64_t i = (int64_t)r * (D / 4) + c4;
      const float4 x = a[i];
      float4 v = o[i];
      v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
      o[i] = v;
      if (ol) store4<T>(ol + 4 * i, v.x, v.y, v.z, v.w);
      acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
    }
  if (dcol.p[g]) {
    if (rl < RGA_RL) part[rl][c4] = acc;
    __syncthreads();
    if (threadIdx.x < D / 4) {
      float4 s = part[0][c4];
      for (int k = 1; k < RGA_RL; ++k) { s.x += part[k][c4].x; s.y += part[k][c4].y; s.z += part[k][c4].z; s.w += part[k][c4].w; }
      if (DET) {
        reinterpret_cast<float4*>(det_part + ((int64_t)g * gridDim.x + blockIdx.x) * D)[c4] = s;
      } else {
        float* d = dcol.p[g] + 4 * c4;
        atomicAdd(d, s.x); atomicAdd(d + 1, s.y); atomicAdd(d + 2, s.z); atomicAdd(d + 3, s.w);
      }
    }
    if constexpr (DET) {
      __syncthreads();
      float* dc = dcol.p[g];
      det_reduce_rows(det_part + (int64_t)g * gridDim.x * D, D, gridDim.x, det_counters + g, &part[0][0].x, RGA_RL * D,
                      [dc](int c, float v) { dc[c] += v; });
    }
  }
}

// ------------------------------------------------------------------------------------------
// loss = -mean_i cos(p_i, z_i) / accum   (torch CosineSimilarity: each norm clamped at 1e-8)
// dp   = grad_scale * d loss / d p.  Single CTA (B rows x 128), deterministic reduction.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cosine_loss_kernel(const float* __restrict__ p,
                                                          const float* __restrict__ z, float* loss,
                                                          float* dp, int B, float inv_count,
                                                          float grad_scale, const float* __restrict__ grad_scale_dev) {
  __shared__ float part[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float eps = 1e-8f;
  float acc = 0.f;
  for (int i = warp; i < B; i += 8) {
    const float4 pv = reinterpret_cast<const float4*>(p + (int64_t)i * V2S_PROJ_OUT)[lane];
    const float4 zv = reinterpret_cast<const float4*>(z + (int64_t)i * V2S_PROJ_OUT)[lane];
    float dot = pv.x * zv.x + pv.y * zv.y + pv.z * zv.z + pv.w * zv.w;
    float pp = pv.x * pv.x + pv.y * pv.y + pv.z * pv.z + pv.w * pv.w;
    float zz = zv.x * zv.x + zv.y * zv.y + zv.z * zv.z + zv.w * zv.w;
    dot = warp_sum(dot); pp = warp_sum(pp); zz = warp_sum(zz);
    const float pn = sqrtf(pp), zn = sqrtf(zz);
    const float pc = fmaxf(pn, eps), zc = fmaxf(zn, eps);
    const float cosv = dot / (pc * zc);
    acc += cosv;
    if (dp) {
      // d cos / d p = z/(pc*zc) - [pn > eps] * cos * p / pn^2
      const float a = 1.0f / (pc * zc);
      const float c = (pn > eps) ? cosv / pp : 0.f;
      const float s = -inv_count * grad_scale * (grad_scale_dev ? __ldg(grad_scale_dev) : 1.0f);
      float4 o;
      o.x = s * (zv.x * a - c * pv.x); o.y = s * (zv.y * a - c * pv.y);
      o.z = s * (zv.z * a - c * pv.z); o.w = s * (zv.w * a - c * pv.w);
      reinterpret_cast<float4*>(dp + (int64_t)i * V2S_PROJ_OUT)[lane] = o;
    }
  }
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += part[w];
    *loss = -t * inv_count;
  }
}

// ------------------------------------------------------------------------------------------
// InfoNCE with global negatives (north_star (3); no reference counterpart, SURVEY D2/D3 — an opt-in loss, never the
// default).  One CTA per local row i: the row of the cosine-similarity matrix p_i . z_j / (|p_i| |z_j| tau) against ALL
// gathered target projections, its log-sum-exp, the cross-entropy against the positive (column label_offset + i) and
// the gradient w.r.t. p_i (z is detached, ref:158) — similarity "GEMM", temperature scale, row logsumexp, CE and its
// backward in one launch; the N x 128 key matrix (512 KB at 8 x 128 keys) streams from L2.
//   loss = mean_i( lse_i - logit_i,label ) / accum   (row_loss[i] holds the per-row term; summed by a second tiny launch
//   in a fixed order, so the result is bit-reproducible)
// ------------------------------------------------------------------------------------------
constexpr int NCE_THREADS = 256;
__global__ void __launch_bounds__(NCE_THREADS) infonce_row_kernel(const float* __restrict__ p, const float* __restrict__ z,
                                                                   float* __restrict__ row_loss, float* __restrict__ dp,
                                                                   int n_keys, long long label_offset, float inv_tau,
                                                                   float grad_mul, const float* __restrict__ grad_scale_dev) {
  extern __shared__ float nce_sm[];
  float* logit = nce_sm;                 // [n_keys]
  float* invn = nce_sm + n_keys;         // [n_keys] 1 / max(|z_j|, eps)
  __shared__ float red[NCE_THREADS / 32];
  __shared__ float ph[V2S_PROJ_OUT];     // normalised p_i
  __shared__ float gh[2][V2S_PROJ_OUT];
  __shared__ float bc[2];
  const int i = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float eps = 1e-8f;
  // ---- p_i / max(|p_i|, eps) ----
  float pn2 = 0.f;
  if (warp == 0) {
    const float4 pv = reinterpret_cast<const float4*>(p + (int64_t)i * V2S_PROJ_OUT)[lane];
    pn2 = warp_sum(pv.x * pv.x + pv.y * pv.y + pv.z * pv.z + pv.w * pv.w);
    const float inv = 1.0f / fmaxf(sqrtf(pn2), eps);
    reinterpret_cast<float4*>(ph)[lane] = make_float4(pv.x * inv, pv.y * inv, pv.z * inv, pv.w * inv);
    if (lane == 0) bc[0] = pn2;
  }
  __syncthreads();
  pn2 = bc[0];
  const float4 pq = reinterpret_cast<const float4*>(ph)[lane];
  // ---- logits: one warp per key row (coalesced 512-byte reads) ----
  float mx = -INFINITY;
  for (int j = warp; j < n_keys; j += NCE_THREADS / 32) {
    const float4 zv = reinterpret_cast<const float4*>(z + (int64_t)j * V2S_PROJ_OUT)[lane];
    const float dot = warp_sum(pq.x * zv.x + pq.y * zv.y + pq.z * zv.z + pq.w * zv.w);
    const float zz = warp_sum(zv.x * zv.x + zv.y * zv.y + zv.z * zv.z + zv.w * zv.w);
    const float iz = 1.0f / fmaxf(sqrtf(zz), eps);
    const float lg = dot * iz * inv_tau;
    if (lane == 0) { logit[j] = lg; invn[j] = iz; }
    mx = fmaxf(mx, lg);
  }
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < NCE_THREADS / 32; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  float se = 0.f;
  for (int j = threadIdx.x; j < n_keys; j += NCE_THREADS) se += __expf(logit[j] - mx);
  se = warp_sum(se);
  if (lane == 0) red[warp] = se;
  __syncthreads();
  se = 0.f;
#pragma unroll
  for (int w = 0; w < NCE_THREADS / 32; ++w) se += red[w];     // fixed order: every thread gets the same sum
  const float lse = mx + __logf(se);
  const int label = (int)(label_offset + i);
  if (threadIdx.x == 0) row_loss[i] = lse - logit[label];
  if (dp == nullptr) return;
  // ---- d loss_i / d p_hat = (1/tau) sum_j (softmax_ij - [j == label]) z_hat_j; thread = (dimension, key parity) ----
  const int d = threadIdx.x & (V2S_PROJ_OUT - 1), par = threadIdx.x >> 7;
  float g = 0.f;
  for (int j = par; j < n_keys; j += 2) {
    const float s = __expf(logit[j] - lse) - (j == label ? 1.0f : 0.0f);
    g = fmaf(s * invn[j], __ldg(z + (int64_t)j * V2S_PROJ_OUT + d), g);
  }
  gh[par][d] = g;
  __syncthreads();
  if (threadIdx.x < V2S_PROJ_OUT) {
    g = (gh[0][d] + gh[1][d]) * inv_tau;
    // through p_hat = p / max(|p|, eps):  (g - [|p| > eps] p_hat (p_hat . g)) / max(|p|, eps)
    const float pd = ph[d];
    float dot = warp_sum(pd * g);
    if (lane == 0) red[warp] = dot;
  }
  __syncthreads();
  if (threadIdx.x < V2S_PROJ_OUT) {
    const float dot = red[0] + red[1] + red[2] + red[3];
    const float pn = sqrtf(pn2);
    const float proj = pn > eps ? ph[d] * dot : 0.f;
    const float sc = grad_mul * (grad_scale_dev ? __ldg(grad_scale_dev) : 1.0f) / fmaxf(pn, eps);
    dp[(int64_t)i * V2S_PROJ_OUT + d] = (g - proj) * sc;
  }
}

__global__ void __launch_bounds__(256) infonce_mean_kernel(const float* __restrict__ row_loss, float* loss, int B, float inv_count) {
  __shared__ float part[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float acc = 0.f;
  for (int i = threadIdx.x; i < B; i += 256) acc += row_loss[i];
  acc = warp_sum(acc);
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += part[w];
    *loss = t * inv_count;
  }
}

// ------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam semantics) over up to 4 flat ranges; optional bf16 shadow refresh
// ------------------------------------------------------------------------------------------
struct AdamRanges {
  v2s_range_t r[4];
  int n;
};

struct AdamHyper { float step_size, bc2_sqrt, skip, gmul; };

// device-resident optimizer-step state (v2s_adam_step_amp): state8[0] = optimizer steps taken, [1..4] = AdamHyper of the
// step being applied.  One thread; double-precision bias corrections like the host path.
__global__ void adam_prologue_kernel(float* state8, double lr, double b1, double b2, double grad_multiplier,
                                     const float* grad_scale_dev, const float* found_inf_dev) {
  const bool skip = found_inf_dev != nullptr && *found_inf_dev != 0.f;
  float step = state8[0];
  if (!skip) step += 1.0f;
  state8[0] = step;
  const double bc1 = 1.0 - pow(b1, (double)step), bc2 = 1.0 - pow(b2, (double)step);
  state8[1] = skip ? 0.f : (float)(lr / bc1);
  state8[2] = skip ? 1.f : (float)sqrt(bc2);
  state8[3] = skip ? 1.f : 0.f;
  state8[4] = (float)(grad_multiplier / (grad_scale_dev ? (double)*grad_scale_dev : 1.0));
}

template <bool DEV>
__global__ void __launch_bounds__(256) adam_kernel(AdamRanges rs, AdamHyper hv, const float* __restrict__ state8, float om_b1,
                                                   float b2, float om_b2, float eps, float wd, int lp_f16) {
  AdamHyper hy = hv;
  if (DEV) { hy.step_size = state8[1]; hy.bc2_sqrt = state8[2]; hy.skip = state8[3]; hy.gmul = state8[4]; }
  if (hy.skip != 0.f) return;                 // GradScaler found an inf / nan: the step changes nothing (ref:216-217)
  const float step_size = hy.step_size, bc2_sqrt = hy.bc2_sqrt, grad_scale = hy.gmul;
  const v2s_range_t r = rs.r[blockIdx.y];
  const int64_t n4 = r.numel / 4;
  float4* p4 = reinterpret_cast<float4*>(r.params);
  const float4* g4 = reinterpret_cast<const float4*>(r.grads);
  float4* m4 = reinterpret_cast<float4*>(r.exp_avg);
  float4* v4 = reinterpret_cast<float4*>(r.exp_avg_sq);
  uint16_t* lp = static_cast<uint16_t*>(r.params_lp);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 p = p4[i], g = g4[i], m = m4[i], v = v4[i];
    float* pp = &p.x; float* gg = &g.x; float* mm = &m.x; float* vv = &v.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float gr = gg[k] * grad_scale;
      if (wd != 0.f) gr = fmaf(wd, pp[k], gr);
      mm[k] = mm[k] + (gr - mm[k]) * om_b1;              // exp_avg.lerp_(grad, 1-beta1), as torch
      vv[k] = b2 * vv[k] + om_b2 * gr * gr;             // mul_(beta2).addcmul_(g, g, 1-beta2)
      const float denom = sqrtf(vv[k]) / bc2_sqrt + eps;
      pp[k] = pp[k] - step_size * (mm[k] / denom);
    }
    p4[i] = p; m4[i] = m; v4[i] = v;
    if (lp) {
      uint2 u;
      u.x = pack_lp(p.x, p.y, lp_f16); u.y = pack_lp(p.z, p.w, lp_f16);
      reinterpret_cast<uint2*>(lp)[i] = u;
    }
  }
  // scalar tail (numel not a multiple of 4)
  if (blockIdx.x == 0 && threadIdx.x < (r.numel & 3)) {
    const int64_t i = n4 * 4 + threadIdx.x;
    float gr = r.grads[i] * grad_scale;
    if (wd != 0.f) gr = fmaf(wd, r.params[i], gr);
    float m = r.exp_avg[i], v = r.exp_avg_sq[i];
    m = m + (gr - m) * om_b1;
    v = b2 * v + om_b2 * gr * gr;
    const float denom = sqrtf(v) / bc2_sqrt + eps;
    const float pn = r.params[i] - step_size * (m / denom);
    r.params[i] = pn; r.exp_avg[i] = m; r.exp_avg_sq[i] = v;
    if (lp) lp[i] = (uint16_t)(pack_lp(pn, 0.f, lp_f16) & 0xffffu);
  }
}

struct EmaPairs {
  float* t[4];
  const float* o[4];
  uint16_t* lp[4];
};

// target = m*target + (1-m)*online, rounded exactly as torch's two multiplies + add (ref:164)
__global__ void __launch_bounds__(256) ema_kernel(EmaPairs pr, int64_t numel, float m, float om, int lp_f16) {
  float4* t4 = reinterpret_cast<float4*>(pr.t[blockIdx.y]);
  const float4* o4 = reinterpret_cast<const float4*>(pr.o[blockIdx.y]);
  uint16_t* lp = pr.lp[blockIdx.y];
  const int64_t n4 = numel / 4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto upd = [&](float4 t, const float4 o, int64_t i) {
    t.x = __fadd_rn(__fmul_rn(m, t.x), __fmul_rn(om, o.x));
    t.y = __fadd_rn(__fmul_rn(m, t.y), __fmul_rn(om, o.y));
    t.z = __fadd_rn(__fmul_rn(m, t.z), __fmul_rn(om, o.z));
    t.w = __fadd_rn(__fmul_rn(m, t.w), __fmul_rn(om, o.w));
    t4[i] = t;
    if (lp) {
      uint2 u;
      u.x = pack_lp(t.x, t.y, lp_f16); u.y = pack_lp(t.z, t.w, lp_f16);
      reinterpret_cast<uint2*>(lp)[i] = u;
    }
  };
  // four independent 16-byte loads of each stream in flight per thread before the first store (a 12 B/element stream
  // needs the memory-level parallelism: 4.3 -> 5+ TB/s)
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n4; i += 4 * stride) {
    const float4 ta = t4[i], tb = t4[i + stride], tc = t4[i + 2 * stride], td = t4[i + 3 * stride];
    const float4 oa = o4[i], ob = o4[i + stride], oc = o4[i + 2 * stride], od = o4[i + 3 * stride];
    upd(ta, oa, i); upd(tb, ob, i + stride); upd(tc, oc, i + 2 * stride); upd(td, od, i + 3 * stride);
  }
  for (; i < n4; i += stride) upd(t4[i], o4[i], i);
}

__global__ void cast_lp_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, int64_t n, int lp_f16) {
  const int64_t n4 = n / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    uint2 u;
    u.x = pack_lp(v.x, v.y, lp_f16); u.y = pack_lp(v.z, v.w, lp_f16);
    reinterpret_cast<uint2*>(dst)[i] = u;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3))
    dst[n4 * 4 + threadIdx.x] = (uint16_t)(pack_lp(src[n4 * 4 + threadIdx.x], 0.f, lp_f16) & 0xffffu);
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void dropout_mask_kernel(float* mask, int64_t n, float p, float keep_scale, uint64_t seed,
                                    uint64_t offset) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t r = splitmix64(splitmix64(seed) ^ (offset + (uint64_t)i));
    const float u = (float)(r >> 40) * (1.0f / 16777216.0f);
    mask[i] = (u >= p) ? keep_scale : 0.f;
  }
}

// uint8 [B,1,28,28] → bilinear (align_corners=False) 224x224 → 3ch → ImageNet normalise
__global__ void preprocess_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, int B) {
  const int64_t total = (int64_t)B * V2S_IMG * V2S_IMG;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int xo = idx % V2S_IMG, yo = (idx / V2S_IMG) % V2S_IMG, b = idx / (V2S_IMG * V2S_IMG);
    const float sc = 28.0f / 224.0f;
    float sx = fmaxf((xo + 0.5f) * sc - 0.5f, 0.f), sy = fmaxf((yo + 0.5f) * sc - 0.5f, 0.f);
    const int x0 = (int)sx, y0 = (int)sy;
    const int x1 = min(x0 + 1, 27), y1 = min(y0 + 1, 27);
    const float lx = sx - x0, ly = sy - y0;
    const uint8_t* s = src + (int64_t)b * 784;
    const float k = 1.0f / 255.0f;
    const float v00 = s[y0 * 28 + x0] * k, v01 = s[y0 * 28 + x1] * k, v10 = s[y1 * 28 + x0] * k, v11 = s[y1 * 28 + x1] * k;
    const float v = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
    const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
#pragma unroll
    for (int c = 0; c < 3; ++c)
      dst[(((int64_t)b * 3 + c) * V2S_IMG + yo) * V2S_IMG + xo] = (v - mean[c]) / stdv[c];
  }
}

// the same values written as the patch matrix [B*196, 768] (k = c*256 + ky*16 + kx) in a 16-bit format: one thread per
// four consecutive kx of one (image, patch, channel, ky)
template <typename T>
__global__ void preprocess_u8_patches_kernel(const uint8_t* __restrict__ src, T* __restrict__ out, int B) {
  const int64_t total = (int64_t)B * NP * (KPE / 4);
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int kx4 = idx % 4, ky = (idx / 4) % 16, c = (idx / 64) % 3, pp = (idx / 192) % NP;
    const int b = idx / (192 * NP);
    const int yo = (pp / 14) * 16 + ky;
    const float sc = 28.0f / 224.0f;
    const float sy = fmaxf((yo + 0.5f) * sc - 0.5f, 0.f);
    const int y0 = (int)sy, y1 = min(y0 + 1, 27);
    const float ly = sy - y0;
    const uint8_t* s = src + (int64_t)b * 784;
    const float k = 1.0f / 255.0f;
    const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
    float r[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int xo = (pp % 14) * 16 + kx4 * 4 + j;
      const float sx = fmaxf((xo + 0.5f) * sc - 0.5f, 0.f);
      const int x0 = (int)sx, x1 = min(x0 + 1, 27);
      const float lx = sx - x0;
      const float v00 = s[y0 * 28 + x0] * k, v01 = s[y0 * 28 + x1] * k, v10 = s[y1 * 28 + x0] * k, v11 = s[y1 * 28 + x1] * k;
      const float v = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
      r[j] = (v - mean[c]) / stdv[c];
    }
    T* dst = out + ((int64_t)b * NP + pp) * KPE + c * 256 + ky * 16 + kx4 * 4;
    dst[0] = from_f<T>(r[0]); dst[1] = from_f<T>(r[1]); dst[2] = from_f<T>(r[2]); dst[3] = from_f<T>(r[3]);
  }
}

inline int grid_for(int64_t n, int threads, int max_blocks = 148 * 8) {
  int64_t b = (n + threads - 1) / threads;
  if (b > max_blocks) b = max_blocks;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
int launch_im2col(const float* const* x, void* const* out, int groups, int B, int at, cudaStream_t s) {
  dim3 grid(grid_for((int64_t)B * NP * (KPE / 4), 256, 148 * 16), groups);
  V2S_DISPATCH_AT(at, im2col_kernel<T><<<grid, 256, 0, s>>>(pack4<const float*>(x, groups), pack4<T*>(out, groups), B));
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_cls_rows(const float* const* params, float* const* hidden, int groups, int B, cudaStream_t s,
                    const uint8_t* const* mask, const float* const* mask_token) {
  const MaskArgs mk = pack_masks(mask, mask_token, groups);
  if (any_mask(mask, groups))
    cls_rows_kernel<true><<<dim3(B, groups), D, 0, s>>>(pack4<const float*>(params, groups), pack4<float*>(hidden, groups), mk);
  else
    cls_rows_kernel<false><<<dim3(B, groups), D, 0, s>>>(pack4<const float*>(params, groups), pack4<float*>(hidden, groups), mk);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_assemble_tokens(const float* const* params, const float* const* tok, float* const* hidden, int groups,
                           int B, cudaStream_t s, const uint8_t* const* mask, const float* const* mask_token) {
  const MaskArgs mk = pack_masks(mask, mask_token, groups);
  if (any_mask(mask, groups))
    assemble_tokens_kernel<true><<<dim3(8, B, groups), 256, 0, s>>>(pack4<const float*>(params, groups),
                                                                  pack4<const float*>(tok, groups), pack4<float*>(hidden, groups), mk);
  else
    assemble_tokens_kernel<false><<<dim3(8, B, groups), 256, 0, s>>>(pack4<const float*>(params, groups),
                                                                   pack4<const float*>(tok, groups), pack4<float*>(hidden, groups), mk);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_gather_patch_rows(const void* const* src, void* const* dst, int groups, int B, int at, cudaStream_t s,
                             const uint8_t* const* mask) {
  dim3 grid(8, B, groups);
  const MaskArgs mk = pack_masks(mask, nullptr, groups);
  if (any_mask(mask, groups)) {
    V2S_DISPATCH_AT(at, (gather_patch_rows_kernel<T, true><<<grid, 256, 0, s>>>(pack4<const T*>(src, groups), pack4<T*>(dst, groups), mk)));
  } else {
    V2S_DISPATCH_AT(at, (gather_patch_rows_kernel<T, false><<<grid, 256, 0, s>>>(pack4<const T*>(src, groups), pack4<T*>(dst, groups), mk)));
  }
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_col2im(const float* const* rows, float* const* img, int groups, int B, cudaStream_t s) {
  dim3 grid(grid_for((int64_t)B * 3 * V2S_IMG * (V2S_IMG / 4), 256, 148 * 16), groups);
  col2im_kernel<<<grid, 256, 0, s>>>(pack4<const float*>(rows, groups), pack4<float*>(img, groups), B);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_ln_fwd(const float* const* x, const float* const* gamma, const float* const* beta, void* const* y,
                  float* const* mean, float* const* rstd, int groups, int M, int at, cudaStream_t s) {
  LnFwdP p;
  memset(&p, 0, sizeof(p));
  for (int g = 0; g < groups; ++g) {
    p.x[g] = x[g]; p.gamma[g] = gamma[g]; p.beta[g] = beta[g]; p.y[g] = y[g];
    p.mean[g] = mean ? mean[g] : nullptr; p.rstd[g] = rstd ? rstd[g] : nullptr;
  }
  p.M = M;
  int bx = (M + 15) / 16;
  if (bx > 148 * 6) bx = 148 * 6;
  dim3 grid(bx, groups);
  V2S_DISPATCH_AT(at, V2S_CUDA_OK(launch_pdl(ln_fwd_kernel<T>, grid, dim3(256), 0, s, p)));
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_ln_bwd(const void* const* dy, const float* const* x, const float* const* mean, const float* const* rstd,
                  const float* const* gamma, float* const* dres, void* const* dres_lp, float* const* dgamma,
                  float* const* dbeta, float* const* dcolsum, int groups, int M, int at, cudaStream_t s,
                  const DetScratch* det) {
  LnBwdP p;
  memset(&p, 0, sizeof(p));
  for (int g = 0; g < groups; ++g) {
    p.dy[g] = dy[g]; p.x[g] = x[g]; p.mean[g] = mean[g]; p.rstd[g] = rstd[g]; p.gamma[g] = gamma[g];
    p.dres[g] = dres[g]; p.dres_lp[g] = dres_lp ? dres_lp[g] : nullptr;
    p.dgamma[g] = dgamma ? dgamma[g] : nullptr; p.dbeta[g] = dbeta ? dbeta[g] : nullptr;
    p.dcolsum[g] = dcolsum ? dcolsum[g] : nullptr;
  }
  p.M = M;
  int bx = (M + 15) / 16;
  if (bx > 148 * 4) bx = 148 * 4;
  if (det && dgamma) {         // a fixed number of row ranges bounds the partial rows the last CTA sums
    if (bx > 148) bx = 148;
    if ((int64_t)groups * bx * 3 * D > det->part_floats) { set_error("ln_bwd: deterministic scratch too small"); return 1; }
    p.det_part = det->part; p.det_counters = det->counters;
  }
  dim3 grid(bx, groups);
  if (!dgamma) { V2S_DISPATCH_AT(at, V2S_CUDA_OK(launch_pdl(ln_bwd_kernel<T, false, false>, grid, dim3(256), 0, s, p))); }
  else if (det) { V2S_DISPATCH_AT(at, V2S_CUDA_OK(launch_pdl(ln_bwd_kernel<T, true, true>, grid, dim3(256), 0, s, p))); }
  else { V2S_DISPATCH_AT(at, V2S_CUDA_OK(launch_pdl(ln_bwd_kernel<T, false, true>, grid, dim3(256), 0, s, p))); }
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_colsum(const void* const* dy, float* const* db, int groups, int M, int N, int t, cudaStream_t s,
                  const DetScratch* det) {
  if (N % 8 || N > 2048) { set_error("colsum: N must be a multiple of 8 and <= 2048 (got %d)", N); return 1; }
  ColsumP p;
  memset(&p, 0, sizeof(p));
  for (int g = 0; g < groups; ++g) { p.dy[g] = dy[g]; p.db[g] = db[g]; }
  p.M = M; p.N = N;
  int rows_t = 256 / (N / 8);
  if (rows_t * N > 2048) rows_t = 2048 / N;
  int bx = (M + rows_t * 16 - 1) / (rows_t * 16);     // >= 16 rows per row-lane
  if (bx > 148 * 4) bx = 148 * 4;
  if (bx < 1) bx = 1;
  if (det) {         // partial rows through the scratch; without scratch (the heads' few rows) one CTA per group
    if (bx > 148) bx = 148;
    if (!det->part) bx = 1;
    if (bx > 1 && (int64_t)groups * bx * N > det->part_floats) { set_error("colsum: deterministic scratch too small"); return 1; }
    p.det_part = det->part; p.det_counters = det->counters;
  }
  p.rows_per_block = (M + bx - 1) / bx;
  dim3 grid(bx, groups);
  if (det) { V2S_DISPATCH_AT(t, (colsum_kernel<T, true><<<grid, 256, 0, s>>>(p))); }
  else { V2S_DISPATCH_AT(t, (colsum_kernel<T, false><<<grid, 256, 0, s>>>(p))); }
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_pool_fwd(const float* const* hidden, float* const* feat, const int64_t* feat_stride, int groups, int B,
                    cudaStream_t s) {
  G4<int64_t> st;
  for (int i = 0; i < MAXG; ++i) st.p[i] = i < groups ? feat_stride[i] : 0;
  pool_fwd_kernel<<<dim3(B, groups), D, 0, s>>>(pack4<const float*>(hidden, groups), pack4<float*>(feat, groups), st);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_pool_bwd(const float* const* dfeat, const int64_t* dfeat_stride, const float* const* dhidden,
                    float* const* dx, void* const* dx_lp, int groups, int B, int at, cudaStream_t s) {
  G4<int64_t> st;
  for (int i = 0; i < MAXG; ++i) st.p[i] = i < groups ? dfeat_stride[i] : 0;
  for (int i = 0; i < groups; ++i)
    if ((dfeat[i] && ((reinterpret_cast<uintptr_t>(dfeat[i]) & 15) || (dfeat_stride[i] & 3))) ||
        (dhidden[i] && (reinterpret_cast<uintptr_t>(dhidden[i]) & 15))) {
      set_error("pool_bwd: dfeat / dhidden must be 16-byte aligned with a row stride that is a multiple of 4 floats");
      return 1;
    }
  dim3 grid(8, B, groups);
  V2S_DISPATCH_AT(at, pool_bwd_kernel<T><<<grid, 256, 0, s>>>(pack4<const float*>(dfeat, groups), st,
                                                             pack4<const float*>(dhidden, groups), pack4<float*>(dx, groups),
                                                             pack4<T*>(dx_lp, groups)));
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_embed_bwd(const float* const* dx, float* const* grads, int groups, int B, cudaStream_t s, const DetScratch* det,
                     const uint8_t* const* mask, float* const* dmask_token) {
  const bool masked = any_mask(mask, groups);
  const MaskArgs mk = pack_masks(mask, nullptr, groups);
  const G4<float*> dt = pack4<float*>(dmask_token, groups);
  const G4<const float*> cdx = pack4<const float*>(dx, groups);
  const G4<float*> gr = pack4<float*>(grads, groups);
  if (det) {
    if ((int64_t)groups * NP * D * (masked ? 2 : 1) > det->part_floats) { set_error("embed_bwd: deterministic scratch too small"); return 1; }
    if (masked) embed_bwd_kernel<true, true><<<dim3(NT, groups), D, 0, s>>>(cdx, gr, B, det->part, det->counters, mk, dt);
    else embed_bwd_kernel<true, false><<<dim3(NT, groups), D, 0, s>>>(cdx, gr, B, det->part, det->counters, mk, dt);
  } else {
    if (masked) embed_bwd_kernel<false, true><<<dim3(NT, groups), D, 0, s>>>(cdx, gr, B, nullptr, nullptr, mk, dt);
    else embed_bwd_kernel<false, false><<<dim3(NT, groups), D, 0, s>>>(cdx, gr, B, nullptr, nullptr, mk, dt);
  }
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_attn_fwd_simt(const void* const* qkv, void* const* ctx, float* const* lse, int groups, int B, int at,
                         cudaStream_t s) {
  const size_t smem = (size_t)(2 * NT * ASTR + 8 * 200 + 8 * DH) * sizeof(float);
  dim3 grid(NH, B, groups);
  V2S_DISPATCH_AT(at, {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_simt_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_fwd_simt_kernel<T><<<grid, 256, smem, s>>>(pack4<const T*>(qkv, groups), pack4<T*>(ctx, groups), pack4<float*>(lse, groups));
  });
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_attn_bwd_simt(const void* const* qkv, const void* const* ctx, const float* const* lse,
                         const void* const* dctx, void* const* dqkv, int groups, int B, int at, cudaStream_t s) {
  const size_t smem = (size_t)(4 * NT * ASTR + 2 * NT + 16 * 200) * sizeof(float);
  dim3 grid(NH, B, groups);
  V2S_DISPATCH_AT(at, {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_simt_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_bwd_simt_kernel<T><<<grid, 256, smem, s>>>(pack4<const T*>(qkv, groups), pack4<const T*>(ctx, groups),
                                                   pack4<const float*>(lse, groups), pack4<const T*>(dctx, groups),
                                                   pack4<T*>(dqkv, groups));
  });
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_attn_probs_simt(const void* const* qkv, const float* const* lse, float* const* probs, int groups, int B, int at,
                           cudaStream_t s) {
  const size_t smem = (size_t)(NT * ASTR + 8 * DH) * sizeof(float);
  dim3 grid(NH, B, groups);
  V2S_DISPATCH_AT(at, {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_probs_simt_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_probs_simt_kernel<T, false><<<grid, 256, smem, s>>>(pack4<const T*>(qkv, groups), pack4<const T*>(qkv, groups),
                                                             pack4<const float*>(lse, groups), pack4<float*>(probs, groups));
  });
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_attn_dprobs_simt(const void* const* qkv, const void* const* dctx, float* const* dprobs, int groups, int B, int at,
                            cudaStream_t s) {
  const size_t smem = (size_t)(NT * ASTR + 8 * DH) * sizeof(float);
  dim3 grid(NH, B, groups);
  V2S_DISPATCH_AT(at, {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_probs_simt_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_probs_simt_kernel<T, true><<<grid, 256, smem, s>>>(pack4<const T*>(qkv, groups), pack4<const T*>(dctx, groups),
                                                            G4<const float*>{}, pack4<float*>(dprobs, groups));
  });
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_residual_grad_add(const float* const* dh, float* const* dx, void* const* dx_lp, float* const* dcol, int groups, int B,
                             int at, cudaStream_t s, const DetScratch* det) {
  for (int i = 0; i < groups; ++i)
    if (reinterpret_cast<uintptr_t>(dh[i]) & 15) { set_error("hidden-state gradients must be 16-byte aligned"); return 1; }
  const int rows = B * NT;
  dim3 grid(grid_for(rows, RGA_RL, 148 * 2), groups);
  if (det && (int64_t)groups * grid.x * D > det->part_floats) { set_error("residual_grad_add: deterministic scratch too small"); return 1; }
  if (det) {
    V2S_DISPATCH_AT(at, (residual_grad_add_kernel<T, true><<<grid, 256, 0, s>>>(
                            pack4<const float*>(dh, groups), pack4<float*>(dx, groups), pack4<T*>(at ? dx_lp : nullptr, groups),
                            pack4<float*>(dcol, groups), rows, det->part, det->counters)));
  } else {
    V2S_DISPATCH_AT(at, (residual_grad_add_kernel<T, false><<<grid, 256, 0, s>>>(
                            pack4<const float*>(dh, groups), pack4<float*>(dx, groups), pack4<T*>(at ? dx_lp : nullptr, groups),
                            pack4<float*>(dcol, groups), rows, nullptr, nullptr)));
  }
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_cosine_loss(const float* p, const float* z, float* loss, float* dp, int B, int accum, float grad_scale,
                       cudaStream_t s, const float* grad_scale_dev) {
  const float inv_count = 1.0f / ((float)B * (float)accum);
  cosine_loss_kernel<<<1, 256, 0, s>>>(p, z, loss, dp, B, inv_count, grad_scale, grad_scale_dev);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_infonce_loss(const float* p, const float* z_all, float* loss, float* row_loss, float* dp, int B, int n_keys,
                        long long label_offset, float temperature, int accum, float grad_scale, cudaStream_t s,
                        const float* grad_scale_dev) {
  if (n_keys < 1 || n_keys > 6000) { set_error("infonce: 1..6000 keys (got %d)", n_keys); return 1; }
  if (label_offset < 0 || label_offset + B > n_keys) { set_error("infonce: the positives [%lld, +%d) are not among the %d keys", label_offset, B, n_keys); return 1; }
  if (!(temperature > 0.f)) { set_error("infonce: temperature must be positive"); return 1; }
  const float inv_count = 1.0f / ((float)B * (float)accum);
  infonce_row_kernel<<<B, NCE_THREADS, (size_t)n_keys * 2 * sizeof(float), s>>>(p, z_all, row_loss, dp, n_keys, label_offset,
                                                                               1.0f / temperature, inv_count * grad_scale,
                                                                               grad_scale_dev);
  V2S_LAUNCH_CHECK();
  infonce_mean_kernel<<<1, 256, 0, s>>>(row_loss, loss, B, inv_count);
  V2S_LAUNCH_CHECK();
  return 0;
}

namespace {
int pack_ranges(const v2s_range_t* ranges, int n, AdamRanges* rs, int64_t* mx) {
  if (n < 1 || n > 4) { set_error("adam: 1..4 ranges"); return 1; }
  *mx = 0;
  for (int i = 0; i < 4; ++i) {
    if (i < n) { rs->r[i] = ranges[i]; if (ranges[i].numel > *mx) *mx = ranges[i].numel; }
    else memset(&rs->r[i], 0, sizeof(v2s_range_t));
  }
  rs->n = n;
  return 0;
}
}  // namespace

int launch_adam(const v2s_range_t* ranges, int n, int64_t step, double lr, double b1, double b2, double eps, double wd,
                double grad_scale, cudaStream_t s, int lp_f16) {
  AdamRanges rs;
  int64_t mx;
  V2S_TRY(pack_ranges(ranges, n, &rs, &mx));
  const double bc1 = 1.0 - pow(b1, (double)step);
  const double bc2 = 1.0 - pow(b2, (double)step);
  AdamHyper hy;
  hy.step_size = (float)(lr / bc1); hy.bc2_sqrt = (float)sqrt(bc2); hy.skip = 0.f; hy.gmul = (float)grad_scale;
  dim3 grid(grid_for(mx / 4 + 1, 256, 148 * 8), n);
  adam_kernel<false><<<grid, 256, 0, s>>>(rs, hy, nullptr, (float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)eps,
                                          (float)wd, lp_f16);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_adam_amp(const v2s_range_t* ranges, int n, float* state8, double lr, double b1, double b2, double eps, double wd,
                    double grad_multiplier, const float* grad_scale_dev, const float* found_inf_dev, int lp_f16, int advance,
                    cudaStream_t s) {
  AdamRanges rs;
  int64_t mx;
  V2S_TRY(pack_ranges(ranges, n, &rs, &mx));
  if (advance) {
    adam_prologue_kernel<<<1, 1, 0, s>>>(state8, lr, b1, b2, grad_multiplier, grad_scale_dev, found_inf_dev);
    V2S_LAUNCH_CHECK();
  }
  AdamHyper hy;
  memset(&hy, 0, sizeof(hy));
  dim3 grid(grid_for(mx / 4 + 1, 256, 148 * 8), n);
  adam_kernel<true><<<grid, 256, 0, s>>>(rs, hy, state8, (float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)eps, (float)wd,
                                         lp_f16);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_ema(float* const* tgt, const float* const* onl, void* const* tgt_lp, int n_pairs, int64_t numel,
               double momentum, cudaStream_t s, int lp_f16) {
  if (n_pairs < 1 || n_pairs > 4) { set_error("ema: 1..4 pairs"); return 1; }
  if (numel % 4) { set_error("ema: numel must be a multiple of 4"); return 1; }
  EmaPairs pr;
  for (int i = 0; i < 4; ++i) {
    pr.t[i] = i < n_pairs ? tgt[i] : nullptr;
    pr.o[i] = i < n_pairs ? onl[i] : nullptr;
    pr.lp[i] = (i < n_pairs && tgt_lp) ? static_cast<uint16_t*>(tgt_lp[i]) : nullptr;
  }
  const float om = (float)(1.0 - momentum);   // python: (1 - momentum) in double, then fp32
  dim3 grid(grid_for(numel / 4, 256, 148 * 4), n_pairs);
  ema_kernel<<<grid, 256, 0, s>>>(pr, numel, (float)momentum, om, lp_f16);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_cast_lp(const float* src, void* dst, int64_t n, cudaStream_t s, int lp_f16) {
  cast_lp_kernel<<<grid_for(n / 4 + 1, 256, 148 * 8), 256, 0, s>>>(src, static_cast<uint16_t*>(dst), n, lp_f16);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_dropout_mask(float* mask, int64_t n, float p, uint64_t seed, uint64_t offset, cudaStream_t s) {
  dropout_mask_kernel<<<grid_for(n, 256), 256, 0, s>>>(mask, n, p, 1.0f / (1.0f - p), seed, offset);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_preprocess_u8_patches(const uint8_t* src, void* out, int B, int lp_f16, cudaStream_t s) {
  const int grid = grid_for((int64_t)B * NP * (KPE / 4), 256, 148 * 16);
  if (lp_f16) preprocess_u8_patches_kernel<f16><<<grid, 256, 0, s>>>(src, static_cast<f16*>(out), B);
  else preprocess_u8_patches_kernel<bf16><<<grid, 256, 0, s>>>(src, static_cast<bf16*>(out), B);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_preprocess_u8(const uint8_t* src, float* dst, int B, cudaStream_t s) {
  preprocess_u8_kernel<<<grid_for((int64_t)B * V2S_IMG * V2S_IMG, 256, 148 * 16), 256, 0, s>>>(src, dst, B);
  V2S_LAUNCH_CHECK();
  return 0;
}

template <bool ADD>
__global__ void splitk_reduce_kernel(float* __restrict__ out, const float* __restrict__ part,
                                     const float* __restrict__ bias, int MN, int N, int splits) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < MN; i += gridDim.x * blockDim.x) {
    float v = ADD ? out[i] : bias ? bias[i % N] : 0.f;
    for (int s = 0; s < splits; ++s) v += part[(int64_t)s * MN + i];      // fixed order: deterministic
    out[i] = v;
  }
}

// out[m,n] = bias[n] + sum_s part[s][m][n] (add: out[m,n] += sum_s part[s][m][n]): deterministic second pass of a split-K GEMM
int launch_splitk_reduce(float* out, const float* part, const float* bias, int M, int N, int splits, cudaStream_t s, bool add) {
  if (add) splitk_reduce_kernel<true><<<grid_for((int64_t)M * N, 256, 148), 256, 0, s>>>(out, part, nullptr, M * N, N, splits);
  else splitk_reduce_kernel<false><<<grid_for((int64_t)M * N, 256, 148), 256, 0, s>>>(out, part, bias, M * N, N, splits);
  V2S_LAUNCH_CHECK();
  return 0;
}

int launch_zero(void* p, int64_t bytes, cudaStream_t s) {
  V2S_CUDA_OK(cudaMemsetAsync(p, 0, (size_t)bytes, s));
  return 0;
}

}  // namespace v2s
