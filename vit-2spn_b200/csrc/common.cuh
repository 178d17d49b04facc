// Shared definitions for the vit2spn sm_100a kernels.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <utility>

#include "../../include/vit2spn.h"

namespace v2s {

typedef __nv_bfloat16 bf16;
typedef __half f16;
// activation type tags used across the launchers: 0 = fp32, 1 = bf16, 2 = fp16
constexpr int AT_F32 = 0, AT_BF16 = 1, AT_F16 = 2;

constexpr int D = V2S_HIDDEN;        // 192
constexpr int NT = V2S_TOKENS;       // 197
constexpr int NP = V2S_PATCHES;      // 196
constexpr int NH = V2S_HEADS;        // 3
constexpr int DH = V2S_HEAD_DIM;     // 64
constexpr int DF = V2S_MLP;          // 768
constexpr int NL = V2S_LAYERS;       // 12
constexpr int KPE = V2S_PATCH_K;     // 768
constexpr int MAXG = V2S_MAX_GROUPS; // 4
constexpr float LN_EPS = 1e-12f;     // HF ViTConfig.layer_norm_eps

// ---- flat parameter layout of one backbone (element offsets, fp32 and bf16 copies alike) ----
constexpr int64_t OFF_CLS = 0;
constexpr int64_t OFF_POS = OFF_CLS + D;
constexpr int64_t OFF_WPE = OFF_POS + (int64_t)NT * D;
constexpr int64_t OFF_BPE = OFF_WPE + (int64_t)D * KPE;
constexpr int64_t OFF_LAYER0 = OFF_BPE + D;
// within a layer
constexpr int64_t L_WQKV = 0;
constexpr int64_t L_BQKV = L_WQKV + 3 * D * D;
constexpr int64_t L_WO = L_BQKV + 3 * D;
constexpr int64_t L_BO = L_WO + D * D;
constexpr int64_t L_W1 = L_BO + D;
constexpr int64_t L_B1 = L_W1 + (int64_t)DF * D;
constexpr int64_t L_W2 = L_B1 + DF;
constexpr int64_t L_B2 = L_W2 + (int64_t)D * DF;
constexpr int64_t L_LN1W = L_B2 + D;
constexpr int64_t L_LN1B = L_LN1W + D;
constexpr int64_t L_LN2W = L_LN1B + D;
constexpr int64_t L_LN2B = L_LN2W + D;
constexpr int64_t LAYER_NUMEL = L_LN2B + D;
constexpr int64_t OFF_ACTIVE_END = OFF_LAYER0 + NL * LAYER_NUMEL;
constexpr int64_t OFF_LNF_W = OFF_ACTIVE_END;
constexpr int64_t OFF_LNF_B = OFF_LNF_W + D;
constexpr int64_t OFF_POOL_W = OFF_LNF_B + D;
constexpr int64_t OFF_POOL_B = OFF_POOL_W + D * D;
constexpr int64_t BACKBONE_NUMEL = OFF_POOL_B + D;
static_assert(BACKBONE_NUMEL == 5561472, "backbone numel");
static_assert(OFF_ACTIVE_END == 5524032, "active numel");

// heads (flat): projection_head.0 W[1024,384],b ; .3 W[128,1024],b ; prediction_head.0 W[128,128],b ; .2 W,b
constexpr int64_t H_W1 = 0;
constexpr int64_t H_B1 = H_W1 + (int64_t)V2S_PROJ_HID * V2S_PROJ_IN;
constexpr int64_t H_W2 = H_B1 + V2S_PROJ_HID;
constexpr int64_t H_B2 = H_W2 + (int64_t)V2S_PROJ_OUT * V2S_PROJ_HID;
constexpr int64_t H_W3 = H_B2 + V2S_PROJ_OUT;
constexpr int64_t H_B3 = H_W3 + V2S_PROJ_OUT * V2S_PROJ_OUT;
constexpr int64_t H_W4 = H_B3 + V2S_PROJ_OUT;
constexpr int64_t H_B4 = H_W4 + V2S_PROJ_OUT * V2S_PROJ_OUT;
constexpr int64_t HEADS_NUMEL = H_B4 + V2S_PROJ_OUT;
static_assert(HEADS_NUMEL == 558464, "heads numel");

inline int64_t layer_off(int l) { return OFF_LAYER0 + (int64_t)l * LAYER_NUMEL; }

// per-device library state (function attributes, error flag, SM count) is indexed by the CURRENT device of the calling
// thread: the host mirror makes the tensors' device current around every call
constexpr int MAX_DEVICES = 16;
inline int cur_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0) d = 0;
  return d < MAX_DEVICES ? d : MAX_DEVICES - 1;
}

// ---- error handling ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern int64_t g_launch_count;

// ---- deterministic mode (v2s_set_deterministic) ------------------------------------------------
// Scratch the fixed-order reductions of a backward call take from the tail of the caller's workspace.  `counters`
// are arrival counters: zero before every launch that uses them (cleared once per backward call, then reset by each
// launch's last arriver).  `part` holds per-CTA partial rows / split-K partial tiles of one launch at a time.
constexpr int DET_COUNTERS = 1024;
struct DetScratch {
  unsigned* counters;
  float* part;
  int64_t part_floats;
};

#define V2S_CUDA_OK(expr)                                                                     \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      v2s::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 1;                                                                               \
    }                                                                                         \
  } while (0)

#define V2S_LAUNCH_CHECK()                                                                    \
  do {                                                                                        \
    ++v2s::g_launch_count;                                                                    \
    cudaError_t _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) {                                                                  \
      v2s::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 1;                                                                               \
    }                                                                                         \
  } while (0)

#define V2S_TRY(expr)             \
  do {                            \
    int _r = (expr);              \
    if (_r != 0) return _r;       \
  } while (0)

// ---- launch with programmatic stream serialization (PDL); the kernel must call ptx::pdl_wait() ----
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---- device helpers ---------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<f16>(f16 v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ f16 from_f<f16>(float v) { return __float2half_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// exact (erf) GELU and its derivative — HF hidden_act="gelu" (modeling_vit.py:297-298)
__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad_f(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752f));
  const float pdf = 0.39894228040143268f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// ---- input image size of the backbone calls (v2s_set_image_size; default 224 x 224) ----------------
// H, W: pixels (multiples of 16); gh x gw: the patch grid; np = gh * gw patches, nt = np + 1 tokens (at most 197)
struct ImageGeom { int H, W, gh, gw, np, nt; };
const ImageGeom& image_geom();
inline bool geom_is_default(const ImageGeom& g) { return g.H == V2S_IMG && g.W == V2S_IMG; }

// per-group pointer bundles passed by value to grouped kernels (blockIdx.z = group)
template <typename T> struct GPtr {
  T* p[MAXG];
};

}  // namespace v2s
