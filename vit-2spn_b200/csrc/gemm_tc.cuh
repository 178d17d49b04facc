// tcgen05 / TMEM / TMA tensor-core GEMM family (bf16 operands, fp32 accumulate) — sm_100a only.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "gemm_simt.cuh"

namespace v2s {

// resolves the driver entry point for tensor-map encoding; 0 on success
int gemm_tc_init();
// tries to run `d` on the tensor-core path; *handled = 1 if it did (0: caller falls back to SIMT,
// only ever taken for shapes/types the tcgen05 kernels do not cover, e.g. fp32 check mode).  A 16-bit GEMM
// before gemm_tc_init is an error, not a fall-back.
int launch_gemm_tc(const GemmDesc& d, int ta, int tb, int to, cudaStream_t stream, int* handled);
// shared with the attention and MLP kernels: cached tensor maps (an error before gemm_tc_init), error flag
int tmap_get_3d(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1_bytes,
                uint64_t s2_bytes, uint32_t b0, uint32_t b1, bool is_bf16, int swizzle_bytes);
// cached rank-2 tensor map of a row-major [d1 rows, d0 cols] 16-bit (is_lp) or fp32 tensor, box b0 x b1
int tmap_get_2d(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t stride1_elems, uint32_t b0,
                uint32_t b1, bool is_lp, int swizzle_bytes);
int tc_num_sms();              // SMs persistent grids may use on the current device (see v2s_set_sm_limit)
void tc_set_sm_limit(int n);
void tc_set_deterministic(int on);   // v2s_set_deterministic
int tc_deterministic();
// floats of DetScratch::part the deterministic split-K wgrad needs on the current device (one wave of fp32 tiles)
int64_t gemm_tc_det_part_floats();
int* tc_err_flag();
long long* tc_dbg_counters();   // 32 device counters when V2S_GEMM_DEBUG is set, else NULL
int gemm_tc_debug_counters(long long* host32);
// reads and clears the device-side protocol error flag (0 = none); synchronises
int gemm_tc_error_flag();
// test hook behind v2s_test_gemm
int gemm_tc_test(int which, const void* a, const void* b, void* c, int m, int n, int k, int variant,
                 cudaStream_t stream);

}  // namespace v2s
