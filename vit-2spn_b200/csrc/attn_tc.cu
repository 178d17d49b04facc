// tcgen05 attention for the 197-token ViT-Tiny blocks (3 heads x 64).  All 197 keys fit one tile (padded to
// 208), so the softmax is a plain two-pass row softmax over a 128 x 208 fp32 score tile held in tensor
// memory - no online rescaling.
//
//   forward:  S = Q K^T (UMMA 128x208x64, both K-major)  ->  P = softmax(S/8) (TMEM -> registers -> bf16
//             pairs back into TMEM over the consumed scores)  ->  O = P V (UMMA 128x64x208, A = P from
//             tensor memory, V MN-major)  -> O / rowsum -> bf16 -> TMA store; log-sum-exp saved for the
//             backward.  attn_fwd_persist_kernel: persistent CTAs, two jobs in flight.
//   backward: see attn_bwd_tc_kernel.
#include <string.h>

#include "gemm_tc.cuh"
#include "kernels.cuh"
#include "ptx.cuh"
#include "tc_math.cuh"

namespace v2s {

namespace {

constexpr int KPAD = 208;                      // keys padded to a multiple of 16
constexpr int QT = 128;                        // query rows per tile (2 tiles cover 197)
constexpr int Q_TILE_BYTES = QT * DH * 2;      // 16384
constexpr int KV_TILE_BYTES = KPAD * DH * 2;   // 26624
constexpr int P_TILE_BYTES = 4 * QT * 128;     // 65536: four 64-key column blocks of 128 rows x 128 B
constexpr float SCALE = 0.125f;                // 64^-0.5
constexpr float SCALE_LOG2E = 0.125f * 1.4426950408889634f;

// one UMMA with SWIZZLE_128B operands given by smem address + leading-dimension byte offset (SBO = 1024)
__device__ __forceinline__ void mma(uint32_t d_tmem, uint32_t a_addr, uint32_t a_lbo, uint32_t b_addr, uint32_t b_lbo,
                                    uint32_t idesc, bool accumulate) {
  ptx::umma_bf16_lohi(d_tmem, ptx::desc_lo(a_addr, a_lbo), ptx::desc_lo(b_addr, b_lbo), ptx::DESC_HI_SW128_SBO1024,
                      idesc, accumulate ? 1u : 0u);
}

// writes 8 consecutive bf16 (one 16-byte chunk) of row r, key group c8 (keys 8*c8..8*c8+7) into a
// K-major SWIZZLE_128B operand tile made of 64-key column blocks of [128 rows x 128 B]
__device__ __forceinline__ void store_p_chunk(uint8_t* tile, int r, int c8, uint4 v) {
  const int block = c8 >> 3, chunk = c8 & 7;
  *reinterpret_cast<uint4*>(tile + block * (QT * 128) + r * 128 + ((chunk ^ (r & 7)) << 4)) = v;
}

// ---- forward, persistent ----------------------------------------------------------------------
// One CTA per SM walks the (query tile, head, image, backbone) jobs.  Three shared-memory stages [Q | K | V]
// are filled by a TMA producer warp ahead of use; a store warp owns the output staging tile; two tensor-memory slots (256 columns each) hold the scores of
// two jobs in flight, each served by its own eight softmax warps (two threads per query row: keys [0,112) and
// [112,208)), so the softmax of one job overlaps the UMMAs and the epilogue of the other.
//   TMEM slot: S [0,208) fp32 -> P bf16x2 in place ([0,56) and [112,160): each thread packs over scores it has
//   already consumed itself) -> O accumulator [160,224).
constexpr int PF_STAGES = 3;
constexpr int PF_STAGE_BYTES = Q_TILE_BYTES + 2 * KV_TILE_BYTES;   // 69632
constexpr int PF_OFF_STG = PF_STAGES * PF_STAGE_BYTES;             // 208896: O staging tile (16 KB)
constexpr int PF_OFF_XCH = PF_OFF_STG + Q_TILE_BYTES;              // 225280: row max / row sum exchange (4 KB)
constexpr int PF_OFF_BAR = PF_OFF_XCH + 4096;                      // 229376
constexpr int PF_SMEM = PF_OFF_BAR + 256 + 1024;                   // 230656
constexpr int PF_THREADS = 96 + 2 * 256;                          // producer, UMMA, store warps + 2 x 8 softmax warps
constexpr int PF_KSPLIT = 112;                                     // keys [0,112) | [112,208)
constexpr int PF_TM_PB = 112;                                      // P columns of the second key half
constexpr int PF_TM_O = 160;
static_assert(PF_STAGE_BYTES % 1024 == 0 && PF_SMEM <= 232448, "persistent attention smem map");

struct alignas(64) AttnFwdPParams {
  CUtensorMap tmQ[MAXG], tmKV[MAXG], tmCtx[MAXG];
  float* lse[MAXG];
  int B, total_jobs;
  int* err_flag;
  long long* dbg;   // optional cycle counters of CTA 0 (V2S_GEMM_DEBUG): [0..3] UMMA warp waits, [8..15] softmax thread phases
  int N, ntiles;    // VAR: tokens (2..197) and query tiles (1 or 2) per image
  int KP;           // VAR: keys padded to round_up(N, 16): the N of the S UMMA, KP / 16 K-steps of P V
};

// DBG: instrumented build (phase cycle counters), launched only when V2S_GEMM_DEBUG is set.  VAR: p.N tokens instead of 197
// (v2s_set_image_size): S = Q K^T is a 128 x KP tile (KP = round_up(N, 16); TMA zero-fills the keys past N per image) and
// P V takes KP / 16 K-steps; 32-key chunks past N are skipped and the one chunk that holds key N is bounds-checked
// (keys >= N get p = 0); with N <= 128 a job is one query tile
template <bool DBG, typename LP, bool VAR = false>
__global__ void __launch_bounds__(PF_THREADS, 1) attn_fwd_persist_kernel(const __grid_constant__ AttnFwdPParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar_load = reinterpret_cast<uint64_t*>(smem + PF_OFF_BAR);   // [3] stage filled
  uint64_t* bar_sfree = bar_load + 3;                                    // [3] stage consumed (P V retired)
  uint64_t* bar_s = bar_sfree + 3;                                       // [2] scores ready
  uint64_t* bar_p = bar_s + 2;                                           // [2] P written (256 threads)
  uint64_t* bar_o = bar_p + 2;                                           // [2] O ready
  uint64_t* bar_tfree = bar_o + 2;                                       // [2] O read out: slot reusable
  uint64_t* bar_full = bar_tfree + 2;                                    // [2] output tile staged (256 threads)
  uint64_t* bar_stgfree = bar_full + 2;                                  // [2] staging tile free for this slot's next job
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar_stgfree + 2);
  float* xch = reinterpret_cast<float*>(smem + PF_OFF_XCH);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 3; ++i) { ptx::mbar_init(&bar_load[i], 1); ptx::mbar_init(&bar_sfree[i], 1); }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bar_s[i], 1); ptx::mbar_init(&bar_p[i], 256); ptx::mbar_init(&bar_o[i], 1); ptx::mbar_init(&bar_tfree[i], 256);
      ptx::mbar_init(&bar_full[i], 256); ptx::mbar_init(&bar_stgfree[i], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_ptr, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();     // after the wait: see the dependent-launch note in gemm_tc.cu

  const int njobs = ((int)blockIdx.x < p.total_jobs) ? (p.total_jobs - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int nt = VAR ? p.N : NT;
  const bool two_tiles = !VAR || p.ntiles == 2;
  auto decode = [&](int n, int& t, int& h, int& b, int& g) {
    const int J = blockIdx.x + n * gridDim.x;
    t = two_tiles ? (J & 1) : 0;
    int r = two_tiles ? (J >> 1) : J;
    h = r % NH; r /= NH;
    b = r % p.B; g = r / p.B;
  };

  if (warp == 0) {
    // ---- TMA producer ----
    for (int n = 0; n < njobs; ++n) {
      const int st = n % PF_STAGES;
      if (n >= PF_STAGES) ptx::mbar_wait(&bar_sfree[st], ((n / PF_STAGES) - 1) & 1, p.err_flag, 31);
      int t, h, b, g;
      decode(n, t, h, b, g);
      if (ptx::elect_one()) {
        uint8_t* stage = smem + st * PF_STAGE_BYTES;
        ptx::mbar_arrive_expect_tx(&bar_load[st], PF_STAGE_BYTES);
        ptx::tma_load_3d(stage, &p.tmQ[g], &bar_load[st], h * DH, t * QT, b);
        ptx::tma_load_3d(stage + Q_TILE_BYTES, &p.tmKV[g], &bar_load[st], D + h * DH, 0, b);
        ptx::tma_load_3d(stage + Q_TILE_BYTES + KV_TILE_BYTES, &p.tmKV[g], &bar_load[st], 2 * D + h * DH, 0, b);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---- UMMA issuer: S(n) as soon as its stage and slot are ready, then P V of job n-1 ----
    const int kp = VAR ? p.KP : KPAD;
    const uint32_t idesc_s = make_idesc_lp(LP::kIdescFmt, QT, kp, 0, 0);
    const uint32_t idesc_o = make_idesc_lp(LP::kIdescFmt, QT, DH, 0, 1);
    const uint32_t sbase = ptx::smem_u32(smem);
    long long w_load = 0, w_tfree = 0, w_p = 0; const long long t_mma0 = clock64();
    for (int n = 0; n <= njobs; ++n) {
      if (n < njobs) {
        const int st = n % PF_STAGES, sl = n & 1;
        long long w0 = DBG ? clock64() : 0;
        ptx::mbar_wait(&bar_load[st], (n / PF_STAGES) & 1, p.err_flag, 32);
        if (DBG) { const long long w1 = clock64(); w_load += w1 - w0; w0 = w1; }
        if (n >= 2) ptx::mbar_wait(&bar_tfree[sl], ((n >> 1) - 1) & 1, p.err_flag, 33);
        if (DBG) w_tfree += clock64() - w0;
        ptx::tc_fence_after();
        const uint32_t sq = sbase + st * PF_STAGE_BYTES, sk = sq + Q_TILE_BYTES;
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < DH / 16; ++k) mma(tmem_base + sl * 256, sq + k * 32, 16, sk + k * 32, 16, idesc_s, k > 0);
          ptx::umma_commit(&bar_s[sl]);
        }
        __syncwarp();
      }
      if (n >= 1) {
        const int m = n - 1, st = m % PF_STAGES, sl = m & 1;
        const long long w0 = DBG ? clock64() : 0;
        ptx::mbar_wait(&bar_p[sl], (m >> 1) & 1, p.err_flag, 34);
        if (DBG) w_p += clock64() - w0;
        ptx::tc_fence_after();
        const uint32_t sv = sbase + st * PF_STAGE_BYTES + Q_TILE_BYTES + KV_TILE_BYTES;
        const uint32_t tslot = tmem_base + sl * 256;
        if (ptx::elect_one()) {
#pragma unroll
          for (int j = 0; j < kp / 16; ++j) {
            const uint32_t a = tslot + (j < PF_KSPLIT / 16 ? 8 * j : PF_TM_PB + 8 * (j - PF_KSPLIT / 16));
            ptx::umma_bf16_ts(tslot + PF_TM_O, a, ptx::desc_lo(sv + j * 2048, 8192), ptx::DESC_HI_SW128_SBO1024, idesc_o,
                              j > 0 ? 1u : 0u);
          }
          ptx::umma_commit(&bar_o[sl]);
          ptx::umma_commit(&bar_sfree[st]);
        }
        __syncwarp();
      }
    }
    if (DBG && blockIdx.x == 0 && lane == 0) { p.dbg[0] = w_load; p.dbg[1] = w_tfree; p.dbg[2] = w_p; p.dbg[3] = clock64() - t_mma0; p.dbg[4] = njobs; }
  } else if (warp == 2) {
    // ---- store warp: staging tile -> global.  Jobs use the single staging tile in job order; its release is
    // signalled to the slot of the NEXT job, so every slot sees its own completions in order. ----
    if (ptx::elect_one()) ptx::mbar_arrive(&bar_stgfree[0]);       // free for job 0
    __syncwarp();
    for (int n = 0; n < njobs; ++n) {
      const int sl = n & 1;
      ptx::mbar_wait(&bar_full[sl], (n >> 1) & 1, p.err_flag, 38);
      int t, h, b, g;
      decode(n, t, h, b, g);
      if (ptx::elect_one()) {
        ptx::tma_store_3d(&p.tmCtx[g], smem + PF_OFF_STG, h * DH, t * QT, b);   // rows >= 197 are clipped by TMA
        ptx::tma_commit_group();
        ptx::tma_wait_group_read<0>();
        ptx::mbar_arrive(&bar_stgfree[sl ^ 1]);
      }
      __syncwarp();
    }
    if (ptx::elect_one()) ptx::tma_wait_group<0>();
    __syncwarp();
  } else {
    // ---- softmax + epilogue warps: slot sl, TMEM lane quarter q, key half hf ----
    const int sw = warp - 3, sl = sw >> 3, hf = (sw & 7) >> 2, q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + sl * 256;
    float* xmax = xch + sl * 512;
    float* xsum = xmax + 256;
    const int bar_id = 1 + sl;
    const int key0 = hf ? PF_KSPLIT : 0;
    const int pcol0 = hf ? PF_TM_PB : 0;
    uint32_t r[32], r2[32];
    long long tk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = 0; 2 * j + sl < njobs; ++j) {
      const int n = 2 * j + sl;
      int t, h, b, g;
      decode(n, t, h, b, g);
      const int qrow = t * QT + row;
      long long c0 = DBG ? clock64() : 0, c1;
#define V2S_TICK(k) if (DBG) { c1 = clock64(); tk[k] += c1 - c0; c0 = c1; }
      ptx::mbar_wait(&bar_s[sl], j & 1, p.err_flag, 35);
      V2S_TICK(0)
      ptx::tc_fence_after();
      // pass 1: maximum over this thread's keys, then over the row.  Tensor-memory loads are issued one chunk
      // ahead of the arithmetic (two register buffers) in both passes.
      float mx = -INFINITY;
      // only the last chunk of the second key half (keys 176..207) contains padding keys (>= 197): every other
      // chunk runs the unmasked variant, so the per-element bound checks stay out of the hot loop
      // VAR: the scores of keys >= N become -inf in the registers of a chunk that reaches past N (they then add nothing
      // to the maximum and give p = 0); a chunk wholly below N is left alone.  It runs right after the chunk's load
      // has landed and before the next load is issued, while only one register buffer is live.
      auto mask32 = [&](uint32_t* v, int kb, int n) {   // keys kb + i, i < n
        if (VAR && kb + n > nt) {
          const int lim = nt - kb;
#pragma unroll
          for (int i = 0; i < n; ++i) v[i] = i < lim ? v[i] : 0xff800000u;
        }
      };
      auto max32 = [&](const uint32_t* v, int kb) {   // VAR: a chunk wholly past N is skipped
        if (VAR && kb >= nt) return;
#pragma unroll
        for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(v[i]));
      };
      auto max32_tail = [&](const uint32_t* v) {       // keys 176 + i
#pragma unroll
        for (int i = 0; i < NT - 176; ++i) mx = fmaxf(mx, __uint_as_float(v[i]));
      };
      ptx::tmem_ld_32x32(taddr + key0, r);
      ptx::tmem_ld_wait();
      mask32(r, key0, 32);
      ptx::tmem_ld_32x32(taddr + key0 + 32, r2);
      max32(r, key0);
      ptx::tmem_ld_wait();
      mask32(r2, key0 + 32, 32);
      ptx::tmem_ld_32x32(taddr + key0 + 64, r);
      max32(r2, key0 + 32);
      ptx::tmem_ld_wait();
      mask32(r, key0 + 64, 32);
      if (hf == 0) ptx::tmem_ld_32x16(taddr + 96, r2);
      if (hf == 0 || VAR) max32(r, key0 + 64);
      else max32_tail(r);
      if (hf == 0) {
        ptx::tmem_ld_wait();
        mask32(r2, 96, 16);
#pragma unroll
        for (int i = 0; i < 16; ++i) mx = fmaxf(mx, __uint_as_float(r2[i]));
      }
      xmax[hf * 128 + row] = mx;
      ptx::tmem_ld_32x32(taddr + key0, r);           // first chunk of pass 2, in flight across the exchange
      V2S_TICK(1)
      ptx::bar_sync(bar_id, 256);
      V2S_TICK(2)
      mx = fmaxf(mx, xmax[(hf ^ 1) * 128 + row]);
      // pass 2: p = exp2((s - max) * scale * log2e); bf16 pairs back into tensor memory
      const float moff = mx * SCALE_LOG2E;
      float sum = 0.f;
      // VAR: masked keys give exp2(-inf) = 0; a chunk wholly past N holds keys >= KP, which P V does not read: skipped
      auto exp32 = [&](const uint32_t* v, int pcol, int kb) {
        if (VAR && kb >= nt) return;
        uint32_t pw[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float e0 = ptx::ex2_approx(fmaf(__uint_as_float(v[2 * i]), SCALE_LOG2E, -moff));
          const float e1 = ptx::ex2_approx(fmaf(__uint_as_float(v[2 * i + 1]), SCALE_LOG2E, -moff));
          sum += e0 + e1;
          pw[i] = LP::pack(e0, e1);
        }
        ptx::tmem_st_32x16(taddr + pcol, pw);
      };
      auto exp32_tail = [&](const uint32_t* v, int pcol) {     // keys 176 + 2i, 177 + 2i: padding keys get p = 0
        uint32_t pw[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float e0 = (176 + 2 * i < NT) ? ptx::ex2_approx(fmaf(__uint_as_float(v[2 * i]), SCALE_LOG2E, -moff)) : 0.f;
          const float e1 = (177 + 2 * i < NT) ? ptx::ex2_approx(fmaf(__uint_as_float(v[2 * i + 1]), SCALE_LOG2E, -moff)) : 0.f;
          sum += e0 + e1;
          pw[i] = LP::pack(e0, e1);
        }
        ptx::tmem_st_32x16(taddr + pcol, pw);
      };
      ptx::tmem_ld_wait();
      mask32(r, key0, 32);
      ptx::tmem_ld_32x32(taddr + key0 + 32, r2);
      exp32(r, pcol0, key0);
      ptx::tmem_ld_wait();
      mask32(r2, key0 + 32, 32);
      ptx::tmem_ld_32x32(taddr + key0 + 64, r);
      exp32(r2, pcol0 + 16, key0 + 32);
      ptx::tmem_ld_wait();
      mask32(r, key0 + 64, 32);
      if (hf == 0) ptx::tmem_ld_32x16(taddr + 96, r2);
      if (hf == 0 || VAR) exp32(r, pcol0 + 32, key0 + 64);
      else exp32_tail(r, pcol0 + 32);
      if (hf == 0) {
        ptx::tmem_ld_wait();
        mask32(r2, 96, 16);
        if (!VAR || 96 < nt) {
          uint32_t pw[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float e0 = ptx::ex2_approx(fmaf(__uint_as_float(r2[2 * i]), SCALE_LOG2E, -moff));
            const float e1 = ptx::ex2_approx(fmaf(__uint_as_float(r2[2 * i + 1]), SCALE_LOG2E, -moff));
            sum += e0 + e1;
            pw[i] = LP::pack(e0, e1);
          }
          ptx::tmem_st_32x8(taddr + 48, pw);
        }
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bar_p[sl]);
      xsum[hf * 128 + row] = sum;
      V2S_TICK(3)
      ptx::bar_sync(bar_id, 256);
      V2S_TICK(4)
      sum += xsum[(hf ^ 1) * 128 + row];
      if (hf == 0 && qrow < nt && p.lse[g]) p.lse[g][((int64_t)b * NH + h) * nt + qrow] = mx * SCALE + __logf(sum);
      const float inv = 1.0f / sum;
      // epilogue: this thread's 32 output columns -> bf16 -> staging tile -> TMA store
      ptx::mbar_wait(&bar_o[sl], j & 1, p.err_flag, 36);
      V2S_TICK(5)
      ptx::tc_fence_after();
      ptx::tmem_ld_32x32(taddr + PF_TM_O + hf * 32, r);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bar_tfree[sl]);
      uint8_t* stg = smem + PF_OFF_STG;
      ptx::mbar_wait(&bar_stgfree[sl], j & 1, p.err_flag, 37);    // the previous job's store has read the tile
      V2S_TICK(6)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        uint4 v;
        v.x = LP::pack(__uint_as_float(r[8 * jj]) * inv, __uint_as_float(r[8 * jj + 1]) * inv);
        v.y = LP::pack(__uint_as_float(r[8 * jj + 2]) * inv, __uint_as_float(r[8 * jj + 3]) * inv);
        v.z = LP::pack(__uint_as_float(r[8 * jj + 4]) * inv, __uint_as_float(r[8 * jj + 5]) * inv);
        v.w = LP::pack(__uint_as_float(r[8 * jj + 6]) * inv, __uint_as_float(r[8 * jj + 7]) * inv);
        *reinterpret_cast<uint4*>(stg + row * 128 + (((hf * 4 + jj) ^ (row & 7)) << 4)) = v;
      }
      ptx::fence_proxy_async();
      ptx::mbar_arrive(&bar_full[sl]);
      V2S_TICK(7)
    }
#undef V2S_TICK
    if (DBG && blockIdx.x == 0 && sw == 0 && lane == 0)
      for (int k = 0; k < 8; ++k) p.dbg[8 + k] = tk[k];
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// ---- backward ---------------------------------------------------------------------------------
// Persistent CTAs (one per SM) over the (head, image, backbone) jobs; the two 128-row query tiles of a job are processed
// one after the other while dK / dV accumulate in tensor memory across both.  A job is a serial chain (S -> P -> dP -> dS
// -> dQ, dK, dV) that needs almost all of shared memory (212 KB: the transposed uses of P and dS must come from shared
// memory), so nothing of the NEXT job can be resident early except what the chain has already released: its K and V are
// loaded as soon as the last dQ UMMAs have retired (they overlap the dQ / dK / dV drains), its Q tile after the last dK
// UMMAs; everything else the job will need (its first dO tile, the second Q / dO tiles) is prefetched into L2 a job /
// a tile ahead, so that the loads the chain does wait for are L2 hits (measured before: 35 % of a job was waiting for
// DRAM-latency TMA loads, one CTA per job).  The dO tile, whose buffer (it doubles as the dQ staging tile) is released
// last, signals its own barrier: only D, dP and dV wait for it, S = Q K^T and the P pass do not.  D = rowsum(dO * O) is
// computed between the P pass and the dS pass, under the dP UMMAs.
//   S  = Q_t K^T                      (UMMA 128x208x64)         -> P = exp2(S*c - lse*log2e)  (bf16, smem)
//   dP = dO_t V^T                     (UMMA 128x208x64)         -> dS = P * (dP - D) / 8      (bf16, smem)
//   dV += P^T dO_t,  dK += dS^T Q_t   (UMMA 128x64x128, A MN-major = the same smem tiles read transposed)
//   dQ_t = dS K                       (UMMA 128x64x208, K MN-major)
// TMEM columns: [0,208) S then dP then dQ_t | [256,384) dK (two 128-key tiles) | [384,512) dV.
constexpr int B_OFF_Q = 0;
constexpr int B_OFF_DO = Q_TILE_BYTES;
constexpr int B_OFF_K = 2 * Q_TILE_BYTES;
constexpr int B_OFF_V = B_OFF_K + KV_TILE_BYTES;
constexpr int B_OFF_P = B_OFF_V + KV_TILE_BYTES;
constexpr int B_OFF_DS = B_OFF_P + P_TILE_BYTES;
constexpr int B_OFF_BAR = B_OFF_DS + P_TILE_BYTES;       // 217088
constexpr int B_SMEM = B_OFF_BAR + 256 + 1024;
constexpr int B_THREADS = 288;
constexpr int TM_DK = 256, TM_DV = 384;
constexpr float LOG2E = 1.4426950408889634f;

struct alignas(64) AttnBwdParams {
  CUtensorMap tmQ[MAXG], tmKV[MAXG], tmDO[MAXG], tmDQKV[MAXG];
  const bf16* ctx[MAXG];
  const float* lse[MAXG];
  int B, total_jobs;
  int* err_flag;
  long long* dbg;   // optional phase cycle counters of CTA 0 (V2S_GEMM_DEBUG): [16..27]
  int N;            // VAR: tokens per image (2..197)
  int ntiles, KP;   // VAR: query tiles per job (1 or 2) and keys padded to round_up(N, 16)
};

// the same accesses through 32-bit shared addresses with the per-row part precomputed (rowbase = tile + r * 128,
// rx = r & 7): the backward softmax threads run at two warps per scheduler, where instruction count is time
__device__ __forceinline__ void store_p_chunk_s(uint32_t rowbase, int rx, int c8, uint4 v) {
  ptx::sts128(rowbase + (c8 >> 3) * (QT * 128) + (((c8 & 7) ^ rx) << 4), v.x, v.y, v.z, v.w);
}
__device__ __forceinline__ uint4 load_p_chunk_s(uint32_t rowbase, int rx, int c8) {
  return ptx::lds128(rowbase + (c8 >> 3) * (QT * 128) + (((c8 & 7) ^ rx) << 4));
}
__device__ __forceinline__ uint4 load_p_chunk(const uint8_t* tile, int r, int c8) {
  const int block = c8 >> 3, chunk = c8 & 7;
  return *reinterpret_cast<const uint4*>(tile + block * (QT * 128) + r * 128 + ((chunk ^ (r & 7)) << 4));
}

// VAR: p.N tokens instead of 197 (v2s_set_image_size): S and dP are 128 x KP tiles (KP = round_up(N, 16)), dQ takes KP / 16
// K-steps and dK / dV cover one 128-key tile when KP <= 128; 32-key chunks past N are skipped and the P chunks that hold
// key N are bounds-checked, so keys >= N get P = 0 and dS = 0; query rows >= N are masked through their lse as the rows
// >= 197 are; with N <= 128 a job is one query tile (dK / dV then accumulate over that one tile)
template <bool DBG, typename LP, bool VAR = false>
__global__ void __launch_bounds__(B_THREADS, 1) attn_bwd_tc_kernel(const __grid_constant__ AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar_load = reinterpret_cast<uint64_t*>(smem + B_OFF_BAR);   // [2]
  uint64_t* bar_s = bar_load + 2;     // [2]
  uint64_t* bar_p = bar_s + 2;        // [2] count 256
  uint64_t* bar_dp = bar_p + 2;       // [2]
  uint64_t* bar_ds = bar_dp + 2;      // [2] count 256
  uint64_t* bar_dq = bar_ds + 2;      // [2]
  uint64_t* bar_kv = bar_dq + 2;      // [2] all MMAs of the tile retired
  uint64_t* bar_free = bar_kv + 2;    // [1] count 256: tile-0 buffers and TMEM[0,208) reusable
  uint64_t* bar_done = bar_free + 1;  // [1] count 256: the dQ store of the job's second tile has read its staging tile
  uint64_t* bar_do = bar_done + 1;    // [2] the dO tile landed (its buffer is released last, so it has its own barrier:
                                      //     S = Q K^T and the P pass do not wait for it)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar_do + 2);
  const int njobs = ((int)blockIdx.x < p.total_jobs) ? (p.total_jobs - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  auto decode = [&](int n, int& h, int& b, int& g) {
    const int J = blockIdx.x + n * gridDim.x;
    h = J % NH;
    const int r = J / NH;
    b = r % p.B; g = r / p.B;
  };
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  const int tl = VAR ? p.ntiles - 1 : 1;        // the job's last query tile
  const int kp = VAR ? p.KP : KPAD;
  const int nmt = VAR && kp <= QT ? 1 : 2;      // 128-key tiles of dK / dV

  if (warp == 0) {
    if (lane == 0) {
      for (int t = 0; t < 2; ++t) {
        ptx::mbar_init(&bar_load[t], 1); ptx::mbar_init(&bar_s[t], 1); ptx::mbar_init(&bar_p[t], 256);
        ptx::mbar_init(&bar_dp[t], 1); ptx::mbar_init(&bar_ds[t], 256); ptx::mbar_init(&bar_dq[t], 1);
        ptx::mbar_init(&bar_kv[t], 1); ptx::mbar_init(&bar_do[t], 1);
      }
      ptx::mbar_init(bar_free, 256);
      ptx::mbar_init(bar_done, 256);
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(tmem_ptr, 512);
    ptx::tmem_relinquish();
  } else {
    // zero the never-written part of the 4th key block (keys 208..255) of P and dS: it is read as
    // garbage rows of the transposed A operand otherwise (harmless, but keep NaNs out of TMEM)
    for (int i = threadIdx.x - 32; i < QT * 6; i += B_THREADS - 32) {
      const int r = i / 6, c = 2 + i % 6;
      const uint4 z = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(smem + B_OFF_P + 3 * (QT * 128) + r * 128 + ((c ^ (r & 7)) << 4)) = z;
      *reinterpret_cast<uint4*>(smem + B_OFF_DS + 3 * (QT * 128) + r * 128 + ((c ^ (r & 7)) << 4)) = z;
    }
    ptx::fence_proxy_async();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
  ptx::pdl_wait();                  // prologue above overlapped the predecessor's tail
  ptx::pdl_launch_dependents();     // after the wait: see the dependent-launch note in gemm_tc.cu

  if (warp == 0) {
    // control warp: every lane walks the same path and waits on the barriers; one elected lane issues
    const uint32_t sbase = ptx::smem_u32(smem);
    const uint32_t sq = sbase + B_OFF_Q, sdo = sbase + B_OFF_DO, sk = sbase + B_OFF_K, sv = sbase + B_OFF_V;
    const uint32_t sp = sbase + B_OFF_P, sds = sbase + B_OFF_DS;
    const uint32_t idesc_s = make_idesc_lp(LP::kIdescFmt, QT, kp, 0, 0);
    const uint32_t idesc_dq = make_idesc_lp(LP::kIdescFmt, QT, DH, 0, 1);
    const uint32_t idesc_kv = make_idesc_lp(LP::kIdescFmt, QT, DH, 1, 1);
    constexpr uint32_t LOAD0_BYTES = Q_TILE_BYTES + 2 * KV_TILE_BYTES;
    if (njobs > 0) {      // the first job: everything at once
      int h, b, g;
      decode(0, h, b, g);
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&bar_load[0], LOAD0_BYTES);
        ptx::mbar_arrive_expect_tx(&bar_do[0], Q_TILE_BYTES);
        ptx::tma_load_3d(smem + B_OFF_Q, &p.tmQ[g], &bar_load[0], h * DH, 0, b);
        ptx::tma_load_3d(smem + B_OFF_DO, &p.tmDO[g], &bar_do[0], h * DH, 0, b);
        ptx::tma_load_3d(smem + B_OFF_K, &p.tmKV[g], &bar_load[0], D + h * DH, 0, b);
        ptx::tma_load_3d(smem + B_OFF_V, &p.tmKV[g], &bar_load[0], 2 * D + h * DH, 0, b);
      }
      __syncwarp();
    }
#pragma unroll 1
    for (int n = 0; n < njobs; ++n) {
      const uint32_t ph = n & 1;
      int h, b, g, h2 = 0, b2 = 0, g2 = 0;
      decode(n, h, b, g);
      const bool has_next = n + 1 < njobs;
      if (has_next) decode(n + 1, h2, b2, g2);
      if (ptx::elect_one()) {      // into L2 now, into shared memory when the chain gets there
        ptx::tma_prefetch_3d(&p.tmQ[g], h * DH, QT, b);
        ptx::tma_prefetch_3d(&p.tmDO[g], h * DH, QT, b);
        if (has_next) {
          ptx::tma_prefetch_3d(&p.tmDO[g2], h2 * DH, 0, b2);
          ptx::tma_prefetch_3d(&p.tmQ[g2], h2 * DH, 0, b2);
        }
      }
      __syncwarp();
#pragma unroll 1
      for (int t = 0; t <= tl; ++t) {
        if (t == 1) {
          ptx::mbar_wait(&bar_kv[0], ph, p.err_flag, 21);     // tile-0 MMAs no longer read Q/dO/P/dS
          ptx::mbar_wait(bar_free, ph, p.err_flag, 22);       // dQ_0 drained, staging store done
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(&bar_load[1], Q_TILE_BYTES);
            ptx::mbar_arrive_expect_tx(&bar_do[1], Q_TILE_BYTES);
            ptx::tma_load_3d(smem + B_OFF_Q, &p.tmQ[g], &bar_load[1], h * DH, QT, b);
            ptx::tma_load_3d(smem + B_OFF_DO, &p.tmDO[g], &bar_do[1], h * DH, QT, b);
          }
          __syncwarp();
        }
        ptx::mbar_wait(&bar_load[t], ph, p.err_flag, 23);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {      // S = Q_t K^T
#pragma unroll
          for (int k = 0; k < DH / 16; ++k) mma(tmem_base, sq + k * 32, 16, sk + k * 32, 16, idesc_s, k > 0);
          ptx::umma_commit(&bar_s[t]);
        }
        __syncwarp();
        // P ready -> dP = dO_t V^T (over S's columns) and dV += P^T dO_t
        ptx::mbar_wait(&bar_p[t], ph, p.err_flag, 24);
        ptx::mbar_wait(&bar_do[t], ph, p.err_flag, 17);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < DH / 16; ++k) mma(tmem_base, sdo + k * 32, 16, sv + k * 32, 16, idesc_s, k > 0);
          ptx::umma_commit(&bar_dp[t]);
#pragma unroll
          for (int mt = 0; mt < nmt; ++mt)
#pragma unroll
            for (int k = 0; k < QT / 16; ++k)
              mma(tmem_base + TM_DV + mt * DH, sp + 2 * mt * (QT * 128) + k * 2048, QT * 128, sdo + k * 2048, 8192,
                  idesc_kv, (t > 0 || k > 0));
        }
        __syncwarp();
        // dS ready -> dQ_t = dS K (over dP's columns) and dK += dS^T Q_t
        ptx::mbar_wait(&bar_ds[t], ph, p.err_flag, 25);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int j = 0; j < kp / 16; ++j)
            mma(tmem_base, sds + (j >> 2) * (QT * 128) + (j & 3) * 32, 16, sk + j * 2048, 8192, idesc_dq, j > 0);
          ptx::umma_commit(&bar_dq[t]);
#pragma unroll
          for (int mt = 0; mt < nmt; ++mt)
#pragma unroll
            for (int k = 0; k < QT / 16; ++k)
              mma(tmem_base + TM_DK + mt * DH, sds + 2 * mt * (QT * 128) + k * 2048, QT * 128, sq + k * 2048, 8192,
                  idesc_kv, (t > 0 || k > 0));
          ptx::umma_commit(&bar_kv[t]);
        }
        __syncwarp();
      }
      if (has_next) {
        // the next job's operands, each as soon as the chain has released its buffer (one barrier phase for all four)
        ptx::mbar_wait(&bar_dq[tl], ph, p.err_flag, 19);      // the last tile's S, dP, dV, dQ retired: K and V are dead
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&bar_load[0], LOAD0_BYTES);
          ptx::tma_load_3d(smem + B_OFF_K, &p.tmKV[g2], &bar_load[0], D + h2 * DH, 0, b2);
          ptx::tma_load_3d(smem + B_OFF_V, &p.tmKV[g2], &bar_load[0], 2 * D + h2 * DH, 0, b2);
        }
        __syncwarp();
        ptx::mbar_wait(&bar_kv[tl], ph, p.err_flag, 20);      // dK retired: Q is dead
        if (ptx::elect_one()) ptx::tma_load_3d(smem + B_OFF_Q, &p.tmQ[g2], &bar_load[0], h2 * DH, 0, b2);
        __syncwarp();
        ptx::mbar_wait(bar_done, ph, p.err_flag, 18);         // the last dQ store has read its staging tile (the dO buffer)
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&bar_do[0], Q_TILE_BYTES);
          ptx::tma_load_3d(smem + B_OFF_DO, &p.tmDO[g2], &bar_do[0], h2 * DH, 0, b2);
        }
        __syncwarp();
      }
    }
  } else {
    const int q = warp & 3;                      // TMEM lane quarter
    const int half = (warp - 1) >> 2;            // column half: 0 → keys [0,112), 1 → keys [112,208)
    const int row = q * 32 + lane;
    const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint8_t* ptile = smem + B_OFF_P;
    uint8_t* dstile = smem + B_OFF_DS;
    const uint32_t prow_s = ptx::smem_u32(ptile) + row * 128, dsrow_s = ptx::smem_u32(dstile) + row * 128;
    const int rx = row & 7;
    const int col0 = half ? 112 : 0;
    uint32_t r[32];
    long long tk[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    long long c0 = DBG ? clock64() : 0, c1;
    const long long t_begin = c0;
#define V2S_TICK(k) if (DBG) { c1 = clock64(); tk[k] += c1 - c0; c0 = c1; }
    // The O row (for D = rowsum(dO * O)) and the row's log-sum-exp come from global memory.  Their loads are issued one
    // tile ahead into registers (this warp role has 200+ registers to spare), so the DRAM latency is never on the chain.
    const int nt = VAR ? p.N : NT;
    uint4 ov[8];
    float lse_nxt = 0.f;
    auto fetch_row = [&](int n2, int t2) {
      int h2, b2, g2;
      decode(n2, h2, b2, g2);
      const int qr = t2 * QT + row;
      if (qr < nt) {
        const uint4* orow = reinterpret_cast<const uint4*>(p.ctx[g2] + ((int64_t)b2 * nt + qr) * D + h2 * DH);
#pragma unroll
        for (int c = 0; c < 8; ++c) ov[c] = __ldg(orow + c);
        lse_nxt = __ldg(p.lse[g2] + ((int64_t)b2 * NH + h2) * nt + qr);
      }
    };
    if (njobs > 0) fetch_row(0, 0);
#pragma unroll 1
    for (int n = 0; n < njobs; ++n) {
    const uint32_t ph = n & 1;
    int h, b, g;
    decode(n, h, b, g);
    for (int t = 0; t <= tl; ++t) {
      const int qrow = t * QT + row;
      const bool valid = qrow < nt;
      // padding query rows (>= 197): lse2 = +huge makes every p underflow to exactly 0, no per-element row mask needed
      const float lse2 = valid ? lse_nxt * LOG2E : 3.0e38f;
      // ---- P = exp(S/8 - lse) ----
      ptx::mbar_wait(&bar_s[t], ph, p.err_flag, 26);
      V2S_TICK(0)
      ptx::tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 3; ++c) {
        if (VAR && col0 + c * 32 >= nt) break;      // keys >= KP: read by neither dQ nor the kept rows of dK / dV
        ptx::tmem_ld_32x32(tlane + col0 + c * 32, r);
        ptx::tmem_ld_wait();
        // only keys 176..207 (second half, last chunk) contain padding keys: the bound check stays out of the other chunks
        const bool tail = (half == 1) && (c == 2);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float e[8];
          if (VAR) {
            const int kb = col0 + c * 32 + j * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              e[i] = (kb + i < nt) ? ptx::ex2_approx(fmaf(__uint_as_float(r[8 * j + i]), SCALE_LOG2E, -lse2)) : 0.f;
          } else if (!tail) {
#pragma unroll
            for (int i = 0; i < 8; ++i) e[i] = ptx::ex2_approx(fmaf(__uint_as_float(r[8 * j + i]), SCALE_LOG2E, -lse2));
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              e[i] = (176 + j * 8 + i < NT) ? ptx::ex2_approx(fmaf(__uint_as_float(r[8 * j + i]), SCALE_LOG2E, -lse2)) : 0.f;
          }
          uint4 v;
          v.x = LP::pack(e[0], e[1]); v.y = LP::pack(e[2], e[3]); v.z = LP::pack(e[4], e[5]); v.w = LP::pack(e[6], e[7]);
          store_p_chunk_s(prow_s, rx, (col0 + c * 32) / 8 + j, v);
        }
      }
      if (half == 0 && (!VAR || 96 < nt)) {      // keys 96..111
        ptx::tmem_ld_32x16(tlane + 96, r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float e[8];
#pragma unroll
          for (int i = 0; i < 8; ++i)
            e[i] = (!VAR || 96 + 8 * j + i < nt) ? ptx::ex2_approx(fmaf(__uint_as_float(r[8 * j + i]), SCALE_LOG2E, -lse2)) : 0.f;
          uint4 v;
          v.x = LP::pack(e[0], e[1]); v.y = LP::pack(e[2], e[3]); v.z = LP::pack(e[4], e[5]); v.w = LP::pack(e[6], e[7]);
          store_p_chunk_s(prow_s, rx, 12 + j, v);
        }
      }
      ptx::fence_proxy_async();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bar_p[t]);
      V2S_TICK(1)
      // D is only needed by the dS pass: computing it here puts it under the dP = dO V^T UMMAs instead of in front of
      // the P pass (the S UMMAs of a tile are long done when the threads get to it)
      ptx::mbar_wait(&bar_do[t], ph, p.err_flag, 30);
      V2S_TICK(2)
      // ---- D = rowsum(dO * O) (both halves compute it) ----
      float Dr = 0.f;
      if (valid) {
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 dv = *reinterpret_cast<const uint4*>(smem + B_OFF_DO + row * 128 + ((c ^ (row & 7)) << 4));
          const uint32_t ow[4] = {ov[c].x, ov[c].y, ov[c].z, ov[c].w}, dw[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            Dr = fmaf(LP::lo(ow[e]), LP::lo(dw[e]), Dr);
            Dr = fmaf(LP::hi(ow[e]), LP::hi(dw[e]), Dr);
          }
        }
      }
      if (t == 0 && tl != 0) fetch_row(n, 1);
      else if (n + 1 < njobs) fetch_row(n + 1, 0);
      V2S_TICK(9)
      // ---- dS = P * (dP - D) / 8 ----
      const float mDs = -Dr * SCALE;
      ptx::mbar_wait(&bar_dp[t], ph, p.err_flag, 27);
      V2S_TICK(3)
      ptx::tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 3; ++c) {
        if (VAR && col0 + c * 32 >= nt) break;
        ptx::tmem_ld_32x32(tlane + col0 + c * 32, r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c8 = (col0 + c * 32) / 8 + j;
          const uint4 pv = load_p_chunk_s(prow_s, rx, c8);
          const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
          float d[8];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            d[2 * e] = LP::lo(pw[e]) * fmaf(__uint_as_float(r[8 * j + 2 * e]), SCALE, mDs);
            d[2 * e + 1] = LP::hi(pw[e]) * fmaf(__uint_as_float(r[8 * j + 2 * e + 1]), SCALE, mDs);
          }
          uint4 v;
          v.x = LP::pack(d[0], d[1]); v.y = LP::pack(d[2], d[3]); v.z = LP::pack(d[4], d[5]); v.w = LP::pack(d[6], d[7]);
          store_p_chunk_s(dsrow_s, rx, c8, v);
        }
      }
      if (half == 0 && (!VAR || 96 < nt)) {
        ptx::tmem_ld_32x16(tlane + 96, r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint4 pv = load_p_chunk_s(prow_s, rx, 12 + j);
          const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
          float d[8];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            d[2 * e] = LP::lo(pw[e]) * fmaf(__uint_as_float(r[8 * j + 2 * e]), SCALE, mDs);
            d[2 * e + 1] = LP::hi(pw[e]) * fmaf(__uint_as_float(r[8 * j + 2 * e + 1]), SCALE, mDs);
          }
          uint4 v;
          v.x = LP::pack(d[0], d[1]); v.y = LP::pack(d[2], d[3]); v.z = LP::pack(d[4], d[5]); v.w = LP::pack(d[6], d[7]);
          store_p_chunk_s(dsrow_s, rx, 12 + j, v);
        }
      }
      ptx::fence_proxy_async();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bar_ds[t]);
      V2S_TICK(4)
      // ---- dQ_t: TMEM [0,64) → bf16 → staged in the (dead) dO buffer → TMA store ----
      ptx::mbar_wait(&bar_dq[t], ph, p.err_flag, 28);
      V2S_TICK(5)
      ptx::tc_fence_after();
      ptx::tmem_ld_32x32(tlane + half * 32, r);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      // bar_dq also covers the dV MMAs issued before dQ, so the dO tile is dead here: stage dQ in it without
      // waiting for the dK MMAs (which still read Q_t and dS)
      uint8_t* stg = smem + B_OFF_DO;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 v;
        v.x = LP::pack(__uint_as_float(r[8 * j]), __uint_as_float(r[8 * j + 1]));
        v.y = LP::pack(__uint_as_float(r[8 * j + 2]), __uint_as_float(r[8 * j + 3]));
        v.z = LP::pack(__uint_as_float(r[8 * j + 4]), __uint_as_float(r[8 * j + 5]));
        v.w = LP::pack(__uint_as_float(r[8 * j + 6]), __uint_as_float(r[8 * j + 7]));
        *reinterpret_cast<uint4*>(stg + row * 128 + (((half * 4 + j) ^ (row & 7)) << 4)) = v;
      }
      ptx::fence_proxy_async();
      ptx::bar_sync(1, 256);
      if (threadIdx.x == 32) {
        ptx::tma_store_3d(&p.tmDQKV[g], stg, h * DH, t * QT, b);
        ptx::tma_commit_group();
        ptx::tma_wait_group_read<0>();
      }
      ptx::mbar_arrive(t == 0 && tl != 0 ? bar_free : bar_done);     // (thread 32: after its store has read the staging tile)
      V2S_TICK(6)
    }
    // ---- dK, dV: TMEM → bf16 → staged in the P buffer → TMA store (rows = keys) ----
    ptx::mbar_wait(&bar_kv[tl], ph, p.err_flag, 29);      // every MMA of the job has retired
    V2S_TICK(7)
    ptx::tc_fence_after();
#pragma unroll 1
    for (int which = 0; which < 2; ++which) {          // 0: dK, 1: dV
#pragma unroll 1
      for (int mt = 0; mt < nmt; ++mt) {
        ptx::tmem_ld_32x32(tlane + (which ? TM_DV : TM_DK) + mt * DH + half * 32, r);
        ptx::tmem_ld_wait();
        uint8_t* stg = smem + B_OFF_P + (which * 2 + mt) * Q_TILE_BYTES;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 v;
          v.x = LP::pack(__uint_as_float(r[8 * j]), __uint_as_float(r[8 * j + 1]));
          v.y = LP::pack(__uint_as_float(r[8 * j + 2]), __uint_as_float(r[8 * j + 3]));
          v.z = LP::pack(__uint_as_float(r[8 * j + 4]), __uint_as_float(r[8 * j + 5]));
          v.w = LP::pack(__uint_as_float(r[8 * j + 6]), __uint_as_float(r[8 * j + 7]));
          *reinterpret_cast<uint4*>(stg + row * 128 + (((half * 4 + j) ^ (row & 7)) << 4)) = v;
        }
      }
    }
    ptx::fence_proxy_async();
    ptx::bar_sync(1, 256);
    if (threadIdx.x == 32) {
      for (int which = 0; which < 2; ++which)
        for (int mt = 0; mt < nmt; ++mt)
          ptx::tma_store_3d(&p.tmDQKV[g], smem + B_OFF_P + (which * 2 + mt) * Q_TILE_BYTES,
                            (1 + which) * D + h * DH, mt * QT, b);
      ptx::tma_commit_group();
      ptx::tma_wait_group_read<0>();
    }
    // the next job's P pass overwrites the staging tiles: nobody leaves before the stores have read them
    ptx::bar_sync(1, 256);
    V2S_TICK(8)
    }   // jobs
    if (threadIdx.x == 32) ptx::tma_wait_group<0>();
#undef V2S_TICK
    if (DBG && blockIdx.x == 0 && threadIdx.x == 32) {
      for (int k = 0; k < 9; ++k) p.dbg[16 + k] = tk[k];
      p.dbg[25] = clock64() - t_begin;
      p.dbg[26] = tk[9];
      p.dbg[27] = njobs;
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// ---- attention probabilities (ViTModel output_attentions) -------------------------------------------
// P = exp(S/8 - lse) as fp32 [B,3,197,197], recomputed from qkv and the forward's log-sum-exp: the hot forward kernel
// never materialises P in fp32.  S = Q K^T is issued exactly as attn_fwd_persist_kernel issues it (same TMA boxes, same
// UMMA 128x208x64 order), so S is bit-identical and each row sums to 1 up to fp32 rounding.  One CTA per (query tile,
// head, image, group), 160 threads: warp 0 loads and issues, warps 1..4 own one query row per thread (TMEM lane quarter
// warp & 3).  A 197-float row is 788 B, not a multiple of 16, so neither TMA nor 128-bit stores can write the output in
// place: the tile is staged densely in shared memory (over the dead Q / K tiles) and copied out with coalesced 4-byte
// stores - the tile's rows are contiguous in the output, so the copy is one linear run of up to 128 x 197 floats.
// DP = true: the same tile of dP = dO V^T, the gradient w.r.t. the probabilities (ViTModel attentions' retain_grad): A is
// the backward's d ctx tile (row stride 192, the box of tmDO in launch_attn_bwd_tc), B is V, and the epilogue is the
// identity (the 1/8 scale sits before the softmax, so dP has none).
constexpr int PR_OFF_Q = 0;
constexpr int PR_OFF_K = Q_TILE_BYTES;                        // 16384
constexpr int PR_STG_BYTES = QT * NT * 4;                     // 100864: [128][197] fp32 (odd row stride: no conflicts)
constexpr int PR_OFF_BAR = PR_STG_BYTES;                      // past both the Q / K tiles and the staging tile
constexpr int PR_SMEM = PR_OFF_BAR + 64 + 1024;
constexpr int PR_THREADS = 160;
static_assert(PR_OFF_K % 1024 == 0 && PR_OFF_K + KV_TILE_BYTES <= PR_STG_BYTES, "attention-probabilities smem map");

struct alignas(64) AttnProbsParams {
  CUtensorMap tmQ[MAXG], tmKV[MAXG];   // tmQ: the A operand, Q (probabilities) or d ctx (DP)
  const float* lse[MAXG];              // unused by DP
  float* probs[MAXG];
  int* err_flag;
  int N, ntiles;                       // VAR: tokens per image and query tiles (grid.x = 3 * ntiles)
  int KP;                              // VAR: keys padded to round_up(N, 16), the N of the S UMMA
};

// VAR: p.N tokens instead of 197 (v2s_set_image_size): a 128 x KP score tile (KP = round_up(N, 16)), output rows of stride N
template <typename LP, bool DP, bool VAR = false>
__global__ void __launch_bounds__(PR_THREADS, 2) attn_probs_tc_kernel(const __grid_constant__ AttnProbsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar_load = reinterpret_cast<uint64_t*>(smem + PR_OFF_BAR);
  uint64_t* bar_s = bar_load + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar_s + 1);
  float* stg = reinterpret_cast<float*>(smem);
  const int nt = VAR ? p.N : NT;
  const bool two_tiles = !VAR || p.ntiles == 2;
  const int t = two_tiles ? blockIdx.x & 1 : 0, h = two_tiles ? blockIdx.x >> 1 : blockIdx.x, b = blockIdx.y, g = blockIdx.z;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int nrows = nt - t * QT < QT ? nt - t * QT : QT;

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_init(bar_load, 1); ptx::mbar_init(bar_s, 1);
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(tmem_ptr, 256);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();     // after the wait: see the dependent-launch note in gemm_tc.cu

  if (warp == 0) {
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx(bar_load, Q_TILE_BYTES + KV_TILE_BYTES);
      ptx::tma_load_3d(smem + PR_OFF_Q, &p.tmQ[g], bar_load, h * DH, t * QT, b);
      ptx::tma_load_3d(smem + PR_OFF_K, &p.tmKV[g], bar_load, (DP ? 2 * D : D) + h * DH, 0, b);   // V or K
    }
    __syncwarp();
    ptx::mbar_wait(bar_load, 0, p.err_flag, 61);
    ptx::tc_fence_after();
    const uint32_t idesc_s = make_idesc_lp(LP::kIdescFmt, QT, VAR ? p.KP : KPAD, 0, 0);
    const uint32_t sq = ptx::smem_u32(smem) + PR_OFF_Q, sk = ptx::smem_u32(smem) + PR_OFF_K;
    if (ptx::elect_one()) {
#pragma unroll
      for (int k = 0; k < DH / 16; ++k) mma(tmem_base, sq + k * 32, 16, sk + k * 32, 16, idesc_s, k > 0);
      ptx::umma_commit(bar_s);
    }
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int qrow = t * QT + row;
    const bool valid = row < nrows;
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
    const float lse2 = !DP && valid ? __ldg(p.lse[g] + ((int64_t)b * NH + h) * nt + qrow) * LOG2E : 0.f;
    auto epi = [&](uint32_t v) { return DP ? __uint_as_float(v) : ptx::ex2_approx(fmaf(__uint_as_float(v), SCALE_LOG2E, -lse2)); };
    float* srow = stg + row * nt;
    uint32_t r[32];
    ptx::mbar_wait(bar_s, 0, p.err_flag, 62);     // S complete: the Q / K tiles are dead, staging may overwrite them
    ptx::tc_fence_after();
#pragma unroll 1
    for (int c = 0; c < 6; ++c) {
      if (VAR && c * 32 >= nt) break;
      ptx::tmem_ld_32x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
      if (valid) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (!VAR || c * 32 + i < nt) srow[c * 32 + i] = epi(r[i]);
      }
    }
    if (!VAR || 192 < nt) ptx::tmem_ld_32x16(taddr + 192, r);
    ptx::tmem_ld_wait();
    if (valid && (!VAR || 192 < nt)) {
#pragma unroll
      for (int i = 0; i < NT - 192; ++i)
        if (!VAR || 192 + i < nt) srow[192 + i] = epi(r[i]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  {
    float* dst = p.probs[g] + (((int64_t)b * NH + h) * nt + t * QT) * nt;
    const int n = nrows * nt;
    for (int i = threadIdx.x; i < n; i += PR_THREADS) dst[i] = stg[i];
  }
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 256);
  }
}

// launches attn_probs_tc_kernel<LP, DP, VAR> over (query tiles x 3 heads, B images, groups)
template <bool DP, bool VAR>
int launch_probs_kernel_t(const AttnProbsParams& p, int groups, int B, cudaStream_t s, int lp_f16) {
  static bool attr[MAX_DEVICES] = {false};
  if (!attr[cur_device()]) {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_probs_tc_kernel<LpBf16, DP, VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_probs_tc_kernel<LpF16, DP, VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM));
    attr[cur_device()] = true;
  }
  const dim3 grid(NH * (VAR ? p.ntiles : 2), B, groups);
  if (lp_f16) V2S_CUDA_OK(launch_pdl(attn_probs_tc_kernel<LpF16, DP, VAR>, grid, dim3(PR_THREADS), (size_t)PR_SMEM, s, p));
  else V2S_CUDA_OK(launch_pdl(attn_probs_tc_kernel<LpBf16, DP, VAR>, grid, dim3(PR_THREADS), (size_t)PR_SMEM, s, p));
  V2S_LAUNCH_CHECK();
  return 0;
}
template <bool DP>
int launch_probs_kernel(AttnProbsParams& p, int groups, int B, cudaStream_t s, int lp_f16) {
  const int nt = image_geom().nt;
  if (nt == NT) return launch_probs_kernel_t<DP, false>(p, groups, B, s, lp_f16);
  p.N = nt; p.ntiles = (nt + QT - 1) / QT; p.KP = (nt + 15) / 16 * 16;
  return launch_probs_kernel_t<DP, true>(p, groups, B, s, lp_f16);
}

}  // namespace

int launch_attn_probs_tc(const void* const* qkv, const float* const* lse, float* const* probs, int groups, int B,
                         cudaStream_t s, int lp_f16) {
  const int nt = image_geom().nt;   // tokens per image: the token dimension of the tensor maps
  AttnProbsParams p;
  memset(&p, 0, sizeof(p));
  p.err_flag = tc_err_flag();
  for (int g = 0; g < groups; ++g) {
    if (!lse[g] || !probs[g]) { set_error("attention probabilities: group %d has no lse / output", g); return 1; }
    V2S_TRY(tmap_get_3d(&p.tmQ[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, QT, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmKV[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, KPAD, true, 128));
    p.lse[g] = lse[g];
    p.probs[g] = probs[g];
  }
  return launch_probs_kernel<false>(p, groups, B, s, lp_f16);
}

int launch_attn_dprobs_tc(const void* const* qkv, const void* const* dctx, float* const* dprobs, int groups, int B,
                          cudaStream_t s, int lp_f16) {
  const int nt = image_geom().nt;   // tokens per image: the token dimension of the tensor maps
  AttnProbsParams p;
  memset(&p, 0, sizeof(p));
  p.err_flag = tc_err_flag();
  for (int g = 0; g < groups; ++g) {
    if (!dctx[g] || !dprobs[g]) { set_error("attention-probability gradient: group %d has no d ctx / output", g); return 1; }
    V2S_TRY(tmap_get_3d(&p.tmQ[g], dctx[g], D, nt, B, D * 2, (uint64_t)nt * D * 2, DH, QT, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmKV[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, KPAD, true, 128));
    p.probs[g] = dprobs[g];
  }
  return launch_probs_kernel<true>(p, groups, B, s, lp_f16);
}

int launch_attn_fwd_tc(const void* const* qkv, void* const* ctx, float* const* lse, int groups, int B,
                       cudaStream_t s, int lp_f16) {
  const int nt = image_geom().nt;   // tokens per image: the token dimension of the tensor maps
  AttnFwdPParams p;
  memset(&p, 0, sizeof(p));
  for (int g = 0; g < groups; ++g) {
    V2S_TRY(tmap_get_3d(&p.tmQ[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, QT, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmKV[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, KPAD, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmCtx[g], ctx[g], D, nt, B, D * 2, (uint64_t)nt * D * 2, DH, QT, true, 128));
    p.lse[g] = lse ? lse[g] : nullptr;
  }
  p.B = B; p.total_jobs = 2 * NH * B * groups; p.err_flag = tc_err_flag(); p.dbg = tc_dbg_counters();
  if (nt != NT) {       // the variable-length instantiation: ceil(N / 128) query tiles per (head, image)
    p.N = nt; p.ntiles = (nt + QT - 1) / QT; p.KP = (nt + 15) / 16 * 16;
    p.total_jobs = p.ntiles * NH * B * groups;
    static bool vattr[MAX_DEVICES] = {false};
    if (!vattr[cur_device()]) {
      V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_persist_kernel<false, LpBf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
      V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_persist_kernel<false, LpF16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
      vattr[cur_device()] = true;
    }
    const int grid = p.total_jobs < tc_num_sms() ? p.total_jobs : tc_num_sms();
    p.dbg = nullptr;
    if (lp_f16) V2S_CUDA_OK(launch_pdl(attn_fwd_persist_kernel<false, LpF16, true>, dim3(grid), dim3(PF_THREADS), (size_t)PF_SMEM, s, p));
    else V2S_CUDA_OK(launch_pdl(attn_fwd_persist_kernel<false, LpBf16, true>, dim3(grid), dim3(PF_THREADS), (size_t)PF_SMEM, s, p));
    V2S_LAUNCH_CHECK();
    return 0;
  }
  static bool pattr[MAX_DEVICES] = {false};
  if (!pattr[cur_device()]) {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_persist_kernel<false, LpBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_persist_kernel<true, LpBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_persist_kernel<false, LpF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_fwd_persist_kernel<true, LpF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
    pattr[cur_device()] = true;
  }
  const int num_sms = tc_num_sms();
  const int grid = p.total_jobs < num_sms ? p.total_jobs : num_sms;
  if (lp_f16) {
    if (p.dbg) V2S_CUDA_OK(launch_pdl(attn_fwd_persist_kernel<true, LpF16>, dim3(grid), dim3(PF_THREADS), (size_t)PF_SMEM, s, p));
    else V2S_CUDA_OK(launch_pdl(attn_fwd_persist_kernel<false, LpF16>, dim3(grid), dim3(PF_THREADS), (size_t)PF_SMEM, s, p));
  } else {
    if (p.dbg) V2S_CUDA_OK(launch_pdl(attn_fwd_persist_kernel<true, LpBf16>, dim3(grid), dim3(PF_THREADS), (size_t)PF_SMEM, s, p));
    else V2S_CUDA_OK(launch_pdl(attn_fwd_persist_kernel<false, LpBf16>, dim3(grid), dim3(PF_THREADS), (size_t)PF_SMEM, s, p));
  }
  V2S_LAUNCH_CHECK();
  return 0;
}

}  // namespace v2s

namespace v2s {

int launch_attn_bwd_tc(const void* const* qkv, const void* const* ctx, const float* const* lse,
                       const void* const* dctx, void* const* dqkv, int groups, int B, cudaStream_t s, int lp_f16) {
  const int nt = image_geom().nt;   // tokens per image: the token dimension of the tensor maps
  AttnBwdParams p;
  memset(&p, 0, sizeof(p));
  p.err_flag = tc_err_flag();
  for (int g = 0; g < groups; ++g) {
    V2S_TRY(tmap_get_3d(&p.tmQ[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, QT, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmKV[g], qkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, KPAD, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmDO[g], dctx[g], D, nt, B, D * 2, (uint64_t)nt * D * 2, DH, QT, true, 128));
    V2S_TRY(tmap_get_3d(&p.tmDQKV[g], dqkv[g], 3 * D, nt, B, 3 * D * 2, (uint64_t)nt * 3 * D * 2, DH, QT, true, 128));
    p.ctx[g] = static_cast<const bf16*>(ctx[g]);
    p.lse[g] = lse[g];
  }
  p.dbg = tc_dbg_counters();
  p.B = B;
  p.total_jobs = NH * B * groups;
  if (nt != NT) {       // the variable-length instantiation: ceil(N / 128) query tiles per job
    p.N = nt; p.ntiles = (nt + QT - 1) / QT; p.KP = (nt + 15) / 16 * 16;
    p.dbg = nullptr;
    static bool vattr[MAX_DEVICES] = {false};
    if (!vattr[cur_device()]) {
      V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, LpBf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
      V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, LpF16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
      vattr[cur_device()] = true;
    }
    const dim3 grid(p.total_jobs < tc_num_sms() ? p.total_jobs : tc_num_sms());
    if (lp_f16) V2S_CUDA_OK(launch_pdl(attn_bwd_tc_kernel<false, LpF16, true>, grid, dim3(B_THREADS), (size_t)B_SMEM, s, p));
    else V2S_CUDA_OK(launch_pdl(attn_bwd_tc_kernel<false, LpBf16, true>, grid, dim3(B_THREADS), (size_t)B_SMEM, s, p));
    V2S_LAUNCH_CHECK();
    return 0;
  }
  static bool attr[MAX_DEVICES] = {false};
  if (!attr[cur_device()]) {
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, LpBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_tc_kernel<true, LpBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, LpF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
    V2S_CUDA_OK(cudaFuncSetAttribute(attn_bwd_tc_kernel<true, LpF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
    attr[cur_device()] = true;
  }
  const int sms = tc_num_sms();
  const dim3 grid(p.total_jobs < sms ? p.total_jobs : sms);
  if (lp_f16) {
    if (p.dbg) V2S_CUDA_OK(launch_pdl(attn_bwd_tc_kernel<true, LpF16>, grid, dim3(B_THREADS), (size_t)B_SMEM, s, p));
    else V2S_CUDA_OK(launch_pdl(attn_bwd_tc_kernel<false, LpF16>, grid, dim3(B_THREADS), (size_t)B_SMEM, s, p));
  } else {
    if (p.dbg) V2S_CUDA_OK(launch_pdl(attn_bwd_tc_kernel<true, LpBf16>, grid, dim3(B_THREADS), (size_t)B_SMEM, s, p));
    else V2S_CUDA_OK(launch_pdl(attn_bwd_tc_kernel<false, LpBf16>, grid, dim3(B_THREADS), (size_t)B_SMEM, s, p));
  }
  V2S_LAUNCH_CHECK();
  return 0;
}

}  // namespace v2s
