// Chained tcgen05 GEMM pair for the MLP half of a ViT block: the 768-wide intermediate stays on chip.
//
//   forward  (HF:modeling_vit.py:296-312,340-346)   u = xn2 W1^T + b1;  h = gelu(u);  x_out = x_mid + b2 + h W2^T
//                                                   (+ LayerNorm of x_out = LN1 of the next block, fused)
//   backward (dgrad chain of the same two layers)   du = (dx W2) * gelu'(u);  dxn2 = du W1
//
// Persistent CTA (768 threads, one per SM) over the (backbone, 128-row m-tile) jobs.  The intermediate dimension is
// walked in twelve chunks of 64 columns; EVERY hand-over between the roles is double-buffered, so that the three
// throughput limits of the kernel (tensor pipe, the issue slots of the GELU warps, L2 -> shared-memory weight
// traffic) overlap instead of adding up:
//   stage 1   acc1 (TMEM, 128 cols) = A1[128x192] * B1 of a SUPER-chunk (two chunks)         12 UMMAs 128x128x16
//             (a UMMA costs about 75 + 0.37 N cycles here: N = 64 instructions made the kernel tensor-pipe bound.)
//             The accumulator is single-buffered but never a bottleneck: the GELU warps pull the whole super-chunk
//             into registers at once and hand the columns back within ~300 cycles.
//   GELU      16 warps (thread = one row x 16 columns of each chunk): bias+GELU or gelu'(u) product -> 16-bit -> the
//             K-major SWIZZLE_128B A operand of stage 2, one [128 x 64] k-block tile A2[c&1] in shared memory
//   stage 2   acc2[tile&1] (TMEM, 2 x 192 cols) += A2_chunk[128x64] * B2_chunk               4 UMMAs 128x192x16
//   drain     a separate warpgroup (thread = one row) empties acc2 of tile i while the other roles already work on
//             tile i+1: forward = + bias + fp32 residual -> x_out, row statistics (the row is parked in its TMEM
//             columns between the statistics pass and the normalise pass), normalised 16-bit row; backward = 16-bit
//             dxn2.  (Measured on the previous single-acc2 version of this kernel: the drain, done by the GELU
//             warps at the end of every tile, was 34 % of the tile time and left the tensor pipe idle.)
// The MMA warp issues S2(2k-1), S1(k+1), S2(2k) while the GELU warps work on super-chunk k: every wait it meets
// was satisfied well before.
//
// Global traffic of the epilogues goes through TMA only (a thread-per-row access pattern costs 32 LSU wavefronts
// per instruction).  Six 16 KB "epilogue buffers":
//   EB0/EB1  the A2 k-block tile of even / odd chunks; the same tiles are the source of the TMA stores of h
//            (forward, online backbones only) / du (backward): no separate staging
//   EB2/EB3  forward: staging of the pre-GELU activation u (stored for the backward pass of the online backbones);
//            backward: the u tiles, TMA-loaded two chunks ahead
//   EB4/EB5  the drain's ring: residual chunk in (TMA load) -> updated in place -> x_out chunk out (TMA store);
//            then the normalised / dxn2 tiles
// Roles: warp 0 TMA producer (A1 per tile, one 24 KB weight slot per chunk stage, 3-slot ring), warp 1 MMA issuer,
// warp 2 chunk stores (h, u / du; backward: also the u-tile loads), warp 3 drain stores (x_out, xn / dxn2; forward:
// also the residual loads, issued the moment the buffer's previous store has been read), warps 4..19 GELU,
// warps 20..23 drain.
#include <string.h>

#include "gemm_tc.cuh"
#include "mlp_tc.cuh"
#include "ptx.cuh"
#include "tc_math.cuh"

namespace v2s {

namespace {

constexpr int BM = 128;                    // rows per m-tile
constexpr int CW = 64;                     // chunk width along the 768-wide intermediate dimension
constexpr int NCH = DF / CW;               // 12 chunks
constexpr int KB1 = D / 64;                // 3 k-blocks in stage 1 (K = 192)
constexpr int KBLK = BM * 128;             // one [128 rows x 128 B] tile: 16384 B
constexpr int A1_BYTES = KB1 * KBLK;       // 49152
constexpr int SW = 2 * CW;                 // stage 1 runs over super-chunks of two chunks: one N = 128 UMMA series
constexpr int NSC = DF / SW;               // 6 super-chunks per tile
constexpr int W_SLOT = 24576;              // holds a stage-1 B k-block [128 x 64] (16 KB) or a stage-2 B block [192 x 64] (24 KB)
constexpr int W_SLOTS = 3;
constexpr int OFF_W = A1_BYTES;
constexpr int N_EB = 6;
constexpr int OFF_EB = OFF_W + W_SLOTS * W_SLOT;       // 122880
constexpr int OFF_BAR = OFF_EB + N_EB * KBLK;          // 221184
constexpr int SMEM_BYTES = OFF_BAR + 1024 + 1024;
constexpr int TM_ACC2 = 128;               // TMEM columns: acc1 0..127 (one super-chunk), acc2[s] at 128 + 192 s
constexpr int N_THREADS = 768;             // 24 warps (see the role list above): 80 registers per thread
constexpr int GELU_THREADS = 512;
constexpr int DRAIN_THREADS = 128;
constexpr int XCH = D / 32;                // 6 column chunks of 32 fp32 when acc2 is drained (forward)
static_assert(SMEM_BYTES <= 232448, "shared-memory budget");
static_assert(OFF_W % 1024 == 0 && OFF_EB % 1024 == 0 && W_SLOT % 1024 == 0, "swizzled tiles need 1024-byte alignment");
static_assert(NCH % 2 == 0, "per-buffer phase bookkeeping assumes an even number of chunks per tile");

struct alignas(64) MlpParams {
  CUtensorMap tmA[MAXG], tmB1[MAXG], tmB2[MAXG];
  CUtensorMap tmH[MAXG];      // [M,768] 16-bit, box 64 x 128: h (forward, optional) / du (backward)
  CUtensorMap tmU[MAXG];      // [M,768] 16-bit, box 64 x 128: u out (forward, optional) / u in (backward)
  CUtensorMap tmRes[MAXG];    // forward: x_mid fp32 [M,192], box 32 x 128
  CUtensorMap tmOut[MAXG];    // forward: x_out fp32 [M,192], box 32 x 128;  backward: dxn2 16-bit [M,192], box 64 x 128
  CUtensorMap tmXn[MAXG];     // forward, optional: normalised row 16-bit [M,192], box 64 x 128
  const float* b1[MAXG]; const float* b2[MAXG];
  const float* ln_gamma[MAXG]; const float* ln_beta[MAXG]; float* ln_mean[MAXG]; float* ln_rstd[MAXG];
  int has_h[MAXG], has_u[MAXG], has_ln[MAXG];
  int M, tiles_m, total_tiles, late_wait;
  int* err_flag;
  long long* dbg;   // optional cycle counters of CTA 0 (V2S_GEMM_DEBUG): see the end of each role
};

template <int MODE, typename LP, bool DBG>
__global__ void __launch_bounds__(N_THREADS, 1) mlp_tc_kernel(const __grid_constant__ MlpParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* a1_full = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* a1_empty = a1_full + 1;
  uint64_t* w_full = a1_empty + 1;          // [3]
  uint64_t* w_empty = w_full + W_SLOTS;     // [3]
  uint64_t* acc1_full = w_empty + W_SLOTS;  // [2] ([0] used) stage-1 UMMAs of the super-chunk retired
  uint64_t* acc1_empty = acc1_full + 2;     // [2] ([0] used) one arrival per GELU warp: the super-chunk is in registers
  uint64_t* a2_full = acc1_empty + 2;       // [2] 512 arrivals: the A2 tile of the chunk is written
  uint64_t* a2_free = a2_full + 2;          // [2] 2 arrivals: stage-2 UMMAs retired + chunk-store warp (h / du store has read it)
  uint64_t* u_full = a2_free + 2;           // [2] forward: 512 arrivals (u staged); backward: the u tile landed (TMA)
  uint64_t* u_free = u_full + 2;            // [2] forward: chunk-store warp (u store has read it); backward: 512 readers done
  uint64_t* acc2_full = u_free + 2;         // [2] all stage-2 UMMAs of the tile retired
  uint64_t* acc2_empty = acc2_full + 2;     // [2] one arrival per drain warp
  uint64_t* rs_full = acc2_empty + 2;       // [2] forward: residual chunk landed in EB4 / EB5
  uint64_t* dst_full = rs_full + 2;         // [2] 128 arrivals: the drain threads finished a chunk / tile in the buffer
  uint64_t* dbuf_free = dst_full + 2;       // [2] drain-store warp: the store has read the buffer
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(dbuf_free + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int g = 0; g * p.tiles_m < p.total_tiles; ++g) {
      ptx::prefetch_tmap(&p.tmA[g]); ptx::prefetch_tmap(&p.tmB1[g]); ptx::prefetch_tmap(&p.tmB2[g]);
    }
  }
  if (warp == 1 && lane == 0) {
    ptx::mbar_init(a1_full, 1); ptx::mbar_init(a1_empty, 1);
    for (int s = 0; s < W_SLOTS; ++s) { ptx::mbar_init(&w_full[s], 1); ptx::mbar_init(&w_empty[s], 1); }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&acc1_full[s], 1); ptx::mbar_init(&acc1_empty[s], 16);
      ptx::mbar_init(&a2_full[s], GELU_THREADS); ptx::mbar_init(&a2_free[s], 2);
      ptx::mbar_init(&u_full[s], MODE == MLP_FWD ? GELU_THREADS : 1);
      ptx::mbar_init(&u_free[s], MODE == MLP_FWD ? 1 : GELU_THREADS);
      ptx::mbar_init(&acc2_full[s], 1); ptx::mbar_init(&acc2_empty[s], 4);
      ptx::mbar_init(&rs_full[s], 1); ptx::mbar_init(&dst_full[s], DRAIN_THREADS); ptx::mbar_init(&dbuf_free[s], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_ptr, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
  if (!p.late_wait) {      // programmatic dependent launch: see the note in gemm_tc.cu
    ptx::pdl_wait();
    ptx::pdl_launch_dependents();
  }

  const int n_my = ((int)blockIdx.x < p.total_tiles) ? (p.total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  auto tile_at = [&](int i, int& g, int& mt) {
    const int t = blockIdx.x + i * gridDim.x;
    g = t / p.tiles_m;
    mt = t - g * p.tiles_m;
  };
  uint8_t* const eb = smem + OFF_EB;
  long long tk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_begin = DBG ? clock64() : 0;
#define V2S_WAIT(slot, bar, par, code)                                   \
  do {                                                                  \
    const long long _t0 = DBG ? clock64() : 0;                          \
    ptx::mbar_wait(bar, par, p.err_flag, code);                         \
    if (DBG) tk[slot] += clock64() - _t0;                               \
  } while (0)

  if (warp == 0) {
    // ================= TMA producer: A1 per tile, one weight slot per chunk stage in the MMA warp's order =========
    int ws = 0; uint32_t wph = 0;
    auto advance = [&]() { if (++ws == W_SLOTS) { ws = 0; wph ^= 1; } };
    auto load_b1 = [&](int g, int k) {          // stage-1 operand of super-chunk k: three k-block slots
#pragma unroll 1
      for (int kb = 0; kb < KB1; ++kb) {
        ptx::mbar_wait(&w_empty[ws], wph ^ 1, p.err_flag, 41);
        if (ptx::elect_one()) {
          uint8_t* slot = smem + OFF_W + ws * W_SLOT;
          ptx::mbar_arrive_expect_tx(&w_full[ws], SW * 128);
          if (MODE == MLP_FWD) {      // W1 rows [k*128, +128), k-block kb: K-major [128 x 64]
            ptx::tma_load_2d(slot, &p.tmB1[g], &w_full[ws], kb * 64, k * SW);
          } else {                    // W2 k-rows [kb*64, +64), columns [k*128, +128): MN-major, two [64 x 64] boxes
            ptx::tma_load_2d(slot, &p.tmB1[g], &w_full[ws], k * SW, kb * 64);
            ptx::tma_load_2d(slot + 8192, &p.tmB1[g], &w_full[ws], k * SW + 64, kb * 64);
          }
        }
        __syncwarp();
        advance();
      }
    };
    auto load_b2 = [&](int g, int j) {          // stage-2 operand of chunk j: one slot
      ptx::mbar_wait(&w_empty[ws], wph ^ 1, p.err_flag, 42);
      if (ptx::elect_one()) {
        uint8_t* slot = smem + OFF_W + ws * W_SLOT;
        ptx::mbar_arrive_expect_tx(&w_full[ws], W_SLOT);
        if (MODE == MLP_FWD) {      // W2 all 192 rows, k columns [j*64, +64): K-major [192 x 64]
          ptx::tma_load_2d(slot, &p.tmB2[g], &w_full[ws], j * CW, 0);
        } else {                    // W1 k-rows [j*64, +64), all 192 columns: MN-major, three [64 x 64] boxes
          ptx::tma_load_2d(slot, &p.tmB2[g], &w_full[ws], 0, j * CW);
          ptx::tma_load_2d(slot + 8192, &p.tmB2[g], &w_full[ws], 64, j * CW);
          ptx::tma_load_2d(slot + 16384, &p.tmB2[g], &w_full[ws], 128, j * CW);
        }
      }
      __syncwarp();
      advance();
    };
    auto load_a1 = [&](int i) {
      int g, mt;
      tile_at(i, g, mt);
      ptx::mbar_wait(a1_empty, (i & 1) ^ 1, p.err_flag, 43);
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(a1_full, A1_BYTES);
#pragma unroll
        for (int kb = 0; kb < KB1; ++kb) ptx::tma_load_2d(smem + kb * KBLK, &p.tmA[g], a1_full, kb * 64, mt * BM);
      }
      __syncwarp();
    };
    // the MMA warp's order over the global super-chunk index K (tile K / 6, super-chunk K % 6):
    //   S1(0);  for K: [S2(2K-1)]  [S1(K+1)]  S2(2K);  S2(last)
    const int n_sc = n_my * NSC;
    auto grp = [&](int K) { int g, mt; tile_at(K / NSC, g, mt); return g; };
    if (n_sc > 0) { load_a1(0); load_b1(grp(0), 0); }
#pragma unroll 1
    for (int K = 0; K < n_sc; ++K) {
      if (K >= 1) load_b2(grp(K - 1), 2 * ((K - 1) % NSC) + 1);
      if (K + 1 < n_sc) {
        if ((K + 1) % NSC == 0) load_a1((K + 1) / NSC);
        load_b1(grp(K + 1), (K + 1) % NSC);
      }
      load_b2(grp(K), 2 * (K % NSC));
    }
    if (n_sc > 0) load_b2(grp(n_sc - 1), 2 * ((n_sc - 1) % NSC) + 1);
  } else if (warp == 1) {
    // ================= MMA issuer: S1(c), then S2(c-2) =================
    constexpr uint32_t b_mn = (MODE == MLP_BWD) ? 1u : 0u;
    const uint32_t idesc2 = make_idesc_lp(LP::kIdescFmt, BM, D, 0, b_mn);
    const uint32_t sbase = ptx::smem_u32(smem);
    const uint32_t b_lbo = b_mn ? 8192u : 16u, b_step = b_mn ? (2048u >> 4) : (32u >> 4);
    int ws = 0; uint32_t wph = 0;
    auto advance = [&]() { if (++ws == W_SLOTS) { ws = 0; wph ^= 1; } };
    const uint32_t idesc1 = make_idesc_lp(LP::kIdescFmt, BM, SW, 0, b_mn);
    auto stage1 = [&](int K) {                  // super-chunk K (global index)
      const int i = K / NSC, k = K - i * NSC;
      V2S_WAIT(0, acc1_empty, (K & 1) ^ 1, 44);
      if (k == 0) V2S_WAIT(1, a1_full, i & 1, 45);
#pragma unroll 1
      for (int kb = 0; kb < KB1; ++kb) {
        V2S_WAIT(2, &w_full[ws], wph, 46);
        ptx::tc_fence_after();
        const uint32_t a_lo = ptx::desc_lo(sbase + kb * KBLK, 16);
        const uint32_t b_lo = ptx::desc_lo(sbase + OFF_W + ws * W_SLOT, b_lbo);
        if (ptx::elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            ptx::umma_bf16_lohi(tmem_base, a_lo + kk * 2, b_lo + kk * b_step, ptx::DESC_HI_SW128_SBO1024, idesc1,
                                (kb > 0 || kk > 0) ? 1u : 0u);
          ptx::umma_commit(&w_empty[ws]);
          if (kb == KB1 - 1) {
            ptx::umma_commit(acc1_full);
            if (k == NSC - 1) ptx::umma_commit(a1_empty);      // the tile's A1 is dead once these retire
          }
        }
        __syncwarp();
        advance();
      }
    };
    auto stage2 = [&](int c) {                  // chunk c (global index)
      const int i = c / NCH, j = c - i * NCH;
      const int s = i & 1, b = c & 1;
      if (j == 0) V2S_WAIT(3, &acc2_empty[s], ((i >> 1) & 1) ^ 1, 47);
      V2S_WAIT(4, &a2_full[b], (c >> 1) & 1, 48);
      V2S_WAIT(5, &w_full[ws], wph, 49);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + TM_ACC2 + s * D;
      const uint32_t a_lo = ptx::desc_lo(sbase + OFF_EB + b * KBLK, 16);
      const uint32_t b_lo = ptx::desc_lo(sbase + OFF_W + ws * W_SLOT, b_lbo);
      if (ptx::elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          ptx::umma_bf16_lohi(d_tmem, a_lo + kk * 2, b_lo + kk * b_step, ptx::DESC_HI_SW128_SBO1024, idesc2,
                              (j > 0 || kk > 0) ? 1u : 0u);
        ptx::umma_commit(&w_empty[ws]);
        ptx::umma_commit(&a2_free[b]);
        if (j == NCH - 1) ptx::umma_commit(&acc2_full[s]);
      }
      __syncwarp();
      advance();
    };
    const int n_sc = n_my * NSC;
    if (n_sc > 0) stage1(0);
#pragma unroll 1
    for (int K = 0; K < n_sc; ++K) {
      if (K >= 1) stage2(2 * K - 1);
      if (K + 1 < n_sc) stage1(K + 1);
      stage2(2 * K);
    }
    if (n_sc > 0) stage2(2 * n_sc - 1);
    if (DBG && blockIdx.x == 0 && lane == 0) {
      for (int k = 0; k < 6; ++k) p.dbg[k] = tk[k];
      p.dbg[6] = clock64() - t_begin; p.dbg[7] = n_my;
    }
  } else if (warp == 2) {
    // ================= chunk-store warp: h / u (forward, online backbones), du (backward) =================
    // (lane 0 issues: bulk async-groups are per thread).  One store group per chunk; a chunk's buffers are handed
    // back while the next chunk's group is in flight.
    int c = 0, nut = 0;
    const int n_chunks = n_my * NCH;
    auto load_u = [&](int cc) {       // backward: u tile of chunk cc into EB2 / EB3 (lane 0)
      const int ti = cc / NCH, jj = cc - ti * NCH;
      int g2, mt2;
      tile_at(ti, g2, mt2);
      ptx::mbar_arrive_expect_tx(&u_full[cc & 1], KBLK);
      ptx::tma_load_2d(eb + (2 + (cc & 1)) * KBLK, &p.tmU[g2], &u_full[cc & 1], jj * CW, mt2 * BM);
    };
    if (MODE == MLP_BWD && lane == 0) {
      if (n_chunks > 0) load_u(0);
      if (n_chunks > 1) load_u(1);
    }
    __syncwarp();
    for (int i = 0; i < n_my; ++i) {
      int g, mt;
      tile_at(i, g, mt);
      const int m0 = mt * BM;
      const bool has_h = p.has_h[g] != 0, has_u = MODE == MLP_FWD && p.has_u[g] != 0;
      const bool stores = has_h || has_u;
#pragma unroll 1
      for (int j = 0; j < NCH; ++j, ++c) {
        const int b = c & 1;
        if (MODE == MLP_BWD && c + 2 < n_chunks) {
          // the readers of chunk c have its u in registers (start of their chunk): fetch the u of chunk c + 2
          ptx::mbar_wait(&u_free[b], (c >> 1) & 1, p.err_flag, 53);
          if (lane == 0) load_u(c + 2);
          __syncwarp();
        }
        ptx::mbar_wait(&a2_full[b], (c >> 1) & 1, p.err_flag, 54);
        if (has_u) ptx::mbar_wait(&u_full[b], (nut * (NCH / 2) + (j >> 1)) & 1, p.err_flag, 55);
        if (lane == 0) {
          if (stores) {
            if (has_h) ptx::tma_store_2d(&p.tmH[g], eb + b * KBLK, j * CW, m0);
            if (has_u) ptx::tma_store_2d(&p.tmU[g], eb + (2 + b) * KBLK, j * CW, m0);
            ptx::tma_commit_group();
            if (j > 0) {                          // the previous chunk's stores have read their buffers
              ptx::tma_wait_group_read<1>();
              ptx::mbar_arrive(&a2_free[b ^ 1]);
              if (has_u) ptx::mbar_arrive(&u_free[b ^ 1]);
            }
            if (j == NCH - 1) {
              ptx::tma_wait_group_read<0>();
              ptx::mbar_arrive(&a2_free[b]);
              if (has_u) ptx::mbar_arrive(&u_free[b]);
            }
          } else {
            ptx::mbar_arrive(&a2_free[b]);
          }
        }
        __syncwarp();
      }
      if (has_u) ++nut;
    }
    if (lane == 0) ptx::tma_wait_group<0>();
    __syncwarp();
  } else if (warp == 3) {
    // ================= drain-store warp: x_out chunks and normalised tiles (forward), dxn2 tiles (backward) =======
    // forward: the residual chunk that uses a buffer next is fetched right here, the moment the buffer's previous
    // store has been read: chunks 0, 1 of a tile are in place long before its accumulator is complete.
    int use0 = 0, use1 = 0;
    auto load_res = [&](int ti, int k) {      // lane 0
      int g2, mt2;
      tile_at(ti, g2, mt2);
      ptx::mbar_arrive_expect_tx(&rs_full[k & 1], KBLK);
      ptx::tma_load_2d(eb + (4 + (k & 1)) * KBLK, &p.tmRes[g2], &rs_full[k & 1], k * 32, mt2 * BM);
    };
    if (MODE == MLP_FWD && n_my > 0 && lane == 0) { load_res(0, 0); load_res(0, 1); }
    __syncwarp();
    for (int i = 0; i < n_my; ++i) {
      int g, mt;
      tile_at(i, g, mt);
      const int m0 = mt * BM;
      const int n_out = MODE == MLP_FWD ? XCH : 0;
      const int n_lp = MODE == MLP_FWD ? (p.has_ln[g] != 0 ? 3 : 0) : 3;
      const int n_all = n_out + n_lp;
#pragma unroll 1
      for (int k = 0; k < n_all; ++k) {
        const int t = k - n_out;                    // >= 0: 16-bit tile t
        const int b = (k < n_out ? k : t) & 1;
        ptx::mbar_wait(&dst_full[b], (b ? use1 : use0) & 1, p.err_flag, 57);
        if (lane == 0) {
          if (k < n_out) ptx::tma_store_2d(&p.tmOut[g], eb + (4 + b) * KBLK, k * 32, m0);
          else ptx::tma_store_2d(MODE == MLP_FWD ? &p.tmXn[g] : &p.tmOut[g], eb + (4 + b) * KBLK, t * 64, m0);
          ptx::tma_commit_group();
          ptx::tma_wait_group_read<0>();
          ptx::mbar_arrive(&dbuf_free[b]);
          if (MODE == MLP_FWD) {
            // next use of buffer b: residual chunk k + 2 of this tile, or chunk b of the next tile when this was the
            // buffer's last use in the tile (uses of a tile: b0 = chunks 0 2 4 [tiles 0 2], b1 = chunks 1 3 5 [tile 1])
            if (k + 2 < n_out) load_res(i, k + 2);
            else if (i + 1 < n_my) {
              const bool last_use = n_lp == 0 ? true : (b == 0 ? t == 2 : t == 1);
              if (last_use) load_res(i + 1, b);
            }
          }
        }
        __syncwarp();
        use0 += b ^ 1; use1 += b;
      }
    }
    if (lane == 0) ptx::tma_wait_group<0>();
    __syncwarp();
  } else if (warp >= 4 && warp < 20) {
    // ================= GELU warps =================
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int cq = (warp - 4) >> 2;              // column quarter: 16 of the chunk's 64 columns
    const int row = q * 32 + lane;
    const int rx = row & 7;
    const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t eb_row = ptx::smem_u32(eb) + row * 128;      // this thread's row in EB0
    const uint32_t pc0 = ((2 * cq) ^ rx) << 4, pc1 = ((2 * cq + 1) ^ rx) << 4;   // its two 16-byte pieces of a tile row
    int c = 0, nut = 0;
    uint32_t rr[32];
    for (int i = 0; i < n_my; ++i) {
      int g, mt;
      tile_at(i, g, mt);
      const bool has_u = MODE == MLP_FWD && p.has_u[g] != 0;
#pragma unroll 1
      for (int j = 0; j < NCH; ++j, ++c) {
        const int b = c & 1;
        uint4 ux0, ux1;
        if (MODE == MLP_BWD) {                                  // pre-GELU activation of the forward pass
          V2S_WAIT(0, &u_full[b], (c >> 1) & 1, 61);
          ux0 = ptx::lds128(eb_row + (2 + b) * KBLK + pc0);
          ux1 = ptx::lds128(eb_row + (2 + b) * KBLK + pc1);
          // The tile is handed back to the TMA engine (the u of chunk c + 2): the loads above must have READ shared
          // memory before the arrival is visible.  Nothing below depends on their data yet, and the hardware lets the
          // barrier arrival overtake loads that are merely issued, so wait for them explicitly.
          __threadfence_block();
          ptx::mbar_arrive(&u_free[b]);
        }
        if (b == 0) {          // a new super-chunk: both halves into registers, the accumulator back to the MMA warp
          V2S_WAIT(1, acc1_full, (c >> 1) & 1, 50);
          ptx::tc_fence_after();
          ptx::tmem_ld_32x16(tl + cq * 16, rr);
          ptx::tmem_ld_32x16(tl + CW + cq * 16, rr + 16);
          ptx::tmem_ld_wait();
          ptx::tc_fence_before();
          if (lane == 0) ptx::mbar_arrive(acc1_empty);
        }
        uint32_t r[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) r[e] = b ? rr[16 + e] : rr[e];
        uint32_t o[8], pu[8];
        if (MODE == MLP_FWD) {
          const float4* b4 = reinterpret_cast<const float4*>(p.b1[g] + j * CW + cq * 16);
          float v[16];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float4 bb = __ldg(b4 + t);
            v[4 * t] = __uint_as_float(r[4 * t]) + bb.x; v[4 * t + 1] = __uint_as_float(r[4 * t + 1]) + bb.y;
            v[4 * t + 2] = __uint_as_float(r[4 * t + 2]) + bb.z; v[4 * t + 3] = __uint_as_float(r[4 * t + 3]) + bb.w;
          }
          if (has_u) {
#pragma unroll
            for (int k = 0; k < 8; ++k) pu[k] = LP::pack(v[2 * k], v[2 * k + 1]);
          }
#pragma unroll
          for (int k = 0; k < 8; ++k) o[k] = LP::pack(gelu_fast(v[2 * k]), gelu_fast(v[2 * k + 1]));
        } else {
          const uint32_t w[8] = {ux0.x, ux0.y, ux0.z, ux0.w, ux1.x, ux1.y, ux1.z, ux1.w};
#pragma unroll
          for (int e = 0; e < 8; ++e)
            o[e] = LP::pack(__uint_as_float(r[2 * e]) * gelu_grad_fast(LP::lo(w[e])),
                            __uint_as_float(r[2 * e + 1]) * gelu_grad_fast(LP::hi(w[e])));
        }
        // A operand of stage 2: the chunk's k-block tile, 16-byte pieces 2 cq, 2 cq + 1 of this row
        V2S_WAIT(2, &a2_free[b], ((c >> 1) & 1) ^ 1, 51);
        ptx::sts128(eb_row + b * KBLK + pc0, o[0], o[1], o[2], o[3]);
        ptx::sts128(eb_row + b * KBLK + pc1, o[4], o[5], o[6], o[7]);
        if (has_u) {      // one proxy fence for both tiles (the fence is the expensive part)
          V2S_WAIT(3, &u_free[b], ((nut * (NCH / 2) + (j >> 1)) & 1) ^ 1, 62);
          ptx::sts128(eb_row + (2 + b) * KBLK + pc0, pu[0], pu[1], pu[2], pu[3]);
          ptx::sts128(eb_row + (2 + b) * KBLK + pc1, pu[4], pu[5], pu[6], pu[7]);
          ptx::fence_proxy_async();
          ptx::mbar_arrive(&a2_full[b]);
          ptx::mbar_arrive(&u_full[b]);
        } else {
          ptx::fence_proxy_async();
          ptx::mbar_arrive(&a2_full[b]);
        }
      }
      if (has_u) ++nut;
    }
    if (DBG && blockIdx.x == 0 && threadIdx.x == 128) {
      for (int k = 0; k < 4; ++k) p.dbg[8 + k] = tk[k];
      p.dbg[12] = clock64() - t_begin;
    }
  } else if (warp >= 20 && warp < 24) {
    // ================= drain warps: thread = one row of the tile =================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int rx = row & 7;
    const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + TM_ACC2;
    const uint32_t eb_row = ptx::smem_u32(eb) + 4 * KBLK + row * 128;      // this thread's row in EB4
    int use0 = 0, use1 = 0, nres0 = 0, nres1 = 0;
    for (int i = 0; i < n_my; ++i) {
      int g, mt;
      tile_at(i, g, mt);
      const int s = i & 1;
      const int64_t grow = (int64_t)mt * BM + row;
      const uint32_t ta = tl + s * D;
      V2S_WAIT(4, &acc2_full[s], (i >> 1) & 1, 52);
      const long long t_d0 = DBG ? clock64() : 0;
      ptx::tc_fence_after();
      if (MODE == MLP_FWD) {
        const bool has_ln = p.has_ln[g] != 0;
        float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
        for (int k = 0; k < XCH; ++k) {
          const int b = k & 1;
          uint32_t r[32];
          ptx::tmem_ld_32x32(ta + k * 32, r);
          const float4* b4 = reinterpret_cast<const float4*>(p.b2[g] + k * 32);
          V2S_WAIT(5, &rs_full[b], (b ? nres1 : nres0) & 1, 63);
          nres0 += b ^ 1; nres1 += b;
          ptx::tmem_ld_wait();
          const uint32_t sb = eb_row + b * KBLK;
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const float4 bb = __ldg(b4 + t);
            const uint32_t sa = sb + ((t ^ rx) << 4);
            const float4 xr = ptx::lds128f(sa);
            const float x0 = __uint_as_float(r[4 * t]) + bb.x + xr.x, x1 = __uint_as_float(r[4 * t + 1]) + bb.y + xr.y;
            const float x2 = __uint_as_float(r[4 * t + 2]) + bb.z + xr.z, x3 = __uint_as_float(r[4 * t + 3]) + bb.w + xr.w;
            ptx::sts128f(sa, x0, x1, x2, x3);
            s1 += (x0 + x1) + (x2 + x3);
            s2 = fmaf(x0, x0, s2); s2 = fmaf(x1, x1, s2); s2 = fmaf(x2, x2, s2); s2 = fmaf(x3, x3, s2);
            r[4 * t] = __float_as_uint(x0); r[4 * t + 1] = __float_as_uint(x1);
            r[4 * t + 2] = __float_as_uint(x2); r[4 * t + 3] = __float_as_uint(x3);
          }
          ptx::fence_proxy_async();
          ptx::mbar_arrive(&dst_full[b]);
          use0 += b ^ 1; use1 += b;
          if (has_ln) ptx::tmem_st_32x32(ta + k * 32, r);       // park the finished row chunk for the normalise pass
        }
        if (has_ln) {
          const float mean = s1 * (1.0f / D);
          const float var = fmaxf(s2 * (1.0f / D) - mean * mean, 0.f);
          const float rstd = 1.0f / sqrtf(var + LN_EPS);
          if (grow < p.M && p.ln_mean[g] != nullptr) { p.ln_mean[g][grow] = mean; p.ln_rstd[g][grow] = rstd; }
          ptx::tmem_st_wait();
#pragma unroll 1
          for (int t = 0; t < 3; ++t) {
            const int b = t & 1;
            const uint32_t sb = eb_row + b * KBLK;
#pragma unroll 1
            for (int hf = 0; hf < 2; ++hf) {
              uint32_t r[32];
              ptx::tmem_ld_32x32(ta + t * 64 + hf * 32, r);
              const float4* g4 = reinterpret_cast<const float4*>(p.ln_gamma[g] + t * 64 + hf * 32);
              const float4* e4 = reinterpret_cast<const float4*>(p.ln_beta[g] + t * 64 + hf * 32);
              if (hf == 0) V2S_WAIT(6, &dbuf_free[b], ((b ? use1 : use0) & 1) ^ 1, 64);     // the buffer's previous store has read it
              ptx::tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float4 ga = __ldg(g4 + 2 * e), gb = __ldg(g4 + 2 * e + 1);
                const float4 ea = __ldg(e4 + 2 * e), eb4 = __ldg(e4 + 2 * e + 1);
                const uint32_t* x = r + 8 * e;
                const uint32_t w0 = LP::pack((__uint_as_float(x[0]) - mean) * rstd * ga.x + ea.x, (__uint_as_float(x[1]) - mean) * rstd * ga.y + ea.y);
                const uint32_t w1 = LP::pack((__uint_as_float(x[2]) - mean) * rstd * ga.z + ea.z, (__uint_as_float(x[3]) - mean) * rstd * ga.w + ea.w);
                const uint32_t w2 = LP::pack((__uint_as_float(x[4]) - mean) * rstd * gb.x + eb4.x, (__uint_as_float(x[5]) - mean) * rstd * gb.y + eb4.y);
                const uint32_t w3 = LP::pack((__uint_as_float(x[6]) - mean) * rstd * gb.z + eb4.z, (__uint_as_float(x[7]) - mean) * rstd * gb.w + eb4.w);
                ptx::sts128(sb + (((hf * 4 + e) ^ rx) << 4), w0, w1, w2, w3);
              }
            }
            ptx::fence_proxy_async();
            ptx::mbar_arrive(&dst_full[b]);
            use0 += b ^ 1; use1 += b;
          }
        }
      } else {
#pragma unroll 1
        for (int t = 0; t < 3; ++t) {
          const int b = t & 1;
          const uint32_t sb = eb_row + b * KBLK;
#pragma unroll 1
          for (int hf = 0; hf < 2; ++hf) {
            uint32_t r[32];
            ptx::tmem_ld_32x32(ta + t * 64 + hf * 32, r);
            if (hf == 0) V2S_WAIT(6, &dbuf_free[b], ((b ? use1 : use0) & 1) ^ 1, 65);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const uint32_t* x = r + 8 * e;
              ptx::sts128(sb + (((hf * 4 + e) ^ rx) << 4), LP::pack(__uint_as_float(x[0]), __uint_as_float(x[1])),
                          LP::pack(__uint_as_float(x[2]), __uint_as_float(x[3])), LP::pack(__uint_as_float(x[4]), __uint_as_float(x[5])),
                          LP::pack(__uint_as_float(x[6]), __uint_as_float(x[7])));
            }
          }
          ptx::fence_proxy_async();
          ptx::mbar_arrive(&dst_full[b]);
          use0 += b ^ 1; use1 += b;
        }
      }
      // every tcgen05.ld of this tile's accumulator has completed (wait::ld above): hand it back to the MMA warp
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc2_empty[s]);
      if (DBG) tk[7] += clock64() - t_d0;
    }
    if (DBG && blockIdx.x == 0 && threadIdx.x == 640) {
      p.dbg[13] = tk[4]; p.dbg[14] = tk[5]; p.dbg[15] = tk[6]; p.dbg[16] = tk[7];
      p.dbg[17] = clock64() - t_begin;
    }
  }
#undef V2S_WAIT

  if (p.late_wait) { ptx::pdl_wait(); ptx::pdl_launch_dependents(); }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

template <int MODE, typename LP>
int launch_impl(const MlpParams& p, int grid, cudaStream_t stream) {
  static bool attr_set[MAX_DEVICES] = {false};
  if (!attr_set[cur_device()]) {
    V2S_CUDA_OK(cudaFuncSetAttribute(mlp_tc_kernel<MODE, LP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    V2S_CUDA_OK(cudaFuncSetAttribute(mlp_tc_kernel<MODE, LP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_set[cur_device()] = true;
  }
  if (p.dbg) V2S_CUDA_OK(launch_pdl(mlp_tc_kernel<MODE, LP, true>, dim3(grid), dim3(N_THREADS), (size_t)SMEM_BYTES, stream, p));
  else V2S_CUDA_OK(launch_pdl(mlp_tc_kernel<MODE, LP, false>, dim3(grid), dim3(N_THREADS), (size_t)SMEM_BYTES, stream, p));
  V2S_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int launch_mlp_tc(const MlpDesc& d, cudaStream_t stream) {
  if (d.groups < 1 || d.groups > MAXG || d.M < 1) { set_error("mlp_tc: bad shape"); return 1; }
  MlpParams p;
  memset(&p, 0, sizeof(p));
  p.M = d.M;
  p.tiles_m = (d.M + BM - 1) / BM;
  p.total_tiles = p.tiles_m * d.groups;
  p.late_wait = d.late_wait ? 1 : 0;
  p.err_flag = tc_err_flag();
  p.dbg = tc_dbg_counters();
  for (int g = 0; g < d.groups; ++g) {
    if (!d.a[g] || !d.w1[g] || !d.w2[g] || !d.out[g]) { set_error("mlp_tc: null operand (group %d)", g); return 1; }
    V2S_TRY(tmap_get_2d(&p.tmA[g], d.a[g], D, d.M, D, 64, BM, true, 128));
    if (d.mode == MLP_FWD) {
      if (!d.b1[g] || !d.b2[g] || !d.resid[g]) { set_error("mlp_tc: forward needs biases and the residual"); return 1; }
      V2S_TRY(tmap_get_2d(&p.tmB1[g], d.w1[g], D, DF, D, 64, SW, true, 128));       // W1 [768,192]: rows x k
      V2S_TRY(tmap_get_2d(&p.tmB2[g], d.w2[g], DF, D, DF, 64, D, true, 128));       // W2 [192,768]: rows x k
      V2S_TRY(tmap_get_2d(&p.tmRes[g], d.resid[g], D, d.M, D, 32, BM, false, 128));
      V2S_TRY(tmap_get_2d(&p.tmOut[g], d.out[g], D, d.M, D, 32, BM, false, 128));
      if (d.h[g]) { V2S_TRY(tmap_get_2d(&p.tmH[g], d.h[g], DF, d.M, DF, 64, BM, true, 128)); p.has_h[g] = 1; }
      if (d.u[g]) { V2S_TRY(tmap_get_2d(&p.tmU[g], d.u[g], DF, d.M, DF, 64, BM, true, 128)); p.has_u[g] = 1; }
      if (d.ln_out[g]) {
        if (!d.ln_gamma[g] || !d.ln_beta[g]) { set_error("mlp_tc: fused LayerNorm needs gamma and beta"); return 1; }
        V2S_TRY(tmap_get_2d(&p.tmXn[g], d.ln_out[g], D, d.M, D, 64, BM, true, 128));
        p.has_ln[g] = 1;
      }
    } else {
      if (!d.u[g] || !d.h[g]) { set_error("mlp_tc: backward needs u and the du buffer"); return 1; }
      V2S_TRY(tmap_get_2d(&p.tmB1[g], d.w2[g], DF, D, DF, 64, 64, true, 128));      // W2 [192(k),768(n)]
      V2S_TRY(tmap_get_2d(&p.tmB2[g], d.w1[g], D, DF, D, 64, 64, true, 128));       // W1 [768(k),192(n)]
      V2S_TRY(tmap_get_2d(&p.tmH[g], d.h[g], DF, d.M, DF, 64, BM, true, 128));
      V2S_TRY(tmap_get_2d(&p.tmU[g], d.u[g], DF, d.M, DF, 64, BM, true, 128));
      V2S_TRY(tmap_get_2d(&p.tmOut[g], d.out[g], D, d.M, D, 64, BM, true, 128));
      p.has_h[g] = 1; p.has_u[g] = 1;
    }
    p.b1[g] = d.b1[g]; p.b2[g] = d.b2[g];
    p.ln_gamma[g] = d.ln_gamma[g]; p.ln_beta[g] = d.ln_beta[g]; p.ln_mean[g] = d.ln_mean[g]; p.ln_rstd[g] = d.ln_rstd[g];
  }
  const int sms = tc_num_sms();
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  if (d.mode == MLP_FWD)
    return d.lp_f16 ? launch_impl<MLP_FWD, LpF16>(p, grid, stream) : launch_impl<MLP_FWD, LpBf16>(p, grid, stream);
  return d.lp_f16 ? launch_impl<MLP_BWD, LpF16>(p, grid, stream) : launch_impl<MLP_BWD, LpBf16>(p, grid, stream);
}

}  // namespace v2s
