// tcgen05 / TMEM / TMA GEMM for sm_100a: persistent, warp-specialised, grouped (up to 4 backbones per
// launch), bf16 operands with fp32 accumulation in tensor memory, fused epilogues staged through shared
// memory and written with TMA (plain store or reduce-add).
//
//   C[M,N] (+)= A[M,K] * B[N,K]^T        A, B: K-major or MN-major (UMMA descriptor major bits)
//
// CTA = 640 threads, one CTA per SM, tile 128 x 192 x 64:
//   warp 0      TMA producer: operand ring in smem (depth chosen per variant from the 227 KB budget;
//               "B-stationary" when K <= 192: the [192 x K] weight tile is loaded once per CTA)
//   warp 1      MMA issuer: tcgen05.mma.cta_group::1.kind::f16 128x192x16, accumulators double-buffered in
//               TMEM (2 x 192 of 512 columns) so the epilogue of tile i overlaps the MMAs of tile i+1;
//               wgrad adds an N=16 MMA against a constant ones tile: bias gradient in columns [192,208)
//   warps 2,3   store warps of the two epilogue groups: own every TMA store / reduce-add and the prefetch of the
//               auxiliary operand (the residual) into the staging ring (warp 2 also owns TMEM)
//   warps 4-19  epilogue: two groups of eight warps; group g drains accumulator stage g (the CTA's even / odd
//               tiles).  Warps w, w+4 of a group read TMEM lane quarter w%4 (tcgen05.ld 32x32b) and take the
//               two 16-column halves of each 32-column chunk: thread = one row x 16 columns.  Epilogues: bias,
//               bias + residual (fp32 stream, updated in place in the staging buffer) with optional fused
//               LayerNorm (row parked in TMEM, second pass writes the normalised bf16 row), fp32 reduce-add
//               (split-K wgrad).
// Staging ring protocol: see the epilogue.  Every mbarrier wait is bounded (ptx::mbar_wait).
#include <string.h>

#include <unordered_map>

#include "gemm_tc.cuh"
#include "ptx.cuh"
#include "tc_math.cuh"

namespace v2s {

namespace {

constexpr int BM = 128, BN = 192, BK = 64;
constexpr int MAX_STAGES = 6;                     // smem ring depth is chosen per variant on the host
constexpr int A_STAGE_BYTES = BM * BK * 2;        // 16384
constexpr int B_STAGE_BYTES = BN * BK * 2;        // 24576
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int CHUNK = 32;                         // epilogue column chunk
constexpr int N_CHUNKS = BN / CHUNK;              // 6
constexpr int SMEM_LIMIT = 232448;                // 227 KB opt-in maximum per CTA
constexpr int SMEM_BAR_BYTES = 8192;             // mbarriers (1 KB) + 2 KB ones tile (row-sum MMA) + 4 KB LayerNorm partial sums
constexpr int TMEM_COLS = 512;
constexpr int ACC_STRIDE = 256;                   // TMEM column stride between accumulator stages
constexpr int N_THREADS = 640;                    // 4 control/idle warps + 16 epilogue warps

enum TcEpi : int {
  T_STORE = 0,   // out = acc (+bias)            OutT = bf16 | fp32
  T_RESID = 1,   // out(fp32) = acc + bias + aux(fp32)
  T_ACCUM = 4,   // global(fp32) += acc          (TMA reduce-add; split-K)
  T_ACCUM_DET = 5,   // deterministic T_ACCUM: partial tiles to a slab, summed in split order by the last CTA to arrive
};

// per-variant epilogue staging: a ring of NSTG buffers of STG bytes per epilogue group.  The residual variant
// (auxiliary operand prefetched two chunks ahead into the ring) and the plain bf16 store use 3 buffers;
// bf16 chunks are 8 KB (SWIZZLE_64B), fp32 chunks 16 KB.
template <int EPI, bool OUT_BF16> struct Cfg {
  static constexpr int NSTG = (EPI == T_ACCUM || EPI == T_ACCUM_DET || (EPI == T_STORE && !OUT_BF16)) ? 2 : 3;
  static constexpr int STG = OUT_BF16 ? 8192 : 16384;
  static constexpr int STAGING_BYTES = 2 * NSTG * STG;
};

struct alignas(64) TcParams {
  CUtensorMap tmA[MAXG], tmB[MAXG], tmOut[MAXG], tmOut2[MAXG], tmAux[MAXG];
  const float* bias[MAXG];
  // T_RESID with fused LayerNorm (ln != 0, N == 192): xn = LN(out) * gamma + beta -> tmOut2 (bf16), stats -> ln_mean/rstd
  const float* ln_gamma[MAXG]; const float* ln_beta[MAXG]; float* ln_mean[MAXG]; float* ln_rstd[MAXG];
  int ln;
  float* rowsum[MAXG];  // T_ACCUM: rowsum[m] += sum_k A(m,k), computed by an extra N=16 MMA against a ones tile
  int M, N, K;
  int tiles_m, tiles_n, splits, kb_total, kb_per_split, groups, total_tiles;
  // hetero (split-K wgrad only): the second half of the groups has its own shape (GemmDesc::M2 / N2)
  int hetero, M2, N2, tiles_m2, tiles_n2, base2;      // base2 = first tile index of the second half
  int a_mn, b_mn;
  int dbg_flags;      // experiments (V2S_GEMM_DEBUG=<n>): 2 skip TMEM loads, 4 skip epilogue math + stores, 16 skip TMA stores only
  int b_stationary;   // K <= 192: the CTA keeps its [192 x K] B tile in smem and walks m-tiles only
  int ctas_per_combo; // b_stationary: CTAs sharing one (group, n_tile)
  int stages;         // smem ring depth: [A|B] slots when streaming, A-only slots when B-stationary
  int op_bytes;       // bytes of the operand region
  int stg_off;        // offset of the epilogue staging ring (after the operands; 0 = overlaid on them, see launch_kernel)
  int bar_off;        // offset of the barrier / constant block
  int late_wait;      // see GemmDesc::late_wait
  int* err_flag;
  long long* dbg;     // optional per-role cycle counters of CTA 0 (V2S_GEMM_DEBUG=1)
  // T_ACCUM_DET: the gradients (+ row stride), the slab of partial tiles (tmOut2[0] maps it: tile slot s = rows
  // [128 s, 128 s + 128)), the partial row sums [slot][128] and one arrival counter per output tile
  float* det_out[MAXG];
  int64_t det_ldc[MAXG];
  float* det_slab;
  float* det_rowpart;
  unsigned* det_counters;
};


// DBG: the instrumented build of the kernel (per-role cycle counters, ablation switches), launched only when
// V2S_GEMM_DEBUG is set: even predicated-off clock reads cost issue slots in the issue-bound epilogues.
template <int EPI, bool OUT_BF16, bool DBG, typename LP>
__global__ void __launch_bounds__(N_THREADS, 1) gemm_tc_kernel(const __grid_constant__ TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int N_STG = Cfg<EPI, OUT_BF16>::NSTG, STG_BYTES = Cfg<EPI, OUT_BF16>::STG;
  const int STAGES = p.stages;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + p.bar_off);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* tfull_bar = empty_bar + MAX_STAGES;  // [2] accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;          // [2] accumulator drained
  uint64_t* aux_bar = tempty_bar + 2;            // [2][3] per epilogue group and staging buffer: aux chunk landed
  uint64_t* bres_bar = aux_bar + 6;              // B-stationary tile landed
  uint64_t* sfull_bar = bres_bar + 1;            // [2][3] staging buffer written by the 256 epilogue threads of a group
  uint64_t* sfree_bar = sfull_bar + 6;           // [2][3] staging buffer released by the group's store warp
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(sfree_bar + 6);
  uint8_t* ones_tile = reinterpret_cast<uint8_t*>(full_bar) + 1024;
  float2* ln_part = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(full_bar) + 3072);   // [2 groups][2 halves][128 rows]   // [16 rows x 128 B] K-major: row 0 = 1.0, rows 1..15 = 0

  // warp index through a shuffle: tells the compiler it is warp-uniform, so that the single-thread
  // roles below compile to straight uniform-datapath code (no per-lane convergence loops around TMA / MMA)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  constexpr bool ACC = EPI == T_ACCUM || EPI == T_ACCUM_DET, DET = EPI == T_ACCUM_DET;
  // T_ACCUM_DET: output tiles whose last split this CTA stored ([0] = count; the LayerNorm scratch is unused here)
  int* fix_list = reinterpret_cast<int*>(ln_part);

  if (warp == 0 && lane == 0) {
    for (int g = 0; g < p.groups; ++g) {
      ptx::prefetch_tmap(&p.tmA[g]);
      ptx::prefetch_tmap(&p.tmB[g]);
      ptx::prefetch_tmap(&p.tmOut[g]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { ptx::mbar_init(&full_bar[s], 1); ptx::mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(&tfull_bar[s], 1); ptx::mbar_init(&tempty_bar[s], 8); }
    for (int s = 0; s < 6; ++s) { ptx::mbar_init(&aux_bar[s], 1); ptx::mbar_init(&sfull_bar[s], 256); ptx::mbar_init(&sfree_bar[s], 1); }
    ptx::mbar_init(bres_bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_ptr, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  if (ACC && warp == 3) {
    // a row of 16-bit 1.0 values; the swizzle only permutes 16-byte chunks inside a row, so a constant row is layout-proof
    for (int i = lane; i < 2048 / 4; i += 32)
      reinterpret_cast<uint32_t*>(ones_tile)[i] = (i < 32) ? LP::kOnePair : 0u;
    if (DET && lane == 0) fix_list[0] = 0;
    ptx::fence_proxy_async();
  }
  // Programmatic dependent launch.  Every kernel of this library waits for its predecessor and only THEN
  // releases its successor (the successor's CTAs cannot become resident before ours exit anyway: shared memory).
  // So when a kernel starts, everything up to its predecessor's predecessor is complete.  A kernel flagged
  // late_wait (the dgrad launched right after the wgrad that shares its inputs: all of them at least two kernels
  // old) uses that: it skips the wait, starts its CTAs as the predecessor's CTAs exit instead of draining it, and
  // waits just before exiting, so that "this kernel complete" still implies "all earlier kernels complete" for
  // whoever follows.
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
  if (!p.late_wait) {
    ptx::pdl_wait();                // everything above overlapped the predecessor's tail; its outputs are visible now
    ptx::pdl_launch_dependents();
  }

  const int tiles_per_group = p.tiles_m * p.splits * p.tiles_n;
  // i-th tile of this CTA (same sequence for every warp role); false when the CTA is done
  auto tile_at = [&](int i, int& g, int& m_tile, int& split, int& n_tile) -> bool {
    if (p.b_stationary) {
      const int combo = blockIdx.x / p.ctas_per_combo, rank = blockIdx.x % p.ctas_per_combo;
      g = combo / p.tiles_n; n_tile = combo % p.tiles_n; split = 0;
      m_tile = rank + i * p.ctas_per_combo;
      return m_tile < p.tiles_m;
    }
    const int t = blockIdx.x + i * gridDim.x;
    if (t >= p.total_tiles) return false;
    if (p.hetero && t >= p.base2) {
      const int per_group2 = p.tiles_m2 * p.splits * p.tiles_n2;
      const int t2 = t - p.base2;
      const int g2 = t2 / per_group2;
      int r = t2 - g2 * per_group2;
      g = p.groups / 2 + g2;
      n_tile = r % p.tiles_n2; r /= p.tiles_n2;
      split = r % p.splits;
      m_tile = r / p.splits;
      return true;
    }
    g = t / tiles_per_group;
    int r = t - g * tiles_per_group;
    n_tile = r % p.tiles_n; r /= p.tiles_n;
    split = r % p.splits;
    m_tile = r / p.splits;
    return true;
  };
  auto rows_of = [&](int g) { return (p.hetero && g >= p.groups / 2) ? p.M2 : p.M; };
  auto cols_of = [&](int g) { return (p.hetero && g >= p.groups / 2) ? p.N2 : p.N; };
  // T_ACCUM_DET: index of an output tile (all splits of it share one arrival counter); its split s has slab slot
  // out_tile * splits + s
  auto out_tile = [&](int g, int m_tile, int n_tile) {
    if (p.hetero && g >= p.groups / 2)
      return p.base2 / p.splits + ((g - p.groups / 2) * p.tiles_m2 + m_tile) * p.tiles_n2 + n_tile;
    return (g * p.tiles_m + m_tile) * p.tiles_n + n_tile;
  };
  // smem map of the operand region: streaming mode = 3 stages of [A 16 KB | B 24 KB];
  // B-stationary mode = [B tile: kb_total (<= 3) k-blocks x 24 KB] followed by a ring of A slots (16 KB)
  uint8_t* bres = smem;
  uint8_t* aring = smem + p.kb_total * B_STAGE_BYTES;

  if (warp == 0) {
    // ================= TMA producer (whole warp walks the loop; one elected lane issues) =================
    long long prod_wait = 0; const long long prod_t0 = clock64();
    int stage = 0; uint32_t phase = 0;
    int g, m_tile, split, n_tile;
    if (p.b_stationary && tile_at(0, g, m_tile, split, n_tile)) {
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(bres_bar, p.kb_total * B_STAGE_BYTES);
        for (int kb = 0; kb < p.kb_total; ++kb) {
          uint8_t* sb = bres + kb * B_STAGE_BYTES;
          if (!p.b_mn) {
            ptx::tma_load_2d(sb, &p.tmB[g], bres_bar, kb * BK, n_tile * BN);
          } else {
            ptx::tma_load_2d(sb, &p.tmB[g], bres_bar, n_tile * BN, kb * BK);
            ptx::tma_load_2d(sb + 8192, &p.tmB[g], bres_bar, n_tile * BN + 64, kb * BK);
            ptx::tma_load_2d(sb + 16384, &p.tmB[g], bres_bar, n_tile * BN + 128, kb * BK);
          }
        }
      }
      __syncwarp();
    }
    for (int i = 0; tile_at(i, g, m_tile, split, n_tile); ++i) {
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      for (int kb = kb0; kb < kb1; ++kb) {
        const long long w0 = DBG ? clock64() : 0;
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1, p.err_flag, 1);
        if (DBG) prod_wait += clock64() - w0;
        if (ptx::elect_one()) {
          uint8_t* sa = p.b_stationary ? aring + stage * A_STAGE_BYTES : smem + stage * STAGE_BYTES;
          uint8_t* sb = sa + A_STAGE_BYTES;
          ptx::mbar_arrive_expect_tx(&full_bar[stage], p.b_stationary ? A_STAGE_BYTES : STAGE_BYTES);
          if (!p.a_mn) {
            ptx::tma_load_2d(sa, &p.tmA[g], &full_bar[stage], kb * BK, m_tile * BM);
          } else {
            ptx::tma_load_2d(sa, &p.tmA[g], &full_bar[stage], m_tile * BM, kb * BK);
            ptx::tma_load_2d(sa + 8192, &p.tmA[g], &full_bar[stage], m_tile * BM + 64, kb * BK);
          }
          if (!p.b_stationary) {
            if (!p.b_mn) {
              ptx::tma_load_2d(sb, &p.tmB[g], &full_bar[stage], kb * BK, n_tile * BN);
            } else {
              ptx::tma_load_2d(sb, &p.tmB[g], &full_bar[stage], n_tile * BN, kb * BK);
              ptx::tma_load_2d(sb + 8192, &p.tmB[g], &full_bar[stage], n_tile * BN + 64, kb * BK);
              ptx::tma_load_2d(sb + 16384, &p.tmB[g], &full_bar[stage], n_tile * BN + 128, kb * BK);
            }
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    if (DBG && blockIdx.x == 0 && lane == 0) { p.dbg[0] = prod_wait; p.dbg[1] = clock64() - prod_t0; }
  } else if (warp == 1) {
    // ================= MMA issuer (whole warp walks the loop; one elected lane issues) =================
    const uint32_t idesc = make_idesc_lp(LP::kIdescFmt, BM, BN, p.a_mn, p.b_mn);
    // descriptor low words per smem slot; a K-step of 16 adds 32 B (K-major) or 2048 B (MN-major), >> 4
    const uint32_t smem_base = ptx::smem_u32(smem);
    const uint32_t a_step = p.a_mn ? (2048u >> 4) : (32u >> 4), b_step = p.b_mn ? (2048u >> 4) : (32u >> 4);
    const uint32_t a_lbo = p.a_mn ? 8192u : 16u, b_lbo = p.b_mn ? 8192u : 16u;
    const uint32_t a_slot0 = p.b_stationary ? p.kb_total * B_STAGE_BYTES : 0, a_slot_stride = p.b_stationary ? A_STAGE_BYTES : STAGE_BYTES;
    const uint32_t b_slot0 = p.b_stationary ? 0 : A_STAGE_BYTES, b_slot_stride = p.b_stationary ? B_STAGE_BYTES : STAGE_BYTES;
    const uint32_t a_lo0 = ptx::desc_lo(smem_base + a_slot0, a_lbo), b_lo0 = ptx::desc_lo(smem_base + b_slot0, b_lbo);
    const uint32_t idesc_rs = make_idesc_lp(LP::kIdescFmt, BM, 16, p.a_mn, 0);
    const uint32_t ones_lo = ptx::desc_lo(ptx::smem_u32(ones_tile), 16);
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    int g, m_tile, split, n_tile;
    long long w_full = 0, w_tempty = 0, ntiles = 0; const long long mma_t0 = clock64();
    if (p.b_stationary && tile_at(0, g, m_tile, split, n_tile)) ptx::mbar_wait(bres_bar, 0, p.err_flag, 6);
    for (int i = 0; tile_at(i, g, m_tile, split, n_tile); ++i) {
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      long long w0 = DBG ? clock64() : 0;
      ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1, p.err_flag, 2);
      if (DBG) { w_tempty += clock64() - w0; ++ntiles; }
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * ACC_STRIDE;
      for (int kb = kb0; kb < kb1; ++kb) {
        if (DBG) w0 = clock64();
        ptx::mbar_wait(&full_bar[stage], phase, p.err_flag, 3);
        if (DBG) w_full += clock64() - w0;
        ptx::tc_fence_after();
        const uint32_t a_lo = a_lo0 + ((stage * a_slot_stride) >> 4);
        const uint32_t b_lo = b_lo0 + (((p.b_stationary ? kb : stage) * b_slot_stride) >> 4);
        if (ptx::elect_one()) {
          ptx::umma_bf16_lohi(d_tmem, a_lo, b_lo, ptx::DESC_HI_SW128_SBO1024, idesc, kb > kb0 ? 1u : 0u);
          ptx::umma_bf16_lohi(d_tmem, a_lo + a_step, b_lo + b_step, ptx::DESC_HI_SW128_SBO1024, idesc, 1u);
          ptx::umma_bf16_lohi(d_tmem, a_lo + 2 * a_step, b_lo + 2 * b_step, ptx::DESC_HI_SW128_SBO1024, idesc, 1u);
          ptx::umma_bf16_lohi(d_tmem, a_lo + 3 * a_step, b_lo + 3 * b_step, ptx::DESC_HI_SW128_SBO1024, idesc, 1u);
          if (ACC && n_tile == 0 && p.rowsum[g] != nullptr && !(DBG && (p.dbg_flags & 32))) {
            // row sums of A (= bias gradient in a wgrad) into accumulator columns [192,208): A x ones
#pragma unroll
            for (int k = 0; k < 4; ++k)
              ptx::umma_bf16_lohi(d_tmem + BN, a_lo + k * a_step, ones_lo, ptx::DESC_HI_SW128_SBO1024, idesc_rs,
                                  (kb > kb0 || k > 0) ? 1u : 0u);
          }
          ptx::umma_commit(&empty_bar[stage]);       // frees the smem slot when these MMAs retire
          if (kb == kb1 - 1) ptx::umma_commit(&tfull_bar[acc]);   // accumulator complete → epilogue
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (DBG && blockIdx.x == 0 && lane == 0) { p.dbg[2] = w_full; p.dbg[3] = w_tempty; p.dbg[4] = clock64() - mma_t0; p.dbg[5] = ntiles; }
  } else if (warp == 2 || warp == 3) {
    // ================= store warp of epilogue group ge (whole warp walks the loop; one elected lane issues) ====
    const int ge = warp - 2;
    uint8_t* stg_base = smem + p.stg_off + ge * N_STG * STG_BYTES;
    uint64_t* abar = aux_bar + ge * 3;
    uint64_t* sfull = sfull_bar + ge * 3;
    uint64_t* sfree = sfree_bar + ge * 3;
    constexpr bool HAS_AUX = EPI == T_RESID;
    constexpr int AUX_BYTES = BM * CHUNK * 4;
    const bool LN = (EPI == T_RESID) && p.ln != 0;
    const int RPT = LN ? 2 * N_CHUNKS : N_CHUNKS;
    // slot n becomes reusable: prefetch the auxiliary operand of its next user into the buffer, or release it
    auto recycle = [&](int n) {
      const int next = n + N_STG, c = next % RPT, b = next % N_STG;
      int g, m_tile, split, n_tile;
      if (!tile_at(ge + 2 * (next / RPT), g, m_tile, split, n_tile)) return;     // no further user
      if (HAS_AUX && c < N_CHUNKS) {
        ptx::mbar_arrive_expect_tx(&abar[b], AUX_BYTES);
        ptx::tma_load_2d(stg_base + b * STG_BYTES, &p.tmAux[g], &abar[b], n_tile * BN + c * CHUNK, m_tile * BM);
      } else {
        ptx::mbar_arrive(&sfree[b]);
      }
    };
    if (HAS_AUX && ptx::elect_one()) {
      for (int n = -N_STG; n < 0; ++n) recycle(n);     // all buffers start free: prefetch for slots 0..N_STG-1
    }
    __syncwarp();
    uint32_t full_par = 0;
    int n = 0;
    int g, m_tile, split, n_tile;
    for (int i = ge; tile_at(i, g, m_tile, split, n_tile); i += 2) {
      const int m0 = m_tile * BM, n0 = n_tile * BN;
#pragma unroll 1
      for (int c = 0; c < RPT; ++c, ++n) {
        const int b = n % N_STG;
        ptx::mbar_wait(&sfull[b], (full_par >> b) & 1, p.err_flag, 8);
        full_par ^= 1u << b;
        if (ptx::elect_one()) {
          uint8_t* stg = stg_base + b * STG_BYTES;
          if (!(DBG && (p.dbg_flags & (4 | 16)))) {
            if (c < N_CHUNKS) {
              const int col0 = n0 + c * CHUNK;
              if (col0 < cols_of(g)) {
                if (DET) ptx::tma_store_2d(&p.tmOut2[0], stg, c * CHUNK, (out_tile(g, m_tile, n_tile) * p.splits + split) * BM);
                else if (EPI == T_ACCUM) ptx::tma_reduce_add_2d(&p.tmOut[g], stg, col0, m0);
                else ptx::tma_store_2d(&p.tmOut[g], stg, col0, m0);
              }
            } else {
              ptx::tma_store_2d(&p.tmOut2[g], stg, (c - N_CHUNKS) * CHUNK, m0);   // normalised row chunk
            }
          }
          ptx::tma_commit_group();
          if (n >= 1) {
            ptx::tma_wait_group_read<1>();             // the store of slot n-1 has left its buffer
            recycle(n - 1);
          }
          if (DET && c == RPT - 1) {
            // the tile's partial (and, through sfull, its row sums) is in global memory: count this split in.  The
            // split that completes the count owns the fix-up; nobody waits for anybody.
            ptx::tma_wait_group<0>();
            ptx::fence_proxy_async_global();
            const int o = out_tile(g, m_tile, n_tile);
            if (ptx::atom_add_acq_rel_gpu(&p.det_counters[o], 1u) == (unsigned)(p.splits - 1))
              fix_list[1 + atomicAdd(&fix_list[0], 1)] = (g << 24) | (m_tile << 12) | n_tile;
          }
        }
        __syncwarp();
      }
    }
    if (ptx::elect_one()) ptx::tma_wait_group<0>();
    __syncwarp();
  } else if (warp >= 4) {
    // ================= epilogue =================
    // 16 warps = 2 groups of 8.  Group ge drains accumulator stage ge.  Inside a group, warps w and w+4 share
    // TMEM lane quarter w%4 and split every 32-column chunk into two 16-column halves (thread = one row x 16 cols).
    const int ge = (warp - 4) >> 3;                 // epilogue group = accumulator stage it drains
    const int q = warp & 3;                         // TMEM lane quarter
    const int hf = ((warp - 4) >> 2) & 1;           // column half of the chunk
    const int row = q * 32 + lane;                  // row within the 128-row tile
    uint8_t* stg_base = smem + p.stg_off + ge * N_STG * STG_BYTES;
    const uint32_t stg_s0 = ptx::smem_u32(stg_base);
    const bool full_n = (p.N % BN) == 0;
    uint64_t* abar = aux_bar + ge * 3;
    uint64_t* sfull = sfull_bar + ge * 3;
    uint64_t* sfree = sfree_bar + ge * 3;
    const int bar_id = 1 + ge;
    constexpr bool HAS_AUX = EPI == T_RESID;
    // With the fused LayerNorm every tile takes 12 ring slots: 6 residual chunks (pass 1) + 6 normalised chunks.
    const bool LN = (EPI == T_RESID) && p.ln != 0;
    const int RPT = LN ? 2 * N_CHUNKS : N_CHUNKS;      // ring slots per tile
    // Staging ring protocol (slot n uses buffer n % N_STG).  The group's store warp (warp 2 + ge) owns all TMA
    // traffic of the ring: it stores a slot once the 256 epilogue threads have arrived on sfull, and when an
    // older store has left its buffer it either prefetches the next auxiliary operand into it (arrival on
    // abar) or releases it (arrival on sfree).  The epilogue threads never wait for a store of their own.
    uint32_t aux_par = 0, free_par = 0;                // per-buffer parities of the next abar / sfree completion
    auto acquire_slot = [&](int n) {
      const int b = n % N_STG;
      if (HAS_AUX && (n % RPT) < N_CHUNKS) {
        ptx::mbar_wait(&abar[b], (aux_par >> b) & 1, p.err_flag, 5);
        aux_par ^= 1u << b;
      } else if (n >= N_STG) {
        ptx::mbar_wait(&sfree[b], (free_par >> b) & 1, p.err_flag, 7);
        free_par ^= 1u << b;
      }
    };
    long long e_pub = 0;
    auto publish_slot = [&](int n) {
      const long long t0 = DBG ? clock64() : 0;
      ptx::fence_proxy_async();
      ptx::mbar_arrive(&sfull[n % N_STG]);
      if (DBG) e_pub += clock64() - t0;
    };

    uint32_t acc_phase = 0;
    int cnt = 0;                                    // running chunk counter of this group
    long long e_tfull = 0, e_aux = 0, e_ld = 0; const long long epi_t0 = clock64();
    (void)bar_id;
    int g, m_tile, split, n_tile;
    for (int i = ge; tile_at(i, g, m_tile, split, n_tile); i += 2) {
      const int m0 = m_tile * BM, n0 = n_tile * BN;
      long long w0 = DBG ? clock64() : 0;
      ptx::mbar_wait(&tfull_bar[ge], acc_phase, p.err_flag, 4);
      if (DBG) e_tfull += clock64() - w0;
      acc_phase ^= 1;
      ptx::tc_fence_after();
      const float* bias = !ACC ? p.bias[g] : nullptr;
      const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16) + ge * ACC_STRIDE;
      float ln_s1 = 0.f, ln_s2 = 0.f;
#pragma unroll 1
      for (int c = 0; c < N_CHUNKS; ++c, ++cnt) {
        const int col0 = n0 + c * CHUNK;            // first column of the chunk
        const int colh = col0 + hf * 16;            // first column of this thread's half
        const int b = cnt % N_STG;
        const uint32_t stg_s = stg_s0 + b * STG_BYTES;
        // bias first (its registers are then live across the tensor-memory load instead of being shuffled around
        // it); the column bound is only checked when N is not a whole number of tiles
        float4 bb[4];
        if (bias != nullptr) {
          const float4* b4 = reinterpret_cast<const float4*>(bias + colh);
          if (full_n) {
#pragma unroll
            for (int k = 0; k < 4; ++k) bb[k] = __ldg(b4 + k);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) bb[k] = (colh + 4 * k < p.N) ? __ldg(b4 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        uint32_t r[16];
        if (DBG) w0 = clock64();
        if (!(DBG && (p.dbg_flags & 2))) {
          ptx::tmem_ld_32x16(tlane + c * CHUNK + hf * 16, r);
          ptx::tmem_ld_wait();
        } else {
#pragma unroll
          for (int k = 0; k < 16; ++k) r[k] = 0;
        }
        if (DBG) e_ld += clock64() - w0;
        if (c == N_CHUNKS - 1 && !LN) {             // accumulator fully read: hand the stage back to the MMA warp
          if (ACC && hf == 0 && n_tile == 0 && p.rowsum[g] != nullptr) {
            uint32_t rs[16];
            ptx::tmem_ld_32x16(tlane + BN, rs);
            ptx::tmem_ld_wait();
            if (DET) {
              p.det_rowpart[(out_tile(g, m_tile, n_tile) * p.splits + split) * BM + row] = __uint_as_float(rs[0]);
              __threadfence();
            } else if (m0 + row < rows_of(g)) {
              atomicAdd(p.rowsum[g] + m0 + row, __uint_as_float(rs[0]));
            }
          }
          ptx::tc_fence_before();
          if (lane == 0) ptx::mbar_arrive(&tempty_bar[ge]);
        }
        float v[16];
        if (bias != nullptr) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            v[4 * k] = __uint_as_float(r[4 * k]) + bb[k].x; v[4 * k + 1] = __uint_as_float(r[4 * k + 1]) + bb[k].y;
            v[4 * k + 2] = __uint_as_float(r[4 * k + 2]) + bb[k].z; v[4 * k + 3] = __uint_as_float(r[4 * k + 3]) + bb[k].w;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] = __uint_as_float(r[k]);
        }
        // fp32 rows are 128 B (8 x 16-B pieces, SWIZZLE_128B), bf16 rows 64 B (4 pieces, SWIZZLE_64B)
        if (DBG) w0 = clock64();
        acquire_slot(cnt);                           // buffer b is ours (and holds the auxiliary operand, if any)
        if (DBG) e_aux += clock64() - w0;
        if (DBG && (p.dbg_flags & 4)) { publish_slot(cnt); continue; }
        if (HAS_AUX) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t slot = stg_s + row * 128 + (((hf * 4 + j) ^ (row & 7)) << 4);
            const float4 a = ptx::lds128f(slot);
            v[4 * j] += a.x; v[4 * j + 1] += a.y; v[4 * j + 2] += a.z; v[4 * j + 3] += a.w;
            ptx::sts128f(slot, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          if (LN) {     // row statistics, and the finished row back into TMEM for the normalisation pass
            uint32_t xr[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) { ln_s1 += v[k]; ln_s2 = fmaf(v[k], v[k], ln_s2); xr[k] = __float_as_uint(v[k]); }
            ptx::tmem_st_32x16(tlane + c * CHUNK + hf * 16, xr);
          }
        } else if (OUT_BF16) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint4 o;
            o.x = LP::pack(v[8 * j], v[8 * j + 1]); o.y = LP::pack(v[8 * j + 2], v[8 * j + 3]);
            o.z = LP::pack(v[8 * j + 4], v[8 * j + 5]); o.w = LP::pack(v[8 * j + 6], v[8 * j + 7]);
            ptx::sts128(stg_s + row * 64 + (((hf * 2 + j) ^ ((row >> 1) & 3)) << 4), o.x, o.y, o.z, o.w);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            ptx::sts128f(stg_s + row * 128 + (((hf * 4 + j) ^ (row & 7)) << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2],
                         v[4 * j + 3]);
        }
        publish_slot(cnt);
      }
      if (EPI == T_RESID && LN) {
        // ---- fused LayerNorm over the finished 192-wide row (two threads per row: exchange partial sums) ----
        ptx::tmem_st_wait();
        ln_part[(ge * 2 + hf) * BM + row] = make_float2(ln_s1, ln_s2);
        ptx::bar_sync(bar_id, 256);
        const float2 other = ln_part[(ge * 2 + (hf ^ 1)) * BM + row];
        const float mean = (ln_s1 + other.x) * (1.0f / BN);
        const float var = fmaxf((ln_s2 + other.y) * (1.0f / BN) - mean * mean, 0.f);
        const float rstd = 1.0f / sqrtf(var + LN_EPS);
        if (hf == 0 && m0 + row < p.M && p.ln_mean[g] != nullptr) {
          p.ln_mean[g][m0 + row] = mean;
          p.ln_rstd[g][m0 + row] = rstd;
        }
        const float* gam = p.ln_gamma[g];
        const float* bet = p.ln_beta[g];
#pragma unroll 1
        for (int c = 0; c < N_CHUNKS; ++c, ++cnt) {
          const int colh = c * CHUNK + hf * 16;
          const int b = cnt % N_STG;
          const uint32_t stg_s = stg_s0 + b * STG_BYTES;
          uint32_t r[16];
          ptx::tmem_ld_32x16(tlane + colh, r);
          ptx::tmem_ld_wait();
          acquire_slot(cnt);
          if (c == N_CHUNKS - 1) {                  // accumulator (now holding the row) fully read
            ptx::tc_fence_before();
            if (lane == 0) ptx::mbar_arrive(&tempty_bar[ge]);
          }
          float v[16];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 gg = __ldg(reinterpret_cast<const float4*>(gam + colh) + k);
            const float4 bb = __ldg(reinterpret_cast<const float4*>(bet + colh) + k);
            v[4 * k] = (__uint_as_float(r[4 * k]) - mean) * rstd * gg.x + bb.x;
            v[4 * k + 1] = (__uint_as_float(r[4 * k + 1]) - mean) * rstd * gg.y + bb.y;
            v[4 * k + 2] = (__uint_as_float(r[4 * k + 2]) - mean) * rstd * gg.z + bb.z;
            v[4 * k + 3] = (__uint_as_float(r[4 * k + 3]) - mean) * rstd * gg.w + bb.w;
          }
#pragma unroll
          for (int j = 0; j < 2; ++j) {             // bf16 chunk: 64-byte rows, SWIZZLE_64B, first 8 KB of the buffer
            uint4 o;
            o.x = LP::pack(v[8 * j], v[8 * j + 1]); o.y = LP::pack(v[8 * j + 2], v[8 * j + 3]);
            o.z = LP::pack(v[8 * j + 4], v[8 * j + 5]); o.w = LP::pack(v[8 * j + 6], v[8 * j + 7]);
            ptx::sts128(stg_s + row * 64 + (((hf * 2 + j) ^ ((row >> 1) & 3)) << 4), o.x, o.y, o.z, o.w);
          }
          publish_slot(cnt);
        }
      }
    }
    if (DBG && blockIdx.x == 0 && (threadIdx.x == 128 || threadIdx.x == 384 + 37)) {
      long long* d = p.dbg + 8 + (threadIdx.x == 128 ? 0 : 8);
      d[0] = e_tfull; d[1] = e_aux; d[2] = e_pub; d[3] = e_ld; d[4] = clock64() - epi_t0; d[5] = cnt;
    }
  }

  if (p.late_wait) { ptx::pdl_wait(); ptx::pdl_launch_dependents(); }
  ptx::tc_fence_before();
  __syncthreads();
  if (DET) {
    // fix-up of the output tiles this CTA completed, by all its threads: gradient += partial 0 + ... + partial S-1
    for (int e = 0; e < fix_list[0]; ++e) {
      const int code = fix_list[1 + e], g = code >> 24, m_tile = (code >> 12) & 4095, n_tile = code & 4095;
      const int o = out_tile(g, m_tile, n_tile), m0 = m_tile * BM, n0 = n_tile * BN;
      const int rows = min(BM, rows_of(g) - m0), c4s = min(BN, cols_of(g) - n0) / 4;
      const float* slab = p.det_slab + (int64_t)o * p.splits * BM * BN;
      for (int i = threadIdx.x; i < rows * c4s; i += N_THREADS) {
        const int r = i / c4s, c4 = i - r * c4s;
        float4* dst = reinterpret_cast<float4*>(p.det_out[g] + (int64_t)(m0 + r) * p.det_ldc[g] + n0) + c4;
        float4 v = *dst;
        for (int s = 0; s < p.splits; ++s) {
          const float4 a = __ldcg(reinterpret_cast<const float4*>(slab + ((int64_t)s * BM + r) * BN) + c4);
          v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
        }
        *dst = v;
      }
      if (n_tile == 0 && p.rowsum[g] != nullptr && threadIdx.x < rows) {
        float v = p.rowsum[g][m0 + threadIdx.x];
        for (int s = 0; s < p.splits; ++s) v += __ldcg(p.det_rowpart + (o * p.splits + s) * BM + threadIdx.x);
        p.rowsum[g][m0 + threadIdx.x] = v;
      }
      if (threadIdx.x == 0) p.det_counters[o] = 0;     // zero again for the next launch
    }
  }
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// host side: tensor-map cache + dispatch
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
int* g_err_flag[MAX_DEVICES] = {nullptr};      // device int per GPU, allocated once at init (4 bytes; the only allocation)
long long* g_dbg[MAX_DEVICES] = {nullptr};     // 32 counters, only with V2S_GEMM_DEBUG=1
int g_num_sms_dev[MAX_DEVICES] = {0};
int g_sm_limit = 0;             // v2s_set_sm_limit: persistent grids leave SMs to a concurrent collective
int g_deterministic = 0;        // v2s_set_deterministic
int g_dbg_flags = 0;

struct MapKey {
  const void* ptr; uint64_t d0, d1, stride1; uint32_t b0, b1, dtype, swz;
  bool operator==(const MapKey& o) const { return memcmp(this, &o, sizeof(MapKey)) == 0; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    const uint64_t* w = reinterpret_cast<const uint64_t*>(&k);
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < sizeof(MapKey) / 8; ++i) { h ^= w[i]; h *= 1099511628211ull; }
    return (size_t)h;
  }
};
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;

// 2-D row-major tensor [d1 rows, d0 cols] of `dtype`, row stride `stride1` elements, box b0 x b1
int get_map(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t stride1_elems, uint32_t b0,
            uint32_t b1, bool is_bf16, CUtensorMapSwizzle swz) {
  MapKey key;
  memset(&key, 0, sizeof(key));
  key.ptr = ptr; key.d0 = d0; key.d1 = d1; key.stride1 = stride1_elems; key.b0 = b0; key.b1 = b1;
  key.dtype = is_bf16 ? 1 : 0; key.swz = (uint32_t)swz;
  auto it = g_maps.find(key);
  if (it != g_maps.end()) { *out = it->second; return 0; }
  const uint64_t es = is_bf16 ? 2 : 4;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((stride1_elems * es) & 15)) {
    set_error("gemm_tc: tensor %p (row stride %llu B) is not 16-byte aligned for TMA", ptr,
              (unsigned long long)(stride1_elems * es));
    return 1;
  }
  cuuint64_t gdim[2] = {d0, d1};
  cuuint64_t gstride[1] = {stride1_elems * es};
  cuuint32_t box[2] = {b0, b1};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = g_encode(&m, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for tensor %p dims %llu x %llu box %u x %u", (int)r, ptr,
              (unsigned long long)d0, (unsigned long long)d1, b0, b1);
    return 1;
  }
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps.emplace(key, m);
  *out = m;
  return 0;
}

}  // namespace

// rank-3 variant used by the attention kernels: tensor [d2][d1][d0] with byte strides s1, s2
int tmap_get_3d(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1_bytes,
                uint64_t s2_bytes, uint32_t b0, uint32_t b1, bool is_bf16, int swizzle_bytes) {
  if (!g_encode) { set_error("tensor maps not initialised (v2s_init)"); return 1; }
  MapKey key;
  memset(&key, 0, sizeof(key));
  key.ptr = ptr; key.d0 = d0; key.d1 = d1 | (d2 << 32); key.stride1 = s1_bytes ^ (s2_bytes << 20); key.b0 = b0; key.b1 = b1;
  key.dtype = (is_bf16 ? 1 : 0) | 0x100; key.swz = (uint32_t)swizzle_bytes;
  auto it = g_maps.find(key);
  if (it != g_maps.end()) { *out = it->second; return 0; }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (s1_bytes & 15) || (s2_bytes & 15)) {
    set_error("tmap_get_3d: tensor %p not 16-byte aligned for TMA", ptr);
    return 1;
  }
  cuuint64_t gdim[3] = {d0, d1, d2};
  cuuint64_t gstride[2] = {s1_bytes, s2_bytes};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle swz = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUtensorMap m;
  CUresult r = g_encode(&m, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                        const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(3d) failed (%d)", (int)r); return 1; }
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps.emplace(key, m);
  *out = m;
  return 0;
}
int tmap_get_2d(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t stride1_elems, uint32_t b0,
                uint32_t b1, bool is_lp, int swizzle_bytes) {
  if (!g_encode) { set_error("tensor maps not initialised (v2s_init)"); return 1; }
  return get_map(out, ptr, d0, d1, stride1_elems, b0, b1, is_lp,
                 swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                 : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
}
int tc_num_sms() {
  const int n = g_num_sms_dev[cur_device()] > 0 ? g_num_sms_dev[cur_device()] : 148;
  return (g_sm_limit > 0 && g_sm_limit < n) ? g_sm_limit : n;
}
void tc_set_sm_limit(int n) { g_sm_limit = n > 0 ? n : 0; }
void tc_set_deterministic(int on) { g_deterministic = on ? 1 : 0; }
int tc_deterministic() { return g_deterministic; }
static int tc_device_sms() { return g_num_sms_dev[cur_device()] > 0 ? g_num_sms_dev[cur_device()] : 148; }
// a deterministic split-K launch has at most one tile per SM of the device (see launch_gemm_tc)
int64_t gemm_tc_det_part_floats() { return (int64_t)tc_device_sms() * (BM * BN + BM); }
int* tc_err_flag() { return g_err_flag[cur_device()]; }
long long* tc_dbg_counters() { return g_dbg[cur_device()]; }

namespace {

template <int EPI, bool OUT_BF16, bool DBG, typename LP>
int launch_kernel_impl(TcParams& p, cudaStream_t stream) {
  static bool attr_set[MAX_DEVICES] = {false};
  if (!attr_set[cur_device()]) {
    V2S_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<EPI, OUT_BF16, DBG, LP>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_set[cur_device()] = true;
  }
  const int g_num_sms = tc_num_sms();
  // split the 227 KB between the operand ring and the epilogue staging ring of this variant
  const int budget = SMEM_LIMIT - 1024 - SMEM_BAR_BYTES - Cfg<EPI, OUT_BF16>::STAGING_BYTES;
  if (p.b_stationary) {
    const int bres = p.kb_total * B_STAGE_BYTES;
    int ring = (budget - bres) / A_STAGE_BYTES;
    if (ring > MAX_STAGES) ring = MAX_STAGES;
    p.stages = ring;
    p.op_bytes = bres + ring * A_STAGE_BYTES;
  } else {
    int st = budget / STAGE_BYTES;
    if (st > MAX_STAGES) st = MAX_STAGES;
    p.stages = st;
    p.op_bytes = st * STAGE_BYTES;
  }
  p.stg_off = p.op_bytes;
  p.bar_off = p.op_bytes + Cfg<EPI, OUT_BF16>::STAGING_BYTES;
  if ((EPI == T_ACCUM || EPI == T_ACCUM_DET) && !p.b_stationary && p.total_tiles <= g_num_sms) {
    // one tile per CTA (the one-wave split-K wgrad): its epilogue starts after the last MMA has retired, when
    // the operand ring is dead, so the staging buffers overlay the ring and the ring gets their 64 KB
    int st = (SMEM_LIMIT - 1024 - SMEM_BAR_BYTES) / STAGE_BYTES;
    if (st > MAX_STAGES) st = MAX_STAGES;
    if (st * STAGE_BYTES >= Cfg<EPI, OUT_BF16>::STAGING_BYTES) {
      p.stages = st;
      p.op_bytes = st * STAGE_BYTES;
      p.stg_off = 0;
      p.bar_off = p.op_bytes;
    }
  }
  if (p.stages < 2) { set_error("gemm_tc: shared-memory budget leaves %d pipeline stages", p.stages); return 1; }
  const int SMEM_TOTAL = p.bar_off + SMEM_BAR_BYTES + 1024;
  int grid = p.total_tiles < g_num_sms ? p.total_tiles : g_num_sms;
  if (p.b_stationary) grid = p.groups * p.tiles_n * p.ctas_per_combo;
  V2S_CUDA_OK(launch_pdl(gemm_tc_kernel<EPI, OUT_BF16, DBG, LP>, dim3(grid), dim3(N_THREADS), (size_t)SMEM_TOTAL, stream, p));
  V2S_LAUNCH_CHECK();
  return 0;
}

template <int EPI, bool OUT_BF16>
int launch_kernel(TcParams& p, int lp_f16, cudaStream_t stream) {
  if (lp_f16)
    return p.dbg ? launch_kernel_impl<EPI, OUT_BF16, true, LpF16>(p, stream) : launch_kernel_impl<EPI, OUT_BF16, false, LpF16>(p, stream);
  return p.dbg ? launch_kernel_impl<EPI, OUT_BF16, true, LpBf16>(p, stream) : launch_kernel_impl<EPI, OUT_BF16, false, LpBf16>(p, stream);
}

}  // namespace

int gemm_tc_init() {
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      set_error("cuTensorMapEncodeTiled entry point not available: %s", cudaGetErrorString(e));
      return 1;
    }
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    if (getenv("V2S_GEMM_DEBUG")) g_dbg_flags = atoi(getenv("V2S_GEMM_DEBUG"));
  }
  // per-device state of the CURRENT device
  const int dev = cur_device();
  if (g_err_flag[dev]) return 0;
  V2S_CUDA_OK(cudaDeviceGetAttribute(&g_num_sms_dev[dev], cudaDevAttrMultiProcessorCount, dev));
  V2S_CUDA_OK(cudaMalloc(&g_err_flag[dev], sizeof(int)));
  V2S_CUDA_OK(cudaMemset(g_err_flag[dev], 0, sizeof(int)));
  if (getenv("V2S_GEMM_DEBUG")) {
    V2S_CUDA_OK(cudaMalloc(&g_dbg[dev], 32 * sizeof(long long)));
    V2S_CUDA_OK(cudaMemset(g_dbg[dev], 0, 32 * sizeof(long long)));
  }
  return 0;
}

int gemm_tc_debug_counters(long long* host32) {
  long long* dbg = tc_dbg_counters();
  if (!dbg) { set_error("V2S_GEMM_DEBUG not set"); return 1; }
  V2S_CUDA_OK(cudaMemcpy(host32, dbg, 32 * sizeof(long long), cudaMemcpyDeviceToHost));
  V2S_CUDA_OK(cudaMemset(dbg, 0, 32 * sizeof(long long)));
  return 0;
}

int gemm_tc_error_flag() {
  int* flag = tc_err_flag();
  if (!flag) return 0;
  int v = 0;
  cudaMemcpy(&v, flag, sizeof(int), cudaMemcpyDeviceToHost);
  if (v) cudaMemset(flag, 0, sizeof(int));
  return v;
}

int launch_gemm_tc(const GemmDesc& d, int ta, int tb, int to, cudaStream_t stream, int* handled) {
  *handled = 0;
  if (ta == 0 || ta != tb) return 0;                      // fp32 check mode stays on the SIMT kernel
  if (to != 0 && to != ta) return 0;
  if (!g_encode) { set_error("tensor maps not initialised (v2s_init)"); return 1; }
  const int lp_f16 = (ta == AT_F16) ? 1 : 0;
  if (d.a_remap || d.b_remap) return 0;
  int epi;
  switch (d.epi) {
    case EPI_STORE: epi = T_STORE; break;
    case EPI_BIAS_RESID: epi = T_RESID; break;
    case EPI_ACCUM: epi = T_ACCUM; break;
    default: return 0;
  }
  if (d.alpha != 1.0f) return 0;
  const bool out_bf16 = (to != 0);                        // 16-bit output (bf16 or fp16, as the operands)
  if ((epi == T_RESID || epi == T_ACCUM) && out_bf16) return 0;
  int a_mn, b_mn;
  int64_t a_ld, b_ld;
  if (d.a_cs == 1) { a_mn = 0; a_ld = d.a_rs; } else if (d.a_rs == 1) { a_mn = 1; a_ld = d.a_cs; } else return 0;
  if (d.b_rs == 1) { b_mn = 0; b_ld = d.b_cs; } else if (d.b_cs == 1) { b_mn = 1; b_ld = d.b_rs; } else return 0;
  if ((a_ld % 8) || (b_ld % 8) || (d.ldc % 8) || (d.N % 8)) return 0;

  const int g_num_sms = tc_num_sms();
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.M = d.M; p.N = d.N; p.K = d.K; p.groups = d.groups;
  p.tiles_m = (d.M + BM - 1) / BM;
  p.tiles_n = (d.N + BN - 1) / BN;
  p.kb_total = (d.K + BK - 1) / BK;
  p.splits = 1;
  const bool hetero = epi == T_ACCUM && d.M2 > 0 && d.N2 > 0;
  if (hetero) {
    if ((d.groups & 1) || !a_mn || !b_mn || (d.M2 % 8) || (d.N2 % 8)) { set_error("gemm_tc: bad two-problem wgrad"); return 1; }
    p.hetero = 1; p.M2 = d.M2; p.N2 = d.N2;
    p.tiles_m2 = (d.M2 + BM - 1) / BM; p.tiles_n2 = (d.N2 + BN - 1) / BN;
  }
  if (epi == T_ACCUM) {
    // split-K so that the launch is ONE balanced wave: base * splits <= #SMs (a second, partial wave of a few
    // tiles would double the makespan of these long-K tiles).  Deterministic mode sizes it for the whole device, so
    // that the summation order does not depend on v2s_set_sm_limit; a limited grid walks several tiles per CTA.
    const int base = hetero ? (d.groups / 2) * (p.tiles_m * p.tiles_n + p.tiles_m2 * p.tiles_n2)
                            : d.groups * p.tiles_m * p.tiles_n;
    int s = (d.det ? tc_device_sms() : g_num_sms) / base;
    const int max_s = p.kb_total / 4 > 0 ? p.kb_total / 4 : 1;
    if (s > max_s) s = max_s;
    if (s < 1) s = 1;
    p.splits = s;
  }
  p.kb_per_split = (p.kb_total + p.splits - 1) / p.splits;
  p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;   // no empty splits
  p.total_tiles = d.groups * p.tiles_m * p.tiles_n * p.splits;
  if (hetero) {
    p.base2 = (d.groups / 2) * p.tiles_m * p.tiles_n * p.splits;
    p.total_tiles = p.base2 + (d.groups / 2) * p.tiles_m2 * p.tiles_n2 * p.splits;
  }
  p.a_mn = a_mn; p.b_mn = b_mn;
  const int combos = d.groups * p.tiles_n;
  if (epi != T_ACCUM && p.kb_total <= 3 && combos <= g_num_sms) {
    int cpc = g_num_sms / combos;
    if (cpc > p.tiles_m) cpc = p.tiles_m;
    p.b_stationary = 1;
    p.ctas_per_combo = cpc;
  }
  p.late_wait = d.late_wait ? 1 : 0;
  p.err_flag = tc_err_flag();
  p.dbg = tc_dbg_counters();
  p.dbg_flags = g_dbg_flags;
  const CUtensorMapSwizzle out_swz = out_bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  for (int g = 0; g < d.groups; ++g) {
    if (hetero && g >= d.groups / 2) {      // second problem: A [K, M2] and B [K, N2] token-major, out [M2, N2]
      V2S_TRY(get_map(&p.tmA[g], d.A[g], d.M2, d.K, d.M2, 64, BK, true, CU_TENSOR_MAP_SWIZZLE_128B));
      V2S_TRY(get_map(&p.tmB[g], d.B[g], d.N2, d.K, d.N2, 64, BK, true, CU_TENSOR_MAP_SWIZZLE_128B));
      V2S_TRY(get_map(&p.tmOut[g], d.out[g], d.N2, d.M2, d.N2, CHUNK, BM, false, out_swz));
      p.bias[g] = nullptr;
      p.rowsum[g] = d.rowsum_out[g];
      continue;
    }
    if (!a_mn) V2S_TRY(get_map(&p.tmA[g], d.A[g], d.K, d.M, a_ld, BK, BM, true, CU_TENSOR_MAP_SWIZZLE_128B));
    else V2S_TRY(get_map(&p.tmA[g], d.A[g], d.M, d.K, a_ld, 64, BK, true, CU_TENSOR_MAP_SWIZZLE_128B));
    if (!b_mn) V2S_TRY(get_map(&p.tmB[g], d.B[g], d.K, d.N, b_ld, BK, BN, true, CU_TENSOR_MAP_SWIZZLE_128B));
    else V2S_TRY(get_map(&p.tmB[g], d.B[g], d.N, d.K, b_ld, 64, BK, true, CU_TENSOR_MAP_SWIZZLE_128B));
    V2S_TRY(get_map(&p.tmOut[g], d.out[g], d.N, d.M, d.ldc, CHUNK, BM, out_bf16, out_swz));
    if (epi == T_RESID) V2S_TRY(get_map(&p.tmAux[g], d.resid[g], d.N, d.M, d.ldc, CHUNK, BM, false, CU_TENSOR_MAP_SWIZZLE_128B));
    p.bias[g] = (epi == T_ACCUM) ? nullptr : d.bias[g];
    p.rowsum[g] = (epi == T_ACCUM) ? d.rowsum_out[g] : nullptr;
    if (epi == T_RESID && d.ln_out[g] != nullptr) {
      if (d.N != BN || d.ldc != BN) { set_error("gemm_tc: fused LayerNorm needs N == 192"); return 1; }
      V2S_TRY(get_map(&p.tmOut2[g], d.ln_out[g], d.N, d.M, d.ldc, CHUNK, BM, true, CU_TENSOR_MAP_SWIZZLE_64B));
      p.ln_gamma[g] = d.ln_gamma[g]; p.ln_beta[g] = d.ln_beta[g]; p.ln_mean[g] = d.ln_mean[g]; p.ln_rstd[g] = d.ln_rstd[g];
      p.ln = 1;
    }
  }
  // deterministic mode: with one split every element already receives exactly one reduce-add (and every row sum one
  // atomic add), so only a split launch needs the slab and the in-kernel fix-up
  if (epi == T_ACCUM && d.det && p.splits > 1) {
    const int64_t slots = p.total_tiles;      // <= SMs of the device: splits > 1 implies base * splits <= SMs
    if (slots * (BM * BN + BM) > d.det->part_floats || slots / p.splits > DET_COUNTERS || slots >= 1024 || !d.det->counters) {
      set_error("gemm_tc: deterministic scratch too small for %lld partial tiles", (long long)slots);
      return 1;
    }
    p.det_slab = d.det->part;
    p.det_rowpart = d.det->part + slots * BM * BN;
    p.det_counters = d.det->counters;
    V2S_TRY(get_map(&p.tmOut2[0], p.det_slab, BN, (uint64_t)slots * BM, BN, CHUNK, BM, false, CU_TENSOR_MAP_SWIZZLE_128B));
    for (int g = 0; g < d.groups; ++g) {
      p.det_out[g] = static_cast<float*>(d.out[g]);
      p.det_ldc[g] = (hetero && g >= d.groups / 2) ? d.N2 : d.ldc;
    }
    epi = T_ACCUM_DET;
  }
  int rc;
  switch (epi) {
    case T_STORE: rc = out_bf16 ? launch_kernel<T_STORE, true>(p, lp_f16, stream) : launch_kernel<T_STORE, false>(p, lp_f16, stream); break;
    case T_RESID: rc = launch_kernel<T_RESID, false>(p, lp_f16, stream); break;
    case T_ACCUM_DET: rc = launch_kernel<T_ACCUM_DET, false>(p, lp_f16, stream); break;
    default: rc = launch_kernel<T_ACCUM, false>(p, lp_f16, stream); break;
  }
  if (rc) return rc;
  *handled = 1;
  return 0;
}

// test hook (v2s_test_gemm): which = 0 NT (A[M,K], B[N,K]), 1 NN/dgrad (A[M,K], B[K,N]),
// 2 TN/wgrad (A[K,M], B[K,N], out fp32 +=), 3 NT with fp32 out, 4 = 2 plus the bias row sums (+=) at c + M*N;
// variant: 0 = tensor-core path, 1 = SIMT reference.  bf16 operands; out bf16 for which 0/1, fp32 accumulate-into for
// which 2/4.  Deterministic mode, which 2/4: the caller's c buffer continues with the scratch a backward call takes
// from its workspace (DetScratch: DET_COUNTERS counters, then gemm_tc_det_part_floats() floats)
int gemm_tc_test(int which, const void* a, const void* b, void* c, int m, int n, int k, int variant,
                 cudaStream_t stream) {
  GemmDesc d = make_gemm_desc();
  d.M = m; d.N = n; d.K = k; d.groups = 1; d.A[0] = a; d.B[0] = b; d.out[0] = c; d.ldc = n;
  int to = 1;
  if (which == 0) { d.a_rs = k; d.a_cs = 1; d.b_rs = 1; d.b_cs = k; d.epi = EPI_STORE; }
  else if (which == 1) { d.a_rs = k; d.a_cs = 1; d.b_rs = n; d.b_cs = 1; d.epi = EPI_STORE; }
  else if (which == 2) { d.a_rs = 1; d.a_cs = m; d.b_rs = n; d.b_cs = 1; d.epi = EPI_ACCUM; to = 0; d.split_k = 1; }
  else if (which == 3) { d.a_rs = k; d.a_cs = 1; d.b_rs = 1; d.b_cs = k; d.epi = EPI_STORE; to = 0; }   // NT, fp32 out
  else if (which == 4) {
    d.a_rs = 1; d.a_cs = m; d.b_rs = n; d.b_cs = 1; d.epi = EPI_ACCUM; to = 0; d.split_k = 1;
    d.rowsum_out[0] = static_cast<float*>(c) + (int64_t)m * n;
  }
  else { set_error("gemm_tc_test: which must be 0..4"); return 1; }
  // variant: bit 0 = SIMT reference instead of the tensor-core path, bit 1 = fp16 instead of bf16 tensors
  const int t16 = (variant & 2) ? AT_F16 : AT_BF16;
  if (to) to = t16;
  if (variant & 1) return launch_gemm_simt(d, t16, t16, to, stream);
  DetScratch det = {nullptr, nullptr, 0};
  if ((which == 2 || which == 4) && tc_deterministic()) {
    if (m % 8) { set_error("gemm_tc_test: deterministic scratch needs M %% 8 == 0"); return 1; }
    det.counters = reinterpret_cast<unsigned*>(static_cast<float*>(c) + (int64_t)m * n + (which == 4 ? m : 0));
    det.part = reinterpret_cast<float*>(det.counters + DET_COUNTERS);
    det.part_floats = gemm_tc_det_part_floats();
    V2S_CUDA_OK(cudaMemsetAsync(det.counters, 0, DET_COUNTERS * sizeof(unsigned), stream));
    d.det = &det;
  }
  int handled = 0;
  V2S_TRY(launch_gemm_tc(d, t16, t16, to, stream, &handled));
  if (!handled) { set_error("gemm_tc_test: shape not handled by the tensor-core path"); return 1; }
  return 0;
}

}  // namespace v2s
