// Host-side orchestration of the grouped ViT-Tiny backbone forward / backward and of the
// heads + loss step, plus the extern "C" boundary (include/vit2spn.h).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "kernels.cuh"
#include "mlp_tc.cuh"

namespace v2s {

static thread_local char g_err[1024] = "";
int64_t g_launch_count = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- optional per-kernel-class device timing (bench.py roofline; off by default) -------------
namespace prof {
constexpr int MAX_REC = 8192;
struct Rec { int cls; double work; double bytes; cudaEvent_t a, b; };
static bool enabled = false;
static Rec recs[MAX_REC];
static int n_recs = 0;
static int n_events = 0;   // events created so far (recs[i].a/b valid for i < n_events)
static const char* names[] = {"gemm_patch", "gemm_qkv", "gemm_proj", "gemm_fc1", "gemm_fc2", "gemm_dgrad",
                              "gemm_wgrad", "attn_fwd", "attn_bwd", "ln_fwd", "ln_bwd", "colsum", "misc", "heads", "gemm_mlp_fwd",
                              "gemm_mlp_bwd", "attn_probs", "gemm_pixels", "attn_dprobs"};
enum { C_PATCH, C_QKV, C_PROJ, C_FC1, C_FC2, C_DGRAD, C_WGRAD, C_ATTN_F, C_ATTN_B, C_LN_F, C_LN_B, C_COLSUM, C_MISC,
       C_HEADS, C_MLP_F, C_MLP_B, C_ATTN_P, C_PIX, C_ATTN_DP, C_COUNT };
struct Scope {
  int idx = -1;
  cudaStream_t st;
  Scope(int cls, double work, cudaStream_t s, double bytes = 0.0) : st(s) {
    if (!enabled || n_recs >= MAX_REC) return;
    idx = n_recs++;
    if (idx >= n_events) { cudaEventCreate(&recs[idx].a); cudaEventCreate(&recs[idx].b); n_events = idx + 1; }
    recs[idx].cls = cls; recs[idx].work = work; recs[idx].bytes = bytes;
    cudaEventRecord(recs[idx].a, st);
  }
  ~Scope() { if (idx >= 0) cudaEventRecord(recs[idx].b, st); }
};
}  // namespace prof

namespace {

inline int64_t align_up(int64_t v, int64_t a = 1024) { return (v + a - 1) / a * a; }

// ---- workspace carve-up ---------------------------------------------------------------------
struct LayerStash {   // byte offsets relative to the slot base
  int64_t mean1, rstd1, xn1, qkv, ctx, lse, x_mid, mean2, rstd2, xn2, u, h;
};
struct Plan {
  int B, at;
  int64_t es;          // activation element size
  int64_t M, MP;
  int64_t heads_bytes;
  // per-group forward scratch (groups that do not save activations)
  int64_t f_patches, f_xa, f_xb, f_xn, f_qkv, f_ctx, f_h, f_bytes;
  // per-slot stash
  int64_t s_patches, s_x[NL + 1];
  LayerStash s_layer[NL];
  int64_t s_bytes;
  // per-slot backward scratch
  int64_t b_dx, b_dxlp, b_big, b_tmp, b_bytes;
};

Plan make_plan(int B, int mode) {
  Plan p;
  memset(&p, 0, sizeof(p));
  p.B = B;
  p.at = mode == V2S_MODE_BF16 ? AT_BF16 : mode == V2S_MODE_FP16 ? AT_F16 : AT_F32;   // activation type tag
  p.es = p.at ? 2 : 4;
  p.M = (int64_t)B * NT;
  p.MP = (int64_t)B * NP;
  p.heads_bytes = align_up((int64_t)B * 8192 * 4 + 4096);
  int64_t o = 0;
  auto take = [&](int64_t bytes) { int64_t r = o; o += align_up(bytes); return r; };
  p.f_patches = take(p.MP * KPE * p.es);
  p.f_xa = take(p.M * D * 4);
  p.f_xb = take(p.M * D * 4);
  p.f_xn = take(p.M * D * p.es);
  p.f_qkv = take(p.M * 3 * D * p.es);
  p.f_ctx = take(p.M * D * p.es);
  p.f_h = take(p.M * DF * p.es);
  p.f_bytes = o;
  o = 0;
  p.s_patches = take(p.MP * KPE * p.es);
  for (int l = 0; l <= NL; ++l) p.s_x[l] = take(p.M * D * 4);
  for (int l = 0; l < NL; ++l) {
    LayerStash& s = p.s_layer[l];
    s.mean1 = take(p.M * 4); s.rstd1 = take(p.M * 4);
    s.xn1 = take(p.M * D * p.es);
    s.qkv = take(p.M * 3 * D * p.es);
    s.ctx = take(p.M * D * p.es);
    s.lse = take((int64_t)B * NH * NT * 4);
    s.x_mid = take(p.M * D * 4);
    s.mean2 = take(p.M * 4); s.rstd2 = take(p.M * 4);
    s.xn2 = take(p.M * D * p.es);
    s.u = take(p.M * DF * p.es);
    s.h = take(p.M * DF * p.es);
  }
  p.s_bytes = o;
  o = 0;
  p.b_dx = take(p.M * D * 4);
  p.b_dxlp = take(p.M * D * p.es);
  p.b_big = take(p.M * DF * p.es);
  p.b_tmp = take(p.M * D * p.es);
  p.b_bytes = o;
  return p;
}

int64_t plan_total(const Plan& p, int n_groups, int n_saved) {
  return p.heads_bytes + (int64_t)n_groups * p.f_bytes + (int64_t)n_saved * (p.s_bytes + p.b_bytes);
}

int wgrad_split(int64_t rows);

// deterministic mode: scratch of a backward call at the tail of the workspace (DetScratch): the arrival counters, then
// one region for the partials of one launch at a time -- the per-CTA rows of the column reductions (at most 296 rows of at
// most 768 columns per group), the tensor-core split-K slab (one wave of fp32 tiles), or the fp32 check mode's split-K
// slabs (one per group)
int64_t det_scratch_bytes(const Plan& p, int n_saved) {
  if (n_saved <= 0) return 0;
  int64_t part = (int64_t)MAXG * 296 * DF;
  const int64_t wg = p.at ? gemm_tc_det_part_floats() : (int64_t)n_saved * wgrad_split(p.M) * DF * D;
  if (wg > part) part = wg;
  return align_up(DET_COUNTERS * sizeof(unsigned)) + align_up(part * 4);
}

int resolve_det(const Plan& p, void* ws, int64_t ws_bytes, int n_saved, DetScratch* det) {
  const int64_t bytes = det_scratch_bytes(p, n_saved);
  if (ws_bytes < plan_total(p, 0, n_saved) + bytes) {
    set_error("deterministic mode: workspace too small (%lld bytes; size it with v2s_workspace_bytes while the switch is on)",
              (long long)ws_bytes);
    return 1;
  }
  char* tail = static_cast<char*>(ws) + ((ws_bytes - bytes) & ~int64_t(1023));
  det->counters = reinterpret_cast<unsigned*>(tail);
  det->part = reinterpret_cast<float*>(tail + align_up(DET_COUNTERS * sizeof(unsigned)));
  det->part_floats = (bytes - align_up(DET_COUNTERS * sizeof(unsigned))) / 4;
  return 0;
}

// base addresses inside the workspace; regions are laid out for the maximum MAXG groups so that
// forward and backward calls agree regardless of how many groups each call carries
struct Regions {
  char* heads;
  char* fwd[MAXG];
  char* stash[MAXG];
  char* bwd[MAXG];
};

int resolve_regions(const Plan& p, void* ws, int64_t ws_bytes, int n_groups, int n_saved, Regions* r) {
  if (n_groups < 0 || n_groups > MAXG || n_saved < 0 || n_saved > MAXG) {
    set_error("workspace: bad group counts");
    return 1;
  }
  // layout: heads | stash[0..n_saved) | bwd[0..n_saved) | fwd[0..n_groups)
  // (stash first so that its addresses do not depend on n_groups)
  const int64_t need = plan_total(p, n_groups, n_saved);
  if (!ws || ws_bytes < need) {
    set_error("workspace too small: have %lld bytes, need %lld", (long long)ws_bytes, (long long)need);
    return 1;
  }
  char* base = static_cast<char*>(ws);
  if ((reinterpret_cast<uintptr_t>(base) & 1023) != 0) {
    set_error("workspace must be 1024-byte aligned");
    return 1;
  }
  r->heads = base;
  char* q = base + p.heads_bytes;
  for (int i = 0; i < MAXG; ++i) { r->stash[i] = i < n_saved ? q : nullptr; if (i < n_saved) q += p.s_bytes; }
  for (int i = 0; i < MAXG; ++i) { r->bwd[i] = i < n_saved ? q : nullptr; if (i < n_saved) q += p.b_bytes; }
  for (int i = 0; i < MAXG; ++i) { r->fwd[i] = i < n_groups ? q : nullptr; if (i < n_groups) q += p.f_bytes; }
  return 0;
}

// number of stash slots the workspace was sized for is implied by the highest slot in use:
// the Python side always allocates with n_saved = 2 (two online streams) or 1; slots index the
// stash region directly, so forward and backward agree as long as the same workspace is passed.
int max_slot(const v2s_group_t* g, int n) {
  int m = -1;
  for (int i = 0; i < n; ++i) if (g[i].slot > m) m = g[i].slot;
  return m;
}

int run_gemm(const GemmDesc& d, int ta, int tb, int to, cudaStream_t s, int cls = prof::C_MISC) {
  // algorithmic HBM bytes: both operands and the output once (+ residual / auxiliary operand, second output)
  const double ea = ta ? 2.0 : 4.0, eb = tb ? 2.0 : 4.0, eo = to ? 2.0 : 4.0;
  double bytes = 0.0;
  for (int g = 0; g < d.groups; ++g) {
    bytes += (double)d.M * d.K * ea + (double)d.N * d.K * eb + (double)d.M * d.N * eo;
    if (d.epi == EPI_BIAS_RESID) bytes += (double)d.M * d.N * 4.0 + (d.ln_out[g] ? (double)d.M * d.N * 2.0 : 0.0);
    // second 16-bit tensor: gelu'(u) operand of the dgrad epilogue; the pre-GELU store only for groups that keep it
    if (d.epi == EPI_DGELU || (d.epi == EPI_BIAS_GELU && d.out[g])) bytes += (double)d.M * d.N * 2.0;
  }
  double flops = 2.0 * d.M * d.N * (double)d.K * d.groups;
  if (d.M2 > 0) {      // two-problem wgrad launch: each half of the groups has its own shape
    bytes = 0.5 * d.groups * (((double)d.M + d.N + d.M2 + d.N2) * d.K * ea + ((double)d.M * d.N + (double)d.M2 * d.N2) * eo);
    flops = d.groups * ((double)d.M * d.N + (double)d.M2 * d.N2) * (double)d.K;
  }
  prof::Scope scope(cls, flops, s, bytes);
  int handled = 0;
  V2S_TRY(launch_gemm_tc(d, ta, tb, to, s, &handled));
  if (handled) return 0;
  if (d.det && ta != AT_F32 && d.epi == EPI_ACCUM && d.split_k > 1) {
    // the SIMT kernel's split-K adds with atomics: in deterministic mode that is an error, not a fall-back
    set_error("deterministic mode: a 16-bit split-K weight gradient the tensor-core kernel declined (M %d N %d K %d)", d.M, d.N, d.K);
    return 1;
  }
  return launch_gemm_simt(d, ta, tb, to, s);
}

inline const void* weight_ptr(const v2s_group_t& g, int at, int64_t off) {
  return at ? static_cast<const void*>(static_cast<const bf16*>(g.params_lp) + off)
            : static_cast<const void*>(g.params + off);
}

int launch_attention_fwd(const void* const* qkv, void* const* ctx, float* const* lse, int groups, int B, int at,
                         cudaStream_t s) {
  prof::Scope scope(prof::C_ATTN_F, 4.0 * B * NH * (double)NT * NT * DH * groups, s, (double)B * NT * 4 * D * 2.0 * groups);
  if (at != AT_F32) return launch_attn_fwd_tc(qkv, ctx, lse, groups, B, s, at == AT_F16);
  return launch_attn_fwd_simt(qkv, ctx, lse, groups, B, at, s);
}
int launch_attention_bwd(const void* const* qkv, const void* const* ctx, const float* const* lse,
                         const void* const* dctx, void* const* dqkv, int groups, int B, int at, cudaStream_t s) {
  prof::Scope scope(prof::C_ATTN_B, 10.0 * B * NH * (double)NT * NT * DH * groups, s, (double)B * NT * 8 * D * 2.0 * groups);
  if (at != AT_F32) return launch_attn_bwd_tc(qkv, ctx, lse, dctx, dqkv, groups, B, s, at == AT_F16);
  return launch_attn_bwd_simt(qkv, ctx, lse, dctx, dqkv, groups, B, at, s);
}

// fp32 attention probabilities of the groups that asked for them (v2s_group_outputs.attn), recomputed from qkv and lse
int launch_attention_probs(const void* const* qkv, const float* const* lse, float* const* probs, int groups, int B, int at,
                           cudaStream_t s) {
  // algorithmic bytes: Q and K read once, lse, the fp32 probabilities written once
  prof::Scope scope(prof::C_ATTN_P, 2.0 * B * NH * (double)NT * NT * DH * groups, s,
                    ((double)B * NT * 2 * D * (at ? 2.0 : 4.0) + (double)B * NH * NT * 4 + (double)B * NH * NT * NT * 4) * groups);
  if (at != AT_F32) return launch_attn_probs_tc(qkv, lse, probs, groups, B, s, at == AT_F16);
  return launch_attn_probs_simt(qkv, lse, probs, groups, B, at, s);
}

// fp32 gradient w.r.t. the attention probabilities of the groups that asked for it, dP = d ctx V^T
int launch_attention_dprobs(const void* const* qkv, const void* const* dctx, float* const* dprobs, int groups, int B, int at,
                            cudaStream_t s) {
  // algorithmic bytes: d ctx and V read once, the fp32 gradient written once
  prof::Scope scope(prof::C_ATTN_DP, 2.0 * B * NH * (double)NT * NT * DH * groups, s,
                    ((double)B * NT * 2 * D * (at ? 2.0 : 4.0) + (double)B * NH * NT * NT * 4) * groups);
  if (at != AT_F32) return launch_attn_dprobs_tc(qkv, dctx, dprobs, groups, B, s, at == AT_F16);
  return launch_attn_dprobs_simt(qkv, dctx, dprobs, groups, B, at, s);
}

// d loss / d hidden_states[k] joins the residual-stream gradient (groups whose dh entry is NULL are skipped); for k > 0 and
// with weight gradients its column sums also go to the fc2 bias gradient of block k - 1, whose output hidden_states[k] is
int add_hidden_grads(int k, const float* const* dh, float* const* dx, void* const* dxlp, const v2s_group_t* gs, int G, int B,
                     int at, const Plan& p, cudaStream_t s, const DetScratch* det, int weight_grads) {
  const float* a[MAXG]; float* o[MAXG]; void* lp[MAXG]; float* cs[MAXG]; int n = 0;
  for (int g = 0; g < G; ++g)
    if (dh[g]) {
      a[n] = dh[g]; o[n] = dx[g]; lp[n] = dxlp[g];
      cs[n] = (k > 0 && weight_grads) ? gs[g].grads + layer_off(k - 1) + L_B2 : nullptr;
      ++n;
    }
  if (!n) return 0;
  prof::Scope sc(prof::C_MISC, (double)p.M * D * (12 + p.es) * n, s);
  return launch_residual_grad_add(a, o, lp, cs, n, B, at, s, det);
}

// v2s_group_outputs checks shared by forward and backward: hidden / attn all or none, 16-byte aligned hidden states
int check_outputs(const v2s_group_outputs_t* o, int g, const char* what) {
  if (!o) return 0;
  int nh = 0, na = 0;
  for (int l = 0; l <= NL; ++l) {
    if (!o->hidden[l]) continue;
    ++nh;
    if (reinterpret_cast<uintptr_t>(o->hidden[l]) & 15) { set_error("%s: group %d: hidden[%d] is not 16-byte aligned", what, g, l); return 1; }
  }
  for (int l = 0; l < NL; ++l) na += o->attn[l] ? 1 : 0;
  if (nh != 0 && nh != NL + 1) { set_error("%s: group %d: %d of the 13 hidden[] set (all or none)", what, g, nh); return 1; }
  if (na != 0 && na != NL) { set_error("%s: group %d: %d of the 12 attn[] set (all or none)", what, g, na); return 1; }
  return 0;
}

// The residual stream of a saved group that supplied hidden[] lives in the caller's tensors, and its backward reads
// them back: remember per (workspace, stash slot) which hidden[0] the forward used, so that a backward given other
// tensors (or none, or some where the forward had none) is an error rather than a silent wrong gradient.  The same
// holds for the patch mask: the backward must be given the mask array its forward used (or none for none).
struct HiddenRec { const void* ws; int slot; const float* h0; const uint8_t* mask; };
static HiddenRec g_hidden_rec[64];
static int g_n_hidden_rec = 0;
void record_hidden(const void* ws, int slot, const float* h0, const uint8_t* mask) {
  for (int i = 0; i < g_n_hidden_rec; ++i)
    if (g_hidden_rec[i].ws == ws && g_hidden_rec[i].slot == slot) { g_hidden_rec[i].h0 = h0; g_hidden_rec[i].mask = mask; return; }
  const int i = g_n_hidden_rec < 64 ? g_n_hidden_rec++ : (int)((reinterpret_cast<uintptr_t>(ws) / 1024 + (uintptr_t)slot) % 64);
  g_hidden_rec[i] = {ws, slot, h0, mask};
}
const HiddenRec* find_hidden(const void* ws, int slot) {
  for (int i = 0; i < g_n_hidden_rec; ++i)
    if (g_hidden_rec[i].ws == ws && g_hidden_rec[i].slot == slot) return &g_hidden_rec[i];
  return nullptr;
}

int wgrad_split(int64_t rows) {
  int64_t s = rows / 1024;
  if (s < 1) s = 1;
  if (s > 16) s = 16;
  return (int)s;
}

}  // namespace

// =============================================================================================
// backbone forward
// =============================================================================================
// masks / mask_tokens (NULL, or one entry per group): the uint8 [B,196] patch mask of each group (NULL entry: none) and its
// fp32 [192] mask token, which replaces each masked patch embedding before the position embeddings are added
static int backbone_forward_impl(const v2s_group_t* gs, const v2s_group_outputs_t* outs, int G, int B, int mode,
                                 void* ws, int64_t ws_bytes, cudaStream_t st, const uint8_t* const* masks = nullptr,
                                 const float* const* mask_tokens = nullptr) {
  if (mode < V2S_MODE_FP32 || mode > V2S_MODE_FP16) { set_error("bad compute mode %d", mode); return 1; }
  if (G < 1 || G > MAXG) { set_error("backbone_forward: 1..4 groups"); return 1; }
  if (B < 1) { set_error("backbone_forward: batch must be >= 1"); return 1; }
  const Plan p = make_plan(B, mode);
  const int at = p.at;
  const int n_saved = max_slot(gs, G) + 1;
  Regions R;
  V2S_TRY(resolve_regions(p, ws, ws_bytes, G, n_saved, &R));
  for (int g = 0; g < G; ++g) {
    if (!gs[g].params || !gs[g].x) { set_error("backbone_forward: group %d has null params/x", g); return 1; }
    if (at && !gs[g].params_lp) { set_error("backbone_forward: the 16-bit modes need params_lp (group %d)", g); return 1; }
    if (gs[g].slot >= MAXG) { set_error("backbone_forward: bad slot"); return 1; }
    if (gs[g].x_format != 0 && (gs[g].x_format != 1 || !at)) {
      set_error("backbone_forward: group %d: x_format %d (1 = 16-bit patch rows, 16-bit modes only)", g, gs[g].x_format);
      return 1;
    }
    V2S_TRY(check_outputs(outs ? &outs[g] : nullptr, g, "backbone_forward"));
  }
  const int64_t M = p.M, MP = p.MP;
  // hidden_states[0..12] / attention probabilities requested by group g (NULL / false: none)
  auto hid = [&](int g) -> float* const* { return outs && outs[g].hidden[0] ? outs[g].hidden : nullptr; };
  auto want_attn = [&](int g) { return outs && outs[g].attn[0]; };
  for (int g = 0; g < G; ++g)
    if (gs[g].slot >= 0) record_hidden(ws, gs[g].slot, hid(g) ? hid(g)[0] : nullptr, masks ? masks[g] : nullptr);

  // ---- buffer resolution ----
  auto saved = [&](int g) { return gs[g].slot >= 0; };
  auto sb = [&](int g, int64_t off) -> char* { return R.stash[gs[g].slot] + off; };
  auto fb = [&](int g, int64_t off) -> char* { return R.fwd[g] + off; };

  // ---- patch embedding: im2col (shared between groups that read the same images) ----
  void* patches[MAXG];
  {
    const float* ux[MAXG]; void* uo[MAXG]; int nu = 0;
    for (int g = 0; g < G; ++g) {
      if (gs[g].x_format == 1) { patches[g] = const_cast<void*>(gs[g].x); continue; }      // the caller's patch matrix
      patches[g] = saved(g) ? sb(g, p.s_patches) : fb(g, p.f_patches);
      int dup = -1;
      // a saved group must own its copy (it outlives the call); unsaved groups may alias
      if (!saved(g))
        for (int k = 0; k < g; ++k) if (gs[k].x == gs[g].x) { dup = k; break; }
      if (dup >= 0) { patches[g] = patches[dup]; continue; }
      ux[nu] = static_cast<const float*>(gs[g].x); uo[nu] = patches[g]; ++nu;
    }
    if (nu > 0) V2S_TRY(launch_im2col(ux, uo, nu, B, at, st));
  }
  float* x_cur[MAXG];
  {
    GemmDesc d = make_gemm_desc();
    d.M = (int)MP; d.N = D; d.K = KPE; d.groups = G;
    d.a_rs = KPE; d.a_cs = 1; d.b_rs = 1; d.b_cs = KPE;
    d.ldc = D;
    const float* pp[MAXG]; const float* tok[MAXG];
    const bool two_pass = at != AT_F32;   // tensor-core GEMM into patch rows, then assemble tokens
    d.epi = two_pass ? EPI_STORE : EPI_PATCH;
    for (int g = 0; g < G; ++g) {
      x_cur[g] = hid(g) ? hid(g)[0] : reinterpret_cast<float*>(saved(g) ? sb(g, p.s_x[0]) : fb(g, p.f_xa));
      // scratch for the [B*196,192] patch rows: the x_mid buffer of block 0 (written later)
      float* tmp = reinterpret_cast<float*>(saved(g) ? sb(g, p.s_layer[0].x_mid) : fb(g, p.f_xb));
      d.A[g] = patches[g];
      d.B[g] = weight_ptr(gs[g], at, OFF_WPE);
      d.bias[g] = gs[g].params + OFF_BPE;
      d.aux[g] = gs[g].params + OFF_POS;
      d.out[g] = two_pass ? tmp : x_cur[g];
      pp[g] = gs[g].params; tok[g] = tmp;
    }
    V2S_TRY(run_gemm(d, at, at, 0, st, prof::C_PATCH));
    // masked patch rows take mask_token + pos in the kernel that writes the token rows
    if (two_pass) V2S_TRY(launch_assemble_tokens(pp, tok, x_cur, G, B, st, masks, mask_tokens));
    else V2S_TRY(launch_cls_rows(pp, x_cur, G, B, st, masks, mask_tokens));
  }

  // ---- 12 pre-LN blocks ----
  // In the 16-bit modes every LayerNorm except the first is fused into the epilogue of the kernel that produces its
  // input row (attention projection → LN2, the chained MLP → LN1 of the next block), and fc1 -> GELU -> fc2 runs as
  // one chained kernel (mlp_tc.cu).  The fp32 check mode runs the separate LayerNorm and GEMM kernels.
  const bool tc = at != AT_F32;
  const int lp_f16 = at == AT_F16 ? 1 : 0;
  for (int l = 0; l < NL; ++l) {
    const int64_t lo = layer_off(l);
    const float *xin[MAXG], *gam[MAXG], *bet[MAXG];
    void *xn[MAXG], *qkv[MAXG], *ctx[MAXG], *u[MAXG], *h[MAXG];
    float *mean[MAXG], *rstd[MAXG], *lse[MAXG], *xmid[MAXG], *xout[MAXG];
    for (int g = 0; g < G; ++g) {
      xin[g] = x_cur[g];
      if (saved(g)) {
        const LayerStash& s = p.s_layer[l];
        xn[g] = sb(g, s.xn1); qkv[g] = sb(g, s.qkv); ctx[g] = sb(g, s.ctx);
        mean[g] = (float*)sb(g, s.mean1); rstd[g] = (float*)sb(g, s.rstd1); lse[g] = (float*)sb(g, s.lse);
        xmid[g] = (float*)sb(g, s.x_mid); u[g] = sb(g, s.u); h[g] = sb(g, s.h);
        xout[g] = (float*)sb(g, p.s_x[l + 1]);
      } else {
        xn[g] = fb(g, p.f_xn); qkv[g] = fb(g, p.f_qkv); ctx[g] = fb(g, p.f_ctx);
        mean[g] = nullptr; rstd[g] = nullptr;
        // the probabilities need the log-sum-exp, and B*3*197 floats fit in f_h: in the 16-bit modes these groups use
        // f_h for nothing else (the chained MLP kernel gets d.h = NULL); in the fp32 mode fc1 writes h there only after
        // the probabilities have been computed
        lse[g] = want_attn(g) ? (float*)fb(g, p.f_h) : nullptr;
        xmid[g] = (float*)fb(g, p.f_xb); u[g] = nullptr; h[g] = fb(g, p.f_h);
        xout[g] = (float*)fb(g, p.f_xa);   // in place: x_in is dead once x_mid exists
      }
      if (hid(g)) xout[g] = hid(g)[l + 1];
      gam[g] = gs[g].params + lo + L_LN1W; bet[g] = gs[g].params + lo + L_LN1B;
    }
    if (l == 0 || !tc) {
      prof::Scope sc(prof::C_LN_F, (double)M * D * (4 + p.es) * G, st);
      V2S_TRY(launch_ln_fwd(xin, gam, bet, xn, mean, rstd, G, (int)M, at, st));
    }
    {  // fused QKV projection
      GemmDesc d = make_gemm_desc();
      d.M = (int)M; d.N = 3 * D; d.K = D; d.groups = G;
      d.a_rs = D; d.a_cs = 1; d.b_rs = 1; d.b_cs = D; d.epi = EPI_STORE; d.ldc = 3 * D;
      for (int g = 0; g < G; ++g) {
        d.A[g] = xn[g]; d.B[g] = weight_ptr(gs[g], at, lo + L_WQKV);
        d.bias[g] = gs[g].params + lo + L_BQKV; d.out[g] = qkv[g];
      }
      V2S_TRY(run_gemm(d, at, at, at, st, prof::C_QKV));
    }
    {
      const void* cq[MAXG];
      for (int g = 0; g < G; ++g) cq[g] = qkv[g];
      V2S_TRY(launch_attention_fwd(cq, ctx, lse, G, B, at, st));
      const float* al[MAXG]; float* ap[MAXG]; int na = 0;
      for (int g = 0; g < G; ++g)
        if (want_attn(g)) { cq[na] = qkv[g]; al[na] = lse[g]; ap[na] = outs[g].attn[l]; ++na; }
      if (na) V2S_TRY(launch_attention_probs(cq, al, ap, na, B, at, st));
    }
    {  // attention output projection + residual
      GemmDesc d = make_gemm_desc();
      d.M = (int)M; d.N = D; d.K = D; d.groups = G;
      d.a_rs = D; d.a_cs = 1; d.b_rs = 1; d.b_cs = D; d.epi = EPI_BIAS_RESID; d.ldc = D;
      for (int g = 0; g < G; ++g) {
        d.A[g] = ctx[g]; d.B[g] = weight_ptr(gs[g], at, lo + L_WO);
        d.bias[g] = gs[g].params + lo + L_BO; d.resid[g] = xin[g]; d.out[g] = xmid[g];
        if (tc) {     // LN2 of this block, fused
          d.ln_out[g] = saved(g) ? (void*)sb(g, p.s_layer[l].xn2) : (void*)fb(g, p.f_xn);
          d.ln_gamma[g] = gs[g].params + lo + L_LN2W; d.ln_beta[g] = gs[g].params + lo + L_LN2B;
          d.ln_mean[g] = saved(g) ? (float*)sb(g, p.s_layer[l].mean2) : nullptr;
          d.ln_rstd[g] = saved(g) ? (float*)sb(g, p.s_layer[l].rstd2) : nullptr;
        }
      }
      V2S_TRY(run_gemm(d, at, at, 0, st, prof::C_PROJ));
    }
    {
      const float* xm[MAXG];
      void* xn2[MAXG]; float *m2[MAXG], *r2[MAXG];
      for (int g = 0; g < G; ++g) {
        xm[g] = xmid[g];
        gam[g] = gs[g].params + lo + L_LN2W; bet[g] = gs[g].params + lo + L_LN2B;
        if (saved(g)) { xn2[g] = sb(g, p.s_layer[l].xn2); m2[g] = (float*)sb(g, p.s_layer[l].mean2); r2[g] = (float*)sb(g, p.s_layer[l].rstd2); }
        else { xn2[g] = fb(g, p.f_xn); m2[g] = nullptr; r2[g] = nullptr; }
      }
      if (tc) {
        // fc1 -> GELU -> fc2 + residual (+ LN1 of the next block) as ONE chained kernel: h never leaves the chip for
        // the EMA-target groups; the online groups still write u and h for the backward pass
        MlpDesc d = make_mlp_desc();
        d.mode = MLP_FWD; d.M = (int)M; d.groups = G; d.lp_f16 = lp_f16;
        double bytes = 0.0;
        for (int g = 0; g < G; ++g) {
          d.a[g] = xn2[g];
          d.w1[g] = weight_ptr(gs[g], at, lo + L_W1); d.w2[g] = weight_ptr(gs[g], at, lo + L_W2);
          d.b1[g] = gs[g].params + lo + L_B1; d.b2[g] = gs[g].params + lo + L_B2;
          d.u[g] = u[g]; d.h[g] = saved(g) ? h[g] : nullptr;
          d.resid[g] = xmid[g]; d.out[g] = xout[g];
          bytes += (double)M * D * (2 + 4 + 4) + 2.0 * D * DF * 2 + (saved(g) ? 2.0 * M * DF * 2 : 0.0);
          if (l + 1 < NL) {     // LN1 of the next block, fused
            const int64_t ln = layer_off(l + 1);
            d.ln_out[g] = saved(g) ? (void*)sb(g, p.s_layer[l + 1].xn1) : (void*)fb(g, p.f_xn);
            d.ln_gamma[g] = gs[g].params + ln + L_LN1W; d.ln_beta[g] = gs[g].params + ln + L_LN1B;
            d.ln_mean[g] = saved(g) ? (float*)sb(g, p.s_layer[l + 1].mean1) : nullptr;
            d.ln_rstd[g] = saved(g) ? (float*)sb(g, p.s_layer[l + 1].rstd1) : nullptr;
            bytes += (double)M * D * 2;
          }
        }
        prof::Scope scope(prof::C_MLP_F, 4.0 * M * D * (double)DF * G, st, bytes);
        V2S_TRY(launch_mlp_tc(d, st));
        for (int g = 0; g < G; ++g) x_cur[g] = xout[g];
        continue;
      }
      {
        prof::Scope sc(prof::C_LN_F, (double)M * D * (4 + p.es) * G, st);
        V2S_TRY(launch_ln_fwd(xm, gam, bet, xn2, m2, r2, G, (int)M, at, st));
      }
      GemmDesc d = make_gemm_desc();   // fc1 + GELU
      d.M = (int)M; d.N = DF; d.K = D; d.groups = G;
      d.a_rs = D; d.a_cs = 1; d.b_rs = 1; d.b_cs = D; d.epi = EPI_BIAS_GELU; d.ldc = DF;
      for (int g = 0; g < G; ++g) {
        d.A[g] = xn2[g]; d.B[g] = weight_ptr(gs[g], at, lo + L_W1);
        d.bias[g] = gs[g].params + lo + L_B1; d.out[g] = u[g]; d.out2[g] = h[g];
      }
      V2S_TRY(run_gemm(d, at, at, at, st, prof::C_FC1));
    }
    {  // fc2 + residual
      GemmDesc d = make_gemm_desc();
      d.M = (int)M; d.N = D; d.K = DF; d.groups = G;
      d.a_rs = DF; d.a_cs = 1; d.b_rs = 1; d.b_cs = DF; d.epi = EPI_BIAS_RESID; d.ldc = D;
      for (int g = 0; g < G; ++g) {
        d.A[g] = h[g]; d.B[g] = weight_ptr(gs[g], at, lo + L_W2);
        d.bias[g] = gs[g].params + lo + L_B2; d.resid[g] = xmid[g]; d.out[g] = xout[g];
      }
      V2S_TRY(run_gemm(d, at, at, 0, st, prof::C_FC2));
    }
    for (int g = 0; g < G; ++g) x_cur[g] = xout[g];
  }

  // ---- outputs: hidden_states[-1] and its mean over the 197 tokens ----
  {
    const float* hid[MAXG]; float* feat[MAXG]; int64_t fs[MAXG]; int nf = 0;
    for (int g = 0; g < G; ++g) {
      if (gs[g].hidden)
        V2S_CUDA_OK(cudaMemcpyAsync(gs[g].hidden, x_cur[g], (size_t)M * D * 4, cudaMemcpyDeviceToDevice, st));
      if (gs[g].feat) { hid[nf] = x_cur[g]; feat[nf] = gs[g].feat; fs[nf] = gs[g].feat_stride > 0 ? gs[g].feat_stride : D; ++nf; }
    }
    if (nf) V2S_TRY(launch_pool_fwd(hid, feat, fs, nf, B, st));
  }
  return 0;
}

// =============================================================================================
// backbone backward
// =============================================================================================
// layers [layer_lo, layer_hi) in descending order; layer_hi == NL starts from the feature / hidden-state gradient,
// layer_lo == 0 finishes with the embedding gradients.  Between two calls the residual-stream gradient lives in the
// workspace, so a full backward may be issued in several ranges (gradient all-reduce overlapped per range).
// dpix_in (whole backward only; NULL or one entry per input group): the groups with dpix_in[g] != NULL also get the fp32
// image gradient [B,3,224,224] (overwritten).  weight_grads = 0: no parameter gradient at all -- no weight-gradient GEMM,
// no bias / LayerNorm-parameter / embedding column sum -- and grads may be NULL.
// masks_in / dmask_in (whole backward only; NULL or one entry per input group): the patch mask the group's forward used,
// and, with weight gradients, d mask_token fp32 [192] (+=, NULL entry: not wanted).  A masked group's masked patch rows
// give no gradient to the patch weight, the patch bias or the pixels.
static int backbone_backward_impl(const v2s_group_t* gs_in, const v2s_group_outputs_t* outs_in, int G_in, int B, int mode,
                                  void* ws, int64_t ws_bytes, cudaStream_t st, int layer_hi, int layer_lo,
                                  float* const* dpix_in, int weight_grads, float* const* dattn_in = nullptr,
                                  const uint8_t* const* masks_in = nullptr, float* const* dmask_in = nullptr) {
  if (layer_lo < 0 || layer_hi > NL || layer_lo >= layer_hi) { set_error("backbone_backward: bad layer range [%d, %d)", layer_lo, layer_hi); return 1; }
  if (any_mask(masks_in, G_in) && (layer_lo != 0 || layer_hi != NL)) {
    set_error("backbone_backward: a masked backward covers the whole range [0, %d), not [%d, %d)", NL, layer_lo, layer_hi);
    return 1;
  }
  // keep only the groups that saved activations and want gradients
  v2s_group_t gs[MAXG];
  const v2s_group_outputs_t* os[MAXG];
  float* dpix[MAXG];
  float* const* dattn[MAXG];   // per group: NL gradients w.r.t. the attention probabilities (NULL entries skipped), or NULL
  const uint8_t* mask[MAXG]; float* dmask[MAXG];
  int G = 0;
  for (int i = 0; i < G_in && i < MAXG; ++i)
    if (gs_in[i].slot >= 0 && (gs_in[i].grads || !weight_grads)) {
      os[G] = outs_in ? &outs_in[i] : nullptr;
      dpix[G] = dpix_in ? dpix_in[i] : nullptr;
      dattn[G] = dattn_in ? dattn_in + (int64_t)i * NL : nullptr;
      mask[G] = masks_in ? masks_in[i] : nullptr;
      dmask[G] = dmask_in && weight_grads ? dmask_in[i] : nullptr;
      if (dpix[G] && gs_in[i].x_format != 0) {
        set_error("backbone_input_backward: group %d: no image gradient for 16-bit patch-row inputs (x_format 1)", i);
        return 1;
      }
      gs[G++] = gs_in[i];
    }
  if (G == 0) { set_error("backbone_backward: no group with slot >= 0 and grads"); return 1; }
  // per group: its saved hidden states (or NULL), d hidden_states[12], and the highest layer its gradient enters at
  // (NL: dfeat / dhidden[12]; k < NL: only intermediate hidden-state gradients, the highest being dhidden[k])
  float* const* hid[MAXG]; const float* dh_top[MAXG]; int top[MAXG];
  int S = -1;              // where the backward starts: the blocks [S, NL) are skipped
  for (int g = 0; g < G; ++g) {
    V2S_TRY(check_outputs(os[g], g, "backbone_backward"));
    hid[g] = os[g] && os[g]->hidden[0] ? os[g]->hidden : nullptr;
    const HiddenRec* rec = find_hidden(ws, gs[g].slot);
    if (rec && rec->h0 != (hid[g] ? hid[g][0] : nullptr)) {
      set_error("backbone_backward: group %d: hidden[] differs from the forward that filled stash slot %d", g, gs[g].slot);
      return 1;
    }
    if (rec && rec->mask != mask[g]) {
      set_error("backbone_backward: group %d: the patch mask (%s) differs from the forward that filled stash slot %d (%s); "
                "a masked forward's backward is v2s_backbone_backward_masked, over the whole range", g,
                mask[g] ? "given" : "none", gs[g].slot, rec->mask ? "masked" : "unmasked");
      return 1;
    }
    const float* dh12 = os[g] ? os[g]->dhidden[NL] : nullptr;
    if (dh12 && gs[g].dhidden) { set_error("backbone_backward: group %d sets both dhidden and outputs dhidden[12]", g); return 1; }
    dh_top[g] = dh12 ? dh12 : gs[g].dhidden;
    top[g] = (gs[g].dfeat || dh_top[g]) ? NL : -1;
    for (int k = NL - 1; top[g] < 0 && k >= 0 && os[g]; --k)
      if (os[g]->dhidden[k]) { top[g] = k; dh_top[g] = os[g]->dhidden[k]; }
    if (top[g] > S) S = top[g];
  }
  if (S < 0) {
    if (layer_hi == NL) { set_error("backbone_backward: group needs dfeat or dhidden"); return 1; }
    S = NL;                // a later range of a backward whose start the caller already issued
  }
  const Plan p = make_plan(B, mode);
  const int at = p.at;
  const int n_saved = max_slot(gs_in, G_in) + 1;
  Regions R;
  V2S_TRY(resolve_regions(p, ws, ws_bytes, 0, n_saved, &R));
  const int64_t M = p.M, MP = p.MP;
  auto sb = [&](int g, int64_t off) -> char* { return R.stash[gs[g].slot] + off; };
  auto bb = [&](int g, int64_t off) -> char* { return R.bwd[gs[g].slot] + off; };
  // deterministic mode (v2s_set_deterministic): every cross-CTA sum below runs in a fixed order through `det`
  DetScratch det_s;
  const DetScratch* det = nullptr;
  if (tc_deterministic() && weight_grads) {     // a weight-free backward has no cross-CTA sum
    V2S_TRY(resolve_det(p, ws, ws_bytes, n_saved, &det_s));
    V2S_CUDA_OK(cudaMemsetAsync(det_s.counters, 0, DET_COUNTERS * sizeof(unsigned), st));
    det = &det_s;
  }

  float* dx[MAXG]; void* dxlp[MAXG]; void* big[MAXG]; void* tmp[MAXG];
  {
    const float *df[MAXG], *dh[MAXG]; int64_t dfs[MAXG]; void* lp[MAXG];
    for (int g = 0; g < G; ++g) {
      dx[g] = (float*)bb(g, p.b_dx);
      dxlp[g] = at ? (void*)bb(g, p.b_dxlp) : (void*)dx[g];
      big[g] = bb(g, p.b_big); tmp[g] = bb(g, p.b_tmp);
      // a group whose gradient enters below S starts from zero and gets its dhidden[] added on the way down
      df[g] = S == NL ? gs[g].dfeat : nullptr; dfs[g] = gs[g].dfeat_stride > 0 ? gs[g].dfeat_stride : D;
      dh[g] = top[g] == S ? dh_top[g] : nullptr;
      lp[g] = at ? dxlp[g] : nullptr;
    }
    if (layer_hi == NL) V2S_TRY(launch_pool_bwd(df, dfs, dh, dx, lp, G, B, at, st));
  }

  const int split = wgrad_split(M);
  // dW[N_out, K_in] += dY[M, N_out]^T * X[M, K_in]   (token dimension is the reduction)
  // bias_goff >= 0: also accumulate the bias gradient (column sums of dY) — inside the tensor-core wgrad
  // kernel (extra N=16 MMA against a ones tile), or with the column-sum kernel on the SIMT path
  const bool tc = at != AT_F32;
  // remap: dy is a token-row gradient [M, n_out] of which the GEMM reads the patch rows; compact: dy is already [MP, n_out]
  auto wgrad = [&](void* const* dy, int n_out, void* const* x, int k_in, int64_t goff, bool remap,
                   int64_t bias_goff = -1, bool compact = false) -> int {
    if (!weight_grads) return 0;
    if (bias_goff >= 0 && !tc) {
      const void* src[MAXG]; float* dst[MAXG];
      for (int g = 0; g < G; ++g) { src[g] = dy[g]; dst[g] = gs[g].grads + bias_goff; }
      prof::Scope sc(prof::C_COLSUM, (double)M * n_out * p.es * G, st);
      V2S_TRY(launch_colsum(src, dst, G, (int)M, n_out, at, st, det));
    }
    GemmDesc d = make_gemm_desc();
    d.M = n_out; d.N = k_in; d.K = (remap || compact) ? (int)MP : (int)M; d.groups = G;
    d.a_rs = 1; d.a_cs = n_out; d.b_rs = k_in; d.b_cs = 1;
    d.a_remap = remap ? 2 : 0;
    d.epi = EPI_ACCUM; d.ldc = k_in; d.split_k = split; d.det = det;
    for (int g = 0; g < G; ++g) {
      d.A[g] = dy[g]; d.B[g] = x[g]; d.out[g] = gs[g].grads + goff;
      d.rowsum_out[g] = (bias_goff >= 0 && tc) ? gs[g].grads + bias_goff : nullptr;
    }
    if (det && !tc && split > 1) {
      // fp32 check mode: the splits write partial slabs, then a fixed-order sum adds them into each gradient
      const int64_t mn = (int64_t)n_out * k_in;
      if ((int64_t)G * split * mn > det->part_floats) { set_error("wgrad: deterministic scratch too small"); return 1; }
      d.epi = EPI_STORE; d.split_stride = mn;
      for (int g = 0; g < G; ++g) d.out[g] = det->part + g * split * mn;
      V2S_TRY(run_gemm(d, at, at, 0, st, prof::C_WGRAD));
      for (int g = 0; g < G; ++g)
        V2S_TRY(launch_splitk_reduce(gs[g].grads + goff, det->part + g * split * mn, nullptr, n_out, k_in, split, st, true));
      return 0;
    }
    return run_gemm(d, at, at, 0, st, prof::C_WGRAD);
  };
  // two weight gradients of one block in ONE split-K launch (tensor-core path, at most two groups): the groups of the
  // second problem follow those of the first (GemmDesc::M2 / N2).  Four ~20 us launches per block become two: one
  // ramp / one tail, longer K ranges per CTA and a third less reduce-add traffic.
  const bool merged = tc && 2 * G <= MAXG;
  auto wgrad2 = [&](void* const* dy1, int n_out1, void* const* x1, int k_in1, int64_t goff1, int64_t bias1,
                    void* const* dy2, int n_out2, void* const* x2, int k_in2, int64_t goff2, int64_t bias2) -> int {
    if (!weight_grads) return 0;
    GemmDesc d = make_gemm_desc();
    d.M = n_out1; d.N = k_in1; d.K = (int)M; d.groups = 2 * G;
    d.a_rs = 1; d.a_cs = n_out1; d.b_rs = k_in1; d.b_cs = 1;
    d.M2 = n_out2; d.N2 = k_in2;
    d.epi = EPI_ACCUM; d.ldc = k_in1; d.split_k = split; d.det = det;
    for (int g = 0; g < G; ++g) {
      d.A[g] = dy1[g]; d.B[g] = x1[g]; d.out[g] = gs[g].grads + goff1;
      d.rowsum_out[g] = bias1 >= 0 ? gs[g].grads + bias1 : nullptr;
      d.A[G + g] = dy2[g]; d.B[G + g] = x2[g]; d.out[G + g] = gs[g].grads + goff2;
      d.rowsum_out[G + g] = bias2 >= 0 ? gs[g].grads + bias2 : nullptr;
    }
    return run_gemm(d, at, at, 0, st, prof::C_WGRAD);
  };
  // dX[M, K_in] = dY[M, N_out] * W[N_out, K_in]
  // late: the kernel launched just before this one is a wgrad whose inputs this GEMM shares, and nothing the wgrad
  // touches is written here (GemmDesc::late_wait).  Without weight gradients the kernel before is the producer of dy:
  // every launch waits.
  auto dgrad = [&](void* const* dy, int n_out, int64_t woff, int k_in, void* const* out, int epi,
                   void* const* aux, bool late = false) -> int {
    GemmDesc d = make_gemm_desc();
    d.M = (int)M; d.N = k_in; d.K = n_out; d.groups = G;
    d.a_rs = n_out; d.a_cs = 1; d.b_rs = k_in; d.b_cs = 1;
    d.epi = epi; d.ldc = k_in; d.late_wait = (late && weight_grads) ? 1 : 0;
    for (int g = 0; g < G; ++g) {
      d.A[g] = dy[g]; d.B[g] = weight_ptr(gs[g], at, woff); d.out[g] = out[g];
      d.aux[g] = aux ? aux[g] : nullptr;
    }
    return run_gemm(d, at, at, at, st, prof::C_DGRAD);
  };
  auto bias_grad = [&](void* const* dy, int n, int64_t goff) -> int {
    if (!weight_grads) return 0;
    const void* src[MAXG]; float* dst[MAXG];
    for (int g = 0; g < G; ++g) { src[g] = dy[g]; dst[g] = gs[g].grads + goff; }
    prof::Scope sc(prof::C_COLSUM, (double)M * n * p.es * G, st);
    return launch_colsum(src, dst, G, (int)M, n, at, st, det);
  };

  // the intermediate hidden-state gradients below the start (dhidden[S] itself started the stream above)
  auto add_dhidden = [&](int k) -> int {
    if (k >= S) return 0;
    const float* a[MAXG];
    for (int g = 0; g < G; ++g) a[g] = os[g] ? os[g]->dhidden[k] : nullptr;
    return add_hidden_grads(k, a, dx, dxlp, gs, G, B, at, p, st, det, weight_grads);
  };
  auto x_in = [&](int g, int l) -> const float* { return hid[g] ? hid[g][l] : (const float*)sb(g, p.s_x[l]); };

  for (int l = (layer_hi < S ? layer_hi : S) - 1; l >= layer_lo; --l) {
    const int64_t lo = layer_off(l);
    const LayerStash& s = p.s_layer[l];
    V2S_TRY(add_dhidden(l + 1));
    void *u[MAXG], *h[MAXG], *xn2[MAXG], *ctx[MAXG], *qkv[MAXG], *xn1[MAXG];
    for (int g = 0; g < G; ++g) {
      u[g] = sb(g, s.u); h[g] = sb(g, s.h); xn2[g] = sb(g, s.xn2);
      ctx[g] = sb(g, s.ctx); qkv[g] = sb(g, s.qkv); xn1[g] = sb(g, s.xn1);
    }
    // Order: the backward chain is dgrad(W2) -> dgrad(W1) -> LN2' -> dgrad(Wo) -> attention' -> dgrad(Wqkv) -> LN1';
    // the wgrads are leaves.  Each dgrad is launched right after the wgrad that reads the same (older) gradient and
    // runs "late" (GemmDesc::late_wait): it does not drain that wgrad.  The mirrored order (wgrads late after the
    // chain kernels, dWo filling the attention kernel's partial last wave) measured the same or slightly slower.
    // ---- MLP ----
    if (!merged) V2S_TRY(wgrad(dxlp, D, h, DF, lo + L_W2, false));      // dW2 [192,768]
    if (l == S - 1) V2S_TRY(bias_grad(dxlp, D, lo + L_B2));                // lower blocks: fused into LN1-bwd above
    if (tc) {
      // du = (dx W2) * gelu'(u) and d xn2 = du W1 chained on chip (du is still written once: dW1 needs it)
      MlpDesc d = make_mlp_desc();
      d.mode = MLP_BWD; d.M = (int)M; d.groups = G; d.lp_f16 = at == AT_F16 ? 1 : 0; d.late_wait = (!merged && l != S - 1 && weight_grads) ? 1 : 0;
      for (int g = 0; g < G; ++g) {
        d.a[g] = dxlp[g]; d.w1[g] = weight_ptr(gs[g], at, lo + L_W1); d.w2[g] = weight_ptr(gs[g], at, lo + L_W2);
        d.u[g] = u[g]; d.h[g] = big[g]; d.out[g] = tmp[g];
      }
      {
        prof::Scope scope(prof::C_MLP_B, 4.0 * M * D * (double)DF * G, st,
                          ((double)M * D * 4 + (double)M * DF * 4 + 2.0 * D * DF * 2) * G);
        V2S_TRY(launch_mlp_tc(d, st));
      }
      if (merged)      // dW2 [192,768] (the gradient dxlp is only overwritten by LN2-bwd below) with dW1 [768,192], d b1
        V2S_TRY(wgrad2(dxlp, D, h, DF, lo + L_W2, -1, big, DF, xn2, D, lo + L_W1, lo + L_B1));
      else
        V2S_TRY(wgrad(big, DF, xn2, D, lo + L_W1, false, lo + L_B1));          // dW1 [768,192] and d b1
    } else {
      V2S_TRY(dgrad(dxlp, D, lo + L_W2, DF, big, EPI_DGELU, u, l != S - 1));    // du = (dx W2) * gelu'(u)
      V2S_TRY(wgrad(big, DF, xn2, D, lo + L_W1, false, lo + L_B1));          // dW1 [768,192] and d b1
      V2S_TRY(dgrad(big, DF, lo + L_W1, D, tmp, EPI_STORE, nullptr, true));  // d xn2
    }
    {
      const void* dy[MAXG]; const float *x[MAXG], *mu[MAXG], *rs[MAXG], *gm[MAXG];
      float *dg[MAXG], *db[MAXG], *cs[MAXG]; void* lp[MAXG];
      for (int g = 0; g < G; ++g) {
        dy[g] = tmp[g]; x[g] = (const float*)sb(g, s.x_mid); mu[g] = (const float*)sb(g, s.mean2);
        rs[g] = (const float*)sb(g, s.rstd2); gm[g] = gs[g].params + lo + L_LN2W;
        lp[g] = at ? dxlp[g] : nullptr;
        if (!weight_grads) continue;
        dg[g] = gs[g].grads + lo + L_LN2W; db[g] = gs[g].grads + lo + L_LN2B;
        cs[g] = gs[g].grads + lo + L_BO;          // d b_o = column sums of the gradient w.r.t. x_mid
      }
      { prof::Scope sc(prof::C_LN_B, (double)M * D * (12 + 2 * p.es) * G, st);
        V2S_TRY(launch_ln_bwd(dy, x, mu, rs, gm, dx, lp, weight_grads ? dg : nullptr, weight_grads ? db : nullptr, weight_grads ? cs : nullptr, G, (int)M, at, st, det)); }
    }
    // ---- attention ----
    if (!merged) V2S_TRY(wgrad(dxlp, D, ctx, D, lo + L_WO, false));        // dWo (d b_o: fused into LN2-bwd)
    V2S_TRY(dgrad(dxlp, D, lo + L_WO, D, tmp, EPI_STORE, nullptr, !merged));  // d ctx
    {
      const void *cq[MAXG], *cc[MAXG], *cd[MAXG]; const float* ls[MAXG];
      for (int g = 0; g < G; ++g) { cq[g] = qkv[g]; cc[g] = ctx[g]; cd[g] = tmp[g]; ls[g] = (const float*)sb(g, s.lse); }
      V2S_TRY(launch_attention_bwd(cq, cc, ls, cd, big, G, B, at, st));    // d qkv in `big` [M,576]
      // d loss / d probabilities = d ctx V^T, while `tmp` still holds d ctx; before the wgrad and its late-wait partner
      const void *aq[MAXG], *ad[MAXG]; float* dp[MAXG]; int n = 0;
      for (int g = 0; g < G; ++g)
        if (dattn[g] && dattn[g][l]) { aq[n] = qkv[g]; ad[n] = tmp[g]; dp[n] = dattn[g][l]; ++n; }
      if (n) V2S_TRY(launch_attention_dprobs(aq, ad, dp, n, B, at, st));
    }
    if (merged)        // dWo [192,192] (its gradient dxlp is only overwritten by LN1-bwd below) with dWqkv [576,192], d b_qkv
      V2S_TRY(wgrad2(dxlp, D, ctx, D, lo + L_WO, -1, big, 3 * D, xn1, D, lo + L_WQKV, lo + L_BQKV));
    else
      V2S_TRY(wgrad(big, 3 * D, xn1, D, lo + L_WQKV, false, lo + L_BQKV));   // dWqkv [576,192] and d b_qkv
    V2S_TRY(dgrad(big, 3 * D, lo + L_WQKV, D, tmp, EPI_STORE, nullptr, true));   // d xn1
    {
      const void* dy[MAXG]; const float *x[MAXG], *mu[MAXG], *rs[MAXG], *gm[MAXG];
      float *dg[MAXG], *db[MAXG], *cs[MAXG]; void* lp[MAXG];
      for (int g = 0; g < G; ++g) {
        dy[g] = tmp[g]; x[g] = x_in(g, l); mu[g] = (const float*)sb(g, s.mean1);
        rs[g] = (const float*)sb(g, s.rstd1); gm[g] = gs[g].params + lo + L_LN1W;
        lp[g] = at ? dxlp[g] : nullptr;
        if (!weight_grads) continue;
        dg[g] = gs[g].grads + lo + L_LN1W; db[g] = gs[g].grads + lo + L_LN1B;
        // d b_2 of the block below = column sums of the gradient w.r.t. this block's input
        cs[g] = l > 0 ? gs[g].grads + layer_off(l - 1) + L_B2 : nullptr;
      }
      { prof::Scope sc(prof::C_LN_B, (double)M * D * (12 + 2 * p.es) * G, st);
        V2S_TRY(launch_ln_bwd(dy, x, mu, rs, gm, dx, lp, weight_grads ? dg : nullptr, weight_grads ? db : nullptr, weight_grads ? cs : nullptr, G, (int)M, at, st, det)); }
    }
  }
  // ---- embeddings: d pos, d cls, d patch bias, d patch weight; the image gradient ----
  if (layer_lo == 0) {
    V2S_TRY(add_dhidden(0));
    const float* cdx[MAXG]; float* gr[MAXG]; void* pt[MAXG];
    // the groups that want the image gradient, compacted: dX_patches [B*196, 768] = dE [B*196, 192] W_pe [192, 768]
    int px[MAXG], npx = 0;
    for (int g = 0; g < G; ++g) {
      cdx[g] = dx[g]; gr[g] = gs[g].grads;
      pt[g] = gs[g].x_format == 1 ? const_cast<void*>(gs[g].x) : static_cast<void*>(sb(g, p.s_patches));
      if (dpix[g]) px[npx++] = g;
    }
    if (weight_grads) V2S_TRY(launch_embed_bwd(cdx, gr, G, B, st, det, mask, dmask));
    GemmDesc dp = make_gemm_desc();
    dp.M = (int)MP; dp.N = KPE; dp.K = D; dp.groups = npx;
    dp.a_rs = D; dp.a_cs = 1; dp.b_rs = KPE; dp.b_cs = 1; dp.ldc = KPE;
    if (tc) {          // compact the patch rows, then the ordinary tensor-core wgrad
      const void* src[MAXG];
      for (int g = 0; g < G; ++g) src[g] = dxlp[g];
      V2S_TRY(launch_gather_patch_rows(src, tmp, G, B, at, st, mask));
      if (weight_grads) {
        GemmDesc d = make_gemm_desc();
        d.M = D; d.N = KPE; d.K = (int)MP; d.groups = G;
        d.a_rs = 1; d.a_cs = D; d.b_rs = KPE; d.b_cs = 1; d.epi = EPI_ACCUM; d.ldc = KPE; d.split_k = split; d.det = det;
        for (int g = 0; g < G; ++g) { d.A[g] = tmp[g]; d.B[g] = pt[g]; d.out[g] = gs[g].grads + OFF_WPE; }
        V2S_TRY(run_gemm(d, at, at, 0, st, prof::C_WGRAD));
      }
      if (npx) {       // the image gradient straight from the epilogue; after the patch wgrad it shares its input rows
        dp.epi = EPI_PIXELS; dp.late_wait = weight_grads;
        for (int i = 0; i < npx; ++i) { dp.A[i] = tmp[px[i]]; dp.B[i] = weight_ptr(gs[px[i]], at, OFF_WPE); dp.out[i] = dpix[px[i]]; }
        V2S_TRY(run_gemm(dp, at, at, 0, st, prof::C_PIX));
      }
    } else {
      // fp32 check mode: the GEMMs read the patch rows of the token-row gradient through the row remap; with a mask they
      // read them compacted, masked rows zeroed, from `tmp` instead
      const bool masked = any_mask(mask, G);
      if (masked) {
        const void* src[MAXG];
        for (int g = 0; g < G; ++g) src[g] = dx[g];
        V2S_TRY(launch_gather_patch_rows(src, tmp, G, B, at, st, mask));
      }
      V2S_TRY(wgrad(masked ? tmp : (void* const*)dxlp, D, pt, KPE, OFF_WPE, !masked, -1, masked));
      if (npx) {       // the patch rows of the image gradient into `big`, then col2im
        const float* rows[MAXG]; float* img[MAXG];
        dp.epi = EPI_STORE; dp.a_remap = masked ? 0 : 1;
        for (int i = 0; i < npx; ++i) {
          dp.A[i] = masked ? tmp[px[i]] : (void*)dx[px[i]]; dp.B[i] = gs[px[i]].params + OFF_WPE; dp.out[i] = big[px[i]];
          rows[i] = static_cast<const float*>(big[px[i]]); img[i] = dpix[px[i]];
        }
        V2S_TRY(run_gemm(dp, at, at, 0, st, prof::C_PIX));
        prof::Scope sc(prof::C_MISC, (double)MP * KPE * 8 * npx, st);
        V2S_TRY(launch_col2im(rows, img, npx, B, st));
      }
    }
  }
  return 0;
}

// =============================================================================================
// heads + loss
// =============================================================================================
namespace {
struct HeadsBufs {
  float *a1, *y1, *a1t, *y1t, *dy1, *z, *y2, *pr, *zt, *dp, *dy2, *dz, *y2b, *part;
};
int heads_bufs(void* ws, int64_t ws_bytes, int B, HeadsBufs* hb) {
  const int64_t need = (int64_t)B * 8192 * 4;
  if (!ws || ws_bytes < need) {
    set_error("heads: workspace too small (%lld < %lld)", (long long)ws_bytes, (long long)need);
    return 1;
  }
  float* w = static_cast<float*>(ws);
  const int PH = V2S_PROJ_HID, PO = V2S_PROJ_OUT;
  hb->a1 = w;  w += (int64_t)B * PH;   // relu(f W1^T + b1)
  hb->y1 = w;  w += (int64_t)B * PH;   // a1 * dropout mask
  hb->a1t = w; w += (int64_t)B * PH;
  hb->y1t = w; w += (int64_t)B * PH;
  hb->dy1 = w; w += (int64_t)B * PH;
  hb->z = w;   w += (int64_t)B * PO;
  hb->y2 = w;  w += (int64_t)B * PO;
  hb->pr = w;  w += (int64_t)B * PO;
  hb->zt = w;  w += (int64_t)B * PO;
  hb->dp = w;  w += (int64_t)B * PO;
  hb->dy2 = w; w += (int64_t)B * PO;
  hb->dz = w;  w += (int64_t)B * PO;
  hb->y2b = w; w += (int64_t)B * PO;
  hb->part = w; w += (int64_t)B * PO * 8;   // split-K partial slabs
  return 0;
}
}  // namespace

// projection_head + prediction_head on the online features, projection_head on the target
// features (ref:ssp_vit2spn_tiny.py:153-158).  Intermediates stay in the workspace heads region.
static int heads_forward_impl(const float* hp, const float* fo, const float* ft, const float* mo, const float* mt,
                              float* pred_out, float* tgt_out, int B, void* ws, int64_t ws_bytes, cudaStream_t st) {
  if (!hp || !fo || !ft) { set_error("heads_forward: null argument"); return 1; }
  HeadsBufs hb;
  V2S_TRY(heads_bufs(ws, ws_bytes, B, &hb));
  const int PH = V2S_PROJ_HID, PO = V2S_PROJ_OUT, PI = V2S_PROJ_IN;
  auto linear = [&](const float* x, int k, int64_t woff, int64_t boff, int n, int epi, float* out, float* out2,
                    const float* mask) -> int {
    GemmDesc d = make_gemm_desc();
    d.M = B; d.N = n; d.K = k; d.a_rs = k; d.a_cs = 1; d.b_rs = 1; d.b_cs = k; d.epi = epi; d.ldc = n;
    d.A[0] = x; d.B[0] = hp + woff; d.bias[0] = hp + boff; d.out[0] = out; d.out2[0] = out2; d.mask[0] = mask;
    return launch_gemm_simt(d, 0, 0, 0, st);
  };
  // K = 1024 with a [B,128] output: too few tiles for a serial K loop → 8 K-splits into partial slabs, then a
  // fixed-order reduction that also adds the bias (deterministic, unlike atomics)
  auto linear_splitk = [&](const float* x, int k, int64_t woff, int64_t boff, int n, float* out) -> int {
    GemmDesc d = make_gemm_desc();
    d.M = B; d.N = n; d.K = k; d.a_rs = k; d.a_cs = 1; d.b_rs = 1; d.b_cs = k; d.epi = EPI_STORE; d.ldc = n;
    d.split_k = 8; d.split_stride = (int64_t)B * n;
    d.A[0] = x; d.B[0] = hp + woff; d.out[0] = hb.part;
    V2S_TRY(launch_gemm_simt(d, 0, 0, 0, st));
    return launch_splitk_reduce(out, hb.part, hp + boff, B, n, 8, st);
  };
  V2S_TRY(linear(fo, PI, H_W1, H_B1, PH, EPI_BIAS_RELU_MASK, hb.a1, hb.y1, mo));
  V2S_TRY(linear_splitk(hb.y1, PH, H_W2, H_B2, PO, hb.z));
  V2S_TRY(linear(hb.z, PO, H_W3, H_B3, PO, EPI_BIAS_RELU_MASK, hb.y2, hb.y2b, nullptr));
  V2S_TRY(linear(hb.y2, PO, H_W4, H_B4, PO, EPI_STORE, hb.pr, nullptr, nullptr));
  V2S_TRY(linear(ft, PI, H_W1, H_B1, PH, EPI_BIAS_RELU_MASK, hb.a1t, hb.y1t, mt));
  V2S_TRY(linear_splitk(hb.y1t, PH, H_W2, H_B2, PO, hb.zt));
  if (pred_out) V2S_CUDA_OK(cudaMemcpyAsync(pred_out, hb.pr, (size_t)B * PO * 4, cudaMemcpyDeviceToDevice, st));
  if (tgt_out) V2S_CUDA_OK(cudaMemcpyAsync(tgt_out, hb.zt, (size_t)B * PO * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// autograd backward of the online branch of the heads: dpred [B,128] -> head grads (+=), dfeat_online
static int heads_backward_impl(const float* hp, float* hg, const float* fo, const float* mo, const float* dpred,
                               float* dfo, int B, void* ws, int64_t ws_bytes, cudaStream_t st) {
  if (!hp || !hg || !fo || !dfo) { set_error("heads_backward: null argument"); return 1; }
  HeadsBufs hb;
  V2S_TRY(heads_bufs(ws, ws_bytes, B, &hb));
  const float* dp = dpred ? dpred : hb.dp;
  const int PH = V2S_PROJ_HID, PO = V2S_PROJ_OUT, PI = V2S_PROJ_IN;
  // deterministic mode: the weight gradients below and dfeat run without a K split (one add per element), the bias
  // gradients sum their B rows in one CTA
  const DetScratch det_rows = {nullptr, nullptr, 0};
  const DetScratch* det = tc_deterministic() ? &det_rows : nullptr;
  auto wgrad = [&](const float* dy, int n, const float* x, int k, int64_t woff) -> int {
    GemmDesc d = make_gemm_desc();
    d.M = n; d.N = k; d.K = B; d.a_rs = 1; d.a_cs = n; d.b_rs = k; d.b_cs = 1; d.epi = EPI_ACCUM; d.ldc = k;
    d.A[0] = dy; d.B[0] = x; d.out[0] = hg + woff;
    return launch_gemm_simt(d, 0, 0, 0, st);
  };
  auto bgrad = [&](const float* dy, int n, int64_t boff) -> int {
    const void* s[1] = {dy}; float* o[1] = {hg + boff};
    return launch_colsum(s, o, 1, B, n, 0, st, det);
  };
  auto dgrad = [&](const float* dy, int n, int64_t woff, int k, float* out, int epi, const float* relu_src,
                   const float* mask) -> int {
    GemmDesc d = make_gemm_desc();
    d.M = B; d.N = k; d.K = n; d.a_rs = n; d.a_cs = 1; d.b_rs = k; d.b_cs = 1; d.epi = epi; d.ldc = k;
    d.A[0] = dy; d.B[0] = hp + woff; d.out[0] = out; d.aux[0] = relu_src; d.mask[0] = mask;
    return launch_gemm_simt(d, 0, 0, 0, st);
  };
  V2S_TRY(wgrad(dp, PO, hb.y2, PO, H_W4));
  V2S_TRY(bgrad(dp, PO, H_B4));
  V2S_TRY(dgrad(dp, PO, H_W4, PO, hb.dy2, EPI_DRELU_MASK, hb.y2, nullptr));
  V2S_TRY(wgrad(hb.dy2, PO, hb.z, PO, H_W3));
  V2S_TRY(bgrad(hb.dy2, PO, H_B3));
  V2S_TRY(dgrad(hb.dy2, PO, H_W3, PO, hb.dz, EPI_STORE, nullptr, nullptr));
  V2S_TRY(wgrad(hb.dz, PO, hb.y1, PH, H_W2));
  V2S_TRY(bgrad(hb.dz, PO, H_B2));
  V2S_TRY(dgrad(hb.dz, PO, H_W2, PH, hb.dy1, EPI_DRELU_MASK, hb.a1, mo));
  V2S_TRY(wgrad(hb.dy1, PH, fo, PI, H_W1));
  V2S_TRY(bgrad(hb.dy1, PH, H_B1));
  {   // d feat = dy1 W1: K = 1024 → split-K accumulate into the zeroed [B,384] output
    V2S_CUDA_OK(cudaMemsetAsync(dfo, 0, (size_t)B * PI * sizeof(float), st));
    GemmDesc d = make_gemm_desc();
    d.M = B; d.N = PI; d.K = PH; d.a_rs = PH; d.a_cs = 1; d.b_rs = PI; d.b_cs = 1; d.epi = EPI_ACCUM; d.ldc = PI;
    d.split_k = det ? 1 : 8;
    d.A[0] = hb.dy1; d.B[0] = hp + H_W1; d.out[0] = dfo;
    V2S_TRY(launch_gemm_simt(d, 0, 0, 0, st));
  }
  return 0;
}

}  // namespace v2s

// =============================================================================================
// extern "C" boundary
// =============================================================================================
using namespace v2s;

extern "C" {

int v2s_abi_version(void) { return V2S_ABI_VERSION; }
const char* v2s_last_error(void) { return g_err; }

int v2s_init(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) { set_error("no CUDA device: %s (there is no CPU fallback)", cudaGetErrorString(e)); return 1; }
  if (device < 0 || device >= n) { set_error("device %d out of range (%d devices)", device, n); return 1; }
  cudaDeviceProp prop;
  V2S_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
    return 1;
  }
  // per-device state is created with `device` current; the caller's current device is left as it was
  int prev = 0;
  V2S_CUDA_OK(cudaGetDevice(&prev));
  V2S_CUDA_OK(cudaSetDevice(device));
  const int rc = gemm_tc_init();
  cudaSetDevice(prev);
  return rc;
}

int64_t v2s_backbone_numel(void) { return BACKBONE_NUMEL; }
int64_t v2s_backbone_active_numel(void) { return OFF_ACTIVE_END; }
int64_t v2s_heads_numel(void) { return HEADS_NUMEL; }

int v2s_backbone_layout(int64_t* o) {
  if (!o) { set_error("null"); return 1; }
  int i = 0;
  o[i++] = OFF_CLS; o[i++] = OFF_POS; o[i++] = OFF_WPE; o[i++] = OFF_BPE;
  for (int l = 0; l < NL; ++l) {
    const int64_t lo = layer_off(l);
    o[i++] = lo + L_WQKV;               o[i++] = lo + L_BQKV;            // query
    o[i++] = lo + L_WQKV + D * D;       o[i++] = lo + L_BQKV + D;        // key
    o[i++] = lo + L_WQKV + 2 * D * D;   o[i++] = lo + L_BQKV + 2 * D;    // value
    o[i++] = lo + L_WO; o[i++] = lo + L_BO;
    o[i++] = lo + L_W1; o[i++] = lo + L_B1;
    o[i++] = lo + L_W2; o[i++] = lo + L_B2;
    o[i++] = lo + L_LN1W; o[i++] = lo + L_LN1B; o[i++] = lo + L_LN2W; o[i++] = lo + L_LN2B;
  }
  o[i++] = OFF_LNF_W; o[i++] = OFF_LNF_B; o[i++] = OFF_POOL_W; o[i++] = OFF_POOL_B;
  return i == 200 ? 0 : 1;
}

int v2s_heads_layout(int64_t* o) {
  if (!o) { set_error("null"); return 1; }
  o[0] = H_W1; o[1] = H_B1; o[2] = H_W2; o[3] = H_B2; o[4] = H_W3; o[5] = H_B3; o[6] = H_W4; o[7] = H_B4;
  return 0;
}

int64_t v2s_workspace_bytes(int batch, int mode, int n_groups, int n_saved) {
  if (batch < 1 || n_groups < 0 || n_groups > MAXG || n_saved < 0 || n_saved > MAXG) return -1;
  const Plan p = make_plan(batch, mode);
  return plan_total(p, n_groups, n_saved) + (tc_deterministic() ? det_scratch_bytes(p, n_saved) : 0);
}

int v2s_backbone_forward(const v2s_group_t* groups, const v2s_group_outputs_t* outputs, int n_groups, int batch, int mode,
                         void* workspace, int64_t workspace_bytes, void* stream) {
  if (!groups) { set_error("null groups"); return 1; }
  return backbone_forward_impl(groups, outputs, n_groups, batch, mode, workspace, workspace_bytes, (cudaStream_t)stream);
}

int v2s_backbone_backward(const v2s_group_t* groups, const v2s_group_outputs_t* outputs, int n_groups, int batch,
                          int mode, void* workspace, int64_t workspace_bytes, int layer_hi, int layer_lo, void* stream) {
  if (!groups) { set_error("null groups"); return 1; }
  return backbone_backward_impl(groups, outputs, n_groups, batch, mode, workspace, workspace_bytes, (cudaStream_t)stream,
                                layer_hi, layer_lo, nullptr, 1);
}

int v2s_backbone_input_backward(const v2s_group_t* groups, const v2s_group_outputs_t* outputs, float* const* dpixels,
                                int weight_grads, int n_groups, int batch, int mode, void* workspace, int64_t workspace_bytes,
                                void* stream) {
  if (!groups || !dpixels) { set_error("backbone_input_backward: null groups / dpixels"); return 1; }
  for (int g = 0; g < n_groups && g < MAXG; ++g)
    if (dpixels[g] && (reinterpret_cast<uintptr_t>(dpixels[g]) & 15)) {
      set_error("backbone_input_backward: dpixels[%d] is not 16-byte aligned", g);
      return 1;
    }
  return backbone_backward_impl(groups, outputs, n_groups, batch, mode, workspace, workspace_bytes, (cudaStream_t)stream,
                                NL, 0, dpixels, weight_grads ? 1 : 0);
}

int v2s_backbone_backward_attn_grads(const v2s_group_t* groups, const v2s_group_outputs_t* outputs, float* const* dattn,
                                     float* const* dpixels, int weight_grads, int n_groups, int batch, int mode,
                                     void* workspace, int64_t workspace_bytes, void* stream) {
  if (!groups || !dattn) { set_error("backbone_backward_attn_grads: null groups / dattn"); return 1; }
  for (int g = 0; g < n_groups && g < MAXG; ++g) {
    for (int l = 0; l < NL; ++l)
      if (reinterpret_cast<uintptr_t>(dattn[g * NL + l]) & 3) {
        set_error("backbone_backward_attn_grads: dattn[%d] (group %d, block %d) is not 4-byte aligned", g * NL + l, g, l);
        return 1;
      }
    if (dpixels && (reinterpret_cast<uintptr_t>(dpixels[g]) & 15)) {
      set_error("backbone_backward_attn_grads: dpixels[%d] is not 16-byte aligned", g);
      return 1;
    }
  }
  return backbone_backward_impl(groups, outputs, n_groups, batch, mode, workspace, workspace_bytes, (cudaStream_t)stream,
                                NL, 0, dpixels, weight_grads ? 1 : 0, dattn);
}

int v2s_backbone_forward_masked(const v2s_group_t* groups, const v2s_group_outputs_t* outputs, const uint8_t* const* masks,
                                const float* const* mask_tokens, int n_groups, int batch, int mode, void* workspace,
                                int64_t workspace_bytes, void* stream) {
  if (!groups) { set_error("backbone_forward_masked: null groups"); return 1; }
  for (int g = 0; masks && g < n_groups && g < MAXG; ++g) {
    if (!masks[g]) continue;
    if (!mask_tokens || !mask_tokens[g]) { set_error("backbone_forward_masked: group %d has a mask but no mask token", g); return 1; }
    if (reinterpret_cast<uintptr_t>(mask_tokens[g]) & 15) {
      set_error("backbone_forward_masked: mask_tokens[%d] is not 16-byte aligned", g);
      return 1;
    }
  }
  return backbone_forward_impl(groups, outputs, n_groups, batch, mode, workspace, workspace_bytes, (cudaStream_t)stream,
                               masks, mask_tokens);
}

int v2s_backbone_backward_masked(const v2s_group_t* groups, const v2s_group_outputs_t* outputs, const uint8_t* const* masks,
                                 float* const* dmask_tokens, float* const* dattn, float* const* dpixels, int weight_grads,
                                 int n_groups, int batch, int mode, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!groups) { set_error("backbone_backward_masked: null groups"); return 1; }
  for (int g = 0; g < n_groups && g < MAXG; ++g) {
    for (int l = 0; dattn && l < NL; ++l)
      if (reinterpret_cast<uintptr_t>(dattn[g * NL + l]) & 3) {
        set_error("backbone_backward_masked: dattn[%d] (group %d, block %d) is not 4-byte aligned", g * NL + l, g, l);
        return 1;
      }
    if (dpixels && (reinterpret_cast<uintptr_t>(dpixels[g]) & 15)) {
      set_error("backbone_backward_masked: dpixels[%d] is not 16-byte aligned", g);
      return 1;
    }
    if (dmask_tokens && (reinterpret_cast<uintptr_t>(dmask_tokens[g]) & 3)) {
      set_error("backbone_backward_masked: dmask_tokens[%d] is not 4-byte aligned", g);
      return 1;
    }
  }
  return backbone_backward_impl(groups, outputs, n_groups, batch, mode, workspace, workspace_bytes, (cudaStream_t)stream,
                                NL, 0, dpixels, weight_grads ? 1 : 0, dattn, masks, dmask_tokens);
}

int v2s_heads_loss_fwd_bwd(const float* head_params, float* head_grads, const float* feat_online,
                           const float* feat_target, const float* mask_online, const float* mask_target,
                           float* dfeat_online, float* pred, float* target_proj, float* loss, int batch,
                           int accumulation_steps, float grad_scale, const float* grad_scale_dev, int with_backward,
                           void* workspace, int64_t workspace_bytes, void* stream) {
  if (batch < 1 || accumulation_steps < 1) { set_error("heads: bad batch/accumulation_steps"); return 1; }
  if (!loss) { set_error("heads: null loss"); return 1; }
  const cudaStream_t st = (cudaStream_t)stream;
  V2S_TRY(heads_forward_impl(head_params, feat_online, feat_target, mask_online, mask_target, pred, target_proj, batch,
                             workspace, workspace_bytes, st));
  HeadsBufs hb;
  V2S_TRY(heads_bufs(workspace, workspace_bytes, batch, &hb));
  V2S_TRY(launch_cosine_loss(hb.pr, hb.zt, loss, with_backward ? hb.dp : nullptr, batch, accumulation_steps, grad_scale,
                             st, grad_scale_dev));
  if (!with_backward) return 0;
  return heads_backward_impl(head_params, head_grads, feat_online, mask_online, nullptr, dfeat_online, batch, workspace,
                             workspace_bytes, st);
}

int v2s_heads_forward(const float* head_params, const float* feat_online, const float* feat_target,
                      const float* mask_online, const float* mask_target, float* pred, float* target_proj, int batch,
                      void* workspace, int64_t workspace_bytes, void* stream) {
  if (batch < 1) { set_error("heads_forward: bad batch"); return 1; }
  return heads_forward_impl(head_params, feat_online, feat_target, mask_online, mask_target, pred, target_proj, batch,
                            workspace, workspace_bytes, (cudaStream_t)stream);
}

int v2s_heads_backward(const float* head_params, float* head_grads, const float* feat_online,
                       const float* mask_online, const float* dpred, float* dfeat_online, int batch, void* workspace,
                       int64_t workspace_bytes, void* stream) {
  if (batch < 1 || !dpred) { set_error("heads_backward: bad argument"); return 1; }
  return heads_backward_impl(head_params, head_grads, feat_online, mask_online, dpred, dfeat_online, batch, workspace,
                             workspace_bytes, (cudaStream_t)stream);
}

int v2s_cosine_loss(const float* pred, const float* target_proj, float* loss, float* dpred, int batch,
                    int accumulation_steps, float grad_scale, void* stream) {
  if (!pred || !target_proj || !loss || batch < 1 || accumulation_steps < 1) { set_error("cosine_loss: bad argument"); return 1; }
  return launch_cosine_loss(pred, target_proj, loss, dpred, batch, accumulation_steps, grad_scale, (cudaStream_t)stream);
}

int v2s_infonce_loss(const float* pred, const float* keys, float* loss, float* row_loss, float* dpred, int batch,
                     int n_keys, int64_t label_offset, float temperature, int accumulation_steps, float grad_scale,
                     const float* grad_scale_dev, void* stream) {
  if (!pred || !keys || !loss || !row_loss || batch < 1 || accumulation_steps < 1) { set_error("infonce_loss: bad argument"); return 1; }
  return launch_infonce_loss(pred, keys, loss, row_loss, dpred, batch, n_keys, label_offset, temperature, accumulation_steps,
                             grad_scale, (cudaStream_t)stream, grad_scale_dev);
}

int v2s_dropout_mask(float* mask, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream) {
  if (!mask || n < 0 || p < 0.f || p >= 1.f) { set_error("dropout_mask: bad argument"); return 1; }
  if (n == 0) return 0;
  return launch_dropout_mask(mask, n, p, seed, offset, (cudaStream_t)stream);
}

static int check_ranges(const v2s_range_t* ranges, int n_ranges) {
  for (int i = 0; i < n_ranges; ++i)
    if ((reinterpret_cast<uintptr_t>(ranges[i].params) | reinterpret_cast<uintptr_t>(ranges[i].grads) |
         reinterpret_cast<uintptr_t>(ranges[i].exp_avg) | reinterpret_cast<uintptr_t>(ranges[i].exp_avg_sq)) & 15) {
      set_error("adam: range %d is not 16-byte aligned", i);
      return 1;
    }
  return 0;
}

int v2s_adam_step(const v2s_range_t* ranges, int n_ranges, int64_t step, double lr, double beta1, double beta2,
                  double eps, double weight_decay, double grad_scale, int lp_format, void* stream) {
  if (!ranges || step < 1) { set_error("adam: bad argument"); return 1; }
  V2S_TRY(check_ranges(ranges, n_ranges));
  return launch_adam(ranges, n_ranges, step, lr, beta1, beta2, eps, weight_decay, grad_scale, (cudaStream_t)stream,
                     lp_format == V2S_LP_FP16);
}

int v2s_adam_step_amp(const v2s_range_t* ranges, int n_ranges, float* state8, double lr, double beta1, double beta2,
                      double eps, double weight_decay, double grad_multiplier, const float* grad_scale_dev,
                      const float* found_inf_dev, int lp_format, int advance_step, void* stream) {
  if (!ranges || !state8) { set_error("adam_amp: bad argument"); return 1; }
  V2S_TRY(check_ranges(ranges, n_ranges));
  return launch_adam_amp(ranges, n_ranges, state8, lr, beta1, beta2, eps, weight_decay, grad_multiplier, grad_scale_dev,
                         found_inf_dev, lp_format == V2S_LP_FP16, advance_step, (cudaStream_t)stream);
}

int v2s_ema_update(float* const* targets, const float* const* onlines, void* const* targets_lp, int n_pairs,
                   int64_t numel, double momentum, int lp_format, void* stream) {
  if (!targets || !onlines) { set_error("ema: null"); return 1; }
  return launch_ema(targets, onlines, targets_lp, n_pairs, numel, momentum, (cudaStream_t)stream, lp_format == V2S_LP_FP16);
}

int v2s_cast_lp(const float* src, void* dst, int64_t numel, int lp_format, void* stream) {
  if (!src || !dst || numel < 0) { set_error("cast: bad argument"); return 1; }
  if (numel == 0) return 0;
  return launch_cast_lp(src, dst, numel, (cudaStream_t)stream, lp_format == V2S_LP_FP16);
}

int v2s_preprocess_u8_patches(const uint8_t* src, void* patch_rows, int n_images, int lp_format, void* stream) {
  if (!src || !patch_rows || n_images < 1 || (lp_format != 0 && lp_format != 1)) { set_error("preprocess_patches: bad argument"); return 1; }
  return launch_preprocess_u8_patches(src, patch_rows, n_images, lp_format, (cudaStream_t)stream);
}

int v2s_preprocess_u8(const uint8_t* src, float* dst, int batch, void* stream) {
  if (!src || !dst || batch < 1) { set_error("preprocess: bad argument"); return 1; }
  return launch_preprocess_u8(src, dst, batch, (cudaStream_t)stream);
}

int v2s_augment_finish_u8(const uint8_t* src, int n, int in_size, const int32_t* bounds, const int32_t* coefs, int ksize,
                          const float* k1d, const int32_t* erase, const float* host_mean3, const float* host_std3,
                          float* dst, void* stream) {
  if (!src || !bounds || !coefs || !host_mean3 || !host_std3 || !dst || n < 1) { set_error("augment: bad argument"); return 1; }
  return launch_augment_finish(src, n, in_size, bounds, coefs, ksize, k1d, erase, host_mean3, host_std3, dst,
                               (cudaStream_t)stream);
}

int64_t v2s_launch_count(void) { return g_launch_count; }

int v2s_set_sm_limit(int n_sms) {
  tc_set_sm_limit(n_sms);
  return 0;
}

int v2s_set_deterministic(int on) {
  tc_set_deterministic(on);
  return 0;
}

int v2s_prof_enable(int on) {
  prof::enabled = on != 0;
  prof::n_recs = 0;
  return 0;
}

// writes one line per kernel class: "<name> <launches> <total_ms> <work> <bytes>" (work = FLOPs for
// GEMM/attention classes, bytes for the memory-bound ones; bytes = algorithmic HBM bytes); synchronises.
int v2s_prof_report(char* host_buf, int64_t buf_bytes) {
  if (!host_buf || buf_bytes < 64) { set_error("prof_report: buffer too small"); return 1; }
  V2S_CUDA_OK(cudaDeviceSynchronize());
  double ms[prof::C_COUNT] = {0}, work[prof::C_COUNT] = {0}, byt[prof::C_COUNT] = {0};
  int cnt[prof::C_COUNT] = {0};
  for (int i = 0; i < prof::n_recs; ++i) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, prof::recs[i].a, prof::recs[i].b) != cudaSuccess) continue;
    ms[prof::recs[i].cls] += t; work[prof::recs[i].cls] += prof::recs[i].work; cnt[prof::recs[i].cls]++;
    byt[prof::recs[i].cls] += prof::recs[i].bytes > 0 ? prof::recs[i].bytes : prof::recs[i].work;
  }
  int64_t off = 0;
  host_buf[0] = 0;
  for (int c = 0; c < prof::C_COUNT; ++c) {
    if (!cnt[c]) continue;
    int n = snprintf(host_buf + off, (size_t)(buf_bytes - off), "%s %d %.6f %.6e %.6e\n", prof::names[c], cnt[c], ms[c], work[c], byt[c]);
    if (n < 0 || off + n >= buf_bytes) break;
    off += n;
  }
  prof::n_recs = 0;
  return 0;
}

// test hook: which = 0 forward (qkv -> ctx, lse), 1 backward (qkv, ctx, lse, dctx -> dqkv), 2 probabilities (qkv, lse ->
// fp32 [batch,3,197,197] in ctx), 3 their gradient (qkv, dctx -> fp32 [batch,3,197,197] in ctx);
// variant 0 = tensor-core kernels, 1 = SIMT reference kernels; bf16 tensors, one backbone
int v2s_test_attention(int which, const void* qkv, void* ctx, float* lse, const void* dctx, void* dqkv, int batch,
                       int variant, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const void* cq[1] = {qkv}; void* cc[1] = {ctx}; float* ls[1] = {lse};
  const void* cctx[1] = {ctx}; const float* cls[1] = {lse}; const void* cd[1] = {dctx}; void* dq[1] = {dqkv};
  // variant: bit 0 = SIMT reference kernels, bit 1 = fp16 instead of bf16 tensors
  const int f16 = (variant & 2) ? 1 : 0, at = f16 ? AT_F16 : AT_BF16;
  if (which == 0) {
    if (variant & 1) return launch_attn_fwd_simt(cq, cc, ls, 1, batch, at, st);
    return launch_attn_fwd_tc(cq, cc, ls, 1, batch, st, f16);
  }
  if (which == 1) {
    if (variant & 1) return launch_attn_bwd_simt(cq, cctx, cls, cd, dq, 1, batch, at, st);
    return launch_attn_bwd_tc(cq, cctx, cls, cd, dq, 1, batch, st, f16);
  }
  if (which == 2) {
    float* pr[1] = {static_cast<float*>(ctx)};
    if (variant & 1) return launch_attn_probs_simt(cq, cls, pr, 1, batch, at, st);
    return launch_attn_probs_tc(cq, cls, pr, 1, batch, st, f16);
  }
  if (which == 3) {
    float* dp[1] = {static_cast<float*>(ctx)};
    if (variant & 1) return launch_attn_dprobs_simt(cq, cd, dp, 1, batch, at, st);
    return launch_attn_dprobs_tc(cq, cd, dp, 1, batch, st, f16);
  }
  set_error("v2s_test_attention: which must be 0, 1, 2 or 3");
  return 1;
}

int v2s_debug_flag(void) { return gemm_tc_error_flag(); }
int v2s_debug_counters(int64_t* host32) { return gemm_tc_debug_counters(reinterpret_cast<long long*>(host32)); }

int v2s_test_mlp(int mode, const void* a, const void* w1, const void* w2, const float* b1, const float* b2, void* u,
                 void* h, const float* resid, void* out, void* ln_out, const float* ln_gamma, const float* ln_beta,
                 float* ln_mean, float* ln_rstd, int m, int lp_f16, void* stream) {
  MlpDesc d = make_mlp_desc();
  d.mode = mode; d.M = m; d.groups = 1; d.lp_f16 = lp_f16;
  d.a[0] = a; d.w1[0] = w1; d.w2[0] = w2; d.b1[0] = b1; d.b2[0] = b2; d.u[0] = u; d.h[0] = h; d.resid[0] = resid;
  d.out[0] = out; d.ln_out[0] = ln_out; d.ln_gamma[0] = ln_gamma; d.ln_beta[0] = ln_beta; d.ln_mean[0] = ln_mean;
  d.ln_rstd[0] = ln_rstd;
  return launch_mlp_tc(d, (cudaStream_t)stream);
}

int v2s_test_gemm(int which, const void* a, const void* b, void* c, int m, int n, int k, int variant, void* stream) {
  return gemm_tc_test(which, a, b, c, m, n, k, variant, (cudaStream_t)stream);
}

}  // extern "C"
