// C-ABI entry points declared in include/gnnjet_b200.h: argument checks, dispatch on precision,
// error reporting.  No torch types; raw device pointers + sizes + cudaStream_t.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "gj_common.cuh"

static thread_local char g_err[512] = "";

void gj_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// programmatic dependent launch of the step's kernel chain (gj_common.cuh): GJ_PDL forces a mode, unset = the default policy
int gj_pdl_mode() { static const int v = getenv("GJ_PDL") ? atoi(getenv("GJ_PDL")) : -1; return v; }

// bitwise-reproducible parameter gradients in the bf16 mode (gj_set_deterministic): read by the backward edge launchers
static int g_deterministic = 0;
bool gj_deterministic() { return g_deterministic != 0; }

int gj_num_sms() {
  static int sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (sms[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    sms[dev] = v;
  }
  return sms[dev];
}

// launchers implemented in the kernel translation units
int gj_node_pre_fwd(const MPLayout&, const float*, const float*, float*, cudaStream_t);
size_t gj_node_pre_bwd_ws_floats(const MPLayout&);
int gj_node_pre_bwd(const MPLayout&, const float*, const float*, const float*, float*, float*, float*, cudaStream_t);
bool gj_node_pre_bwd_tc_supported(const MPLayout&);
size_t gj_node_pre_bwd_tc_ws_floats(const MPLayout&);
int gj_node_pre_bwd_tc(const MPLayout&, const float*, const float*, const float*, float*, float*, int*, cudaStream_t);
int gj_reduce_pre_partials(const MPLayout&, const float*, int, float*, cudaStream_t);
int gj_node_post_fwd(const MPLayout&, const float*, const float*, const float*, float*, cudaStream_t);
size_t gj_node_post_bwd_ws_floats(const MPLayout&);
bool gj_node_post_bwd_tc_supported(const MPLayout&);
size_t gj_node_post_bwd_tc_ws_floats(const MPLayout&);
int gj_node_post_bwd_tc(const MPLayout&, const float*, const float*, const float*, const float*, float*, float*, float*, int*, float*, cudaStream_t);
int gj_reduce_step_partials(const MPLayout&, const float*, int, const float*, int, const float*, int, float*, cudaStream_t);
int gj_reduce_partials(const float*, int, int, float*, cudaStream_t);
int gj_node_post_bwd(const MPLayout&, const float*, const float*, const float*, const float*, float*, float*, float*, float*,
                     cudaStream_t);
int gj_edge_grid(int);
int gj_edge_fwd_simt(MPLayout, const float*, const float*, const float*, float*, cudaStream_t);
int gj_edge_bwd_simt(MPLayout, const float*, const float*, const float*, const float*, float*, float*, float*, float*,
                     cudaStream_t);
int gj_edge_fwd_tc(MPLayout, const float*, const float*, const float*, float*, cudaStream_t);
bool gj_fwd2_supported(const MPLayout&);
size_t gj_fwd2_ws_floats(const MPLayout&);
int gj_edge_fwd2(const MPLayout&, const float*, const float*, const float*, float*, float*, float*, float*, cudaStream_t, bool, bool);
int gj_pack_batch2(int, const MPLayout*, const float* const*, float* const*, cudaStream_t);
size_t gj_bwd2_part_floats(const MPLayout&);
int gj_bwd2_nparts(const MPLayout&);
int gj_node_pre_bwd_tc_nparts(const MPLayout&);
int gj_node_post_bwd_tc_nparts(const MPLayout&);
int gj_reduce_steps_partials(int, const MPLayout*, const float* const*, const int*, const float* const*, const int*, const float* const*,
                             const int*, float* const*, cudaStream_t);
size_t gj_wimage_floats();
void gj_fwd2_plan(const MPLayout&, int*, int*);
void gj_bwd2_plan(const MPLayout&, int*, int*);
bool gj_bwd2_supported(const MPLayout&);
size_t gj_bwd2_ws_floats(const MPLayout&);
int gj_edge_bwd2(const MPLayout&, const float*, const float*, const float*, const float*, float*, float*, float*, float*, float*, float*, bool,
                 cudaStream_t, int, const float**, int*, float*);
size_t gj_edge_bwd_tc_ws_floats(const MPLayout&);
int gj_edge_bwd_tc(MPLayout, const float*, const float*, const float*, const float*, float*, float*, float*, float*,
                   cudaStream_t);
int gj_umma_selftest_launch(int, int, int, int, int, const float*, const float*, float*, cudaStream_t);
bool gj_edge3_supported(const MPLayout&);
size_t gj_edge3_wimage_floats(const MPLayout&);
size_t gj_edge3_fwd_ws_floats(const MPLayout&);
size_t gj_edge3_bwd_ws_floats(const MPLayout&);
int gj_edge_fwd3(const MPLayout&, const float*, const float*, const float*, float*, float*, float*, float*, cudaStream_t);
int gj_edge_bwd3(const MPLayout&, const float*, const float*, const float*, const float*, float*, float*, float*, float*, float*, float*, bool,
                 cudaStream_t);
bool gj_node_generic_fits(const MPLayout&);
bool gj_edge_simt_fits(MPLayout, const float*);
bool gj_edge_tc_fits(MPLayout);
size_t gj_edge_mat_ws_floats(const MPLayout&, bool);
int gj_edge_mat_launches(const MPLayout&, bool);
int gj_edge_mat_fwd(const MPLayout&, const float*, const float*, const float*, float*, float*, int, cudaStream_t);
int gj_edge_mat_bwd(const MPLayout&, const float*, const float*, const float*, const float*, float*, float*, float*, float*, int, cudaStream_t);
size_t gj_dense_ws_floats(const MPLayout&, bool);
int gj_dense_launches(const MPLayout&, bool);
int gj_dense_pre_fwd(const MPLayout&, const float*, const float*, float*, int, cudaStream_t);
size_t gj_dense_ysave_floats(const MPLayout&);
int gj_dense_post_fwd(const MPLayout&, const float*, const float*, const float*, float*, float*, float*, int, cudaStream_t);
int gj_dense_post_bwd(const MPLayout&, const float*, const float*, const float*, const float*, float*, float*, float*, float*, const float*, int,
                      cudaStream_t);
int gj_dense_pre_bwd(const MPLayout&, const float*, const float*, const float*, float*, float*, float*, int, cudaStream_t);
void gj_tc_plan_info(MPLayout, int*);
int gj_chamfer_launch(int, int, int, int, int, float, float, const float*, const float*, float*, float*, float*, cudaStream_t);
int gj_pair_min_dist_launch(int, int, int, int, int, const float*, const float*, float*, float*, cudaStream_t);
int gj_assignment_launch(int, int, int, int, const float*, const float*, int*, float*, cudaStream_t);
int gj_emd_check(int, int, int, float, float, int);
int gj_emd_launch(int, int, int, const float*, const float*, float, float, int, double*, double*, float*, double*, int*, cudaStream_t);
size_t gj_emd_loss_ws_bytes(int);
int gj_emd_loss_check(int, int, int, int, float, float, int, size_t);
int gj_emd_loss_launch(int, int, int, int, const float*, const float*, float, float, int, float, float*, float*, float*, void*, cudaStream_t);
size_t gj_hmse_ws_bytes(int);
int gj_hmse_check(int, int, int, int, size_t);
int gj_hmse_launch(int, int, int, int, const float*, const float*, float, float*, float*, int*, void*, cudaStream_t);
int gj_linear_fwd_launch(int, int, int, const float*, const float*, const float*, float*, cudaStream_t);
size_t gj_linear_bwd_ws_bytes(int, int, int);
int gj_linear_bwd_launch(int, int, int, const float*, const float*, const float*, float*, float*, float*, void*, size_t, cudaStream_t);
int gj_adam_launch(float*, const float*, float*, float*, size_t, float, float, float, float, int, float, float, float,
                   cudaStream_t);
size_t gj_norms_ws_bytes(size_t);
int gj_optimizer_launch(int, float*, const float*, float*, float*, size_t, float, float, float, float, float, float, float, cudaStream_t);
int gj_nonfinite_flag_launch(const float*, int, float*, cudaStream_t);
int gj_nonfinite_check_launch(const float*, size_t, int*, float*, cudaStream_t);
int gj_adam_guarded_launch(float*, const float*, float*, float*, size_t, float, float, float, float, const int*, int*, float, float, float,
                           cudaStream_t);
int gj_optimizer_guarded_launch(int, float*, const float*, float*, float*, size_t, float, float, float, float, float, float, float,
                                const int*, int*, cudaStream_t);
int gj_norms_launch(const float*, size_t, float*, void*, size_t, cudaStream_t);
int gj_latent_mean_fwd_launch(int, int, int, const float*, float*, cudaStream_t);
int gj_latent_mean_bwd_launch(int, int, int, const float*, float*, cudaStream_t);
int gj_latent_extreme_fwd_launch(int, int, int, int, const float*, float*, cudaStream_t);
int gj_latent_extreme_bwd_launch(int, int, int, const float*, const float*, const float*, float*, cudaStream_t);
int gj_out_transform_launch(size_t, int, int, int, float, const float*, const float*, float*, cudaStream_t);
size_t gj_mse_ws_bytes();
int gj_mse_launch(size_t, double, const float*, const float*, float*, float*, void*, size_t, cudaStream_t);

extern "C" {

const char* gj_last_error(void) { return g_err; }
int32_t gj_abi_version(void) { return 1; }
const char* gj_build_arch(void) { return "sm_100a"; }

int32_t gj_set_deterministic(int32_t on) {
  const int prev = g_deterministic;
  g_deterministic = on != 0;
  return prev;
}

// The kernels one message-passing step runs, resolved once per (layout, precision) by step_plan(); every launch sequence,
// workspace plan and launch count below reads it.  Edge kernels: SIMT (edge_simt.cu), first-generation tcgen05 (edge_tc.cu),
// the second- and third-generation fused kernels (edge_fwd2.cu / edge_bwd2.cu, edge3.cu), and the edge MLP as generic GEMMs
// over the materialised edge rows of a chunk of jets (dense.cu).
enum StepEdge { EDGE_SIMT, EDGE_TC1, EDGE_TC2, EDGE_TC3, EDGE_MAT };
struct StepPath {
  int precision;
  StepEdge edge;
  bool dense_node;      // the node level (P|Q projections, node MLP and their adjoints) as generic GEMMs (dense.cu)
  bool post_tc, pre_tc;      // the node-MLP adjoint / the projections' adjoint on tcgen05 (node_tc.cu); EDGE_TC2 only
  // the backward with both node-level adjoints on tcgen05: their partials and the edge kernel's are reduced together
  bool tail_fused() const { return post_tc && pre_tc; }
  // the fused kernels can keep P|Q, the parameter image and the pair distances for the backward (gj_mp_step_saved_bytes)
  bool saves() const { return edge == EDGE_TC2 || edge == EDGE_TC3; }
};

static StepPath resolve_path(const MPLayout& L, int precision) {
  StepPath p = {precision, EDGE_MAT, false, false, false};
  const bool tc = precision == GJ_PREC_BF16 && L.Le > 1;      // a one-layer edge network runs the SIMT kernels in either mode
  if (tc && gj_fwd2_supported(L) && gj_bwd2_supported(L)) p.edge = EDGE_TC2;      // forward and backward cover the same widths
  else if (tc && gj_edge3_supported(L)) p.edge = EDGE_TC3;      // two-layer edge networks [H, H], H = 64 / 128 (BASELINE config 5)
  else if (tc ? gj_edge_tc_fits(L) : gj_edge_simt_fits(L, nullptr)) p.edge = tc ? EDGE_TC1 : EDGE_SIMT;
  // else EDGE_MAT: the widths no edge kernel has a plan for (e.g. edge_sizes [[256, 256]])
  const bool tc2 = p.edge == EDGE_TC2;
  p.post_tc = tc2 && gj_node_post_bwd_tc_supported(L);
  p.pre_tc = tc2 && gj_node_pre_bwd_tc_supported(L);
  // Generic-GEMM node level wherever a node-level weight matrix does not fit the fused node kernels' shared-memory plans, and
  // for wide layers (BASELINE config 5: H >= 64), where the GEMM formulation -- tcgen05 in the bf16 mode -- is the faster one
  int wmax = L.H > L.E[0] ? L.H : L.E[0];
  for (int m = 0; m < L.Ln; ++m) if (L.O[m] > wmax) wmax = L.O[m];
  p.dense_node = !tc2 && (p.edge == EDGE_MAT || !gj_node_generic_fits(L) || wmax >= 64);
  return p;
}

// Validates the descriptor, fills the layout and resolves the step's path.  An entry point that reports errors passes its name
// (a chain entry point also the step's index) and gets "<who>: <reason>" as the last error; the size queries pass none.
static int step_plan(const gj_mp_desc* d, MPLayout* L, StepPath* p, const char* who = nullptr, int step = -1) {
  const char* why;
  if (int rc = gj_fill_arch(d, L, &why)) {
    if (who && step >= 0) gj_set_error("%s: %s (step %d)", who, why, step);
    else if (who) gj_set_error("%s: %s", who, why);
    return rc;
  }
  *p = resolve_path(*L, d->precision);
  return GJ_OK;
}

size_t gj_mp_param_count(const gj_mp_desc* d) {
  MPLayout L; StepPath p;
  if (step_plan(d, &L, &p)) return 0;
  return (size_t)L.nparams;
}

static size_t align_floats(size_t n) { return (n + 63) & ~(size_t)63; }   // keep every region 256-byte aligned

struct StepWs {   // offsets in floats
  size_t pq, dpq, de, part, part_post, part_pre, epart, wimg, dist, ysave, dense, emat, total;
};

// caller-owned buffer of a step whose parameter-gradient reduction is deferred (gj_mp_step_bwd_deferred): per-CTA partials of the
// edge kernel, the projections' adjoint and the node-MLP adjoint (offsets in floats)
struct PartialsPlan { size_t edge, pre, post, total; };
static PartialsPlan plan_partials(const MPLayout& L) {
  PartialsPlan p; size_t off = 0;
  p.edge = off; off += align_floats(gj_bwd2_part_floats(L));
  p.pre = off; off += align_floats(gj_node_pre_bwd_tc_ws_floats(L));
  p.post = off; off += align_floats(gj_node_post_bwd_tc_ws_floats(L));
  p.total = off;
  return p;
}
static bool can_defer(const MPLayout& L, const StepPath& p) { return L.B > 0 && p.tail_fused(); }

static StepWs plan_ws(const MPLayout& L, const StepPath& p, bool backward) {
  StepWs w; size_t off = 0;
  const size_t rows = (size_t)L.B * L.N;
  // P|Q, the packed edge-parameter image and the pair distances come first: a caller-owned "saved" buffer of
  // gj_mp_step_saved_bytes() has exactly this prefix layout
  w.pq = off; off += align_floats(rows * 2 * L.E0p);
  w.wimg = w.dist = off;
  if (p.saves()) {
    w.wimg = off; off += align_floats(p.edge == EDGE_TC3 ? gj_edge3_wimage_floats(L) : gj_wimage_floats());
    w.dist = off; off += align_floats(rows * (size_t)(((L.N + 31) / 32) * 32));
  }
  w.ysave = off;
  if (p.edge == EDGE_TC3) off += align_floats(gj_dense_ysave_floats(L));      // node-MLP activations (the saved prefix ends here)
  w.epart = off;
  if (!backward && p.edge == EDGE_TC2) off += align_floats(gj_fwd2_ws_floats(L));   // per-j-block partial aggregates (N > 32)
  if (!backward && p.edge == EDGE_TC3) off += align_floats(gj_edge3_fwd_ws_floats(L));
  w.dpq = w.de = w.part = off;
  if (backward) {
    w.dpq = off; off += align_floats(rows * 2 * L.E0p);
    w.de = off; off += align_floats(rows * L.EL);
    // per-CTA parameter-gradient partials of the node-level and edge adjoints, which use the region one after another.  The fused
    // node kernels' and the first-generation edge adjoint's sizes count on every path (the latter also covers the SIMT adjoint)
    size_t n = std::max({gj_node_post_bwd_ws_floats(L), gj_node_pre_bwd_ws_floats(L), gj_edge_bwd_tc_ws_floats(L), (size_t)64});
    if (p.post_tc) n = std::max(n, gj_node_post_bwd_tc_ws_floats(L));
    if (p.pre_tc) n = std::max(n, gj_node_pre_bwd_tc_ws_floats(L));
    if (p.edge == EDGE_TC2) n = std::max(n, gj_bwd2_ws_floats(L));
    if (p.edge == EDGE_TC3) n = std::max(n, gj_edge3_bwd_ws_floats(L));
    w.part = off; off += align_floats(n);
    // the all-tensor-core backward keeps the node-MLP and projection partials next to the edge kernel's, so that one
    // launch reduces all three at the end of the step
    w.part_post = w.part_pre = w.part;
    if (p.tail_fused()) {
      w.part_post = off; off += align_floats(gj_node_post_bwd_tc_ws_floats(L));
      w.part_pre = off; off += align_floats(gj_node_pre_bwd_tc_ws_floats(L));
    }
  }
  w.dense = off;
  if (p.dense_node) off += align_floats(gj_dense_ws_floats(L, backward));
  w.emat = off;
  if (p.edge == EDGE_MAT) off += align_floats(gj_edge_mat_ws_floats(L, backward));
  w.total = off;
  return w;
}

// The step's edge kernel, forward: e from h and P|Q.  `pre` is the caller's saved buffer or the workspace (same layout).
static int edge_fwd(const MPLayout& L, const StepPath& p, const StepWs& w, float* ws, float* pre, bool saved, bool prepacked,
                    const float* h, const float* params, float* e_out, cudaStream_t st) {
  switch (p.edge) {
    case EDGE_SIMT: return gj_edge_fwd_simt(L, h, pre + w.pq, params, e_out, st);
    case EDGE_TC1: return gj_edge_fwd_tc(L, h, pre + w.pq, params, e_out, st);
    case EDGE_TC2: return gj_edge_fwd2(L, h, pre + w.pq, params, e_out, ws + w.epart, pre + w.wimg, saved ? pre + w.dist : nullptr, st, false, prepacked);
    case EDGE_TC3: return gj_edge_fwd3(L, h, pre + w.pq, params, e_out, ws + w.epart, pre + w.wimg, pre + w.dist, st);
    case EDGE_MAT: break;
  }
  return gj_edge_mat_fwd(L, h, pre + w.pq, params, e_out, ws + w.emat, p.precision, st);
}

// The step's edge adjoint: dP|dQ, the distance-path dh and the edge parameter gradients from de
static int edge_bwd(const MPLayout& L, const StepPath& p, const StepWs& w, float* ws, float* pre, bool saved, const float* h,
                    const float* params, float* dh, float* dparams, cudaStream_t st) {
  switch (p.edge) {
    case EDGE_SIMT: return gj_edge_bwd_simt(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, st);
    case EDGE_TC1: return gj_edge_bwd_tc(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, st);
    case EDGE_TC2:
      return gj_edge_bwd2(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist, saved,
                          st, 0, nullptr, nullptr, nullptr);
    case EDGE_TC3: return gj_edge_bwd3(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist, saved, st);
    case EDGE_MAT: break;
  }
  return gj_edge_mat_bwd(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.emat, p.precision, st);
}

size_t gj_mp_step_fwd_workspace(const gj_mp_desc* d) {
  MPLayout L; StepPath p;
  if (step_plan(d, &L, &p)) return 0;
  return plan_ws(L, p, false).total * sizeof(float);
}

// saved: optional caller-owned buffer of gj_mp_step_saved_bytes(): receives P|Q, the packed edge parameters and the pair
// distances, which gj_mp_step_bwd_saved then reuses instead of recomputing them
static int mp_step_fwd_impl(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* saved,
                            void* workspace, size_t workspace_bytes, void* stream, const char* who, bool prepacked = false) {
  g_err[0] = 0;
  if (!d || !h || !params || !h_out || !e_out || !workspace) { gj_set_error("%s: null pointer", who); return GJ_ERR_INVALID; }
  if (d->precision != GJ_PREC_FP32 && d->precision != GJ_PREC_BF16) { gj_set_error("%s: unknown precision %d", who, d->precision); return GJ_ERR_INVALID; }
  MPLayout L; StepPath p;
  int rc = step_plan(d, &L, &p, who);
  if (rc) return rc;
  if (L.B == 0) return GJ_OK;
  const StepWs w = plan_ws(L, p, false);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("%s: workspace too small", who); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  if (saved && !p.saves()) { gj_set_error("%s: this step has nothing to save (gj_mp_step_saved_bytes is 0)", who); return GJ_ERR_INVALID; }
  if (prepacked && !(p.edge == EDGE_TC2 && saved)) {
    gj_set_error("%s: this step has no packed parameter image (gj_mp_step_partials_bytes is 0)", who); return GJ_ERR_INVALID; }
  float* pre = saved ? (float*)saved : ws;      // P|Q, parameter image, pair distances: same layout in either buffer
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = p.dense_node ? gj_dense_pre_fwd(L, h, params, pre + w.pq, d->precision, st) : gj_node_pre_fwd(L, h, params, pre + w.pq, st))) return rc;
  if ((rc = edge_fwd(L, p, w, ws, pre, saved != nullptr, prepacked, h, params, e_out, st))) return rc;
  if (p.dense_node) return gj_dense_post_fwd(L, e_out, h, params, h_out, ws + w.dense, (saved && p.edge == EDGE_TC3) ? pre + w.ysave : nullptr, d->precision, st);
  return gj_node_post_fwd(L, e_out, h, params, h_out, st);
}

int gj_mp_step_fwd(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* workspace,
                   size_t workspace_bytes, void* stream) {
  return mp_step_fwd_impl(d, h, params, h_out, e_out, nullptr, workspace, workspace_bytes, stream, "gj_mp_step_fwd");
}

int gj_mp_step_launches(const gj_mp_desc* d, int backward, int with_saved) {
  MPLayout L; StepPath p;
  if (step_plan(d, &L, &p)) return 0;
  const int njb = L.N > 32 ? 1 : 0;      // the fused kernels' per-j-block partial sums (forward: e, backward: dP)
  if (p.dense_node) {
    const int node = gj_dense_launches(L, backward != 0);
    if (p.edge == EDGE_MAT) return node + gj_edge_mat_launches(L, backward != 0);
    if (p.edge == EDGE_TC3)      // + parameter image, pair distances, edge kernel [, j-block sum]; backward also the distance adjoint and the reduction
      return node + 3 + njb + (backward ? 2 : 0) - ((backward && with_saved) ? 4 + L.Ln + 1 : 0);
    return node + (backward ? 2 : 1);      // + the edge kernel(s)
  }
  if (!backward) return p.edge == EDGE_TC2 ? 4 + njb : 3;      // projections, [parameter image], edge kernel, [j-block sum], node MLP
  if (p.edge != EDGE_TC2) return 8;
  // node MLP adjoint, [projections, parameter image, pair distances unless saved], edge kernel, [dP j-block sum],
  // pair-distance adjoint, projections' adjoint, and one reduction (all-tensor-core tail) or three
  return 4 + (p.tail_fused() ? 1 : 3) + njb + (with_saved ? 0 : 3);
}

size_t gj_mp_step_saved_bytes(const gj_mp_desc* d) {
  MPLayout L; StepPath p;
  if (step_plan(d, &L, &p) || !p.saves()) return 0;
  return plan_ws(L, p, false).epart * sizeof(float);      // the prefix P|Q, parameter image, pair distances
}

int gj_mp_step_fwd_saving(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* saved,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (!saved) { g_err[0] = 0; gj_set_error("gj_mp_step_fwd_saving: null pointer"); return GJ_ERR_INVALID; }
  return mp_step_fwd_impl(d, h, params, h_out, e_out, saved, workspace, workspace_bytes, stream, "gj_mp_step_fwd_saving");
}

size_t gj_mp_step_bwd_workspace(const gj_mp_desc* d) {
  MPLayout L; StepPath p;
  if (step_plan(d, &L, &p)) return 0;
  return plan_ws(L, p, true).total * sizeof(float);
}

// partials (optional, with saved): caller-owned buffer of gj_mp_step_partials_bytes(); the per-CTA parameter-gradient partials are
// left there and dparams is NOT written (gj_mp_steps_reduce reduces them later)
static int mp_step_bwd_impl(const gj_mp_desc* d, const float* h, const float* e, const float* params, const float* dh_out, float* dh,
                            float* dparams, const void* saved, void* workspace, size_t workspace_bytes, void* stream, const char* who,
                            float* partials = nullptr) {
  g_err[0] = 0;
  if (!d || !h || !e || !params || !dh_out || !dh || (!dparams && !partials) || !workspace) { gj_set_error("%s: null pointer", who); return GJ_ERR_INVALID; }
  if (d->precision != GJ_PREC_FP32 && d->precision != GJ_PREC_BF16) { gj_set_error("%s: unknown precision %d", who, d->precision); return GJ_ERR_INVALID; }
  MPLayout L; StepPath p;
  int rc = step_plan(d, &L, &p, who);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (L.B == 0 && partials) { gj_set_error("%s: empty batch", who); return GJ_ERR_INVALID; }
  if (L.B == 0) { cudaMemsetAsync(dparams, 0, (size_t)L.nparams * sizeof(float), st); return GJ_OK; }
  const StepWs w = plan_ws(L, p, true);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("%s: workspace too small", who); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  if (saved && !p.saves()) { gj_set_error("%s: this step has nothing saved (gj_mp_step_saved_bytes is 0)", who); return GJ_ERR_INVALID; }
  float* pre = saved ? (float*)saved : ws;      // read-only when it is the caller's saved buffer
  if (partials && !(p.tail_fused() && saved)) {
    gj_set_error("%s: this step cannot defer its reduction (gj_mp_step_partials_bytes is 0)", who); return GJ_ERR_INVALID; }
  if (p.tail_fused()) {
    // node MLP adjoint (also clears dP|dQ), P|Q unless saved, edge adjoint, projections' adjoint, one reduction of all partials
    int np_post = 0, np_pre = 0, np_edge = 0;
    const float* part_edge = nullptr;
    const PartialsPlan pp = plan_partials(L);
    float* part_e = partials ? partials + pp.edge : nullptr;
    float* part_post = partials ? partials + pp.post : ws + w.part_post;
    float* part_pre = partials ? partials + pp.pre : ws + w.part_pre;
    if ((rc = gj_node_post_bwd_tc(L, e, h, params, dh_out, ws + w.de, dh, part_post, &np_post, ws + w.dpq, st))) return rc;
    if (!saved && (rc = gj_node_pre_fwd(L, h, params, pre + w.pq, st))) return rc;
    if ((rc = gj_edge_bwd2(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist,
                           saved != nullptr, st, 2, &part_edge, &np_edge, part_e))) return rc;
    if ((rc = gj_node_pre_bwd_tc(L, h, params, ws + w.dpq, dh, part_pre, &np_pre, st))) return rc;
    if (partials) return GJ_OK;      // reduced later, together with the other steps' (gj_mp_steps_reduce)
    return gj_reduce_step_partials(L, part_edge, np_edge, part_pre, np_pre, part_post, np_post, dparams, st);
  }
  if (p.dense_node) {      // generic-GEMM node level (dense.cu) around the edge adjoint
    if ((rc = gj_dense_post_bwd(L, e, h, params, dh_out, ws + w.de, dh, dparams, ws + w.dense,
                                (saved && p.edge == EDGE_TC3) ? pre + w.ysave : nullptr, d->precision, st))) return rc;
    if (!saved && (rc = gj_dense_pre_fwd(L, h, params, pre + w.pq, d->precision, st))) return rc;
    if ((rc = edge_bwd(L, p, w, ws, pre, saved != nullptr, h, params, dh, dparams, st))) return rc;
    return gj_dense_pre_bwd(L, h, params, ws + w.dpq, dh, dparams, ws + w.dense, d->precision, st);
  }
  // node MLP adjoint: de, node-path dh, node parameter gradients
  if (p.post_tc) {      // bf16 mode: the node MLP adjoint on tcgen05
    int nparts = 0;
    if ((rc = gj_node_post_bwd_tc(L, e, h, params, dh_out, ws + w.de, dh, ws + w.part, &nparts, nullptr, st))) return rc;
    if ((rc = gj_reduce_partials(ws + w.part, nparts, L.nparams - L.pV[0], dparams + L.pV[0], st))) return rc;
  } else if ((rc = gj_node_post_bwd(L, e, h, params, dh_out, ws + w.de, dh, dparams, ws + w.part, st))) return rc;
  // P|Q (recomputed unless saved by the forward call), then the edge adjoint
  if (!saved && (rc = gj_node_pre_fwd(L, h, params, pre + w.pq, st))) return rc;
  if ((rc = edge_bwd(L, p, w, ws, pre, saved != nullptr, h, params, dh, dparams, st))) return rc;
  // first-layer projections' adjoint: dh += Wa^T dP + Wb^T dQ, dWa, dWb, db0
  if (p.pre_tc) {      // bf16 mode: the projections' adjoint on tcgen05
    int nparts = 0;
    if ((rc = gj_node_pre_bwd_tc(L, h, params, ws + w.dpq, dh, ws + w.part, &nparts, st))) return rc;
    return gj_reduce_pre_partials(L, ws + w.part, nparts, dparams, st);
  }
  return gj_node_pre_bwd(L, h, params, ws + w.dpq, dh, dparams, ws + w.part, st);
}

int gj_mp_step_bwd(const gj_mp_desc* d, const float* h, const float* e, const float* params, const float* dh_out, float* dh,
                   float* dparams, void* workspace, size_t workspace_bytes, void* stream) {
  return mp_step_bwd_impl(d, h, e, params, dh_out, dh, dparams, nullptr, workspace, workspace_bytes, stream, "gj_mp_step_bwd");
}

int gj_mp_step_bwd_saved(const gj_mp_desc* d, const float* h, const float* e, const float* params, const float* dh_out, float* dh,
                         float* dparams, const void* saved, void* workspace, size_t workspace_bytes, void* stream) {
  if (!saved) { g_err[0] = 0; gj_set_error("gj_mp_step_bwd_saved: null pointer"); return GJ_ERR_INVALID; }
  return mp_step_bwd_impl(d, h, e, params, dh_out, dh, dparams, saved, workspace, workspace_bytes, stream, "gj_mp_step_bwd_saved");
}

// ---- a chain of steps: ONE launch packs every step's parameter image, ONE launch reduces every step's gradient partials ----
size_t gj_mp_step_partials_bytes(const gj_mp_desc* d) {
  MPLayout L; StepPath p;
  if (step_plan(d, &L, &p) || !can_defer(L, p)) return 0;
  return plan_partials(L).total * sizeof(float);
}

int gj_mp_steps_pack(int32_t n, const gj_mp_desc* const* descs, const float* const* params, void* const* saved, void* stream) {
  g_err[0] = 0;
  if (n < 0 || n > 64 || (n > 0 && (!descs || !params || !saved))) { gj_set_error("gj_mp_steps_pack: bad arguments"); return GJ_ERR_INVALID; }
  MPLayout Ls[64]; float* img[64];
  for (int s = 0; s < n; ++s) {
    StepPath p;
    if (!descs[s] || !params[s] || !saved[s]) { gj_set_error("gj_mp_steps_pack: null pointer (step %d)", s); return GJ_ERR_INVALID; }
    if (int rc = step_plan(descs[s], &Ls[s], &p, "gj_mp_steps_pack", s)) return rc;
    if (!can_defer(Ls[s], p)) {
      gj_set_error("gj_mp_steps_pack: step %d does not run the fused tensor-core kernels (gj_mp_step_partials_bytes is 0)", s); return GJ_ERR_INVALID; }
    img[s] = (float*)saved[s] + plan_ws(Ls[s], p, false).wimg;
  }
  return n ? gj_pack_batch2(n, Ls, params, img, (cudaStream_t)stream) : GJ_OK;
}

int gj_mp_step_fwd_packed(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* saved,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (!saved) { g_err[0] = 0; gj_set_error("gj_mp_step_fwd_packed: null pointer"); return GJ_ERR_INVALID; }
  return mp_step_fwd_impl(d, h, params, h_out, e_out, saved, workspace, workspace_bytes, stream, "gj_mp_step_fwd_packed", true);
}

int gj_mp_step_bwd_deferred(const gj_mp_desc* d, const float* h, const float* e, const float* params, const float* dh_out, float* dh,
                            const void* saved, void* partials, void* workspace, size_t workspace_bytes, void* stream) {
  if (!saved || !partials) { g_err[0] = 0; gj_set_error("gj_mp_step_bwd_deferred: null pointer"); return GJ_ERR_INVALID; }
  return mp_step_bwd_impl(d, h, e, params, dh_out, dh, nullptr, saved, workspace, workspace_bytes, stream, "gj_mp_step_bwd_deferred",
                          (float*)partials);
}

int gj_mp_steps_reduce(int32_t n, const gj_mp_desc* const* descs, const void* const* partials, float* const* dparams, void* stream) {
  g_err[0] = 0;
  if (n < 0 || n > 64 || (n > 0 && (!descs || !partials || !dparams))) { gj_set_error("gj_mp_steps_reduce: bad arguments"); return GJ_ERR_INVALID; }
  MPLayout Ls[64];
  const float* pE[64]; const float* pP[64]; const float* pN[64];
  int nE[64], nP[64], nN[64];
  for (int s = 0; s < n; ++s) {
    StepPath p;
    if (!descs[s] || !partials[s] || !dparams[s]) { gj_set_error("gj_mp_steps_reduce: null pointer (step %d)", s); return GJ_ERR_INVALID; }
    if (int rc = step_plan(descs[s], &Ls[s], &p, "gj_mp_steps_reduce", s)) return rc;
    if (!can_defer(Ls[s], p)) {
      gj_set_error("gj_mp_steps_reduce: step %d cannot defer its reduction (gj_mp_step_partials_bytes is 0)", s); return GJ_ERR_INVALID; }
    const PartialsPlan pp = plan_partials(Ls[s]);
    const float* base = (const float*)partials[s];
    pE[s] = base + pp.edge; pP[s] = base + pp.pre; pN[s] = base + pp.post;
    nE[s] = gj_bwd2_nparts(Ls[s]); nP[s] = gj_node_pre_bwd_tc_nparts(Ls[s]); nN[s] = gj_node_post_bwd_tc_nparts(Ls[s]);
  }
  return n ? gj_reduce_steps_partials(n, Ls, pE, nE, pP, nP, pN, nN, dparams, (cudaStream_t)stream) : GJ_OK;
}

int gj_chamfer_fwd_bwd(int32_t batch, int32_t np_, int32_t nq, int32_t dim, int32_t norm, float w_chamfer, float w_jet,
                       const float* p, const float* q, float* jet_terms, float* terms, float* dp, void* stream) {
  g_err[0] = 0;
  if (!p || !q || !jet_terms || !terms) { gj_set_error("gj_chamfer_fwd_bwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_chamfer_launch(batch, np_, nq, dim, norm, w_chamfer, w_jet, p, q, jet_terms, terms, dp, (cudaStream_t)stream);
}

int gj_pair_min_dist(int32_t batch, int32_t np_, int32_t nq, int32_t dim, int32_t lorentz, const float* p, const float* q,
                     float* min_pq, float* min_qp, void* stream) {
  g_err[0] = 0;
  if (batch > 0 && (!p || !q || !min_pq || !min_qp)) { gj_set_error("gj_pair_min_dist: null pointer"); return GJ_ERR_INVALID; }
  return gj_pair_min_dist_launch(batch, np_, nq, dim, lorentz, p, q, min_pq, min_qp, (cudaStream_t)stream);
}

int gj_assignment(int32_t batch, int32_t n, int32_t dim, int32_t lorentz, const float* p, const float* q, int32_t* col_for_row,
                  float* total_cost, void* stream) {
  g_err[0] = 0;
  if (batch > 0 && (!p || !q || !col_for_row)) { gj_set_error("gj_assignment: null pointer"); return GJ_ERR_INVALID; }
  return gj_assignment_launch(batch, n, dim, lorentz, p, q, col_for_row, total_cost, (cudaStream_t)stream);
}

// the solver keeps its whole state in shared memory
size_t gj_emd_workspace(int32_t, int32_t, int32_t) { return 0; }

int gj_emd(int32_t batch, int32_t np_, int32_t nq, const float* p, const float* q, float R, float beta, int32_t flags, double* emd_out,
           double* flow_out, float* dp_out, double* potentials_out, int32_t* status_out, void*, size_t, void* stream) {
  g_err[0] = 0;
  if (int rc = gj_emd_check(batch, np_, nq, R, beta, flags)) return rc;
  if (batch > 0 && (!p || !q || !emd_out)) { gj_set_error("gj_emd: null pointer"); return GJ_ERR_INVALID; }
  return gj_emd_launch(batch, np_, nq, p, q, R, beta, flags, emd_out, flow_out, dp_out, potentials_out, status_out, (cudaStream_t)stream);
}

size_t gj_emd_loss_workspace(int32_t batch, int32_t) { return gj_emd_loss_ws_bytes(batch); }

int gj_emd_loss(int32_t batch, int32_t n, int32_t dim, int32_t coords, const float* p, const float* q, float R, float beta,
                int32_t flags, float scale, float* terms, float* failed, float* dp, void* workspace, size_t workspace_bytes,
                void* stream) {
  g_err[0] = 0;
  if (int rc = gj_emd_loss_check(batch, n, dim, coords, R, beta, flags, workspace_bytes)) return rc;
  if (!terms || !failed || (batch > 0 && (!p || !q || !workspace))) { gj_set_error("gj_emd_loss: null pointer"); return GJ_ERR_INVALID; }
  return gj_emd_loss_launch(batch, n, dim, coords, p, q, R, beta, flags, scale, terms, failed, dp, workspace, (cudaStream_t)stream);
}

size_t gj_hungarian_mse_loss_workspace(int32_t batch, int32_t) { return gj_hmse_ws_bytes(batch); }

int gj_hungarian_mse_loss(int32_t batch, int32_t n, int32_t dim, int32_t coords, const float* p, const float* q, float scale,
                          float* terms, float* dp, int32_t* col_for_row, void* workspace, size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  if (int rc = gj_hmse_check(batch, n, dim, coords, workspace_bytes)) return rc;
  if (!terms || (batch > 0 && (!p || !q || !dp || !workspace))) { gj_set_error("gj_hungarian_mse_loss: null pointer"); return GJ_ERR_INVALID; }
  return gj_hmse_launch(batch, n, dim, coords, p, q, scale, terms, dp, col_for_row, workspace, (cudaStream_t)stream);
}

int gj_linear_fwd(int32_t rows, int32_t in_f, int32_t out_f, const float* x, const float* w, const float* b, float* y,
                  void* stream) {
  g_err[0] = 0;
  if (rows < 0 || in_f < 1 || out_f < 1) { gj_set_error("gj_linear_fwd: bad shape"); return GJ_ERR_INVALID; }
  if (rows && (!x || !w || !y)) { gj_set_error("gj_linear_fwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_linear_fwd_launch(rows, in_f, out_f, x, w, b, y, (cudaStream_t)stream);
}

size_t gj_linear_bwd_workspace(int32_t rows, int32_t in_f, int32_t out_f) { return gj_linear_bwd_ws_bytes(rows, in_f, out_f); }

int gj_linear_bwd(int32_t rows, int32_t in_f, int32_t out_f, const float* x, const float* w, const float* dy, float* dx,
                  float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  if (rows < 0 || in_f < 1 || out_f < 1) { gj_set_error("gj_linear_bwd: bad shape"); return GJ_ERR_INVALID; }
  if (!w || !dw || !workspace || (rows && (!x || !dy))) { gj_set_error("gj_linear_bwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_linear_bwd_launch(rows, in_f, out_f, x, w, dy, dx, dw, db, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gj_adam_step_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1,
                      float beta2, float eps, int32_t step, float grad_scale, float l1_lambda, float l2_lambda, void* stream) {
  g_err[0] = 0;
  if (n && (!param || !grad || !exp_avg || !exp_avg_sq)) { gj_set_error("gj_adam_step_flat: null pointer"); return GJ_ERR_INVALID; }
  return gj_adam_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, grad_scale, l1_lambda, l2_lambda,
                        (cudaStream_t)stream);
}

int gj_optimizer_step_flat(int32_t kind, float* param, const float* grad, float* momentum_buf, float* sq_acc, size_t n, float lr,
                           float alpha, float momentum, float eps, float grad_scale, float l1_lambda, float l2_lambda, void* stream) {
  g_err[0] = 0;
  if (kind < GJ_OPT_RMSPROP || kind > GJ_OPT_SGD) { gj_set_error("gj_optimizer_step_flat: unknown optimiser %d", kind); return GJ_ERR_INVALID; }
  if (n && (!param || !grad || !momentum_buf || !sq_acc)) { gj_set_error("gj_optimizer_step_flat: null pointer"); return GJ_ERR_INVALID; }
  return gj_optimizer_launch(kind, param, grad, momentum_buf, sq_acc, n, lr, alpha, momentum, eps, grad_scale, l1_lambda, l2_lambda,
                             (cudaStream_t)stream);
}

int gj_nonfinite_flag(const float* terms, int32_t count, float* out, void* stream) {
  g_err[0] = 0;
  if (count < 0 || count > 64) { gj_set_error("gj_nonfinite_flag: 0 <= count <= 64, got %d", count); return GJ_ERR_INVALID; }
  if (!out || (count && !terms)) { gj_set_error("gj_nonfinite_flag: null pointer"); return GJ_ERR_INVALID; }
  return gj_nonfinite_flag_launch(terms, count, out, (cudaStream_t)stream);
}

int gj_nonfinite_check(const float* x, size_t n, int32_t* skip, float* flag, void* stream) {
  g_err[0] = 0;
  if (!skip || (n && !x)) { gj_set_error("gj_nonfinite_check: null pointer"); return GJ_ERR_INVALID; }
  return gj_nonfinite_check_launch(x, n, skip, flag, (cudaStream_t)stream);
}

int gj_adam_step_flat_guarded(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1,
                              float beta2, float eps, const int32_t* skip, int32_t* step_state, float grad_scale, float l1_lambda,
                              float l2_lambda, void* stream) {
  g_err[0] = 0;
  if (!skip || !step_state || (n && (!param || !grad || !exp_avg || !exp_avg_sq))) {
    gj_set_error("gj_adam_step_flat_guarded: null pointer"); return GJ_ERR_INVALID; }
  return gj_adam_guarded_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, skip, step_state, grad_scale, l1_lambda,
                                l2_lambda, (cudaStream_t)stream);
}

int gj_optimizer_step_flat_guarded(int32_t kind, float* param, const float* grad, float* momentum_buf, float* sq_acc, size_t n, float lr,
                                   float alpha, float momentum, float eps, float grad_scale, float l1_lambda, float l2_lambda,
                                   const int32_t* skip, int32_t* step_state, void* stream) {
  g_err[0] = 0;
  if (kind < GJ_OPT_RMSPROP || kind > GJ_OPT_SGD) { gj_set_error("gj_optimizer_step_flat_guarded: unknown optimiser %d", kind); return GJ_ERR_INVALID; }
  if (!skip || (n && (!param || !grad || !momentum_buf || !sq_acc))) {
    gj_set_error("gj_optimizer_step_flat_guarded: null pointer"); return GJ_ERR_INVALID; }
  return gj_optimizer_guarded_launch(kind, param, grad, momentum_buf, sq_acc, n, lr, alpha, momentum, eps, grad_scale, l1_lambda,
                                     l2_lambda, skip, step_state, (cudaStream_t)stream);
}

size_t gj_param_norms_workspace(size_t n) { return gj_norms_ws_bytes(n); }

int gj_param_norms(const float* param, size_t n, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  if (!out || !workspace || (n && !param)) { gj_set_error("gj_param_norms: null pointer"); return GJ_ERR_INVALID; }
  return gj_norms_launch(param, n, out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gj_latent_mean_fwd(int32_t batch, int32_t num_nodes, int32_t width, const float* y, float* z, void* stream) {
  g_err[0] = 0;
  if (batch < 0 || num_nodes < 1 || width < 1) { gj_set_error("gj_latent_mean_fwd: bad shape"); return GJ_ERR_INVALID; }
  return gj_latent_mean_fwd_launch(batch, num_nodes, width, y, z, (cudaStream_t)stream);
}

int gj_latent_mean_bwd(int32_t batch, int32_t num_nodes, int32_t width, const float* dz, float* dy, void* stream) {
  g_err[0] = 0;
  if (batch < 0 || num_nodes < 1 || width < 1) { gj_set_error("gj_latent_mean_bwd: bad shape"); return GJ_ERR_INVALID; }
  return gj_latent_mean_bwd_launch(batch, num_nodes, width, dz, dy, (cudaStream_t)stream);
}

int gj_latent_extreme_fwd(int32_t batch, int32_t num_nodes, int32_t width, int32_t is_min, const float* y, float* z, void* stream) {
  g_err[0] = 0;
  if (batch < 0 || num_nodes < 1 || width < 1) { gj_set_error("gj_latent_extreme_fwd: bad shape"); return GJ_ERR_INVALID; }
  if (batch > 0 && (!y || !z)) { gj_set_error("gj_latent_extreme_fwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_latent_extreme_fwd_launch(batch, num_nodes, width, is_min != 0, y, z, (cudaStream_t)stream);
}

int gj_latent_extreme_bwd(int32_t batch, int32_t num_nodes, int32_t width, const float* y, const float* z, const float* dz, float* dy,
                          void* stream) {
  g_err[0] = 0;
  if (batch < 0 || num_nodes < 1 || width < 1) { gj_set_error("gj_latent_extreme_bwd: bad shape"); return GJ_ERR_INVALID; }
  if (batch > 0 && (!y || !z || !dz || !dy)) { gj_set_error("gj_latent_extreme_bwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_latent_extreme_bwd_launch(batch, num_nodes, width, y, z, dz, dy, (cudaStream_t)stream);
}

int gj_output_transform_fwd(size_t rows, int32_t dim, int32_t use_tanh, int32_t clamp_mask, float eps, const float* x, float* y, void* stream) {
  g_err[0] = 0;
  if (dim < 1 || dim > 31) { gj_set_error("gj_output_transform_fwd: bad width"); return GJ_ERR_INVALID; }
  if (rows > 0 && (!x || !y)) { gj_set_error("gj_output_transform_fwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_out_transform_launch(rows * (size_t)dim, dim, use_tanh != 0, clamp_mask, eps, x, nullptr, y, (cudaStream_t)stream);
}

int gj_output_transform_bwd(size_t rows, int32_t dim, int32_t use_tanh, int32_t clamp_mask, float eps, const float* x, const float* dy,
                            float* dx, void* stream) {
  g_err[0] = 0;
  if (dim < 1 || dim > 31) { gj_set_error("gj_output_transform_bwd: bad width"); return GJ_ERR_INVALID; }
  if (rows > 0 && (!x || !dy || !dx)) { gj_set_error("gj_output_transform_bwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_out_transform_launch(rows * (size_t)dim, dim, use_tanh != 0, clamp_mask, eps, x, dy, dx, (cudaStream_t)stream);
}

size_t gj_mse_workspace(void) { return gj_mse_ws_bytes(); }

int gj_mse_fwd_bwd(size_t count, double denom, const float* p, const float* q, float* terms, float* dp, void* workspace,
                   size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  if (!(denom > 0.0)) { gj_set_error("gj_mse_fwd_bwd: denom must be positive"); return GJ_ERR_INVALID; }
  if (!terms || !workspace || (count > 0 && (!p || !q || !dp))) { gj_set_error("gj_mse_fwd_bwd: null pointer"); return GJ_ERR_INVALID; }
  return gj_mse_launch(count, denom, p, q, terms, dp, workspace, workspace_bytes, (cudaStream_t)stream);
}

/* Measurement hooks (declared in the header under "benchmark support"): relaunch ONLY the fused edge kernel of a step on
 * the workspace that a preceding full gj_mp_step_fwd / gj_mp_step_bwd call with the same arguments has populated. */
static int bench_step(const gj_mp_desc* d, bool pointers, size_t workspace_bytes, bool backward, const char* who, MPLayout* L, StepWs* w) {
  g_err[0] = 0;
  StepPath p;
  if (int rc = step_plan(d, L, &p, who)) return rc;
  if (!pointers) { gj_set_error("%s: null pointer", who); return GJ_ERR_INVALID; }
  if (p.edge != EDGE_TC2) { gj_set_error("%s: step does not run the fused tensor-core kernel", who); return GJ_ERR_INVALID; }
  *w = plan_ws(*L, p, backward);
  if (workspace_bytes < w->total * sizeof(float)) { gj_set_error("%s: workspace too small", who); return GJ_ERR_WORKSPACE; }
  return GJ_OK;
}

int gj_bench_edge_fwd_only(const gj_mp_desc* d, const float* h, const float* params, float* e_out, void* workspace,
                           size_t workspace_bytes, void* stream) {
  MPLayout L; StepWs w;
  if (int rc = bench_step(d, h && params && e_out && workspace, workspace_bytes, false, "gj_bench_edge_fwd_only", &L, &w)) return rc;
  float* ws = (float*)workspace;
  return gj_edge_fwd2(L, h, ws + w.pq, params, e_out, ws + w.epart, ws + w.wimg, nullptr, (cudaStream_t)stream, true, false);
}

int gj_bench_edge_bwd_only(const gj_mp_desc* d, const float* h, const float* params, float* dh, float* dparams, void* workspace,
                           size_t workspace_bytes, void* stream) {
  MPLayout L; StepWs w;
  if (int rc = bench_step(d, h && params && dh && dparams && workspace, workspace_bytes, true, "gj_bench_edge_bwd_only", &L, &w)) return rc;
  float* ws = (float*)workspace;
  return gj_edge_bwd2(L, h, ws + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, ws + w.wimg, ws + w.dist, true,
                      (cudaStream_t)stream, 1, nullptr, nullptr, nullptr);
}

/* As gj_bench_edge_bwd_only, for the step as the trainer runs it: `saved` was filled by gj_mp_step_fwd_saving and `workspace`
 * by the gj_mp_step_bwd_saved call that followed. */
int gj_bench_edge_bwd_saved_only(const gj_mp_desc* d, const float* h, const float* params, float* dh, float* dparams, const void* saved,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  MPLayout L; StepWs w;
  if (int rc = bench_step(d, h && params && dh && dparams && saved && workspace, workspace_bytes, true, "gj_bench_edge_bwd_saved_only", &L, &w))
    return rc;
  float* ws = (float*)workspace;
  float* pre = (float*)saved;
  return gj_edge_bwd2(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist, true,
                      (cudaStream_t)stream, 1, nullptr, nullptr, nullptr);
}

int gj_mp_plan_info(const gj_mp_desc* d, int32_t* info) {
  g_err[0] = 0;
  MPLayout L; StepPath p;
  if (int rc = step_plan(d, &L, &p, "gj_mp_plan_info")) return rc;
  if (!info) { gj_set_error("gj_mp_plan_info: null pointer"); return GJ_ERR_INVALID; }
  gj_tc_plan_info(L, info);
  // the second-generation kernels take over where their widths are compiled in
  if (p.edge == EDGE_TC2) { gj_fwd2_plan(L, info + 0, info + 1); gj_bwd2_plan(L, info + 2, info + 3); }
  return GJ_OK;
}

int gj_umma_selftest(int32_t m, int32_t n, int32_t k, int32_t a_major, int32_t b_major, const float* a, const float* b,
                     float* out, void* stream) {
  g_err[0] = 0;
  if (!a || !b || !out) { gj_set_error("gj_umma_selftest: null pointer"); return GJ_ERR_INVALID; }
  return gj_umma_selftest_launch(m, n, k, a_major, b_major, a, b, out, (cudaStream_t)stream);
}

}  // extern "C"
