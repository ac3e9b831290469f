// C-ABI entry points declared in include/gnnjet_b200.h: argument checks, dispatch on precision,
// error reporting.  No torch types; raw device pointers + sizes + cudaStream_t.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

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

size_t gj_mp_param_count(const gj_mp_desc* d) {
  MPLayout L; const char* why;
  if (gj_fill_arch(d, &L, &why)) return 0;
  return (size_t)L.nparams;
}

static size_t align_floats(size_t n) { return (n + 63) & ~(size_t)63; }   // keep every region 256-byte aligned

struct StepWs {   // offsets in floats
  size_t pq, dpq, de, part, part_post, part_pre, epart, wimg, dist, ysave, dense, emat, total;
};

static bool use_tc(const MPLayout& L, int precision) { return precision == GJ_PREC_BF16 && L.Le > 1; }
// the step runs the second-generation fused kernels (forward and backward are covered by the same widths)
static bool tc2_path(const MPLayout& L, int precision) {
  return use_tc(L, precision) && gj_fwd2_supported(L) && gj_bwd2_supported(L);
}

static bool edge_mat(const MPLayout& L, int precision);
// the step runs the third-generation fused kernels (two-layer edge networks [H, H], H = 64 / 128: BASELINE config 5)
static bool tc3_path(const MPLayout& L, int precision) {
  return use_tc(L, precision) && !tc2_path(L, precision) && gj_edge3_supported(L);
}

// Node-level work (P|Q projections, node MLP and their adjoints) as generic GEMMs (dense.cu): wherever a node-level weight
// matrix does not fit the fused node kernels' shared-memory plans, and for wide layers (BASELINE config 5: H >= 64), where the
// GEMM formulation -- tcgen05 in the bf16 mode -- is the faster one
static bool dense_node(const MPLayout& L, int precision) {
  if (edge_mat(L, precision)) return true;
  if (tc2_path(L, precision)) return false;
  if (!gj_node_generic_fits(L)) return true;
  int wmax = L.H > L.E[0] ? L.H : L.E[0];
  for (int m = 0; m < L.Ln; ++m) if (L.O[m] > wmax) wmax = L.O[m];
  return wmax >= 64;
}

// The edge MLP as generic GEMMs over the materialised edge rows of a chunk of jets (dense.cu): for the widths no fused edge
// kernel has a plan for (e.g. edge_sizes [[256, 256]])
static bool edge_mat(const MPLayout& L, int precision) {
  if (tc2_path(L, precision) || tc3_path(L, precision)) return false;
  return use_tc(L, precision) ? !gj_edge_tc_fits(L) : !gj_edge_simt_fits(L, nullptr);
}

// backward of the bf16 step with both node-level adjoints on tcgen05: their partials and the edge kernel's are reduced together
static bool node_tail_fused(const MPLayout& L, int precision) {
  return tc2_path(L, precision) && gj_node_post_bwd_tc_supported(L) && gj_node_pre_bwd_tc_supported(L);
}

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

static StepWs plan_ws(const MPLayout& L, int precision, bool backward) {
  StepWs w; size_t off = 0;
  const size_t rows = (size_t)L.B * L.N;
  // P|Q, the packed edge-parameter image and the pair distances come first: a caller-owned "saved" buffer of
  // gj_mp_step_saved_bytes() has exactly this prefix layout
  w.pq = off; off += align_floats(rows * 2 * L.E0p);
  w.wimg = w.dist = off;
  if (tc2_path(L, precision) || tc3_path(L, precision)) {
    w.wimg = off; off += align_floats(tc3_path(L, precision) ? gj_edge3_wimage_floats(L) : gj_wimage_floats());
    w.dist = off; off += align_floats(rows * (size_t)(((L.N + 31) / 32) * 32));
  }
  w.ysave = off;
  if (tc3_path(L, precision)) off += align_floats(gj_dense_ysave_floats(L));      // node-MLP activations (the saved prefix ends here)
  w.epart = off;
  if (!backward && tc2_path(L, precision)) off += align_floats(gj_fwd2_ws_floats(L));   // per-j-block partial aggregates (N > 32)
  if (!backward && tc3_path(L, precision)) off += align_floats(gj_edge3_fwd_ws_floats(L));
  w.dpq = w.de = w.part = off;
  if (backward) {
    w.dpq = off; off += align_floats(rows * 2 * L.E0p);
    w.de = off; off += align_floats(rows * L.EL);
    size_t p = gj_node_post_bwd_ws_floats(L);
    if (tc2_path(L, precision) && gj_node_post_bwd_tc_supported(L)) { const size_t p2 = gj_node_post_bwd_tc_ws_floats(L); if (p2 > p) p = p2; }
    size_t q = gj_node_pre_bwd_ws_floats(L);
    if (tc2_path(L, precision) && gj_node_pre_bwd_tc_supported(L)) { const size_t q2 = gj_node_pre_bwd_tc_ws_floats(L); if (q2 > q) q = q2; }
    size_t r = use_tc(L, precision) ? gj_edge_bwd_tc_ws_floats(L) : (size_t)gj_edge_grid(L.B) * L.pV[0];
    if (tc2_path(L, precision)) { const size_t r2 = gj_bwd2_ws_floats(L); if (r2 > r) r = r2; }
    if (tc3_path(L, precision)) { const size_t r2 = gj_edge3_bwd_ws_floats(L); if (r2 > r) r = r2; }
    if (q > p) p = q;
    if (r > p) p = r;
    if (p < 64) p = 64;
    w.part = off; off += align_floats(p);
    // the all-tensor-core backward keeps the node-MLP and projection partials next to the edge kernel's, so that one
    // launch reduces all three at the end of the step
    w.part_post = w.part_pre = w.part;
    if (node_tail_fused(L, precision)) {
      w.part_post = off; off += align_floats(gj_node_post_bwd_tc_ws_floats(L));
      w.part_pre = off; off += align_floats(gj_node_pre_bwd_tc_ws_floats(L));
    }
  }
  w.dense = off;
  if (dense_node(L, precision)) off += align_floats(gj_dense_ws_floats(L, backward));
  w.emat = off;
  if (edge_mat(L, precision)) off += align_floats(gj_edge_mat_ws_floats(L, backward));
  w.total = off;
  return w;
}

size_t gj_mp_step_fwd_workspace(const gj_mp_desc* d) {
  MPLayout L; const char* why;
  if (gj_fill_arch(d, &L, &why)) return 0;
  return plan_ws(L, d->precision, false).total * sizeof(float);
}

// saved: optional caller-owned buffer of gj_mp_step_saved_bytes(): receives P|Q, the packed edge parameters and the pair
// distances, which gj_mp_step_bwd_saved then reuses instead of recomputing them
static int mp_step_fwd_impl(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* saved,
                            void* workspace, size_t workspace_bytes, void* stream, const char* who, bool prepacked = false) {
  g_err[0] = 0;
  if (!d || !h || !params || !h_out || !e_out || !workspace) { gj_set_error("%s: null pointer", who); return GJ_ERR_INVALID; }
  if (d->precision != GJ_PREC_FP32 && d->precision != GJ_PREC_BF16) { gj_set_error("%s: unknown precision %d", who, d->precision); return GJ_ERR_INVALID; }
  MPLayout L; const char* why;
  int rc = gj_fill_arch(d, &L, &why);
  if (rc) { gj_set_error("%s: %s", who, why); return rc; }
  if (L.B == 0) return GJ_OK;
  const StepWs w = plan_ws(L, d->precision, false);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("%s: workspace too small", who); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  const bool emat = edge_mat(L, d->precision);
  const bool tc2 = tc2_path(L, d->precision);
  const bool tc3 = tc3_path(L, d->precision);
  if (saved && !tc2 && !tc3) { gj_set_error("%s: this step has nothing to save (gj_mp_step_saved_bytes is 0)", who); return GJ_ERR_INVALID; }
  if (prepacked && !(tc2 && saved)) { gj_set_error("%s: this step has no packed parameter image (gj_mp_step_partials_bytes is 0)", who); return GJ_ERR_INVALID; }
  float* pre = saved ? (float*)saved : ws;      // P|Q, parameter image, pair distances: same layout in either buffer
  cudaStream_t st = (cudaStream_t)stream;
  const bool dense = dense_node(L, d->precision);
  if ((rc = dense ? gj_dense_pre_fwd(L, h, params, pre + w.pq, d->precision, st) : gj_node_pre_fwd(L, h, params, pre + w.pq, st))) return rc;
  if (emat) rc = gj_edge_mat_fwd(L, h, ws + w.pq, params, e_out, ws + w.emat, d->precision, st);
  else if (tc3) rc = gj_edge_fwd3(L, h, pre + w.pq, params, e_out, ws + w.epart, pre + w.wimg, pre + w.dist, st);
  else if (tc2) rc = gj_edge_fwd2(L, h, pre + w.pq, params, e_out, ws + w.epart, pre + w.wimg, saved ? pre + w.dist : nullptr, st, false, prepacked);
  else rc = use_tc(L, d->precision) ? gj_edge_fwd_tc(L, h, ws + w.pq, params, e_out, st)
                                    : gj_edge_fwd_simt(L, h, ws + w.pq, params, e_out, st);
  if (rc) return rc;
  if (dense) return gj_dense_post_fwd(L, e_out, h, params, h_out, ws + w.dense, (saved && tc3) ? pre + w.ysave : nullptr, d->precision, st);
  return gj_node_post_fwd(L, e_out, h, params, h_out, st);
}

int gj_mp_step_fwd(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* workspace,
                   size_t workspace_bytes, void* stream) {
  return mp_step_fwd_impl(d, h, params, h_out, e_out, nullptr, workspace, workspace_bytes, stream, "gj_mp_step_fwd");
}

int gj_mp_step_launches(const gj_mp_desc* d, int backward, int with_saved) {
  MPLayout L; const char* why;
  if (gj_fill_arch(d, &L, &why)) return 0;
  const bool tc2 = tc2_path(L, d->precision);
  const int njb = (tc2 && L.N > 32) ? 1 : 0;      // per-j-block partial sums (forward: e, backward: dP)
  if (edge_mat(L, d->precision)) return gj_dense_launches(L, backward != 0) + gj_edge_mat_launches(L, backward != 0);
  if (tc3_path(L, d->precision))      // + parameter image, pair distances, edge kernel [, j-block sum]; backward also the distance adjoint and the reduction
    return gj_dense_launches(L, backward != 0) + 3 + (L.N > 32 ? 1 : 0) + (backward ? 2 : 0) - ((backward && with_saved) ? 4 + L.Ln + 1 : 0);
  if (dense_node(L, d->precision)) return gj_dense_launches(L, backward != 0) + (backward ? 2 : 1);      // + the edge kernel(s)
  if (!backward) return tc2 ? 4 + njb : 3;        // projections, [parameter image], edge kernel, [j-block sum], node MLP
  if (!tc2) return 8;
  // node MLP adjoint, [projections, parameter image, pair distances unless saved], edge kernel, [dP j-block sum],
  // pair-distance adjoint, projections' adjoint, and one reduction (all-tensor-core tail) or three
  const int reductions = node_tail_fused(L, d->precision) ? 1 : 3;
  return 4 + reductions + njb + ((with_saved && tc2) ? 0 : 3);
}

size_t gj_mp_step_saved_bytes(const gj_mp_desc* d) {
  MPLayout L; const char* why;
  if (gj_fill_arch(d, &L, &why) || !(tc2_path(L, d->precision) || tc3_path(L, d->precision))) return 0;
  const StepWs w = plan_ws(L, d->precision, false);
  return w.epart * sizeof(float);      // the prefix P|Q, parameter image, pair distances
}

int gj_mp_step_fwd_saving(const gj_mp_desc* d, const float* h, const float* params, float* h_out, float* e_out, void* saved,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (!saved) { g_err[0] = 0; gj_set_error("gj_mp_step_fwd_saving: null pointer"); return GJ_ERR_INVALID; }
  return mp_step_fwd_impl(d, h, params, h_out, e_out, saved, workspace, workspace_bytes, stream, "gj_mp_step_fwd_saving");
}

size_t gj_mp_step_bwd_workspace(const gj_mp_desc* d) {
  MPLayout L; const char* why;
  if (gj_fill_arch(d, &L, &why)) return 0;
  return plan_ws(L, d->precision, true).total * sizeof(float);
}

// partials (optional, with saved): caller-owned buffer of gj_mp_step_partials_bytes(); the per-CTA parameter-gradient partials are
// left there and dparams is NOT written (gj_mp_steps_reduce reduces them later)
static int mp_step_bwd_impl(const gj_mp_desc* d, const float* h, const float* e, const float* params, const float* dh_out, float* dh,
                            float* dparams, const void* saved, void* workspace, size_t workspace_bytes, void* stream, const char* who,
                            float* partials = nullptr) {
  g_err[0] = 0;
  if (!d || !h || !e || !params || !dh_out || !dh || (!dparams && !partials) || !workspace) { gj_set_error("%s: null pointer", who); return GJ_ERR_INVALID; }
  if (d->precision != GJ_PREC_FP32 && d->precision != GJ_PREC_BF16) { gj_set_error("%s: unknown precision %d", who, d->precision); return GJ_ERR_INVALID; }
  MPLayout L; const char* why;
  int rc = gj_fill_arch(d, &L, &why);
  if (rc) { gj_set_error("%s: %s", who, why); return rc; }
  cudaStream_t st = (cudaStream_t)stream;
  if (L.B == 0 && partials) { gj_set_error("%s: empty batch", who); return GJ_ERR_INVALID; }
  if (L.B == 0) { cudaMemsetAsync(dparams, 0, (size_t)L.nparams * sizeof(float), st); return GJ_OK; }
  const StepWs w = plan_ws(L, d->precision, true);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("%s: workspace too small", who); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  const bool emat = edge_mat(L, d->precision);
  const bool tc2 = tc2_path(L, d->precision);
  const bool tc3 = tc3_path(L, d->precision);
  if (saved && !tc2 && !tc3) { gj_set_error("%s: this step has nothing saved (gj_mp_step_saved_bytes is 0)", who); return GJ_ERR_INVALID; }
  float* pre = saved ? (float*)saved : ws;      // read-only when it is the caller's saved buffer
  if (partials && !(node_tail_fused(L, d->precision) && saved)) {
    gj_set_error("%s: this step cannot defer its reduction (gj_mp_step_partials_bytes is 0)", who); return GJ_ERR_INVALID; }
  if (node_tail_fused(L, d->precision)) {
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
  const bool dense = dense_node(L, d->precision);
  if (dense) {      // generic-GEMM node level (dense.cu) around the edge adjoint
    if ((rc = gj_dense_post_bwd(L, e, h, params, dh_out, ws + w.de, dh, dparams, ws + w.dense, (saved && tc3) ? pre + w.ysave : nullptr,
                                d->precision, st))) return rc;
    if (!saved && (rc = gj_dense_pre_fwd(L, h, params, pre + w.pq, d->precision, st))) return rc;
    rc = emat ? gj_edge_mat_bwd(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.emat, d->precision, st)
       : tc3 ? gj_edge_bwd3(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist,
                            saved != nullptr, st)
       : use_tc(L, d->precision) ? gj_edge_bwd_tc(L, h, ws + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, st)
                                 : gj_edge_bwd_simt(L, h, ws + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, st);
    if (rc) return rc;
    return gj_dense_pre_bwd(L, h, params, ws + w.dpq, dh, dparams, ws + w.dense, d->precision, st);
  }
  // node MLP adjoint: de, node-path dh, node parameter gradients
  if (tc2 && gj_node_post_bwd_tc_supported(L)) {      // bf16 mode: the node MLP adjoint on tcgen05
    int nparts = 0;
    if ((rc = gj_node_post_bwd_tc(L, e, h, params, dh_out, ws + w.de, dh, ws + w.part, &nparts, nullptr, st))) return rc;
    if ((rc = gj_reduce_partials(ws + w.part, nparts, L.nparams - L.pV[0], dparams + L.pV[0], st))) return rc;
  } else if ((rc = gj_node_post_bwd(L, e, h, params, dh_out, ws + w.de, dh, dparams, ws + w.part, st))) return rc;
  // P|Q (recomputed unless saved by the forward call), then the edge adjoint: dP|dQ, distance-path dh, edge parameter gradients
  if (!saved && (rc = gj_node_pre_fwd(L, h, params, pre + w.pq, st))) return rc;
  if (tc2)
    rc = gj_edge_bwd2(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist, saved != nullptr,
                      st, 0, nullptr, nullptr, nullptr);
  else
    rc = use_tc(L, d->precision) ? gj_edge_bwd_tc(L, h, ws + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, st)
                                 : gj_edge_bwd_simt(L, h, ws + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, st);
  if (rc) return rc;
  // first-layer projections' adjoint: dh += Wa^T dP + Wb^T dQ, dWa, dWb, db0
  if (tc2 && gj_node_pre_bwd_tc_supported(L)) {      // bf16 mode: the projections' adjoint on tcgen05
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
  MPLayout L; const char* why;
  if (gj_fill_arch(d, &L, &why) || L.B == 0 || !node_tail_fused(L, d->precision)) return 0;
  return plan_partials(L).total * sizeof(float);
}

int gj_mp_steps_pack(int32_t n, const gj_mp_desc* const* descs, const float* const* params, void* const* saved, void* stream) {
  g_err[0] = 0;
  if (n < 0 || n > 64 || (n > 0 && (!descs || !params || !saved))) { gj_set_error("gj_mp_steps_pack: bad arguments"); return GJ_ERR_INVALID; }
  MPLayout Ls[64]; float* img[64];
  for (int s = 0; s < n; ++s) {
    const char* why;
    if (!descs[s] || !params[s] || !saved[s]) { gj_set_error("gj_mp_steps_pack: null pointer (step %d)", s); return GJ_ERR_INVALID; }
    if (int rc = gj_fill_arch(descs[s], &Ls[s], &why)) { gj_set_error("gj_mp_steps_pack: %s (step %d)", why, s); return rc; }
    if (gj_mp_step_partials_bytes(descs[s]) == 0) {
      gj_set_error("gj_mp_steps_pack: step %d does not run the fused tensor-core kernels (gj_mp_step_partials_bytes is 0)", s); return GJ_ERR_INVALID; }
    img[s] = (float*)saved[s] + plan_ws(Ls[s], descs[s]->precision, false).wimg;
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
    const char* why;
    if (!descs[s] || !partials[s] || !dparams[s]) { gj_set_error("gj_mp_steps_reduce: null pointer (step %d)", s); return GJ_ERR_INVALID; }
    if (int rc = gj_fill_arch(descs[s], &Ls[s], &why)) { gj_set_error("gj_mp_steps_reduce: %s (step %d)", why, s); return rc; }
    if (gj_mp_step_partials_bytes(descs[s]) == 0) {
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
int gj_bench_edge_fwd_only(const gj_mp_desc* d, const float* h, const float* params, float* e_out, void* workspace,
                           size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  MPLayout L; const char* why;
  int rc = gj_fill_arch(d, &L, &why);
  if (rc || !h || !params || !e_out || !workspace) { gj_set_error("gj_bench_edge_fwd_only: %s", rc ? why : "null pointer"); return GJ_ERR_INVALID; }
  if (!tc2_path(L, d->precision)) { gj_set_error("gj_bench_edge_fwd_only: step does not run the fused tensor-core kernel"); return GJ_ERR_INVALID; }
  const StepWs w = plan_ws(L, d->precision, false);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("gj_bench_edge_fwd_only: workspace too small"); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  return gj_edge_fwd2(L, h, ws + w.pq, params, e_out, ws + w.epart, ws + w.wimg, nullptr, (cudaStream_t)stream, true, false);
}

int gj_bench_edge_bwd_only(const gj_mp_desc* d, const float* h, const float* params, float* dh, float* dparams, void* workspace,
                           size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  MPLayout L; const char* why;
  int rc = gj_fill_arch(d, &L, &why);
  if (rc || !h || !params || !dh || !dparams || !workspace) { gj_set_error("gj_bench_edge_bwd_only: %s", rc ? why : "null pointer"); return GJ_ERR_INVALID; }
  if (!tc2_path(L, d->precision)) { gj_set_error("gj_bench_edge_bwd_only: step does not run the fused tensor-core kernel"); return GJ_ERR_INVALID; }
  const StepWs w = plan_ws(L, d->precision, true);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("gj_bench_edge_bwd_only: workspace too small"); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  return gj_edge_bwd2(L, h, ws + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, ws + w.wimg, ws + w.dist, true,
                      (cudaStream_t)stream, 1, nullptr, nullptr, nullptr);
}

/* As gj_bench_edge_bwd_only, for the step as the trainer runs it: `saved` was filled by gj_mp_step_fwd_saving and `workspace`
 * by the gj_mp_step_bwd_saved call that followed. */
int gj_bench_edge_bwd_saved_only(const gj_mp_desc* d, const float* h, const float* params, float* dh, float* dparams, const void* saved,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  g_err[0] = 0;
  MPLayout L; const char* why;
  int rc = gj_fill_arch(d, &L, &why);
  if (rc || !h || !params || !dh || !dparams || !saved || !workspace) { gj_set_error("gj_bench_edge_bwd_saved_only: %s", rc ? why : "null pointer"); return GJ_ERR_INVALID; }
  if (!tc2_path(L, d->precision)) { gj_set_error("gj_bench_edge_bwd_saved_only: step does not run the fused tensor-core kernel"); return GJ_ERR_INVALID; }
  const StepWs w = plan_ws(L, d->precision, true);
  if (workspace_bytes < w.total * sizeof(float)) { gj_set_error("gj_bench_edge_bwd_saved_only: workspace too small"); return GJ_ERR_WORKSPACE; }
  float* ws = (float*)workspace;
  float* pre = (float*)saved;
  return gj_edge_bwd2(L, h, pre + w.pq, params, ws + w.de, ws + w.dpq, dh, dparams, ws + w.part, pre + w.wimg, pre + w.dist, true,
                      (cudaStream_t)stream, 1, nullptr, nullptr, nullptr);
}

int gj_mp_plan_info(const gj_mp_desc* d, int32_t* info) {
  g_err[0] = 0;
  MPLayout L; const char* why;
  int rc = gj_fill_arch(d, &L, &why);
  if (rc || !info) { gj_set_error("gj_mp_plan_info: %s", rc ? why : "null pointer"); return GJ_ERR_INVALID; }
  gj_tc_plan_info(L, info);
  {      // the second-generation kernels take over where their widths are compiled in
    if (tc2_path(L, d->precision)) { gj_fwd2_plan(L, info + 0, info + 1); gj_bwd2_plan(L, info + 2, info + 3); }
  }
  return GJ_OK;
}

int gj_umma_selftest(int32_t m, int32_t n, int32_t k, int32_t a_major, int32_t b_major, const float* a, const float* b,
                     float* out, void* stream) {
  g_err[0] = 0;
  if (!a || !b || !out) { gj_set_error("gj_umma_selftest: null pointer"); return GJ_ERR_INVALID; }
  return gj_umma_selftest_launch(m, n, k, a_major, b_major, a, b, out, (cudaStream_t)stream);
}

}  // extern "C"
