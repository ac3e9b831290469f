// Shared host/device definitions for the GraphNet message-passing kernels (sm_100a).
//
// One message-passing step (reference models/graphnet.py:154-168) is evaluated per jet as
//   P_i = Wa h_i + b0,  Q_j = Wb h_j,  d_ij = metric(h_j - h_i + eps)            (node level, N rows)
//   a0_ij = leaky(P_i + Q_j + wd d_ij)                                           (first edge layer, factorised:
//                                                    W0 [h_i|h_j|d] = Wa h_i + Wb h_j + wd d, graphnet.py:220)
//   a_l = leaky(W_l a_{l-1} + b_l), l = 1..Le-1                                  (dense edge layers, N^2 rows)
//   e_i = sum_j a_{Le-1,ij};  h'_i = NodeNet([e_i | h_i])                        (graphnet.py:243-246,266-268)
// Edge rows are tiled as (TI i's) x (32 j's); padded j's and i's are masked at the sum / at dz_{Le-1}.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "gnnjet_b200.h"

#define GJ_THREADS 256
#define GJ_EPS 1e-16f   // reference utils/const.py:5
#define GJ_IB 32        // nodes per i-block

struct MPLayout {
  int B, N, H, Hs, Npad;
  int ld, cols;  // row stride of h / dh in HBM, columns present in memory (rest are zeros)
  int Le, Ln;
  int E[GJ_MAX_LAYERS], Ep[GJ_MAX_LAYERS];  // edge layer output widths, padded to 16
  int K[GJ_MAX_LAYERS], Kp[GJ_MAX_LAYERS];  // edge layer input widths (K[0] = 2H+1; Kp[0] unused)
  int pW[GJ_MAX_LAYERS], pb[GJ_MAX_LAYERS]; // offsets into the packed parameter block
  int O[GJ_MAX_LAYERS], I[GJ_MAX_LAYERS], Is[GJ_MAX_LAYERS];
  int pV[GJ_MAX_LAYERS], pc[GJ_MAX_LAYERS];
  int nparams;
  int Hout, EL, ELp, ELs, E0p, E0s, Ws;
  float alpha;
  int mink;      // 1: minkowskian signs (+,-,-,-) (only when H == 4)
  int R, Rs;     // rows per tile, padded row stride of activation buffers (floats)
  // shared-memory offsets, in floats
  int o_wE[GJ_MAX_LAYERS], o_bE[GJ_MAX_LAYERS];
  int o_wa, o_wb, o_wd;
  int o_V[GJ_MAX_LAYERS], o_c[GJ_MAX_LAYERS];
  int o_h, o_hj, o_Q, o_P, o_e;
  int n_edge_dpar;
  int o_act[GJ_MAX_LAYERS];
  int o_node[GJ_MAX_LAYERS + 3];
  // backward only
  int o_dpar, o_dh, o_dQ, o_dP, o_de, o_G, Gs, o_drow;
  int smem_floats;
};

static inline int gj_round_up(int x, int m) { return (x + m - 1) / m * m; }

// Validates the descriptor and fills the architecture part of the layout. Returns 0 or GJ_ERR_*.
static inline int gj_fill_arch(const gj_mp_desc* d, MPLayout* L, const char** why) {
  memset(L, 0, sizeof(*L));
  *why = "";
  if (!d) { *why = "null descriptor"; return GJ_ERR_INVALID; }
  if (d->batch < 0 || d->num_nodes < 1 || d->node_in < 1) { *why = "batch/num_nodes/node_in out of range"; return GJ_ERR_INVALID; }
  if (d->n_edge_layers < 1 || d->n_edge_layers > GJ_MAX_LAYERS || d->n_node_layers < 1 || d->n_node_layers > GJ_MAX_LAYERS) {
    *why = "layer count out of range"; return GJ_ERR_INVALID; }
  if (!(d->alpha >= 0.f)) { *why = "alpha must be >= 0 (the LeakyReLU mask is recovered from the output sign)"; return GJ_ERR_INVALID; }
  L->B = d->batch; L->N = d->num_nodes; L->H = d->node_in; L->Hs = d->node_in | 1;
  L->Npad = gj_round_up(L->N, 32);
  L->ld = d->h_ld > 0 ? d->h_ld : L->H;
  L->cols = d->h_cols > 0 ? d->h_cols : L->H;
  if (L->cols > L->H || L->cols > L->ld) { *why = "h_cols must be <= node_in and <= h_ld"; return GJ_ERR_INVALID; }
  L->Le = d->n_edge_layers; L->Ln = d->n_node_layers;
  L->alpha = d->alpha;
  L->mink = (d->metric == GJ_METRIC_MINKOWSKIAN && d->node_in == 4) ? 1 : 0;
  int off = 0;
  for (int l = 0; l < L->Le; ++l) {
    if (d->edge_widths[l] < 1 || d->edge_widths[l] > 256) { *why = "edge width out of range [1,256]"; return GJ_ERR_INVALID; }
    L->E[l] = d->edge_widths[l]; L->Ep[l] = gj_round_up(L->E[l], 16);
    L->K[l] = l == 0 ? 2 * L->H + 1 : L->E[l - 1];
    L->Kp[l] = l == 0 ? 0 : L->Ep[l - 1];
    L->pW[l] = off; off += L->E[l] * L->K[l];
    L->pb[l] = off; off += L->E[l];
  }
  L->EL = L->E[L->Le - 1]; L->ELp = L->Ep[L->Le - 1]; L->ELs = L->ELp + 1;
  L->E0p = L->Ep[0]; L->E0s = L->E0p + 1;
  int wmax = L->EL + L->H;
  for (int m = 0; m < L->Ln; ++m) {
    if (d->node_widths[m] < 1 || d->node_widths[m] > 1024) { *why = "node width out of range"; return GJ_ERR_INVALID; }
    L->O[m] = d->node_widths[m];
    L->I[m] = m == 0 ? L->EL + L->H : L->O[m - 1];
    L->Is[m] = L->I[m] | 1;
    L->pV[m] = off; off += L->O[m] * L->I[m];
    L->pc[m] = off; off += L->O[m];
    if (L->O[m] > wmax) wmax = L->O[m];
  }
  L->Ws = wmax | 1;
  L->Hout = L->O[L->Ln - 1];
  L->nparams = off;
  return GJ_OK;
}

#ifdef __CUDACC__
// ---- programmatic dependent launch (PDL) ----
// A kernel launched with the programmatic-stream-serialization attribute may be launched, and its CTAs made resident, while
// the preceding kernel of the stream still runs.  Correctness rests on one rule: every kernel launched through gj_launch /
// gj_launch_edge executes gj_pdl_wait() as its FIRST statement, before any global-memory access and before any early return
// (the wait returns when every preceding grid has completed and its memory is visible, so dependencies stay transitive along
// the chain).  gj_pdl_trigger() lets the dependent grid launch: short kernels call it right after the wait, the persistent
// edge kernels after their tile loop.  Both instructions are no-ops in a kernel launched without the attribute.
// Measured on a B200 (profiles/r02_pdl_ab.txt, config 2): on the persistent edge kernels the attribute hides their
// prologue (barriers, TMEM allocation, the TMA of the parameter image) behind the predecessor's tail, 482.5 -> 479.5 us per
// backward launch; on the 5-40 us node-level kernels it helps when the step is launched kernel by kernel (4.88 -> 4.81 ms)
// and HURTS inside a CUDA graph, whose kernel-to-kernel hand-over is already tighter than a programmatic edge (4.72 -> 4.80
// ms).  Default therefore: edge kernels always, the other kernels only when the stream is not being captured;
// GJ_PDL = 0 / 1 / 2 / 3 forces none / small only / edge only / all.
__device__ __forceinline__ void gj_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void gj_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void gj_pdl_sync() { gj_pdl_wait(); gj_pdl_trigger(); }

int gj_pdl_mode();      // api.cu: environment GJ_PDL (bit 0: node-level / small kernels, bit 1: edge kernels), -1 = default policy

// <<<grid, block, smem, stream>>> with the PDL attribute (kernel class `mask`: 1 small, 2 edge); the kernel MUST start with
// gj_pdl_wait() / gj_pdl_sync()
template <typename... KArgs, typename... Args>
static inline cudaError_t gj_launch_masked(int mask, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                           Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  const int mode = gj_pdl_mode();
  bool on;
  if (mode >= 0) on = (mode & mask) != 0;
  else if (mask & 2) on = true;
  else {      // small kernels: not inside a graph capture (the legacy default stream cannot be captured)
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    on = stream == nullptr || (cudaStreamIsCapturing(stream, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone);
  }
  cfg.attrs = attr; cfg.numAttrs = on ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<Args&&>(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t gj_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  return gj_launch_masked(1, kern, grid, block, smem, stream, static_cast<Args&&>(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t gj_launch_edge(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  return gj_launch_masked(2, kern, grid, block, smem, stream, static_cast<Args&&>(args)...);
}

__device__ __forceinline__ float gj_leaky(float z, float a) { return z > 0.f ? z : a * z; }
// LeakyReLU as FMUL + FMNMX: max(z, a z) for a <= 1, min(z, a z) for a > 1 (a >= 0 is validated on the host)
__device__ __forceinline__ float gj_leaky2(float z, float a, bool a_le_1) { const float y = a * z; return a_le_1 ? fmaxf(z, y) : fminf(z, y); }
__device__ __forceinline__ float gj_slope(float y, float a) { return y > 0.f ? 1.f : a; }
__device__ __forceinline__ float gj_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// losses._to_polar of one Cartesian momentum, operation by operation and without contraction, so that a loss kernel sees the
// values torch computes: pt = sqrt(px^2 + py^2 + eps), eta = asinh(pz / (pt + eps)), phi = atan2(py + eps, px + eps)
__device__ __forceinline__ float3 gj_to_polar(float px, float py, float pz) {
  const float pt = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(px, px), __fmul_rn(py, py)), GJ_EPS));
  return make_float3(pt, asinhf(__fdiv_rn(pz, __fadd_rn(pt, GJ_EPS))), atan2f(__fadd_rn(py, GJ_EPS), __fadd_rn(px, GJ_EPS)));
}

// Chain rule through gj_to_polar: the gradient (g_pt, g_eta, g_phi) at (px, py, pz) in fp64 -> (d/dpx, d/dpy, d/dpz)
__device__ __forceinline__ void gj_to_polar_grad(float px, float py, float pz, double g0, double g1, double g2, double& gx,
                                                 double& gy, double& gz) {
  const float pt = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(px, px), __fmul_rn(py, py)), GJ_EPS));
  const double den = (double)__fadd_rn(pt, GJ_EPS), sh = (double)__fdiv_rn(pz, __fadd_rn(pt, GJ_EPS));
  const double deta = g1 / sqrt(1.0 + sh * sh);                       // d/d(pz / (pt + eps))
  const double gpt = g0 - deta * sh / den;                              // total d/dpt
  const double xe = (double)__fadd_rn(px, GJ_EPS), ye = (double)__fadd_rn(py, GJ_EPS), r2 = xe * xe + ye * ye;
  gx = gpt * (double)px / (double)pt - g2 * ye / r2;
  gy = gpt * (double)py / (double)pt + g2 * xe / r2;
  gz = deta / den;
}
#endif
