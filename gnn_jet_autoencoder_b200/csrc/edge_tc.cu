// bf16 (GJ_PREC_BF16) edge kernels on tcgen05 tensor cores with TMEM accumulators.
//
// Work decomposition: a CTA holds NWG independent warpgroups (128 threads = 128 TMEM lanes each).  Every
// warpgroup walks whole jets on its own: for a jet the N x N pair set is visited as (32 i's) x (32 j's) blocks,
// each block as tiles of 128 edge rows (4 i's x 32 j's, j on the lanes).  Per tile:
//   a0 = leaky(P_i + Q_j + wd d_ij)            CUDA cores, fp32 -> bf16 A operand in shared memory
//   a_l = leaky(W_l a_{l-1} + b_l), l >= 1     tcgen05.mma (M = 128 rows, N = layer width, K = previous width)
//                                              issued by one elected thread, accumulator in the warpgroup's TMEM
//                                              columns, epilogue tcgen05.ld -> bias + LeakyReLU -> bf16 -> smem
//   e_i = sum_j a_last                         warp shuffles (fp32)
// While one warpgroup runs an epilogue, the other's MMAs occupy the tensor pipe.  Edge activations never leave
// the SM.  Replaces the edge part of reference models/graphnet.py:154-168 and its autograd adjoint.
#include "gj_common.cuh"
#include <stdlib.h>

#include "umma.cuh"

namespace {

using namespace umma;

struct Carver {
  int off = 0;
  int take(int n) { int o = off; off += (n + 3) & ~3; return o; }
};

int next_pow2_cols(int c) { int p = 32; while (p < c) p <<= 1; return p; }

// Optional timeline of the issuer / warpgroup handshake (GJ_TRACE=1 in the environment): (tag, clock) pairs of CTA 0.
__device__ long long g_trace[8192];
__device__ int g_trace_n[4];
#define GJ_TRACE_PT(who, tag)                                                                         \
  do { if (T.trace && blockIdx.x == 0 && tr_i < 1024) { g_trace[(who) * 2048 + 2 * tr_i] = (tag);     \
         g_trace[(who) * 2048 + 2 * tr_i + 1] = clock64(); ++tr_i; } } while (0)
#define GJ_TRACE_END(who) do { if (T.trace && blockIdx.x == 0) g_trace_n[who] = tr_i; } while (0)

struct TCPlan {
  int nwg, trace;
  int o_bar, o_tmem_slot, o_tbl;
  int o_wT[GJ_MAX_LAYERS];  // bf16 interleaved edge weights, layers >= 1 (bytes from smem base)
  int o_shared_f32;         // float region shared by all warpgroups (biases, wd)
  int wg_base, wg_stride;   // per-warpgroup region
  int w_act[GJ_MAX_LAYERS]; // bf16 activation buffers inside the warpgroup region (bytes)
  int w_f32;                // float region inside the warpgroup region
  int acc_cols, tmem_cols_per_wg, tmem_cols_total;   // two accumulator buffers of acc_cols columns per warpgroup
  int smem_bytes;
};

// Fills the float offsets of L relative to the two float regions and the byte plan T.
// row strides of the fp32 blocks: multiples of 4 floats with (stride / 4) odd, so that per-lane rows can be read with
// conflict-free 16-byte loads
static void tc_strides(MPLayout* L) {
  L->Hs = ((L->H + 7) & ~7) + 4;
  L->E0s = L->E0p + 4;
  L->ELs = L->ELp + 4;
  L->Gs = 36;
}

void plan_tc_fwd(MPLayout* L, TCPlan* T, int nwg) {
  L->R = 128; L->Rs = 0;
  tc_strides(L);
  T->nwg = nwg; T->trace = 0;
  Carver c;
  for (int l = 1; l < L->Le; ++l) L->o_bE[l] = c.take(L->Ep[l]);
  L->o_wd = c.take(L->E0p);
  Carver w;
  L->o_h = w.take(GJ_IB * L->Hs);
  L->o_hj = w.take(32 * L->Hs);
  L->o_P = w.take(GJ_IB * L->E0s);
  L->o_Q = w.take(32 * L->E0s);
  L->o_e = w.take(GJ_IB * L->ELs);
  int off = 0;
  T->o_bar = off; off += gj_round_up(nwg * (1 + 16) * 8, 64);
  T->o_tmem_slot = off; off += 64;
  T->o_tbl = off; off += gj_round_up(nwg * GJ_MAX_LAYERS * 40, 128);
  for (int l = 1; l < L->Le; ++l) { T->o_wT[l] = off; off += L->Ep[l] * L->Kp[l] * 2; }
  T->o_shared_f32 = off; off += c.off * 4;
  off = gj_round_up(off, 128);
  T->wg_base = off;
  int wo = 0;
  for (int l = 0; l + 1 < L->Le; ++l) { T->w_act[l] = wo; wo += L->Ep[l] * 128 * 2; }
  T->w_f32 = wo; wo += w.off * 4;
  wo = gj_round_up(wo, 128);
  T->wg_stride = wo;
  T->smem_bytes = T->wg_base + nwg * wo;
  int mx = 32;
  for (int l = 1; l < L->Le; ++l) if (L->Ep[l] > mx) mx = L->Ep[l];
  T->acc_cols = gj_round_up(mx, 32);
  T->tmem_cols_per_wg = 2 * T->acc_cols;
  T->tmem_cols_total = next_pow2_cols(T->tmem_cols_per_wg * nwg);
}

__device__ void stage_small(const MPLayout& L, const float* __restrict__ params, float* smf, int tid, int nthr) {
  for (int l = 1; l < L.Le; ++l)
    for (int c = tid; c < L.Ep[l]; c += nthr) smf[L.o_bE[l] + c] = c < L.E[l] ? __ldg(params + L.pb[l] + c) : 0.f;
  for (int c = tid; c < L.E0p; c += nthr) smf[L.o_wd + c] = c < L.E[0] ? __ldg(params + L.pW[0] + c * L.K[0] + 2 * L.H) : 0.f;
}

// bf16 interleaved staging of edge weights l >= 1 as the K-major B operand (N = out feature rows, K = in).
__device__ void stage_edge_weights_bf16(const MPLayout& L, const int* o_wT, const float* __restrict__ params, uint8_t* smem,
                                        int tid, int nthr) {
  for (int l = 1; l < L.Le; ++l) {
    uint8_t* w = smem + o_wT[l];
    const int Ep = L.Ep[l], Kp = L.Kp[l], E = L.E[l], K = L.K[l];
    for (int idx = tid; idx < Ep * Kp; idx += nthr) {
      int n = idx / Kp, k = idx - n * Kp;
      float v = (n < E && k < K) ? __ldg(params + L.pW[l] + n * K + k) : 0.f;
      *reinterpret_cast<__nv_bfloat16*>(w + il_off(n, k, Ep)) = __float2bfloat16_rn(v);
    }
  }
}

// rows [r0, r0 + 32) of h (zero padded) and of the P or Q half of PQ, by one warpgroup.  Loads are batched
// (all of a thread's global loads are issued before the first use) and 16 bytes wide where the layout allows.
__device__ void wg_load_block(const MPLayout& L, const float* __restrict__ hjet, const float* __restrict__ pqjet, int half,
                              int r0, float* sh, float* spq, int t, int nthr = 128) {
  const int q4 = L.E0p >> 2;                       // float4 per P/Q row (E0p is a multiple of 16)
#pragma unroll 2
  for (int idx = t; idx < 32 * q4; idx += nthr) {
    const int n = idx / q4, c = (idx - n * q4) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + n < L.N) v = __ldg(reinterpret_cast<const float4*>(pqjet + (size_t)(r0 + n) * 2 * L.E0p + half * L.E0p + c));
    *reinterpret_cast<float4*>(spq + n * L.E0s + c) = v;
  }
#pragma unroll 4
  for (int idx = t; idx < 32 * L.H; idx += nthr) {
    int n = idx / L.H, k = idx - n * L.H;
    sh[n * L.Hs + k] = (r0 + n < L.N && k < L.cols) ? __ldg(hjet + (size_t)(r0 + n) * L.ld + k) : 0.f;
  }
}

// first edge layer of one tile on CUDA cores: thread t owns row (i = it*4 + wq, j = lane); returns d_ij.
// All shared-memory rows are read 16 bytes at a time (h_i, P_i, wd: warp broadcasts; h_j, Q_j: one row per lane).
// With two warps per TMEM lane quadrant (NH = 2) the warp pair of a row splits the channels 8 by 8 (part = 0 / 1).
__device__ __forceinline__ float tc_layer0(const MPLayout& L, const float* sm_h, const float* sm_hj, const float* sm_P,
                                           const float* sm_Q, const float* wd, uint8_t* a0, int il, int lane, int t,
                                           int part = 0, int nparts = 1) {
  const float* hi = sm_h + il * L.Hs;
  const float* hj = sm_hj + lane * L.Hs;
  float d = 0.f;
  if (L.mink) {          // width 4 only: x0^2 - x1^2 - x2^2 - x3^2 (graphnet.py:320-323)
    const float4 a = *reinterpret_cast<const float4*>(hi), b = *reinterpret_cast<const float4*>(hj);
    const float x0 = b.x - a.x + GJ_EPS, x1 = b.y - a.y + GJ_EPS, x2 = b.z - a.z + GJ_EPS, x3 = b.w - a.w + GJ_EPS;
    d = x0 * x0 - x1 * x1 - x2 * x2 - x3 * x3;
  } else {
    const int H4 = L.H & ~3;
    for (int k = 0; k < H4; k += 4) {
      const float4 a = *reinterpret_cast<const float4*>(hi + k), b = *reinterpret_cast<const float4*>(hj + k);
      const float x0 = b.x - a.x + GJ_EPS, x1 = b.y - a.y + GJ_EPS, x2 = b.z - a.z + GJ_EPS, x3 = b.w - a.w + GJ_EPS;
      d = fmaf(x0, x0, d); d = fmaf(x1, x1, d); d = fmaf(x2, x2, d); d = fmaf(x3, x3, d);
    }
    for (int k = H4; k < L.H; ++k) { const float x = hj[k] - hi[k] + GJ_EPS; d = fmaf(x, x, d); }
  }
  const float* P = sm_P + il * L.E0s;
  const float* Q = sm_Q + lane * L.E0s;
  const bool a_le_1 = L.alpha <= 1.f;
  for (int c0 = 8 * part; c0 < L.E0p; c0 += 8 * nparts) {
    float p[8], q[8], w[8], v[8];
    *reinterpret_cast<float4*>(p) = *reinterpret_cast<const float4*>(P + c0);
    *reinterpret_cast<float4*>(p + 4) = *reinterpret_cast<const float4*>(P + c0 + 4);
    *reinterpret_cast<float4*>(q) = *reinterpret_cast<const float4*>(Q + c0);
    *reinterpret_cast<float4*>(q + 4) = *reinterpret_cast<const float4*>(Q + c0 + 4);
    *reinterpret_cast<float4*>(w) = *reinterpret_cast<const float4*>(wd + c0);
    *reinterpret_cast<float4*>(w + 4) = *reinterpret_cast<const float4*>(wd + c0 + 4);
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float z = fmaf(w[i], d, p[i] + q[i]); v[i] = fmaxf(z, L.alpha * z); }
    uint4 pk = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    *reinterpret_cast<uint4*>(a0 + (c0 >> 3) * 2048 + t * 16) = pk;
  }
  return d;
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Wait of a whole tile group on an mbarrier: only its first warp polls (a polling warp burns issue slots every time
// the hardware sleep is woken by unrelated barrier traffic); the other warps block on a hardware named barrier, which
// costs no issue slots, and are released when the polling warp joins it.
__device__ __forceinline__ void group_wait(uint64_t* bar, uint32_t parity, bool poller, int bar_id, int nthreads) {
  if (poller) mbar_wait(bar, parity);
  named_bar_sync(bar_id, nthreads);
}

// one arrival per warp (the barrier counts warps): 128-256 same-address arrivals would serialise in the smem atomic unit
__device__ __forceinline__ void warp_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
}

// transpose-reduce of 16 per-lane values over the 32 lanes of a warp: returns, in every lane, the sum over all lanes
// of channel (lane >> 1) & 15   (31 adds + 16 shuffles instead of 80 + 80)
__device__ __forceinline__ float warp_transpose_sum16(const float (&v)[16], int lane) {
  float w8[8], w4[4], w2[2];
  bool up = lane & 16;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    float send = up ? v[q] : v[q + 8], keep = up ? v[q + 8] : v[q];
    w8[q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  up = lane & 8;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float send = up ? w8[q] : w8[q + 4], keep = up ? w8[q + 4] : w8[q];
    w4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  up = lane & 4;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    float send = up ? w4[q] : w4[q + 2], keep = up ? w4[q + 2] : w4[q];
    w2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  up = lane & 2;
  float send = up ? w2[0] : w2[1], keep = up ? w2[1] : w2[0];
  float w1 = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  return w1 + __shfl_xor_sync(0xffffffffu, w1, 1);
}

// ---- the issuer's MMA batches -----------------------------------------------------------------------------
// A/B K-major buffer with nrows rows: next 8 rows +128 B (SBO), next 8 columns +nrows*16 B (LBO), 16 columns per MMA
// A/B MN-major view of the same bytes (MN = column, K = row): next 8 columns +nrows*16 B (SBO), next 8 rows +128 B (LBO)
// One group = the k-steps of one GEMM: descriptors of k-step 0 plus the per-step advance, built once per kernel.
// v[q] = leaky(v[q] + b[q]) for 16 values; the alpha <= 1 test is taken once, not per value (FADD + FMUL + FMNMX each)
// (the tensor-core kernels are only launched for 0 <= alpha <= 1, where LeakyReLU(z) = max(z, alpha z))
__device__ __forceinline__ void bias_leaky16(float (&v)[16], const float* bq, float alpha, bool) {
#pragma unroll
  for (int q = 0; q < 16; ++q) { const float z = v[q] + bq[q]; v[q] = fmaxf(z, alpha * z); }
}

// Epilogue walk over a thread's 16-column accumulator chunks (chunk = part, part + nparts, ...) with two register
// sets: the next chunk's TMEM load flies while the current one is processed.
template <typename F>
__device__ __forceinline__ void for_chunks(uint32_t tmem_row, int nch, int part, int nparts, F&& process) {
  float va[16], vb[16];
  int ch = part;
  if (ch >= nch) return;
  tmem_ld16_issue(tmem_row + (uint32_t)(ch << 4), va);
  for (; ch < nch; ch += 2 * nparts) {
    tmem_wait16(va);
    if (ch + nparts < nch) tmem_ld16_issue(tmem_row + (uint32_t)((ch + nparts) << 4), vb);
    process(va, ch << 4);
    if (ch + nparts < nch) {
      tmem_wait16(vb);
      if (ch + 2 * nparts < nch) tmem_ld16_issue(tmem_row + (uint32_t)((ch + 2 * nparts) << 4), va);
      process(vb, (ch + nparts) << 4);
    }
  }
}

struct MmaGroup {
  unsigned long long a, b;
  uint32_t d, idesc, astep, bstep;   // astep/bstep in 16-byte units
  short nk, commit;                  // commit: after this group, tcgen05.commit to 0 nothing / 1 done[wg] / 2 done2[wg]
  int accbit;                        // accbit >= 0: shared accumulator id (accumulate unless it is the first write)
};

static_assert(sizeof(MmaGroup) == 40, "plan_tc_bwd reserves 40 bytes per group");

__device__ __forceinline__ MmaGroup grp_fwd(uint32_t d, uint32_t a, uint32_t w, int N, int K) {
  // acc[128 x N] = act[128 x K] W[N x K]^T, both K-major
  return MmaGroup{make_smem_desc(a, 2048, 128), make_smem_desc(w, N * 16, 128), d, make_idesc_bf16(128, N, 0, 0), 4096u >> 4,
                  (uint32_t)(2 * N * 16) >> 4, (short)(K / 16), 0, -1};
}
__device__ __forceinline__ MmaGroup grp_dgrad(uint32_t d, uint32_t dz, uint32_t w, int Kin, int Eout) {
  // acc[128 x Kin] = dz[128 x Eout] W[Eout x Kin]: A = dz K-major, B = W viewed MN-major (MN = in feature, K = out feature)
  return MmaGroup{make_smem_desc(dz, 2048, 128), make_smem_desc(w, 128, Eout * 16), d, make_idesc_bf16(128, Kin, 0, 1), 4096u >> 4,
                  256u >> 4, (short)(Eout / 16), 0, -1};
}
__device__ __forceinline__ MmaGroup grp_wgrad(uint32_t d, uint32_t x, uint32_t y, int M, int N, int accbit) {
  // D[M x N] += X^T Y over the 128 tile rows: both operands MN-major views of 128-row buffers
  return MmaGroup{make_smem_desc(x, 128, 2048), make_smem_desc(y, 128, 2048), d, make_idesc_bf16(M, N, 1, 1), 256u >> 4, 256u >> 4, 8, 0,
                  accbit};
}
__device__ __forceinline__ MmaGroup grp_colsum(uint32_t d, uint32_t x, uint32_t ones, int M, int accbit) {
  // D[M x 16] += X^T 1: column sums of a 128-row buffer (ones operand: K-major [16][128])
  return MmaGroup{make_smem_desc(x, 128, 2048), make_smem_desc(ones, 256, 128), d, make_idesc_bf16(M, 16, 1, 0), 256u >> 4, 512u >> 4, 8, 0,
                  accbit};
}
// executed by all 32 lanes of the issuer warp (convergent); fields are broadcast so they live in uniform registers
__device__ __forceinline__ int run_group(const MmaGroup* g, uint32_t& inited) {
  const uint64_t a = uni64(g->a), b = uni64(g->b);
  const uint32_t d = uni(g->d), idesc = uni(g->idesc), astep = uni(g->astep), bstep = uni(g->bstep);
  const int nk = (int)uni((uint32_t)g->nk), accbit = (int)uni((uint32_t)g->accbit), commit = (int)uni((uint32_t)g->commit);
  uint32_t accumulate = 0;
  if (accbit >= 0) { accumulate = (inited >> accbit) & 1u; inited |= 1u << accbit; }
  for (int ks = 0; ks < nk; ++ks)
    mma_bf16_ss_elect(d, desc_advance(a, astep, ks), desc_advance(b, bstep, ks), idesc, (accumulate | (uint32_t)(ks > 0)));
  return commit;
}

__device__ __forceinline__ int tiles_of_jet(const MPLayout& L) {
  int n = 0;
  const int njb = (L.N + 31) / 32;
  for (int i0 = 0; i0 < L.N; i0 += GJ_IB) n += ((min(GJ_IB, L.N - i0) + 3) / 4) * njb;
  return n;
}

// pieces of the first edge layer for the streaming forward kernel
__device__ __forceinline__ float tc_pair_distance(const MPLayout& L, const float* hi, const float* hj) {
  float d = 0.f;
  if (L.mink) {
    const float4 a = *reinterpret_cast<const float4*>(hi), b = *reinterpret_cast<const float4*>(hj);
    const float x0 = b.x - a.x + GJ_EPS, x1 = b.y - a.y + GJ_EPS, x2 = b.z - a.z + GJ_EPS, x3 = b.w - a.w + GJ_EPS;
    d = x0 * x0 - x1 * x1 - x2 * x2 - x3 * x3;
  } else {
    const int H4 = L.H & ~3;
    for (int k = 0; k < H4; k += 4) {
      const float4 a = *reinterpret_cast<const float4*>(hi + k), b = *reinterpret_cast<const float4*>(hj + k);
      const float x0 = b.x - a.x + GJ_EPS, x1 = b.y - a.y + GJ_EPS, x2 = b.z - a.z + GJ_EPS, x3 = b.w - a.w + GJ_EPS;
      d = fmaf(x0, x0, d); d = fmaf(x1, x1, d); d = fmaf(x2, x2, d); d = fmaf(x3, x3, d);
    }
    for (int k = H4; k < L.H; ++k) { const float x = hj[k] - hi[k] + GJ_EPS; d = fmaf(x, x, d); }
  }
  return d;
}
// channels [c0, c0 + 16) of a0 = leaky(P_i + Q_j + wd d_ij) for one row -> bf16 A operand (dst already points at the row)
__device__ __forceinline__ void tc_layer0_chunk(const MPLayout& L, const float* P, const float* Q, const float* wd, uint8_t* dst,
                                                int c0, float d, bool a_le_1) {
#pragma unroll
  for (int h8 = 0; h8 < 2; ++h8) {
    const int c = c0 + 8 * h8;
    float p[8], q[8], w[8], v[8];
    *reinterpret_cast<float4*>(p) = *reinterpret_cast<const float4*>(P + c);
    *reinterpret_cast<float4*>(p + 4) = *reinterpret_cast<const float4*>(P + c + 4);
    *reinterpret_cast<float4*>(q) = *reinterpret_cast<const float4*>(Q + c);
    *reinterpret_cast<float4*>(q + 4) = *reinterpret_cast<const float4*>(Q + c + 4);
    *reinterpret_cast<float4*>(w) = *reinterpret_cast<const float4*>(wd + c);
    *reinterpret_cast<float4*>(w + 4) = *reinterpret_cast<const float4*>(wd + c + 4);
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float z = fmaf(w[i], d, p[i] + q[i]); v[i] = fmaxf(z, L.alpha * z); }
    *reinterpret_cast<uint4*>(dst + (c >> 3) * 2048) =
        make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  }
}

// Handshake between the compute warpgroups and the MMA-issuer warp (both tensor-core kernels):
//   warpgroup: write operands to smem -> fence.proxy.async -> arrive(ready[wg])      wait(done[wg]) -> epilogue from TMEM
//   issuer   : wait(ready[wg]) -> issue the stage's tcgen05.mma batch -> tcgen05.commit -> arrive(done[wg])
// The issuer warp runs warp-convergent code only, so its descriptors stay in uniform registers.

// NH = warps per TMEM lane quadrant of a tile: 1 -> 128 threads per tile, 2 -> 256 (the pair splits the column chunks).
//
// The forward kernel STREAMS layer l+1's MMA behind layer l's epilogue: the epilogue publishes every 16-column chunk of
// a_l (one k-step of layer l+1) on its own mbarrier, the issuer issues that k-step as soon as the chunk is complete, and
// the accumulators alternate between two TMEM buffers (layer l reads buffer l&1 while layer l+1 fills the other), so a
// warpgroup only waits for the tail of an MMA batch instead of the whole batch.
#define GJ_MAX_CHUNKS 16
template <int NWG, int NH>
__global__ void __launch_bounds__(NWG * 128 * NH + NWG * 32, 1)
edge_fwd_tc_kernel(const MPLayout L, const TCPlan T, const float* __restrict__ h, const float* __restrict__ pq,
                   const float* __restrict__ params, float* __restrict__ e_out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int TGT = 128 * NH;            // threads per tile group
  constexpr int NT = NWG * TGT + NWG * 32;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = (int)uni((uint32_t)(tid >> 5));     // provably warp-uniform
  const bool is_issuer = warp >= NWG * 4 * NH;
  float* smf = reinterpret_cast<float*>(smem + T.o_shared_f32);
  // barriers: done[wg] = bars[wg]; chunk[wg][c] = bars[NWG + wg * GJ_MAX_CHUNKS + c]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + T.o_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + T.o_tmem_slot);
  const int Le = L.Le;

  stage_small(L, params, smf, tid, NT);
  stage_edge_weights_bf16(L, T.o_wT, params, smem, tid, NT);
  if (tid == 0) {
    for (int w = 0; w < NWG; ++w) {
      mbar_init(bars + w, 1);
      for (int c = 0; c < GJ_MAX_CHUNKS; ++c) mbar_init(bars + NWG + w * GJ_MAX_CHUNKS + c, 4);   // the 4 row quadrants
    }
    fence_barrier_init();
  }
  if (warp == NWG * 4 * NH) tmem_alloc(tmem_slot, (uint32_t)T.tmem_cols_total);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  int tr_i = 0;      // trace cursor (register; written back once at the end)

  if (is_issuer) {
    // =================================== MMA issuers (warp-convergent) ===================================
    // One issuer warp per warpgroup (the forward kernel has no shared accumulators, so no ordering between them is
    // needed): it sleeps on the next chunk barrier and issues that k-step the moment the chunk is complete.
    const int w = warp - NWG * 4 * NH;
    const int S = Le - 1;
    const int tpj = tiles_of_jet(L);
    MmaGroup* tbl = reinterpret_cast<MmaGroup*>(smem + T.o_tbl) + w * S;      // [NWG][S]
    if (lane == 0) {
      const uint32_t wgb = smem_u32(smem + T.wg_base + w * T.wg_stride);
      for (int l = 1; l < Le; ++l)
        tbl[l - 1] = grp_fwd(tmem_base + (uint32_t)(w * T.tmem_cols_per_wg + (l & 1) * T.acc_cols), wgb + T.w_act[l - 1],
                             smem_u32(smem + T.o_wT[l]), L.Ep[l], L.Kp[l]);
    }
    __syncwarp();
    const int first = blockIdx.x * NWG + w;
    const int njets = first < L.B ? (L.B - first + gridDim.x * NWG - 1) / (gridDim.x * NWG) : 0;
    uint64_t* chunk = bars + NWG + w * GJ_MAX_CHUNKS;
    uint32_t cpar = 0;                     // parity bit per chunk barrier
    for (int tile = 0; tile < njets * tpj; ++tile) {
      for (int st = 0; st < S; ++st) {
        const MmaGroup* g = tbl + st;
        const uint64_t ga = uni64(g->a), gb = uni64(g->b);
        const uint32_t gd = uni(g->d), gi = uni(g->idesc), gas = uni(g->astep), gbs = uni(g->bstep);
        const int gnk = (int)uni((uint32_t)g->nk);
        for (int ck = 0; ck < gnk; ++ck) {
          mbar_wait(chunk + ck, (cpar >> ck) & 1u);
          __syncwarp();
          tc_fence_after();
          if (lane == 0 && ck == 0 && w == 0) GJ_TRACE_PT(2, st);
          mma_bf16_ss_elect(gd, desc_advance(ga, gas, ck), desc_advance(gb, gbs, ck), gi, ck > 0 ? 1u : 0u);
        }
        cpar ^= (1u << gnk) - 1u;
        mma_commit_elect(bars + w);
        if (lane == 0 && w == 0) GJ_TRACE_PT(2, 1000 + st);
      }
    }
    if (lane == 0 && w == 0) GJ_TRACE_END(2);
  } else {
    // =================================== compute warpgroups ===================================
    const int wg = warp / (4 * NH), w8 = warp % (4 * NH), wq = w8 & 3, part = w8 >> 2;
    const int t = tid - wg * TGT, row = wq * 32 + lane;
    uint8_t* wgb = smem + T.wg_base + wg * T.wg_stride;
    float* wgf = reinterpret_cast<float*>(wgb + T.w_f32);
    uint64_t* done = bars + wg;
    uint64_t* chunk = bars + NWG + wg * GJ_MAX_CHUNKS;
    const uint32_t tmem_row0 = tmem_base + (uint32_t)(wg * T.tmem_cols_per_wg) + ((uint32_t)(wq * 32) << 16);
    uint32_t phase = 0;
    const int bar_id = 1 + wg;
    float* sm_h = wgf + L.o_h;
    float* sm_hj = wgf + L.o_hj;
    float* sm_Q = wgf + L.o_Q;
    float* sm_P = wgf + L.o_P;
    float* sm_e = wgf + L.o_e;
    const float* wd = smf + L.o_wd;
    const bool a_le_1 = L.alpha <= 1.f;

    for (int jet = blockIdx.x * NWG + wg; jet < L.B; jet += gridDim.x * NWG) {
      const float* hjet = h + (size_t)jet * L.N * L.ld;
      const float* pqjet = pq + (size_t)jet * L.N * 2 * L.E0p;
      for (int i0 = 0; i0 < L.N; i0 += GJ_IB) {
        const int ni = min(GJ_IB, L.N - i0);
        named_bar_sync(bar_id, TGT);
        wg_load_block(L, hjet, pqjet, 0, i0, sm_h, sm_P, t, TGT);
        for (int idx = t; idx < GJ_IB * L.ELs; idx += TGT) sm_e[idx] = 0.f;
        for (int j0 = 0; j0 < L.N; j0 += 32) {
          const int nj = min(32, L.N - j0);
          named_bar_sync(bar_id, TGT);
          wg_load_block(L, hjet, pqjet, 1, j0, sm_hj, sm_Q, t, TGT);
          named_bar_sync(bar_id, TGT);
          const int nit = (ni + 3) / 4;
          for (int it = 0; it < nit; ++it) {
            const int il = it * 4 + wq;
            const bool valid = il < ni && lane < nj;
            // first layer: 16-column chunks, published one by one (each is one k-step of layer 1)
            {
              const float dij = tc_pair_distance(L, sm_h + il * L.Hs, sm_hj + lane * L.Hs);
              const int nch0 = L.E0p >> 4;
              for (int ch = part; ch < nch0; ch += NH) {
                tc_layer0_chunk(L, sm_P + il * L.E0s, sm_Q + lane * L.E0s, wd, wgb + T.w_act[0] + row * 16, ch << 4, dij, a_le_1);
                fence_proxy_async();
                warp_arrive(chunk + ch, lane);
              }
            }
            if (t == 0) GJ_TRACE_PT(wg, 10);
            for (int l = 1; l < Le; ++l) {
              group_wait(done, phase, w8 == 0, 8 + wg, TGT); phase ^= 1u;
              tc_fence_after();
              if (t == 0) GJ_TRACE_PT(wg, 20 + l);
              const bool last = (l == Le - 1);
              const float* bias = smf + L.o_bE[l];
              uint8_t* al = wgb + T.w_act[l] + row * 16;
              const int nch = L.Ep[l] >> 4;
              const uint32_t tmem_row = tmem_row0 + (uint32_t)((l & 1) * T.acc_cols);
              auto process = [&](float (&v)[16], int c0) {
                float bq[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(bq + 4 * q) = *reinterpret_cast<const float4*>(bias + c0 + 4 * q);
                bias_leaky16(v, bq, L.alpha, a_le_1);
                if (!last) {
                  uint4 p0 = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                  uint4 p1 = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
                  *reinterpret_cast<uint4*>(al + (c0 >> 3) * 2048) = p0;
                  *reinterpret_cast<uint4*>(al + ((c0 >> 3) + 1) * 2048) = p1;
                  fence_proxy_async();
                  tc_fence_before();
                  warp_arrive(chunk + (c0 >> 4), lane);      // this chunk is one k-step of the next layer
                } else {
                  // e_i += sum_j a_last (padded rows masked AFTER the activation: leaky(b) != 0); transpose-reduce over
                  // the 32 j's of the warp: lane L ends up with channel c0 + (L >> 1)
#pragma unroll
                  for (int q = 0; q < 16; ++q) v[q] = valid ? v[q] : 0.f;
                  const float s = warp_transpose_sum16(v, lane);
                  if ((lane & 1) == 0) sm_e[il * L.ELs + c0 + (lane >> 1)] += s;
                }
              };
              for_chunks(tmem_row, nch, part, NH, process);
              if (last) { tc_fence_before(); if (t == 0) GJ_TRACE_PT(wg, 60); }
              else if (t == 0) GJ_TRACE_PT(wg, 30 + l);
            }
          }
        }
        named_bar_sync(bar_id, TGT);
        for (int idx = t; idx < ni * L.EL; idx += TGT) {
          int n = idx / L.EL, c = idx - n * L.EL;
          e_out[((size_t)jet * L.N + i0 + n) * L.EL + c] = sm_e[n * L.ELs + c];
        }
      }
    }
    if (t == 0) GJ_TRACE_END(wg);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NWG * 4 * NH) tmem_dealloc(tmem_base, (uint32_t)T.tmem_cols_total);
}

// ------------------------------------------------------------------------------------------------
// backward: recompute + dgrad + wgrad on tensor cores
// ------------------------------------------------------------------------------------------------
// CTA = NWG compute warpgroups + one MMA-issuer warp.  A warpgroup owns the tiles of its jets and only ever
// touches shared memory and its TMEM accumulator; ALL tcgen05.mma are issued by one thread of the issuer warp,
// strictly round-robin over the warpgroups (fixed accumulation order => deterministic gradients), which lets the
// weight-gradient accumulators be shared by the warpgroups and stay resident in TMEM for the whole kernel.
// Per tile and warpgroup the issuer runs 2(Le-1) stages, each followed by a warpgroup epilogue:
//   F_l (l = 1..Le-1): acc = a_{l-1} W_l^T                     epilogue: a_l -> bf16 smem (last: dz_last = de*leaky')
//   B_l (l = Le-1..1): dW_l += dz_l^T a_{l-1} ; acc = dz_l W_l  epilogue: dz_{l-1} = acc * leaky'(a_{l-1}) in place
//                      (at l = 1 also the bias gradients: column sums of ALL dz_l as one M=128 MMA per 128 columns
//                       against a ones operand, the dz_l buffers being contiguous in shared memory)
// The first layer's adjoint (dP, dQ, distance gradient, d wd) is reduced on the CUDA cores from dz_0 in fp32.
struct BwdPlan {
  int nwg, Le, trace;
  // shared regions (bytes from smem base)
  int o_bar, o_tmem_slot, o_ones, o_shared_f32, o_tbl, groups_per_wg;
  int o_wT[GJ_MAX_LAYERS];
  int wg_base, wg_stride;
  // per-warpgroup (bytes from the warpgroup base)
  int w_a0, w_comb, w_f32;
  int coff[GJ_MAX_LAYERS];      // column offset of layer l's buffer inside the combined dz buffer (l >= 1)
  int ctot;
  // TMEM (columns from the allocation base)
  int nacc;                     // per-warpgroup forward/dgrad accumulator width
  int t_wg[GJ_MAX_LAYERS];      // weight-gradient accumulator of layer l
  int wg_orient[GJ_MAX_LAYERS]; // 0: lanes = out features (M from dz_l), 1: lanes = in features (M from a_{l-1})
  int wg_M[GJ_MAX_LAYERS], wg_N[GJ_MAX_LAYERS];
  int nbias, t_bias[4], bias_M[4];
  int tmem_cols;
  int smem_bytes;
};

// returns 0 if the configuration is supported by the tensor-core backward
int plan_tc_bwd(MPLayout* L, BwdPlan* T, int nwg) {
  memset(T, 0, sizeof(*T));
  T->nwg = nwg; T->Le = L->Le;
  L->R = 128;
  tc_strides(L);
  if (L->Le < 2) return 1;
  if (L->E0p != 16 && L->E0p != 32 && L->E0p != 48 && L->E0p != 64) return 1;
  int ctot = 0, nacc = 32;
  for (int l = 1; l < L->Le; ++l) {
    if (L->Ep[l] > 256 || L->Kp[l] > 256) return 1;
    T->coff[l] = ctot; ctot += L->Ep[l];
    if (L->Ep[l] > nacc) nacc = L->Ep[l];
    if (L->Kp[l] > nacc) nacc = L->Kp[l];
  }
  T->ctot = ctot; T->nacc = nacc;
  int tcol = nwg * nacc;
  for (int l = 1; l < L->Le; ++l) {
    const int Ma = gj_round_up(L->Ep[l], 64), Mb = gj_round_up(L->Kp[l], 64);
    const bool oka = Ma <= 128, okb = Mb <= 128;
    if (!oka && !okb) return 1;
    int orient;
    if (oka && okb) {
      if (L->Kp[l] != L->Ep[l]) orient = L->Kp[l] < L->Ep[l] ? 0 : 1;      // fewer TMEM columns
      else orient = (Ma == L->Ep[l] || Mb != L->Kp[l]) ? 0 : 1;             // prefer an unpadded M
    } else orient = oka ? 0 : 1;
    T->wg_orient[l] = orient;
    T->wg_M[l] = orient == 0 ? Ma : Mb;
    T->wg_N[l] = orient == 0 ? L->Kp[l] : L->Ep[l];
    T->t_wg[l] = tcol; tcol += T->wg_N[l];
  }
  int rem = ctot, nb = 0;
  while (rem > 0) {
    if (nb >= 4) return 1;
    T->bias_M[nb] = rem > 64 ? 128 : 64;
    T->t_bias[nb] = tcol; tcol += 16;
    rem -= 128; ++nb;
  }
  T->nbias = nb;
  if (tcol > 512) return 1;
  T->tmem_cols = next_pow2_cols(tcol);
  // shared floats
  Carver c;
  for (int l = 1; l < L->Le; ++l) L->o_bE[l] = c.take(L->Ep[l]);
  L->o_wd = c.take(L->E0p);
  L->o_dpar = c.take(nwg * L->E0p);     // per-warpgroup d(wd) partials at kernel end
  // per-warpgroup floats
  Carver w;
  L->o_h = w.take(GJ_IB * L->Hs);
  L->o_hj = w.take(32 * L->Hs);
  L->o_P = w.take(GJ_IB * L->E0s);
  L->o_Q = w.take(32 * L->E0s);
  L->o_e = w.take(GJ_IB * L->ELs);
  L->o_dP = w.take(GJ_IB * L->E0s);
  L->o_dQ = L->o_Q;                    // dQ_j is flushed after the block's last tile, when Q_j is dead: same storage
  L->o_dh = w.take(GJ_IB * L->Hs);
  L->o_G = w.take(GJ_IB * L->Gs);
  int off = 0;
  T->o_bar = off; off += 64;
  T->o_tmem_slot = off; off += 64;
  T->o_ones = off; off += 16 * 128 * 2;
  T->groups_per_wg = (L->Le - 1) + 2 * (L->Le - 1) + nb;
  T->o_tbl = off; off += nwg * T->groups_per_wg * 40 + (2 * GJ_MAX_LAYERS + 2) * 4;
  off = gj_round_up(off, 16);
  for (int l = 1; l < L->Le; ++l) { T->o_wT[l] = off; off += L->Ep[l] * L->Kp[l] * 2; }
  T->o_shared_f32 = off; off += c.off * 4;
  off = gj_round_up(off, 128);
  T->wg_base = off;
  int wo = 0;
  T->w_a0 = wo; wo += L->E0p * 256;
  T->w_comb = wo; wo += ctot * 256;
  T->w_f32 = wo; wo += w.off * 4;
  // MN-major operands with a padded M read up to 127 columns past their buffer: keep those reads inside the
  // warpgroup's own region (what they fetch only lands in accumulator rows nobody reads)
  const int overshoot = 128 * 256;
  if (w.off * 4 < overshoot) wo += overshoot - w.off * 4;
  wo = gj_round_up(wo, 128);
  T->wg_stride = wo;
  T->smem_bytes = T->wg_base + nwg * wo;
  return T->smem_bytes > 227 * 1024 ? 1 : 0;
}

__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}

template <int NWG, int NH, int E0P>
__global__ void __launch_bounds__(NWG * 128 * NH + 32, 1)
edge_bwd_tc_kernel(const MPLayout L, const BwdPlan T, const float* __restrict__ h, const float* __restrict__ pq,
                   const float* __restrict__ params, const float* __restrict__ de, float* __restrict__ dpq,
                   float* __restrict__ dh, float* __restrict__ part) {
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int TGT = 128 * NH;                    // threads per tile group (NH warps per TMEM lane quadrant)
  constexpr int NT = NWG * TGT + 32;
  constexpr int NCH0 = E0P / 16;                   // 16-column chunks of the first layer
  constexpr int OWN = ((NCH0 + NH - 1) / NH) * 16; // first-layer channels a thread owns (chunks part, part + NH, ...)
  const int tid = threadIdx.x;
  const int warp = (int)uni((uint32_t)(tid >> 5)), lane = tid & 31;     // provably warp-uniform
  const bool is_issuer = warp == NWG * 4 * NH;
  float* smf = reinterpret_cast<float*>(smem + T.o_shared_f32);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + T.o_bar);   // ready[wg] = bars[wg], done[wg] = bars[NWG + wg]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + T.o_tmem_slot);
  const int Le = L.Le;

  stage_small(L, params, smf, tid, NT);
  stage_edge_weights_bf16(L, T.o_wT, params, smem, tid, NT);
  for (int idx = tid; idx < 16 * 128; idx += NT) reinterpret_cast<__nv_bfloat16*>(smem + T.o_ones)[idx] = __float2bfloat16_rn(1.f);
  if (tid == 0) {
    for (int w = 0; w < NWG; ++w) { mbar_init(bars + w, 4 * NH); mbar_init(bars + NWG + w, 1); mbar_init(bars + 2 * NWG + w, 1); }
    fence_barrier_init();
  }
  if (is_issuer) tmem_alloc(tmem_slot, (uint32_t)T.tmem_cols);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int jets_total = L.B;
  int tr_i = 0;      // trace cursor (register; written back once at the end)

  if (is_issuer) {
    // =================================== MMA issuer ===================================
    // The whole warp runs this code convergently; only the tcgen05 instructions themselves are elected to one lane.
    {
      const int S = 2 * (Le - 1);
      const int tpj = tiles_of_jet(L);
      int total[NWG], done_st[NWG];
      uint32_t par[NWG];
      bool any = false;
#pragma unroll
      for (int w = 0; w < NWG; ++w) {
        const int first = blockIdx.x * NWG + w;
        const int njets = first < jets_total ? (jets_total - first + gridDim.x * NWG - 1) / (gridDim.x * NWG) : 0;
        total[w] = njets * tpj * S; done_st[w] = 0; par[w] = 0;
        any |= total[w] > 0;
      }
      // group table in shared memory: per warpgroup, stage s owns groups [gbeg[s], gbeg[s + 1])
      MmaGroup* tbl = reinterpret_cast<MmaGroup*>(smem + T.o_tbl);
      int* gbeg = reinterpret_cast<int*>(smem + T.o_tbl + NWG * T.groups_per_wg * 40);
      if (lane == 0) {
        for (int w = 0; w < NWG; ++w) {
          const uint32_t wgb = smem_u32(smem + T.wg_base + w * T.wg_stride);
          const uint32_t a0 = wgb + T.w_a0, comb = wgb + T.w_comb;
          const uint32_t acc = tmem_base + (uint32_t)(w * T.nacc);
          int ng = 0;
          MmaGroup* tw = tbl + w * T.groups_per_wg;
          for (int s2 = 0; s2 < S; ++s2) {
            gbeg[s2] = ng;
            if (s2 < Le - 1) {
              const int l = s2 + 1;
              const uint32_t ain = l == 1 ? a0 : comb + (T.coff[l - 1] >> 3) * 2048;
              tw[ng] = grp_fwd(acc, ain, smem_u32(smem + T.o_wT[l]), L.Ep[l], L.Kp[l]);
              tw[ng++].commit = 1;
            } else {
              const int l = Le - 1 - (s2 - (Le - 1));
              const uint32_t dz = comb + (T.coff[l] >> 3) * 2048;
              const uint32_t ain = l == 1 ? a0 : comb + (T.coff[l - 1] >> 3) * 2048;
              const MmaGroup wgrad = T.wg_orient[l] == 0 ? grp_wgrad(tmem_base + T.t_wg[l], dz, ain, T.wg_M[l], T.wg_N[l], l)
                                                         : grp_wgrad(tmem_base + T.t_wg[l], ain, dz, T.wg_M[l], T.wg_N[l], l);
              MmaGroup dgrad = grp_dgrad(acc, dz, smem_u32(smem + T.o_wT[l]), L.Kp[l], L.Ep[l]);
              if (l > 1) {
                // the epilogue overwrites a_{l-1} in place, which the weight gradient reads: both must complete first
                tw[ng++] = wgrad;
                dgrad.commit = 1;
                tw[ng++] = dgrad;
              } else {
                // nothing the last epilogue writes is read by an MMA: release the warpgroup after dgrad and let the
                // weight-gradient and bias column-sum batches run behind its epilogue (done2 gates the next tile)
                dgrad.commit = 1;
                tw[ng++] = dgrad;
                tw[ng++] = wgrad;
                for (int b = 0; b < T.nbias; ++b)
                  tw[ng++] = grp_colsum(tmem_base + T.t_bias[b], comb + b * 16 * 2048, smem_u32(smem + T.o_ones), T.bias_M[b], 16 + b);
                tw[ng - 1].commit = 2;
              }
            }
          }
          gbeg[S] = ng;
        }
      }
      __syncwarp();
      uint32_t inited = 0;    // bit id: that shared gradient accumulator has been written
      while (any) {
#pragma unroll
        for (int w = 0; w < NWG; ++w) {
          if (done_st[w] >= total[w]) continue;
          mbar_wait(bars + w, par[w]);
          par[w] ^= 1u;
          __syncwarp();
          tc_fence_after();
          const int s2 = done_st[w] % S;
          if (lane == 0) GJ_TRACE_PT(2, w * 100 + s2);
          const MmaGroup* tw = tbl + w * T.groups_per_wg;
          const int g0 = (int)uni((uint32_t)gbeg[s2]), g1 = (int)uni((uint32_t)gbeg[s2 + 1]);
          for (int g = g0; g < g1; ++g) {
            const int commit = run_group(tw + g, inited);
            if (commit == 1) mma_commit_elect(bars + NWG + w);
            else if (commit == 2) mma_commit_elect(bars + 2 * NWG + w);
          }
          if (lane == 0) GJ_TRACE_PT(2, 1000 + w * 100 + s2);
          ++done_st[w];
        }
        any = false;
#pragma unroll
        for (int w = 0; w < NWG; ++w) any |= done_st[w] < total[w];
      }
      if (lane == 0) GJ_TRACE_END(2);
    }
    __syncwarp();
  } else {
    // =================================== compute warpgroups ===================================
    const int wg = warp / (4 * NH), w8 = warp % (4 * NH), wq = w8 & 3, part = w8 >> 2;     // warp-uniform
    const int t = tid - wg * TGT, row = wq * 32 + lane;
    uint8_t* wgb = smem + T.wg_base + wg * T.wg_stride;
    float* wgf = reinterpret_cast<float*>(wgb + T.w_f32);
    uint8_t* A0 = wgb + T.w_a0;
    uint8_t* COMB = wgb + T.w_comb;
    uint64_t* ready = bars + wg;
    uint64_t* done = bars + NWG + wg;
    uint64_t* done2 = bars + 2 * NWG + wg;     // the previous tile's background weight-gradient batch has completed
    const uint32_t tmem_row = tmem_base + (uint32_t)(wg * T.nacc) + ((uint32_t)(wq * 32) << 16);
    uint32_t phase = 0, phase2 = 0;
    bool pending2 = false;
    const int bar_id = 1 + wg;
    float* sm_h = wgf + L.o_h;
    float* sm_hj = wgf + L.o_hj;
    float* sm_Q = wgf + L.o_Q;
    float* sm_P = wgf + L.o_P;
    float* sm_de = wgf + L.o_e;
    float* sm_dP = wgf + L.o_dP;
    float* sm_dQ = wgf + L.o_dQ;
    float* sm_dh = wgf + L.o_dh;
    float* sm_G = wgf + L.o_G;
    const float* wd = smf + L.o_wd;
    const int H = L.H, W2 = 2 * L.E0p;
    const bool a_le_1 = L.alpha <= 1.f;
    float dwd[OWN];
#pragma unroll
    for (int c = 0; c < OWN; ++c) dwd[c] = 0.f;

    for (int jet = blockIdx.x * NWG + wg; jet < L.B; jet += gridDim.x * NWG) {
      const float* hjet = h + (size_t)jet * L.N * L.ld;
      const float* pqjet = pq + (size_t)jet * L.N * W2;
      float* dpqjet = dpq + (size_t)jet * L.N * W2;
      float* dhjet = dh + (size_t)jet * L.N * L.ld;
      for (int i0 = 0; i0 < L.N; i0 += GJ_IB) {
        const int ni = min(GJ_IB, L.N - i0);
        named_bar_sync(bar_id, TGT);
        wg_load_block(L, hjet, pqjet, 0, i0, sm_h, sm_P, t, TGT);
#pragma unroll 4
        for (int idx = t; idx < GJ_IB * L.ELs; idx += TGT) {
          int n = idx / L.ELs, c = idx - n * L.ELs;
          sm_de[idx] = (n < ni && c < L.EL) ? __ldg(de + ((size_t)jet * L.N + i0 + n) * L.EL + c) : 0.f;
        }
        for (int idx = t; idx < GJ_IB * L.E0s; idx += TGT) sm_dP[idx] = 0.f;
        for (int idx = t; idx < GJ_IB * L.Hs; idx += TGT) sm_dh[idx] = 0.f;
        for (int j0 = 0; j0 < L.N; j0 += 32) {
          const int nj = min(32, L.N - j0);
          named_bar_sync(bar_id, TGT);
          wg_load_block(L, hjet, pqjet, 1, j0, sm_hj, sm_Q, t, TGT);
          for (int idx = t; idx < GJ_IB * L.Gs; idx += TGT) sm_G[idx] = 0.f;
          float dq[OWN];
#pragma unroll
          for (int c = 0; c < OWN; ++c) dq[c] = 0.f;
          named_bar_sync(bar_id, TGT);
          const int nit = (ni + 3) / 4;
          for (int it = 0; it < nit; ++it) {
            const int il = it * 4 + wq;
            const bool valid = il < ni && lane < nj;
            if (pending2) { group_wait(done2, phase2, w8 == 0, 8 + wg, TGT); phase2 ^= 1u; }     // A0 / dz buffers are free again
            pending2 = true;
            const float dij = tc_layer0(L, sm_h, sm_hj, sm_P, sm_Q, wd, A0, il, lane, row, part, NH);
            fence_proxy_async();
            tc_fence_before();
            warp_arrive(ready, lane);
            if (t == 0) GJ_TRACE_PT(wg, 10);
            // ---- forward stages ----
            for (int l = 1; l < Le; ++l) {
              group_wait(done, phase, w8 == 0, 8 + wg, TGT); phase ^= 1u;
              tc_fence_after();
              if (t == 0) GJ_TRACE_PT(wg, 20 + l);
              const bool last = (l == Le - 1);
              const float* bias = smf + L.o_bE[l];
              uint8_t* out = COMB + (T.coff[l] >> 3) * 2048 + row * 16;
              const int nch = L.Ep[l] >> 4;
              auto process = [&](float (&v)[16], int c0) {
                float bq[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(bq + 4 * q) = *reinterpret_cast<const float4*>(bias + c0 + 4 * q);
                if (!last) {
                  bias_leaky16(v, bq, L.alpha, a_le_1);
                } else {
                  // dz_last = de_i * leaky'(z_last), zero on padded rows (this masks everything downstream)
                  const float* dei = sm_de + il * L.ELs + c0;
#pragma unroll
                  for (int q = 0; q < 16; ++q) {
                    const float z = v[q] + bq[q];
                    v[q] = valid ? dei[q] * (z > 0.f ? 1.f : L.alpha) : 0.f;
                  }
                }
                uint4 p0 = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                uint4 p1 = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
                *reinterpret_cast<uint4*>(out + (c0 >> 3) * 2048) = p0;
                *reinterpret_cast<uint4*>(out + ((c0 >> 3) + 1) * 2048) = p1;
              };
              for_chunks(tmem_row, nch, part, NH, process);
              fence_proxy_async();
              tc_fence_before();
              warp_arrive(ready, lane);
              if (t == 0) GJ_TRACE_PT(wg, 30 + l);
            }
            // ---- backward stages ----
            for (int l = Le - 1; l >= 1; --l) {
              group_wait(done, phase, w8 == 0, 8 + wg, TGT); phase ^= 1u;
              tc_fence_after();
              if (t == 0) GJ_TRACE_PT(wg, 40 + l);
              if (l > 1) {
                // dz_{l-1} = da_{l-1} * leaky'(a_{l-1}), in place over a_{l-1}
                uint8_t* buf = COMB + (T.coff[l - 1] >> 3) * 2048 + row * 16;
                const int nch = L.Kp[l] >> 4;
                auto process = [&](float (&v)[16], int c0) {
                  float a[16];
                  unpack_bf16x8(*reinterpret_cast<const uint4*>(buf + (c0 >> 3) * 2048), a);
                  unpack_bf16x8(*reinterpret_cast<const uint4*>(buf + ((c0 >> 3) + 1) * 2048), a + 8);
#pragma unroll
                  for (int q = 0; q < 16; ++q) v[q] = a[q] > 0.f ? v[q] : L.alpha * v[q];
                  uint4 p0 = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                  uint4 p1 = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
                  *reinterpret_cast<uint4*>(buf + (c0 >> 3) * 2048) = p0;
                  *reinterpret_cast<uint4*>(buf + ((c0 >> 3) + 1) * 2048) = p1;
                };
                for_chunks(tmem_row, nch, part, NH, process);
                fence_proxy_async();
                tc_fence_before();
                warp_arrive(ready, lane);
                if (t == 0) GJ_TRACE_PT(wg, 50 + l);
              } else {
                // dz_0 = da_0 * leaky'(a_0), consumed in fp32: G_ij, dQ_j, dP_i, d(wd)
                float g = 0.f;
#pragma unroll
                for (int kk = 0; kk < OWN / 16; ++kk) {
                  const int c0 = 16 * (part + NH * kk);            // this thread's kk-th chunk
                  if (c0 < E0P) {
                    float v[16], a[16];
                    tmem_ld16(tmem_row + (uint32_t)c0, v);
                    unpack_bf16x8(*reinterpret_cast<const uint4*>(A0 + (c0 >> 3) * 2048 + row * 16), a);
                    unpack_bf16x8(*reinterpret_cast<const uint4*>(A0 + ((c0 >> 3) + 1) * 2048 + row * 16), a + 8);
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                      v[q] *= (a[q] > 0.f ? 1.f : L.alpha);
                      g = fmaf(v[q], wd[c0 + q], g);
                      dq[16 * kk + q] += v[q];
                      dwd[16 * kk + q] = fmaf(v[q], dij, dwd[16 * kk + q]);
                    }
                    const float s = warp_transpose_sum16(v, lane);
                    if ((lane & 1) == 0) sm_dP[il * L.E0s + c0 + (lane >> 1)] += s;
                  }
                }
                if (NH == 1) sm_G[il * L.Gs + lane] = g;
                else atomicAdd(sm_G + il * L.Gs + lane, g);   // two addends onto a zeroed cell: order-independent, deterministic
                tc_fence_before();
                if (t == 0) GJ_TRACE_PT(wg, 60);
              }
            }
          }
          // ---- (i block, j block) epilogue ----
          named_bar_sync(bar_id, TGT);            // every warp is done reading Q_j: its storage now receives dQ_j
          for (int w = 0; w < 4; ++w) {           // the four warps hold different i's of the same j: fixed order 0..3
            if (wq == w) {
#pragma unroll
              for (int kk = 0; kk < OWN / 16; ++kk) {
                const int c0 = 16 * (part + NH * kk);
                if (c0 < E0P) {
#pragma unroll
                  for (int c = 0; c < 16; c += 4) {
                    float4* p = reinterpret_cast<float4*>(sm_dQ + lane * L.E0s + c0 + c);
                    float4 v = w == 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : *p;
                    v.x += dq[16 * kk + c]; v.y += dq[16 * kk + c + 1]; v.z += dq[16 * kk + c + 2]; v.w += dq[16 * kk + c + 3];
                    *p = v;
                  }
                }
              }
            }
            named_bar_sync(bar_id, TGT);
          }
          for (int idx = t; idx < nj * L.E0p; idx += TGT) {
            int n = idx / L.E0p, c = idx - n * L.E0p;
            float* p = dpqjet + (size_t)(j0 + n) * W2 + L.E0p + c;
            float v = sm_dQ[n * L.E0s + c];
            *p = (i0 == 0) ? v : (*p + v);
          }
          for (int idx = t; idx < nj * H; idx += TGT) {
            int n = idx / H, k = idx - n * H;
            const float sgn = (L.mink && k > 0) ? -2.f : 2.f;
            const float hjk = sm_hj[n * L.Hs + k];
            float acc = 0.f;
            for (int i = 0; i < ni; ++i) acc = fmaf(sm_G[i * L.Gs + n], hjk - sm_h[i * L.Hs + k] + GJ_EPS, acc);
            if (k < L.cols) dhjet[(size_t)(j0 + n) * L.ld + k] += sgn * acc;
          }
          for (int idx = t; idx < ni * H; idx += TGT) {
            int n = idx / H, k = idx - n * H;
            const float sgn = (L.mink && k > 0) ? -2.f : 2.f;
            const float hik = sm_h[n * L.Hs + k];
            float acc = 0.f;
            for (int j = 0; j < nj; ++j) acc = fmaf(sm_G[n * L.Gs + j], sm_hj[j * L.Hs + k] - hik + GJ_EPS, acc);
            sm_dh[n * L.Hs + k] -= sgn * acc;
          }
        }
        named_bar_sync(bar_id, TGT);
        for (int idx = t; idx < ni * L.E0p; idx += TGT) {
          int n = idx / L.E0p, c = idx - n * L.E0p;
          dpqjet[(size_t)(i0 + n) * W2 + c] = sm_dP[n * L.E0s + c];
        }
        for (int idx = t; idx < ni * L.cols; idx += TGT) {
          int n = idx / L.cols, k = idx - n * L.cols;
          dhjet[(size_t)(i0 + n) * L.ld + k] += sm_dh[n * L.Hs + k];
        }
      }
    }
    if (t == 0) GJ_TRACE_END(wg);
    if (pending2) { mbar_wait(done2, phase2); phase2 ^= 1u; }       // all of this warpgroup's MMAs have completed
    // d(wd)[c] = sum over this warpgroup's rows: lanes by shuffles, warps through shared memory (fixed order)
    named_bar_sync(bar_id, TGT);
    float* red = sm_dQ;    // [4][E0P]
#pragma unroll
    for (int kk = 0; kk < OWN / 16; ++kk) {
      const int c0 = 16 * (part + NH * kk);
#pragma unroll
      for (int q = 0; q < 16; ++q) {
        const float s = gj_warp_sum(dwd[16 * kk + q]);
        if (lane == 0 && c0 < E0P) red[wq * E0P + c0 + q] = s;
      }
    }
    named_bar_sync(bar_id, TGT);
    for (int c = t; c < E0P; c += TGT) smf[L.o_dpar + wg * L.E0p + c] = (red[c] + red[E0P + c]) + (red[2 * E0P + c] + red[3 * E0P + c]);
  }

  // =================================== gradient read-out ===================================
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  float* out = part + (size_t)blockIdx.x * L.pV[0];
  if (!is_issuer) {
    const int wq = warp & 3, wgi = warp >> 2;      // wgi: 0 .. NWG*NH-1, every one of them covers the 128 lanes
    const bool wrote = (blockIdx.x * NWG) < jets_total;     // a CTA without jets never initialised its accumulators
    // wd column
    for (int c = tid; c < L.E[0]; c += NWG * TGT) {
      float s = 0.f;
      for (int w = 0; w < NWG; ++w) s += smf[L.o_dpar + w * L.E0p + c];
      out[L.pW[0] + c * L.K[0] + 2 * L.H] = wrote ? s : 0.f;
    }
    // weight gradients: accumulator row m <-> lane (M = 128: lane m; M = 64: lane (m / 16) * 32 + m % 16)
    for (int l = 1; l < Le; ++l) {
      const int M = T.wg_M[l], N = T.wg_N[l];
      const int m = M == 128 ? wq * 32 + lane : (lane < 16 ? wq * 16 + lane : -1);
      const int nchunks = N / 16;
      for (int ch = wgi; ch < nchunks; ch += NWG * NH) {       // warp-uniform: every lane of the warp issues the load
        float v[16];
        tmem_ld16(tmem_base + (uint32_t)(T.t_wg[l] + ch * 16) + ((uint32_t)(wq * 32) << 16), v);
        if (m < 0) continue;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const int n = ch * 16 + q;
          const int c = T.wg_orient[l] == 0 ? m : n;       // out feature
          const int k = T.wg_orient[l] == 0 ? n : m;       // in feature
          if (c < L.E[l] && k < L.K[l]) out[L.pW[l] + c * L.K[l] + k] = wrote ? v[q] : 0.f;
        }
      }
    }
    // bias gradients: column sums of the combined dz buffer, chunk b covers columns [128 b, 128 b + M)
    if (wgi == 0) {
      for (int b = 0; b < T.nbias; ++b) {
        float v[16];
        tmem_ld16(tmem_base + (uint32_t)T.t_bias[b] + ((uint32_t)(wq * 32) << 16), v);
        const int M = T.bias_M[b];
        const int m = M == 128 ? wq * 32 + lane : (lane < 16 ? wq * 16 + lane : -1);
        if (m < 0) continue;
        const int col = b * 128 + m;
        for (int l = 1; l < Le; ++l) {
          const int c = col - T.coff[l];
          if (c >= 0 && c < L.E[l]) out[L.pb[l] + c] = wrote ? v[0] : 0.f;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (is_issuer) tmem_dealloc(tmem_base, (uint32_t)T.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// tcgen05 self-test: one CTA, D = A * B^T with selectable operand major-ness; dumps raw TMEM.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128, 1)
umma_selftest_kernel(int M, int N, int K, int a_mn, int b_mn, const float* __restrict__ A, const float* __restrict__ B,
                     float* __restrict__ out, int tmem_cols, int b_off) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + 16);
  uint8_t* sa = smem + 1024;
  uint8_t* sb = smem + b_off;
  const int tid = threadIdx.x;
  for (int idx = tid; idx < M * K; idx += 128) {
    int m = idx / K, k = idx - m * K;
    uint32_t off = a_mn ? il_off(k, m, K) : il_off(m, k, M);
    *reinterpret_cast<__nv_bfloat16*>(sa + off) = __float2bfloat16_rn(A[idx]);
  }
  for (int idx = tid; idx < N * K; idx += 128) {
    int n = idx / K, k = idx - n * K;
    uint32_t off = b_mn ? il_off(k, n, K) : il_off(n, k, N);
    *reinterpret_cast<__nv_bfloat16*>(sb + off) = __float2bfloat16_rn(B[idx]);
  }
  if (tid == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  if (tid < 32) tmem_alloc(slot, (uint32_t)tmem_cols);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *slot;
  if (tid == 0) {
    const uint32_t idesc = make_idesc_bf16(M, N, a_mn, b_mn);
    for (int ks = 0; ks < K / 16; ++ks) {
      uint64_t ad = a_mn ? make_smem_desc(smem_u32(sa) + ks * 256, 128, K * 16)
                         : make_smem_desc(smem_u32(sa) + ks * (2 * M * 16), M * 16, 128);
      uint64_t bd = b_mn ? make_smem_desc(smem_u32(sb) + ks * 256, 128, K * 16)
                         : make_smem_desc(smem_u32(sb) + ks * (2 * N * 16), N * 16, 128);
      mma_bf16_ss(tbase, ad, bd, idesc, ks > 0 ? 1u : 0u);
    }
    mma_commit(bar);
  }
  __syncwarp();
  mbar_wait(bar, 0);
  tc_fence_after();
  const int wq = tid >> 5, lane = tid & 31;
  for (int c0 = 0; c0 < N; c0 += 16) {
    float v[16];
    tmem_ld16(tbase + ((uint32_t)(wq * 32) << 16) + (uint32_t)c0, v);
    for (int q = 0; q < 16 && c0 + q < N; ++q) out[(size_t)(wq * 32 + lane) * N + c0 + q] = v[q];
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 32) tmem_dealloc(tbase, (uint32_t)tmem_cols);
}

}  // namespace

int gj_num_sms();
void gj_set_error(const char* fmt, ...);
int gj_edge_grid(int);
int gj_edge_bwd_simt(MPLayout, const float*, const float*, const float*, const float*, float*, float*, float*, float*,
                     cudaStream_t);

int gj_edge_fwd_simt(MPLayout, const float*, const float*, const float*, float*, cudaStream_t);

int gj_edge_fwd_tc(MPLayout L, const float* h, const float* pq, const float* params, float* e_out, cudaStream_t stream) {
  if (L.alpha > 1.f) return gj_edge_fwd_simt(L, h, pq, params, e_out, stream);   // max(z, alpha z) form needs alpha <= 1
  for (int l = 1; l < L.Le; ++l)
    if (L.Ep[l] > 256 || L.Kp[l] > 256) { gj_set_error("gj_mp_step_fwd(bf16): edge widths above 256 unsupported"); return GJ_ERR_INVALID; }
  TCPlan T;
  int NWG = 2;
  plan_tc_fwd(&L, &T, NWG);
  for (int l = 0; l < L.Le; ++l)
    if (L.Ep[l] > 16 * GJ_MAX_CHUNKS) { gj_set_error("gj_mp_step_fwd(bf16): edge widths above 256 unsupported"); return GJ_ERR_INVALID; }
  if (T.smem_bytes > 227 * 1024 || T.tmem_cols_total > 512) {      // wide layers: one warpgroup per CTA
    NWG = 1;
    plan_tc_fwd(&L, &T, NWG);
  }
  if (T.smem_bytes > 227 * 1024 || T.tmem_cols_total > 512) {
    gj_set_error("gj_mp_step_fwd(bf16): needs %d B shared memory / %d TMEM columns (limits 232448 / 512)", T.smem_bytes, T.tmem_cols_total);
    return GJ_ERR_SMEM;
  }
  static const int trace_fwd = getenv("GJ_TRACE") ? atoi(getenv("GJ_TRACE")) : 0;
  T.trace = trace_fwd == 2;
  if (T.trace) { int z[4] = {0, 0, 0, 0}; cudaMemcpyToSymbolAsync(g_trace_n, z, sizeof(z), 0, cudaMemcpyHostToDevice, stream); }
  constexpr int NH = 2;
  auto kern = NWG == 1 ? edge_fwd_tc_kernel<1, NH> : edge_fwd_tc_kernel<2, NH>;
  cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T.smem_bytes);
  if (ce != cudaSuccess) { gj_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  int sms = gj_num_sms();
  int grid = (L.B + NWG - 1) / NWG; if (grid > sms) grid = sms;
  kern<<<grid, NWG * 128 * NH + NWG * 32, T.smem_bytes, stream>>>(L, T, h, pq, params, e_out);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("edge_fwd_tc launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

bool gj_edge_simt_fits(MPLayout, const float*);
// the first-generation tensor-core forward has a plan for these widths and the backward either has one or can hand over to the
// fp32 kernel (otherwise the step runs the materialised path of dense.cu)
bool gj_edge_tc_fits(MPLayout L) {
  if (L.alpha > 1.f) return gj_edge_simt_fits(L, nullptr);
  for (int l = 0; l < L.Le; ++l)
    if (L.Ep[l] > 256 || (l > 0 && L.Kp[l] > 256) || L.Ep[l] > 16 * GJ_MAX_CHUNKS) return false;
  TCPlan T; MPLayout Lf = L;
  plan_tc_fwd(&Lf, &T, 2);
  if (T.smem_bytes > 227 * 1024 || T.tmem_cols_total > 512) { Lf = L; plan_tc_fwd(&Lf, &T, 1); }
  if (T.smem_bytes > 227 * 1024 || T.tmem_cols_total > 512) return false;
  BwdPlan Bp; MPLayout Lb = L;
  if (plan_tc_bwd(&Lb, &Bp, 2) == 0) return true;
  return gj_edge_simt_fits(L, nullptr);
}

int gj_reduce_edge_partials(const MPLayout& L, const float* part, int nparts, float* dparams, cudaStream_t stream);

static int tc_bwd_grid(int batch, int nwg) {
  int sms = gj_num_sms();
  int grid = (batch + nwg - 1) / nwg;
  return grid > sms ? sms : (grid < 1 ? 1 : grid);
}

size_t gj_edge_bwd_tc_ws_floats(const MPLayout& L) {
  // large enough for either backward (tensor-core or the SIMT fallback for unsupported widths)
  size_t a = (size_t)gj_edge_grid(L.B) * L.pV[0], b = (size_t)tc_bwd_grid(L.B, 2) * L.pV[0];
  return a > b ? a : b;
}

template <int E0P>
static int launch_tc_bwd(const MPLayout& L, const BwdPlan& T, const float* h, const float* pq, const float* params,
                         const float* de, float* dpq, float* dh, float* part, int grid, cudaStream_t stream) {
  constexpr int NWG = 2;
  // NH = 1: with NH = 2 (256 threads per tile) the backward kernel is measured slower, since 17 warps cap it at 96 registers
  // and the first-layer adjoint spills
  constexpr int NH = 1;
  auto kern = edge_bwd_tc_kernel<NWG, NH, E0P>;
  cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T.smem_bytes);
  if (ce != cudaSuccess) { gj_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  kern<<<grid, NWG * 128 * NH + 32, T.smem_bytes, stream>>>(L, T, h, pq, params, de, dpq, dh, part);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("edge_bwd_tc launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_edge_bwd_tc(MPLayout L, const float* h, const float* pq, const float* params, const float* de, float* dpq, float* dh,
                   float* dparams, float* part, cudaStream_t stream) {
  BwdPlan T;
  MPLayout Lt = L;
  if (L.alpha > 1.f || plan_tc_bwd(&Lt, &T, 2)) {
    // widths the tensor-core backward does not cover (first layer wider than 64, layers wider than 128 on both sides,
    // more than 512 combined dz columns): the fp32 kernel computes the gradient instead
    return gj_edge_bwd_simt(L, h, pq, params, de, dpq, dh, dparams, part, stream);
  }
  const int grid = tc_bwd_grid(Lt.B, 2);
  static const int trace_env = getenv("GJ_TRACE") ? atoi(getenv("GJ_TRACE")) : 0;
  T.trace = trace_env == 1;
  if (T.trace) { int z[4] = {0, 0, 0, 0}; cudaMemcpyToSymbolAsync(g_trace_n, z, sizeof(z), 0, cudaMemcpyHostToDevice, stream); }
  int rc;
  switch (Lt.E0p) {
    case 16: rc = launch_tc_bwd<16>(Lt, T, h, pq, params, de, dpq, dh, part, grid, stream); break;
    case 32: rc = launch_tc_bwd<32>(Lt, T, h, pq, params, de, dpq, dh, part, grid, stream); break;
    case 48: rc = launch_tc_bwd<48>(Lt, T, h, pq, params, de, dpq, dh, part, grid, stream); break;
    default: rc = launch_tc_bwd<64>(Lt, T, h, pq, params, de, dpq, dh, part, grid, stream); break;
  }
  if (rc) return rc;
  return gj_reduce_edge_partials(Lt, part, grid, dparams, stream);
}

// info[0..3]: forward smem bytes, forward TMEM columns, backward smem bytes (0 = fp32 fallback), backward TMEM columns
void gj_tc_plan_info(MPLayout L, int* info) {
  TCPlan F; MPLayout Lf = L; plan_tc_fwd(&Lf, &F, 2);
  info[0] = F.smem_bytes; info[1] = F.tmem_cols_total;
  BwdPlan T; MPLayout Lb = L;
  if (L.Le < 2 || plan_tc_bwd(&Lb, &T, 2)) { info[2] = 0; info[3] = 0; }
  else { info[2] = T.smem_bytes; info[3] = T.tmem_cols; }
}

// debugging aid (not part of the ABI header): copies the handshake timeline of the last traced launch
extern "C" int gj_debug_read_trace(long long* out, int* counts) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out, g_trace, sizeof(long long) * 8192) != cudaSuccess) return 1;
  if (cudaMemcpyFromSymbol(counts, g_trace_n, sizeof(int) * 4) != cudaSuccess) return 1;
  return 0;
}

int gj_umma_selftest_launch(int M, int N, int K, int a_mn, int b_mn, const float* a, const float* b, float* out,
                            cudaStream_t stream) {
  if ((M != 64 && M != 128) || N < 8 || N > 256 || (N % 8) || K < 16 || K > 256 || (K % 16)) {
    gj_set_error("gj_umma_selftest: unsupported shape m=%d n=%d k=%d", M, N, K);
    return GJ_ERR_INVALID;
  }
  int a_bytes = gj_round_up(M * K * 2, 1024), b_bytes = gj_round_up(N * K * 2, 1024);
  int b_off = 1024 + a_bytes;
  int smem = b_off + b_bytes;
  int cols = 32; while (cols < N) cols <<= 1;
  cudaError_t ce = cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (ce != cudaSuccess) { gj_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  umma_selftest_kernel<<<1, 128, smem, stream>>>(M, N, K, a_mn, b_mn, a, b, out, cols, b_off);
  ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("umma_selftest launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
