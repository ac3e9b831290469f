// Exact energy mover's distance between the particle sets of two jets, one CTA per jet (the EMD of energyflow.emd.emd,
// Komiske, Metodiev, Thaler, PRL 123, 041801, which reference utils/jet_analysis/anomaly_detection.py computes jet by jet on
// the host and utils/losses/emd_loss.py wraps through jetnet).
//
// Problem.  Rows i < Np are the particles of p with weight a_i = max(pt_i, 0), columns j < Nq those of q with b_j, and
// c_ij = (theta_ij / R)^beta, theta_ij = sqrt(deta^2 + dphi^2).  The imbalance |W_p - W_q| is modelled as energyflow does: a
// dummy row (index Np) carries max(W_q - W_p, 0) and a dummy column (index Nq) max(W_p - W_q, 0), at cost 1 to every real
// particle (a particle at distance R) and 0 between each other (that arc never carries flow: one of the two is empty).  The
// result is a balanced transportation problem on (Np + 1) x (Nq + 1) whose optimum is the EMD.  norm: a_i /= W_p, b_j /= W_q,
// and the dummies carry weight only if exactly one jet is empty.
//
// Solver.  Successive shortest paths with Johnson potentials: u (rows) and v (columns) keep every reduced cost
// c_ij - u_i - v_j >= 0 and reach 0 wherever f_ij > 0.  Each augmentation runs a dense Dijkstra over the residual graph from
// all rows with residual supply (distance 0) to the nearest column with residual demand; forward arcs i -> j always exist,
// reverse arcs j -> i where f_ij > 0 (reduced cost 0).  Thread j owns column j: relax, block arg-min and the potential update
// run across the threads, one column settled per step; the rows reached over reverse arcs of the settled column relax all
// columns.  The path then moves min(residual supply, residual demand, smallest reverse flow on the path), which zeroes that
// quantity exactly, and the potentials move by min(distance, D).  Costs are fp32 and recomputed from the staged particles
// (the fp64 flow matrix takes the shared memory: 182 KB at 150 x 150), potentials, flows and the EMD are fp64.
// Bounded: at most N1 N2 + 4 (N1 + N2) + 64 augmentations (N1 = Np + 1, N2 = Nq + 1) of at most N2 steps each; a jet that
// hits the cap gets status 1, one for which no augmenting path is found status 3 (not seen on finite costs).  A jet with a NaN or
// infinite staged (pt, eta, phi) never reaches the solver: status 2, EMD NaN, gradient rows 0.
#include <math.h>

#include "gj_common.cuh"

namespace {

constexpr int kEmdMaxParticles = 150;

__device__ __forceinline__ float emd_dphi(float d, int periodic) {
  if (!periodic) return d;
  const float two_pi = 6.283185307179586f;
  return d - two_pi * floorf((d + 3.14159265358979f) * (1.f / two_pi));      // into [-pi, pi)
}

// (theta / R)^beta of two real particles (eta, phi)
__device__ __forceinline__ float emd_pair_cost(float2 a, float2 b, float r, float beta, int periodic) {
  const float de = a.x - b.x, dp = emd_dphi(a.y - b.y, periodic);
  const float t2 = de * de + dp * dp;
  if (beta == 1.f) return sqrtf(t2) / r;
  if (beta == 2.f) return t2 / (r * r);
  return t2 > 0.f ? powf(t2 / (r * r), 0.5f * beta) : 0.f;
}

// pt, eta and phi of a staged particle are finite (checked before the solver: a NaN cost never enters its comparisons)
__device__ __forceinline__ bool emd_finite(float pt, float2 ep) { return isfinite(pt) & isfinite(ep.x) & isfinite(ep.y); }

// Per-CTA solver state, carved from the dynamic shared memory (emd_smem bytes).  A kernel stages its jet pair into sp / wa (rows
// i < Np: (eta, phi) and max(pt, 0); the dummy row Np: (0, 0) and 0) and sq / resb (the same for the columns) and calls emd_solve.
struct EmdState {
  double *flow, *u, *drow, *resa, *wa, *v, *resb, *red_v, *scal;
  float2 *sp, *sq;
  int *rpred, *rset, *rlist, *cpred, *red_j, *ctl;
};

__device__ __forceinline__ EmdState emd_state(int np_, int nq) {
  const int n1 = np_ + 1, n2 = nq + 1;                  // + the dummy row / column
  extern __shared__ double emd_smem[];
  EmdState S;
  S.flow = emd_smem;                                    // [n1][n2]
  S.u = S.flow + (size_t)n1 * n2;                       // [n1] row potentials
  S.drow = S.u + n1;                                    // [n1] Dijkstra distance of settled rows
  S.resa = S.drow + n1;                                 // [n1] residual supply
  S.wa = S.resa + n1;                                   // [n1] row weights
  S.v = S.wa + n1;                                      // [n2] column potentials
  S.resb = S.v + n2;                                    // [n2] residual demand
  S.red_v = S.resb + n2;                                // [32]
  S.scal = S.red_v + 32;                                // [4]: W_p, W_q, sum_i a_i u_i
  S.sp = reinterpret_cast<float2*>(S.scal + 4);         // [n1] (eta, phi) of p
  S.sq = S.sp + n1;                                     // [n2] (eta, phi) of q
  S.rpred = reinterpret_cast<int*>(S.sq + n2);          // [n1] column a settled row was reached from (-1: source)
  S.rset = S.rpred + n1;                                // [n1] row settled
  S.rlist = S.rset + n1;                                // [n1] rows settled in the current step
  S.cpred = S.rlist + n1;                               // [n2] row a column was reached from
  S.red_j = S.cpred + n2;                               // [32]
  S.ctl = S.red_j + 32;                                 // [2]: rows in rlist, status
  return S;
}

// The solver and the EMD sum on the staged jet pair (the whole CTA calls it).  Returns the EMD in every thread and leaves the
// status in S.ctl[1], the flow in S.flow, the potentials in S.u / S.v and W_p, W_q, sum_i a_i u_i in S.scal.
__device__ double emd_solve(const EmdState& S, int np_, int nq, float r, float beta, int norm, int periodic) {
  const int n1 = np_ + 1, n2 = nq + 1;
  double* const flow = S.flow; double* const u = S.u; double* const drow = S.drow; double* const resa = S.resa;
  double* const wa = S.wa; double* const v = S.v; double* const resb = S.resb; double* const red_v = S.red_v;
  double* const scal = S.scal; const float2* const sp = S.sp; const float2* const sq = S.sq;
  int* const rpred = S.rpred; int* const rset = S.rset; int* const rlist = S.rlist; int* const cpred = S.cpred;
  int* const red_j = S.red_j; int* const ctl = S.ctl;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;

  for (int idx = tid; idx < n1 * n2; idx += blockDim.x) flow[idx] = 0.0;
  for (int i = tid; i < n1; i += blockDim.x) u[i] = 0.0;
  for (int j = tid; j < n2; j += blockDim.x) v[j] = 0.0;
  if (tid == 0) { ctl[0] = 0; ctl[1] = 0; }
  __syncthreads();
  if (tid < 2) {        // jet totals in a fixed order
    const double* w = tid == 0 ? wa : resb;
    const int n = tid == 0 ? np_ : nq;
    double s = 0.0;
    for (int k = 0; k < n; ++k) s += w[k];
    scal[tid] = s;
  }
  __syncthreads();
  const double wp = scal[0], wq = scal[1];
  const double sa = norm ? (wp > 0.0 ? 1.0 : 0.0) : wp, sb = norm ? (wq > 0.0 ? 1.0 : 0.0) : wq;
  for (int i = tid; i < n1; i += blockDim.x) {
    if (i < np_) { if (norm && wp > 0.0) wa[i] /= wp; }
    else wa[i] = sb > sa ? sb - sa : 0.0;
    resa[i] = wa[i];
  }
  for (int j = tid; j < n2; j += blockDim.x) {
    if (j < nq) { if (norm && wq > 0.0) resb[j] /= wq; }
    else resb[j] = sa > sb ? sa - sb : 0.0;
  }
  __syncthreads();

  const int j = tid;                                    // this thread's column
  const bool has_col = j < n2, dummy_col = j == nq;
  const float2 qj = has_col ? sq[j] : make_float2(0.f, 0.f);
  // reduced cost c_ij - u_i - v_j of the forward arc i -> j, clamped at 0 (rounding of the potential updates)
  auto reduced = [&](int i) -> double {
    float c;
    if (i == np_ || dummy_col) c = (i == np_ && dummy_col) ? 0.f : 1.f;
    else c = emd_pair_cost(sp[i], qj, r, beta, periodic);
    return fmax((double)c - u[i] - v[j], 0.0);
  };
  // The augmentations that saturate a reverse arc grow faster than n1 + n2 (normalised compact jets against wide ones: up to
  // 2.4 (n1 + n2) at 30 x 30, 6.6 (n1 + n2) at 150 x 150) but stay below 0.16 n1 n2; the cap leaves a margin of about 8x.
  const int max_aug = n1 * n2 + 4 * (n1 + n2) + 64;
  int aug = 0;
  while (true) {
    const int any_row = __syncthreads_or(tid < n1 && resa[tid] > 0.0);
    const int any_col = __syncthreads_or(has_col && resb[j] > 0.0);
    if (!any_row || !any_col) break;
    if (aug++ == max_aug) { if (tid == 0) ctl[1] = 1; break; }
    // Dijkstra: every row with residual supply is a source at distance 0
    for (int i = tid; i < n1; i += blockDim.x) {
      const bool src = resa[i] > 0.0;
      rset[i] = src; drow[i] = src ? 0.0 : INFINITY; rpred[i] = -1;
    }
    __syncthreads();
    double dcol = INFINITY;
    int pred = -1;
    bool csettled = false;
    if (has_col)
      for (int i = 0; i < n1; ++i)
        if (rset[i]) { const double c = reduced(i); if (c < dcol) { dcol = c; pred = i; } }
    double D = INFINITY;
    int sink = -1;
    for (int step = 0; step < n2; ++step) {
      // settle the unsettled column nearest to the sources (ties: smallest column)
      double cand = has_col && !csettled ? dcol : INFINITY;
      int cj = has_col && !csettled ? j : 0x7fffffff;
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, cand, d);
        const int oj = __shfl_xor_sync(0xffffffffu, cj, d);
        if (ov < cand || (ov == cand && oj < cj)) { cand = ov; cj = oj; }
      }
      if (lane == 0) { red_v[warp] = cand; red_j[warp] = cj; }
      __syncthreads();
      double delta = red_v[0]; int js = red_j[0];
      for (int w = 1; w < nwarps; ++w) {
        const double ov = red_v[w]; const int oj = red_j[w];
        if (ov < delta || (ov == delta && oj < js)) { delta = ov; js = oj; }
      }
      if (!(delta < INFINITY)) break;                   // unreachable: forward arcs connect every source to every column
      if (j == js) csettled = true;
      if (resb[js] > 0.0) { D = delta; sink = js; break; }
      // rows reached over the reverse arcs js -> i (f_i,js > 0, reduced cost 0)
      for (int i = tid; i < n1; i += blockDim.x)
        if (!rset[i] && flow[(size_t)i * n2 + js] > 0.0) {
          rset[i] = 1; drow[i] = delta; rpred[i] = js;
          rlist[atomicAdd(&ctl[0], 1)] = i;
        }
      __syncthreads();
      const int nnew = ctl[0];
      if (has_col && !csettled)                         // min with index tie-break: independent of the list order
        for (int k = 0; k < nnew; ++k) {
          const int i = rlist[k];
          const double c = delta + reduced(i);
          if (c < dcol || (c == dcol && i < pred)) { dcol = c; pred = i; }
        }
      __syncthreads();
      if (tid == 0) ctl[0] = 0;
    }
    if (sink < 0) { if (tid == 0) ctl[1] = 3; break; }
    if (has_col) cpred[j] = pred;
    __syncthreads();
    if (tid == 0) {       // bottleneck of the path sink <- row <- column <- ... <- source row, then augment
      double amt = resb[sink];
      int jj = sink, i = cpred[jj], src = -1;
      for (int k = 0; k <= n1 + n2; ++k) {
        if (rpred[i] < 0) { amt = fmin(amt, resa[i]); src = i; break; }
        jj = rpred[i];
        amt = fmin(amt, flow[(size_t)i * n2 + jj]);
        i = cpred[jj];
      }
      if (src < 0) ctl[1] = 3;
      else {
        jj = sink; i = cpred[jj];
        for (int k = 0; k <= n1 + n2; ++k) {
          flow[(size_t)i * n2 + jj] += amt;
          if (rpred[i] < 0) break;
          jj = rpred[i];
          flow[(size_t)i * n2 + jj] -= amt;
          i = cpred[jj];
        }
        resa[src] -= amt;
        resb[sink] -= amt;
      }
    }
    for (int i = tid; i < n1; i += blockDim.x) u[i] -= rset[i] ? fmin(drow[i], D) : D;
    if (has_col) v[j] += csettled ? fmin(dcol, D) : D;
    __syncthreads();
    if (ctl[1]) break;
  }
  __syncthreads();

  // EMD = sum_ij f_ij c_ij (dummy arcs included), fixed order: column sums, then the warps in order
  double part = 0.0;
  if (has_col)
    for (int i = 0; i < n1; ++i) {
      const double f = flow[(size_t)i * n2 + j];
      if (f != 0.0) {
        const float c = (i == np_ || dummy_col) ? ((i == np_ && dummy_col) ? 0.f : 1.f) : emd_pair_cost(sp[i], qj, r, beta, periodic);
        part += f * (double)c;
      }
    }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) part += __shfl_down_sync(0xffffffffu, part, d);
  if (lane == 0) red_v[warp] = part;
  if (tid == 0 && norm) { double s = 0.0; for (int i = 0; i < np_; ++i) s += wa[i] * u[i]; scal[2] = s; }
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < nwarps; ++w) t += red_v[w];
  return t;
}

// Gradient of the EMD w.r.t. (pt, eta, phi) of the real row i < Np after emd_solve, in the order (pt, eta, phi)
__device__ __forceinline__ void emd_row_grad(const EmdState& S, int i, int np_, int nq, float r, float beta, int norm, int periodic,
                                             double& gw, double& ge, double& gp) {
  const int n2 = nq + 1;
  const double wp = S.scal[0], wq = S.scal[1];
  // d/d(eta_i, phi_i) sum_j f_ij (theta_ij / R)^beta = sum_j f_ij beta c_ij / theta_ij^2 (deta, dphi), 0 at theta = 0
  const float2 a = S.sp[i];
  ge = 0.0; gp = 0.0;
  for (int jq = 0; jq < nq; ++jq) {
    const double f = S.flow[(size_t)i * n2 + jq];
    if (f > 0.0) {
      const float2 c = S.sq[jq];
      const float de = a.x - c.x, dph = emd_dphi(a.y - c.y, periodic), t2 = de * de + dph * dph;
      if (t2 > 0.f) {
        const double k = f * (double)beta * (double)emd_pair_cost(a, c, r, beta, periodic) / (double)t2;
        ge += k * de; gp += k * dph;
      }
    }
  }
  // d/da_i of the optimum is the row's dual minus that of the dummy whose weight a_i changes (+ the normalisation's chain rule)
  gw = 0.0;
  if (S.wa[i] > 0.0) {
    if (norm) gw = (S.u[i] - S.scal[2]) / wp;
    else gw = wp <= wq ? S.u[i] - S.u[np_] : S.u[i] + S.v[nq];
  }
}

__global__ void emd_kernel(int np_, int nq, float r, float beta, int norm, int periodic, const float* __restrict__ p,
                           const float* __restrict__ q, double* __restrict__ emd_out, double* __restrict__ flow_out,
                           float* __restrict__ dp_out, double* __restrict__ pot_out, int* __restrict__ status_out) {
  gj_pdl_sync();
  const int n1 = np_ + 1, n2 = nq + 1;
  const EmdState S = emd_state(np_, nq);
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* pg = p + (size_t)b * np_ * 3;
  const float* qg = q + (size_t)b * nq * 3;
  bool finite = true;
  for (int i = tid; i < n1; i += blockDim.x) {
    const bool real = i < np_;
    const float pt = real ? __ldg(pg + i * 3) : 0.f;
    S.sp[i] = real ? make_float2(__ldg(pg + i * 3 + 1), __ldg(pg + i * 3 + 2)) : make_float2(0.f, 0.f);
    S.wa[i] = real ? fmax((double)pt, 0.0) : 0.0;
    finite &= emd_finite(pt, S.sp[i]);
  }
  for (int j = tid; j < n2; j += blockDim.x) {
    const bool real = j < nq;
    const float pt = real ? __ldg(qg + j * 3) : 0.f;
    S.sq[j] = real ? make_float2(__ldg(qg + j * 3 + 1), __ldg(qg + j * 3 + 2)) : make_float2(0.f, 0.f);
    S.resb[j] = real ? fmax((double)pt, 0.0) : 0.0;
    finite &= emd_finite(pt, S.sq[j]);
  }
  if (__syncthreads_or(!finite)) {      // not solved: status 2, EMD NaN, no flow, NaN potentials, zero gradient rows
    if (tid == 0) { emd_out[b] = __longlong_as_double(0x7ff8000000000000ll); if (status_out) status_out[b] = 2; }
    if (flow_out) for (int idx = tid; idx < np_ * nq; idx += blockDim.x) flow_out[(size_t)b * np_ * nq + idx] = 0.0;
    if (pot_out) for (int k = tid; k < n1 + n2; k += blockDim.x) pot_out[(size_t)b * (n1 + n2) + k] = __longlong_as_double(0x7ff8000000000000ll);
    if (dp_out) for (int k = tid; k < np_ * 3; k += blockDim.x) dp_out[(size_t)b * np_ * 3 + k] = 0.f;
    return;
  }
  const double t = emd_solve(S, np_, nq, r, beta, norm, periodic);
  if (tid == 0) {
    emd_out[b] = t;
    if (status_out) status_out[b] = S.ctl[1];
  }
  if (flow_out)
    for (int idx = tid; idx < np_ * nq; idx += blockDim.x) {
      const int i = idx / nq, jq = idx - i * nq;
      flow_out[(size_t)b * np_ * nq + idx] = S.flow[(size_t)i * n2 + jq];
    }
  if (pot_out) {
    double* po = pot_out + (size_t)b * (n1 + n2);
    for (int i = tid; i < n1; i += blockDim.x) po[i] = S.u[i];
    if (tid < n2) po[n1 + tid] = S.v[tid];
  }
  if (dp_out && tid < np_) {
    double gw, ge, gp;
    emd_row_grad(S, tid, np_, nq, r, beta, norm, periodic, gw, ge, gp);
    float* o = dp_out + ((size_t)b * np_ + tid) * 3;
    o[0] = (float)gw; o[1] = (float)ge; o[2] = (float)gp;
  }
}

// (pt, eta, phi) of particle k of a (.., dim) jet: the first three features (polar) or converted from the last three (Cartesian)
__device__ __forceinline__ float3 emd_load_polar(const float* __restrict__ x, int k, int dim, int cartesian) {
  const float* e = x + (size_t)k * dim;
  if (cartesian) return gj_to_polar(__ldg(e + dim - 3), __ldg(e + dim - 2), __ldg(e + dim - 1));
  return make_float3(__ldg(e), __ldg(e + 1), __ldg(e + 2));
}

// The EMD loss of the training step: one CTA per jet pair (p = reconstruction, q = target, both (B, N, dim)), the solver of
// emd_kernel, and as epilogue the per-jet EMD and status into the workspace and scale * dEMD/dp in p's own coordinates.
__global__ void emd_loss_kernel(int n, int dim, int cartesian, float r, float beta, int norm, int periodic, float scale,
                                const float* __restrict__ p, const float* __restrict__ q, float* __restrict__ dp,
                                double* __restrict__ jet_emd, int* __restrict__ jet_status) {
  gj_pdl_sync();
  const int n1 = n + 1;
  const EmdState S = emd_state(n, n);
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* pg = p + (size_t)b * n * dim;
  const float* qg = q + (size_t)b * n * dim;
  bool finite = true;
  for (int i = tid; i < n1; i += blockDim.x) {
    const bool real = i < n;
    const float3 a = real ? emd_load_polar(pg, i, dim, cartesian) : make_float3(0.f, 0.f, 0.f);
    const float3 c = real ? emd_load_polar(qg, i, dim, cartesian) : make_float3(0.f, 0.f, 0.f);
    S.sp[i] = make_float2(a.y, a.z); S.wa[i] = real ? fmax((double)a.x, 0.0) : 0.0;
    S.sq[i] = make_float2(c.y, c.z); S.resb[i] = real ? fmax((double)c.x, 0.0) : 0.0;
    finite &= emd_finite(a.x, S.sp[i]) & emd_finite(c.x, S.sq[i]);
  }
  if (__syncthreads_or(!finite)) {      // not solved: status 2, EMD NaN, zero gradient rows
    if (tid == 0) { jet_emd[b] = __longlong_as_double(0x7ff8000000000000ll); jet_status[b] = 2; }
    if (dp) for (int k = tid; k < n * dim; k += blockDim.x) dp[(size_t)b * n * dim + k] = 0.f;
    return;
  }
  const double t = emd_solve(S, n, n, r, beta, norm, periodic);
  if (tid == 0) { jet_emd[b] = t; jet_status[b] = S.ctl[1]; }
  if (dp && tid < n) {
    double gw, ge, gp;
    emd_row_grad(S, tid, n, n, r, beta, norm, periodic, gw, ge, gp);
    // the fp32 gradient gj_emd writes, scaled in fp64 as autograd scales it
    const double s = (double)scale;
    const double g0 = (double)(float)gw * s, g1 = (double)(float)ge * s, g2 = (double)(float)gp * s;
    float* o = dp + ((size_t)b * n + tid) * dim;
    if (!cartesian) { o[0] = (float)g0; o[1] = (float)g1; o[2] = (float)g2; return; }
    // chain rule through gj_to_polar; the energy of a 4-vector does not enter the EMD
    const float* e = pg + (size_t)tid * dim + dim - 3;
    double gx, gy, gz;
    gj_to_polar_grad(__ldg(e), __ldg(e + 1), __ldg(e + 2), g0, g1, g2, gx, gy, gz);
    if (dim == 4) o[0] = 0.f;
    o[dim - 3] = (float)gx;
    o[dim - 2] = (float)gy;
    o[dim - 1] = (float)gz;
  }
}

// Fixed-order sum of the per-jet EMDs and count of the jets whose solver stopped without the optimum (a jet with non-finite input,
// status 2, is not counted: its EMD is NaN and makes the sum NaN)
__global__ void __launch_bounds__(256) emd_loss_sum_kernel(int batch, float scale, const double* __restrict__ jet_emd,
                                                           const int* __restrict__ jet_status, float* __restrict__ terms,
                                                           float* __restrict__ failed) {
  gj_pdl_sync();
  __shared__ double red[8];
  __shared__ int redf[8];
  double s = 0.0;
  int f = 0;
  for (int b = threadIdx.x; b < batch; b += 256) { s += jet_emd[b]; f += jet_status[b] != 0 && jet_status[b] != 2; }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { s += __shfl_down_sync(0xffffffffu, s, d); f += __shfl_down_sync(0xffffffffu, f, d); }
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = s; redf[threadIdx.x >> 5] = f; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    int nf = 0;
    for (int w = 0; w < 8; ++w) { t += red[w]; nf += redf[w]; }
    terms[0] = (float)t; terms[1] = 0.f; terms[2] = (float)((double)scale * t);
    failed[0] = (float)nf;
  }
}

}  // namespace

void gj_set_error(const char* fmt, ...);

static size_t emd_smem(int np_, int nq) {
  const size_t n1 = (size_t)np_ + 1, n2 = (size_t)nq + 1;
  return (n1 * n2 + 4 * n1 + 2 * n2 + 32 + 4) * sizeof(double) + (n1 + n2) * sizeof(float2) + (3 * n1 + n2 + 32 + 2) * sizeof(int);
}

int gj_emd_check(int batch, int np_, int nq, float r, float beta, int flags) {
  if (batch < 0 || np_ < 1 || nq < 1 || np_ > kEmdMaxParticles || nq > kEmdMaxParticles) {
    gj_set_error("gj_emd: 1 <= particles per jet <= %d on both sides (fp64 flow matrix in shared memory), got %d and %d",
                 kEmdMaxParticles, np_, nq);
    return GJ_ERR_INVALID;
  }
  if (!(r > 0.f) || !isfinite(r)) { gj_set_error("gj_emd: R must be positive and finite, got %g", (double)r); return GJ_ERR_INVALID; }
  if (!(beta > 0.f) || !isfinite(beta)) { gj_set_error("gj_emd: beta must be positive and finite, got %g", (double)beta); return GJ_ERR_INVALID; }
  if (flags & ~(GJ_EMD_NORM | GJ_EMD_PERIODIC_PHI)) { gj_set_error("gj_emd: unknown flags 0x%x", flags); return GJ_ERR_INVALID; }
  return GJ_OK;
}

int gj_emd_launch(int batch, int np_, int nq, const float* p, const float* q, float r, float beta, int flags, double* emd_out,
                  double* flow_out, float* dp_out, double* pot_out, int* status_out, cudaStream_t stream) {
  if (batch == 0) return GJ_OK;
  const size_t smem = emd_smem(np_, nq);
  const int n = (np_ > nq ? np_ : nq) + 1;
  cudaError_t ce = cudaSuccess;
  if (smem > 48 * 1024) ce = cudaFuncSetAttribute(emd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ce == cudaSuccess) {
    gj_launch(emd_kernel, batch, gj_round_up(n, 32), smem, stream, np_, nq, r, beta, (flags & GJ_EMD_NORM) ? 1 : 0,
              (flags & GJ_EMD_PERIODIC_PHI) ? 1 : 0, p, q, emd_out, flow_out, dp_out, pot_out, status_out);
    ce = cudaGetLastError();
  }
  if (ce != cudaSuccess) { gj_set_error("emd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

size_t gj_emd_loss_ws_bytes(int batch) { return batch > 0 ? (size_t)batch * (sizeof(double) + sizeof(int)) : 0; }

int gj_emd_loss_check(int batch, int n, int dim, int coords, float r, float beta, int flags, size_t ws_bytes) {
  if (batch < 0 || n < 1 || n > kEmdMaxParticles) {
    gj_set_error("gj_emd_loss: batch >= 0 and 1 <= particles per jet <= %d (fp64 flow matrix in shared memory), got %d and %d",
                 kEmdMaxParticles, batch, n);
    return GJ_ERR_INVALID;
  }
  if (dim != 3 && dim != 4) { gj_set_error("gj_emd_loss: features per particle must be 3 or 4, got %d", dim); return GJ_ERR_INVALID; }
  if (coords != GJ_EMD_COORDS_POLAR && coords != GJ_EMD_COORDS_CARTESIAN) {
    gj_set_error("gj_emd_loss: unknown coordinates %d", coords); return GJ_ERR_INVALID; }
  if (coords == GJ_EMD_COORDS_POLAR && dim != 3) {
    gj_set_error("gj_emd_loss: polar coordinates are [pt, eta, phi] (3 features), got %d", dim); return GJ_ERR_INVALID; }
  if (!(r > 0.f) || !isfinite(r)) { gj_set_error("gj_emd_loss: R must be positive and finite, got %g", (double)r); return GJ_ERR_INVALID; }
  if (!(beta > 0.f) || !isfinite(beta)) { gj_set_error("gj_emd_loss: beta must be positive and finite, got %g", (double)beta); return GJ_ERR_INVALID; }
  if (flags & ~(GJ_EMD_NORM | GJ_EMD_PERIODIC_PHI)) { gj_set_error("gj_emd_loss: unknown flags 0x%x", flags); return GJ_ERR_INVALID; }
  if (ws_bytes < gj_emd_loss_ws_bytes(batch)) {
    gj_set_error("gj_emd_loss: workspace too small (%zu bytes, needs %zu)", ws_bytes, gj_emd_loss_ws_bytes(batch));
    return GJ_ERR_WORKSPACE;
  }
  return GJ_OK;
}

int gj_emd_loss_launch(int batch, int n, int dim, int coords, const float* p, const float* q, float r, float beta, int flags,
                       float scale, float* terms, float* failed, float* dp, void* ws, cudaStream_t stream) {
  double* jet_emd = (double*)ws;
  int* jet_status = (int*)(jet_emd + batch);
  cudaError_t ce = cudaSuccess;
  if (batch > 0) {
    const size_t smem = emd_smem(n, n);
    if (smem > 48 * 1024) ce = cudaFuncSetAttribute(emd_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce == cudaSuccess)
      ce = gj_launch(emd_loss_kernel, batch, gj_round_up(n + 1, 32), smem, stream, n, dim, coords == GJ_EMD_COORDS_CARTESIAN ? 1 : 0,
                     r, beta, (flags & GJ_EMD_NORM) ? 1 : 0, (flags & GJ_EMD_PERIODIC_PHI) ? 1 : 0, scale, p, q, dp, jet_emd,
                     jet_status);
  }
  if (ce == cudaSuccess) ce = gj_launch(emd_loss_sum_kernel, 1, 256, 0, stream, batch, scale, (const double*)jet_emd,
                                        (const int*)jet_status, terms, failed);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("emd loss launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
