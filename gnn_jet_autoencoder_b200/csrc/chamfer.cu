// Fused Chamfer / jet-sum loss, forward + gradient w.r.t. the reconstruction, one CTA per jet.
// Replaces reference utils/losses/chamfer_loss/chamfer_loss.py:11-42 and
// utils/losses/chamfer_loss/distance_sq.py:4-77 (which materialise two (B,N,N,D) repeats).
// HBM-bound: 3*N*D*4 bytes per jet; gradients flow through the arg-mins only (torch.min semantics,
// first index on ties).
#include "gj_common.cuh"

namespace {

__global__ void chamfer_kernel(int np_, int nq, int dim, int mink, int mink_jet, float wc, float wj, const float* __restrict__ p,
                               const float* __restrict__ q, float* __restrict__ jet_terms, float* __restrict__ dp) {
  gj_pdl_sync();
  extern __shared__ float sm[];
  float* sp = sm;                       // [np][4]
  float* sq = sp + np_ * 4;             // [nq][4]
  int* jstar = reinterpret_cast<int*>(sq + nq * 4);   // [np]
  int* istar = jstar + np_;                            // [nq]
  float* red = reinterpret_cast<float*>(istar + nq);   // [blockDim/32 * 2] + [8] jet diff
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* pg = p + (size_t)b * np_ * dim;
  const float* qg = q + (size_t)b * nq * dim;
  for (int idx = tid; idx < np_ * 4; idx += blockDim.x) { int n = idx >> 2, c = idx & 3; sp[idx] = c < dim ? __ldg(pg + n * dim + c) : 0.f; }
  for (int idx = tid; idx < nq * 4; idx += blockDim.x) { int n = idx >> 2, c = idx & 3; sq[idx] = c < dim ? __ldg(qg + n * dim + c) : 0.f; }
  __syncthreads();
  const float s1 = mink ? -1.f : 1.f;       // sign of components 1..3 in the pairwise distances
  const float sj = mink_jet ? -1.f : 1.f;   // ... and in the jet term (chamfer_loss.py:40 passes loss_norm_choice unchanged)
  float local = 0.f;
  if (tid < np_) {          // nearest target for each reconstructed particle
    float4 a = *reinterpret_cast<const float4*>(sp + tid * 4);
    float best = INFINITY; int bj = 0;
    for (int j = 0; j < nq; ++j) {
      float4 c = *reinterpret_cast<const float4*>(sq + j * 4);
      float dx = a.x - c.x, dy = a.y - c.y, dz = a.z - c.z, dw = a.w - c.w;
      float d = dx * dx + s1 * (dy * dy + dz * dz + dw * dw);
      if (d < best) { best = d; bj = j; }
    }
    jstar[tid] = bj; local += best;
  }
  if (tid < nq) {           // nearest reconstructed particle for each target
    float4 c = *reinterpret_cast<const float4*>(sq + tid * 4);
    float best = INFINITY; int bi = 0;
    for (int i = 0; i < np_; ++i) {
      float4 a = *reinterpret_cast<const float4*>(sp + i * 4);
      float dx = a.x - c.x, dy = a.y - c.y, dz = a.z - c.z, dw = a.w - c.w;
      float d = dx * dx + s1 * (dy * dy + dz * dz + dw * dw);
      if (d < best) { best = d; bi = i; }
    }
    istar[tid] = bi; local += best;
  }
  // jet feature difference: sum_i p_i - sum_j q_j, one warp, fixed order
  float* jd = red + 64;
  if (tid < 4) {
    float acc = 0.f;
    for (int i = 0; i < np_; ++i) acc += sp[i * 4 + tid];
    float acc2 = 0.f;
    for (int j = 0; j < nq; ++j) acc2 += sq[j * 4 + tid];
    jd[tid] = acc - acc2;
  }
  float ws = gj_warp_sum(local);
  if ((tid & 31) == 0) red[tid >> 5] = ws;
  __syncthreads();
  if (tid == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    float jt = jd[0] * jd[0] + sj * (jd[1] * jd[1] + jd[2] * jd[2] + jd[3] * jd[3]);
    jet_terms[b * 2 + 0] = tot;
    jet_terms[b * 2 + 1] = jt;
  }
  if (dp && tid < np_) {
    const float sgn[4] = {2.f, 2.f * s1, 2.f * s1, 2.f * s1};
    const float sgj[4] = {2.f, 2.f * sj, 2.f * sj, 2.f * sj};
    float g[4];
    const float* a = sp + tid * 4;
    const float* c = sq + jstar[tid] * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) g[k] = a[k] - c[k];
    for (int j = 0; j < nq; ++j)
      if (istar[j] == tid) {
#pragma unroll
        for (int k = 0; k < 4; ++k) g[k] += a[k] - sq[j * 4 + k];
      }
    for (int k = 0; k < dim; ++k) dp[((size_t)b * np_ + tid) * dim + k] = sgn[k] * wc * g[k] + sgj[k] * wj * jd[k];
  }
}

// terms[t] = sum_b jet_terms[b][t], single block, fixed tree => deterministic
__global__ void chamfer_reduce_kernel(int batch, float wc, float wj, const float* __restrict__ jet_terms,
                                      float* __restrict__ terms) {
  gj_pdl_sync();
  __shared__ float red[2][32];
  float a0 = 0.f, a1 = 0.f;
  for (int b = threadIdx.x; b < batch; b += blockDim.x) { a0 += jet_terms[b * 2]; a1 += jet_terms[b * 2 + 1]; }
  a0 = gj_warp_sum(a0); a1 = gj_warp_sum(a1);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a0; red[1][threadIdx.x >> 5] = a1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t0 = 0.f, t1 = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { t0 += red[0][w]; t1 += red[1][w]; }
    terms[0] = t0; terms[1] = t1; terms[2] = wc * t0 + wj * t1;
  }
}

// Per-particle nearest-neighbour distances of the anomaly scores (reference utils/jet_analysis/anomaly_detection.py:
// chamfer :459-488 with the Euclidean norm, chamfer_lorentz :491-510 with E^2 - px^2 - py^2 - pz^2), one CTA per jet:
// min_pq[b][i] = min_j dist(p_i, q_j), min_qp[b][j] = min_i dist(p_i, q_j).  No (B,N,N,D) difference tensor is built.
__global__ void pair_min_dist_kernel(int np_, int nq, int dim, int lorentz, const float* __restrict__ p, const float* __restrict__ q,
                                     float* __restrict__ min_pq, float* __restrict__ min_qp) {
  gj_pdl_sync();
  extern __shared__ float sm[];
  float* sp = sm;                       // [np][4]
  float* sq = sp + np_ * 4;             // [nq][4]
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* pg = p + (size_t)b * np_ * dim;
  const float* qg = q + (size_t)b * nq * dim;
  for (int idx = tid; idx < np_ * 4; idx += blockDim.x) { int n = idx >> 2, c = idx & 3; sp[idx] = c < dim ? __ldg(pg + n * dim + c) : 0.f; }
  for (int idx = tid; idx < nq * 4; idx += blockDim.x) { int n = idx >> 2, c = idx & 3; sq[idx] = c < dim ? __ldg(qg + n * dim + c) : 0.f; }
  __syncthreads();
  const float s1 = lorentz ? -1.f : 1.f;
  for (int i = tid; i < np_; i += blockDim.x) {
    const float4 a = *reinterpret_cast<const float4*>(sp + i * 4);
    float best = INFINITY;
    for (int j = 0; j < nq; ++j) {
      const float4 c = *reinterpret_cast<const float4*>(sq + j * 4);
      const float dx = a.x - c.x, dy = a.y - c.y, dz = a.z - c.z, dw = a.w - c.w;
      best = fminf(best, dx * dx + s1 * (dy * dy + dz * dz + dw * dw));
    }
    min_pq[(size_t)b * np_ + i] = lorentz ? best : sqrtf(best);      // the minimum of the norms is the norm at the minimum square
  }
  for (int j = tid; j < nq; j += blockDim.x) {
    const float4 c = *reinterpret_cast<const float4*>(sq + j * 4);
    float best = INFINITY;
    for (int i = 0; i < np_; ++i) {
      const float4 a = *reinterpret_cast<const float4*>(sp + i * 4);
      const float dx = a.x - c.x, dy = a.y - c.y, dz = a.z - c.z, dw = a.w - c.w;
      best = fminf(best, dx * dx + s1 * (dy * dy + dz * dz + dw * dw));
    }
    min_qp[(size_t)b * nq + j] = lorentz ? best : sqrtf(best);
  }
}

// Optimal assignment between the particles of p and q per jet (the matching step of reference
// utils/jet_analysis/anomaly_detection.py: hungarian :513-547, hungarian_lorentz :550-590, and of
// utils/losses/hungarian_mse/hungarian_mse.py:51-56, which call scipy.optimize.linear_sum_assignment jet by jet on the
// host).  One CTA per jet, thread j owns column j: the O(n^3) shortest-augmenting-path Hungarian method with row / column
// potentials (u, v), where the scan over the columns of every path step -- relax, arg-min, potential update -- runs across
// the threads.  Costs are fp32 (|p_i - q_j|_2 or the Lorentz norm squared), potentials and slacks fp64.  A jet with a cost that is
// not finite is not solved (identity matching, NaN cost or loss, zero gradient rows): asg_cost checks before asg_solve runs.
// col_for_row[b][i] = column assigned to row i (linear_sum_assignment's second array for a square matrix).
constexpr int kAsgMaxParticles = 220;     // the largest n with assignment_smem(n) <= 200 KB

// Per-CTA solver state, carved from the dynamic shared memory (assignment_smem bytes).  A kernel stages its jet pair into sp / sq
// ([n][4], components beyond the jet's zero) and calls asg_cost, then asg_solve.
struct AsgState {
  float *sp, *sq, *cost;
  double *u, *red_v;
  int *red_j, *prow, *way, *ctl;
};

__device__ __forceinline__ AsgState asg_state(int n) {
  extern __shared__ float4 asg_smem[];
  AsgState S;
  S.sp = reinterpret_cast<float*>(asg_smem);                  // [n][4]
  S.sq = S.sp + n * 4;                                        // [n][4]
  S.u = reinterpret_cast<double*>(S.sq + n * 4);              // [n + 1] row potentials (1-based, 0 = none)
  S.red_v = S.u + (n + 1);                                    // [32] per-warp minima
  S.red_j = reinterpret_cast<int*>(S.red_v + 32);             // [32]
  S.prow = S.red_j + 32;                                      // [n + 1] row matched to column j (0 = free)
  S.way = S.prow + (n + 1);                                   // [n + 1]
  S.ctl = S.way + (n + 1);                                    // [2]: current column j0, spare
  S.cost = reinterpret_cast<float*>(S.ctl + 2);               // [n][n]
  return S;
}

// cost[i][j] = |sp_i - sq_j|_2 (lorentz: E^2 - px^2 - py^2 - pz^2 of the difference) and the solver's initial state; the staged
// jets must be visible to the whole CTA (a __syncthreads after the staging).  Returns, in every thread, whether every cost is finite:
// the caller must not run asg_solve otherwise -- a NaN or infinite cost never wins a comparison, so the path search would leave
// stale entries in way[] and its augmentation walk need not end.
__device__ __forceinline__ bool asg_cost(const AsgState& S, int n, int lorentz) {
  const int tid = threadIdx.x;
  for (int idx = tid; idx <= n; idx += blockDim.x) { S.u[idx] = 0.0; S.prow[idx] = 0; S.way[idx] = 0; }
  const float s1 = lorentz ? -1.f : 1.f;
  bool finite = true;
  for (int idx = tid; idx < n * n; idx += blockDim.x) {
    const int i = idx / n, j = idx - i * n;
    const float4 a = *reinterpret_cast<const float4*>(S.sp + i * 4), c = *reinterpret_cast<const float4*>(S.sq + j * 4);
    const float dx = a.x - c.x, dy = a.y - c.y, dz = a.z - c.z, dw = a.w - c.w;
    const float d2 = dx * dx + s1 * (dy * dy + dz * dz + dw * dw);
    const float cij = lorentz ? d2 : sqrtf(d2);
    S.cost[idx] = cij;
    finite &= isfinite(cij);
  }
  return !__syncthreads_or(!finite);
}

// The shortest-augmenting-path solve on S.cost (the whole CTA calls it); leaves the matching in S.prow: prow[j] = 1-based row
// assigned to the 1-based column j.
__device__ void asg_solve(const AsgState& S, int n) {
  double* const u = S.u; double* const red_v = S.red_v; const float* const cost = S.cost;
  int* const red_j = S.red_j; int* const prow = S.prow; int* const way = S.way; int* const ctl = S.ctl;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int j = tid + 1;                 // this thread's column (1-based); threads beyond n idle along
  const bool has_col = j <= n;
  double v = 0.0, minv = 0.0;
  bool used = false;
  for (int i = 1; i <= n; ++i) {
    if (tid == 0) { prow[0] = i; ctl[0] = 0; }
    minv = INFINITY; used = false;
    __syncthreads();
    while (true) {
      const int j0 = ctl[0], i0 = prow[j0];
      if (has_col && j == j0) used = true;
      double cand = INFINITY;
      if (has_col && !used) {
        const double cur = (double)cost[(size_t)(i0 - 1) * n + (j - 1)] - u[i0] - v;
        if (cur < minv) { minv = cur; way[j] = j0; }
        cand = minv;
      }
      // block arg-min of cand (ties: smallest column)
      int cj = has_col && !used ? j : 0x7fffffff;
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, cand, d);
        const int oj = __shfl_xor_sync(0xffffffffu, cj, d);
        if (ov < cand || (ov == cand && oj < cj)) { cand = ov; cj = oj; }
      }
      if (lane == 0) { red_v[warp] = cand; red_j[warp] = cj; }
      __syncthreads();
      double delta = red_v[0]; int j1 = red_j[0];
      for (int w = 1; w < nwarps; ++w) {
        const double ov = red_v[w]; const int oj = red_j[w];
        if (ov < delta || (ov == delta && oj < j1)) { delta = ov; j1 = oj; }
      }
      // potentials: matched (used) columns move with their rows, free columns get closer by delta
      if (has_col) {
        if (used) { u[prow[j]] += delta; v -= delta; }
        else minv -= delta;
      }
      if (tid == 0) { u[prow[0]] += delta; ctl[0] = j1; }
      __syncthreads();
      if (prow[j1] == 0) break;
    }
    if (tid == 0) {      // augment along the recorded path
      int j0 = ctl[0];
      do { const int jn = way[j0]; prow[j0] = prow[jn]; j0 = jn; } while (j0);
    }
    __syncthreads();
  }
}

__global__ void assignment_kernel(int n, int dim, int lorentz, const float* __restrict__ p, const float* __restrict__ q,
                                  int* __restrict__ col_for_row, float* __restrict__ total_cost) {
  gj_pdl_sync();
  const AsgState S = asg_state(n);
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const float* pg = p + (size_t)b * n * dim;
  const float* qg = q + (size_t)b * n * dim;
  for (int idx = tid; idx < n * 4; idx += blockDim.x) {
    const int r = idx >> 2, c = idx & 3;
    S.sp[idx] = c < dim ? __ldg(pg + r * dim + c) : 0.f;
    S.sq[idx] = c < dim ? __ldg(qg + r * dim + c) : 0.f;
  }
  __syncthreads();
  if (!asg_cost(S, n, lorentz)) {      // not solved: identity matching, NaN cost
    for (int i = tid; i < n; i += blockDim.x) col_for_row[(size_t)b * n + i] = i;
    if (total_cost && tid == 0) total_cost[b] = __int_as_float(0x7fffffff);
    return;
  }
  asg_solve(S, n);
  const int j = tid + 1;
  const bool has_col = j <= n;
  if (has_col) col_for_row[(size_t)b * n + (S.prow[j] - 1)] = j - 1;
  if (total_cost) {
    float c = has_col ? S.cost[(size_t)(S.prow[j] - 1) * n + (j - 1)] : 0.f;
    c = gj_warp_sum(c);
    __syncthreads();
    if (lane == 0) S.red_v[warp] = (double)c;
    __syncthreads();
    if (tid == 0) { double t = 0.0; for (int w = 0; w < nwarps; ++w) t += S.red_v[w]; total_cost[b] = (float)t; }
  }
}

// _relative_polar of one particle's (pt, eta, phi) to the jet axis: pt / (pt_jet + eps), eta - eta_jet and
// remainder(phi - phi_jet + pi, 2 pi) - pi (torch's remainder: fmod, moved into the divisor's sign)
__device__ __forceinline__ float3 hmse_relative(float3 t, float3 axis) {
  const float pi = 3.14159265358979f, two_pi = 6.283185307179586f;
  float m = fmodf(__fadd_rn(__fsub_rn(t.z, axis.z), pi), two_pi);
  if (m < 0.f) m = __fadd_rn(m, two_pi);
  return make_float3(__fdiv_rn(t.x, __fadd_rn(axis.x, GJ_EPS)), __fsub_rn(t.y, axis.y), __fsub_rn(m, pi));
}

// T(x_k) of particle k of a (.., dim) jet into out[4] (components beyond the loss's zero)
__device__ __forceinline__ void hmse_stage(const float* __restrict__ x, int k, int dim, int coords, float3 axis, float* out) {
  const float* e = x + (size_t)k * dim;
  if (coords == GJ_HMSE_ABS_CARTESIAN) {
    for (int c = 0; c < 4; ++c) out[c] = c < dim ? __ldg(e + c) : 0.f;
    return;
  }
  float3 t = gj_to_polar(__ldg(e + dim - 3), __ldg(e + dim - 2), __ldg(e + dim - 1));
  if (coords != GJ_HMSE_ABS_POLAR) t = hmse_relative(t, axis);
  out[3] = 0.f;
  if (coords == GJ_HMSE_REL_CARTESIAN) {      // _polar_to_cartesian with the reference's py = pt cos(phi)
    const float cp = cosf(t.z);
    out[0] = __fmul_rn(t.x, cp); out[1] = __fmul_rn(t.x, cp); out[2] = __fmul_rn(t.x, sinhf(t.y));
    return;
  }
  out[0] = t.x; out[1] = t.y; out[2] = t.z;
}

// The Hungarian-matched MSE of reference utils/losses/hungarian_mse/hungarian_mse.py:27-58 (losses.HungarianMSELoss) as a training
// loss: one CTA per jet pair (p = reconstruction, q = target, both (B, N, dim)).
//   1. both jets staged in the loss's coordinates T (losses.hungarian_preprocess, operation by operation as torch computes them);
//   2. the assignment of assignment_kernel on cost |T(p)_i - T(q)_j|_2, sigma = col_for_row;
//   3. the jet's loss sum_i |T(p)_sigma(i) - T(q)_i|^2 (the module gathers the reconstruction with the column indices), fp64, to
//      jet_loss[b];
//   4. dp_k = 2 scale (T(p)_k - T(q)_sigma^-1(k)) J_T(p_k) in p's own coordinates; the matching is piecewise constant and the target
//      jet's axis a constant, so J_T is per particle.
// Relative coordinates are taken to the axis of the TARGET jet, the sum of its particles converted by _to_polar.
__global__ void hungarian_mse_loss_kernel(int n, int dim, int coords, float scale, const float* __restrict__ p,
                                          const float* __restrict__ q, float* __restrict__ dp, int* __restrict__ col_for_row,
                                          double* __restrict__ jet_loss) {
  gj_pdl_sync();
  __shared__ float jet_s[4];
  const AsgState S = asg_state(n);
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const float* pg = p + (size_t)b * n * dim;
  const float* qg = q + (size_t)b * n * dim;
  const bool relative = coords == GJ_HMSE_REL_POLAR || coords == GJ_HMSE_REL_CARTESIAN;
  if (relative && tid < dim) {      // the target jet, summed in particle order, one thread per component
    float s = 0.f;
    for (int k = 0; k < n; ++k) s += __ldg(qg + (size_t)k * dim + tid);
    jet_s[tid] = s;
  }
  __syncthreads();
  const float3 axis = relative ? gj_to_polar(jet_s[dim - 3], jet_s[dim - 2], jet_s[dim - 1]) : make_float3(0.f, 0.f, 0.f);
  for (int k = tid; k < n; k += blockDim.x) {
    hmse_stage(pg, k, dim, coords, axis, S.sp + k * 4);
    hmse_stage(qg, k, dim, coords, axis, S.sq + k * 4);
  }
  __syncthreads();
  if (!asg_cost(S, n, 0)) {      // not solved: identity matching, NaN loss, zero gradient rows
    for (int k = tid; k < n; k += blockDim.x) {
      if (col_for_row) col_for_row[(size_t)b * n + k] = k;
      for (int m = 0; m < dim; ++m) dp[((size_t)b * n + k) * dim + m] = 0.f;
    }
    if (tid == 0) jet_loss[b] = __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  asg_solve(S, n);
  // thread k owns particle k of p, matched to particle i = sigma^-1(k) of q
  const int k = tid;
  double e = 0.0;
  if (k < n) {
    const int i = S.prow[k + 1] - 1;
    if (col_for_row) col_for_row[(size_t)b * n + i] = k;
    double g[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const float d = __fsub_rn(S.sp[k * 4 + m], S.sq[i * 4 + m]);
      e += (double)d * (double)d;
      g[m] = 2.0 * (double)scale * (double)d;
    }
    float* o = dp + ((size_t)b * n + k) * dim;
    if (coords == GJ_HMSE_ABS_CARTESIAN) {
      o[0] = (float)g[0]; o[1] = (float)g[1]; o[2] = (float)g[2];
      if (dim == 4) o[3] = (float)g[3];
    } else {
      const float* x = pg + (size_t)k * dim + dim - 3;
      const float px = __ldg(x), py = __ldg(x + 1), pz = __ldg(x + 2);
      if (relative) {
        const float3 r = hmse_relative(gj_to_polar(px, py, pz), axis);
        if (coords == GJ_HMSE_REL_CARTESIAN) {      // d/d(pt', eta', phi') of (pt' cos phi', pt' cos phi', pt' sinh eta')
          const double pt = r.x, eta = r.y, phi = r.z, gxy = g[0] + g[1];
          g[0] = gxy * cos(phi) + g[2] * sinh(eta);
          g[1] = g[2] * pt * cosh(eta);
          g[2] = -gxy * pt * sin(phi);
        }
        g[0] /= (double)__fadd_rn(axis.x, GJ_EPS);      // pt' = pt / (pt_jet + eps); the shifts and the wrap have slope 1
      }
      double gx, gy, gz;
      gj_to_polar_grad(px, py, pz, g[0], g[1], g[2], gx, gy, gz);
      if (dim == 4) o[0] = 0.f;
      o[dim - 3] = (float)gx;
      o[dim - 2] = (float)gy;
      o[dim - 1] = (float)gz;
    }
  }
  // the jet's loss: per particle, then a shuffle tree per warp, then the warps in order
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) e += __shfl_down_sync(0xffffffffu, e, d);
  if (lane == 0) S.red_v[warp] = e;
  __syncthreads();
  if (tid == 0) { double t = 0.0; for (int w = 0; w < nwarps; ++w) t += S.red_v[w]; jet_loss[b] = t; }
}

// Fixed-order sum of the per-jet losses into the loss slots
__global__ void __launch_bounds__(256) hungarian_mse_sum_kernel(int batch, float scale, const double* __restrict__ jet_loss,
                                                                float* __restrict__ terms) {
  gj_pdl_sync();
  __shared__ double red[8];
  double s = 0.0;
  for (int b = threadIdx.x; b < batch; b += 256) s += jet_loss[b];
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    terms[0] = (float)t; terms[1] = 0.f; terms[2] = (float)((double)scale * t);
  }
}

}  // namespace

void gj_set_error(const char* fmt, ...);

static size_t assignment_smem(int n) {
  return (size_t)(n + 1 + 32) * sizeof(double) + (size_t)(32 + 2 * (n + 1) + 2) * sizeof(int) + ((size_t)n * n + 8 * (size_t)n) * sizeof(float) + 16;
}

int gj_assignment_launch(int batch, int n, int dim, int lorentz, const float* p, const float* q, int* col_for_row, float* total_cost,
                         cudaStream_t stream) {
  if (batch < 0 || n < 1 || n > kAsgMaxParticles) {
    gj_set_error("gj_assignment: 1 <= particles per jet <= %d (cost matrix in shared memory), got %d", kAsgMaxParticles, n);
    return GJ_ERR_INVALID;
  }
  if (dim < 1 || dim > 4 || (lorentz && dim != 4)) { gj_set_error("gj_assignment: 1..4 components (4 for the Lorentz norm), got %d", dim); return GJ_ERR_INVALID; }
  if (batch == 0) return GJ_OK;
  const size_t smem = assignment_smem(n);
  cudaError_t ce = cudaSuccess;
  if (smem > 48 * 1024) ce = cudaFuncSetAttribute(assignment_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ce == cudaSuccess) {
    gj_launch(assignment_kernel, batch, gj_round_up(n, 32), smem, stream, n, dim, lorentz, p, q, col_for_row, total_cost);
    ce = cudaGetLastError();
  }
  if (ce != cudaSuccess) { gj_set_error("assignment launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_pair_min_dist_launch(int batch, int np_, int nq, int dim, int lorentz, const float* p, const float* q, float* min_pq,
                            float* min_qp, cudaStream_t stream) {
  if (batch < 0 || np_ < 1 || nq < 1 || (size_t)(np_ + nq) * 16 > 200 * 1024) {
    gj_set_error("gj_pair_min_dist: particle counts out of range"); return GJ_ERR_INVALID; }
  if (dim < 1 || dim > 4 || (lorentz && dim != 4)) { gj_set_error("gj_pair_min_dist: 1..4 components (4 for the Lorentz norm), got %d", dim); return GJ_ERR_INVALID; }
  if (batch == 0) return GJ_OK;
  const int nmax = np_ > nq ? np_ : nq;
  int threads = gj_round_up(nmax, 32); if (threads > 256) threads = 256;
  const size_t smem = (size_t)(np_ + nq) * 4 * sizeof(float);
  cudaError_t ce = cudaSuccess;
  if (smem > 48 * 1024) ce = cudaFuncSetAttribute(pair_min_dist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ce == cudaSuccess) {
    gj_launch(pair_min_dist_kernel, batch, threads, smem, stream, np_, nq, dim, lorentz, p, q, min_pq, min_qp);
    ce = cudaGetLastError();
  }
  if (ce != cudaSuccess) { gj_set_error("pair_min_dist launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_chamfer_launch(int batch, int np_, int nq, int dim, int norm, float wc, float wj, const float* p, const float* q,
                      float* jet_terms, float* terms, float* dp, cudaStream_t stream) {
  if (batch < 0 || np_ < 1 || nq < 1 || np_ > 1024 || nq > 1024) { gj_set_error("gj_chamfer_fwd_bwd: particle counts must be in [1,1024]"); return GJ_ERR_INVALID; }
  if (dim != 3 && dim != 4) { gj_set_error("gj_chamfer_fwd_bwd: p and q must be 3- or 4-vectors (got %d)", dim); return GJ_ERR_INVALID; }
  if (batch == 0) { cudaMemsetAsync(terms, 0, 3 * sizeof(float), stream); return GJ_OK; }
  // distance_sq.py:43-44 forces cartesian for 3-vectors inside pairwise_distance_sq ONLY; the jet term of chamfer_loss.py:40
  // calls normsq with the loss's norm choice directly, so 3-vectors with 'minkowskian' / 'polar' get p0^2 - p1^2 - p2^2 there
  const int mink = (dim != 3 && norm != 0) ? 1 : 0, mink_jet = norm != 0 ? 1 : 0;
  int nmax = np_ > nq ? np_ : nq;
  int threads = gj_round_up(nmax, 32);
  if (threads < 32) threads = 32;
  size_t smem = (size_t)(np_ + nq) * 4 * sizeof(float) + (size_t)(np_ + nq) * sizeof(int) + (64 + 8) * sizeof(float);
  gj_launch(chamfer_kernel, batch, threads, smem, stream, np_, nq, dim, mink, mink_jet, wc, wj, p, q, jet_terms, dp);
  gj_launch(chamfer_reduce_kernel, 1, 1024, 0, stream, batch, wc, wj, jet_terms, terms);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("chamfer launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

size_t gj_hmse_ws_bytes(int batch) { return batch > 0 ? (size_t)batch * sizeof(double) : 0; }

int gj_hmse_check(int batch, int n, int dim, int coords, size_t ws_bytes) {
  if (batch < 0 || n < 1 || n > kAsgMaxParticles) {
    gj_set_error("gj_hungarian_mse_loss: batch >= 0 and 1 <= particles per jet <= %d (cost matrix in shared memory), got %d and %d",
                 kAsgMaxParticles, batch, n);
    return GJ_ERR_INVALID;
  }
  if (dim != 3 && dim != 4) { gj_set_error("gj_hungarian_mse_loss: features per particle must be 3 or 4, got %d", dim); return GJ_ERR_INVALID; }
  if (coords < GJ_HMSE_ABS_CARTESIAN || coords > GJ_HMSE_REL_CARTESIAN) {
    gj_set_error("gj_hungarian_mse_loss: unknown coordinates %d", coords); return GJ_ERR_INVALID; }
  if (ws_bytes < gj_hmse_ws_bytes(batch)) {
    gj_set_error("gj_hungarian_mse_loss: workspace too small (%zu bytes, needs %zu)", ws_bytes, gj_hmse_ws_bytes(batch));
    return GJ_ERR_WORKSPACE;
  }
  return GJ_OK;
}

int gj_hmse_launch(int batch, int n, int dim, int coords, const float* p, const float* q, float scale, float* terms, float* dp,
                   int* col_for_row, void* ws, cudaStream_t stream) {
  double* jet_loss = (double*)ws;
  cudaError_t ce = cudaSuccess;
  if (batch > 0) {
    const size_t smem = assignment_smem(n);
    if (smem > 48 * 1024) ce = cudaFuncSetAttribute(hungarian_mse_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce == cudaSuccess)
      ce = gj_launch(hungarian_mse_loss_kernel, batch, gj_round_up(n, 32), smem, stream, n, dim, coords, scale, p, q, dp, col_for_row,
                     jet_loss);
  }
  if (ce == cudaSuccess) ce = gj_launch(hungarian_mse_sum_kernel, 1, 256, 0, stream, batch, scale, (const double*)jet_loss, terms);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("hungarian mse loss launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
