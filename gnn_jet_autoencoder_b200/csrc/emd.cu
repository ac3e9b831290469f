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
// hits the cap gets status 1.
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

__global__ void emd_kernel(int np_, int nq, float r, float beta, int norm, int periodic, const float* __restrict__ p,
                           const float* __restrict__ q, double* __restrict__ emd_out, double* __restrict__ flow_out,
                           float* __restrict__ dp_out, double* __restrict__ pot_out, int* __restrict__ status_out) {
  gj_pdl_sync();
  const int n1 = np_ + 1, n2 = nq + 1;                  // + the dummy row / column
  extern __shared__ double emd_smem[];
  double* flow = emd_smem;                              // [n1][n2]
  double* u = flow + (size_t)n1 * n2;                   // [n1] row potentials
  double* drow = u + n1;                                // [n1] Dijkstra distance of settled rows
  double* resa = drow + n1;                             // [n1] residual supply
  double* wa = resa + n1;                               // [n1] row weights
  double* v = wa + n1;                                  // [n2] column potentials
  double* resb = v + n2;                                // [n2] residual demand
  double* red_v = resb + n2;                            // [32]
  double* scal = red_v + 32;                            // [4]: W_p, W_q, sum_i a_i u_i
  float2* sp = reinterpret_cast<float2*>(scal + 4);     // [n1] (eta, phi) of p
  float2* sq = sp + n1;                                 // [n2] (eta, phi) of q
  int* rpred = reinterpret_cast<int*>(sq + n2);         // [n1] column a settled row was reached from (-1: source)
  int* rset = rpred + n1;                               // [n1] row settled
  int* rlist = rset + n1;                               // [n1] rows settled in the current step
  int* cpred = rlist + n1;                              // [n2] row a column was reached from
  int* red_j = cpred + n2;                              // [32]
  int* ctl = red_j + 32;                                // [2]: rows in rlist, status
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const float* pg = p + (size_t)b * np_ * 3;
  const float* qg = q + (size_t)b * nq * 3;

  for (int idx = tid; idx < n1 * n2; idx += blockDim.x) flow[idx] = 0.0;
  for (int i = tid; i < n1; i += blockDim.x) {
    const bool real = i < np_;
    sp[i] = real ? make_float2(__ldg(pg + i * 3 + 1), __ldg(pg + i * 3 + 2)) : make_float2(0.f, 0.f);
    wa[i] = real ? fmax((double)__ldg(pg + i * 3), 0.0) : 0.0;
    u[i] = 0.0;
  }
  for (int j = tid; j < n2; j += blockDim.x) {
    const bool real = j < nq;
    sq[j] = real ? make_float2(__ldg(qg + j * 3 + 1), __ldg(qg + j * 3 + 2)) : make_float2(0.f, 0.f);
    resb[j] = real ? fmax((double)__ldg(qg + j * 3), 0.0) : 0.0;
    v[j] = 0.0;
  }
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
    if (sink < 0) { if (tid == 0) ctl[1] = 2; break; }
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
      if (src < 0) ctl[1] = 2;
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
  if (tid == 0) {
    double t = 0.0;
    for (int w = 0; w < nwarps; ++w) t += red_v[w];
    emd_out[b] = t;
    if (status_out) status_out[b] = ctl[1];
  }
  if (flow_out)
    for (int idx = tid; idx < np_ * nq; idx += blockDim.x) {
      const int i = idx / nq, jq = idx - i * nq;
      flow_out[(size_t)b * np_ * nq + idx] = flow[(size_t)i * n2 + jq];
    }
  if (pot_out) {
    double* po = pot_out + (size_t)b * (n1 + n2);
    for (int i = tid; i < n1; i += blockDim.x) po[i] = u[i];
    if (has_col) po[n1 + j] = v[j];
  }
  if (dp_out && tid < np_) {
    // d/d(eta_i, phi_i) sum_j f_ij (theta_ij / R)^beta = sum_j f_ij beta c_ij / theta_ij^2 (deta, dphi), 0 at theta = 0
    const int i = tid;
    const float2 a = sp[i];
    double ge = 0.0, gp = 0.0;
    for (int jq = 0; jq < nq; ++jq) {
      const double f = flow[(size_t)i * n2 + jq];
      if (f > 0.0) {
        const float2 c = sq[jq];
        const float de = a.x - c.x, dph = emd_dphi(a.y - c.y, periodic), t2 = de * de + dph * dph;
        if (t2 > 0.f) {
          const double k = f * (double)beta * (double)emd_pair_cost(a, c, r, beta, periodic) / (double)t2;
          ge += k * de; gp += k * dph;
        }
      }
    }
    // d/da_i of the optimum is the row's dual minus that of the dummy whose weight a_i changes (+ the normalisation's chain rule)
    double gw = 0.0;
    if (wa[i] > 0.0) {
      if (norm) gw = (u[i] - scal[2]) / wp;
      else gw = wp <= wq ? u[i] - u[np_] : u[i] + v[nq];
    }
    float* o = dp_out + ((size_t)b * np_ + i) * 3;
    o[0] = (float)gw; o[1] = (float)ge; o[2] = (float)gp;
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
