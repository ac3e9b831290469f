// Node-level kernels of one message-passing step (fp32 SIMT, shared by both precision modes).
//
// Everything in reference models/graphnet.py:154-168 that is O(N) per jet -- as opposed to the O(N^2) edge MLP --
// runs here, over all B*N node rows at once (rows are independent), so that the edge kernels hold nothing but
// pair tiles:
//   node_pre_fwd   : P_i = Wa h_i + b0, Q_j = Wb h_j    (the factorised first edge layer, W0 [h_i|h_j|d] =
//                    Wa h_i + Wb h_j + wd d, column order of graphnet.py:220)
//   node_post_fwd  : h'_i = NodeNet([e_i | h_i])          (graphnet.py:243-246, 266-268)
//   node_post_bwd  : adjoint of node_post_fwd -> de, dh (node path), dV, dc
//   node_pre_bwd   : dh += Wa^T dP + Wb^T dQ ; dWa, dWb, db0
// A CTA stages R node rows at a time in shared memory and runs register-tiled small GEMMs on them; parameter
// gradients accumulate in shared memory across the CTA's row blocks and leave as one partial per CTA
// (deterministic fixed-order reduction afterwards).
#include "gj_common.cuh"

#define NK_THREADS 256

namespace {

// ---------------------------------------------------------------------------------------------------------
// register-tiled helpers on shared-memory operands (all strides multiples of 4 floats, (stride/4) odd)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float dot4(const float4& a, const float4& b, float acc) {
  acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc); acc = fmaf(a.z, b.z, acc); return fmaf(a.w, b.w, acc);
}

// out[r][o] = epi( bias[o] + sum_k X[r][k] W[o][k] ),  r < R (even), o < Op (mult of 4), k < Kp (mult of 4).
// EPI 0: identity; 1: leaky; 2: multiply by leaky'(aux[r][o]) (aux has stride os).
template <int EPI>
__device__ void nk_gemm_rows(const float* __restrict__ X, int xs, const float* __restrict__ W, int ws,
                             const float* __restrict__ bias, float* __restrict__ out, int os, const float* __restrict__ aux,
                             int R, int Op, int Kp, float alpha) {
  const int half = R >> 1;
  const int items = half * (Op >> 2);
  for (int item = threadIdx.x; item < items; item += NK_THREADS) {
    const int rp = item % half, oq = item / half;
    float acc[2][4];
#pragma unroll
    for (int q = 0; q < 4; ++q) { float b = bias ? bias[oq * 4 + q] : 0.f; acc[0][q] = b; acc[1][q] = b; }
    const float* x0 = X + rp * xs;
    const float* x1 = X + (rp + half) * xs;
    const float* w = W + (oq * 4) * ws;
    for (int k = 0; k < Kp; k += 4) {
      const float4 a0 = *reinterpret_cast<const float4*>(x0 + k);
      const float4 a1 = *reinterpret_cast<const float4*>(x1 + k);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 wv = *reinterpret_cast<const float4*>(w + q * ws + k);
        acc[0][q] = dot4(a0, wv, acc[0][q]);
        acc[1][q] = dot4(a1, wv, acc[1][q]);
      }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int r = rp + i * half;
      float4 o = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      if (EPI == 1) { o.x = gj_leaky(o.x, alpha); o.y = gj_leaky(o.y, alpha); o.z = gj_leaky(o.z, alpha); o.w = gj_leaky(o.w, alpha); }
      if (EPI == 2) {
        const float4 y = *reinterpret_cast<const float4*>(aux + r * os + oq * 4);
        o.x *= gj_slope(y.x, alpha); o.y *= gj_slope(y.y, alpha); o.z *= gj_slope(y.z, alpha); o.w *= gj_slope(y.w, alpha);
      }
      *reinterpret_cast<float4*>(out + r * os + oq * 4) = o;
    }
  }
}

// dW[o][k] += sum_r G[r][o] Y[r][k] (o < O, k < K, stored unpadded with row length K at dW), db[o] += sum_r G[r][o].
// An item (4 o x 4 k) is owned by 8 consecutive lanes that split the rows and combine by shuffles (fixed order).
__device__ void nk_wgrad(const float* __restrict__ G, int gs, const float* __restrict__ Y, int ys, float* __restrict__ dW,
                         float* __restrict__ db, int R, int O, int K) {
  const int Oq = (O + 3) >> 2, Kq = (K + 3) >> 2;
  const int items = Oq * Kq;
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  const int rounds = (items + (NK_THREADS / 8) - 1) / (NK_THREADS / 8);
  for (int it = 0; it < rounds; ++it) {
    const int item = it * (NK_THREADS / 8) + grp;
    const bool live = item < items;
    const int kq = live ? item % Kq : 0, oq = live ? item / Kq : 0;
    float acc[4][4];
    float bs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int a = 0; a < 4; ++a) { acc[a][0] = 0.f; acc[a][1] = 0.f; acc[a][2] = 0.f; acc[a][3] = 0.f; }
    if (live) {
      for (int r = sub; r < R; r += 8) {
        const float4 g = *reinterpret_cast<const float4*>(G + r * gs + oq * 4);
        const float4 y = *reinterpret_cast<const float4*>(Y + r * ys + kq * 4);
        const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          acc[a][0] = fmaf(gv[a], y.x, acc[a][0]); acc[a][1] = fmaf(gv[a], y.y, acc[a][1]);
          acc[a][2] = fmaf(gv[a], y.z, acc[a][2]); acc[a][3] = fmaf(gv[a], y.w, acc[a][3]);
          bs[a] += gv[a];
        }
      }
    }
#pragma unroll
    for (int s = 1; s < 8; s <<= 1) {
#pragma unroll
      for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] += __shfl_xor_sync(0xffffffffu, acc[a][b], s);
        bs[a] += __shfl_xor_sync(0xffffffffu, bs[a], s);
      }
    }
    if (live && sub == 0) {
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int o = oq * 4 + a;
        if (o < O) {
#pragma unroll
          for (int b = 0; b < 4; ++b) { const int k = kq * 4 + b; if (k < K) dW[o * K + k] += acc[a][b]; }
          if (kq == 0 && db) db[o] += bs[a];
        }
      }
    }
  }
}

__device__ __forceinline__ int rup4(int x) { return (x + 3) & ~3; }
__host__ __device__ __forceinline__ int nk_stride(int w) { return ((w + 7) & ~7) + 4; }   // (stride/4) odd

// ---------------------------------------------------------------------------------------------------------
// node_pre: P|Q projections and their adjoint
// ---------------------------------------------------------------------------------------------------------
struct PreArgs {
  int rows, H, ld, cols, E0, E0p, K0;   // K0 = 2H+1 (row length of edge_net[t][0].weight)
  int R, hs, ws, ps;                    // rows per block; smem strides of h rows, weight rows, PQ rows
  int o_w, o_b, o_h, o_pq, o_dpar, smem_floats;
};

// PQ[row][0..E0p) = Wa h + b0 ; PQ[row][E0p..2E0p) = Wb h
__global__ void __launch_bounds__(NK_THREADS) node_pre_fwd_kernel(const PreArgs A, const float* __restrict__ h,
                                                                   const float* __restrict__ w0, const float* __restrict__ b0,
                                                                   float* __restrict__ pq) {
  gj_pdl_sync();
  extern __shared__ float4 nk_smem_raw[];
  float* sm = reinterpret_cast<float*>(nk_smem_raw);
  float* W = sm + A.o_w;     // [2*E0p][ws]: rows 0..E0p-1 = Wa, E0p.. = Wb, zero padded
  float* bias = sm + A.o_b;  // [2*E0p]: b0 | 0
  const int Hp = rup4(A.H);
  for (int idx = threadIdx.x; idx < 2 * A.E0p * A.ws; idx += NK_THREADS) {
    const int o = idx / A.ws, k = idx - o * A.ws;
    const int c = o < A.E0p ? o : o - A.E0p;
    float v = 0.f;
    if (c < A.E0 && k < A.H) v = __ldg(w0 + c * A.K0 + (o < A.E0p ? k : A.H + k));
    W[idx] = v;
  }
  for (int o = threadIdx.x; o < 2 * A.E0p; o += NK_THREADS) bias[o] = (o < A.E0) ? __ldg(b0 + o) : 0.f;
  float* X = sm + A.o_h;
  float* O = sm + A.o_pq;
  const int width = 2 * A.E0p;
  for (int r0 = blockIdx.x * A.R; r0 < A.rows; r0 += gridDim.x * A.R) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < A.R * Hp; idx += NK_THREADS) {
      const int r = idx / Hp, k = idx - r * Hp;
      const int row = r0 + r;
      X[r * A.hs + k] = (row < A.rows && k < A.cols) ? __ldg(h + (size_t)row * A.ld + k) : 0.f;
    }
    __syncthreads();
    nk_gemm_rows<0>(X, A.hs, W, A.ws, bias, O, A.ps, nullptr, A.R, width, Hp, 0.f);
    __syncthreads();
    const int nvalid = min(A.R, A.rows - r0);
    const int w4 = width >> 2;
    for (int idx = threadIdx.x; idx < nvalid * w4; idx += NK_THREADS) {
      const int r = idx / w4, q = idx - r * w4;
      *reinterpret_cast<float4*>(pq + (size_t)(r0 + r) * width + q * 4) = *reinterpret_cast<const float4*>(O + r * A.ps + q * 4);
    }
  }
}

// dh[row][k] += sum_c dP[row][c] Wa[c][k] + dQ[row][c] Wb[c][k]   (k < cols)
// dW0[c][k] += sum_rows dP h ; dW0[c][H+k] += sum_rows dQ h ; db0[c] += sum_rows dP     (partial per CTA)
__global__ void __launch_bounds__(NK_THREADS) node_pre_bwd_kernel(const PreArgs A, const float* __restrict__ h,
                                                                   const float* __restrict__ w0, const float* __restrict__ dpq,
                                                                   float* __restrict__ dh, float* __restrict__ part) {
  gj_pdl_sync();
  extern __shared__ float4 nk_smem_raw[];
  float* sm = reinterpret_cast<float*>(nk_smem_raw);
  // Wt[k][c'] with c' over 2*E0p (dP | dQ channels): dh[r][k] = sum_c' dPQ[r][c'] Wt[k][c']
  float* Wt = sm + A.o_w;
  const int Hp = rup4(A.H), width = 2 * A.E0p;
  for (int idx = threadIdx.x; idx < Hp * A.ws; idx += NK_THREADS) {
    const int k = idx / A.ws, o = idx - k * A.ws;
    float v = 0.f;
    if (o < width && k < A.H) {
      const int c = o < A.E0p ? o : o - A.E0p;
      if (c < A.E0) v = __ldg(w0 + c * A.K0 + (o < A.E0p ? k : A.H + k));
    }
    Wt[idx] = v;
  }
  const int ndpar = A.E0 * 2 * A.H + A.E0;
  float* out = part + (size_t)blockIdx.x * ndpar;
  // [E0][2H] (Wa | Wb gradients, row length 2H) then [E0] bias gradient; wide layers accumulate in the CTA's global partial
  float* dpar = A.o_dpar >= 0 ? sm + A.o_dpar : out;
  for (int idx = threadIdx.x; idx < ndpar; idx += NK_THREADS) dpar[idx] = 0.f;
  float* X = sm + A.o_h;    // h rows [R][hs]
  float* G = sm + A.o_pq;   // dPQ rows [R][ps]
  float* D = X;             // dh rows reuse... (kept separate below)
  (void)D;
  float* Dh = sm + A.o_b;   // [R][hs] output staging
  for (int r0 = blockIdx.x * A.R; r0 < A.rows; r0 += gridDim.x * A.R) {
    __syncthreads();
    const int nvalid = min(A.R, A.rows - r0);
    for (int idx = threadIdx.x; idx < A.R * Hp; idx += NK_THREADS) {
      const int r = idx / Hp, k = idx - r * Hp;
      const int row = r0 + r;
      X[r * A.hs + k] = (row < A.rows && k < A.cols) ? __ldg(h + (size_t)row * A.ld + k) : 0.f;
    }
    const int w4 = width >> 2;
    for (int idx = threadIdx.x; idx < A.R * w4; idx += NK_THREADS) {
      const int r = idx / w4, q = idx - r * w4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nvalid) v = *reinterpret_cast<const float4*>(dpq + (size_t)(r0 + r) * width + q * 4);
      *reinterpret_cast<float4*>(G + r * A.ps + q * 4) = v;
    }
    __syncthreads();
    nk_gemm_rows<0>(G, A.ps, Wt, A.ws, nullptr, Dh, A.hs, nullptr, A.R, Hp, width, 0.f);
    // dWa: G[:, 0:E0p] x h ; dWb: G[:, E0p:] x h
    nk_wgrad(G, A.ps, X, A.hs, dpar, dpar + A.E0 * 2 * A.H, A.R, A.E0, A.H);          // placeholder layout fixed below
    __syncthreads();
    nk_wgrad(G + A.E0p, A.ps, X, A.hs, dpar + A.E0 * A.H, nullptr, A.R, A.E0, A.H);
    __syncthreads();
    for (int idx = threadIdx.x; idx < nvalid * A.cols; idx += NK_THREADS) {
      const int r = idx / A.cols, k = idx - r * A.cols;
      float* p = dh + (size_t)(r0 + r) * A.ld + k;
      *p += Dh[r * A.hs + k];
    }
  }
  __syncthreads();
  // partial layout: [Wa grads E0*H][Wb grads E0*H][b0 grads E0]
  if (dpar != out)
    for (int idx = threadIdx.x; idx < ndpar; idx += NK_THREADS) out[idx] = dpar[idx];
}

// ---------------------------------------------------------------------------------------------------------
// node_post: the node MLP and its adjoint
// ---------------------------------------------------------------------------------------------------------
struct PostArgs {
  int rows, H, ld, cols, EL, Ln;
  int O[GJ_MAX_LAYERS], I[GJ_MAX_LAYERS], pV[GJ_MAX_LAYERS], pc[GJ_MAX_LAYERS];   // offsets in the packed params
  int p_first;                 // offset of the first node parameter in the packed block
  int n_node_params;
  float alpha;
  int R, S;                    // rows per block, activation row stride
  int o_V[GJ_MAX_LAYERS], vs[GJ_MAX_LAYERS], o_c[GJ_MAX_LAYERS];     // weights [Op][vs]
  int o_Vt[GJ_MAX_LAYERS], vts[GJ_MAX_LAYERS];                        // transposed weights [Ip][vts] (bwd only)
  int o_Y[GJ_MAX_LAYERS + 1], o_g0, o_g1, o_dpar, smem_floats;
  int wide;                    // backward of wide layers: ONE weight area, (re)staged before every GEMM; gradients in global memory
};

// wide mode: layer m's weights (or their transpose) into the shared weight area, biases stay resident
__device__ void post_stage_one(const PostArgs& A, const float* __restrict__ params, float* sm, int m, bool transposed) {
  const int O = A.O[m], I = A.I[m], Op = rup4(O), Ip = rup4(I);
  if (!transposed) {
    for (int idx = threadIdx.x; idx < Op * A.vs[m]; idx += NK_THREADS) {
      const int o = idx / A.vs[m], k = idx - o * A.vs[m];
      sm[A.o_V[m] + idx] = (o < O && k < I) ? __ldg(params + A.pV[m] + o * I + k) : 0.f;
    }
  } else {
    for (int idx = threadIdx.x; idx < Ip * A.vts[m]; idx += NK_THREADS) {
      const int k = idx / A.vts[m], o = idx - k * A.vts[m];
      sm[A.o_Vt[m] + idx] = (o < O && k < I) ? __ldg(params + A.pV[m] + o * I + k) : 0.f;
    }
  }
}

__device__ void post_stage_weights(const PostArgs& A, const float* __restrict__ params, float* sm, bool transposed) {
  for (int m = 0; m < A.Ln; ++m) {
    const int O = A.O[m], I = A.I[m], Op = rup4(O), Ip = rup4(I);
    for (int idx = threadIdx.x; idx < Op * A.vs[m]; idx += NK_THREADS) {
      const int o = idx / A.vs[m], k = idx - o * A.vs[m];
      sm[A.o_V[m] + idx] = (o < O && k < I) ? __ldg(params + A.pV[m] + o * I + k) : 0.f;
    }
    for (int o = threadIdx.x; o < Op; o += NK_THREADS) sm[A.o_c[m] + o] = o < O ? __ldg(params + A.pc[m] + o) : 0.f;
    if (transposed) {
      for (int idx = threadIdx.x; idx < Ip * A.vts[m]; idx += NK_THREADS) {
        const int k = idx / A.vts[m], o = idx - k * A.vts[m];
        sm[A.o_Vt[m] + idx] = (o < O && k < I) ? __ldg(params + A.pV[m] + o * I + k) : 0.f;
      }
    }
  }
}

// Y0[r] = [e | h | 0-pad]
__device__ void post_load_rows(const PostArgs& A, const float* __restrict__ e, const float* __restrict__ h, float* Y0, int r0) {
  const int I0 = A.EL + A.H, I0p = rup4(I0);
  for (int idx = threadIdx.x; idx < A.R * I0p; idx += NK_THREADS) {
    const int r = idx / I0p, k = idx - r * I0p;
    const int row = r0 + r;
    float v = 0.f;
    if (row < A.rows) {
      if (k < A.EL) v = __ldg(e + (size_t)row * A.EL + k);
      else if (k - A.EL < A.cols) v = __ldg(h + (size_t)row * A.ld + (k - A.EL));
    }
    Y0[r * A.S + k] = v;
  }
}

__global__ void __launch_bounds__(NK_THREADS) node_post_fwd_kernel(const PostArgs A, const float* __restrict__ e,
                                                                    const float* __restrict__ h, const float* __restrict__ params,
                                                                    float* __restrict__ h_out) {
  gj_pdl_sync();
  extern __shared__ float4 nk_smem_raw[];
  float* sm = reinterpret_cast<float*>(nk_smem_raw);
  post_stage_weights(A, params, sm, false);
  const int Hout = A.O[A.Ln - 1];
  for (int r0 = blockIdx.x * A.R; r0 < A.rows; r0 += gridDim.x * A.R) {
    __syncthreads();
    post_load_rows(A, e, h, sm + A.o_Y[0], r0);
    __syncthreads();
    for (int m = 0; m < A.Ln; ++m) {
      nk_gemm_rows<1>(sm + A.o_Y[m & 1], A.S, sm + A.o_V[m], A.vs[m], sm + A.o_c[m], sm + A.o_Y[(m + 1) & 1], A.S, nullptr, A.R,
                      rup4(A.O[m]), rup4(A.I[m]), A.alpha);
      __syncthreads();
    }
    const float* Y = sm + A.o_Y[A.Ln & 1];
    const int nvalid = min(A.R, A.rows - r0);
    for (int idx = threadIdx.x; idx < nvalid * Hout; idx += NK_THREADS) {
      const int r = idx / Hout, o = idx - r * Hout;
      h_out[(size_t)(r0 + r) * Hout + o] = Y[r * A.S + o];
    }
  }
}

// in : e, h, dh_out ; out: de (rows, EL), dh (rows, ld; first `cols` columns OVERWRITTEN with the node-path gradient),
//      per-CTA partial of the node parameters (packed order, n_node_params floats).
__global__ void __launch_bounds__(NK_THREADS) node_post_bwd_kernel(const PostArgs A, const float* __restrict__ e,
                                                                    const float* __restrict__ h, const float* __restrict__ params,
                                                                    const float* __restrict__ dh_out, float* __restrict__ de,
                                                                    float* __restrict__ dh, float* __restrict__ part) {
  gj_pdl_sync();
  extern __shared__ float4 nk_smem_raw[];
  float* sm = reinterpret_cast<float*>(nk_smem_raw);
  if (!A.wide) post_stage_weights(A, params, sm, true);
  else
    for (int m = 0; m < A.Ln; ++m)
      for (int o = threadIdx.x; o < rup4(A.O[m]); o += NK_THREADS) sm[A.o_c[m] + o] = o < A.O[m] ? __ldg(params + A.pc[m] + o) : 0.f;
  float* out = part + (size_t)blockIdx.x * A.n_node_params;
  float* dpar = A.o_dpar >= 0 ? sm + A.o_dpar : out;
  for (int idx = threadIdx.x; idx < A.n_node_params; idx += NK_THREADS) dpar[idx] = 0.f;
  const int Hout = A.O[A.Ln - 1], Houtp = rup4(Hout);
  for (int r0 = blockIdx.x * A.R; r0 < A.rows; r0 += gridDim.x * A.R) {
    __syncthreads();
    const int nvalid = min(A.R, A.rows - r0);
    post_load_rows(A, e, h, sm + A.o_Y[0], r0);
    __syncthreads();
    for (int m = 0; m < A.Ln; ++m) {
      if (A.wide) { post_stage_one(A, params, sm, m, false); __syncthreads(); }
      nk_gemm_rows<1>(sm + A.o_Y[m], A.S, sm + A.o_V[m], A.vs[m], sm + A.o_c[m], sm + A.o_Y[m + 1], A.S, nullptr, A.R,
                      rup4(A.O[m]), rup4(A.I[m]), A.alpha);
      __syncthreads();
    }
    float* g = sm + A.o_g0;
    float* gp = sm + A.o_g1;
    {  // gz = dh_out * leaky'(y_last); rows beyond the batch and padded columns are zero
      const float* Yl = sm + A.o_Y[A.Ln];
      for (int idx = threadIdx.x; idx < A.R * Houtp; idx += NK_THREADS) {
        const int r = idx / Houtp, o = idx - r * Houtp;
        float v = 0.f;
        if (r < nvalid && o < Hout) v = __ldg(dh_out + (size_t)(r0 + r) * Hout + o) * gj_slope(Yl[r * A.S + o], A.alpha);
        g[r * A.S + o] = v;
      }
    }
    __syncthreads();
    for (int m = A.Ln - 1; m >= 0; --m) {
      const int O = A.O[m], I = A.I[m];
      nk_wgrad(g, A.S, sm + A.o_Y[m], A.S, dpar + (A.pV[m] - A.p_first), dpar + (A.pc[m] - A.p_first), A.R, O, I);
      if (A.wide) { post_stage_one(A, params, sm, m, true); __syncthreads(); }
      if (m > 0) nk_gemm_rows<2>(g, A.S, sm + A.o_Vt[m], A.vts[m], nullptr, gp, A.S, sm + A.o_Y[m], A.R, rup4(I), rup4(O), A.alpha);
      else       nk_gemm_rows<0>(g, A.S, sm + A.o_Vt[m], A.vts[m], nullptr, gp, A.S, nullptr, A.R, rup4(I), rup4(O), A.alpha);
      __syncthreads();
      float* t = g; g = gp; gp = t;
    }
    // g = d[e | h]
    for (int idx = threadIdx.x; idx < nvalid * A.EL; idx += NK_THREADS) {
      const int r = idx / A.EL, k = idx - r * A.EL;
      de[(size_t)(r0 + r) * A.EL + k] = g[r * A.S + k];
    }
    for (int idx = threadIdx.x; idx < nvalid * A.cols; idx += NK_THREADS) {
      const int r = idx / A.cols, k = idx - r * A.cols;
      dh[(size_t)(r0 + r) * A.ld + k] = g[r * A.S + A.EL + k];
    }
  }
  __syncthreads();
  if (dpar != out)
    for (int idx = threadIdx.x; idx < A.n_node_params; idx += NK_THREADS) out[idx] = dpar[idx];
}

// ---------------------------------------------------------------------------------------------------------
// thread-per-row kernels for the usual small widths (compile-time sizes: every loop unrolls, activations live in
// registers, weights are read as warp-broadcast 16-byte shared-memory loads -> FFMA bound)
// ---------------------------------------------------------------------------------------------------------
#define NF_THREADS 128
// tile staging with asynchronous 4-byte copies: a load -> store loop would wait for every load in turn
__device__ __forceinline__ void nf_cp_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void nf_cp_async_wait() {
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}
#define NF_BWD_CTAS_PER_SM 4      // adjoint kernels: CTAs per SM the grid is sized for (one parameter-gradient partial per CTA)
// y[o] = bias[o] + sum_k W[o][k] x[k]  for o in [o0, o0 + 4): W rows are KP floats long (zero padded), in shared memory
template <int KP>
__device__ __forceinline__ float4 nf_dot4(const float (&x)[KP], const float* __restrict__ W, const float* __restrict__ bias, int o0) {
  float acc[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    acc[q] = bias[o0 + q];
    const float4* w = reinterpret_cast<const float4*>(W + (o0 + q) * KP);
#pragma unroll
    for (int k = 0; k < KP / 4; ++k) { const float4 v = w[k]; acc[q] = dot4(make_float4(x[4 * k], x[4 * k + 1], x[4 * k + 2], x[4 * k + 3]), v, acc[q]); }
  }
  return make_float4(acc[0], acc[1], acc[2], acc[3]);
}

// Global traffic goes through shared-memory tiles of NF_THREADS rows so that it is coalesced (a thread reading / writing
// its own row straight from HBM touches 32 sectors per instruction); tile rows have a stride of 4 * odd floats, so the
// per-thread 16-byte accesses are conflict free.
template <int KP>
__device__ __forceinline__ float4 nf_dot4_nobias(const float (&x)[KP], const float* __restrict__ W, int o0) {
  float acc[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    acc[q] = 0.f;
    const float4* w = reinterpret_cast<const float4*>(W + (o0 + q) * KP);
#pragma unroll
    for (int k = 0; k < KP / 4; ++k) { const float4 v = w[k]; acc[q] = dot4(make_float4(x[4 * k], x[4 * k + 1], x[4 * k + 2], x[4 * k + 3]), v, acc[q]); }
  }
  return make_float4(acc[0], acc[1], acc[2], acc[3]);
}

// ---------------------------------------------------------------------------------------------------------
// Warp-autonomous forward kernels (projections and node MLP).  A CTA-wide tile loop would run one serial chain per 128-row
// tile -- stage weights, stage the tile, compute, store, with CTA-wide barriers in between -- on 592-960 CTAs, each of which
// re-stages the weights: 3-6x the HBM / FFMA floor.  Here a CTA of 8 warps stages the weights ONCE and every warp then walks
// its own 32-row tiles with no CTA-wide synchronisation: the next tile's rows are fetched (cp.async, 16-byte pieces where the
// layout allows) into the warp's staging rows as soon as every lane holds its row in registers, so the fetch runs under the
// ~2000 FFMA / LDS of the current tile; outputs leave as 16-byte coalesced stores (a tile's output rows are one contiguous
// block).  Tiles are dealt round-robin to CTAs first, then to the warps of a CTA, so every SM gets the same number of tiles
// (+-1).
// ---------------------------------------------------------------------------------------------------------
#define NW_WARPS 8
__device__ __forceinline__ void nf_cp_async16(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void nf_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void nf_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// rows [r0, r0 + nrows) x columns [0, cols) of a row-major matrix (row stride ld) -> dst[r][c0 + k] (row stride XS), lane-strided
template <int XS>
__device__ __forceinline__ void nw_stage_rows(float* dst, int c0, const float* __restrict__ src, int ld, int cols, size_t r0, int nrows,
                                              bool vec, int lane) {
  if (vec) {      // 16-byte pieces: cols, ld multiples of 4 and a 16-byte aligned base
    const int c4 = cols >> 2;
    for (int idx = lane; idx < nrows * c4; idx += 32) {
      const int r = idx / c4, k = idx - r * c4;
      nf_cp_async16(dst + r * XS + c0 + 4 * k, src + (r0 + r) * (size_t)ld + 4 * k);
    }
  } else {
    for (int idx = lane; idx < nrows * cols; idx += 32) {
      const int r = idx / cols, k = idx - r * cols;
      nf_cp_async4(dst + r * XS + c0 + k, src + (r0 + r) * (size_t)ld + k);
    }
  }
}
// a warp's [nrows][O] output rows (shared memory, row stride OS) -> out[(r0 + r) * ostride + o0 ..], coalesced
template <int OS>
__device__ __forceinline__ void nw_store_rows(float* __restrict__ out, int ostride, int o0, int O, const float* sO, size_t r0, int nrows,
                                              bool vec, int lane) {
  if (vec) {
    const int o4 = O >> 2;
    for (int idx = lane; idx < nrows * o4; idx += 32) {
      const int r = idx / o4, q = idx - r * o4;
      *reinterpret_cast<float4*>(out + (r0 + r) * (size_t)ostride + o0 + 4 * q) = *reinterpret_cast<const float4*>(sO + r * OS + 4 * q);
    }
  } else {
    for (int idx = lane; idx < nrows * O; idx += 32) {
      const int r = idx / O, o = idx - r * O;
      out[(r0 + r) * (size_t)ostride + o0 + o] = sO[r * OS + o];
    }
  }
}
__device__ __forceinline__ bool nw_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <int KP>
struct NwPreSmem {
  static constexpr int XS = KP + 4, OS = 36;
  static constexpr int o_bias = 64 * KP, o_warp = o_bias + 64, warp_floats = 32 * XS + 32 * OS;
  static constexpr int bytes = (o_warp + NW_WARPS * warp_floats) * 4;
};

// PQ[row][0..32) = Wa h + b0 ; PQ[row][32..64) = Wb h      (E0 = 32; KP = columns of h present in memory, padded to 4)
template <int KP>
__global__ void __launch_bounds__(NW_WARPS * 32, 2) node_pre_fwd_warp_kernel(int rows, int H, int cols, int ld, int K0,
                                                                            const float* __restrict__ h, const float* __restrict__ w0,
                                                                            const float* __restrict__ b0, float* __restrict__ pq) {
  gj_pdl_sync();
  using S = NwPreSmem<KP>;
  constexpr int XS = S::XS, OS = S::OS;
  extern __shared__ __align__(16) float nw_smem[];
  float* W = nw_smem;
  float* bias = nw_smem + S::o_bias;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* sX = nw_smem + S::o_warp + warp * S::warp_floats;      // [32][XS]
  float* sO = sX + 32 * XS;                                     // [32][OS]
  for (int idx = threadIdx.x; idx < 64 * KP; idx += NW_WARPS * 32) {
    const int o = idx / KP, k = idx - o * KP;
    if (k < cols) nf_cp_async4(W + idx, w0 + (o & 31) * K0 + (o < 32 ? k : H + k));
    else W[idx] = 0.f;
  }
  if (threadIdx.x < 64) bias[threadIdx.x] = threadIdx.x < 32 ? __ldg(b0 + threadIdx.x) : 0.f;
  for (int idx = lane; idx < 32 * (KP - cols); idx += 32) {      // the padding columns of the staging rows stay zero
    const int r = idx / (KP - cols), k = idx - r * (KP - cols);
    sX[r * XS + cols + k] = 0.f;
  }
  const int T = (rows + 31) >> 5, G = gridDim.x;
  const bool vin = (cols & 3) == 0 && (ld & 3) == 0 && nw_aligned16(h);
  int t = blockIdx.x + G * warp;
  if (t < T) nw_stage_rows<XS>(sX, 0, h, ld, cols, (size_t)t * 32, min(32, rows - t * 32), vin, lane);
  nf_cp_async_commit();
  nf_cp_async_wait_all();
  __syncthreads();      // weights, biases (and this warp's first tile) have landed
  while (t < T) {
    const size_t r0 = (size_t)t * 32;
    const int nrows = min(32, rows - t * 32);
    float x[KP];
#pragma unroll
    for (int k = 0; k < KP; k += 4) {
      const float4 v = *reinterpret_cast<const float4*>(sX + lane * XS + k);
      x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
    }
    __syncwarp();
    const int tn = t + G * NW_WARPS;      // every lane holds its row: fetch the next tile under this tile's arithmetic
    if (tn < T) nw_stage_rows<XS>(sX, 0, h, ld, cols, (size_t)tn * 32, min(32, rows - tn * 32), vin, lane);
    nf_cp_async_commit();
#pragma unroll
    for (int half = 0; half < 2; ++half) {      // P then Q
#pragma unroll
      for (int o0 = 0; o0 < 32; o0 += 4)
        *reinterpret_cast<float4*>(sO + lane * OS + o0) = nf_dot4<KP>(x, W, bias, 32 * half + o0);
      __syncwarp();
      nw_store_rows<OS>(pq, 64, 32 * half, 32, sO, r0, nrows, true, lane);
      __syncwarp();
    }
    nf_cp_async_wait_all();
    __syncwarp();
    t = tn;
  }
}

template <int I0P, int O0P, int O1P>
struct NwPostSmem {
  static constexpr int XS = 4 * ((I0P / 4) | 1), OS = 4 * ((O1P / 4) | 1);
  static constexpr int o_v1 = O0P * I0P, o_c0 = o_v1 + O1P * O0P, o_c1 = o_c0 + O0P, o_warp = (o_c1 + O1P + 3) & ~3;
  static constexpr int warp_floats = 32 * XS + 32 * OS;
  static constexpr int bytes = (o_warp + NW_WARPS * warp_floats) * 4;
};

// h' = leaky(V1 leaky(V0 [e | h] + c0) + c1)      (two node layers; I0P, O0P, O1P = widths padded to 4; EL = 16)
template <int I0P, int O0P, int O1P>
__global__ void __launch_bounds__(NW_WARPS * 32, 2) node_post_fwd_warp_kernel(int rows, int EL, int cols, int ld, int I0, int O0, int O1,
                                                                             float alpha, const float* __restrict__ e,
                                                                             const float* __restrict__ h, const float* __restrict__ V0,
                                                                             const float* __restrict__ c0, const float* __restrict__ V1,
                                                                             const float* __restrict__ c1, float* __restrict__ h_out) {
  gj_pdl_sync();
  using S = NwPostSmem<I0P, O0P, O1P>;
  constexpr int XS = S::XS, OS = S::OS, HP = I0P - 16;
  extern __shared__ __align__(16) float nw_smem[];
  float* sV0 = nw_smem;
  float* sV1 = nw_smem + S::o_v1;
  float* sc0 = nw_smem + S::o_c0;
  float* sc1 = nw_smem + S::o_c1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* sX = nw_smem + S::o_warp + warp * S::warp_floats;      // [32][XS]: e (16 columns) | h
  float* sO = sX + 32 * XS;                                     // [32][OS]
  for (int idx = threadIdx.x; idx < O0P * I0P; idx += NW_WARPS * 32) {
    const int o = idx / I0P, k = idx - o * I0P;
    if (o < O0 && k < I0) nf_cp_async4(sV0 + idx, V0 + o * I0 + k);
    else sV0[idx] = 0.f;
  }
  for (int idx = threadIdx.x; idx < O1P * O0P; idx += NW_WARPS * 32) {
    const int o = idx / O0P, k = idx - o * O0P;
    if (o < O1 && k < O0) nf_cp_async4(sV1 + idx, V1 + o * O0 + k);
    else sV1[idx] = 0.f;
  }
  for (int o = threadIdx.x; o < O0P; o += NW_WARPS * 32) sc0[o] = o < O0 ? __ldg(c0 + o) : 0.f;
  for (int o = threadIdx.x; o < O1P; o += NW_WARPS * 32) sc1[o] = o < O1 ? __ldg(c1 + o) : 0.f;
  for (int idx = lane; idx < 32 * (HP - cols); idx += 32) {      // the padding columns of the staging rows stay zero
    const int r = idx / (HP - cols), k = idx - r * (HP - cols);
    sX[r * XS + 16 + cols + k] = 0.f;
  }
  const int T = (rows + 31) >> 5, G = gridDim.x;
  const bool ve = nw_aligned16(e);      // EL == 16
  const bool vh = (cols & 3) == 0 && (ld & 3) == 0 && nw_aligned16(h);
  const bool vo = (O1 & 3) == 0 && nw_aligned16(h_out);
  auto stage = [&](int tt) {
    const size_t r0 = (size_t)tt * 32;
    const int nrows = min(32, rows - tt * 32);
    nw_stage_rows<XS>(sX, 0, e, EL, 16, r0, nrows, ve, lane);
    nw_stage_rows<XS>(sX, 16, h, ld, cols, r0, nrows, vh, lane);
  };
  int t = blockIdx.x + G * warp;
  if (t < T) stage(t);
  nf_cp_async_commit();
  nf_cp_async_wait_all();
  __syncthreads();      // weights, biases (and this warp's first tile) have landed
  while (t < T) {
    const size_t r0 = (size_t)t * 32;
    const int nrows = min(32, rows - t * 32);
    float x[I0P];
#pragma unroll
    for (int k = 0; k < I0P; k += 4) {
      const float4 v = *reinterpret_cast<const float4*>(sX + lane * XS + k);
      x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
    }
    __syncwarp();
    const int tn = t + G * NW_WARPS;      // every lane holds its row: fetch the next tile under this tile's arithmetic
    if (tn < T) stage(tn);
    nf_cp_async_commit();
    float y0[O0P];
#pragma unroll
    for (int o0 = 0; o0 < O0P; o0 += 4) {
      const float4 v = nf_dot4<I0P>(x, sV0, sc0, o0);
      y0[o0] = fmaxf(v.x, alpha * v.x); y0[o0 + 1] = fmaxf(v.y, alpha * v.y); y0[o0 + 2] = fmaxf(v.z, alpha * v.z); y0[o0 + 3] = fmaxf(v.w, alpha * v.w);
    }
#pragma unroll
    for (int o0 = 0; o0 < O1P; o0 += 4) {
      const float4 v = nf_dot4<O0P>(y0, sV1, sc1, o0);
      *reinterpret_cast<float4*>(sO + lane * OS + o0) =
          make_float4(fmaxf(v.x, alpha * v.x), fmaxf(v.y, alpha * v.y), fmaxf(v.z, alpha * v.z), fmaxf(v.w, alpha * v.w));
    }
    __syncwarp();
    nw_store_rows<OS>(h_out, O1, 0, O1, sO, r0, nrows, vo, lane);
    nf_cp_async_wait_all();
    __syncwarp();
    t = tn;
  }
}

// ---- thread-per-row adjoints: dgrad per thread from registers, wgrad as a second pass over the CTA's row tile ----
// Weight gradients: the O x KP outputs are dealt out in units of 4 consecutive k; a thread keeps its units in registers
// across all tiles of the CTA and sweeps the tile's rows, reading g[r][o] and the 16 bytes y[r][4 k4 ..] from the tiles.
template <int UNITS>
struct NfAcc { float4 v[UNITS]; float b[UNITS]; };

// acc[u] += sum_r G[r][o_u] * Y[r][4 k4_u ..] ; bacc[u] += sum_r G[r][o_u] (used only where k4_u == 0)
template <int KP4, int NOUT, int UNITS>
__device__ __forceinline__ void nf_wgrad_tile(NfAcc<UNITS>& acc, const float* __restrict__ G, int gs, const float* __restrict__ Y, int ys, int nrows) {
  int o[UNITS], k4[UNITS];
#pragma unroll
  for (int u = 0; u < UNITS; ++u) { const int unit = threadIdx.x + u * NF_THREADS; o[u] = unit / KP4; k4[u] = unit - o[u] * KP4; }
  for (int r = 0; r < nrows; ++r) {
#pragma unroll
    for (int u = 0; u < UNITS; ++u) {
      if (o[u] < NOUT) {
        const float g = G[r * gs + o[u]];
        const float4 y = *reinterpret_cast<const float4*>(Y + r * ys + 4 * k4[u]);
        acc.v[u].x = fmaf(g, y.x, acc.v[u].x); acc.v[u].y = fmaf(g, y.y, acc.v[u].y);
        acc.v[u].z = fmaf(g, y.z, acc.v[u].z); acc.v[u].w = fmaf(g, y.w, acc.v[u].w);
        acc.b[u] += g;
      }
    }
  }
}
// per-CTA partial: dW[o][k] (row length K, unpadded) and db[o]
template <int KP4, int NOUT, int UNITS>
__device__ __forceinline__ void nf_wgrad_store(const NfAcc<UNITS>& acc, float* __restrict__ dW, float* __restrict__ db, int O, int K) {
#pragma unroll
  for (int u = 0; u < UNITS; ++u) {
    const int unit = threadIdx.x + u * NF_THREADS, o = unit / KP4, k4 = unit - o * KP4;
    if (o < O && o < NOUT) {
      const float v[4] = {acc.v[u].x, acc.v[u].y, acc.v[u].z, acc.v[u].w};
#pragma unroll
      for (int q = 0; q < 4; ++q) if (4 * k4 + q < K) dW[o * K + 4 * k4 + q] = v[q];
      if (k4 == 0 && db) db[o] = acc.b[u];
    }
  }
}

// adjoint of the two-layer node MLP: de (rows, 16), dh (rows, ld; first `cols` columns OVERWRITTEN), per-CTA partial of the
// node parameters in packed order [V0 | c0 | V1 | c1]
template <int I0P, int O0P, int O1P>
__global__ void __launch_bounds__(NF_THREADS) node_post_bwd_fast_kernel(int rows, int EL, int cols, int ld, int I0, int O0, int O1, float alpha,
                                                                        int n_node_params, const float* __restrict__ e,
                                                                        const float* __restrict__ h, const float* __restrict__ V0,
                                                                        const float* __restrict__ c0, const float* __restrict__ V1,
                                                                        const float* __restrict__ c1, const float* __restrict__ dh_out,
                                                                        float* __restrict__ de, float* __restrict__ dh, float* __restrict__ part) {
  gj_pdl_sync();
  constexpr int XS = 4 * ((I0P / 4) | 1), YS = 4 * ((O0P / 4) | 1), G1S = 4 * ((O1P / 4) | 1);
  constexpr int U0 = (O0P * (I0P / 4) + NF_THREADS - 1) / NF_THREADS, U1 = (O1P * (O0P / 4) + NF_THREADS - 1) / NF_THREADS;
  extern __shared__ float4 nk_smem_raw[];
  float* sm = reinterpret_cast<float*>(nk_smem_raw);
  float* sV0 = sm;                         // [O0P][I0P]
  float* sV1 = sV0 + O0P * I0P;            // [O1P][O0P]
  float* sV0t = sV1 + O1P * O0P;           // [I0P][O0P]
  float* sV1t = sV0t + I0P * O0P;          // [O0P][O1P]
  float* sc0 = sV1t + O0P * O1P;           // [O0P]
  float* sc1 = sc0 + O0P;                  // [O1P]
  float* sX = sc1 + O1P;                   // [NF_THREADS][XS]   x = [e | h]
  float* sY0 = sX + NF_THREADS * XS;       // [NF_THREADS][YS]   y0, then (second use) g0
  float* sG1 = sY0 + NF_THREADS * YS;      // [NF_THREADS][G1S]  dh_out, then g1
  float* sG0 = sG1 + NF_THREADS * G1S;     // [NF_THREADS][YS]   g0
  for (int idx = threadIdx.x; idx < O0P * I0P; idx += NF_THREADS) {
    const int o = idx / I0P, k = idx - o * I0P;
    const float v = (o < O0 && k < I0) ? __ldg(V0 + o * I0 + k) : 0.f;
    sV0[idx] = v; sV0t[k * O0P + o] = v;
  }
  for (int idx = threadIdx.x; idx < O1P * O0P; idx += NF_THREADS) {
    const int o = idx / O0P, k = idx - o * O0P;
    const float v = (o < O1 && k < O0) ? __ldg(V1 + o * O0 + k) : 0.f;
    sV1[idx] = v; sV1t[k * O1P + o] = v;
  }
  for (int o = threadIdx.x; o < O0P; o += NF_THREADS) sc0[o] = o < O0 ? __ldg(c0 + o) : 0.f;
  for (int o = threadIdx.x; o < O1P; o += NF_THREADS) sc1[o] = o < O1 ? __ldg(c1 + o) : 0.f;
  NfAcc<U0> acc0;
  NfAcc<U1> acc1;
#pragma unroll
  for (int u = 0; u < U0; ++u) { acc0.v[u] = make_float4(0.f, 0.f, 0.f, 0.f); acc0.b[u] = 0.f; }
#pragma unroll
  for (int u = 0; u < U1; ++u) { acc1.v[u] = make_float4(0.f, 0.f, 0.f, 0.f); acc1.b[u] = 0.f; }
  for (int row0 = blockIdx.x * NF_THREADS; row0 < rows; row0 += gridDim.x * NF_THREADS) {
    const int nrows = min(NF_THREADS, rows - row0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < nrows * 16; idx += NF_THREADS) {
      const int r = idx >> 4, k = idx & 15;
      nf_cp_async4(sX + r * XS + k, e + (size_t)(row0 + r) * EL + k);
    }
    for (int idx = threadIdx.x; idx < nrows * (I0P - 16); idx += NF_THREADS) {
      const int r = idx / (I0P - 16), k = idx - r * (I0P - 16);
      if (k < cols) nf_cp_async4(sX + r * XS + 16 + k, h + (size_t)(row0 + r) * ld + k);
      else sX[r * XS + 16 + k] = 0.f;
    }
    for (int idx = threadIdx.x; idx < nrows * O1P; idx += NF_THREADS) {
      const int r = idx / O1P, o = idx - r * O1P;
      if (o < O1) nf_cp_async4(sG1 + r * G1S + o, dh_out + (size_t)(row0 + r) * O1 + o);
      else sG1[r * G1S + o] = 0.f;
    }
    nf_cp_async_wait();
    __syncthreads();
    if (threadIdx.x < nrows) {
      const int t = threadIdx.x;
      float x[I0P];
#pragma unroll
      for (int k = 0; k < I0P; k += 4) {
        const float4 v = *reinterpret_cast<const float4*>(sX + t * XS + k);
        x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
      }
      float y0[O0P];
#pragma unroll
      for (int o0 = 0; o0 < O0P; o0 += 4) {
        const float4 v = nf_dot4<I0P>(x, sV0, sc0, o0);
        y0[o0] = fmaxf(v.x, alpha * v.x); y0[o0 + 1] = fmaxf(v.y, alpha * v.y); y0[o0 + 2] = fmaxf(v.z, alpha * v.z); y0[o0 + 3] = fmaxf(v.w, alpha * v.w);
        *reinterpret_cast<float4*>(sY0 + t * YS + o0) = make_float4(y0[o0], y0[o0 + 1], y0[o0 + 2], y0[o0 + 3]);
      }
      // g1 = dh_out * leaky'(y1)
      float g1[O1P];
#pragma unroll
      for (int o0 = 0; o0 < O1P; o0 += 4) {
        const float4 v = nf_dot4<O0P>(y0, sV1, sc1, o0);
        const float4 d = *reinterpret_cast<const float4*>(sG1 + t * G1S + o0);
        g1[o0] = d.x * (v.x > 0.f ? 1.f : alpha); g1[o0 + 1] = d.y * (v.y > 0.f ? 1.f : alpha);
        g1[o0 + 2] = d.z * (v.z > 0.f ? 1.f : alpha); g1[o0 + 3] = d.w * (v.w > 0.f ? 1.f : alpha);
        *reinterpret_cast<float4*>(sG1 + t * G1S + o0) = make_float4(g1[o0], g1[o0 + 1], g1[o0 + 2], g1[o0 + 3]);
      }
      // g0 = (V1^T g1) * leaky'(y0)
      float g0[O0P];
#pragma unroll
      for (int o0 = 0; o0 < O0P; o0 += 4) {
        const float4 v = nf_dot4_nobias<O1P>(g1, sV1t, o0);
        g0[o0] = v.x; g0[o0 + 1] = v.y; g0[o0 + 2] = v.z; g0[o0 + 3] = v.w;
      }
#pragma unroll
      for (int o = 0; o < O0P; ++o) g0[o] *= (y0[o] > 0.f ? 1.f : alpha);
#pragma unroll
      for (int o0 = 0; o0 < O0P; o0 += 4) *reinterpret_cast<float4*>(sG0 + t * YS + o0) = make_float4(g0[o0], g0[o0 + 1], g0[o0 + 2], g0[o0 + 3]);
      // dx = V0^T g0 -> de | dh
      float* de_row = de + (size_t)(row0 + t) * EL;
      float* dh_row = dh + (size_t)(row0 + t) * ld;
#pragma unroll
      for (int k0 = 0; k0 < I0P; k0 += 4) {
        const float4 v = nf_dot4_nobias<O0P>(g0, sV0t, k0);
        if (k0 < 16) *reinterpret_cast<float4*>(de_row + k0) = v;
        else {
          const float r4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) if (k0 - 16 + q < cols) dh_row[k0 - 16 + q] = r4[q];
        }
      }
    }
    __syncthreads();
    nf_wgrad_tile<I0P / 4, O0P, U0>(acc0, sG0, YS, sX, XS, nrows);      // dV0 += g0^T x, dc0 += sum g0
    nf_wgrad_tile<O0P / 4, O1P, U1>(acc1, sG1, G1S, sY0, YS, nrows);    // dV1 += g1^T y0, dc1 += sum g1
  }
  float* out = part + (size_t)blockIdx.x * n_node_params;
  nf_wgrad_store<I0P / 4, O0P, U0>(acc0, out, out + O0 * I0, O0, I0);
  nf_wgrad_store<O0P / 4, O1P, U1>(acc1, out + O0 * I0 + O0, out + O0 * I0 + O0 + O1 * O0, O1, O0);
}

// Fixed-order reduction of per-CTA partials: block = 32 outputs x 8 slices; slice y sums partials y, y+8, ... and the
// 8 slice sums are combined through shared memory in slice order (deterministic for a given grid size).
#define RED_SLICES 8
__device__ __forceinline__ float reduce_column(const float* __restrict__ part, int nparts, int n, int p) {
  __shared__ float red[RED_SLICES][33];
  float acc = 0.f;
  if (p < n) {
    int c = threadIdx.y;
    for (; c + 3 * RED_SLICES < nparts; c += 4 * RED_SLICES) {      // four loads in flight; same summation order as one by one
      const float v0 = part[(size_t)c * n + p], v1 = part[(size_t)(c + RED_SLICES) * n + p];
      const float v2 = part[(size_t)(c + 2 * RED_SLICES) * n + p], v3 = part[(size_t)(c + 3 * RED_SLICES) * n + p];
      acc += v0; acc += v1; acc += v2; acc += v3;
    }
    for (; c < nparts; c += RED_SLICES) acc += part[(size_t)c * n + p];
  }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  float tot = 0.f;
  if (threadIdx.y == 0) {
#pragma unroll
    for (int y = 0; y < RED_SLICES; ++y) tot += red[y][threadIdx.x];
  }
  return tot;
}

__global__ void reduce_partials_kernel(const float* __restrict__ part, int nparts, int n, float* __restrict__ out) {
  gj_pdl_sync();
  const int p = blockIdx.x * 32 + threadIdx.x;
  const float v = reduce_column(part, nparts, n, p);
  if (threadIdx.y == 0 && p < n) out[p] = v;
}

// dW0 scatter: the node_pre partials are [Wa E0*H][Wb E0*H][b0 E0]; the packed layout is W0 (E0, 2H+1) then b0.
__global__ void reduce_pre_partials_kernel(const float* __restrict__ part, int nparts, int E0, int H, float* __restrict__ dW0,
                                           float* __restrict__ db0) {
  gj_pdl_sync();
  const int n = E0 * 2 * H + E0;
  const int p = blockIdx.x * 32 + threadIdx.x;
  const float acc = reduce_column(part, nparts, n, p);
  if (threadIdx.y != 0 || p >= n) return;
  const int K0 = 2 * H + 1;
  if (p < E0 * H) { const int c = p / H, k = p - c * H; dW0[c * K0 + k] = acc; }
  else if (p < 2 * E0 * H) { const int q = p - E0 * H; const int c = q / H, k = q - c * H; dW0[c * K0 + H + k] = acc; }
  else db0[p - 2 * E0 * H] = acc;
}

// One launch for the three fixed-order partial reductions of a backward step (bf16 tensor-core path): blocks [0, nbE) the
// edge-kernel partials (all edge parameters but the Wa | Wb columns of W0 and b0), [nbE, nbE + nbP) the projection-adjoint
// partials (those columns and b0), the rest the node-MLP partials.  Same per-output summation order as the single kernels.
struct StepReduce {
  const float* partE; const float* partP; const float* partN;
  int npE, nE, nbE, npP, nbP, npN, nN, E0, H;
  float* dedge; float* dW0; float* db0; float* dnode;
};
__device__ __forceinline__ void reduce_step_partials_body(const StepReduce& R, int bx) {
  const int K0 = 2 * R.H + 1, E0 = R.E0, H = R.H;
  if (bx < R.nbE) {
    const int p = bx * 32 + threadIdx.x;
    const int first = E0 * K0 + E0;          // W0 then b0: only the wd column (index 2H of each row) belongs to the edge kernel
    const bool mine = p < R.nE && !(p < first && !(p < E0 * K0 && (p % K0) == K0 - 1));
    const float acc = reduce_column(R.partE, R.npE, R.nE, mine ? p : R.nE);
    if (threadIdx.y == 0 && mine) R.dedge[p] = acc;
  } else if (bx < R.nbE + R.nbP) {
    const int n = E0 * 2 * H + E0;
    const int p = (bx - R.nbE) * 32 + threadIdx.x;
    const float acc = reduce_column(R.partP, R.npP, n, p);
    if (threadIdx.y != 0 || p >= n) return;
    if (p < E0 * H) { const int c = p / H, k = p - c * H; R.dW0[c * K0 + k] = acc; }
    else if (p < 2 * E0 * H) { const int q = p - E0 * H; const int c = q / H, k = q - c * H; R.dW0[c * K0 + H + k] = acc; }
    else R.db0[p - 2 * E0 * H] = acc;
  } else {
    const int p = (bx - R.nbE - R.nbP) * 32 + threadIdx.x;
    const float acc = reduce_column(R.partN, R.npN, R.nN, p);
    if (threadIdx.y == 0 && p < R.nN) R.dnode[p] = acc;
  }
}
__global__ void reduce_step_partials_kernel(const __grid_constant__ StepReduce R) {
  gj_pdl_sync();
  reduce_step_partials_body(R, blockIdx.x);
}
// the reductions of up to REDUCE_BATCH_MAX steps in ONE launch (gj_mp_steps_reduce): blockIdx.y = step
constexpr int REDUCE_BATCH_MAX = 16;
struct StepReduceBatch { StepReduce r[REDUCE_BATCH_MAX]; };
__global__ void reduce_steps_partials_kernel(const __grid_constant__ StepReduceBatch Bt) {
  gj_pdl_sync();
  const StepReduce& R = Bt.r[blockIdx.y];
  if ((int)blockIdx.x >= R.nbE + R.nbP + (R.nN + 31) / 32) return;      // block-uniform
  reduce_step_partials_body(R, blockIdx.x);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
int gj_num_sms();
void gj_set_error(const char* fmt, ...);

static const int kSmemLimit = 227 * 1024;
static const int kSmemTarget = 54 * 1024;   // <= this many bytes per CTA lets 4 CTAs share an SM (latency hiding)
static const int kSmemTargetBwd = 110 * 1024;   // backward: 2 CTAs per SM, larger row blocks (fewer partials, longer wgrad loops)

static int pre_plan_impl(const MPLayout& L, PreArgs* A, bool backward, bool dpar_global) {
  memset(A, 0, sizeof(*A));
  A->rows = L.B * L.N; A->H = L.H; A->ld = L.ld; A->cols = L.cols; A->E0 = L.E[0]; A->E0p = L.E0p; A->K0 = L.K[0];
  const int Hp = (L.H + 3) & ~3, width = 2 * L.E0p;
  A->hs = nk_stride(L.H);
  A->ps = nk_stride(width);
  for (int R = 128; R >= 8; R >>= 1) {
    A->R = R;
    int off = 0;
    auto take = [&](int n) { int o = off; off += (n + 3) & ~3; return o; };
    if (!backward) {
      A->ws = nk_stride(L.H);
      A->o_w = take(width * A->ws);
      A->o_b = take(width);
      A->o_h = take(R * A->hs);
      A->o_pq = take(R * A->ps);
    } else {
      A->ws = nk_stride(width);
      A->o_w = take(Hp * A->ws);
      A->o_b = take(R * A->hs);      // dh staging
      A->o_h = take(R * A->hs);
      A->o_pq = take(R * A->ps);
      A->o_dpar = dpar_global ? -1 : take(L.E[0] * 2 * L.H + L.E[0]);
    }
    A->smem_floats = off;
    if (off * 4 <= (R > 16 ? (backward ? kSmemTargetBwd : kSmemTarget) : kSmemLimit)) return off * 4;
  }
  return -1;
}
// wide layers (backward): the parameter-gradient accumulators move to the CTA's partial in global memory
static int pre_plan(const MPLayout& L, PreArgs* A, bool backward) {
  int bytes = pre_plan_impl(L, A, backward, false);
  if (bytes < 0 && backward) bytes = pre_plan_impl(L, A, backward, true);
  return bytes;
}

static int post_plan_impl(const MPLayout& L, PostArgs* A, bool backward, bool wide) {
  memset(A, 0, sizeof(*A));
  A->wide = wide ? 1 : 0;
  A->rows = L.B * L.N; A->H = L.H; A->ld = L.ld; A->cols = L.cols; A->EL = L.EL; A->Ln = L.Ln; A->alpha = L.alpha;
  int wmax = L.EL + L.H;
  for (int m = 0; m < L.Ln; ++m) {
    A->O[m] = L.O[m]; A->I[m] = L.I[m]; A->pV[m] = L.pV[m]; A->pc[m] = L.pc[m];
    if (L.O[m] > wmax) wmax = L.O[m];
  }
  A->p_first = L.pV[0];
  A->n_node_params = L.nparams - L.pV[0];
  A->S = nk_stride(wmax);
  for (int R = 128; R >= 8; R >>= 1) {
    A->R = R;
    int off = 0;
    auto take = [&](int n) { int o = off; off += (n + 3) & ~3; return o; };
    int wmaxf = 0;      // wide: one weight area for the largest matrix in either orientation
    for (int m = 0; m < L.Ln; ++m) {
      const int Op = (L.O[m] + 3) & ~3, Ip = (L.I[m] + 3) & ~3;
      A->vs[m] = nk_stride(L.I[m]);
      if (backward) A->vts[m] = nk_stride(L.O[m]);
      if (Op * A->vs[m] > wmaxf) wmaxf = Op * A->vs[m];
      if (backward && Ip * A->vts[m] > wmaxf) wmaxf = Ip * A->vts[m];
    }
    const int o_wide = wide ? take(wmaxf) : 0;
    for (int m = 0; m < L.Ln; ++m) {
      const int Op = (L.O[m] + 3) & ~3, Ip = (L.I[m] + 3) & ~3;
      A->o_V[m] = wide ? o_wide : take(Op * A->vs[m]);
      A->o_c[m] = take(Op);
      if (backward) A->o_Vt[m] = wide ? o_wide : take(Ip * A->vts[m]);
    }
    const int nY = backward ? L.Ln + 1 : 2;
    for (int m = 0; m < nY; ++m) A->o_Y[m] = take(R * A->S);
    if (backward) { A->o_g0 = take(R * A->S); A->o_g1 = take(R * A->S); A->o_dpar = wide ? -1 : take(A->n_node_params); }
    A->smem_floats = off;
    if (off * 4 <= (R > 16 ? (backward ? kSmemTargetBwd : kSmemTarget) : kSmemLimit)) return off * 4;
  }
  return -1;
}
// wide layers (backward): V and its transpose do not fit side by side; see PostArgs::wide
static int post_plan(const MPLayout& L, PostArgs* A, bool backward) {
  int bytes = post_plan_impl(L, A, backward, false);
  if (bytes < 0 && backward) bytes = post_plan_impl(L, A, backward, true);
  return bytes;
}

// every generic node kernel (projections, node MLP and both adjoints) has a shared-memory plan for these widths
bool gj_node_generic_fits(const MPLayout& L) {
  PreArgs A; PostArgs B;
  return pre_plan(L, &A, false) >= 0 && pre_plan(L, &A, true) >= 0 && post_plan(L, &B, false) >= 0 && post_plan(L, &B, true) >= 0;
}

static int nk_grid(int rows, int R, int smem_bytes) {
  int blocks = (rows + R - 1) / R;
  int per_sm = kSmemLimit / (smem_bytes + 1024);
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  int cap = gj_num_sms() * per_sm;
  return blocks < cap ? (blocks > 0 ? blocks : 1) : cap;
}

#define NK_CHECK_LAUNCH(what)                                                                         \
  do { cudaError_t ce_ = cudaGetLastError();                                                          \
       if (ce_ != cudaSuccess) { gj_set_error(what ": %s", cudaGetErrorString(ce_)); return GJ_ERR_CUDA; } } while (0)

template <typename K>
static int nk_set_smem(K kern, int bytes) {
  cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (ce != cudaSuccess) { gj_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

// warp-autonomous forward kernels: CTAs of NW_WARPS warps, two per SM, tiles of 32 rows dealt round-robin
static int nw_grid(int rows) {
  const int tiles = (rows + 31) / 32, cap = gj_num_sms() * 2;
  const int blocks = (tiles + NW_WARPS - 1) / NW_WARPS;
  return blocks < cap ? (blocks > 0 ? blocks : 1) : cap;
}
template <int KP>
static int nw_pre_launch(const MPLayout& L, const float* h, const float* w0, const float* b0, float* pq, cudaStream_t st) {
  using S = NwPreSmem<KP>;
  if (int rc = nk_set_smem(node_pre_fwd_warp_kernel<KP>, S::bytes)) return rc;
  const int rows = L.B * L.N;
  gj_launch(node_pre_fwd_warp_kernel<KP>, nw_grid(rows), NW_WARPS * 32, S::bytes, st, rows, L.H, L.cols, L.ld, L.K[0], h, w0, b0, pq);
  NK_CHECK_LAUNCH("node_pre_fwd launch");
  return GJ_OK;
}
template <int I0P, int O0P, int O1P>
static int nw_post_launch(const MPLayout& L, const float* e, const float* h, const float* params, float* h_out, cudaStream_t st) {
  using S = NwPostSmem<I0P, O0P, O1P>;
  if (int rc = nk_set_smem(node_post_fwd_warp_kernel<I0P, O0P, O1P>, S::bytes)) return rc;
  const int rows = L.B * L.N;
  gj_launch(node_post_fwd_warp_kernel<I0P, O0P, O1P>, nw_grid(rows), NW_WARPS * 32, S::bytes, st, rows, L.EL, L.cols, L.ld, L.I[0], L.O[0],
            L.O[1], L.alpha, e, h, params + L.pV[0], params + L.pc[0], params + L.pV[1], params + L.pc[1], h_out);
  NK_CHECK_LAUNCH("node_post_fwd launch");
  return GJ_OK;
}

int gj_node_pre_fwd(const MPLayout& L, const float* h, const float* params, float* pq, cudaStream_t st) {
  if (L.E[0] == 32 && L.E0p == 32 && L.cols <= 32) {      // thread-per-row kernel (the usual first edge width)
    const int kp = L.cols <= 4 ? 4 : (L.cols <= 8 ? 8 : (L.cols <= 16 ? 16 : 32));
    const float* w0 = params + L.pW[0];
    const float* b0 = params + L.pb[0];
    if (kp == 4) return nw_pre_launch<4>(L, h, w0, b0, pq, st);
    if (kp == 8) return nw_pre_launch<8>(L, h, w0, b0, pq, st);
    if (kp == 16) return nw_pre_launch<16>(L, h, w0, b0, pq, st);
    return nw_pre_launch<32>(L, h, w0, b0, pq, st);
  }
  PreArgs A; int bytes = pre_plan(L, &A, false);
  if (bytes < 0) { gj_set_error("node_pre_fwd: widths do not fit shared memory"); return GJ_ERR_SMEM; }
  if (int rc = nk_set_smem(node_pre_fwd_kernel, bytes)) return rc;
  gj_launch(node_pre_fwd_kernel, nk_grid(A.rows, A.R, bytes), NK_THREADS, bytes, st, A, h, params + L.pW[0], params + L.pb[0], pq);
  NK_CHECK_LAUNCH("node_pre_fwd launch");
  return GJ_OK;
}

size_t gj_node_pre_bwd_ws_floats(const MPLayout& L) {
  PreArgs A; int bytes = pre_plan(L, &A, true);
  if (bytes < 0) return 0;
  return (size_t)nk_grid(A.rows, A.R, bytes) * (L.E[0] * 2 * L.H + L.E[0]);
}

static int nf_bwd_grid(int rows) {      // the per-CTA partials are reduced afterwards: keep their number small
  int blocks = (rows + NF_THREADS - 1) / NF_THREADS, cap = gj_num_sms() * NF_BWD_CTAS_PER_SM;
  return blocks < cap ? (blocks > 0 ? blocks : 1) : cap;
}

// fixed-order reduction of per-CTA [dWa | dWb | db0] partials into the packed W0 / b0 gradients
int gj_reduce_pre_partials(const MPLayout& L, const float* part, int nparts, float* dparams, cudaStream_t st) {
  const int n = L.E[0] * 2 * L.H + L.E[0];
  gj_launch(reduce_pre_partials_kernel, (n + 31) / 32, dim3(32, RED_SLICES), 0, st, part, nparts, L.E[0], L.H, dparams + L.pW[0], dparams + L.pb[0]);
  NK_CHECK_LAUNCH("reduce_pre_partials launch");
  return GJ_OK;
}

static StepReduce step_reduce_args(const MPLayout& L, const float* partE, int npE, const float* partP, int npP, const float* partN, int npN,
                                   float* dparams) {
  StepReduce R;
  R.partE = partE; R.partP = partP; R.partN = partN;
  R.npE = npE; R.nE = L.pV[0]; R.nbE = (R.nE + 31) / 32;
  R.npP = npP; R.nbP = (L.E[0] * 2 * L.H + L.E[0] + 31) / 32;
  R.npN = npN; R.nN = L.nparams - L.pV[0];
  R.E0 = L.E[0]; R.H = L.H;
  R.dedge = dparams; R.dW0 = dparams + L.pW[0]; R.db0 = dparams + L.pb[0]; R.dnode = dparams + L.pV[0];
  return R;
}

int gj_reduce_step_partials(const MPLayout& L, const float* partE, int npE, const float* partP, int npP, const float* partN, int npN,
                            float* dparams, cudaStream_t st) {
  const StepReduce R = step_reduce_args(L, partE, npE, partP, npP, partN, npN, dparams);
  gj_launch(reduce_step_partials_kernel, R.nbE + R.nbP + (R.nN + 31) / 32, dim3(32, RED_SLICES), 0, st, R);
  NK_CHECK_LAUNCH("reduce_step_partials launch");
  return GJ_OK;
}

// the same reduction for n steps in one launch; partE / partP / partN / np*: per step
int gj_reduce_steps_partials(int n, const MPLayout* Ls, const float* const* partE, const int* npE, const float* const* partP, const int* npP,
                             const float* const* partN, const int* npN, float* const* dparams, cudaStream_t st) {
  for (int s0 = 0; s0 < n; s0 += REDUCE_BATCH_MAX) {
    const int m = n - s0 < REDUCE_BATCH_MAX ? n - s0 : REDUCE_BATCH_MAX;
    StepReduceBatch Bt;
    memset(&Bt, 0, sizeof(Bt));
    int nbmax = 1;
    for (int s = 0; s < m; ++s) {
      const int g = s0 + s;
      Bt.r[s] = step_reduce_args(Ls[g], partE[g], npE[g], partP[g], npP[g], partN[g], npN[g], dparams[g]);
      const int nb = Bt.r[s].nbE + Bt.r[s].nbP + (Bt.r[s].nN + 31) / 32;
      if (nb > nbmax) nbmax = nb;
    }
    gj_launch(reduce_steps_partials_kernel, dim3(nbmax, m), dim3(32, RED_SLICES), 0, st, Bt);
    NK_CHECK_LAUNCH("reduce_steps_partials launch");
  }
  return GJ_OK;
}

int gj_node_pre_bwd(const MPLayout& L, const float* h, const float* params, const float* dpq, float* dh, float* dparams,
                    float* part, cudaStream_t st) {
  PreArgs A; int bytes = pre_plan(L, &A, true);
  if (bytes < 0) { gj_set_error("node_pre_bwd: widths do not fit shared memory"); return GJ_ERR_SMEM; }
  if (int rc = nk_set_smem(node_pre_bwd_kernel, bytes)) return rc;
  const int grid = nk_grid(A.rows, A.R, bytes);
  gj_launch(node_pre_bwd_kernel, grid, NK_THREADS, bytes, st, A, h, params + L.pW[0], dpq, dh, part);
  const int n = L.E[0] * 2 * L.H + L.E[0];
  gj_launch(reduce_pre_partials_kernel, (n + 31) / 32, dim3(32, RED_SLICES), 0, st, part, grid, L.E[0], L.H, dparams + L.pW[0], dparams + L.pb[0]);
  NK_CHECK_LAUNCH("node_pre_bwd launch");
  return GJ_OK;
}

int gj_node_post_fwd(const MPLayout& L, const float* e, const float* h, const float* params, float* h_out, cudaStream_t st) {
  if (L.Ln == 2 && L.EL == 16 && L.alpha <= 1.f && L.cols <= L.H) {      // thread-per-row kernels for the usual node widths
    const int i0p = (L.I[0] + 3) & ~3, o0p = (L.O[0] + 3) & ~3, o1p = (L.O[1] + 3) & ~3;
    if (i0p == 32 && o0p == 16 && o1p == 32) return nw_post_launch<32, 16, 32>(L, e, h, params, h_out, st);
    if (i0p == 48 && o0p == 32 && o1p == 8) return nw_post_launch<48, 32, 8>(L, e, h, params, h_out, st);
    if (i0p == 24 && o0p == 8 && o1p == 20) return nw_post_launch<24, 8, 20>(L, e, h, params, h_out, st);
    if (i0p == 24 && o0p == 8 && o1p == 4) return nw_post_launch<24, 8, 4>(L, e, h, params, h_out, st);
  }
  PostArgs A; int bytes = post_plan(L, &A, false);
  if (bytes < 0) { gj_set_error("node_post_fwd: widths do not fit shared memory"); return GJ_ERR_SMEM; }
  if (int rc = nk_set_smem(node_post_fwd_kernel, bytes)) return rc;
  gj_launch(node_post_fwd_kernel, nk_grid(A.rows, A.R, bytes), NK_THREADS, bytes, st, A, e, h, params, h_out);
  NK_CHECK_LAUNCH("node_post_fwd launch");
  return GJ_OK;
}

size_t gj_node_post_bwd_ws_floats(const MPLayout& L) {
  if (L.Ln == 2 && L.EL == 16) {      // thread-per-row adjoint (see gj_node_post_bwd)
    int blocks = (L.B * L.N + NF_THREADS - 1) / NF_THREADS, cap = gj_num_sms() * NF_BWD_CTAS_PER_SM;
    const size_t fast = (size_t)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap) * (size_t)(L.nparams - L.pV[0]);
    PostArgs A0; int b0 = post_plan(L, &A0, true);
    const size_t gen = b0 < 0 ? 0 : (size_t)nk_grid(A0.rows, A0.R, b0) * A0.n_node_params;
    return fast > gen ? fast : gen;
  }
  PostArgs A; int bytes = post_plan(L, &A, true);
  if (bytes < 0) return 0;
  return (size_t)nk_grid(A.rows, A.R, bytes) * A.n_node_params;
}

static int nf_post_shape(const MPLayout& L) {      // index of the compiled (I0P, O0P, O1P) combination, -1 if none
  if (!(L.Ln == 2 && L.EL == 16 && L.alpha <= 1.f && L.cols <= L.H)) return -1;
  const int i0p = (L.I[0] + 3) & ~3, o0p = (L.O[0] + 3) & ~3, o1p = (L.O[1] + 3) & ~3;
  if (i0p == 32 && o0p == 16 && o1p == 32) return 0;
  if (i0p == 48 && o0p == 32 && o1p == 8) return 1;
  if (i0p == 24 && o0p == 8 && o1p == 20) return 2;
  if (i0p == 24 && o0p == 8 && o1p == 4) return 3;
  return -1;
}
template <int I0P, int O0P, int O1P>
static int nf_post_bwd_launch(const MPLayout& L, const float* e, const float* h, const float* params, const float* dh_out, float* de,
                              float* dh, float* part, int grid, cudaStream_t st) {
  constexpr int XS = 4 * ((I0P / 4) | 1), YS = 4 * ((O0P / 4) | 1), G1S = 4 * ((O1P / 4) | 1);
  const int bytes = (2 * O0P * I0P + 2 * O1P * O0P + O0P + O1P + NF_THREADS * (XS + 2 * YS + G1S)) * 4;
  if (int rc = nk_set_smem(node_post_bwd_fast_kernel<I0P, O0P, O1P>, bytes)) return rc;
  gj_launch(node_post_bwd_fast_kernel<I0P, O0P, O1P>, grid, NF_THREADS, bytes, st,
      L.B * L.N, L.EL, L.cols, L.ld, L.I[0], L.O[0], L.O[1], L.alpha, L.nparams - L.pV[0], e, h, params + L.pV[0], params + L.pc[0],
      params + L.pV[1], params + L.pc[1], dh_out, de, dh, part);
  return GJ_OK;
}

int gj_node_post_bwd(const MPLayout& L, const float* e, const float* h, const float* params, const float* dh_out, float* de,
                     float* dh, float* dparams, float* part, cudaStream_t st) {
  const int shape = nf_post_shape(L);
  if (shape >= 0) {
    const int grid = nf_bwd_grid(L.B * L.N), n = L.nparams - L.pV[0];
    int rc = shape == 0 ? nf_post_bwd_launch<32, 16, 32>(L, e, h, params, dh_out, de, dh, part, grid, st)
           : shape == 1 ? nf_post_bwd_launch<48, 32, 8>(L, e, h, params, dh_out, de, dh, part, grid, st)
           : shape == 2 ? nf_post_bwd_launch<24, 8, 20>(L, e, h, params, dh_out, de, dh, part, grid, st)
                        : nf_post_bwd_launch<24, 8, 4>(L, e, h, params, dh_out, de, dh, part, grid, st);
    if (rc) return rc;
    gj_launch(reduce_partials_kernel, (n + 31) / 32, dim3(32, RED_SLICES), 0, st, part, grid, n, dparams + L.pV[0]);
    NK_CHECK_LAUNCH("node_post_bwd launch");
    return GJ_OK;
  }
  PostArgs A; int bytes = post_plan(L, &A, true);
  if (bytes < 0) { gj_set_error("node_post_bwd: widths do not fit shared memory"); return GJ_ERR_SMEM; }
  if (int rc = nk_set_smem(node_post_bwd_kernel, bytes)) return rc;
  const int grid = nk_grid(A.rows, A.R, bytes);
  gj_launch(node_post_bwd_kernel, grid, NK_THREADS, bytes, st, A, e, h, params, dh_out, de, dh, part);
  gj_launch(reduce_partials_kernel, (A.n_node_params + 31) / 32, dim3(32, RED_SLICES), 0, st, part, grid, A.n_node_params, dparams + A.p_first);
  NK_CHECK_LAUNCH("node_post_bwd launch");
  return GJ_OK;
}

int gj_reduce_partials(const float* part, int nparts, int n, float* out, cudaStream_t st) {
  if (n <= 0) return GJ_OK;
  gj_launch(reduce_partials_kernel, (n + 31) / 32, dim3(32, RED_SLICES), 0, st, part, nparts, n, out);
  NK_CHECK_LAUNCH("reduce_partials launch");
  return GJ_OK;
}
