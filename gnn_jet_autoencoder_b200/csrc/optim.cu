// Flat fused Adam (+L1/L2 regulariser gradients), parameter norms, and the 'mean' latent map.
// Replaces torch.optim.Adam as built in reference utils/initialize.py:152-153 (about 100 tiny foreach
// kernels per step), the regularisers of utils/train.py:376-384 / models/encoder.py:173-179, and
// models/encoder.py:147-149.  All HBM-bound elementwise / reduction work.
#include "gj_common.cuh"

namespace {

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float lr_over_bc1, float inv_sqrt_bc2, float b1, float b2,
                            float eps, float gscale, float l1, float l2) {
  gj_pdl_sync();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float pi = p[i];
    float gi = g[i] * gscale;
    if (l1 != 0.f) gi += l1 * (pi > 0.f ? 1.f : (pi < 0.f ? -1.f : 0.f));
    if (l2 != 0.f) gi += 2.f * l2 * pi;
    float mi = b1 * m[i] + (1.f - b1) * gi;
    float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
    p[i] = pi - lr_over_bc1 * (mi / denom);
  }
}

// The other optimisers of utils/initialize.py:154-170 over the same flat buffers (buf = momentum buffer, acc = squared-gradient
// statistic): 1 RMSprop (alpha 0.99, momentum), 2 Adagrad, 3 SGD with momentum -- torch.optim semantics, regulariser gradients folded in
__global__ void optimizer_kernel(int kind, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf,
                                 float* __restrict__ acc, size_t n, float lr, float alpha, float momentum, float eps, float gscale,
                                 float l1, float l2) {
  gj_pdl_sync();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const float pi = p[i];
    float gi = g[i] * gscale;
    if (l1 != 0.f) gi += l1 * (pi > 0.f ? 1.f : (pi < 0.f ? -1.f : 0.f));
    if (l2 != 0.f) gi += 2.f * l2 * pi;
    float upd;
    if (kind == 1) {
      const float sq = alpha * acc[i] + (1.f - alpha) * gi * gi;
      acc[i] = sq;
      const float b = momentum * buf[i] + gi / (sqrtf(sq) + eps);
      buf[i] = b;
      upd = b;
    } else if (kind == 2) {
      const float sq = acc[i] + gi * gi;
      acc[i] = sq;
      upd = gi / (sqrtf(sq) + eps);
    } else {
      const float b = momentum * buf[i] + gi;
      buf[i] = b;
      upd = b;
    }
    p[i] = pi - lr * upd;
  }
}

// ---- the non-finite step guard (GNNAETrainer(nonfinite="skip" | "raise")) ----
// out[0] = 0 if terms[0..count) are all finite, else NaN.  The trainer writes it into the element past the end of the flat gradient,
// so that the gradient all-reduce carries a non-finite loss of one rank to every rank, as it carries a non-finite gradient.
__global__ void nonfinite_flag_kernel(const float* __restrict__ terms, int count, float* __restrict__ out) {
  gj_pdl_sync();
  if (threadIdx.x != 0) return;
  bool ok = true;
  for (int k = 0; k < count; ++k) ok &= isfinite(terms[k]);
  out[0] = ok ? 0.f : __int_as_float(0x7fffffff);
}

// skip[0] = 1 if any of x[0..n) is not finite, else 0; flag[0] (optional) the same as a float.  One CTA: the decision is a few
// hundred KB at most (the flat gradient of a training step), and one CTA needs no cross-CTA combination.
constexpr int kCheckThreads = 1024;
__global__ void __launch_bounds__(kCheckThreads) nonfinite_check_kernel(const float* __restrict__ x, size_t n, int vec,
                                                                        int* __restrict__ skip, float* __restrict__ flag) {
  gj_pdl_sync();
  bool ok = true;
  size_t i = threadIdx.x;
  if (vec) {      // 16-byte aligned: float4 reads, four loads in flight per thread
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const size_t n4 = n / 4;
    for (; i + 3 * kCheckThreads < n4; i += 4 * kCheckThreads) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(x4 + i + (size_t)u * kCheckThreads);
#pragma unroll
      for (int u = 0; u < 4; ++u) ok &= isfinite(v[u].x) & isfinite(v[u].y) & isfinite(v[u].z) & isfinite(v[u].w);
    }
    for (; i < n4; i += kCheckThreads) { const float4 v = __ldg(x4 + i); ok &= isfinite(v.x) & isfinite(v.y) & isfinite(v.z) & isfinite(v.w); }
    i = 4 * n4 + threadIdx.x;
  }
  for (; i < n; i += kCheckThreads) ok &= isfinite(__ldg(x + i));
  const int bad = __syncthreads_or(!ok);
  if (threadIdx.x == 0) {
    skip[0] = bad;
    if (flag) flag[0] = bad ? 1.f : 0.f;
  }
}

// Called by every CTA of a guarded optimiser launch that applied its update, after its last read of state[0]: the last CTA to
// arrive advances the applied-step count state[0]; atomicInc wraps the arrival counter state[1] back to 0 for the next launch.
__device__ __forceinline__ void guard_count_applied(int* state) {
  __syncthreads();
  if (threadIdx.x == 0 && atomicInc(reinterpret_cast<unsigned*>(state + 1), gridDim.x - 1) == gridDim.x - 1) state[0] += 1;
}

// adam_kernel behind the guard: nothing is written when skip[0] != 0; otherwise the update is step state[0] + 1 (bias correction
// computed as gj_adam_launch computes it on the host) and state[0] advances
__global__ void adam_guarded_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                    size_t n, float lr, float b1, float b2, float eps, float gscale, float l1, float l2,
                                    const int* __restrict__ skip, int* state) {
  gj_pdl_sync();
  if (*skip) return;
  __shared__ float coef[2];
  if (threadIdx.x == 0) {
    const int step = *(volatile int*)state + 1;
    const double bc1 = 1.0 - pow((double)b1, (double)step), bc2 = 1.0 - pow((double)b2, (double)step);
    coef[0] = (float)(lr / bc1); coef[1] = (float)(1.0 / sqrt(bc2));
  }
  __syncthreads();
  const float lr_over_bc1 = coef[0], inv_sqrt_bc2 = coef[1];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float pi = p[i];
    float gi = g[i] * gscale;
    if (l1 != 0.f) gi += l1 * (pi > 0.f ? 1.f : (pi < 0.f ? -1.f : 0.f));
    if (l2 != 0.f) gi += 2.f * l2 * pi;
    float mi = b1 * m[i] + (1.f - b1) * gi;
    float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
    p[i] = pi - lr_over_bc1 * (mi / denom);
  }
  guard_count_applied(state);
}

// optimizer_kernel behind the guard (state, optional: the count of applied updates)
__global__ void optimizer_guarded_kernel(int kind, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf,
                                         float* __restrict__ acc, size_t n, float lr, float alpha, float momentum, float eps,
                                         float gscale, float l1, float l2, const int* __restrict__ skip, int* state) {
  gj_pdl_sync();
  if (*skip) return;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const float pi = p[i];
    float gi = g[i] * gscale;
    if (l1 != 0.f) gi += l1 * (pi > 0.f ? 1.f : (pi < 0.f ? -1.f : 0.f));
    if (l2 != 0.f) gi += 2.f * l2 * pi;
    float upd;
    if (kind == 1) {
      const float sq = alpha * acc[i] + (1.f - alpha) * gi * gi;
      acc[i] = sq;
      const float b = momentum * buf[i] + gi / (sqrtf(sq) + eps);
      buf[i] = b;
      upd = b;
    } else if (kind == 2) {
      const float sq = acc[i] + gi * gi;
      acc[i] = sq;
      upd = gi / (sqrtf(sq) + eps);
    } else {
      const float b = momentum * buf[i] + gi;
      buf[i] = b;
      upd = b;
    }
    p[i] = pi - lr * upd;
  }
  if (state) guard_count_applied(state);
}

__global__ void norms_stage1(const float* __restrict__ p, size_t n, float* __restrict__ part) {
  gj_pdl_sync();
  __shared__ float red[2][8];
  float a = 0.f, s = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float x = p[i]; a += fabsf(x); s = fmaf(x, x, s);
  }
  a = gj_warp_sum(a); s = gj_warp_sum(s);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = s; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t0 = 0.f, t1 = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { t0 += red[0][w]; t1 += red[1][w]; }
    part[blockIdx.x * 2] = t0; part[blockIdx.x * 2 + 1] = t1;
  }
}

__global__ void norms_stage2(const float* __restrict__ part, int nblk, float* __restrict__ out) {
  gj_pdl_sync();
  if (threadIdx.x == 0) {
    float t0 = 0.f, t1 = 0.f;
    for (int b = 0; b < nblk; ++b) { t0 += part[b * 2]; t1 += part[b * 2 + 1]; }
    out[0] = t0; out[1] = t1;
  }
}

__global__ void latent_mean_fwd_kernel(int N, int W, const float* __restrict__ y, float* __restrict__ z, int total) {
  gj_pdl_sync();
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int b = idx / W, c = idx - b * W;
  const float* yp = y + (size_t)b * N * W + c;
  float acc = 0.f;
  for (int n = 0; n < N; ++n) acc += yp[(size_t)n * W];
  z[idx] = acc / (float)N;
}

__global__ void latent_mean_bwd_kernel(int N, int W, const float* __restrict__ dz, float* __restrict__ dy, size_t total) {
  gj_pdl_sync();
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  size_t b = idx / ((size_t)N * W);
  int c = (int)(idx % W);
  dy[idx] = dz[b * W + c] / (float)N;
}

// 'max' / 'min' latent maps (encoder.py:150-155, torch.amax / torch.amin over the particle axis).  The adjoint follows
// torch: the gradient of an extremum is shared evenly by the entries that attain it.
__global__ void latent_extreme_fwd_kernel(int N, int W, int is_min, const float* __restrict__ y, float* __restrict__ z, int total) {
  gj_pdl_sync();
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int b = idx / W, c = idx - b * W;
  const float* yp = y + (size_t)b * N * W + c;
  float m = yp[0];
  for (int n = 1; n < N; ++n) { const float v = yp[(size_t)n * W]; m = is_min ? fminf(m, v) : fmaxf(m, v); }
  z[idx] = m;
}
__global__ void latent_extreme_bwd_kernel(int N, int W, const float* __restrict__ y, const float* __restrict__ z,
                                          const float* __restrict__ dz, float* __restrict__ dy, int total) {
  gj_pdl_sync();
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int b = idx / W, c = idx - b * W;
  const float* yp = y + (size_t)b * N * W + c;
  float* dp = dy + (size_t)b * N * W + c;
  const float m = z[idx];
  int ties = 0;
  for (int n = 0; n < N; ++n) ties += yp[(size_t)n * W] == m;
  const float g = dz[idx] / (float)max(ties, 1);
  for (int n = 0; n < N; ++n) dp[(size_t)n * W] = yp[(size_t)n * W] == m ? g : 0.f;
}

// Output transform between the decoder and the loss: y = clamp_k(tanh(x)) -- tanh if the decoder normalises its output
// (decoder.py:123-124), lower clamp at eps of the components in clamp_mask (train.py:55-65, polar coordinates).
__global__ void out_transform_fwd_kernel(size_t n, int dim, int use_tanh, int clamp_mask, float eps, const float* __restrict__ x,
                                         float* __restrict__ y) {
  gj_pdl_sync();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float v = x[i];
    if (use_tanh) v = tanhf(v);
    if ((clamp_mask >> (int)(i % dim)) & 1) v = fmaxf(v, eps);
    y[i] = v;
  }
}
// dx = dy * [tanh(x) >= eps on clamped components] * (1 - tanh(x)^2)
__global__ void out_transform_bwd_kernel(size_t n, int dim, int use_tanh, int clamp_mask, float eps, const float* __restrict__ x,
                                         const float* __restrict__ dy, float* __restrict__ dx) {
  gj_pdl_sync();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float v = x[i], g = dy[i];
    if (use_tanh) v = tanhf(v);
    if (((clamp_mask >> (int)(i % dim)) & 1) && v < eps) g = 0.f;
    if (use_tanh) g *= 1.f - v * v;
    dx[i] = g;
  }
}

// nn.MSELoss (train.py:359-361): value = sum (p - q)^2 / denom, dp = 2 (p - q) / denom; per-block partial sums, fixed order
__global__ void __launch_bounds__(256) mse_stage1(size_t n, float inv_denom, const float* __restrict__ p, const float* __restrict__ q,
                                                  float* __restrict__ dp, float* __restrict__ part) {
  gj_pdl_sync();
  float acc = 0.f;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
    const float d = p[i] - q[i];
    acc = fmaf(d, d, acc);
    dp[i] = 2.f * d * inv_denom;
  }
  __shared__ float red[8];
  acc = gj_warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) { float t = 0.f; for (int w = 0; w < 8; ++w) t += red[w]; part[blockIdx.x] = t; }
}
__global__ void mse_stage2(const float* __restrict__ part, int nblk, float inv_denom, float* __restrict__ terms) {
  gj_pdl_sync();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int b = 0; b < nblk; ++b) t += part[b];
    terms[0] = 0.f; terms[1] = 0.f; terms[2] = (float)(t * inv_denom);
  }
}

}  // namespace

void gj_set_error(const char* fmt, ...);
static const int kNormBlocks = 64;

int gj_latent_extreme_fwd_launch(int B, int N, int W, int is_min, const float* y, float* z, cudaStream_t stream) {
  const int total = B * W;
  if (total == 0) return GJ_OK;
  gj_launch(latent_extreme_fwd_kernel, (total + 255) / 256, 256, 0, stream, N, W, is_min, y, z, total);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("latent_extreme_fwd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
int gj_latent_extreme_bwd_launch(int B, int N, int W, const float* y, const float* z, const float* dz, float* dy, cudaStream_t stream) {
  const int total = B * W;
  if (total == 0) return GJ_OK;
  gj_launch(latent_extreme_bwd_kernel, (total + 255) / 256, 256, 0, stream, N, W, y, z, dz, dy, total);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("latent_extreme_bwd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
int gj_out_transform_launch(size_t n, int dim, int use_tanh, int clamp_mask, float eps, const float* x, const float* dy, float* out,
                            cudaStream_t stream) {
  if (n == 0) return GJ_OK;
  unsigned blocks = (unsigned)((n + 255) / 256); if (blocks > 148 * 8) blocks = 148 * 8;
  if (dy) gj_launch(out_transform_bwd_kernel, blocks, 256, 0, stream, n, dim, use_tanh, clamp_mask, eps, x, dy, out);
  else gj_launch(out_transform_fwd_kernel, blocks, 256, 0, stream, n, dim, use_tanh, clamp_mask, eps, x, out);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("out_transform launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
size_t gj_mse_ws_bytes() { return kNormBlocks * sizeof(float); }
int gj_mse_launch(size_t n, double denom, const float* p, const float* q, float* terms, float* dp, void* ws, size_t ws_bytes,
                  cudaStream_t stream) {
  if (ws_bytes < gj_mse_ws_bytes()) { gj_set_error("gj_mse_fwd_bwd: workspace too small"); return GJ_ERR_WORKSPACE; }
  const float inv = (float)(1.0 / denom);
  gj_launch(mse_stage1, kNormBlocks, 256, 0, stream, n, inv, p, q, dp, (float*)ws);
  gj_launch(mse_stage2, 1, 32, 0, stream, (const float*)ws, kNormBlocks, inv, terms);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("mse launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_adam_launch(float* param, const float* grad, float* m, float* v, size_t n, float lr, float b1, float b2, float eps,
                   int step, float gscale, float l1, float l2, cudaStream_t stream) {
  if (n == 0) return GJ_OK;
  if (step < 1) { gj_set_error("gj_adam_step_flat: step must be >= 1"); return GJ_ERR_INVALID; }
  double bc1 = 1.0 - pow((double)b1, step), bc2 = 1.0 - pow((double)b2, step);
  int blocks = (int)((n + 255) / 256); if (blocks > 148 * 8) blocks = 148 * 8;
  gj_launch(adam_kernel, blocks, 256, 0, stream, param, grad, m, v, n, (float)(lr / bc1), (float)(1.0 / sqrt(bc2)), b1, b2, eps,
                                          gscale, l1, l2);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("adam launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_optimizer_launch(int kind, float* param, const float* grad, float* buf, float* acc, size_t n, float lr, float alpha, float momentum,
                        float eps, float gscale, float l1, float l2, cudaStream_t stream) {
  if (n == 0) return GJ_OK;
  int blocks = (int)((n + 255) / 256); if (blocks > 148 * 8) blocks = 148 * 8;
  gj_launch(optimizer_kernel, blocks, 256, 0, stream, kind, param, grad, buf, acc, n, lr, alpha, momentum, eps, gscale, l1, l2);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("optimizer launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_nonfinite_flag_launch(const float* terms, int count, float* out, cudaStream_t stream) {
  gj_launch(nonfinite_flag_kernel, 1, 32, 0, stream, terms, count, out);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("nonfinite_flag launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_nonfinite_check_launch(const float* x, size_t n, int* skip, float* flag, cudaStream_t stream) {
  const int vec = ((uintptr_t)x & 15) == 0;
  gj_launch(nonfinite_check_kernel, 1, kCheckThreads, 0, stream, x, n, vec, skip, flag);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("nonfinite_check launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_adam_guarded_launch(float* param, const float* grad, float* m, float* v, size_t n, float lr, float b1, float b2, float eps,
                           const int* skip, int* state, float gscale, float l1, float l2, cudaStream_t stream) {
  if (n == 0) return GJ_OK;
  int blocks = (int)((n + 255) / 256); if (blocks > 148 * 8) blocks = 148 * 8;
  gj_launch(adam_guarded_kernel, blocks, 256, 0, stream, param, grad, m, v, n, lr, b1, b2, eps, gscale, l1, l2, skip, state);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("guarded adam launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_optimizer_guarded_launch(int kind, float* param, const float* grad, float* buf, float* acc, size_t n, float lr, float alpha,
                                float momentum, float eps, float gscale, float l1, float l2, const int* skip, int* state,
                                cudaStream_t stream) {
  if (n == 0) return GJ_OK;
  int blocks = (int)((n + 255) / 256); if (blocks > 148 * 8) blocks = 148 * 8;
  gj_launch(optimizer_guarded_kernel, blocks, 256, 0, stream, kind, param, grad, buf, acc, n, lr, alpha, momentum, eps, gscale, l1, l2,
            skip, state);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("guarded optimizer launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

size_t gj_norms_ws_bytes(size_t) { return kNormBlocks * 2 * sizeof(float); }

int gj_norms_launch(const float* p, size_t n, float* out, void* ws, size_t ws_bytes, cudaStream_t stream) {
  if (ws_bytes < gj_norms_ws_bytes(n)) { gj_set_error("gj_param_norms: workspace too small"); return GJ_ERR_WORKSPACE; }
  gj_launch(norms_stage1, kNormBlocks, 256, 0, stream, p, n, (float*)ws);
  gj_launch(norms_stage2, 1, 32, 0, stream, (const float*)ws, kNormBlocks, out);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("norms launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_latent_mean_fwd_launch(int B, int N, int W, const float* y, float* z, cudaStream_t stream) {
  int total = B * W;
  if (total == 0) return GJ_OK;
  gj_launch(latent_mean_fwd_kernel, (total + 255) / 256, 256, 0, stream, N, W, y, z, total);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("latent_mean_fwd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

int gj_latent_mean_bwd_launch(int B, int N, int W, const float* dz, float* dy, cudaStream_t stream) {
  size_t total = (size_t)B * N * W;
  if (total == 0) return GJ_OK;
  gj_launch(latent_mean_bwd_kernel, (unsigned)((total + 255) / 256), 256, 0, stream, N, W, dz, dy, total);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("latent_mean_bwd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

// ------------------------------------------------------------------------------------------------
// small dense layers at node / graph level (decoder.py:127-136, encoder.py:156-161)
// ------------------------------------------------------------------------------------------------
namespace {

constexpr int kLinRB = 8;            // rows per CTA of the forward / input-gradient kernels (staged in shared memory)
constexpr int kLinChunk = 32;        // rows per weight-gradient partial (fewer when K is so large that the x tile would not fit)
constexpr int kLinKT = 32;           // in-features a weight-gradient thread accumulates in registers

// y[r][o] = b[o] + sum_k x[r][k] w[o][k].  A CTA owns kLinRB rows (x staged in shared memory, read as broadcasts) and
// walks the outputs 256 at a time; a thread reads its weight row once for all the CTA's rows.
__global__ void __launch_bounds__(256) linear_fwd_kernel(int rows, int K, int O, const float* __restrict__ x, const float* __restrict__ w,
                                                         const float* __restrict__ b, float* __restrict__ y) {
  gj_pdl_sync();
  extern __shared__ float lin_smem[];      // [kLinRB][K]
  const int r0 = blockIdx.x * kLinRB, nr = min(kLinRB, rows - r0);
  for (int idx = threadIdx.x; idx < nr * K; idx += 256) lin_smem[idx] = __ldg(x + (size_t)r0 * K + idx);
  for (int idx = nr * K + threadIdx.x; idx < kLinRB * K; idx += 256) lin_smem[idx] = 0.f;
  __syncthreads();
  for (int o = threadIdx.x; o < O; o += 256) {
    float acc[kLinRB];
    const float bias = b ? __ldg(b + o) : 0.f;
#pragma unroll
    for (int r = 0; r < kLinRB; ++r) acc[r] = bias;
    const float* wo = w + (size_t)o * K;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      const float wv = __ldg(wo + k);
#pragma unroll
      for (int r = 0; r < kLinRB; ++r) acc[r] = fmaf(lin_smem[r * K + k], wv, acc[r]);
    }
    for (int r = 0; r < nr; ++r) y[(size_t)(r0 + r) * O + o] = acc[r];
  }
}

// dx[r][k] = sum_o dy[r][o] w[o][k], generic form: one thread per (row, k)
__global__ void linear_dx_kernel(int rows, int K, int O, const float* __restrict__ dy, const float* __restrict__ w,
                                 float* __restrict__ dx) {
  gj_pdl_sync();
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)rows * K) return;
  int r = (int)(idx / K), k = (int)(idx - (size_t)r * K);
  const float* g = dy + (size_t)r * O;
  float acc = 0.f;
  for (int o = 0; o < O; ++o) acc = fmaf(__ldg(g + o), __ldg(w + (size_t)o * K + k), acc);
  dx[idx] = acc;
}

// Same for K <= 32 (decoder input layer, local mix): w staged in shared memory, one warp per row, lanes split the O
// outputs and keep K running sums each, combined by shuffles at the end of the row.
constexpr int kDxRowsPerBlock = 8;       // one row per warp
constexpr int kDxOC = 512;               // outputs per staged weight chunk (a lane keeps its 16 dy values of the chunk in registers)
template <bool VEC>
__global__ void __launch_bounds__(256) linear_dx_smallk_kernel(int rows, int K, int O, const float* __restrict__ dy,
                                                               const float* __restrict__ w, float* __restrict__ dx) {
  gj_pdl_sync();
  extern __shared__ float4 lin_smem4[];      // [kDxOC][K]
  float* lin_smem = reinterpret_cast<float*>(lin_smem4);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = blockIdx.x * kDxRowsPerBlock + warp;
  float acc[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) acc[k] = 0.f;
  for (int o0 = 0; o0 < O; o0 += kDxOC) {
    const int oc = min(kDxOC, O - o0);
    float g[kDxOC / 32];
#pragma unroll
    for (int j = 0; j < kDxOC / 32; ++j) g[j] = (r < rows && lane + 32 * j < oc) ? __ldg(dy + (size_t)r * O + o0 + lane + 32 * j) : 0.f;
    if (o0 > 0) __syncthreads();      // the previous chunk has been consumed
    for (int idx = threadIdx.x; idx < oc * K; idx += 256)      // asynchronous copies: the loads do not wait for one another
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(lin_smem + idx)), "l"(w + (size_t)o0 * K + idx) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kDxOC / 32; ++j) {
      if (32 * j >= oc) break;      // uniform
      const int o = min(lane + 32 * j, oc - 1);      // lanes past the end carry g = 0
      const float* wo = lin_smem + o * K;
      if (VEC) {      // K % 4 == 0: 16-byte reads (lanes are K floats apart: conflict free for K = 4 * odd)
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4) {
          if (4 * q4 < K) {
            const float4 v = *reinterpret_cast<const float4*>(wo + 4 * q4);
            acc[4 * q4] = fmaf(g[j], v.x, acc[4 * q4]); acc[4 * q4 + 1] = fmaf(g[j], v.y, acc[4 * q4 + 1]);
            acc[4 * q4 + 2] = fmaf(g[j], v.z, acc[4 * q4 + 2]); acc[4 * q4 + 3] = fmaf(g[j], v.w, acc[4 * q4 + 3]);
          }
        }
      } else {
#pragma unroll
        for (int k = 0; k < 32; ++k) if (k < K) acc[k] = fmaf(g[j], wo[k], acc[k]);
      }
    }
  }
  if (r >= rows) return;
  float mine = 0.f;
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    if (k < K) {      // uniform
      float v = acc[k];
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
      if (lane == k) mine = v;
    }
  }
  if (lane < K) dx[(size_t)r * K + lane] = mine;
}

// Per chunk of rows: part[chunk][o * (K + 1) + k] = sum_r dy[r][o] x[r][k]; slot k == K holds the bias gradient (x extended
// by a column of ones).  A thread owns one output o and kLinKT consecutive k in registers; the x tile rows are padded to a
// multiple of 4 floats and read as 16-byte broadcasts.
__global__ void __launch_bounds__(256) linear_dw_partial_kernel(int rows, int K, int O, int chunk, const float* __restrict__ x,
                                                                const float* __restrict__ dy, float* __restrict__ part) {
  gj_pdl_sync();
  extern __shared__ float4 lin_smem4[];      // [chunk][K1p]
  float* xs = reinterpret_cast<float*>(lin_smem4);
  const int K1 = K + 1, K1p = (K1 + 3) & ~3, r0 = blockIdx.y * chunk, nr = min(chunk, rows - r0);
  for (int idx = threadIdx.x; idx < chunk * K1p; idx += 256) {
    const int r = idx / K1p, k = idx - r * K1p;
    xs[idx] = r < nr ? (k < K ? __ldg(x + (size_t)(r0 + r) * K + k) : (k == K ? 1.f : 0.f)) : 0.f;
  }
  __syncthreads();
  const int kchunks = (K1 + kLinKT - 1) / kLinKT, items = O * kchunks;
  for (int item = blockIdx.x * 256 + threadIdx.x; item < items; item += gridDim.x * 256) {
    const int kc = item / O, o = item - kc * O, k0 = kc * kLinKT;
    float acc[kLinKT];
#pragma unroll
    for (int q = 0; q < kLinKT; ++q) acc[q] = 0.f;
    float g[kLinChunk];      // the chunk's dy column first: the loads overlap one another
#pragma unroll
    for (int r = 0; r < kLinChunk; ++r) g[r] = r < nr ? __ldg(dy + (size_t)(r0 + r) * O + o) : 0.f;
#pragma unroll
    for (int r = 0; r < kLinChunk; ++r) {
      if (r >= nr) continue;      // uniform
      const float4* xr = reinterpret_cast<const float4*>(xs + r * K1p + k0);
#pragma unroll
      for (int q4 = 0; q4 < kLinKT / 4; ++q4) {
        if (k0 + 4 * q4 < K1) {      // uniform
          const float4 v = xr[q4];
          acc[4 * q4] = fmaf(g[r], v.x, acc[4 * q4]); acc[4 * q4 + 1] = fmaf(g[r], v.y, acc[4 * q4 + 1]);
          acc[4 * q4 + 2] = fmaf(g[r], v.z, acc[4 * q4 + 2]); acc[4 * q4 + 3] = fmaf(g[r], v.w, acc[4 * q4 + 3]);
        }
      }
    }
    float* dst = part + (size_t)blockIdx.y * O * K1 + (size_t)o * K1 + k0;
#pragma unroll
    for (int q = 0; q < kLinKT; ++q) if (k0 + q < K1) dst[q] = acc[q];
  }
}

// fixed-order sum of the chunk partials: block = 32 outputs x 8 slices; slice y sums chunks y, y + 8, ... and the slice
// sums are combined in slice order
__global__ void __launch_bounds__(256) linear_dw_reduce_kernel(int nchunks, int K, int O, const float* __restrict__ part,
                                                               float* __restrict__ dw, float* __restrict__ db) {
  gj_pdl_sync();
  __shared__ float red[8][33];
  const int K1 = K + 1, total = K1 * O;
  const int idx = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (idx < total)
    for (int c = threadIdx.y; c < nchunks; c += 8) acc += part[(size_t)c * total + idx];
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && idx < total) {
    float tot = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) tot += red[y][threadIdx.x];
    const int o = idx / K1, k = idx - o * K1;
    if (k < K) dw[(size_t)o * K + k] = tot;
    else if (db) db[o] = tot;
  }
}

}  // namespace

static int lin_set_smem(const void* kern, size_t bytes, const char* who) {
  if (bytes > 200 * 1024) { gj_set_error("%s: layer too wide for the shared-memory row tile (%zu bytes)", who, bytes); return GJ_ERR_SMEM; }
  if (bytes > 48 * 1024) {
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (ce != cudaSuccess) { gj_set_error("%s: %s", who, cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  }
  return GJ_OK;
}

int gj_linear_fwd_launch(int rows, int K, int O, const float* x, const float* w, const float* b, float* y, cudaStream_t stream) {
  if ((size_t)rows * O == 0) return GJ_OK;
  const size_t smem = (size_t)kLinRB * K * sizeof(float);
  if (int rc = lin_set_smem((const void*)linear_fwd_kernel, smem, "linear_fwd")) return rc;
  gj_launch(linear_fwd_kernel, (rows + kLinRB - 1) / kLinRB, 256, smem, stream, rows, K, O, x, w, b, y);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("linear_fwd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

static int lin_chunk_rows(int K) { int c = kLinChunk; while (c > 1 && (size_t)c * (K + 4) * sizeof(float) > 96 * 1024) c >>= 1; return c; }
static int lin_chunks(int rows, int K) { const int cr = lin_chunk_rows(K); int c = (rows + cr - 1) / cr; return c < 1 ? 1 : c; }

size_t gj_linear_bwd_ws_bytes(int rows, int K, int O) { return (size_t)lin_chunks(rows, K) * (K + 1) * O * sizeof(float); }

int gj_linear_bwd_launch(int rows, int K, int O, const float* x, const float* w, const float* dy, float* dx, float* dw,
                         float* db, void* ws, size_t ws_bytes, cudaStream_t stream) {
  if (ws_bytes < gj_linear_bwd_ws_bytes(rows, K, O)) { gj_set_error("gj_linear_bwd: workspace too small"); return GJ_ERR_WORKSPACE; }
  const int total = (K + 1) * O;
  const int nch = rows > 0 ? lin_chunks(rows, K) : 0, chunk = lin_chunk_rows(K);
  if (rows > 0) {
    if (dx) {
      const size_t smem = (size_t)(O < kDxOC ? O : kDxOC) * K * sizeof(float);
      if (K <= 32) {
        auto kern = (K & 3) == 0 ? linear_dx_smallk_kernel<true> : linear_dx_smallk_kernel<false>;
        if (int rc = lin_set_smem((const void*)kern, smem, "linear_bwd")) return rc;
        gj_launch(kern, (rows + kDxRowsPerBlock - 1) / kDxRowsPerBlock, 256, smem, stream, rows, K, O, dy, w, dx);
      } else {
        gj_launch(linear_dx_kernel, (unsigned)(((size_t)rows * K + 255) / 256), 256, 0, stream, rows, K, O, dy, w, dx);
      }
    }
    const size_t smem = (size_t)chunk * ((K + 4) & ~3) * sizeof(float);
    if (int rc = lin_set_smem((const void*)linear_dw_partial_kernel, smem, "linear_bwd")) return rc;
    const int items = O * ((K + 1 + kLinKT - 1) / kLinKT);
    dim3 grid((items + 255) / 256, nch);
    gj_launch(linear_dw_partial_kernel, grid, 256, smem, stream, rows, K, O, chunk, x, dy, (float*)ws);
  }
  gj_launch(linear_dw_reduce_kernel, (total + 31) / 32, dim3(32, 8), 0, stream, nch, K, O, (const float*)ws, dw, db);
  cudaError_t ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("linear_bwd launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
