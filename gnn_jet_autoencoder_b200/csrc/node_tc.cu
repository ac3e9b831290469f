// Node-level adjoint kernels on tcgen05 (GJ_PREC_BF16 only; the fp32 mode keeps the SIMT kernels of node_kernels.cu).
//
// node_pre_bwd_tc_kernel: adjoint of the first-edge-layer projections P_i = Wa h_i + b0, Q_j = Wb h_j
// (the factorised W0 [h_i | h_j | d] of reference models/graphnet.py:220) over all B*N node rows:
//     dh[row]   += dPQ[row] (64) . [Wa ; Wb] (64 x H)                      one GEMM per 128-row tile, accumulator in TMEM
//     [dWa ; dWb | db0] += dPQ^T [h | 1]    (64 x (H + 16), K = rows)      accumulator resident in TMEM for the whole kernel
// A CTA is one 128-thread tile group (thread = node row = TMEM lane) with a 128-column TMEM allocation, so four CTAs share
// an SM and hide each other's staging / GEMM / epilogue phases.  The row tile is staged as bf16 in the UMMA SWIZZLE_NONE
// slab layout ([8-channel slab][128 rows][8]), which serves as K-major A operand of the dgrad GEMM and as MN-major operand
// (K = tile row) of the weight-gradient GEMM alike.  bf16 operands, fp32 accumulation: the same precision class as the
// edge-MLP weight gradients.
// All global traffic is coalesced (a thread walking its own row touches 32 lines per instruction, which made the first
// version L1-wavefront bound): the dPQ rows are read four whole rows per warp instruction straight into slab entries (and
// prefetched one tile ahead, in registers, behind the GEMMs); the h and dh row tiles are copied with cp.async into padded
// fp32 tiles, converted / accumulated thread-per-row there, and the dh tile is written back with coalesced stores.
#include <stdlib.h>

#include "tc2_common.cuh"

namespace {
using namespace tc2;

__device__ __forceinline__ void ntc_cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void ntc_cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void ntc_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void ntc_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <int HP>
struct PreBwdSmem {
  static constexpr int TS = HP + 4;                          // fp32 tile row stride (4 * odd floats: per-row 16-byte accesses are conflict free)
  static constexpr int o_bar = 0;
  static constexpr int o_slot = 16;
  static constexpr int o_wt = 1024;                          // [HP][64] bf16 K-major B operand: WabT[n][c] = [Wa ; Wb][c][n]
  static constexpr int o_g = o_wt + HP * 64 * 2;             // dPQ tile: 8 slabs
  static constexpr int o_h = o_g + 8 * 2048;                 // h tile: HP / 8 slabs, then the ones slab and a zero slab
  static constexpr int o_th = o_h + (HP / 8 + 2) * 2048;     // fp32 h tile [128][TS] (coalesced copy of the global rows)
  static constexpr int o_td = o_th + 128 * TS * 4;           // fp32 dh tile [128][TS]: read, accumulated, written back
  static constexpr int total = o_td + 128 * TS * 4;
};

// dPQ rows of one tile as this thread's 8 (row, 8-channel slab) entries: entry it covers row (it * 4 + warp) * 4 + (lane & 3),
// slab lane >> 2, so that a warp instruction reads four whole 256-byte rows
struct DpqRegs { float4 v[16]; };
__device__ __forceinline__ void ntc_load_dpq(DpqRegs& R, const float* __restrict__ dpq, int row0, int rows, int warp, int lane) {
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int row = row0 + (it * 4 + warp) * 4 + (lane & 3);
    const float4* src = reinterpret_cast<const float4*>(dpq + (size_t)row * 64 + (lane >> 2) * 8);
    if (row < rows) { R.v[2 * it] = __ldg(src); R.v[2 * it + 1] = __ldg(src + 1); }
    else { R.v[2 * it] = make_float4(0.f, 0.f, 0.f, 0.f); R.v[2 * it + 1] = R.v[2 * it]; }
  }
}

template <int HP>
__global__ void __launch_bounds__(128) node_pre_bwd_tc_kernel(int rows, int H, int cols, int ld, int K0, const float* __restrict__ h,
                                                              const float* __restrict__ w0, const float* __restrict__ dpq,
                                                              float* __restrict__ dh, float* __restrict__ part) {
  gj_pdl_sync();
  using S = PreBwdSmem<HP>;
  constexpr int TS = S::TS;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = (int)uni((uint32_t)(tid >> 5));
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::o_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::o_slot);
  float* sH = reinterpret_cast<float*>(smem + S::o_th);
  float* sD = reinterpret_cast<float*>(smem + S::o_td);
  const int ntiles = (rows + 127) / 128;
  DpqRegs R;
  if ((int)blockIdx.x < ntiles) ntc_load_dpq(R, dpq, blockIdx.x * 128, rows, warp, lane);
  // ---- one-time staging: transposed projection weights, constant slabs, barrier, TMEM ----
  // W0 (32 rows of K0 = 2 H + 1 floats) first lands in the h / dh tile area through asynchronous copies (overlapping loads)
  float* raw = reinterpret_cast<float*>(smem + S::o_th);
  const bool raw_fits = 32 * K0 * 4 <= 2 * 128 * S::TS * 4;
  if (raw_fits) for (int idx = tid; idx < 32 * K0; idx += 128) ntc_cp_async4(raw + idx, w0 + idx);
  ntc_cp_async_commit();
  for (int idx = tid; idx < 1024; idx += 128)      // ones slab (channel HP = 1.0, HP + 1 .. HP + 7 = 0), zero slab
    reinterpret_cast<uint32_t*>(smem + S::o_h + (HP / 8) * 2048)[idx] = (idx < 512 && (idx & 3) == 0) ? 0x00003F80u : 0u;
  ntc_cp_async_wait_all();
  __syncthreads();
  for (int idx = tid; idx < HP * 64; idx += 128) {
    const int n = idx >> 6, c = idx & 63, src = (c & 31) * K0 + (c < 32 ? n : H + n);
    const float v = n < cols ? (raw_fits ? raw[src] : __ldg(w0 + src)) : 0.f;
    *reinterpret_cast<__nv_bfloat16*>(smem + S::o_wt + (c >> 3) * (HP * 16) + n * 16 + (c & 7) * 2) = __float2bfloat16_rn(v);
  }
  __syncthreads();      // the tile area is free for the first tile's copies
  if (tid == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(tmem_slot, 128);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
  {      // the gradient accumulator [64, 64 + HP + 16) starts at zero: every weight-gradient MMA accumulates
    uint32_t z[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) z[c] = 0u;
#pragma unroll
    for (int c0 = 0; c0 < HP + 16; c0 += 16) tmem_st16(lane_base + 64 + c0, z);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const uint32_t ga = smem_u32(smem + S::o_g), ha = smem_u32(smem + S::o_h), wta = smem_u32(smem + S::o_wt);
  const bool vec = (ld & 3) == 0 && ((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(dh)) & 15) == 0;
  const int q4 = min((ld + 3) >> 2, HP / 4);      // 16-byte pieces fetched per row (they cover the `cols` live columns)
  uint32_t ph = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * 128, nrows = min(128, rows - row0);
    // ---- coalesced copies of the h and dh row tiles into shared memory ----
    if (vec) {
      for (int idx = tid; idx < nrows * q4; idx += 128) {
        const int r = idx / q4, k = idx - r * q4;
        ntc_cp_async16(sH + r * TS + 4 * k, h + (size_t)(row0 + r) * ld + 4 * k);
        ntc_cp_async16(sD + r * TS + 4 * k, dh + (size_t)(row0 + r) * ld + 4 * k);
      }
    } else {
      for (int idx = tid; idx < nrows * cols; idx += 128) {
        const int r = idx / cols, k = idx - r * cols;
        sH[r * TS + k] = __ldg(h + (size_t)(row0 + r) * ld + k);
        sD[r * TS + k] = dh[(size_t)(row0 + r) * ld + k];
      }
    }
    ntc_cp_async_commit();
    // ---- this tile's dPQ entries (prefetched during the previous tile) -> bf16 slabs ----
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const float4 a = R.v[2 * it], b = R.v[2 * it + 1];
      const int r = (it * 4 + warp) * 4 + (lane & 3);
      *reinterpret_cast<uint4*>(smem + S::o_g + (lane >> 2) * 2048 + r * 16) =
          make_uint4(bf2_as_u32(__floats2bfloat162_rn(a.x, a.y)), bf2_as_u32(__floats2bfloat162_rn(a.z, a.w)),
                     bf2_as_u32(__floats2bfloat162_rn(b.x, b.y)), bf2_as_u32(__floats2bfloat162_rn(b.z, b.w)));
    }
    ntc_cp_async_wait_all();
    __syncthreads();
    // ---- this thread's h row -> bf16 slabs (zero beyond `cols` and beyond the last row) ----
    {
      const bool live = tid < nrows;
#pragma unroll
      for (int s = 0; s < HP / 8; ++s) {
        const float4 a = *reinterpret_cast<const float4*>(sH + tid * TS + 8 * s), b = *reinterpret_cast<const float4*>(sH + tid * TS + 8 * s + 4);
        const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        float w[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) w[q] = (live && 8 * s + q < cols) ? v[q] : 0.f;
        *reinterpret_cast<uint4*>(smem + S::o_h + s * 2048 + tid * 16) =
            make_uint4(bf2_as_u32(__floats2bfloat162_rn(w[0], w[1])), bf2_as_u32(__floats2bfloat162_rn(w[2], w[3])),
                       bf2_as_u32(__floats2bfloat162_rn(w[4], w[5])), bf2_as_u32(__floats2bfloat162_rn(w[6], w[7])));
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      // dgrad: acc[0, HP) = dPQ (A, K-major) . [Wa ; Wb] (B = WabT, K-major), K = 64
      const uint32_t i_d = make_idesc_bf16(128, HP, 0, 0);
#pragma unroll
      for (int s = 0; s < 4; ++s)
        mma_bf16_ss_elect(tmem_base, make_smem_desc(ga + s * 4096, 2048, 128), make_smem_desc(wta + s * 2 * HP * 16, HP * 16, 128), i_d, s > 0);
      // wgrad: acc[64, 64 + HP + 16) += dPQ^T [h | 1 | 0] (both MN-major views, K = tile row)
      const uint32_t i_g = make_idesc_bf16(64, HP + 16, 1, 1);
#pragma unroll
      for (int s = 0; s < 8; ++s)
        mma_bf16_ss_elect(tmem_base + 64, make_smem_desc(ga + s * 256, 128, 2048), make_smem_desc(ha + s * 256, 128, 2048), i_g, 1u);
      mma_commit_elect(bar);
    }
    if (tile + (int)gridDim.x < ntiles) ntc_load_dpq(R, dpq, (tile + gridDim.x) * 128, rows, warp, lane);      // in flight behind the GEMMs
    mbar_wait(bar, ph); ph ^= 1u;
    tc_fence_after();
    // ---- epilogue: dh tile row += acc, then the tile goes back to global memory with coalesced stores ----
#pragma unroll
    for (int c0 = 0; c0 < HP; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + c0, v);
      tmem_ld_wait(); tmem_pin16(v);
#pragma unroll
      for (int q = 0; q < 16; q += 4) {
        float4 o = *reinterpret_cast<const float4*>(sD + tid * TS + c0 + q);
        o.x += __uint_as_float(v[q]); o.y += __uint_as_float(v[q + 1]); o.z += __uint_as_float(v[q + 2]); o.w += __uint_as_float(v[q + 3]);
        *reinterpret_cast<float4*>(sD + tid * TS + c0 + q) = o;
      }
    }
    tc_fence_before();
    __syncthreads();      // the staging buffers and acc[0, HP) are free again; the dh tile is complete
    if (vec) {
      for (int idx = tid; idx < nrows * q4; idx += 128) {
        const int r = idx / q4, k = idx - r * q4;
        float* dst = dh + (size_t)(row0 + r) * ld + 4 * k;
        const float4 o = *reinterpret_cast<const float4*>(sD + r * TS + 4 * k);
        if (4 * k + 3 < cols) *reinterpret_cast<float4*>(dst) = o;
        else {
          const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) if (4 * k + q < cols) dst[q] = ov[q];
        }
      }
    } else {
      for (int idx = tid; idx < nrows * cols; idx += 128) {
        const int r = idx / cols, k = idx - r * cols;
        dh[(size_t)(row0 + r) * ld + k] = sD[r * TS + k];
      }
    }
    __syncthreads();      // the next tile's copies overwrite the dh tile
  }
  // ---- gradient read-out: M = 64 accumulator, channel m at lane (m / 16) * 32 + m % 16; column k < HP = in feature, HP = bias ----
  tc_fence_after();
  float* out = part + (size_t)blockIdx.x * (64 * H + 32);
  {
    const int m = warp * 16 + (lane & 15);      // 0..31: Wa / b0 rows, 32..63: Wb rows (lanes 16..31 hold nothing)
    float* rowp = out + (m < 32 ? m * H : 32 * H + (m - 32) * H);
#pragma unroll
    for (int c0 = 0; c0 < HP + 16; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + 64 + c0, v);      // .aligned: every lane of the warp issues the load
      tmem_ld_wait(); tmem_pin16(v);
      if (lane < 16) {
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const int k = c0 + q;
          if (k < H && k < HP) rowp[k] = k < cols ? __uint_as_float(v[q]) : 0.f;
          if (k == HP && m < 32) out[64 * H + m] = __uint_as_float(v[q]);
        }
      }
    }
    if (lane < 16) for (int k = HP; k < H; ++k) rowp[k] = 0.f;      // columns of W0 that multiply the zero padding of h
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 128);
}


// ---------------------------------------------------------------------------------------------------------------------
// node_post_bwd_tc_kernel: adjoint of the two-layer node MLP  h' = leaky(V1 leaky(V0 [e | h] + c0) + c1)  (reference
// models/graphnet.py:249-271) over all B*N node rows, 128 rows per tile, thread = row = TMEM lane.  Per tile a chain of
// four small GEMMs with register epilogues in between, and the two weight-gradient GEMMs accumulating in TMEM for the
// whole kernel:
//   Y0  = [X | 1] [V0 | c0]^T  -> y0 = leaky(Y0) as bf16 slabs, sign mask kept in a register
//   Y1  = [y0 | 1] [V1 | c1]^T -> g1 = dh' * leaky'(Y1) as bf16 slabs
//   G0  = g1 V1                -> g0 = G0 * leaky'(Y0) as bf16 slabs
//   DX  = g0 V0                -> de (first 16 columns) | dh (OVERWRITES the first `cols` columns)
//   [dV0 | dc0] += g0^T [X | 1]   (M = 64, TMEM columns [64, 128), lanes 0..15 of every quadrant)
//   [dV1 | dc1] += g1^T [y0 | 1]  (M = 64, same columns, lanes 16..31 of every quadrant)
// I0P / O0P / O1P = layer widths padded to 16.  TMEM: 128 columns per CTA (chain accumulators alias one another in
// [0, 64)), so up to four CTAs share an SM.  Biases ride as an extra k-step (hi + lo bf16 halves) against a constant
// slab whose channels 0 and 1 are one; the same slab is the B operand of the bias-gradient MMAs.
// ---------------------------------------------------------------------------------------------------------------------
template <int I0P, int O0P, int O1P>
struct PostBwdSmem {
  static constexpr int XS = I0P / 8, YS = O0P / 8, G1S = O1P / 8;
  static constexpr int o_bar = 0;                              // chain barrier, weight-gradient barrier
  static constexpr int o_slot = 16;
  static constexpr int o_g0 = 1024;                            // the M = 64 weight-gradient A operands read 8 slabs from
  static constexpr int o_g1 = o_g0 + YS * 2048;                // their base: whatever follows g0 / g1 lands in unused rows
  static constexpr int o_x = o_g1 + G1S * 2048;
  static constexpr int o_y0 = o_x + XS * 2048;
  static constexpr int o_ones = o_y0 + YS * 2048;              // ones slab (channels 0, 1), zero slab
  static constexpr int o_b1 = o_ones + 2 * 2048;               // [V0 | c0]: K-major B, K = I0P + 16, N = O0P
  static constexpr int o_b2 = o_b1 + (I0P + 16) * O0P * 2;     // [V1 | c1]: K = O0P + 16, N = O1P
  static constexpr int o_b3 = o_b2 + (O0P + 16) * O1P * 2;     // V1^T: K = O1P, N = O0P
  static constexpr int o_b4 = o_b3 + O1P * O0P * 2;            // V0^T: K = O0P, N = I0P
  static constexpr int total = o_b4 + O0P * I0P * 2;
  static_assert(G1S + XS + YS + 2 >= 8 && YS + G1S + XS >= 8, "weight-gradient A operands must stay inside the allocation");
};

__device__ __forceinline__ void ntc_put_bf16(uint8_t* base, int nrows_b, int k, int n, float v) {      // K-major B element (k, n)
  *reinterpret_cast<__nv_bfloat16*>(base + (k >> 3) * (nrows_b * 16) + n * 16 + (k & 7) * 2) = __float2bfloat16_rn(v);
}
__device__ __forceinline__ uint4 ntc_pack8(const float (&v)[8]) {
  return make_uint4(bf2_as_u32(__floats2bfloat162_rn(v[0], v[1])), bf2_as_u32(__floats2bfloat162_rn(v[2], v[3])),
                    bf2_as_u32(__floats2bfloat162_rn(v[4], v[5])), bf2_as_u32(__floats2bfloat162_rn(v[6], v[7])));
}
// 8 consecutive floats k0 .. k0 + 7 of a row of `ld` floats; columns >= cols read as zero
__device__ __forceinline__ void ntc_load8(const float* __restrict__ rowp, int k0, int cols, int ld, bool vec, bool live, float (&v)[8]) {
#pragma unroll
  for (int q = 0; q < 8; ++q) v[q] = 0.f;
  if (!live) return;
  if (vec) {
    if (k0 < cols) { const float4 a = __ldg(reinterpret_cast<const float4*>(rowp + k0)); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; }
    if (k0 + 4 < cols) { const float4 b = __ldg(reinterpret_cast<const float4*>(rowp + k0 + 4)); v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w; }
#pragma unroll
    for (int q = 0; q < 8; ++q) if (k0 + q >= cols) v[q] = 0.f;
  } else {
#pragma unroll
    for (int q = 0; q < 8; ++q) if (k0 + q < cols) v[q] = __ldg(rowp + k0 + q);
  }
}

template <int I0P, int O0P, int O1P>
__global__ void __launch_bounds__(128) node_post_bwd_tc_kernel(int rows, int cols, int ld, int I0, int O0, int O1, float alpha,
                                                               int n_node_params, const float* __restrict__ e,
                                                               const float* __restrict__ h, const float* __restrict__ V0,
                                                               const float* __restrict__ c0, const float* __restrict__ V1,
                                                               const float* __restrict__ c1, const float* __restrict__ dh_out,
                                                               float* __restrict__ de, float* __restrict__ dh, float* __restrict__ part,
                                                               float* __restrict__ zero64) {
  gj_pdl_sync();
  using S = PostBwdSmem<I0P, O0P, O1P>;
  constexpr int HS = S::XS - 2;      // h slabs of the X tile (the first two hold e)
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = (int)uni((uint32_t)(tid >> 5));
  uint64_t* barA = reinterpret_cast<uint64_t*>(smem + S::o_bar);
  uint64_t* barW = barA + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::o_slot);
  // ---- one-time staging: the four weight operands, constant slabs, barriers, TMEM ----
  // the fp32 parameters first land in the (still unused) slab area through asynchronous copies, so that the loads overlap
  float* raw = reinterpret_cast<float*>(smem + S::o_g0);      // [V0 | V1 | c0 | c1]
  for (int idx = tid; idx < O0 * I0; idx += 128) ntc_cp_async4(raw + idx, V0 + idx);
  for (int idx = tid; idx < O1 * O0; idx += 128) ntc_cp_async4(raw + O0 * I0 + idx, V1 + idx);
  for (int n = tid; n < O0; n += 128) ntc_cp_async4(raw + O0 * I0 + O1 * O0 + n, c0 + n);
  for (int n = tid; n < O1; n += 128) ntc_cp_async4(raw + O0 * I0 + O1 * O0 + O0 + n, c1 + n);
  ntc_cp_async_commit();
  for (int idx = tid; idx < (S::total - S::o_b1) / 4; idx += 128) reinterpret_cast<uint32_t*>(smem + S::o_b1)[idx] = 0u;
  for (int idx = tid; idx < 1024; idx += 128)
    reinterpret_cast<uint32_t*>(smem + S::o_ones)[idx] = (idx < 512 && (idx & 3) == 0) ? 0x3F803F80u : 0u;
  ntc_cp_async_wait_all();
  __syncthreads();
  for (int idx = tid; idx < O0 * I0; idx += 128) {
    const int n = idx / I0, k = idx - n * I0;
    const float v = raw[idx];
    ntc_put_bf16(smem + S::o_b1, O0P, k, n, v);
    ntc_put_bf16(smem + S::o_b4, I0P, n, k, v);
  }
  for (int idx = tid; idx < O1 * O0; idx += 128) {
    const int n = idx / O0, k = idx - n * O0;
    const float v = raw[O0 * I0 + idx];
    ntc_put_bf16(smem + S::o_b2, O1P, k, n, v);
    ntc_put_bf16(smem + S::o_b3, O0P, n, k, v);
  }
  for (int n = tid; n < O0; n += 128) {
    const float b = raw[O0 * I0 + O1 * O0 + n], hi = __bfloat162float(__float2bfloat16_rn(b));
    ntc_put_bf16(smem + S::o_b1, O0P, I0P, n, hi);
    ntc_put_bf16(smem + S::o_b1, O0P, I0P + 1, n, b - hi);
  }
  for (int n = tid; n < O1; n += 128) {
    const float b = raw[O0 * I0 + O1 * O0 + O0 + n], hi = __bfloat162float(__float2bfloat16_rn(b));
    ntc_put_bf16(smem + S::o_b2, O1P, O0P, n, hi);
    ntc_put_bf16(smem + S::o_b2, O1P, O0P + 1, n, b - hi);
  }
  if (tid == 0) { mbar_init(barA, 1); mbar_init(barW, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(tmem_slot, 128);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
  {      // both weight-gradient accumulators (all 32 lanes of every quadrant, columns [64, 128)) start at zero
    uint32_t z[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) z[c] = 0u;
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 16) tmem_st16(lane_base + 64 + c0, z);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const uint32_t g0a = smem_u32(smem + S::o_g0), g1a = smem_u32(smem + S::o_g1), xa = smem_u32(smem + S::o_x), y0a = smem_u32(smem + S::o_y0);
  const uint32_t onesa = smem_u32(smem + S::o_ones), b1a = smem_u32(smem + S::o_b1), b2a = smem_u32(smem + S::o_b2);
  const uint32_t b3a = smem_u32(smem + S::o_b3), b4a = smem_u32(smem + S::o_b4);
  const bool vec = (ld & 3) == 0 && ((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(dh)) & 15) == 0;
  const bool vec_o = (O1 & 3) == 0 && (reinterpret_cast<uintptr_t>(dh_out) & 15) == 0;
  uint32_t phA = 0, phW = 0;
  bool pendingW = false;
  const int ntiles = (rows + 127) / 128;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * 128, row = row0 + tid;
    const bool live = row < rows;
    if (zero64) {      // the dP|dQ accumulator of the edge adjoint that follows (64 floats per row) starts at zero
      float4* z = reinterpret_cast<float4*>(zero64 + (size_t)row0 * 64);
      const int n4 = min(128, rows - row0) * 16;
      for (int idx = tid; idx < n4; idx += 128) z[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // ---- global loads of the tile: e and h as (row, slab) entries (a warp instruction covers whole rows), dh' per row ----
    float ev[2][8], hv[HS][8];
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int idx = it * 128 + tid, r = idx >> 1, sl = idx & 1;
      ntc_load8(e + (size_t)(row0 + r) * 16, 8 * sl, 16, 16, true, row0 + r < rows, ev[it]);
    }
#pragma unroll
    for (int it = 0; it < HS; ++it) {
      const int idx = it * 128 + tid, r = idx / HS, sl = idx - r * HS;
      ntc_load8(h + (size_t)(row0 + r) * ld, 8 * sl, cols, ld, vec, row0 + r < rows, hv[it]);
    }
    float dout[O1P];
#pragma unroll
    for (int q = 0; q < O1P; ++q) dout[q] = 0.f;
    if (live) {
      const float* src = dh_out + (size_t)row * O1;
      if (vec_o) {
#pragma unroll
        for (int q = 0; q < O1P; q += 4)
          if (q < O1) { const float4 a = __ldg(reinterpret_cast<const float4*>(src + q)); dout[q] = a.x; dout[q + 1] = a.y; dout[q + 2] = a.z; dout[q + 3] = a.w; }
      } else {
#pragma unroll
        for (int q = 0; q < O1P; ++q) if (q < O1) dout[q] = __ldg(src + q);
      }
    }
    if (pendingW) { mbar_wait(barW, phW); phW ^= 1u; pendingW = false; }      // the previous tile's weight-gradient MMAs have read every slab
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int idx = it * 128 + tid, r = idx >> 1, sl = idx & 1;
      *reinterpret_cast<uint4*>(smem + S::o_x + sl * 2048 + r * 16) = ntc_pack8(ev[it]);
    }
#pragma unroll
    for (int it = 0; it < HS; ++it) {
      const int idx = it * 128 + tid, r = idx / HS, sl = idx - r * HS;
      *reinterpret_cast<uint4*>(smem + S::o_x + (2 + sl) * 2048 + r * 16) = ntc_pack8(hv[it]);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {      // Y0 = [X | 1] [V0 | c0]^T
      tc_fence_after();
      const uint32_t id = make_idesc_bf16(128, O0P, 0, 0);
#pragma unroll
      for (int s = 0; s < I0P / 16; ++s)
        mma_bf16_ss_elect(tmem_base, make_smem_desc(xa + s * 4096, 2048, 128), make_smem_desc(b1a + s * 2 * O0P * 16, O0P * 16, 128), id, s > 0);
      mma_bf16_ss_elect(tmem_base, make_smem_desc(onesa, 2048, 128), make_smem_desc(b1a + (I0P / 16) * 2 * O0P * 16, O0P * 16, 128), id, 1u);
      mma_commit_elect(barA);
    }
    mbar_wait(barA, phA); phA ^= 1u;
    tc_fence_after();
    uint32_t mask0 = 0u;
#pragma unroll
    for (int c0 = 0; c0 < O0P; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + c0, v);
      tmem_ld_wait(); tmem_pin16(v);
      float y[16];
#pragma unroll
      for (int q = 0; q < 16; ++q) {
        const float f = __uint_as_float(v[q]);
        if (f > 0.f) mask0 |= 1u << (c0 + q);
        y[q] = fmaxf(f, alpha * f);
      }
      const float ylo[8] = {y[0], y[1], y[2], y[3], y[4], y[5], y[6], y[7]}, yhi[8] = {y[8], y[9], y[10], y[11], y[12], y[13], y[14], y[15]};
      *reinterpret_cast<uint4*>(smem + S::o_y0 + (c0 / 8) * 2048 + tid * 16) = ntc_pack8(ylo);
      *reinterpret_cast<uint4*>(smem + S::o_y0 + (c0 / 8 + 1) * 2048 + tid * 16) = ntc_pack8(yhi);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {      // Y1 = [y0 | 1] [V1 | c1]^T
      tc_fence_after();
      const uint32_t id = make_idesc_bf16(128, O1P, 0, 0);
#pragma unroll
      for (int s = 0; s < O0P / 16; ++s)
        mma_bf16_ss_elect(tmem_base + 32, make_smem_desc(y0a + s * 4096, 2048, 128), make_smem_desc(b2a + s * 2 * O1P * 16, O1P * 16, 128), id, s > 0);
      mma_bf16_ss_elect(tmem_base + 32, make_smem_desc(onesa, 2048, 128), make_smem_desc(b2a + (O0P / 16) * 2 * O1P * 16, O1P * 16, 128), id, 1u);
      mma_commit_elect(barA);
    }
    mbar_wait(barA, phA); phA ^= 1u;
    tc_fence_after();
#pragma unroll
    for (int c0 = 0; c0 < O1P; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + 32 + c0, v);
      tmem_ld_wait(); tmem_pin16(v);
      float g[16];
#pragma unroll
      for (int q = 0; q < 16; ++q) g[q] = dout[c0 + q] * (__uint_as_float(v[q]) > 0.f ? 1.f : alpha);
      const float glo[8] = {g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7]}, ghi[8] = {g[8], g[9], g[10], g[11], g[12], g[13], g[14], g[15]};
      *reinterpret_cast<uint4*>(smem + S::o_g1 + (c0 / 8) * 2048 + tid * 16) = ntc_pack8(glo);
      *reinterpret_cast<uint4*>(smem + S::o_g1 + (c0 / 8 + 1) * 2048 + tid * 16) = ntc_pack8(ghi);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {      // G0 = g1 V1, then [dV1 | dc1] += g1^T [y0 | 1] behind it
      tc_fence_after();
      const uint32_t id = make_idesc_bf16(128, O0P, 0, 0);
#pragma unroll
      for (int s = 0; s < O1P / 16; ++s)
        mma_bf16_ss_elect(tmem_base + 32, make_smem_desc(g1a + s * 4096, 2048, 128), make_smem_desc(b3a + s * 2 * O0P * 16, O0P * 16, 128), id, s > 0);
      mma_commit_elect(barA);
      const uint32_t iw = make_idesc_bf16(64, O0P, 1, 1), ib = make_idesc_bf16(64, 16, 1, 1);
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        mma_bf16_ss_elect(tmem_base + 64 + (16u << 16), make_smem_desc(g1a + s * 256, 128, 2048), make_smem_desc(y0a + s * 256, 128, 2048), iw, 1u);
        mma_bf16_ss_elect(tmem_base + 64 + O0P + (16u << 16), make_smem_desc(g1a + s * 256, 128, 2048), make_smem_desc(onesa + s * 256, 128, 2048), ib, 1u);
      }
    }
    mbar_wait(barA, phA); phA ^= 1u;
    tc_fence_after();
#pragma unroll
    for (int c0 = 0; c0 < O0P; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + 32 + c0, v);
      tmem_ld_wait(); tmem_pin16(v);
      float g[16];
#pragma unroll
      for (int q = 0; q < 16; ++q) g[q] = __uint_as_float(v[q]) * (((mask0 >> (c0 + q)) & 1u) ? 1.f : alpha);
      const float glo[8] = {g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7]}, ghi[8] = {g[8], g[9], g[10], g[11], g[12], g[13], g[14], g[15]};
      *reinterpret_cast<uint4*>(smem + S::o_g0 + (c0 / 8) * 2048 + tid * 16) = ntc_pack8(glo);
      *reinterpret_cast<uint4*>(smem + S::o_g0 + (c0 / 8 + 1) * 2048 + tid * 16) = ntc_pack8(ghi);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {      // DX = g0 V0, then [dV0 | dc0] += g0^T [X | 1] behind it
      tc_fence_after();
      const uint32_t id = make_idesc_bf16(128, I0P, 0, 0);
#pragma unroll
      for (int s = 0; s < O0P / 16; ++s)
        mma_bf16_ss_elect(tmem_base, make_smem_desc(g0a + s * 4096, 2048, 128), make_smem_desc(b4a + s * 2 * I0P * 16, I0P * 16, 128), id, s > 0);
      mma_commit_elect(barA);
      const uint32_t iw = make_idesc_bf16(64, I0P, 1, 1), ib = make_idesc_bf16(64, 16, 1, 1);
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        mma_bf16_ss_elect(tmem_base + 64, make_smem_desc(g0a + s * 256, 128, 2048), make_smem_desc(xa + s * 256, 128, 2048), iw, 1u);
        mma_bf16_ss_elect(tmem_base + 64 + I0P, make_smem_desc(g0a + s * 256, 128, 2048), make_smem_desc(onesa + s * 256, 128, 2048), ib, 1u);
      }
      mma_commit_elect(barW);
    }
    pendingW = true;
    mbar_wait(barA, phA); phA ^= 1u;
    tc_fence_after();
    // ---- DX -> de | dh ----
#pragma unroll
    for (int c0 = 0; c0 < I0P; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + c0, v);
      tmem_ld_wait(); tmem_pin16(v);
      if (live) {
        if (c0 == 0) {
          float4* dst = reinterpret_cast<float4*>(de + (size_t)row * 16);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            dst[q] = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        } else {
          float* dst = dh + (size_t)row * ld + (c0 - 16);
#pragma unroll
          for (int q = 0; q < 16; q += 4) {
            const int k = c0 - 16 + q;
            if (vec && k + 3 < cols)
              *reinterpret_cast<float4*>(dst + q) = make_float4(__uint_as_float(v[q]), __uint_as_float(v[q + 1]), __uint_as_float(v[q + 2]), __uint_as_float(v[q + 3]));
            else {
#pragma unroll
              for (int u = 0; u < 4; ++u) if (k + u < cols) dst[q + u] = __uint_as_float(v[q + u]);
            }
          }
        }
      }
    }
    tc_fence_before();
    __syncthreads();      // DX has been read back: the next tile's first GEMM may overwrite the chain accumulators
  }
  if (pendingW) { mbar_wait(barW, phW); }
  // ---- gradient read-out: lanes 0..15 of a quadrant hold dV0 | dc0 channels, lanes 16..31 dV1 | dc1 channels ----
  tc_fence_after();
  float* out = part + (size_t)blockIdx.x * n_node_params;
  {
    const int o = warp * 16 + (lane & 15);      // output channel (quadrants 2, 3 hold the unused rows 32..63)
    const bool first = lane < 16;
    const int K = first ? I0 : O0, KPad = first ? I0P : O0P, O = first ? O0 : O1;
    float* wrow = out + (first ? o * I0 : O0 * I0 + O0 + o * O0);
    float* brow = out + (first ? O0 * I0 : O0 * I0 + O0 + O1 * O0);
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lane_base + 64 + c0, v);      // .aligned: every lane issues the load
      tmem_ld_wait(); tmem_pin16(v);
      if (warp < 2 && o < O) {
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const int k = c0 + q;
          if (k < K) wrow[k] = __uint_as_float(v[q]);
          if (k == KPad) brow[o] = __uint_as_float(v[q]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 128);
}

}  // namespace

int gj_num_sms();
void gj_set_error(const char* fmt, ...);

bool gj_node_pre_bwd_tc_supported(const MPLayout& L) { return L.E[0] == 32 && L.E0p == 32 && L.cols <= 32; }
static int pre_bwd_tc_grid(const MPLayout& L) {      // every CTA gets the same number of tiles (+-1) with 3-4 CTAs per SM resident
  const int tiles = (L.B * L.N + 127) / 128, cap = (L.cols <= 16 ? 4 : 3) * gj_num_sms();
  if (tiles <= cap) return tiles > 0 ? tiles : 1;
  const int rounds = (tiles + cap - 1) / cap;
  return (tiles + rounds - 1) / rounds;
}
// per-CTA partials [Wa grads 32*H][Wb grads 32*H][b0 grads 32], reduced by reduce_pre_partials_kernel
size_t gj_node_pre_bwd_tc_ws_floats(const MPLayout& L) { return (size_t)pre_bwd_tc_grid(L) * (64 * L.H + 32); }

int gj_node_pre_bwd_tc_nparts(const MPLayout& L) { return pre_bwd_tc_grid(L); }

// launches the kernel; *nparts receives the number of per-CTA partials written to `part`
int gj_node_pre_bwd_tc(const MPLayout& L, const float* h, const float* params, const float* dpq, float* dh, float* part, int* nparts,
                       cudaStream_t st) {
  const int grid = pre_bwd_tc_grid(L), rows = L.B * L.N;
  *nparts = grid;
  cudaError_t ce;
  if (L.cols <= 16) {
    using S = PreBwdSmem<16>;
    ce = cudaFuncSetAttribute(node_pre_bwd_tc_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::total);
    if (ce == cudaSuccess) gj_launch(node_pre_bwd_tc_kernel<16>, grid, 128, S::total, st, rows, L.H, L.cols, L.ld, L.K[0], h, params + L.pW[0], dpq, dh, part);
  } else {
    using S = PreBwdSmem<32>;
    ce = cudaFuncSetAttribute(node_pre_bwd_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::total);
    if (ce == cudaSuccess) gj_launch(node_pre_bwd_tc_kernel<32>, grid, 128, S::total, st, rows, L.H, L.cols, L.ld, L.K[0], h, params + L.pW[0], dpq, dh, part);
  }
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) { gj_set_error("node_pre_bwd_tc launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}

// ---- node MLP adjoint on tcgen05 ----
static int post_tc_shape(const MPLayout& L) {      // index of the compiled (I0P, O0P, O1P) combination, -1 if none
  if (!(L.Ln == 2 && L.EL == 16 && L.alpha <= 1.f && L.cols <= L.H && L.I[0] == 16 + L.H)) return -1;
  const int i0p = (L.I[0] + 15) & ~15, o0p = (L.O[0] + 15) & ~15, o1p = (L.O[1] + 15) & ~15;
  if (i0p == 32 && o0p == 16 && o1p == 32) return 0;
  if (i0p == 48 && o0p == 32 && o1p == 16) return 1;
  if (i0p == 32 && o0p == 16 && o1p == 16) return 2;
  if (i0p == 48 && o0p == 32 && o1p == 32) return 3;
  return -1;
}
bool gj_node_post_bwd_tc_supported(const MPLayout& L) { return post_tc_shape(L) >= 0; }
static int post_bwd_tc_grid(const MPLayout& L) {
  const int tiles = (L.B * L.N + 127) / 128, cap = 4 * gj_num_sms();
  if (tiles <= cap) return tiles > 0 ? tiles : 1;
  const int rounds = (tiles + cap - 1) / cap;
  return (tiles + rounds - 1) / rounds;
}
size_t gj_node_post_bwd_tc_ws_floats(const MPLayout& L) { return (size_t)post_bwd_tc_grid(L) * (L.nparams - L.pV[0]); }

int gj_node_post_bwd_tc_nparts(const MPLayout& L) { return post_bwd_tc_grid(L); }

template <int I0P, int O0P, int O1P>
static cudaError_t post_bwd_tc_launch(const MPLayout& L, int grid, const float* e, const float* h, const float* params, const float* dh_out,
                                      float* de, float* dh, float* part, float* zero64, cudaStream_t st) {
  using S = PostBwdSmem<I0P, O0P, O1P>;
  cudaError_t ce = cudaFuncSetAttribute(node_post_bwd_tc_kernel<I0P, O0P, O1P>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::total);
  if (ce != cudaSuccess) return ce;
  gj_launch(node_post_bwd_tc_kernel<I0P, O0P, O1P>, grid, 128, S::total, st, L.B * L.N, L.cols, L.ld, L.I[0], L.O[0], L.O[1], L.alpha,
            L.nparams - L.pV[0], e, h, params + L.pV[0], params + L.pc[0], params + L.pV[1], params + L.pc[1], dh_out, de, dh, part, zero64);
  return cudaGetLastError();
}

// launches the kernel; *nparts receives the number of per-CTA partials (packed [V0 | c0 | V1 | c1]) written to `part`;
// zero64 (optional): a (rows, 64) buffer the kernel clears on the way (the edge adjoint's dP|dQ accumulator)
int gj_node_post_bwd_tc(const MPLayout& L, const float* e, const float* h, const float* params, const float* dh_out, float* de, float* dh,
                        float* part, int* nparts, float* zero64, cudaStream_t st) {
  const int grid = post_bwd_tc_grid(L), shape = post_tc_shape(L);
  *nparts = grid;
  cudaError_t ce = shape == 0 ? post_bwd_tc_launch<32, 16, 32>(L, grid, e, h, params, dh_out, de, dh, part, zero64, st)
                 : shape == 1 ? post_bwd_tc_launch<48, 32, 16>(L, grid, e, h, params, dh_out, de, dh, part, zero64, st)
                 : shape == 2 ? post_bwd_tc_launch<32, 16, 16>(L, grid, e, h, params, dh_out, de, dh, part, zero64, st)
                 : shape == 3 ? post_bwd_tc_launch<48, 32, 32>(L, grid, e, h, params, dh_out, de, dh, part, zero64, st)
                              : cudaErrorInvalidValue;
  if (ce != cudaSuccess) { gj_set_error("node_post_bwd_tc launch: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  return GJ_OK;
}
