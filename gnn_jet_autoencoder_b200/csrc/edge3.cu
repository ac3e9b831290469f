// Third-generation fused edge kernels (GJ_PREC_BF16): TWO-layer edge networks [E0, E1] with compile-time widths, the shape of
// BASELINE config 5's deep / wide sweep (edge_sizes [[H, H]], node_sizes [[H]]; instantiated for H = 64 and H = 128).
//
// Replaces the edge part of one iteration of reference models/graphnet.py:154-168 (_getA :186-223, _edge_conv :273-289, the
// sum over j of _concat :243) and its adjoint.  With the first layer factorised (W0 [h_i | h_j | d] = Wa h_i + Wb h_j + wd d,
// graphnet.py:220) only ONE dense product per edge row is left:
//   a0 = leaky(P_i + Q_j + wd d_ij)          CUDA cores (P, Q from the node-level projections, d from pair_dist_fwd)
//   a1 = leaky(W1 a0 + b1)                   tcgen05.mma, bias as one extra k-step
//   e_i = sum_j a1                           warp transpose-reduce
// Decomposition as in edge_fwd2.cu: a warp owns a (jet, 32-wide j block), lane = j, and walks i; four warps (one TMEM lane
// quadrant each, possibly four jets) form a tile group of 128 edge rows.
//
// Forward: a0 goes straight to TENSOR MEMORY as the A operand (tcgen05.st, double buffered so that the next tile's first layer
// runs behind the current GEMM), W1 (bf16, K-major) is resident in shared memory.
// Backward (recompute + dgrad + wgrad per tile): a0 and dz1 are staged in shared memory in the UMMA slab layout, which serves the
// forward / dgrad GEMMs (K-major view) and the weight-gradient GEMM (MN-major view, K = tile row) alike; [dW1 | db1]
// accumulates in TMEM for the whole kernel.  The first-layer adjoint needs per-thread accumulators for dQ_j and d(wd) -- E0
// each -- so a row's channels are SPLIT over S threads (S warps share a TMEM lane quadrant): S = 1 for E0 = 64, 2 for 128.
#include <stdlib.h>

#include "tc2_common.cuh"
#include "tma.cuh"

namespace {
using namespace tc2;

__device__ __forceinline__ void e3_cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void e3_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void e3_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// transpose-reduce of 16 per-lane values over the 32 lanes of a warp: every lane returns the sum over all lanes of
// channel (lane >> 1) & 15
__device__ __forceinline__ float e3_transpose_sum16(const float (&v)[16], int lane) {
  float w8[8], w4[4], w2[2];
  bool up = lane & 16;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float send = up ? v[q] : v[q + 8], keep = up ? v[q + 8] : v[q];
    w8[q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  up = lane & 8;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float send = up ? w8[q] : w8[q + 4], keep = up ? w8[q + 4] : w8[q];
    w4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  up = lane & 4;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const float send = up ? w4[q] : w4[q + 2], keep = up ? w4[q + 2] : w4[q];
    w2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  up = lane & 2;
  const float send = up ? w2[0] : w2[1], keep = up ? w2[1] : w2[0];
  const float w1 = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  return w1 + __shfl_xor_sync(0xffffffffu, w1, 1);
}

// ---- packed image of the step's dense edge layer: [b1: per out feature (b_hi, b_lo, 0 x 6) bf16][W1: bf16 K-major] ----
template <int E0, int E1>
struct WImage3 {
  static constexpr int o_b1 = 0;
  static constexpr int o_w1 = ((E1 * 16 + 1023) / 1024) * 1024;
  static constexpr int bytes = o_w1 + E1 * E0 * 2;
};
template <int E0, int E1>
__global__ void __launch_bounds__(256) pack3_kernel(const float* __restrict__ params, int pW1, int pb1, uint8_t* __restrict__ img) {
  using I = WImage3<E0, E1>;
  const int tid = blockIdx.x * 256 + threadIdx.x, nthr = gridDim.x * 256;
  for (int idx = tid; idx < (I::o_w1 - E1 * 16) / 4; idx += nthr) reinterpret_cast<uint32_t*>(img + E1 * 16)[idx] = 0u;
  pack_bias_chunk<E1>(img + I::o_b1, params + pb1, tid, nthr);
  if (((reinterpret_cast<uintptr_t>(params) | (uintptr_t)(pW1 * 4)) & 15) == 0) pack_weight_kmajor<E1, E0>(img + I::o_w1, params + pW1, tid, nthr);
  else pack_weight_kmajor_unaligned<E1, E0>(img + I::o_w1, params + pW1, tid, nthr);
}

struct E3Args {
  const float* pq; const float* d; const float* params; const uint8_t* wimg;
  float* e_out;                                                // forward: (per-j-block partial) edge aggregates
  const float* de; float* dpq; float* dp_part; float* G; float* part;      // backward
  int B, N, NJB, NJ32;
  int pW1, pb1, pWd, K0, nedge;
  float alpha;
  int tiles_total, ngroups;
};

// =====================================================================================================================
// forward
// =====================================================================================================================
template <int E0, int E1, int NWG, int IC>
struct Fwd3Smem {
  static constexpr int o_bar = 0;                       // NWG mbarriers
  static constexpr int o_slot = 128;
  static constexpr int o_wd = 256;                      // E0 floats
  static constexpr int o_img = 1024;
  static constexpr int o_b1 = o_img + WImage3<E0, E1>::o_b1;
  static constexpr int o_w1 = o_img + WImage3<E0, E1>::o_w1;
  static constexpr int o_ones = o_img + WImage3<E0, E1>::bytes;      // [128][8] (1, 1, 0, ...) then [128][8] zeros (second k-chunk of the bias operands)
  static constexpr int o_warp = o_ones + 4096;
  static constexpr int warp_bytes = 2 * IC * E0 * 4;    // P_i chunks, double buffered
  static constexpr int total = o_warp + NWG * 4 * warp_bytes;
  static_assert(E1 * 16 <= 2048, "the zero chunk behind the ones chunk doubles as the second k-chunk of the bias B operand");
};

template <int E0, int E1, int NWG, int IC>
__global__ void __launch_bounds__(NWG * 128, 1) edge_fwd3_kernel(const E3Args A, const __grid_constant__ CUtensorMap tm_w) {
  static_assert(E0 % 16 == 0 && E1 % 16 == 0 && E0 <= 128 && E1 <= 128, "widths");
  constexpr int SLOT = E0 + E1;      // TMEM columns of a tile group: two packed a0 buffers (E0 / 2 each), then the accumulator
  static_assert(NWG * SLOT <= 512, "TMEM columns");
  using S = Fwd3Smem<E0, E1, NWG, IC>;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = (int)uni((uint32_t)(tid >> 5));
  const int wg = warp >> 2, wq = warp & 3;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::o_bar) + wg;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::o_slot);
  float* s_wd = reinterpret_cast<float*>(smem + S::o_wd);

  for (int c = tid; c < E0; c += NWG * 128) s_wd[c] = __ldg(A.params + A.pWd + c * A.K0);
  for (int idx = tid; idx < 1024; idx += NWG * 128)
    reinterpret_cast<uint32_t*>(smem + S::o_ones)[idx] = (idx < 512 && (idx & 3) == 0) ? 0x3F803F80u : 0u;
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(smem + S::o_bar) + 15;      // byte 120: the parameter image (TMA) has landed
  static_assert(NWG <= 15, "mbarrier slots");
  if (tid == 0) {
    for (int b = 0; b < NWG; ++b) mbar_init(reinterpret_cast<uint64_t*>(smem + S::o_bar) + b, 1);
    mbar_init(bar_w, 1);
    fence_barrier_init();
    tma::prefetch_map(&tm_w);
    tma::mbar_expect_tx(bar_w, WImage3<E0, E1>::bytes);
    tma::load_2d(smem + S::o_img, &tm_w, 0, 0, bar_w);
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  mbar_wait(bar_w, 0u);
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t slot = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(wg * SLOT);
  const uint32_t slot0 = tmem_base + (uint32_t)(wg * SLOT);
  const uint32_t acc = slot + E0, acc0 = slot0 + E0;
  const __nv_bfloat162 alpha2 = __float2bfloat162_rn(A.alpha);
  const float alpha = A.alpha;

  const uint32_t idesc = make_idesc_bf16(128, E1, 0, 0);
  const uint64_t dW1 = wdesc_kmajor(smem_u32(smem + S::o_w1), E1);
  const uint32_t zero_a = smem_u32(smem + S::o_ones + 2048);
  const uint64_t dB1 = make_smem_desc(smem_u32(smem + S::o_b1), zero_a - smem_u32(smem + S::o_b1), 128);
  const uint64_t dOnes = make_smem_desc(smem_u32(smem + S::o_ones), 2048, 128);

  float* s_pi = reinterpret_cast<float*>(smem + S::o_warp + warp * S::warp_bytes);      // [2][IC][E0]

  const int ngroups = gridDim.x * NWG, gidx = blockIdx.x * NWG + wg;
  const long long T = A.tiles_total;
  const int g0 = (int)(T * gidx / ngroups), g1 = (int)(T * (gidx + 1) / ngroups);
  const int N = A.N, ntasks = A.B * A.NJB;
  int k = g0 / N, i = g0 - k * N;
  bool fresh = true, p_active = false, p_valid = false;
  uint32_t p_vmask = 0u;      // lanes (j) of the warp's j block that are real particles
  uint32_t q[E0 / 2];      // Q_j as bf16 pairs
  size_t node0 = 0;
  float* e_dst = nullptr;
  int jb = 0;
  float d_cur = 0.f;

  auto stage_chunk = [&](int c) {
    const int ib = c * IC, n = min(IC, N - ib);
    float* dst = s_pi + (c & 1) * IC * E0;
    for (int idx = lane; idx < n * (E0 / 4); idx += 32) {
      const int r = idx / (E0 / 4), c4 = idx - r * (E0 / 4);
      e3_cp_async16(dst + r * E0 + 4 * c4, A.pq + (node0 + ib + r) * (2 * E0) + 4 * c4);
    }
    e3_cp_async_commit();
  };

  // first edge layer of tile (k, i) -> packed bf16 pairs in TMEM buffer `buf`; advances (k, i)
  auto prepare = [&](int buf, bool& t_active, bool& t_valid, float*& t_erow, uint32_t& t_vmask) {
    if (fresh) {
      const int task = 4 * k + wq;
      p_active = task < ntasks;
      const int tk = p_active ? task : 0;
      const int jet = tk / A.NJB;
      jb = tk - jet * A.NJB;
      const int j = jb * 32 + lane;
      p_valid = p_active && j < N;
      p_vmask = __ballot_sync(0xffffffffu, p_valid);
      node0 = (size_t)jet * N;
      e_dst = A.e_out + ((size_t)jb * A.B + jet) * N * E1;
      e3_cp_async_wait<0>();
      __syncwarp();
      stage_chunk(i / IC);
      if ((i / IC + 1) * IC < N) stage_chunk(i / IC + 1);
      if (j < N) {
        const float4* src = reinterpret_cast<const float4*>(A.pq + (node0 + j) * (2 * E0) + E0);
#pragma unroll
        for (int c = 0; c < E0 / 4; ++c) {
          const float4 v = __ldg(src + c);
          q[2 * c] = bf2_as_u32(__floats2bfloat162_rn(v.x, v.y)); q[2 * c + 1] = bf2_as_u32(__floats2bfloat162_rn(v.z, v.w));
        }
      } else {
#pragma unroll
        for (int c = 0; c < E0 / 2; ++c) q[c] = 0u;
      }
      d_cur = __ldg(A.d + (node0 + i) * A.NJ32 + jb * 32 + lane);
      if ((i / IC + 1) * IC < N) e3_cp_async_wait<1>(); else e3_cp_async_wait<0>();
      __syncwarp();
    } else if ((i % IC) == 0) {
      e3_cp_async_wait<0>();
      __syncwarp();
      if ((i / IC + 1) * IC < N) stage_chunk(i / IC + 1);
    }
    fresh = false;
    const float dij = d_cur;
    if (i + 1 < N) d_cur = __ldg(A.d + (node0 + i + 1) * A.NJ32 + jb * 32 + lane);
    {
      const float* Pi = s_pi + (((i / IC) & 1) * IC + (i % IC)) * E0;
      const float2 d2 = make_float2(dij, dij);
      const uint32_t dst = slot + (uint32_t)(buf * (E0 / 2));
#pragma unroll
      for (int c = 0; c < E0; c += 16) {
        uint32_t o[8];
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) {
          const int cc = c + 4 * hh;
          const float4 p = *reinterpret_cast<const float4*>(Pi + cc);
          const float4 w = *reinterpret_cast<const float4*>(s_wd + cc);
          const float2 z0 = fma2(make_float2(w.x, w.y), d2, add2(make_float2(p.x, p.y), unpack_bf2(q[cc / 2])));
          const float2 z1 = fma2(make_float2(w.z, w.w), d2, add2(make_float2(p.z, p.w), unpack_bf2(q[cc / 2 + 1])));
          o[2 * hh] = leaky_pack(z0.x, z0.y, alpha2);
          o[2 * hh + 1] = leaky_pack(z1.x, z1.y, alpha2);
        }
        tmem_st8(dst + (uint32_t)(c / 2), o);
      }
      tmem_st_wait();
    }
    t_active = p_active; t_valid = p_valid; t_erow = e_dst + (size_t)i * E1; t_vmask = p_vmask;
    if (++i == N) { i = 0; ++k; fresh = true; }
  };

  uint32_t ph = 0;
  bool n_active = false, n_valid = false;
  float* n_erow = nullptr;
  uint32_t n_vmask = 0u;
  if (g0 < g1) prepare(0, n_active, n_valid, n_erow, n_vmask);

  for (int g = g0; g < g1; ++g) {
    const int buf = (g - g0) & 1;
    const bool active = n_active, valid = n_valid;
    float* const erow = n_erow;
    const uint32_t valid_mask = n_vmask;
    tc_fence_before();
    named_bar_sync(1 + wg, 128);      // the group's a0 rows are in TMEM; the previous tile's accumulator has been read
    if (wq == 0) {
      tc_fence_after();
#pragma unroll
      for (int s = 0; s < E0 / 16; ++s)
        mma_ts_elect(acc0, slot0 + (uint32_t)(buf * (E0 / 2) + 8 * s), dW1 + (uint64_t)(s * ((2 * E1 * 16) >> 4)), idesc, s > 0);
      mma_bf16_ss_elect(acc0, dOnes, dB1, idesc, 1u);
      mma_commit_elect(bar);
    }
    if (g + 1 < g1) prepare(buf ^ 1, n_active, n_valid, n_erow, n_vmask);      // behind the GEMM
    mbar_wait(bar, ph);
    tc_fence_after();
    // e_i = sum over the quadrant's 32 lanes (j) of leaky(acc), padded rows masked: the accumulator is read as matrix fragments
    // (tmem_ld_frag16: this thread holds lanes g, g + 8, g + 16, g + 24, g = lane / 4, of columns 2q, 2q + 1, 8 + 2q, 9 + 2q of each
    // 16-column chunk), so the sum is local adds and three shuffle rounds over g per chunk
    {
      const uint32_t vm = valid_mask >> (lane >> 2);
      const float m0 = (vm & 1u) ? 1.f : 0.f, m1 = (vm & 0x100u) ? 1.f : 0.f, m2 = (vm & 0x10000u) ? 1.f : 0.f, m3 = (vm & 0x1000000u) ? 1.f : 0.f;
      uint32_t fa[2][8], fb[2][8];
      tmem_ld_frag16(acc, fa[0]);
      tmem_ld_frag16(acc + (16u << 16), fb[0]);
#pragma unroll
      for (int c0 = 0; c0 < E1; c0 += 16) {
        const int cur = (c0 >> 4) & 1;
        tmem_ld_wait(); tmem_pin8(fa[cur]); tmem_pin8(fb[cur]);
        if (c0 + 16 < E1) {
          tmem_ld_frag16(acc + (uint32_t)(c0 + 16), fa[cur ^ 1]);
          tmem_ld_frag16(acc + (uint32_t)(c0 + 16) + (16u << 16), fb[cur ^ 1]);
        }
        float s[4];
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const float z0 = __uint_as_float(fa[cur][4 * kk + c]) * m0, z1 = __uint_as_float(fa[cur][4 * kk + 2 + c]) * m1;
            const float z2 = __uint_as_float(fb[cur][4 * kk + c]) * m2, z3 = __uint_as_float(fb[cur][4 * kk + 2 + c]) * m3;
            s[2 * kk + c] = (fmaxf(z0, alpha * z0) + fmaxf(z1, alpha * z1)) + (fmaxf(z2, alpha * z2) + fmaxf(z3, alpha * z3));
          }
        }
#pragma unroll
        for (int off = 4; off < 32; off <<= 1) {
#pragma unroll
          for (int c = 0; c < 4; ++c) s[c] += __shfl_xor_sync(0xffffffffu, s[c], off);
        }
        if (active && lane < 4) {
          *reinterpret_cast<float2*>(erow + c0 + 2 * lane) = make_float2(s[0], s[1]);
          *reinterpret_cast<float2*>(erow + c0 + 8 + 2 * lane) = make_float2(s[2], s[3]);
        }
      }
    }
    ph ^= 1u;
  }
  e3_cp_async_wait<0>();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// e_i = sum over the j blocks' partial aggregates (N > 32), fixed order
__global__ void __launch_bounds__(256) e3_sum_jblocks_kernel(const float4* __restrict__ part, int njb, size_t n4, float4* __restrict__ out) {
  const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (idx >= n4) return;
  float4 s = __ldg(part + idx);
  for (int b = 1; b < njb; ++b) {
    const float4 v = __ldg(part + b * n4 + idx);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  out[idx] = s;
}

// =====================================================================================================================
// backward
// =====================================================================================================================
template <int E0, int E1, int NWG, int S, int IC>
struct Bwd3Smem {
  static constexpr int C0 = E0 / S, C1 = E1 / S;
  static constexpr int o_bar = 0;                        // per group: done[2], doneW[2]
  static constexpr int o_slot = 128;
  static constexpr int o_wd = 256;                       // E0 floats
  static constexpr int o_img = 1024;
  static constexpr int o_b1 = o_img + WImage3<E0, E1>::o_b1;
  static constexpr int o_w1 = o_img + WImage3<E0, E1>::o_w1;
  static constexpr int o_grp = ((o_img + WImage3<E0, E1>::bytes + 1023) / 1024) * 1024;
  // per group and tile slot: A0 = [a0: E0 / 8 slabs][ones slab][zero slab], D1 = [dz1: E1 / 8 slabs]
  static constexpr int t_a0 = 0;
  static constexpr int t_ones = (E0 / 8) * 2048;
  static constexpr int t_d1 = t_ones + 4096;
  static constexpr int tile_bytes = t_d1 + (E1 / 8) * 2048;
  static constexpr int g_gs = 2 * tile_bytes;            // [S][128] floats: the G partials of the upper channel parts
  static constexpr int grp_bytes = g_gs + S * 128 * 4;
  static constexpr int o_warp = o_grp + NWG * grp_bytes;
  static constexpr int warp_bytes = 2 * IC * (C0 + C1) * 4;      // this warp's channel part of P_i and de_i, double buffered
  static constexpr int o_red = o_warp + NWG * S * 4 * warp_bytes;      // [warps][C0] floats: d(wd) partials
  static constexpr int o_zero = ((o_red + NWG * S * 4 * C0 * 4 + 127) / 128) * 128;      // [128][8] zeros: second k-chunk of the bias operands
  static constexpr int total = o_zero + 2048;                                            // (last, so that descriptor strides to it are positive)
};

// Two tiles of a group are in flight (slots 0 / 1: private A0 / D1 slabs, TMEM accumulator and barriers), handled by the SAME
// threads in the order  E1(t) -> L0(t + 1) -> E0(t): the GEMMs of one tile run on the tensor pipe while the CUDA cores work on
// the other, and the per-thread dQ_j / d(wd) accumulators are shared (consecutive tiles are consecutive i of the same j).
struct E3Slot {
  bool active, valid, last_i, pendW;
  int i, jb, slot;
  size_t node0;
  float dij;
  const float* st;      // staged [P_i part | de_i part] of the tile
};

template <int E0, int E1, int NWG, int S, int IC>
__global__ void __launch_bounds__(NWG * S * 128, 1) edge_bwd3_kernel(const E3Args A, const __grid_constant__ CUtensorMap tm_w) {
  using SM = Bwd3Smem<E0, E1, NWG, S, IC>;
  constexpr int C0 = SM::C0, C1 = SM::C1;
  static_assert(C0 % 16 == 0 && C1 % 16 == 0 && E0 <= 128 && E1 <= 128 && (E1 == 64 || E1 == 128), "widths");
  constexpr int ACC = E0 > E1 ? E0 : E1;           // TMEM columns of a tile slot: F1 accumulator, then (same columns) the dgrad accumulator
  constexpr int GW = NWG * 2 * ACC;                // first column of the [dW1 | db1] accumulator (E0 + 16 columns)
  static_assert(GW + E0 + 16 <= 512, "TMEM columns");
  constexpr int TCOLS = GW + E0 + 16 <= 256 ? 256 : 512;
  constexpr int NT = NWG * S * 128, GT = S * 128;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = (int)uni((uint32_t)(tid >> 5));
  const int wg = warp / (4 * S), wl = warp - wg * 4 * S;      // group, warp within the group
  const int wq = wl & 3, part = wl >> 2;                       // TMEM lane quadrant (= task of the tile), channel part
  const int row = wq * 32 + lane;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::o_bar) + 4 * wg;      // done[0], done[1], doneW[0], doneW[1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM::o_slot);
  float* s_wd = reinterpret_cast<float*>(smem + SM::o_wd);
  float* s_red = reinterpret_cast<float*>(smem + SM::o_red);

  for (int idx = tid; idx < 512; idx += NT) reinterpret_cast<uint32_t*>(smem + SM::o_zero)[idx] = 0u;
  for (int c = tid; c < E0; c += NT) s_wd[c] = __ldg(A.params + A.pWd + c * A.K0);
  for (int idx = tid; idx < NWG * 2 * 1024; idx += NT) {      // ones slab (channels E0, E0 + 1 = 1.0: bias hi + lo) and zero slab of every tile slot
    const int gs = idx >> 10, w = idx & 1023;
    reinterpret_cast<uint32_t*>(smem + SM::o_grp + (gs >> 1) * SM::grp_bytes + (gs & 1) * SM::tile_bytes + SM::t_ones)[w] =
        (w < 512 && (w & 3) == 0) ? 0x3F803F80u : 0u;
  }
  for (int idx = tid; idx < NWG * 2 * (E1 / 8) * 512; idx += NT) {      // dz1 slabs start finite
    const int gs = idx / ((E1 / 8) * 512), w = idx - gs * ((E1 / 8) * 512);
    reinterpret_cast<uint32_t*>(smem + SM::o_grp + (gs >> 1) * SM::grp_bytes + (gs & 1) * SM::tile_bytes + SM::t_d1)[w] = 0u;
  }
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(smem + SM::o_bar) + 15;      // byte 120: the parameter image (TMA) has landed
  static_assert(4 * NWG <= 15, "mbarrier slots");
  if (tid == 0) {
    for (int b = 0; b < 4 * NWG; ++b) mbar_init(reinterpret_cast<uint64_t*>(smem + SM::o_bar) + b, 1);
    mbar_init(bar_w, 1);
    fence_barrier_init();
    tma::prefetch_map(&tm_w);
    tma::mbar_expect_tx(bar_w, WImage3<E0, E1>::bytes);
    tma::load_2d(smem + SM::o_img, &tm_w, 0, 0, bar_w);
  }
  if (warp == 0) tmem_alloc(tmem_slot, TCOLS);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  mbar_wait(bar_w, 0u);
  const uint32_t tmem_base = *tmem_slot;
  if (warp < 4) {      // the shared gradient accumulator starts at zero: every weight-gradient MMA accumulates
    uint32_t z[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) z[c] = 0u;
#pragma unroll
    for (int c0 = 0; c0 < E0 + 16; c0 += 16) tmem_st16(tmem_base + ((uint32_t)(warp * 32) << 16) + GW + c0, z);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const long long T = A.tiles_total;
  const int N = A.N;
  auto range_lo = [&](int g) { return g < A.ngroups ? (int)(T * g / A.ngroups) : (int)T; };

  const uint32_t smem0 = smem_u32(smem);
  const uint32_t w1a = smem0 + SM::o_w1, b1a = smem0 + SM::o_b1, zero_a = smem0 + SM::o_zero;
  uint8_t* gb = smem + SM::o_grp + wg * SM::grp_bytes;
  float* s_g = reinterpret_cast<float*>(gb + SM::g_gs);
  float* s_st = reinterpret_cast<float*>(smem + SM::o_warp + warp * SM::warp_bytes);      // [2][IC][C0 + C1]
  const __nv_bfloat162 alpha2 = __float2bfloat162_rn(A.alpha);
  const float alpha = A.alpha;
  const int gidx = blockIdx.x * NWG + wg;
  const int g0 = range_lo(gidx), g1 = range_lo(gidx + 1);
  const int ntasks = A.B * A.NJB;
  // ---- cursor over the (task, i) tile list: advanced by L0 ----
  int k = g0 / N, i = g0 - k * N;
  bool fresh = true, c_active = false, c_valid = false;
  size_t node0 = 0;
  int jb = 0;
  uint32_t q[C0 / 2];
  float dq[C0], dwd[C0];
#pragma unroll
  for (int c = 0; c < C0; ++c) { dq[c] = 0.f; dwd[c] = 0.f; }
#pragma unroll
  for (int c = 0; c < C0 / 2; ++c) q[c] = 0u;
  float d_cur = 0.f;
  uint32_t ph_bits = 0u;      // bit s: parity of done[s]; bit 2 + s: parity of doneW[s] (phases belong to the slot, not to the record)

  auto stage_chunk = [&](int c) {      // this warp's channel parts of P_i and de_i for i in [c IC, ...) -> buffer c & 1
    const int ib = c * IC, n = min(IC, N - ib);
    float* dst = s_st + (c & 1) * IC * (C0 + C1);
    for (int idx = lane; idx < n * ((C0 + C1) / 4); idx += 32) {
      const int r = idx / ((C0 + C1) / 4), c4 = idx - r * ((C0 + C1) / 4);
      const float* src = 4 * c4 < C0 ? A.pq + (node0 + ib + r) * (2 * E0) + part * C0 + 4 * c4
                                     : A.de + (node0 + ib + r) * E1 + part * C1 + (4 * c4 - C0);
      e3_cp_async16(dst + r * (C0 + C1) + 4 * c4, src);
    }
    e3_cp_async_commit();
  };

  // ---- L0 of the cursor's tile into tile slot `ts`: a0 (this thread's channel part) -> shared A0, then F1 is issued ----
  auto L0 = [&](E3Slot& sl, const int ts) {
    uint8_t* tb = gb + ts * SM::tile_bytes;
    const uint32_t tba = smem_u32(tb);
    if (fresh) {
      const int task = 4 * k + wq;
      c_active = task < ntasks;
      const int tk = c_active ? task : 0;
      const int jet = tk / A.NJB;
      jb = tk - jet * A.NJB;
      const int j = jb * 32 + lane;
      c_valid = c_active && j < N;
      node0 = (size_t)jet * N;
      e3_cp_async_wait<0>();
      __syncwarp();
      stage_chunk(i / IC);
      if ((i / IC + 1) * IC < N) stage_chunk(i / IC + 1);
      if (j < N) {
        const float4* src = reinterpret_cast<const float4*>(A.pq + (node0 + j) * (2 * E0) + E0 + part * C0);
#pragma unroll
        for (int c = 0; c < C0 / 4; ++c) {
          const float4 v = __ldg(src + c);
          q[2 * c] = bf2_as_u32(__floats2bfloat162_rn(v.x, v.y)); q[2 * c + 1] = bf2_as_u32(__floats2bfloat162_rn(v.z, v.w));
        }
      } else {
#pragma unroll
        for (int c = 0; c < C0 / 2; ++c) q[c] = 0u;
      }
      d_cur = __ldg(A.d + (node0 + i) * A.NJ32 + jb * 32 + lane);
      if ((i / IC + 1) * IC < N) e3_cp_async_wait<1>(); else e3_cp_async_wait<0>();
      __syncwarp();
      fresh = false;
    } else if ((i % IC) == 0) {
      e3_cp_async_wait<0>();
      __syncwarp();
      if ((i / IC + 1) * IC < N) stage_chunk(i / IC + 1);
    }
    sl.active = c_active; sl.valid = c_valid; sl.i = i; sl.jb = jb; sl.node0 = node0; sl.last_i = (i + 1 == N); sl.slot = ts;
    sl.dij = d_cur;
    sl.st = s_st + (((i / IC) & 1) * IC + (i % IC)) * (C0 + C1);
    if (!sl.last_i) d_cur = __ldg(A.d + (node0 + i + 1) * A.NJ32 + jb * 32 + lane);
    // the weight-gradient GEMM of the tile that used this slot two tiles ago must have read A0 / D1
    if (sl.pendW) { mbar_wait(bars + 2 + sl.slot, (ph_bits >> (2 + sl.slot)) & 1u); ph_bits ^= 4u << sl.slot; sl.pendW = false; }
    {
      uint8_t* a0_row = tb + SM::t_a0 + row * 16;
      const float* st = sl.st;
      const float2 d2 = make_float2(sl.dij, sl.dij);
#pragma unroll
      for (int c = 0; c < C0; c += 8) {
        uint32_t o[4];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int cc = c + 4 * hh;
          const float4 p = *reinterpret_cast<const float4*>(st + cc);
          const float4 w = *reinterpret_cast<const float4*>(s_wd + part * C0 + cc);
          const float2 z0 = fma2(make_float2(w.x, w.y), d2, add2(make_float2(p.x, p.y), unpack_bf2(q[cc / 2])));
          const float2 z1 = fma2(make_float2(w.z, w.w), d2, add2(make_float2(p.z, p.w), unpack_bf2(q[cc / 2 + 1])));
          o[2 * hh] = leaky_pack(z0.x, z0.y, alpha2);
          o[2 * hh + 1] = leaky_pack(z1.x, z1.y, alpha2);
        }
        *reinterpret_cast<uint4*>(a0_row + ((part * C0 + c) >> 3) * 2048) = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
    fence_proxy_async();
    tc_fence_before();
    named_bar_sync(1 + wg, GT);
    if (wl == 0) {      // F1: acc = A0 W1^T + b1
      tc_fence_after();
      const uint32_t acc0 = tmem_base + (uint32_t)((wg * 2 + ts) * ACC);
      const uint64_t dA0k = make_smem_desc(tba + SM::t_a0, 2048, 128), dW1f = wdesc_kmajor(w1a, E1);
      const uint64_t dBiasA = make_smem_desc(tba + SM::t_ones, zero_a - (tba + SM::t_ones), 128);
      const uint32_t idesc = make_idesc_bf16(128, E1, 0, 0);
#pragma unroll
      for (int s = 0; s < E0 / 16; ++s) mma_bf16_ss_elect(acc0, dA0k + (uint64_t)(s * 256), dW1f + (uint64_t)(s * 2 * E1), idesc, s > 0);
      mma_bf16_ss_elect(acc0, dBiasA, make_smem_desc(b1a, zero_a - b1a, 128), idesc, 1u);
      mma_commit_elect(bars + ts);
    }
    if (++i == N) { i = 0; ++k; fresh = true; }
  };

  // ---- E1: dz1 = de_i leaky'(z1) (zero on padded rows) for this thread's channel part -> shared D1; dgrad and wgrad are issued ----
  auto E1f = [&](E3Slot& sl, const int ts) {
    uint8_t* tb = gb + ts * SM::tile_bytes;
    const uint32_t tba = smem_u32(tb);
    const uint32_t acc0 = tmem_base + (uint32_t)((wg * 2 + ts) * ACC), acc = acc0 + ((uint32_t)(wq * 32) << 16);
    uint8_t* d1_row = tb + SM::t_d1 + row * 16;
    mbar_wait(bars + ts, (ph_bits >> ts) & 1u); ph_bits ^= 1u << ts;
    tc_fence_after();
    const float* dei = sl.st + C0;
    const bool valid = sl.valid;
#pragma unroll
    for (int c0 = 0; c0 < C1; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(acc + (uint32_t)(part * C1 + c0), v);
      tmem_ld_wait(); tmem_pin16(v);
      uint32_t o[8];
#pragma unroll
      for (int p4 = 0; p4 < 4; ++p4) {
        const float4 dv = *reinterpret_cast<const float4*>(dei + c0 + 4 * p4);
        const float g0v = valid ? dv.x * (__uint_as_float(v[4 * p4]) > 0.f ? 1.f : alpha) : 0.f;
        const float g1v = valid ? dv.y * (__uint_as_float(v[4 * p4 + 1]) > 0.f ? 1.f : alpha) : 0.f;
        const float g2v = valid ? dv.z * (__uint_as_float(v[4 * p4 + 2]) > 0.f ? 1.f : alpha) : 0.f;
        const float g3v = valid ? dv.w * (__uint_as_float(v[4 * p4 + 3]) > 0.f ? 1.f : alpha) : 0.f;
        o[2 * p4] = bf2_as_u32(__floats2bfloat162_rn(g0v, g1v));
        o[2 * p4 + 1] = bf2_as_u32(__floats2bfloat162_rn(g2v, g3v));
      }
      *reinterpret_cast<uint4*>(d1_row + ((part * C1 + c0) >> 3) * 2048) = make_uint4(o[0], o[1], o[2], o[3]);
      *reinterpret_cast<uint4*>(d1_row + (((part * C1 + c0) >> 3) + 1) * 2048) = make_uint4(o[4], o[5], o[6], o[7]);
    }
    fence_proxy_async();
    tc_fence_before();
    named_bar_sync(1 + wg, GT);
    if (wl == 1) {      // dgrad: acc = dz1 W1
      tc_fence_after();
      const uint64_t dD1k = make_smem_desc(tba + SM::t_d1, 2048, 128), dW1b = make_smem_desc(w1a, 128, E1 * 16);
      const uint32_t idesc = make_idesc_bf16(128, E0, 0, 1);
#pragma unroll
      for (int s = 0; s < E1 / 16; ++s) mma_bf16_ss_elect(acc0, dD1k + (uint64_t)(s * 256), dW1b + (uint64_t)(s * 16), idesc, s > 0);
      mma_commit_elect(bars + ts);
    } else if (wl == 2) {      // wgrad: [dW1 | db1] += dz1^T [a0 | 1]
      tc_fence_after();
      const uint64_t dD1n = make_smem_desc(tba + SM::t_d1, 128, 2048), dA0n = make_smem_desc(tba + SM::t_a0, 128, 2048);
      const uint32_t idesc = make_idesc_bf16(E1 == 128 ? 128 : 64, E0 + 16, 1, 1);
#pragma unroll
      for (int s = 0; s < 8; ++s) mma_bf16_ss_elect(tmem_base + GW, dD1n + (uint64_t)(s * 16), dA0n + (uint64_t)(s * 16), idesc, 1u);
      mma_commit_elect(bars + 2 + ts);
    }
    sl.pendW = true;
  };

  auto flush_dq = [&](const E3Slot& sl) {      // dQ_j of the (jet, j block) just finished (at most two groups add into one row)
    if (sl.valid) {
      float* dst = A.dpq + (sl.node0 + sl.jb * 32 + lane) * (2 * E0) + E0 + part * C0;
#pragma unroll
      for (int c = 0; c < C0; ++c) atomicAdd(dst + c, dq[c]);
    }
#pragma unroll
    for (int c = 0; c < C0; ++c) dq[c] = 0.f;
  };

  // ---- E0: dz0 = acc leaky'(a0) in fp32 -> dP_i (lane reduce), dQ_j, d(wd), G_ij ----
  auto E0f = [&](E3Slot& sl, const int ts, bool last_of_range) {
    uint8_t* tb = gb + ts * SM::tile_bytes;
    const uint32_t acc = tmem_base + (uint32_t)((wg * 2 + ts) * ACC) + ((uint32_t)(wq * 32) << 16);
    const uint8_t* a0_row = tb + SM::t_a0 + row * 16;
    mbar_wait(bars + ts, (ph_bits >> ts) & 1u); ph_bits ^= 1u << ts;
    tc_fence_after();
    float gsum = 0.f;
    const float dij = sl.dij;
    float* dp_dst = (A.NJB > 1 ? A.dp_part + ((size_t)sl.jb * A.B * N + sl.node0 + sl.i) * E0 : A.dpq + (sl.node0 + sl.i) * (2 * E0)) + part * C0;
#pragma unroll
    for (int c0 = 0; c0 < C0; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(acc + (uint32_t)(part * C0 + c0), v);
      const uint4 s0 = *reinterpret_cast<const uint4*>(a0_row + ((part * C0 + c0) >> 3) * 2048);
      const uint4 s1 = *reinterpret_cast<const uint4*>(a0_row + (((part * C0 + c0) >> 3) + 1) * 2048);
      const uint32_t sg[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
      tmem_ld_wait(); tmem_pin16(v);
      float z[16];
#pragma unroll
      for (int p = 0; p < 8; ++p) {
        const float alo = __uint_as_float(sg[p] << 16), ahi = __uint_as_float(sg[p] & 0xffff0000u);
        z[2 * p] = __uint_as_float(v[2 * p]) * (alo > 0.f ? 1.f : alpha);
        z[2 * p + 1] = __uint_as_float(v[2 * p + 1]) * (ahi > 0.f ? 1.f : alpha);
      }
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        const float4 w = *reinterpret_cast<const float4*>(s_wd + part * C0 + c0 + 4 * c4);
        gsum = fmaf(z[4 * c4], w.x, gsum); gsum = fmaf(z[4 * c4 + 1], w.y, gsum);
        gsum = fmaf(z[4 * c4 + 2], w.z, gsum); gsum = fmaf(z[4 * c4 + 3], w.w, gsum);
      }
#pragma unroll
      for (int c = 0; c < 16; ++c) { dq[c0 + c] += z[c]; dwd[c0 + c] = fmaf(z[c], dij, dwd[c0 + c]); }
      const float s = e3_transpose_sum16(z, lane);
      if (sl.active && (lane & 1) == 0) dp_dst[c0 + (lane >> 1)] = s;
    }
    tc_fence_before();
    if (S > 1) {      // G_ij: the channel parts' sums meet in shared memory, part 0 writes the row's value
      if (part > 0) s_g[(part - 1) * 128 + row] = gsum;
      named_bar_sync(1 + wg, GT);
      if (part == 0) {
#pragma unroll
        for (int p = 1; p < S; ++p) gsum += s_g[(p - 1) * 128 + row];
      }
      named_bar_sync(1 + wg, GT);      // s_g is free again before the next tile's partials arrive
    }
    if (part == 0 && sl.active) A.G[(sl.node0 + sl.i) * A.NJ32 + sl.jb * 32 + lane] = sl.valid ? gsum : 0.f;
    if (sl.last_i || last_of_range) flush_dq(sl);      // a (jet, j block) that ends mid-way: the next group adds the rest
  };

  E3Slot sA, sB;
  sA.pendW = sB.pendW = false;
  sA.active = sA.valid = sA.last_i = sB.active = sB.valid = sB.last_i = false;
  sA.i = sB.i = sA.jb = sB.jb = 0; sA.slot = 0; sB.slot = 1; sA.node0 = sB.node0 = 0; sA.dij = sB.dij = 0.f; sA.st = sB.st = s_st;
  const int ntile = g1 - g0;
  // One copy of each stage in the instruction stream (the unrolled stages are several thousand instructions: two copies per
  // slot thrash the instruction cache): the slot is a run-time index and the two slot records swap after every tile.
  int ts = 0;
  if (ntile > 0) L0(sA, 0);
#pragma unroll 1
  for (int t = 0; t < ntile; ++t) {
    E1f(sA, ts);
    if (t + 1 < ntile) L0(sB, ts ^ 1);
    E0f(sA, ts, t + 1 == ntile);
    const E3Slot tmp = sA; sA = sB; sB = tmp;
    ts ^= 1;
  }
  // all of this group's MMAs have completed: the slot a record last used is kept in the record
  if (sA.pendW) { mbar_wait(bars + 2 + sA.slot, (ph_bits >> (2 + sA.slot)) & 1u); ph_bits ^= 4u << sA.slot; }
  if (sB.pendW) { mbar_wait(bars + 2 + sB.slot, (ph_bits >> (2 + sB.slot)) & 1u); ph_bits ^= 4u << sB.slot; }
  e3_cp_async_wait<0>();
  // d(wd): lanes by shuffles, warps through shared memory (fixed order)
#pragma unroll
  for (int c = 0; c < C0; ++c) { const float s = gj_warp_sum(dwd[c]); if (lane == 0) s_red[warp * C0 + c] = s; }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // =================================== gradient read-out ===================================
  float* out = A.part + (size_t)blockIdx.x * A.nedge;
  if (tid < E0) {      // channel c = tid: the warps holding its part are (wg, part = c / C0, any quadrant)
    const int c = tid, p = c / C0, cl = c - p * C0;
    float s = 0.f;
    for (int g = 0; g < NWG; ++g)
      for (int w4 = 0; w4 < 4; ++w4) s += s_red[((g * S + p) * 4 + w4) * C0 + cl];
    out[A.pWd + c * A.K0] = s;
  }
  if (warp < 4) {
    const uint32_t lb = tmem_base + ((uint32_t)(warp * 32) << 16);
    // [dW1 | db1]: M = 128: lane = out feature; M = 64: out feature m at lane (m / 16) * 32 + m % 16 (lanes 16..31 of a quadrant unused)
    const bool has = E1 == 128 || lane < 16;
    const int m = E1 == 128 ? warp * 32 + lane : warp * 16 + (lane & 15);
    for (int c0 = 0; c0 < E0 + 16; c0 += 16) {
      uint32_t v[16];
      tmem_ld16_u(lb + GW + c0, v);
      tmem_ld_wait(); tmem_pin16(v);
      if (has) {
        if (c0 < E0) {
#pragma unroll
          for (int c = 0; c < 16; ++c) out[A.pW1 + m * E0 + c0 + c] = __uint_as_float(v[c]);
        } else {
          out[A.pb1 + m] = __uint_as_float(v[0]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, TCOLS);
}

// dP_i = sum over the j blocks' partial dP (N > 32), fixed order
__global__ void __launch_bounds__(256) e3_sum_dp_parts_kernel(const float4* __restrict__ part, int njb, size_t rows, int E0, float* __restrict__ dpq) {
  const size_t n4 = rows * (size_t)(E0 / 4), idx = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (idx >= n4) return;
  float4 s = __ldg(part + idx);
  for (int b = 1; b < njb; ++b) {
    const float4 v = __ldg(part + (size_t)b * n4 + idx);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  const size_t r = idx / (size_t)(E0 / 4);
  const int c4 = (int)(idx - r * (size_t)(E0 / 4));
  *reinterpret_cast<float4*>(dpq + r * 2 * E0 + 4 * c4) = s;
}

}  // namespace

int gj_num_sms();
bool gj_deterministic();
void gj_set_error(const char* fmt, ...);
int gj_reduce_edge_partials(const MPLayout& L, const float* part, int nparts, float* dparams, cudaStream_t stream);
int gj_pair_dist_fwd(const MPLayout& L, const float* h, float* d, cudaStream_t stream);
int gj_pair_dist_bwd(const MPLayout& L, const float* h, const float* G, float* dh, cudaStream_t stream);
bool gj_pair_dist_bwd_fits(const MPLayout& L);

#define E3_CHECK(what)                                                                                \
  do { cudaError_t ce_ = cudaGetLastError();                                                          \
       if (ce_ != cudaSuccess) { gj_set_error(what ": %s", cudaGetErrorString(ce_)); return GJ_ERR_CUDA; } } while (0)

// widths covered by the compiled instantiations
static int e3_shape(const MPLayout& L) {
  if (!(L.Le == 2 && L.alpha <= 1.f && L.E[0] == L.E[1] && L.H >= 1)) return -1;
  if (L.E[0] == 64) return 0;
  if (L.E[0] == 128) return 1;
  return -1;
}
bool gj_edge3_supported(const MPLayout& L) {
  return e3_shape(L) >= 0 && gj_pair_dist_bwd_fits(L);
}
size_t gj_edge3_wimage_floats(const MPLayout& L) { return ((size_t)(e3_shape(L) == 0 ? WImage3<64, 64>::bytes : WImage3<128, 128>::bytes) + 255) / 256 * 64; }
// forward workspace: per-j-block partial aggregates (N > 32)
size_t gj_edge3_fwd_ws_floats(const MPLayout& L) {
  const size_t njb = (L.N + 31) / 32;
  return njb > 1 ? njb * L.B * L.N * L.E[1] : 0;
}
static int e3_bwd_grid() { return gj_num_sms(); }
// backward workspace: G (B N NJ32) | dP partials (NJB > 1) | per-CTA parameter-gradient partials
size_t gj_edge3_bwd_ws_floats(const MPLayout& L) {
  const size_t njb = (L.N + 31) / 32, rows = (size_t)L.B * L.N;
  size_t n = rows * njb * 32 + 64;
  if (njb > 1) n += njb * rows * L.E[0] + 64;
  n += (size_t)e3_bwd_grid() * L.pV[0] + 64;
  return n;
}

static void e3_fill(const MPLayout& L, E3Args& A) {
  memset(&A, 0, sizeof(A));
  A.B = L.B; A.N = L.N; A.NJB = (L.N + 31) / 32; A.NJ32 = A.NJB * 32;
  A.pW1 = L.pW[1]; A.pb1 = L.pb[1]; A.pWd = L.pW[0] + 2 * L.H; A.K0 = L.K[0]; A.nedge = L.pV[0];
  A.alpha = L.alpha;
  const long long tasks4 = ((long long)L.B * A.NJB + 3) / 4;
  A.tiles_total = (int)(tasks4 * L.N);
}

template <int E0, int E1, int NWG, int IC>
static int e3_launch_fwd(const MPLayout& L, E3Args& A, float* e_out, float* ws, cudaStream_t stream) {
  using SM = Fwd3Smem<E0, E1, NWG, IC>;
  static_assert(SM::total <= 227 * 1024, "forward shared-memory plan");
  auto kern = edge_fwd3_kernel<E0, E1, NWG, IC>;
  cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::total);
  if (ce != cudaSuccess) { gj_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  int grid = gj_num_sms();
  const int max_grid = (A.tiles_total + NWG - 1) / NWG;
  if (grid > max_grid) grid = max_grid;
  CUtensorMap tm_w;      // the parameter image as rows of 1 KB, one box
  static_assert(WImage3<E0, E1>::bytes % 1024 == 0 && WImage3<E0, E1>::bytes / 1024 <= 256, "one TMA box");
  if (int rc = gj_tmap_2d(&tm_w, A.wimg, 256, WImage3<E0, E1>::bytes / 1024, 1024, 256, WImage3<E0, E1>::bytes / 1024)) return rc;
  kern<<<grid, NWG * 128, SM::total, stream>>>(A, tm_w);
  E3_CHECK("edge_fwd3 launch");
  return GJ_OK;
}

// pq: (B N, 2 E0) projections; wimg: receives the packed parameter image; d: receives the pair distances (both reused by the
// backward call when the caller keeps them)
int gj_edge_fwd3(const MPLayout& L, const float* h, const float* pq, const float* params, float* e_out, float* ws, float* wimg, float* d,
                 cudaStream_t stream) {
  E3Args A; e3_fill(L, A);
  if (((long long)L.B * A.NJB + 3) / 4 * L.N > 0x7fffffffLL) { gj_set_error("gj_mp_step_fwd(bf16): batch * nodes too large"); return GJ_ERR_INVALID; }
  const int shape = e3_shape(L);
  if (shape == 0) pack3_kernel<64, 64><<<4, 256, 0, stream>>>(params, L.pW[1], L.pb[1], reinterpret_cast<uint8_t*>(wimg));
  else pack3_kernel<128, 128><<<8, 256, 0, stream>>>(params, L.pW[1], L.pb[1], reinterpret_cast<uint8_t*>(wimg));
  if (int rc = gj_pair_dist_fwd(L, h, d, stream)) return rc;
  A.pq = pq; A.d = d; A.params = params; A.wimg = reinterpret_cast<const uint8_t*>(wimg);
  A.e_out = A.NJB > 1 ? ws : e_out;
  int rc = shape == 0 ? e3_launch_fwd<64, 64, 4, 4>(L, A, e_out, ws, stream) : e3_launch_fwd<128, 128, 2, 2>(L, A, e_out, ws, stream);
  if (rc) return rc;
  if (A.NJB > 1) {
    const size_t n4 = (size_t)L.B * L.N * (L.E[1] / 4);
    e3_sum_jblocks_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const float4*>(ws), A.NJB, n4, reinterpret_cast<float4*>(e_out));
    E3_CHECK("edge_fwd3 j-block sum launch");
  }
  return GJ_OK;
}

template <int E0, int E1, int NWG, int S, int IC>
static int e3_launch_bwd(E3Args& A, int grid, cudaStream_t stream) {
  using SM = Bwd3Smem<E0, E1, NWG, S, IC>;
  static_assert(SM::total <= 227 * 1024, "backward shared-memory plan");
  auto kern = edge_bwd3_kernel<E0, E1, NWG, S, IC>;
  cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::total);
  if (ce != cudaSuccess) { gj_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  long long ng = (long long)grid * NWG;      // every (jet, j block) is shared by at most two groups (two-addend atomic dQ sums)
  const long long tasks4 = ((long long)A.B * A.NJB + 3) / 4;
  if (ng > tasks4) ng = tasks4;
  A.ngroups = (int)(ng < 1 ? 1 : ng);
  CUtensorMap tm_w;
  static_assert(WImage3<E0, E1>::bytes % 1024 == 0 && WImage3<E0, E1>::bytes / 1024 <= 256, "one TMA box");
  if (int rc = gj_tmap_2d(&tm_w, A.wimg, 256, WImage3<E0, E1>::bytes / 1024, 1024, 256, WImage3<E0, E1>::bytes / 1024)) return rc;
  kern<<<grid, NWG * S * 128, SM::total, stream>>>(A, tm_w);
  E3_CHECK("edge_bwd3 launch");
  return GJ_OK;
}

// edge adjoint: dpq (OVERWRITTEN), dh += distance path, dparams: W1, b1 and the wd column of W0.  have_saved: wimg and d hold the
// forward call's parameter image and pair distances; otherwise they are recomputed here.
int gj_edge_bwd3(const MPLayout& L, const float* h, const float* pq, const float* params, const float* de, float* dpq, float* dh, float* dparams,
                 float* ws, float* wimg, float* d, bool have_saved, cudaStream_t stream) {
  E3Args A; e3_fill(L, A);
  const size_t njb = A.NJB, rows = (size_t)L.B * L.N;
  float* G = ws;
  float* dp_part = G + rows * A.NJ32 + 64;
  float* part = njb > 1 ? dp_part + njb * rows * L.E[0] + 64 : dp_part;
  const int shape = e3_shape(L);
  if (!have_saved) {
    if (shape == 0) pack3_kernel<64, 64><<<4, 256, 0, stream>>>(params, L.pW[1], L.pb[1], reinterpret_cast<uint8_t*>(wimg));
    else pack3_kernel<128, 128><<<8, 256, 0, stream>>>(params, L.pW[1], L.pb[1], reinterpret_cast<uint8_t*>(wimg));
    if (int rc = gj_pair_dist_fwd(L, h, d, stream)) return rc;
  }
  cudaError_t ce = cudaMemsetAsync(dpq, 0, rows * 2 * L.E[0] * sizeof(float), stream);
  if (ce != cudaSuccess) { gj_set_error("cudaMemsetAsync: %s", cudaGetErrorString(ce)); return GJ_ERR_CUDA; }
  A.pq = pq; A.d = d; A.params = params; A.wimg = reinterpret_cast<const uint8_t*>(wimg);
  A.de = de; A.dpq = dpq; A.dp_part = dp_part; A.G = G; A.part = part;
  const int grid = e3_bwd_grid();
  // two tile groups per CTA (H = 64) share the TMEM gradient accumulator in a timing-dependent order: the deterministic mode
  // (gj_set_deterministic) runs one
  int rc = shape == 0 ? (gj_deterministic() ? e3_launch_bwd<64, 64, 1, 1, 2>(A, grid, stream) : e3_launch_bwd<64, 64, 2, 1, 2>(A, grid, stream))
                      : e3_launch_bwd<128, 128, 1, 2, 2>(A, grid, stream);
  if (rc) return rc;
  if (njb > 1) {
    const size_t n4 = rows * (size_t)(L.E[0] / 4);
    e3_sum_dp_parts_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const float4*>(dp_part), (int)njb, rows, L.E[0], dpq);
    E3_CHECK("edge_bwd3 dP sum launch");
  }
  if ((rc = gj_pair_dist_bwd(L, h, G, dh, stream))) return rc;
  return gj_reduce_edge_partials(L, part, grid, dparams, stream);
}
