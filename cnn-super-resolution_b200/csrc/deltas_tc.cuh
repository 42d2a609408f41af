// Deltas below an f = 1 layer on the tensor cores (layer 1 of 9-1-5, n1 = 64, n2 = 32):
//     target[p][n] = [lo[p][n] > 0] * sum_k W[n][k] * dn[p][k]        p over all S*oh*ow pixels
// reference: src/kernel/layer_deltas.cl:42-127 with f_next = 1.
//
// The contraction is a plain [P x 32] . [32 x 64] GEMM, 4 096 FLOP for 640 bytes per pixel: on
// the FP32 pipe it is compute-bound (f1_deltas_kernel: 330 us per 2 048 patches), on the tensor
// cores it is an HBM stream (~130 us).  Same machinery as the fused forward kernels: tiles of
// 128 pixels, the A operand (dn, split into TF32 hi + lo: gradients have no fixed range, so no
// FP16 here) written to TENSOR MEMORY by the loader warps, stacked weights [W_hi; W_lo] as the
// shared-memory B operand, two MMAs per K-step, accumulators in TMEM, double buffering.
//
//   L (4 warps)  dn tile -> split -> A[i&1] (TMEM)                       -> a_full
//   I (1 warp)   D[i&1] = A_hi x [W_hi; W_lo] + A_lo x W_hi (8 MMAs)     -> mma_done
//   E (8 warps)  D -> sum of the two halves -> ReLU mask of lo -> target -> d_free
#pragma once
#include <cuda_runtime.h>

#include "context.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace d1tc {

struct Cfg {
  static constexpr int N = 64, K = 32, M = 128;
  static constexpr int W_L = 0, W_E = 4, N_E = 8, W_I = 12;
  static constexpr int NT = 13 * 32;
  // tensor memory: A[2] = 2 x (32 hi + 32 lo) columns, D[2] = 2 x 128 columns
  static constexpr uint32_t cA = 0, cD = 128, TMEM_COLS = 512;
};

__global__ void __launch_bounds__(Cfg::NT, 1) f1_deltas_tc_kernel(const float* __restrict__ dn,
                                                                  const float* __restrict__ lo,
                                                                  float* __restrict__ target,
                                                                  const float* __restrict__ W,
                                                                  long long P, int n_tiles_total) {
  using C = Cfg;
  using namespace tc;
  using tc::mbar_arrive;
  __shared__ __align__(128) float sW[2 * C::N * C::K];   // [128][K]: rows 0..63 hi, 64..127 lo
  __shared__ __align__(8) uint64_t a_full[2], mma_done[2], d_free[2];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  for (int i = tid; i < 2 * C::N * C::K; i += C::NT) {
    const int n = i / C::K, k = i % C::K;
    float hi, lw;
    split_tf32(__ldg(W + (n & (C::N - 1)) * C::K + k), hi, lw);
    sW[kmajor_offset(n, k, C::K)] = n < C::N ? hi : lw;
  }
  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    for (int i = 0; i < 2; i++) {
      mbar_init(&a_full[i], 128);
      mbar_init(&mma_done[i], 1);
      mbar_init(&d_free[i], C::N_E * 32);
    }
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  // tiles blockIdx.x, blockIdx.x + gridDim.x, ...
  const int my_tiles = (n_tiles_total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp < C::W_E) {
    // ============================ L: dn tile -> TF32 hi/lo -> A (TMEM) =====================
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    for (int i = 0; i < my_tiles; i++) {
      const long long p = ((long long)blockIdx.x + (long long)i * gridDim.x) * C::M + warp * 32 + lane;
      float4 v[C::K / 4];
#pragma unroll
      for (int q = 0; q < C::K / 4; q++)
        v[q] = p < P ? __ldg(reinterpret_cast<const float4*>(dn + p * C::K) + q)
                     : make_float4(0.f, 0.f, 0.f, 0.f);
      // A[i&1] is free once MMA(i-2) has completed
      if (i >= 2) mbar_wait(&mma_done[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
      tcgen05_fence_after();
      const uint32_t a = tmem + lane_base + C::cA + 64u * (uint32_t)(i & 1);
#pragma unroll
      for (int q = 0; q < C::K / 8; q++) {
        float hi[8], lw[8];
        split_tf32(v[2 * q].x, hi[0], lw[0]);
        split_tf32(v[2 * q].y, hi[1], lw[1]);
        split_tf32(v[2 * q].z, hi[2], lw[2]);
        split_tf32(v[2 * q].w, hi[3], lw[3]);
        split_tf32(v[2 * q + 1].x, hi[4], lw[4]);
        split_tf32(v[2 * q + 1].y, hi[5], lw[5]);
        split_tf32(v[2 * q + 1].z, hi[6], lw[6]);
        split_tf32(v[2 * q + 1].w, hi[7], lw[7]);
        tmem_st8(a + q * 8, hi);
        tmem_st8(a + C::K + q * 8, lw);
      }
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive(&a_full[i & 1]);
    }
  } else if (warp == C::W_I) {
    // ============================ I: MMA issuer ============================================
    const uint32_t idesc_hi = make_idesc_tf32(C::M, 2 * C::N);   // A_hi x [W_hi; W_lo]
    const uint32_t idesc_lo = make_idesc_tf32(C::M, C::N);       // A_lo x W_hi
    const uint64_t wdesc = make_desc_kmajor(sW, 0, 128, 128 * (C::K / 4));
    for (int i = 0; i < my_tiles; i++) {
      mbar_wait(&a_full[i & 1], (uint32_t)((i >> 1) & 1));
      if (i >= 2) mbar_wait(&d_free[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
      tcgen05_fence_after();
      const uint32_t a = tmem + C::cA + 64u * (uint32_t)(i & 1);
      const uint32_t d = tmem + C::cD + 128u * (uint32_t)(i & 1);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::K / 8; ks++) {
          mma_tf32_ts(d, a + ks * 8, wdesc + 16 * ks, idesc_hi, ks > 0);
          mma_tf32_ts(d, a + C::K + ks * 8, wdesc + 16 * ks, idesc_lo, 1);
        }
        mma_commit(&mma_done[i & 1]);
      }
      __syncwarp();
    }
  } else {
    // ============================ E: D -> mask -> target ===================================
    // warp w: TMEM lane quarter w & 3, outputs 32 * ((w - W_E) >> 2) .. + 31 of its pixel
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int n0 = ((warp - C::W_E) >> 2) * 32;
    for (int i = 0; i < my_tiles; i++) {
      const long long p = ((long long)blockIdx.x + (long long)i * gridDim.x) * C::M + (warp & 3) * 32 + lane;
      // the mask operand does not depend on the MMA: fetch it while waiting
      float4 o[8];
#pragma unroll
      for (int q = 0; q < 8; q++)
        o[q] = p < P ? __ldg(reinterpret_cast<const float4*>(lo + p * C::N + n0) + q)
                     : make_float4(0.f, 0.f, 0.f, 0.f);
      mbar_wait(&mma_done[i & 1], (uint32_t)((i >> 1) & 1));
      tcgen05_fence_after();
      const uint32_t d = tmem + lane_base + C::cD + 128u * (uint32_t)(i & 1) + n0;
      float va[32], vb[32];
      tmem_ld16_nowait(d, va);
      tmem_ld16_nowait(d + 16, va + 16);
      tmem_ld16_nowait(d + C::N, vb);
      tmem_ld16_nowait(d + C::N + 16, vb + 16);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&d_free[i & 1]);
      if (p < P) {
        float4* dst = reinterpret_cast<float4*>(target + p * C::N + n0);
#pragma unroll
        for (int q = 0; q < 8; q++) {
          float4 r;
          r.x = o[q].x > 0.f ? va[4 * q + 0] + vb[4 * q + 0] : 0.f;
          r.y = o[q].y > 0.f ? va[4 * q + 1] + vb[4 * q + 1] : 0.f;
          r.z = o[q].z > 0.f ? va[4 * q + 2] + vb[4 * q + 2] : 0.f;
          r.w = o[q].w > 0.f ? va[4 * q + 3] + vb[4 * q + 3] : 0.f;
          dst[q] = r;
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
}

// returns true when it launched
inline bool f1_deltas_tc(srcnn_ctx* ctx, const float* dn, const float* lo, float* target,
                         const float* W, int n_curr, int f_next, int n_next, int ow, int oh, int S) {
  if (f_next != 1 || n_curr != Cfg::N || n_next != Cfg::K) return false;
  if ((reinterpret_cast<uintptr_t>(dn) | reinterpret_cast<uintptr_t>(lo) |
       reinterpret_cast<uintptr_t>(target)) & 15u)
    return false;
  const long long P = (long long)S * ow * oh;
  const long long tiles = (P + Cfg::M - 1) / Cfg::M;
  if (tiles > 0x7fffffff) return false;
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  const int grid = (int)(tiles < sms ? tiles : sms);
  f1_deltas_tc_kernel<<<grid, Cfg::NT, 0, ctx->stream>>>(dn, lo, target, W, P, (int)tiles);
  return true;
}

}  // namespace d1tc
}  // namespace srcnn
