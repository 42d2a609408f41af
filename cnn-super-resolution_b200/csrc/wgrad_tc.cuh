// Weight / bias gradient of layer 1 (k = 1, f = 9, n = 64) on the tensor cores:
//     gW[dy][dx][n] += sum_{s,row,col} in[s][row+dy][col+dx] * d[s][row][col][n],  gB[n] += sum d
// reference: src/kernel/backpropagate.cl:56-114 (one work-item per weight, serial over all
// pixels, racy `+=` across samples; here deterministic).
//
// The contraction index is the PIXEL -- the slow index of both operands -- and tcgen05 has no
// MN-major TF32 operands (probe/mn_probe.cu: the MMA is a no-op), so the producers transpose on
// the way into shared memory: a thread owns one operand ROW (a filter tap / an output channel)
// for four consecutive pixels, its four loads are coalesced across the warp (consecutive rows
// are consecutive addresses in the pixel-major tensors), and its one STS.128 lands in the
// canonical K-major layout without bank conflicts.  Per tile of 64 pixels:
//     A_hi, A_lo [88 taps][64 px]   im2col of the input patches, TF32 hi / lo
//     B          [64 ch hi; 64 ch lo][64 px]   the deltas
//     D_hi[tap][0..127] += A_hi x B (N = 128),  D_lo[tap][0..63] += A_lo x B_hi (N = 64)
// 16 MMAs, accumulators stay in tensor memory for ALL tiles of the (persistent) CTA; one
// partial [81*64 + 64] per CTA goes to the fixed-order partial_reduce_kernel.
//
//   PA (8 warps)  im2col gather -> split -> A tiles                      -> full[i&1]
//   PB (4 warps)  delta tile -> split -> B tile, bias sums               -> full[i&1]
//   I  (1 warp)   8 K-steps x 2 MMAs                                     -> empty[i&1]
#pragma once
#include <cuda_runtime.h>

#include "context.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace wgtc {

struct Cfg {
  static constexpr int F = 9, T = F * F, TP = 88, N = 64;   // taps, padded taps, channels
  static constexpr int PX = 64;                             // pixels per tile (K of the GEMM)
  static constexpr int N_PA = 8, W_PB = N_PA, W_I = W_PB + 4;   // warps: PA 0..7, PB 8..11, I 12
  static constexpr int NT = (W_I + 1) * 32;
  static constexpr int PA_ITEMS = (T * (PX / 4) + N_PA * 32 - 1) / (N_PA * 32);   // per thread
  static constexpr int SBO = 128 * (PX / 4);                // bytes between 8-row groups
  // shared memory per stage (floats): A_hi, A_lo (TP rows), B (2N rows)
  static constexpr int A_FLOATS = TP * PX, B_FLOATS = 2 * N * PX;
  static constexpr int STAGE = 2 * A_FLOATS + B_FLOATS;
  static constexpr int oBase = 2 * STAGE;                   // per-pixel input offsets [2][PX]
  // staged input rows for the im2col gather (STAGED, as in wgrad1_fused_tc.cuh): 2 x [NSLOT][SPITCH]
  static constexpr int NSLOT = 20, SPITCH = 40, MIN_OW = 22;
  static constexpr int oStage = oBase + 2 * PX;
  static constexpr int TOTAL = oStage + 2 * NSLOT * SPITCH;
  // the M = 128 MMA also reads rows TP..127 of an A tile: they must lie inside the allocation
  // (their products land in accumulator rows nobody reads)
  static constexpr size_t SMEM_BYTES = sizeof(float) * (size_t)(TOTAL + (128 - TP) * PX);
  static constexpr uint32_t cDhi = 0, cDlo = 128, TMEM_COLS = 256;
};

// STAGED: the input rows a tile's windows touch are copied to shared memory with coalesced
// cp.async loads, one tile ahead, and the im2col gather reads them from there (gathering from
// global memory costs one L1 tag lookup per 128-byte line a warp's 32 taps touch, ~8 per load
// instruction).  Needs MIN_OW <= ow, ow + 8 <= SPITCH and oh >= 3: a tile then spans at most 4
// output rows of at most 2 samples = NSLOT input rows.  The scheme of wgrad1_fused_tc_kernel.
template <bool STAGED>
__global__ void __launch_bounds__(Cfg::NT, 1) wgrad1_tc_kernel(const float* __restrict__ d,
                                                               const float* __restrict__ in,
                                                               float* __restrict__ partial, int ow,
                                                               int oh, long long P,
                                                               int n_tiles_total) {
  using C = Cfg;
  using namespace tc;
  using tc::mbar_arrive;
  using tc::named_bar_sync;
  extern __shared__ __align__(128) float wg_smem[];
  int* sBase = reinterpret_cast<int*>(wg_smem + C::oBase);
  __shared__ __align__(8) uint64_t full[2], empty[2], done;
  __shared__ float gb_part[2][C::N];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int iw = ow + C::F - 1, ih = oh + C::F - 1;

  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    for (int i = 0; i < 2; i++) {
      mbar_init(&full[i], C::N_PA * 32 + 128);
      mbar_init(&empty[i], 1);
    }
    mbar_init(&done, 1);
  }
  // the zero rows of the im2col tiles (taps 81..87) are written once
  for (int i = tid; i < 2 * 2 * (C::TP - C::T) * C::PX; i += C::NT) {
    const int tile = i / ((C::TP - C::T) * C::PX), r = i % ((C::TP - C::T) * C::PX);
    const int t = C::T + r / C::PX, k = r % C::PX;
    wg_smem[(tile >> 1) * C::STAGE + (tile & 1) * C::A_FLOATS + kmajor_offset(t, k, C::PX)] = 0.f;
  }
  for (int i = tid; i < 2 * C::NSLOT * C::SPITCH; i += C::NT) wg_smem[C::oStage + i] = 0.f;
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  const int my_tiles = (n_tiles_total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const long long per = (long long)ow * oh;

  if (warp < C::W_PB) {
    // ============================ PA: im2col tiles ========================================
    float* sStage = wg_smem + C::oStage;
    // STAGED: pixel offsets and input rows of tile i -> buffers i&1, asynchronously (cp.async):
    // issued one tile ahead, so the L2 latency hides behind the gather / stores of the tile
    // before.  slot k of the stage = one input row: rows row0 .. ih-1 of sample s0 (count0 of
    // them), then rows 0 .. of sample s0+1.  A pixel (sample s, output row `row`, column col)
    // reads slots first .. first+8 at columns col .. col+8
    // Tile geometry without integer divisions in the loop (a dependent chain of ten of them was
    // 1 500 cycles per tile): (sample, output row, column) of the tile's first pixel advance by
    // a fixed step from tile to tile.
    int g_p0 = 0, g_s = 0, g_row = 0, g_col = 0, d_s = 0, d_row = 0, d_col = 0;
    const float inv_iw = 1.f / (float)iw;
    if (STAGED) {
      g_p0 = (int)blockIdx.x * C::PX;
      const int g = g_p0 / ow;
      g_col = g_p0 - g * ow;
      g_s = g / oh;
      g_row = g - g_s * oh;
      const int step = (int)gridDim.x * C::PX, sg = step / ow;
      d_col = step - sg * ow;
      d_s = sg / oh;
      d_row = sg - d_s * oh;
    }
    auto stage_issue = [&](int i) {
      if (i >= my_tiles) return;
      const int ip0 = g_p0, s0 = g_s, row0 = g_row, col0 = g_col, count0 = ih - row0;
      // advance to the next tile of this CTA
      g_p0 += (int)gridDim.x * C::PX;
      g_col += d_col;
      if (g_col >= ow) { g_col -= ow; g_row++; }
      g_row += d_row;
      if (g_row >= oh) { g_row -= oh; g_s++; }
      g_s += d_s;
      float* st = sStage + (i & 1) * (C::NSLOT * C::SPITCH);
      // pixel j of the tile: column col0 + j wraps at most three times (ow >= MIN_OW)
      auto first_slot = [&](int j, int& col) {
        const int c = col0 + j;
        const int w = (c >= ow) + (c >= 2 * ow) + (c >= 3 * ow);
        col = c - w * ow;
        const int row = row0 + w;
        return row < oh ? w : count0 + row - oh;
      };
      if (tid < C::PX) {
        int col;
        const int f = first_slot(tid, col);
        sBase[(i & 1) * C::PX + tid] = ip0 + tid < P ? f * C::SPITCH + col : 0;
      }
      const long long left = P - ip0;
      int col_l;
      const int n_elems = (first_slot((left < C::PX ? (int)left : C::PX) - 1, col_l) + C::F) * iw;
#pragma unroll
      for (int u = 0; u < (C::NSLOT * C::SPITCH + C::N_PA * 32 - 1) / (C::N_PA * 32); u++) {
        const int e = tid + C::N_PA * 32 * u;
        if (e < n_elems) {
          const int k = __float2int_rz(((float)e + 0.5f) * inv_iw), x = e - k * iw;
          const int src = k < count0 ? (s0 * ih + row0 + k) : ((s0 + 1) * ih + (k - count0));
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(
                           smem_u32(st + k * C::SPITCH + x)),
                       "l"(in + src * iw + x)
                       : "memory");
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // loop-invariant per item: stage offset of the tap, first pixel of the quad, tile offset
    int item_toff[C::PA_ITEMS], item_q4[C::PA_ITEMS], item_off[C::PA_ITEMS];
#pragma unroll
    for (int u = 0; u < C::PA_ITEMS; u++) {
      const int it = tid + C::N_PA * 32 * u;
      const bool ok = it < C::T * (C::PX / 4);
      const int t = ok ? it % C::T : 0, q = ok ? it / C::T : 0;
      item_toff[u] = (t / C::F) * C::SPITCH + (t % C::F);
      item_q4[u] = 4 * q;
      item_off[u] = ok ? kmajor_offset(t, 4 * q, C::PX) : -1;
    }
    if (STAGED) stage_issue(0);
    for (int i = 0; i < my_tiles; i++) {
      const long long p0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * C::PX;
      int* base = sBase + (i & 1) * C::PX;
      float v[C::PA_ITEMS][4];
      if (STAGED) {
        const float* st = sStage + (i & 1) * (C::NSLOT * C::SPITCH);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        named_bar_sync(1, C::N_PA * 32);   // tile i staged; everybody is done with tile i-1
        stage_issue(i + 1);
#pragma unroll
        for (int u = 0; u < C::PA_ITEMS; u++) {
          const int4 b4 = *reinterpret_cast<const int4*>(base + item_q4[u]);
          v[u][0] = st[b4.x + item_toff[u]];
          v[u][1] = st[b4.y + item_toff[u]];
          v[u][2] = st[b4.z + item_toff[u]];
          v[u][3] = st[b4.w + item_toff[u]];
        }
        // the stage is separate from the operand tiles: only the stores wait for MMA(i-2)
        if (i >= 2) mbar_wait(&empty[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
      } else {
        if (i >= 2) mbar_wait(&empty[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
        // input offset of the window origin of each pixel of the tile (-1: past the end)
        if (tid < C::PX) {
          const long long p = p0 + tid;
          int b = -1;
          if (p < P) {
            const long long sm = p / per;
            const int rem = (int)(p - sm * per), row = rem / ow, col = rem - row * ow;
            b = (int)((sm * ih + row) * iw + col);
          }
          base[tid] = b;
        }
        named_bar_sync(1, C::N_PA * 32);
        // item = (tap t, pixel quad q); consecutive lanes take consecutive taps.  All loads of
        // a thread are issued before the first is used
#pragma unroll
        for (int u = 0; u < C::PA_ITEMS; u++) {
          const int it = tid + C::N_PA * 32 * u;
          const int t = it % C::T, q = it / C::T;
          const int toff = (t / C::F) * iw + (t % C::F);
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const int b = it < C::T * (C::PX / 4) ? base[4 * q + j] : -1;
            v[u][j] = b >= 0 ? __ldg(in + b + toff) : 0.f;
          }
        }
      }
      float* sAh = wg_smem + (i & 1) * C::STAGE;
      float* sAl = sAh + C::A_FLOATS;
#pragma unroll
      for (int u = 0; u < C::PA_ITEMS; u++) {
        if (item_off[u] >= 0) {
          float hi[4], lo[4];
#pragma unroll
          for (int j = 0; j < 4; j++) split_tf32(v[u][j], hi[j], lo[j]);
          *reinterpret_cast<float4*>(sAh + item_off[u]) = make_float4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<float4*>(sAl + item_off[u]) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_proxy_async();
      mbar_arrive(&full[i & 1]);
    }
  } else if (warp < C::W_I) {
    // ============================ PB: delta tiles + bias sums ==============================
    const int pw = warp - C::W_PB;                 // 0..3
    const int c = (pw & 1) * 32 + lane;            // output channel of this thread
    float gb = 0.f;
    for (int i = 0; i < my_tiles; i++) {
      const long long p0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * C::PX;
      float* sB = wg_smem + (i & 1) * C::STAGE + 2 * C::A_FLOATS;
      float v[C::PX / 8][4];   // this thread's 8 pixel quads, all loads in flight together
#pragma unroll
      for (int u = 0; u < C::PX / 8; u++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const long long p = p0 + 4 * ((pw >> 1) + 2 * u) + j;
          v[u][j] = p < P ? __ldg(d + p * C::N + c) : 0.f;
        }
      if (i >= 2) mbar_wait(&empty[i & 1], (uint32_t)(((i - 2) >> 1) & 1));   // (loads first, as in PA)
#pragma unroll
      for (int u = 0; u < C::PX / 8; u++) {
        const int q = (pw >> 1) + 2 * u;
        float hi[4], lo[4];
        gb += (v[u][0] + v[u][1]) + (v[u][2] + v[u][3]);
#pragma unroll
        for (int j = 0; j < 4; j++) split_tf32(v[u][j], hi[j], lo[j]);
        *reinterpret_cast<float4*>(sB + kmajor_offset(c, 4 * q, C::PX)) =
            make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(sB + kmajor_offset(C::N + c, 4 * q, C::PX)) =
            make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_proxy_async();
      mbar_arrive(&full[i & 1]);
    }
    gb_part[pw >> 1][c] = gb;
  } else {
    // ============================ I: MMA issuer ============================================
    const uint32_t idesc_hi = make_idesc_tf32(128, 2 * C::N);   // A_hi x [B_hi; B_lo]
    const uint32_t idesc_lo = make_idesc_tf32(128, C::N);       // A_lo x B_hi
    for (int i = 0; i < my_tiles; i++) {
      mbar_wait(&full[i & 1], (uint32_t)((i >> 1) & 1));
      tcgen05_fence_after();
      const float* st = wg_smem + (i & 1) * C::STAGE;
      const uint64_t ah = make_desc_kmajor(st, 0, 128, C::SBO);
      const uint64_t al = make_desc_kmajor(st + C::A_FLOATS, 0, 128, C::SBO);
      const uint64_t bd = make_desc_kmajor(st + 2 * C::A_FLOATS, 0, 128, C::SBO);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::PX / 8; ks++) {
          mma_tf32(tmem + C::cDhi, ah + 16 * ks, bd + 16 * ks, idesc_hi, (i | ks) > 0);
          mma_tf32(tmem + C::cDlo, al + 16 * ks, bd + 16 * ks, idesc_lo, (i | ks) > 0);
        }
        mma_commit(&empty[i & 1]);
        if (i == my_tiles - 1) mma_commit(&done);
      }
      __syncwarp();
    }
  }

  // ---- epilogue: one partial [T*N + N] per CTA; thread = filter tap (TMEM lane)
  __syncthreads();   // gb_part complete, all producers done
  float* dst = partial + (long long)blockIdx.x * (C::T * C::N + C::N);
  if (warp < 3) {
    if (my_tiles > 0) {
      mbar_wait(&done, 0);
      tcgen05_fence_after();
    }
    const int t = warp * 32 + lane;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
#pragma unroll 1
    for (int g = 0; g < C::N / 16; g++) {
      float a[16], b[16], l[16];
      if (my_tiles > 0) {
        tmem_ld16_nowait(tmem + lane_base + C::cDhi + g * 16, a);
        tmem_ld16_nowait(tmem + lane_base + C::cDhi + C::N + g * 16, b);
        tmem_ld16_nowait(tmem + lane_base + C::cDlo + g * 16, l);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 16; j++) a[j] = b[j] = l[j] = 0.f;
      }
      if (t < C::T) {
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          *reinterpret_cast<float4*>(dst + t * C::N + g * 16 + j) =
              make_float4((a[j] + b[j]) + l[j], (a[j + 1] + b[j + 1]) + l[j + 1],
                          (a[j + 2] + b[j + 2]) + l[j + 2], (a[j + 3] + b[j + 3]) + l[j + 3]);
      }
    }
  }
  if (tid < C::N) dst[C::T * C::N + tid] = gb_part[0][tid] + gb_part[1][tid];
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------
// Weight / bias gradient of an f = 1 layer (layer 2 of 9-1-5, k = 64 -> n = 32):
//     gW[m][n] += sum_p in[p][m] * d[p][n],   gB[n] += sum_p d[p][n]
// Same scheme; both operands are plain transposes, and with 64 + 64 rows of A (hi, lo) and
// 32 + 32 rows of B all four partial products come out of ONE M = 128, N = 64 MMA per K-step:
//     D[m][n] = hi.hi   D[m][32+n] = hi.lo   D[64+m][n] = lo.hi   (D[64+m][32+n] = lo.lo, unused)
struct Cfg2 {
  static constexpr int K = 64, N = 32, PX = 64;
  static constexpr int N_PA = 8, W_PB = N_PA, W_I = W_PB + 4;
  static constexpr int NT = (W_I + 1) * 32;
  static constexpr int SBO = 128 * (PX / 4);
  static constexpr int A_FLOATS = 2 * K * PX, B_FLOATS = 2 * N * PX;
  static constexpr int STAGE = A_FLOATS + B_FLOATS;
  static constexpr int NS = 4;                               // stages (two tiles per producer step)
  static constexpr int oX = NS * STAGE;                      // epilogue exchange [K][N]
  static constexpr size_t SMEM_BYTES = sizeof(float) * (size_t)(oX + K * N);
  static constexpr uint32_t TMEM_COLS = 64;
};

__global__ void __launch_bounds__(Cfg2::NT, 1) wgrad2_tc_kernel(const float* __restrict__ d,
                                                                const float* __restrict__ in,
                                                                float* __restrict__ partial,
                                                                long long P, int n_tiles_total) {
  using C = Cfg2;
  using namespace tc;
  using tc::mbar_arrive;
  extern __shared__ __align__(128) float wg_smem[];
  float* sX = wg_smem + C::oX;
  __shared__ __align__(8) uint64_t full[C::NS], empty[C::NS], done;
  __shared__ float gb_part[4][C::N];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    for (int i = 0; i < C::NS; i++) {
      mbar_init(&full[i], C::N_PA * 32 + 128);
      mbar_init(&empty[i], 1);
    }
    mbar_init(&done, 1);
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  const int my_tiles = (n_tiles_total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp < C::W_PB) {
    // ============================ PA: layer input, transposed ==============================
    const int c = (warp & 1) * 32 + lane;          // input channel (row of A)
    // two tiles per step: the loads of both are in flight together (with one, the producers
    // waited on HBM latency every tile and the kernel sat at 58 % of the HBM peak)
    for (int i = 0; i < my_tiles; i += 2) {
      float v[2][4][4];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const long long p0 = ((long long)blockIdx.x + (long long)(i + h) * gridDim.x) * C::PX;
        const bool on = i + h < my_tiles;
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const long long p = p0 + 4 * ((warp >> 1) + 4 * u) + j;
            v[h][u][j] = (on && p < P) ? __ldg(in + p * C::K + c) : 0.f;
          }
      }
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int t = i + h, st = t & (C::NS - 1);
        if (t < my_tiles) {
          if (t >= C::NS) mbar_wait(&empty[st], (uint32_t)(((t - C::NS) / C::NS) & 1));
          float* sA = wg_smem + st * C::STAGE;
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int q = (warp >> 1) + 4 * u;
            float hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; j++) split_tf32(v[h][u][j], hi[j], lo[j]);
            *reinterpret_cast<float4*>(sA + kmajor_offset(c, 4 * q, C::PX)) =
                make_float4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<float4*>(sA + kmajor_offset(C::K + c, 4 * q, C::PX)) =
                make_float4(lo[0], lo[1], lo[2], lo[3]);
          }
          fence_proxy_async();
          mbar_arrive(&full[st]);
        }
      }
    }
  } else if (warp < C::W_I) {
    // ============================ PB: deltas, transposed + bias sums =======================
    const int pw = warp - C::W_PB;                 // 0..3: pixel quads pw, pw+4, ..
    float gb = 0.f;
    for (int i = 0; i < my_tiles; i += 2) {
      float v[2][4][4];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const long long p0 = ((long long)blockIdx.x + (long long)(i + h) * gridDim.x) * C::PX;
        const bool on = i + h < my_tiles;
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const long long p = p0 + 4 * (pw + 4 * u) + j;
            v[h][u][j] = (on && p < P) ? __ldg(d + p * C::N + lane) : 0.f;
          }
      }
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int t = i + h, st = t & (C::NS - 1);
        if (t < my_tiles) {
          if (t >= C::NS) mbar_wait(&empty[st], (uint32_t)(((t - C::NS) / C::NS) & 1));
          float* sB = wg_smem + st * C::STAGE + C::A_FLOATS;
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int q = pw + 4 * u;
            float hi[4], lo[4];
            gb += (v[h][u][0] + v[h][u][1]) + (v[h][u][2] + v[h][u][3]);
#pragma unroll
            for (int j = 0; j < 4; j++) split_tf32(v[h][u][j], hi[j], lo[j]);
            *reinterpret_cast<float4*>(sB + kmajor_offset(lane, 4 * q, C::PX)) =
                make_float4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<float4*>(sB + kmajor_offset(C::N + lane, 4 * q, C::PX)) =
                make_float4(lo[0], lo[1], lo[2], lo[3]);
          }
          fence_proxy_async();
          mbar_arrive(&full[st]);
        }
      }
    }
    gb_part[pw][lane] = gb;
  } else {
    // ============================ I: MMA issuer ============================================
    const uint32_t idesc = make_idesc_tf32(128, 2 * C::N);
    for (int i = 0; i < my_tiles; i++) {
      const int sg = i & (C::NS - 1);
      mbar_wait(&full[sg], (uint32_t)((i / C::NS) & 1));
      tcgen05_fence_after();
      const float* st = wg_smem + sg * C::STAGE;
      const uint64_t ad = make_desc_kmajor(st, 0, 128, C::SBO);
      const uint64_t bd = make_desc_kmajor(st + C::A_FLOATS, 0, 128, C::SBO);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::PX / 8; ks++)
          mma_tf32(tmem, ad + 16 * ks, bd + 16 * ks, idesc, (i | ks) > 0);
        mma_commit(&empty[sg]);
        if (i == my_tiles - 1) mma_commit(&done);
      }
      __syncwarp();
    }
  }

  // ---- epilogue: gW[m][n] = D[m][n] + D[m][32+n] + D[64+m][n]; thread = TMEM lane
  __syncthreads();
  float* dst = partial + (long long)blockIdx.x * (C::K * C::N + C::N);
  if (warp < 4) {
    mbar_wait(&done, 0);
    tcgen05_fence_after();
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    const int r = warp * 32 + lane;   // accumulator row
    float a[32], b[32];
    tmem_ld16_nowait(tmem + lane_base, a);
    tmem_ld16_nowait(tmem + lane_base + 16, a + 16);
    tmem_ld16_nowait(tmem + lane_base + 32, b);
    tmem_ld16_nowait(tmem + lane_base + 48, b + 16);
    tmem_ld_wait();
    if (r >= C::K) {   // lo.hi rows -> exchange buffer
#pragma unroll
      for (int j = 0; j < C::N; j++) sX[(r - C::K) * C::N + j] = a[j];
    }
    asm volatile("bar.sync 2, 128;" ::: "memory");
    if (r < C::K) {
#pragma unroll
      for (int j = 0; j < C::N; j += 4) {
        const float4 x = *reinterpret_cast<const float4*>(sX + r * C::N + j);
        *reinterpret_cast<float4*>(dst + r * C::N + j) =
            make_float4((a[j] + b[j]) + x.x, (a[j + 1] + b[j + 1]) + x.y,
                        (a[j + 2] + b[j + 2]) + x.z, (a[j + 3] + b[j + 3]) + x.w);
      }
    }
  }
  if (tid < C::N)
    dst[C::K * C::N + tid] = (gb_part[0][tid] + gb_part[1][tid]) + (gb_part[2][tid] + gb_part[3][tid]);
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
}

inline int wgrad2_tc(srcnn_ctx* ctx, const float* d, const float* in, int n, int k, int f, int ow,
                     int oh, int S, int* count) {
  if (f != 1 || k != Cfg2::K || n != Cfg2::N) return 0;
  const long long P = (long long)S * ow * oh;
  const long long tiles = (P + Cfg2::PX - 1) / Cfg2::PX;
  if (tiles > 0x7fffffffLL) return 0;
  SRCNN_TRY(ensure_func_setup(ctx, wgrad2_tc_kernel, Cfg2::SMEM_BYTES));
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  const int grid = (int)(tiles < sms ? tiles : sms);
  *count = grid;
  SRCNN_TRY(ensure_scratch(ctx, &ctx->splitk_scratch, &ctx->splitk_bytes,
                           sizeof(float) * (size_t)grid * (Cfg2::K * Cfg2::N + Cfg2::N)));
  wgrad2_tc_kernel<<<grid, Cfg2::NT, Cfg2::SMEM_BYTES, ctx->stream>>>(
      d, in, (float*)ctx->splitk_scratch, P, (int)tiles);
  return 1;
}

// returns 1 when it launched (partials in ctx->splitk_scratch, *count of them), 0 when not
// handled, < 0 on error
inline int wgrad1_tc(srcnn_ctx* ctx, const float* d, const float* in, int n, int k, int f, int ow,
                     int oh, int S, int* count) {
  if (k != 1 || f != Cfg::F || n != Cfg::N) return 0;
  const long long P = (long long)S * ow * oh;
  const long long in_elems = (long long)S * (ow + f - 1) * (oh + f - 1);
  if (in_elems > 0x7fffffffLL) return 0;   // 32-bit input offsets
  const long long tiles = (P + Cfg::PX - 1) / Cfg::PX;
  if (tiles > 0x7fffffffLL) return 0;
  const bool staged = ow >= Cfg::MIN_OW && ow + Cfg::F - 1 <= Cfg::SPITCH && oh >= 3;
  if (staged) SRCNN_TRY(ensure_func_setup(ctx, wgrad1_tc_kernel<true>, Cfg::SMEM_BYTES));
  else SRCNN_TRY(ensure_func_setup(ctx, wgrad1_tc_kernel<false>, Cfg::SMEM_BYTES));
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  const int grid = (int)(tiles < sms ? tiles : sms);
  *count = grid;
  SRCNN_TRY(ensure_scratch(ctx, &ctx->splitk_scratch, &ctx->splitk_bytes,
                           sizeof(float) * (size_t)grid * (Cfg::T * Cfg::N + Cfg::N)));
  if (staged)
    wgrad1_tc_kernel<true><<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(
        d, in, (float*)ctx->splitk_scratch, ow, oh, P, (int)tiles);
  else
    wgrad1_tc_kernel<false><<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(
        d, in, (float*)ctx->splitk_scratch, ow, oh, P, (int)tiles);
  return 1;
}

}  // namespace wgtc
}  // namespace srcnn
