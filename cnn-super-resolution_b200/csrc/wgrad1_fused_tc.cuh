// Layer-1 deltas FUSED into the layer-1 weight / bias gradient (9-1-5, n1 = 64, n2 = 32):
//     d1[p][c]        = [out1[p][c] > 0] * sum_k W2[c][k] * d2[p][k]            (never stored)
//     gW1[dy][dx][c] += sum_p in[p + (dy,dx)] * d1[p][c],     gB1[c] += sum_p d1[p][c]
// reference: src/kernel/layer_deltas.cl:42-127 (f_next = 1) followed by
// src/kernel/backpropagate.cl:56-114; ConfigBasedDataPipeline.cpp:258-320 runs them as two
// launches with the layer-1 deltas (n1 floats per pixel, 328 MB per 2 048 patches) written and
// read back in between.
//
// wgrad1_tc_kernel (wgrad_tc.cuh) wants its B operand TRANSPOSED: rows = channels, K = the 64
// pixels of a tile.  The delta GEMM can deliver exactly that: with A = W2 (rows = channels,
// K-major as stored) and B = the d2 tile (rows = pixels, K-major as stored) the accumulator is
//     DT[c][p] = sum_k W2[c][k] * d2[p][k]          TMEM lane = channel, column = pixel
// so the PB warps of the gradient kernel read their operand row out of tensor memory instead of
// global memory, mask it with out1 (loaded with the access pattern they used for d1), split it
// and store it as before.  3xTF32 into ONE accumulator (hi.hi + hi.lo + lo.hi).  W2 is stored
// twice along M (rows 64..127 repeat rows 0..63): lanes 64..127 then hold a copy of the tile,
// and the four PB warps -- one per TMEM lane quarter -- split the pixels of a tile in halves
// without exchanging anything.
//
// Measured and not kept: (1) the PB warps rewriting DT in place (hi parts in lanes 0..63, lo
// parts in the duplicate lanes 64..127) so that the gradient MMAs take their channel operand
// from TMEM: -32 KB of STS and -32 KB of tensor-core reads per tile, but every PB thread then
// needs the mask of all 64 pixels and the chunk went from 0.784 to 1.00 ms (a 1-bit mask written
// by the forward kernel would remove that); (2) keeping next-tile loads in registers across a
// tile (the compiler serialises load -> compare chains); (3) staging the input rows from the two
// LD warps instead of the producers (cp.async completion on an mbarrier): 0.784 -> 0.889 ms, the
// LD warps sit on the delta-GEMM chain and 64 threads are too few for 660 copies per tile;
// (4) 12 producer warps + one PB group: 0.831 ms.  The im2col producers (PA) are the critical
// path: ~3 000 cycles per tile for 400 instructions per thread in dependent chains.
//
//   LD (2 warps)  d2 tile -> TF32 hi / lo -> smem                               -> d2_full
//   I2 (1 warp)   DT[i&1] = [W2;W2] x d2^T, 12 MMAs                             -> dt_full
//   PB (2x4 warps) DT -> mask(out1) -> bias sums -> split -> B tile              -> full, dt_free
//   PA (8 warps)  im2col gather -> split -> A tiles                             -> full
//   I  (1 warp)   8 K-steps x 2 MMAs into the resident gradient accumulators    -> empty
#pragma once
#include <cuda_runtime.h>

#include "context.cuh"
#include "tc_common.cuh"
#include "wgrad_tc.cuh"

namespace srcnn {
namespace wgf {

struct Cfg {
  static constexpr int F = 9, T = F * F, TP = 88, N = 64, K2 = 32;
  static constexpr int PX = 64;
  static constexpr int N_PA = 8, W_PB = N_PA, N_PB = 8, W_I = W_PB + N_PB, W_LD = W_I + 1,
                       W_I2 = W_LD + 2;
  static constexpr int NT = (W_I2 + 1) * 32;
  static constexpr int PA_ITEMS = (T * (PX / 4) + N_PA * 32 - 1) / (N_PA * 32);
  static constexpr int SBO = 128 * (PX / 4);     // tiles with K = 64 pixels
  static constexpr int SBO2 = 128 * (K2 / 4);    // operands of the delta GEMM, K = 32
  // shared memory (floats).  An M = 128 MMA reads rows TP..127 of an A tile: they fall into
  // the arrays behind it (A_lo, B), inside the allocation; nobody reads those accumulator rows
  static constexpr int A_FLOATS = TP * PX, B_FLOATS = 2 * N * PX;
  static constexpr int STAGE = 2 * A_FLOATS + B_FLOATS;
  static constexpr int oBase = 2 * STAGE;                // per-pixel input offsets [2][PX]
  static constexpr int oD2 = oBase + 2 * PX;             // d2 stages: 2 x (hi [PX][K2], lo)
  static constexpr int D2_FLOATS = PX * K2;
  // staged input rows for the im2col gather: 2 x [NSLOT][SPITCH]
  static constexpr int NSLOT = 20, SPITCH = 40, MIN_OW = 22;
  static constexpr int oStage = oD2 + 2 * 2 * D2_FLOATS;
  static constexpr int TOTAL = oStage + 2 * NSLOT * SPITCH;
  static constexpr size_t SMEM_BYTES = sizeof(float) * (size_t)TOTAL;
  // tensor memory: the gradient accumulator D[channel rows: hi 0..63, lo 64..127][2*TP columns:
  // taps of A_hi, taps of A_lo], DT[2] (64 columns each), and W2 (TF32 hi 32 columns + lo 32) as
  // the TMEM-resident A operand of the delta GEMM
  static constexpr uint32_t cD = 0, cDT = 192, cW2 = 320, TMEM_COLS = 512;
  static_assert(2 * TP <= 192, "accumulator columns");
};
static_assert(Cfg::SMEM_BYTES + 2560 <= 227 * 1024, "shared memory budget (dynamic + static)");

#ifdef WGF_TRACE
__device__ long long wgf_trace[8][20];
#define WGF_EV(i, e) \
  { if (blockIdx.x == 0 && lane == 0 && (i) >= 50 && (i) < 58) wgf_trace[(i) - 50][e] = clock64(); }
#else
#define WGF_EV(i, e) {}
#endif

// STAGED: the input rows a tile's windows touch are copied to shared memory with coalesced
// loads first and the im2col gather reads them from there.  Gathering from global memory costs
// one L1 tag lookup per 128-byte line a warp's 32 taps touch (~8 per load instruction): 2 700
// of the 3 300 cycles a tile took.  Needs MIN_OW <= ow, ow + 8 <= SPITCH and oh >= 3 (a tile
// then spans at most 4 output rows of at most 2 samples: NSLOT input rows)
template <bool STAGED>
__global__ void __launch_bounds__(Cfg::NT, 1)
    wgrad1_fused_tc_kernel(const float* __restrict__ d2, const float* __restrict__ out1,
                           const float* __restrict__ W2, const float* __restrict__ in,
                           float* __restrict__ partial, int ow, int oh, long long P,
                           int n_tiles_total) {
  using C = Cfg;
  using namespace tc;
  using tc::mbar_arrive;
  using tc::named_bar_sync;
  extern __shared__ __align__(128) float wg_smem[];
  int* sBase = reinterpret_cast<int*>(wg_smem + C::oBase);
  float* sD2 = wg_smem + C::oD2;
  __shared__ __align__(8) uint64_t full[2], empty[2], d2_full[2], dt_full[2], dt_free[2], done;
  __shared__ float gb_part[4][C::N];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int iw = ow + C::F - 1, ih = oh + C::F - 1;

  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    for (int i = 0; i < 2; i++) {
      mbar_init(&full[i], C::N_PA * 32 + 128);
      mbar_init(&empty[i], 1);
      mbar_init(&d2_full[i], 64);
      mbar_init(&dt_full[i], 1);
      mbar_init(&dt_free[i], 128);
    }
    mbar_init(&done, 1);
  }
  // the zero rows of the im2col tiles (taps 81..87) are written once
  for (int i = tid; i < 2 * 2 * (C::TP - C::T) * C::PX; i += C::NT) {
    const int tile = i / ((C::TP - C::T) * C::PX), r = i % ((C::TP - C::T) * C::PX);
    const int t = C::T + r / C::PX, k = r % C::PX;
    wg_smem[(tile >> 1) * C::STAGE + (tile & 1) * C::A_FLOATS + kmajor_offset(t, k, C::PX)] = 0.f;
  }
  // the stage only ever holds finite values: pixels past the end of the last tile may then
  // read anything (their deltas are zero)
  for (int i = tid; i < 2 * C::NSLOT * C::SPITCH; i += C::NT) wg_smem[C::oStage + i] = 0.f;
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  // A operand of the delta GEMM, resident in tensor memory: lane r holds W2[r & 63][0..31] as
  // TF32 hi (32 columns) and lo (32 columns)
  if (warp < 4) {
    const int r = warp * 32 + lane;
    const float4* src = reinterpret_cast<const float4*>(W2 + (r & (C::N - 1)) * C::K2);
    const uint32_t a = tmem + ((uint32_t)(warp * 32) << 16) + C::cW2;
#pragma unroll
    for (int q = 0; q < C::K2 / 8; q++) {
      const float4 x = __ldg(src + 2 * q), y = __ldg(src + 2 * q + 1);
      float hi[8], lo[8];
      split_tf32(x.x, hi[0], lo[0]);
      split_tf32(x.y, hi[1], lo[1]);
      split_tf32(x.z, hi[2], lo[2]);
      split_tf32(x.w, hi[3], lo[3]);
      split_tf32(y.x, hi[4], lo[4]);
      split_tf32(y.y, hi[5], lo[5]);
      split_tf32(y.z, hi[6], lo[6]);
      split_tf32(y.w, hi[7], lo[7]);
      tmem_st8(a + q * 8, hi);
      tmem_st8(a + C::K2 + q * 8, lo);
    }
    tmem_st_wait();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const int my_tiles = (n_tiles_total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const long long per = (long long)ow * oh;

  if (warp < C::W_PB) {
    // ============================ PA: im2col tiles (as wgrad1_tc_kernel) ===================
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
        if (warp == 0) WGF_EV(i, 1)
        stage_issue(i + 1);
        if (warp == 0) WGF_EV(i, 15)
#pragma unroll
        for (int u = 0; u < C::PA_ITEMS; u++) {
          const int4 b4 = *reinterpret_cast<const int4*>(base + item_q4[u]);
          v[u][0] = st[b4.x + item_toff[u]];
          v[u][1] = st[b4.y + item_toff[u]];
          v[u][2] = st[b4.z + item_toff[u]];
          v[u][3] = st[b4.w + item_toff[u]];
        }
        if (warp == 0) WGF_EV(i, 16)
        // the stage is separate from the operand tiles: only the stores wait for MMA(i-2)
        if (i >= 2) mbar_wait(&empty[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
        if (warp == 0) WGF_EV(i, 0)
      } else {
        if (i >= 2) mbar_wait(&empty[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
        if (warp == 0) WGF_EV(i, 0)
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
        if (warp == 0) WGF_EV(i, 1)
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
      if (warp == 0) WGF_EV(i, 2)
    }
  } else if (warp < C::W_I) {
    // ============================ PB: DT -> mask -> B tile, bias sums ======================
    // warp pw = TMEM lane quarter pw: channel 32*(pw&1) + lane, pixels 32*(pw>>1) .. +31.
    // Two groups of four warps take alternate tiles (group g: stage g, DT[g]): a warp's loads
    // only have one tile to land, and with one group every tile waited on HBM latency
    const int pw = (warp - C::W_PB) & 3, grp = (warp - C::W_PB) >> 2;
    const int c = (pw & 1) * 32 + lane;
    const int px0 = (pw >> 1) * 32;
    const uint32_t lane_base = (uint32_t)(pw * 32) << 16;
    float gb = 0.f;
    for (int i = grp; i < my_tiles; i += 2) {
      const long long p0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * C::PX + px0;
      // the mask operand does not depend on the MMA: all loads in flight while waiting
      float o[32];
#pragma unroll
      for (int j = 0; j < 32; j++) o[j] = p0 + j < P ? __ldg(out1 + (p0 + j) * C::N + c) : 0.f;
      if (pw == 0) WGF_EV(i, 3)
      mbar_wait(&dt_full[i & 1], (uint32_t)((i >> 1) & 1));
      if (pw == 0) WGF_EV(i, 4)
      tcgen05_fence_after();
      float v[32];
      const uint32_t dt = tmem + lane_base + C::cDT + 64u * (uint32_t)(i & 1) + (uint32_t)px0;
      tmem_ld16_nowait(dt, v);
      tmem_ld16_nowait(dt + 16, v + 16);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&dt_free[i & 1]);
      if (pw == 0) WGF_EV(i, 5)
      if (i >= 2) mbar_wait(&empty[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
      if (pw == 0) WGF_EV(i, 6)
      float* sB = wg_smem + (i & 1) * C::STAGE + 2 * C::A_FLOATS;
#pragma unroll
      for (int u = 0; u < 8; u++) {
        float d[4], hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = o[4 * u + j] > 0.f ? v[4 * u + j] : 0.f;
        gb += (d[0] + d[1]) + (d[2] + d[3]);
#pragma unroll
        for (int j = 0; j < 4; j++) split_tf32(d[j], hi[j], lo[j]);
        *reinterpret_cast<float4*>(sB + kmajor_offset(c, px0 + 4 * u, C::PX)) =
            make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(sB + kmajor_offset(C::N + c, px0 + 4 * u, C::PX)) =
            make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_proxy_async();
      mbar_arrive(&full[i & 1]);
      if (pw == 0) WGF_EV(i, 7)
    }
    gb_part[2 * grp + (pw >> 1)][c] = gb;
  } else if (warp == C::W_I) {
    // ============================ I: gradient MMA issuer ===================================
    // D[ch hi; ch lo][taps of A_hi | taps of A_lo] += [B_hi; B_lo] x [A_hi; A_lo]^T: M = 128
    // channel rows (no padding), N = 176 tap columns, all four partial products from ONE MMA
    // per K-step (shared-memory operand reads are what bounds this kernel)
    const uint32_t idesc = make_idesc_tf32(128, 2 * C::TP);
    for (int i = 0; i < my_tiles; i++) {
      mbar_wait(&full[i & 1], (uint32_t)((i >> 1) & 1));
      WGF_EV(i, 8)
      tcgen05_fence_after();
      const float* st = wg_smem + (i & 1) * C::STAGE;
      const uint64_t taps = make_desc_kmajor(st, 0, 128, C::SBO);   // A_hi rows, then A_lo rows
      const uint64_t chan = make_desc_kmajor(st + 2 * C::A_FLOATS, 0, 128, C::SBO);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::PX / 8; ks++)
          mma_tf32(tmem + C::cD, chan + 16 * ks, taps + 16 * ks, idesc, (i | ks) > 0);
        mma_commit(&empty[i & 1]);
        if (i == my_tiles - 1) mma_commit(&done);
      }
      __syncwarp();
      WGF_EV(i, 9)
    }
  } else if (warp < C::W_I2) {
    // ============================ LD: d2 tile -> TF32 hi / lo (rows = pixels) ==============
    // item u of a thread = (pixel px_of(u), 16-byte chunk ck_of(u)): the 8 lanes of a quarter
    // warp take 8 consecutive pixels (conflict-free STS.128 into the K-major tile: the 16-byte
    // slot inside a core matrix is the pixel & 7), the four quarters four consecutive chunks, so
    // one load instruction touches 8 lines of 64 bytes (thread = pixel row: 32 lines of 16)
    const int lw = warp - C::W_LD;
    auto px_of = [&](int u) { return 8 * (4 * lw + (u >> 1)) + (lane & 7); };
    auto ck_of = [&](int u) { return (lane >> 3) + 4 * (u & 1); };
    // one tile ahead in registers, for the same reason as the mask of the PB warps
    auto load_tile = [&](int i, float4 (&v)[C::K2 / 4]) {
      const long long p0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * C::PX;
#pragma unroll
      for (int u = 0; u < C::K2 / 4; u++) {
        const long long p = p0 + px_of(u);
        v[u] = (i < my_tiles && p < P)
                   ? __ldg(reinterpret_cast<const float4*>(d2 + p * C::K2) + ck_of(u))
                   : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    float4 v[C::K2 / 4], nv[C::K2 / 4];
    load_tile(0, v);
    for (int i = 0; i < my_tiles; i++) {
      load_tile(i + 1, nv);
      if (warp == C::W_LD) WGF_EV(i, 10)
      // the stage is free once the delta GEMM of tile i-2 has completed
      if (i >= 2) mbar_wait(&dt_full[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
      if (warp == C::W_LD) WGF_EV(i, 11)
      float* sh = sD2 + (i & 1) * 2 * C::D2_FLOATS;
      float* sl = sh + C::D2_FLOATS;
#pragma unroll
      for (int q = 0; q < C::K2 / 4; q++) {
        float hi[4], lo[4];
        split_tf32(v[q].x, hi[0], lo[0]);
        split_tf32(v[q].y, hi[1], lo[1]);
        split_tf32(v[q].z, hi[2], lo[2]);
        split_tf32(v[q].w, hi[3], lo[3]);
        const int off = kmajor_offset(px_of(q), 4 * ck_of(q), C::K2);
        *reinterpret_cast<float4*>(sh + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(sl + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_proxy_async();
      mbar_arrive(&d2_full[i & 1]);
      if (warp == C::W_LD) WGF_EV(i, 12)
#pragma unroll
      for (int q = 0; q < C::K2 / 4; q++) v[q] = nv[q];
    }
  } else {
    // ============================ I2: delta GEMM issuer ====================================
    const uint32_t idesc = make_idesc_tf32(128, C::PX);
    const uint32_t wh = tmem + C::cW2, wl = tmem + C::cW2 + C::K2;
    for (int i = 0; i < my_tiles; i++) {
      mbar_wait(&d2_full[i & 1], (uint32_t)((i >> 1) & 1));
      // DT[i&1] is free once the PB warps have read tile i-2 out of it
      if (i >= 2) mbar_wait(&dt_free[i & 1], (uint32_t)(((i - 2) >> 1) & 1));
      WGF_EV(i, 13)
      tcgen05_fence_after();
      const float* st = sD2 + (i & 1) * 2 * C::D2_FLOATS;
      const uint64_t dh = make_desc_kmajor(st, 0, 128, C::SBO2);
      const uint64_t dl = make_desc_kmajor(st + C::D2_FLOATS, 0, 128, C::SBO2);
      const uint32_t dt = tmem + C::cDT + 64u * (uint32_t)(i & 1);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::K2 / 8; ks++) {
          mma_tf32_ts(dt, wh + 8 * ks, dh + 16 * ks, idesc, ks > 0);
          mma_tf32_ts(dt, wh + 8 * ks, dl + 16 * ks, idesc, 1);
          mma_tf32_ts(dt, wl + 8 * ks, dh + 16 * ks, idesc, 1);
        }
        mma_commit(&dt_full[i & 1]);
      }
      __syncwarp();
      WGF_EV(i, 14)
    }
  }

  // ---- epilogue: one partial [T*N + N] per CTA.  TMEM lane = channel (lanes 64.. : the lo
  // rows of the same channels), columns = taps (88.. : the A_lo taps): four terms per weight
  __syncthreads();   // gb_part complete, all producers done
  float* dst = partial + (long long)blockIdx.x * (C::T * C::N + C::N);
  float* sX = wg_smem;   // [T][N] exchange between the lane halves (the stages are idle now)
  if (warp < 4) {
    if (my_tiles > 0) {
      mbar_wait(&done, 0);
      tcgen05_fence_after();
    }
    const int ch = (warp & 1) * 32 + lane;
    const uint32_t d = tmem + ((uint32_t)(warp * 32) << 16) + C::cD;
#pragma unroll 1
    for (int g = 0; g < C::TP / 8; g++) {
      float a[8], b[8];
      if (my_tiles > 0) {
        tmem_ld8(d + g * 8, a);
        tmem_ld8(d + C::TP + g * 8, b);
      } else {
#pragma unroll
        for (int j = 0; j < 8; j++) a[j] = b[j] = 0.f;
      }
      if (warp >= 2) {
#pragma unroll
        for (int j = 0; j < 8; j++)
          if (g * 8 + j < C::T) sX[(g * 8 + j) * C::N + ch] = a[j] + b[j];
      }
      named_bar_sync(2, 128);
      if (warp < 2) {
#pragma unroll
        for (int j = 0; j < 8; j++)
          if (g * 8 + j < C::T)
            dst[(g * 8 + j) * C::N + ch] = (a[j] + b[j]) + sX[(g * 8 + j) * C::N + ch];
      }
    }
  }
  if (tid < C::N)
    dst[C::T * C::N + tid] = (gb_part[0][tid] + gb_part[1][tid]) + (gb_part[2][tid] + gb_part[3][tid]);
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
#ifdef WGF_TRACE
  if (blockIdx.x == 0 && tid == 0 && my_tiles > 60) {
    const long long t0 = wgf_trace[0][0];
    for (int t = 0; t < 8; t++)
      printf("tile %d: PA issued %6lld gathered %6lld\n", 50 + t, wgf_trace[t][15] - t0, wgf_trace[t][16] - t0);
    for (int t = 0; t < 8; t++)
      printf("tile %d: PA free %6lld base %6lld done %6lld | LD top %6lld free %6lld done %6lld | I2 %6lld..%6lld | "
             "PB top %6lld dt %6lld ld %6lld free %6lld done %6lld | I %6lld..%6lld\n",
             50 + t, wgf_trace[t][0] - t0, wgf_trace[t][1] - t0, wgf_trace[t][2] - t0,
             wgf_trace[t][10] - t0, wgf_trace[t][11] - t0, wgf_trace[t][12] - t0,
             wgf_trace[t][13] - t0, wgf_trace[t][14] - t0, wgf_trace[t][3] - t0, wgf_trace[t][4] - t0,
             wgf_trace[t][5] - t0, wgf_trace[t][6] - t0, wgf_trace[t][7] - t0, wgf_trace[t][8] - t0,
             wgf_trace[t][9] - t0);
  }
#endif
}

// Layer-1 deltas + layer-1 gradients of an f2 = 1 network in one launch: per-CTA partials go to
// ctx->splitk_scratch (`count` of them) for partial_reduce_kernel.  Returns 1 when it launched,
// 0 when the shape has no instantiation.
inline int wgrad1_fused_tc(srcnn_ctx* ctx, const float* d2, const float* out1, const float* W2,
                           const float* in, int n1, int n2, int f1, int f2, int ow, int oh, int S,
                           int* count) {
  if (f1 != Cfg::F || f2 != 1 || n1 != Cfg::N || n2 != Cfg::K2) return 0;
  if ((reinterpret_cast<uintptr_t>(d2) & 15u) != 0) return 0;
  const long long P = (long long)S * ow * oh;
  const long long in_elems = (long long)S * (ow + f1 - 1) * (oh + f1 - 1);
  if (in_elems > 0x7fffffffLL) return 0;   // 32-bit input offsets
  const long long tiles = (P + Cfg::PX - 1) / Cfg::PX;
  if (tiles > 0x7fffffffLL) return 0;
  if (P > 0x7fffffffLL - Cfg::PX) return 0;
  SRCNN_TRY(ensure_func_setup(ctx, wgrad1_fused_tc_kernel<true>, Cfg::SMEM_BYTES));
  SRCNN_TRY(ensure_func_setup(ctx, wgrad1_fused_tc_kernel<false>, Cfg::SMEM_BYTES));
  const bool staged = ow >= Cfg::MIN_OW && ow + Cfg::F - 1 <= Cfg::SPITCH && oh >= 3;
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  const int grid = (int)(tiles < sms ? tiles : sms);
  *count = grid;
  SRCNN_TRY(ensure_scratch(ctx, &ctx->splitk_scratch, &ctx->splitk_bytes,
                           sizeof(float) * (size_t)grid * (Cfg::T * Cfg::N + Cfg::N)));
  if (staged)
    wgrad1_fused_tc_kernel<true><<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(
        d2, out1, W2, in, (float*)ctx->splitk_scratch, ow, oh, P, (int)tiles);
  else
    wgrad1_fused_tc_kernel<false><<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(
        d2, out1, W2, in, (float*)ctx->splitk_scratch, ow, oh, P, (int)tiles);
  return 1;
}

}  // namespace wgf
}  // namespace srcnn
