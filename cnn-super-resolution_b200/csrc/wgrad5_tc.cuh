// Weight / bias gradient of the 5x5 layer 2 of the 9-5-5 network (k = 64 -> n = 32; BASELINE
// config C4) on the tensor cores:
//     gW[dy][dx][k][n] += sum_{s,y,x} d2[s][y][x][n] * out1[s][y+dy][x+dx][k],  gB[n] += sum d2
// reference: src/kernel/backpropagate.cl:56-114 (one work-item per weight, serial over all
// pixels, racy `+=` across samples; here deterministic: per-CTA partials + fixed-order reduce).
//
// The contraction runs over PIXELS, the slow index of both tensors.  With the samples of a chunk
// flattened to one pixel stream on out1's grid, P = (s*h1 + y)*w1 + x, and d2 zero-padded to that
// grid, a filter tap is a constant shift:  gW[t] = sum_P d2pad[P] (x) out1[P + dy*w1 + dx].
// tcgen05 takes MN-major (transposed) FP16 operands whose K rows (pixels) are 16 bytes apart
// (tools/probe/mn16_probe.cu), which is exactly a "plane" [8-channel group][pixel][8 halves] --
// and a 16-byte shifted base address shifts the pixel index by one.  So out1 is converted ONCE
// into FP16 hi/lo planes in a shared-memory ring, and every tap reads the same planes at its
// own offset: no im2col, no transposes.
//
// The whole gradient (1600 x 32 floats) has to stay in tensor memory (256 KB), so an
// accumulator row holds (tap, n): the A operand is M = 128 = 4 shifted copies of the d2 tile
// (32 channels each), one MMA = 4 taps.  Copy sets:  H = shifts {0,-1,-2,-3} (4 dx of one dy),
// V = shifts {0,-w1,-2w1,-3w1} (4 dy of dx = 4).  7 groups x 64 columns = 448 columns:
//     g = 0..4: set H, out1 shift dy*w1          -> taps (dy = g, dx = 0..3)
//     g = 5   : set V, out1 shift 4              -> taps (dy = 0..3, dx = 4)
//     g = 6   : set H, out1 shift 4*w1 + 4       -> tap (4, 4) (+ 3 unused rows)
// Operands are split x*s = hi + lo (unscaled lo, power-of-two s from the tensors' maxima); the
// three products share the accumulator.  21 MMAs (M128 N64 K16) per 16 pixels.
//
//   PA (8 warps)  d2 tile -> 8 shifted, masked copies (hi/lo) + bias sums       -> full_a[stage]
//   PB (4 warps)  out1 block of 16 pixels -> planes of the ring (hi/lo)         -> bfull[slot]
//   I0, I1        groups {0,2,4,6} / {1,3,5}: 3 products each                   -> empty_a, bempty
//   epilogue      (PA warps 0-3) TMEM -> per-CTA partial [t][k][n] | [n]
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "context.cuh"
#include "conv5_tc.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace wg5 {

struct Cfg {
  static constexpr int F = 5, T = 25, K = 64, N = 32;   // taps, input / output channels
  static constexpr int KS = 16;                         // pixels per K-step (one f16 MMA)
  static constexpr int RBN = 32;                        // ring blocks of 16 pixels
  static constexpr int RPX = RBN * KS + KS;             // plane entries: ring + mirror block
  // bytes per 8-channel plane, + 16: the four plane pairs a quarter-warp of PB threads writes
  // then start 32 bytes apart modulo 128 (all in the same banks without it: 16 instead of 4
  // wavefronts per store, profiles/r2s)
  static constexpr int PLANE = RPX * 16 + 16;
  static constexpr int oBh = 0, oBl = oBh + 8 * PLANE;  // out1 hi / lo: 8 planes each
  static constexpr int NSTAGE = 3;
  static constexpr int TILE = 16 * KS * 16;             // one A tile: 16 groups x 16 px x 16 B
  static constexpr int STAGE = 4 * TILE;                // H_hi, H_lo, V_hi, V_lo
  static constexpr int oA = oBl + 8 * PLANE;
  static constexpr size_t SMEM_BYTES = (size_t)oA + NSTAGE * STAGE;
  static constexpr int N_PA = 8, W_PB = N_PA, N_PB = 4, W_I = W_PB + N_PB, NT = (W_I + 2) * 32;
  static constexpr int NG = 7;
  static constexpr uint32_t TMEM_COLS = 512;
  static constexpr int MAX_W1 = 100;                    // 4*w1 + 20 <= 16 * (RBN - 4)
  static_assert(SMEM_BYTES + 1024 <= 232448, "shared memory");
};

__host__ __device__ __forceinline__ uint32_t idesc_f16_mn(int Mm, int Nn) {
  // c F32, a/b F16, A and B MN-major (transposed)
  return (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(Nn >> 3) << 17) | ((uint32_t)(Mm >> 4) << 24);
}

struct Args {
  const float* d2;        // [S][oh2][ow2][32]
  const float* out1;      // [S][h1][w1][64]
  float* partial;         // [grid][(1600 + 1) * 32]
  const unsigned* d2_max;     // bit patterns of the tensors' |x| maxima
  const unsigned* out1_max;
  int S, w1, h1;
  long long total_px;     // S * h1 * w1
  int blocks_per_cta;     // 16-pixel blocks of the flat stream per CTA
};

__global__ void __launch_bounds__(Cfg::NT, 1) wgrad5_tc_kernel(Args a) {
  using C = Cfg;
  using namespace tc;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_a[C::NSTAGE], empty_a[C::NSTAGE], bfull[C::RBN],
      bempty[C::RBN], done;
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int w1 = a.w1, h1 = a.h1, ow2 = w1 - (C::F - 1), oh2 = h1 - (C::F - 1);
  const long long Q0 = (long long)blockIdx.x * a.blocks_per_cta * C::KS;
  const long long Q1 = min(a.total_px, Q0 + (long long)a.blocks_per_cta * C::KS);
  // K-steps: this CTA's pixels plus the largest lag of a copy (3 * w1)
  const int n_ks = Q1 > Q0 ? (int)((Q1 - Q0 + 3 * w1 + C::KS - 1) / C::KS) : 0;
  const int NB = (4 * w1 + 4 + C::KS + C::KS - 1) / C::KS;   // ring blocks one K-step reads
  const int n_blocks = n_ks + NB - 1;                        // out1 blocks this CTA loads

  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    if (smem_u32(smem_raw) & 127u) __trap();
    for (int i = 0; i < C::NSTAGE; i++) {
      mbar_init(&full_a[i], C::N_PA * 32);
      mbar_init(&empty_a[i], 2);
    }
    for (int i = 0; i < C::RBN; i++) {
      mbar_init(&bfull[i], 64);
      mbar_init(&bempty[i], 2);
    }
    mbar_init(&done, 2);
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  const float s_d = c5::scale_for(__uint_as_float(__ldg(a.d2_max)));
  const float s_o = c5::scale_for(__uint_as_float(__ldg(a.out1_max)));
  float* part = a.partial + (size_t)blockIdx.x * ((size_t)(C::T * C::K + 1) * C::N);

  if (warp < C::N_PA) {
    // ============================ PA: the 8 shifted copies of the d2 tile ======================
    // thread = (set, copy j, pixel kk, 16-channel half): value d2pad[Q0 + 16 i + kk - lag]
    // (the channel half in lane bit 0 costs the stores a 2-way bank conflict -- the two
    // destinations are 512 bytes apart -- but keeps a quarter-warp's loads within 4 lines; with the
    // pixel in the low bits the stores are conflict-free and the chunk's gradients 10 % SLOWER)
    const int set = tid >> 7, j = (tid >> 5) & 3, kk = (tid >> 1) & 15, half = tid & 1;
    const int lag = set == 0 ? j : j * w1;
    // first K-step whose pixel is not before Q0, and that pixel's (sample, y, x)
    const int i0 = lag > kk ? (lag - kk + C::KS - 1) / C::KS : 0;
    long long q = Q0 + (long long)i0 * C::KS + kk - lag;
    int sx, sy;
    long long ss;
    {
      const long long per = (long long)h1 * w1;
      ss = q / per;
      const int rem = (int)(q - ss * per);
      sy = rem / w1;
      sx = rem - sy * w1;
    }
    // tile offsets of this thread's two 8-channel groups: group = 4 j + 2 half + c
    uint8_t* dst = smem_raw + C::oA + (set * 2) * C::TILE + (4 * j + 2 * half) * (C::KS * 16) + kk * 16;
    float gb[16];
#pragma unroll
    for (int c = 0; c < 16; c++) gb[c] = 0.f;
    const bool bias_thread = set == 0 && j == 0;
    // loads run two K-steps ahead of their use (v: this K-step, vn: the next)
    float4 v[4], vn[4];
    auto load = [&](float4 (&dstv)[4], int i) {
      const bool ok = i >= i0 && i < n_ks && q < Q1 && sy < oh2 && sx < ow2;
      if (ok) {
        const float4* p = reinterpret_cast<const float4*>(
            a.d2 + (((size_t)ss * oh2 + sy) * ow2 + sx) * C::N + half * 16);
#pragma unroll
        for (int c = 0; c < 4; c++) dstv[c] = __ldg(p + c);
      } else {
#pragma unroll
        for (int c = 0; c < 4; c++) dstv[c] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (i >= i0) {   // advance to the pixel of the next K-step
        q += C::KS;
        sx += C::KS;
        while (sx >= w1) { sx -= w1; sy++; }
        while (sy >= h1) { sy -= h1; ss++; }
      }
    };
    if (n_ks > 0) { load(v, 0); load(vn, 1); }
    for (int i = 0; i < n_ks; i++) {
      const int stage = i % C::NSTAGE;
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int c = 0; c < 4; c++) {
        split_h2(v[c].x * s_d, v[c].y * s_d, hi[2 * c], lo[2 * c]);
        split_h2(v[c].z * s_d, v[c].w * s_d, hi[2 * c + 1], lo[2 * c + 1]);
        if (bias_thread) {
          gb[4 * c] += v[c].x; gb[4 * c + 1] += v[c].y; gb[4 * c + 2] += v[c].z; gb[4 * c + 3] += v[c].w;
        }
      }
#pragma unroll
      for (int c = 0; c < 4; c++) v[c] = vn[c];
      load(vn, i + 2);                 // in flight while waiting for the stage
      if (i >= C::NSTAGE) mbar_wait(&empty_a[stage], (uint32_t)(((i / C::NSTAGE) - 1) & 1));
      uint8_t* s = dst + stage * C::STAGE;
      *reinterpret_cast<uint4*>(s) = make_uint4(hi[0], hi[1], hi[2], hi[3]);                        // hi, group c=0
      *reinterpret_cast<uint4*>(s + C::KS * 16) = make_uint4(hi[4], hi[5], hi[6], hi[7]);           // hi, group c=1
      *reinterpret_cast<uint4*>(s + C::TILE) = make_uint4(lo[0], lo[1], lo[2], lo[3]);              // lo tile
      *reinterpret_cast<uint4*>(s + C::TILE + C::KS * 16) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      fence_proxy_async();
      mbar_arrive(&full_a[stage]);
    }
    // bias gradient: warp 0 holds every pixel of the CTA exactly once (set H, copy 0)
    if (warp == 0) {
#pragma unroll
      for (int c = 0; c < 16; c++) {
        float s = gb[c];
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        s += __shfl_xor_sync(0xffffffffu, s, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if (lane < 2) part[(size_t)C::T * C::K * C::N + lane * 16 + c] = s;
      }
    }
    // ============================ epilogue: accumulators -> partial [t][k][n] =================
    if (warp < 4) {
      mbar_wait(&done, 0);
      tcgen05_fence_after();
      const uint32_t lane_base = (uint32_t)(warp * 32) << 16;   // TMEM lane = 32 * copy + n
      const int cj = warp, n = lane;
      const float cs = 1.f / (s_d * s_o);
      for (int g = 0; g < C::NG; g++) {
        int t;
        if (g < 5) t = g * C::F + cj;          // set H: (dy = g, dx = copy)
        else if (g == 5) t = cj * C::F + 4;    // set V: (dy = copy, dx = 4)
        else t = cj == 0 ? C::T - 1 : -1;      // (4, 4)
#pragma unroll
        for (int kc = 0; kc < C::K / 16; kc++) {
          float v16[16];
          tmem_ld16_nowait(tmem + lane_base + (uint32_t)(g * C::K + kc * 16), v16);
          tmem_ld_wait();
          if (t >= 0) {
#pragma unroll
            for (int c = 0; c < 16; c++)
              part[((size_t)t * C::K + kc * 16 + c) * C::N + n] = n_ks > 0 ? v16[c] * cs : 0.f;
          }
        }
      }
    }
  } else if (warp < C::W_I) {
    // ============================ PB: out1 blocks -> planes of the ring =======================
    // a warp pair owns every other block; thread = (pixel, 16-channel slice)
    const int pair = (warp - C::W_PB) >> 1;
    const int pt = tid - (C::W_PB + 2 * pair) * 32;     // 0..63
    const int px = pt >> 2, sl = pt & 3;
    float4 v[4];
    auto load = [&](int b) {
      const long long gp = Q0 + (long long)b * C::KS + px;
      if (gp < a.total_px) {
        const float4* p = reinterpret_cast<const float4*>(a.out1 + (size_t)gp * C::K + sl * 16);
#pragma unroll
        for (int c = 0; c < 4; c++) v[c] = __ldg(p + c);
      } else {
#pragma unroll
        for (int c = 0; c < 4; c++) v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    if (pair < n_blocks) load(pair);
    for (int b = pair; b < n_blocks; b += 2) {
      const int slot = b % C::RBN;
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int c = 0; c < 4; c++) {
        split_h2(v[c].x * s_o, v[c].y * s_o, hi[2 * c], lo[2 * c]);
        split_h2(v[c].z * s_o, v[c].w * s_o, hi[2 * c + 1], lo[2 * c + 1]);
      }
      if (b + 2 < n_blocks) load(b + 2);
      if (b >= C::RBN) mbar_wait(&bempty[slot], (uint32_t)(((b / C::RBN) - 1) & 1));
      // planes 2 sl and 2 sl + 1 (8 channels each), entry slot * 16 + px (+ the mirror of slot 0)
      uint8_t* h = smem_raw + C::oBh + (2 * sl) * C::PLANE + (slot * C::KS + px) * 16;
      uint8_t* l = smem_raw + C::oBl + (2 * sl) * C::PLANE + (slot * C::KS + px) * 16;
      const uint4 h0 = make_uint4(hi[0], hi[1], hi[2], hi[3]), h1v = make_uint4(hi[4], hi[5], hi[6], hi[7]);
      const uint4 l0 = make_uint4(lo[0], lo[1], lo[2], lo[3]), l1v = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      *reinterpret_cast<uint4*>(h) = h0;
      *reinterpret_cast<uint4*>(h + C::PLANE) = h1v;
      *reinterpret_cast<uint4*>(l) = l0;
      *reinterpret_cast<uint4*>(l + C::PLANE) = l1v;
      if (slot == 0) {
        constexpr int MIR = C::RBN * C::KS * 16;
        *reinterpret_cast<uint4*>(h + MIR) = h0;
        *reinterpret_cast<uint4*>(h + C::PLANE + MIR) = h1v;
        *reinterpret_cast<uint4*>(l + MIR) = l0;
        *reinterpret_cast<uint4*>(l + C::PLANE + MIR) = l1v;
      }
      fence_proxy_async();
      mbar_arrive(&bfull[slot]);
    }
  } else {
    // ============================ I0 / I1: MMA issuers ========================================
    const int me = warp - C::W_I;
    const uint32_t idesc = idesc_f16_mn(128, C::K);
    const uint32_t sA = smem_u32(smem_raw + C::oA);
    const uint32_t sBh = smem_u32(smem_raw + C::oBh), sBl = smem_u32(smem_raw + C::oBl);
    // MN-major, no swizzle: LBO = 128 (next 8 K rows), SBO = stride between 8-element M/N groups
    auto desc = [](uint32_t addr, uint32_t sbo) -> uint64_t {
      return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) |
             ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
    };
    for (int i = 0; i < n_ks; i++) {
      const int stage = i % C::NSTAGE;
      mbar_wait(&full_a[stage], (uint32_t)((i / C::NSTAGE) & 1));
      {   // the last ring block this K-step reads (blocks are filled in order)
        const int b = i + NB - 1;
        mbar_wait(&bfull[b % C::RBN], (uint32_t)((b / C::RBN) & 1));
        // ... and the one before it, filled by the other warp pair
        const int b1 = b - 1;
        if (b1 >= 0) mbar_wait(&bfull[b1 % C::RBN], (uint32_t)((b1 / C::RBN) & 1));
      }
      tcgen05_fence_after();
      if (elect_one()) {
        const uint32_t st = sA + stage * C::STAGE;
        const uint32_t ring = (uint32_t)((i % C::RBN) * C::KS * 16);   // entry of local pixel 16 i
#pragma unroll
        for (int g = me; g < C::NG; g += 2) {
          const uint32_t set = g == 5 ? 1u : 0u;
          const uint32_t shift = g < 5 ? (uint32_t)(g * w1) : (g == 5 ? 4u : (uint32_t)(4 * w1 + 4));
          // ring entry of the first pixel: (16 i + shift) mod ring length; the mirror block
          // makes the 16-pixel read contiguous
          const uint32_t e = (ring + shift * 16u) % (uint32_t)(C::RBN * C::KS * 16);
          const uint64_t ah = desc(st + set * 2 * C::TILE, C::KS * 16);
          const uint64_t al = desc(st + set * 2 * C::TILE + C::TILE, C::KS * 16);
          const uint64_t bh = desc(sBh + e, C::PLANE), bl = desc(sBl + e, C::PLANE);
          const uint32_t d = tmem + (uint32_t)(g * C::K);
          mma_f16_ss(d, ah, bh, idesc, i > 0 ? 1u : 0u);
          mma_f16_ss(d, ah, bl, idesc, 1u);
          mma_f16_ss(d, al, bh, idesc, 1u);
        }
        mma_commit(&empty_a[stage]);
        mma_commit(&bempty[i % C::RBN]);
        if (i == n_ks - 1) mma_commit(&done);
      }
      __syncwarp();
    }
    if (n_ks == 0 && elect_one()) mbar_arrive(&done);
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
}

// returns 1 when it launched (partials in ctx->splitk_scratch, *count of them), 0 when the shape
// is not handled, < 0 on error.  `mx` holds the maxima of out1 and d2 (c5::Maxes).
inline int wgrad5_tc(srcnn_ctx* ctx, const float* d2, const float* out1, const c5::Maxes* mx, int n,
                     int k, int f, int ow2, int oh2, int S, int* count) {
  using C = Cfg;
  if (n != C::N || k != C::K || f != C::F) return 0;
  const int w1 = ow2 + f - 1, h1 = oh2 + f - 1;
  if (w1 > C::MAX_W1) return 0;
  const long long total = (long long)S * h1 * w1;
  if (total >= (1LL << 40)) return 0;
  SRCNN_TRY(ensure_func_setup(ctx, wgrad5_tc_kernel, C::SMEM_BYTES));
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  const long long nblk = (total + C::KS - 1) / C::KS;
  const int grid = (int)std::min<long long>(sms, std::max<long long>(1, nblk / 8));
  const long long per = (nblk + grid - 1) / grid;
  if (per > 0x7fffffffLL / C::KS) return 0;
  *count = grid;
  SRCNN_TRY(ensure_scratch(ctx, &ctx->splitk_scratch, &ctx->splitk_bytes,
                           sizeof(float) * (size_t)grid * (C::T * C::K + 1) * C::N));
  Args a{d2, out1, (float*)ctx->splitk_scratch, &mx->d2, &mx->out1, S, w1, h1, total, (int)per};
  wgrad5_tc_kernel<<<grid, C::NT, C::SMEM_BYTES, ctx->stream>>>(a);
  return 1;
}

}  // namespace wg5
}  // namespace srcnn
