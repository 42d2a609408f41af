// The two 5x5 contractions over ACTIVATIONS of the 9-5-5 network (BASELINE config C4) on the
// 5th-gen tensor cores, one kernel template:
//
//   MODE 0  layer-2 forward   out2[s][y][x][n] = relu(b2[n] + sum_{dy,dx,k} W2[dy][dx][k][n] *
//                                                     out1[s][y+dy][x+dx][k])          (K = 25*64)
//           reference: src/kernel/layer_uber_kernel.cl:36-96 with F_SPATIAL_SIZE=5,
//           PREVIOUS_FILTER_COUNT=64, CURRENT_FILTER_COUNT=32
//   MODE 1  layer-1 deltas    d1[s][j][i][n] = [out1[s][j][i][n] > 0] * sum_{dy,dx,k}
//                                              W2[dy][dx][n][k] * d2[s][j-dy][i-dx][k]  (K = 25*32)
//           reference: src/kernel/layer_deltas.cl:42-127 (zero outside d2's extent)
//
// Both are "out[y][x][co] = sum_{dy,dx,ci} Wg[dy][dx][ci][co] * in[y+dy-P][x+dx-P][ci]" (P = 0 /
// 4, in = 0 outside; for MODE 1 Wg is W2 with the taps flipped and the channel roles swapped),
// i.e. implicit GEMMs  M = pixels, N = co, K = 25 taps x ci.
//
// No im2col.  The samples of a chunk (33x33 patches -> 25x25 maps) lie side by side as one
// VIRTUAL image whose slots are 25 columns wide (MODE 1: a 21-wide d2 row + 4 zero columns, which
// also are the left padding of the next sample).  A CTA owns a strip of 128 virtual output
// columns and marches down the INPUT rows.  One input row slice (132 pixels x 16 channels) is
// converted ONCE into FP16 hi/lo "planes" [8-channel chunk][pixel][8 halves]: with SBO = 128 the
// 128 rows of a K-major A operand are consecutive 16-byte units, so the tile of tap (dy, dx) is
// the same plane read at base + dx*16 bytes -- the 25 taps of an input row reuse one conversion
// and one shared-memory copy.  The 5 output rows an input row contributes to (dy = 0..4) each
// have their own accumulator in tensor memory, side by side in a ring of 16 (forward) / 8
// (deltas) slots (row rho in slot rho % NACC), so that ONE instruction A x [W(dy=4); ...; W(dy=0)] feeds all five (N = 5 * C_out
// = 160 forward; deltas 4 + 1 rows of 64): "dy-stacked" MMAs, see Cfg.  A row leaves
// through the epilogue when its last input row has been issued.  W (hi | lo, 204 800 bytes)
// stays resident in shared memory, stored [hi | lo][dx][slice][(4 - dy) * C_out + n][16] so that
// a range of filter rows is one B operand.
//
// Precision: operands are split x*s = hi + lo into two halves (lo unscaled), products
// hi.hi + hi.lo + lo.hi: 22 operand bits, all three in ONE FP32 accumulator per output row
// (same scheme as the wide inference kernel, fused_forward_hpw.cuh; one issuer, so the
// summation order is fixed).  s is a power of two that
// maps the largest |x| of the tensor (found on the device by absmax_kernel) to 2^14; the
// weights likewise.
//
//   P  (5 warps)  input row slice -> split -> planes (loads two slices ahead)  -> full[slot]
//   I  (1 warp)   MMA issuer: per (slice, dx) one instruction per product and piece of the
//                 row range (pieces: where the ring wraps, and <= 256 / C_out rows)
//                                                                            -> empty[slot], done[acc]
//   E  (4 warps)  accumulator -> bias + relu / relu' mask -> global          -> acc_free[acc]
//                 (deltas: 16x256b fragments, mask loaded before the accumulator wait)
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "context.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace c5 {

// per-chunk device scalars: bit patterns of max |x| (non-negative floats order like unsigned)
struct Maxes {
  unsigned out1, d2, in, out2, d3;
};

// |x| maximum of a tensor, as an unsigned bit pattern (atomicMax); `out` must be zeroed first.
// `x` only needs float alignment: up to 3 leading and 3 trailing floats are read singly.
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ x, size_t n,
                                                     unsigned* out) {
  const size_t head = min(n, (size_t)((16 - (reinterpret_cast<uintptr_t>(x) & 15)) & 15) / 4);
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  const size_t n4 = (n - head) / 4;
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(x4 + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  if (blockIdx.x == 0) {
    if (threadIdx.x < head) m = fmaxf(m, fabsf(__ldg(x + threadIdx.x)));
    const size_t tail = head + 4 * n4;
    if (threadIdx.x < n - tail) m = fmaxf(m, fabsf(__ldg(x + tail + threadIdx.x)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

// 2^14 / pow2ceil(max): the scale that maps the tensor into the FP16 range with headroom
__host__ __device__ __forceinline__ float scale_for(float mx) {
  if (!(mx > 0.f) || !(mx < 1e30f)) return 1.f;
  int e;
  frexpf(mx, &e);   // mx = f * 2^e, f in [0.5, 1)
  return ldexpf(1.f, min(14 - e, 100));   // (a tensor of denormal-sized values keeps a finite scale)
}

constexpr int F = 5, T = F * F;

template <int CIN_, int COUT_, int MODE_>
struct Cfg {
  static constexpr int CIN = CIN_, COUT = COUT_, MODE = MODE_;
  static constexpr int KT = T * CIN;                  // K of the GEMM (halves per weight row)
  static constexpr int NSLICE = CIN / 16;             // 16-channel slices of an input row
  static constexpr int M = 128;                       // output pixels per strip
  static constexpr int PW = 136;                      // plane entries (>= M + F - 1)
  static constexpr int PB = PW * 16;                  // bytes per plane
  static constexpr int SLOT_BYTES = 4 * PB;           // hi chunk 0, hi chunk 1, lo chunk 0, lo chunk 1
  // dy-stacked MMAs: the five filter rows dy of an input row slice use the SAME A tile (same
  // input row, same dx shift) and only differ in the output row they feed.  With the
  // accumulators of consecutive output rows side by side in tensor memory, ONE instruction
  // A x [W(dy=4); W(dy=3); ... ; W(dy=0)] (N = 5 * COUT = 160) serves all five: 3 instructions per
  // (slice, dx), one per product, instead of 10, and each is math-bound (80 cycles of tensor math
  // against 72 of operand fetch) where the per-dy instructions were fetch-bound (94 cycles per 48
  // of math: the kernel's tensor pipe was 74 % busy at 39 % math, profiles/r3j_ncu_summary.txt).
  // Output row rho lives in slot rho % NACC; a range of rows that wraps around the ring is issued
  // as two instructions.  All three products of a row go into its one accumulator, issued by one
  // warp (the summation order is fixed).  The forward (C_out = 32) has 16 slots: a range of 5 rows
  // wraps in 4 of 16 input rows instead of 4 of 8 (chunk of 3 028 patches 2.229 -> 2.207 ms); the
  // deltas (C_out = 64) fill tensor memory with 8.
  static constexpr int NSLOT = 3, NACC = COUT_ * 16 <= 512 ? 16 : 8;
  static constexpr int BLK_BYTES = F * COUT * 32;     // image block of one (dx, slice)
  static constexpr int IMG_L = F * NSLICE * BLK_BYTES;   // byte offset of the W_lo blocks
  static constexpr int W_BYTES = 2 * COUT * KT * 2;   // [W_hi blocks ; W_lo blocks] halves
  static constexpr int oW = 0, oSlots = W_BYTES, oBias = oSlots + NSLOT * SLOT_BYTES;
  static constexpr size_t SMEM_BYTES = (size_t)oBias + COUT * 4;
  // warps: epilogue, plane producers, the MMA issuer
  static constexpr int W_E = 0, W_P = 4, N_P = 5, W_I = W_P + N_P, NT = (W_I + 1) * 32;
  static constexpr int ITEMS = (2 * PW + N_P * 32 - 1) / (N_P * 32);   // plane items per producer thread
  static constexpr uint32_t TMEM_COLS = 512;
  static_assert(NACC * COUT <= 512, "accumulators must fit tensor memory");
  static constexpr int MAXROWS = 256 / COUT;          // output rows per instruction (N <= 256)
  static_assert(CIN % 16 == 0 && COUT % 16 == 0, "channel counts");
  static_assert(SMEM_BYTES + 1024 <= 232448, "shared memory");
};

// header + packed weight images of the 9-5-5 layer 2 (fp16 hi | lo, canonical K-major), built
// once per parameter change by prepare_kernel
struct Images {
  float sw, inv_sw;        // weights were multiplied by sw
  float pad_[2];
  // [hi | lo][dx][slice][row = (4 - dy) * C_out + n][16 ci], every block canonical K-major
  // (8-row groups 256 bytes apart); n = n2 (forward) / n1 (deltas)
  unsigned char fwd[Cfg<64, 32, 0>::W_BYTES];
  unsigned char d1[Cfg<32, 64, 1>::W_BYTES];
};
static_assert(offsetof(Images, fwd) % 16 == 0 && offsetof(Images, d1) % 16 == 0, "uint4 copies");

// W2 [5][5][64][32] -> both images.  Every CTA recomputes max|W2| (51 200 loads) and packs its
// share.
__global__ void __launch_bounds__(256) prepare_kernel(const float* __restrict__ w2, Images* img) {
  __shared__ float red[8];
  __shared__ float s_sw;
  constexpr int N1 = 64, N2 = 32, NW = T * N1 * N2;
  float m = 0.f;
  for (int i = threadIdx.x; i < NW; i += 256) m = fmaxf(m, fabsf(__ldg(w2 + i)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    float r = red[0];
    for (int w = 1; w < 8; w++) r = fmaxf(r, red[w]);
    s_sw = scale_for(r);
    if (blockIdx.x == 0) {
      img->sw = s_sw;
      img->inv_sw = 1.f / s_sw;
    }
  }
  __syncthreads();
  const float sw = s_sw;
  __half* f = reinterpret_cast<__half*>(img->fwd);
  __half* d = reinterpret_cast<__half*>(img->d1);
  const int gtid = blockIdx.x * 256 + threadIdx.x, gn = gridDim.x * 256;
  {   // forward image: Wg[t][ci][n] = W2[t][ci][n]
    constexpr int KT = T * N1;
    for (int i = gtid; i < N2 * KT; i += gn) {
      const int n = i / KT, k = i % KT;            // k = t*64 + ci
      unsigned short hi, lo;
      tc::split_h(__ldg(w2 + (size_t)k * N2 + n) * sw, hi, lo);
      using FC = Cfg<64, 32, 0>;
      const int t = k / N1, ci = k % N1, dy = t / F, dx = t % F, c = ci / 16, kk = ci % 16;
      const int row = (F - 1 - dy) * N2 + n;
      const int off = ((dx * FC::NSLICE + c) * FC::BLK_BYTES) / 2 + (row >> 3) * 128 + (kk >> 3) * 64 +
                      (row & 7) * 8 + (kk & 7);
      f[off] = __ushort_as_half(hi);
      f[FC::IMG_L / 2 + off] = __ushort_as_half(lo);
    }
  }
  {   // deltas image: Wg[t][ci = k2][co = n1] = W2[24 - t][n1][k2]
    constexpr int KT = T * N2;
    for (int i = gtid; i < N1 * KT; i += gn) {
      const int n = i / KT, k = i % KT;            // k = t*32 + ci
      const int t = k / N2, ci = k % N2;
      unsigned short hi, lo;
      tc::split_h(__ldg(w2 + ((size_t)(T - 1 - t) * N1 + n) * N2 + ci) * sw, hi, lo);
      using DC = Cfg<32, 64, 1>;
      const int dy = t / F, dx = t % F, c = ci / 16, kk = ci % 16;
      const int row = (F - 1 - dy) * N1 + n;
      const int off = ((dx * DC::NSLICE + c) * DC::BLK_BYTES) / 2 + (row >> 3) * 128 + (kk >> 3) * 64 +
                      (row & 7) * 8 + (kk & 7);
      d[off] = __ushort_as_half(hi);
      d[DC::IMG_L / 2 + off] = __ushort_as_half(lo);
    }
  }
}

struct Args {
  const float* in;       // MODE 0: out1 [S][h1][w1][64];  MODE 1: d2 [S][h1-4][w1-4][32]
  const float* aux;      // MODE 0: b2 [32];               MODE 1: out1 (relu' mask)
  float* out;            // MODE 0: out2 [S][h1-4][w1-4][32];  MODE 1: d1 [S][h1][w1][64]
  const unsigned char* wimg;   // packed weight image of this mode
  const float* sw;       // -> Images::sw
  const unsigned* in_max;      // bit pattern of max |in|
  int S, w1, h1;         // samples, extent of the layer-1 map (25 x 25 for 33 x 33 patches)
  unsigned* out_max;     // MODE 0, may be null: receives max |out2| (zeroed by the launcher)
};

template <class C>
__global__ void __launch_bounds__(C::NT, 1) conv5_tc_kernel(Args a) {
  using namespace tc;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full[C::NSLOT], empty[C::NSLOT], done[C::NACC], acc_free[C::NACC];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int P = C::MODE == 0 ? 0 : F - 1;               // zero padding of the input
  const int iw = C::MODE == 0 ? a.w1 : a.w1 - (F - 1);       // input map extent
  const int ih = C::MODE == 0 ? a.h1 : a.h1 - (F - 1);
  const int ow = C::MODE == 0 ? a.w1 - (F - 1) : a.w1;       // output map extent
  const int oh = C::MODE == 0 ? a.h1 - (F - 1) : a.h1;
  const int slot_w = a.w1;                                   // virtual-image slot of one sample
  const long long vw = (long long)a.S * slot_w;              // virtual width
  const long long X0 = (long long)blockIdx.x * C::M;         // first output column of the strip

  // ---- resident B operand: the packed image, and the bias ------------------------------------
  {
    const uint4* src = reinterpret_cast<const uint4*>(a.wimg);
    uint4* dst = reinterpret_cast<uint4*>(smem_raw + C::oW);
    for (int i = tid; i < C::W_BYTES / 16; i += C::NT) dst[i] = __ldg(src + i);
    // plane pads are read by the tensor core (rows beyond the strip, times real weights, into
    // accumulator rows nobody stores): keep them finite
    uint32_t* z = reinterpret_cast<uint32_t*>(smem_raw + C::oSlots);
    for (int i = tid; i < C::NSLOT * C::SLOT_BYTES / 4; i += C::NT) z[i] = 0u;
    if (C::MODE == 0) {
      float* sB = reinterpret_cast<float*>(smem_raw + C::oBias);
      for (int i = tid; i < C::COUT; i += C::NT) sB[i] = __ldg(a.aux + i);
    }
  }
  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    if (smem_u32(smem_raw) & 127u) __trap();
    for (int i = 0; i < C::NSLOT; i++) {
      mbar_init(&full[i], C::N_P * 32);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < C::NACC; i++) {
      mbar_init(&done[i], 1);
      mbar_init(&acc_free[i], 128);
    }
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;

  const float s_in = scale_for(__uint_as_float(__ldg(a.in_max)));
  const float sw = __ldg(a.sw);

  if (warp >= C::W_P && warp < C::W_P + C::N_P) {
    // ============================ P: plane producers ==========================================
    // item = (plane entry q = virtual input column X0 - P + q, 8-channel chunk ch of the slice);
    // a thread owns items t and t + 160.  Two lanes per pixel: a quarter-warp's 16-byte loads
    // fall into 4 lines (one lane per pixel with the whole 64-byte slice: 8 lines per quarter
    // and 32 per instruction -- the L1 pipe these kernels are bound by counts lines)
    const int t = tid - C::W_P * 32;
    long long base[C::ITEMS];       // float offset of (sample, row 0, x, channel 8 ch), -1 = zero column
    uint8_t* my[C::ITEMS];
    bool live[C::ITEMS];
#pragma unroll
    for (int k = 0; k < C::ITEMS; k++) {
      const int item = t + k * (C::N_P * 32), q = item >> 1, ch = item & 1;
      const long long vin = X0 - P + q;
      base[k] = -1;
      live[k] = q < C::PW;
      if (q < C::PW && vin >= 0 && vin < vw) {
        const int smp = (int)(vin / slot_w), x = (int)(vin - (long long)smp * slot_w);
        if (x < iw) base[k] = (((long long)smp * ih) * iw + x) * C::CIN + ch * 8;
      }
      my[k] = smem_raw + C::oSlots + ch * C::PB + q * 16;
    }
    const long long row_stride = (long long)iw * C::CIN;
    // Loads run TWO slices ahead of their use (v = this slice, v1 = the next, v2 = the one after):
    // with the dy-stacked MMAs a slice is consumed every ~1 300 cycles, less than one HBM round
    // trip, so a single slice in flight per thread made the producers the bound.
    float4 v[C::ITEMS][2], v1[C::ITEMS][2], v2[C::ITEMS][2];
    auto load = [&](float4 (&dst)[C::ITEMS][2], int i) {   // slice index i = r * NSLICE + c
      const int r = i / C::NSLICE, c = i % C::NSLICE;
#pragma unroll
      for (int k = 0; k < C::ITEMS; k++) {
        if (base[k] >= 0 && r < ih) {
          const float4* p = reinterpret_cast<const float4*>(a.in + base[k] + r * row_stride + c * 16);
          dst[k][0] = __ldg(p);
          dst[k][1] = __ldg(p + 1);
        } else {
          dst[k][0] = dst[k][1] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    load(v, 0);
    load(v1, 1);
    int it = 0;
    for (int r = 0; r < ih; r++) {
      for (int c = 0; c < C::NSLICE; c++, it++) {
        const int slot = it % C::NSLOT;
        load(v2, it + 2);
        uint32_t hi[C::ITEMS][4], lo[C::ITEMS][4];
#pragma unroll
        for (int k = 0; k < C::ITEMS; k++)
#pragma unroll
          for (int j = 0; j < 2; j++) {
            split_h2(v[k][j].x * s_in, v[k][j].y * s_in, hi[k][2 * j], lo[k][2 * j]);
            split_h2(v[k][j].z * s_in, v[k][j].w * s_in, hi[k][2 * j + 1], lo[k][2 * j + 1]);
          }
#pragma unroll
        for (int k = 0; k < C::ITEMS; k++)
#pragma unroll
          for (int j = 0; j < 2; j++) { v[k][j] = v1[k][j]; v1[k][j] = v2[k][j]; }
        if (it >= C::NSLOT) mbar_wait(&empty[slot], (uint32_t)(((it / C::NSLOT) - 1) & 1));
#pragma unroll
        for (int k = 0; k < C::ITEMS; k++)
          if (live[k]) {
            uint8_t* sdst = my[k] + slot * C::SLOT_BYTES;
            *reinterpret_cast<uint4*>(sdst) = make_uint4(hi[k][0], hi[k][1], hi[k][2], hi[k][3]);
            *reinterpret_cast<uint4*>(sdst + 2 * C::PB) = make_uint4(lo[k][0], lo[k][1], lo[k][2], lo[k][3]);
          }
        fence_proxy_async();
        mbar_arrive(&full[slot]);
      }
    }
  } else if (warp >= C::W_I) {
    // ============================ I: MMA issuer ===============================================
    // Input row r feeds output rows rho = r - dy + P; a row is first touched at input row
    // max(rho - P, 0) (slice 0, dx = 0) and complete after input row min(rho - P + 4, ih - 1).
    const uint32_t sW = smem_u32(smem_raw + C::oW);
    const uint32_t sS = smem_u32(smem_raw + C::oSlots);
    auto adesc = [](uint32_t addr) -> uint64_t {        // K-major, LBO = plane stride, SBO = 128
      return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((C::PB >> 4) & 0x3FFF) << 16) |
             ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    };
    auto bdesc = [](uint32_t addr) -> uint64_t {        // image block: LBO = 128, SBO = 256
      return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) |
             ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
    };
    constexpr uint64_t kImgL = (uint64_t)(C::IMG_L >> 4);             // descriptor address units
    constexpr uint64_t kDx = (uint64_t)((C::NSLICE * C::BLK_BYTES) >> 4);
    int it = 0;
    for (int r = 0; r < ih; r++) {
      const int dy_lo = max(0, r + P - (oh - 1)), dy_hi = min(F - 1, r + P);
      // the instructions of one (slice, dx) step of this input row: rows of dy = dy_hi .. dy_lo
      // (rho ascending) -> slots (r - dy + P) % NACC, cut where the ring wraps and at MAXROWS
      // rows.  At most 3 pieces; computed once per input row, the issue loop only adds offsets.
      uint32_t seg_d[3], seg_i[3];
      uint64_t seg_b[3];
      int nseg = 0;
      auto cut = [&](int a0, int b0, uint32_t (&sd)[3], uint64_t (&sb)[3], uint32_t (&si)[3]) {
        int n_out = 0, b = b0;
#pragma unroll
        for (int q = 0; q < 3; q++)      // static indices: the tables stay in registers
          if (b >= a0) {
            const int s0 = (r - b + P) % C::NACC;
            const int n = min(min(b - a0 + 1, C::NACC - s0), C::MAXROWS);
            sd[q] = (uint32_t)(s0 * C::COUT);
            sb[q] = (uint64_t)(((F - 1 - b) * C::COUT * 32) >> 4);
            si[q] = make_idesc_f16(C::M, n * C::COUT);
            n_out = q + 1;
            b -= n;
          }
        return n_out;
      };
      nseg = cut(dy_lo, dy_hi, seg_d, seg_b, seg_i);
      for (int c = 0; c < C::NSLICE; c++, it++) {
        const int slot = it % C::NSLOT;
        mbar_wait(&full[slot], (uint32_t)((it / C::NSLOT) & 1));
        if (c == 0 && dy_lo == 0 && r + P >= C::NACC)   // row r + P starts: its slot's last row has left
          mbar_wait(&acc_free[(r + P) % C::NACC], (uint32_t)((((r + P) / C::NACC) - 1) & 1));
        tcgen05_fence_after();
        const uint32_t ah = sS + slot * C::SLOT_BYTES, al = ah + 2 * C::PB;
        if (elect_one()) {
          const uint64_t dah0 = adesc(ah), dal0 = adesc(al);
          const uint64_t blk0 = bdesc(sW + (uint32_t)(c * C::BLK_BYTES));
          // all products of the pieces, in a fixed order
          auto step = [&](uint64_t dah, uint64_t dal, uint64_t blk, int ns, const uint32_t (&sd)[3],
                          const uint64_t (&sb)[3], const uint32_t (&si)[3], uint32_t acc_flag) {
#pragma unroll
            for (int q = 0; q < 3; q++)
              if (q < ns) {
                mma_f16_ss(tmem + sd[q], dah, blk + sb[q], si[q], acc_flag);      // hi.w_hi
                mma_f16_ss(tmem + sd[q], dah, blk + kImgL + sb[q], si[q], 1u);    // hi.w_lo
                mma_f16_ss(tmem + sd[q], dal, blk + sb[q], si[q], 1u);            // lo.w_hi
              }
          };
          int dx0 = 0;
          if (c == 0 && (r == 0 || dy_lo == 0)) {      // rows start here: their first product overwrites
            uint32_t fd[3], fi[3];
            uint64_t fb[3];
            const int f_hi = r == 0 ? dy_hi : 0;       // at r = 0 every row is new, later only dy = 0
            int nf = cut(dy_lo, f_hi, fd, fb, fi);
            step(dah0, dal0, blk0, nf, fd, fb, fi, 0u);
            if (f_hi < dy_hi) {
              nf = cut(f_hi + 1, dy_hi, fd, fb, fi);
              step(dah0, dal0, blk0, nf, fd, fb, fi, 1u);
            }
            dx0 = 1;
          }
          if (dx0 == 0) step(dah0, dal0, blk0, nseg, seg_d, seg_b, seg_i, 1u);
#pragma unroll
          for (int dx = 1; dx < F; dx++)
            step(dah0 + dx, dal0 + dx, blk0 + dx * kDx, nseg, seg_d, seg_b, seg_i, 1u);
          if (c == C::NSLICE - 1)
            for (int dy = dy_lo; dy <= dy_hi; dy++) {
              const int rho = r - dy + P;
              if (r == min(rho - P + (F - 1), ih - 1)) mma_commit(&done[rho % C::NACC]);
            }
          mma_commit(&empty[slot]);
        }
        __syncwarp();
      }
    }
  } else if (C::MODE == 1) {
    // ============================ E: epilogue of the deltas ===================================
    // The accumulator is read as 16x256b fragments (the layout of an mma accumulator:
    // a thread holds 2 adjacent channels of rows lane/4 and lane/4 + 8 of a 16-lane half, for
    // every group of 8 channels), so that 4 lanes cover 32 contiguous bytes of a pixel and an
    // 8-byte access per lane touches 8 lines per instruction.  With one pixel per lane (64
    // channels = 256 bytes apart) every 16-byte access of a warp touched 32 lines, and the L1
    // pipe -- mask loads and d1 stores of the epilogue -- was what bound the kernel (81 % busy
    // at 53 % tensor-pipe activity, profiles/r3l_ncu_summary.txt).
    const int q4 = lane >> 2, l4 = lane & 3;
    long long ob[4];   // pixels (warp & 3) * 32 + j * 8 + lane / 4
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const long long vo = X0 + (warp & 3) * 32 + j * 8 + q4;
      ob[j] = -1;
      if (vo < vw) {
        const int smp = (int)(vo / slot_w), x = (int)(vo - (long long)smp * slot_w);
        if (x < ow) ob[j] = (((long long)smp * oh) * ow + x) * C::COUT + 2 * l4;
      }
    }
    const long long orow_f = (long long)ow * C::COUT;
    const float csf = 1.f / (s_in * sw);
    for (int rho = 0; rho < oh; rho++) {
      const int acc = rho % C::NACC;
      // the relu' mask of this row does not depend on the accumulator: all its loads are in
      // flight while the row's MMAs finish (issued after the wait, their HBM round trips --
      // several dependent batches per row -- were the row period)
      float2 gm[4][C::COUT / 8];
#pragma unroll
      for (int j = 0; j < 4; j++)
#pragma unroll
        for (int g = 0; g < C::COUT / 8; g++)
          gm[j][g] = ob[j] >= 0 ? __ldg(reinterpret_cast<const float2*>(a.aux + ob[j] + rho * orow_f + 8 * g))
                                : make_float2(0.f, 0.f);
      mbar_wait(&done[acc], (uint32_t)((rho / C::NACC) & 1));
      tcgen05_fence_after();
      uint32_t f[2][32];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32 + h * 16) << 16);
        const uint32_t ta = tl + (uint32_t)(acc * C::COUT);
        asm volatile(
            "tcgen05.ld.sync.aligned.16x256b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
            "%13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, "
            "[%32];"
            : "=r"(f[h][0]), "=r"(f[h][1]), "=r"(f[h][2]), "=r"(f[h][3]), "=r"(f[h][4]), "=r"(f[h][5]),
              "=r"(f[h][6]), "=r"(f[h][7]), "=r"(f[h][8]), "=r"(f[h][9]), "=r"(f[h][10]), "=r"(f[h][11]),
              "=r"(f[h][12]), "=r"(f[h][13]), "=r"(f[h][14]), "=r"(f[h][15]), "=r"(f[h][16]),
              "=r"(f[h][17]), "=r"(f[h][18]), "=r"(f[h][19]), "=r"(f[h][20]), "=r"(f[h][21]),
              "=r"(f[h][22]), "=r"(f[h][23]), "=r"(f[h][24]), "=r"(f[h][25]), "=r"(f[h][26]),
              "=r"(f[h][27]), "=r"(f[h][28]), "=r"(f[h][29]), "=r"(f[h][30]), "=r"(f[h][31])
            : "r"(ta));
      }
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&acc_free[acc]);
      // f[h][4 g + 2 s + e] = D[row h*16 + s*8 + lane/4][channel 8 g + 2 (lane%4) + e]
#pragma unroll
      for (int j = 0; j < 4; j++) {
        if (ob[j] < 0) continue;
        const int h = j >> 1, sidx = j & 1;
        float* o = a.out + ob[j] + rho * orow_f;
#pragma unroll
        for (int g = 0; g < C::COUT / 8; g++) {
          const float x0 = __uint_as_float(f[h][4 * g + 2 * sidx]) * csf;
          const float x1 = __uint_as_float(f[h][4 * g + 2 * sidx + 1]) * csf;
          *reinterpret_cast<float2*>(o + 8 * g) =
              make_float2(gm[j][g].x > 0.f ? x0 : 0.f, gm[j][g].y > 0.f ? x1 : 0.f);
        }
      }
    }
  } else {
    // ============================ E: epilogue of the forward ==================================
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int m = (warp & 3) * 32 + lane;
    const long long vout = X0 + m;
    long long obase = -1;   // float offset of (sample, row 0, x, channel 0) of the output
    if (vout < vw) {
      const int smp = (int)(vout / slot_w), x = (int)(vout - (long long)smp * slot_w);
      if (x < ow) obase = (((long long)smp * oh) * ow + x) * C::COUT;
    }
    const long long orow = (long long)ow * C::COUT;
    const float cs = 1.f / (s_in * sw);
    const float* sB = reinterpret_cast<const float*>(smem_raw + C::oBias);
    float omax = 0.f;
    for (int rho = 0; rho < oh; rho++) {
      const int acc = rho % C::NACC;
      mbar_wait(&done[acc], (uint32_t)((rho / C::NACC) & 1));
      tcgen05_fence_after();
      float v[C::COUT];
      const uint32_t c0 = (uint32_t)(acc * C::COUT);
#pragma unroll
      for (int g = 0; g < C::COUT / 16; g++)
        tmem_ld16_nowait(tmem + lane_base + c0 + g * 16, v + g * 16);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&acc_free[acc]);
      if (obase < 0) continue;
      float4* o = reinterpret_cast<float4*>(a.out + obase + rho * orow);
#pragma unroll
      for (int j = 0; j < C::COUT / 4; j++) {
        const float4 r = make_float4(fmaxf(fmaf(v[4 * j], cs, sB[4 * j]), 0.f),
                                     fmaxf(fmaf(v[4 * j + 1], cs, sB[4 * j + 1]), 0.f),
                                     fmaxf(fmaf(v[4 * j + 2], cs, sB[4 * j + 2]), 0.f),
                                     fmaxf(fmaf(v[4 * j + 3], cs, sB[4 * j + 3]), 0.f));
        o[j] = r;
        omax = fmaxf(fmaxf(omax, fmaxf(r.x, r.y)), fmaxf(r.z, r.w));
      }
    }
    if (a.out_max) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) omax = fmaxf(omax, __shfl_xor_sync(0xffffffffu, omax, o));
      if (lane == 0 && omax > 0.f) atomicMax(a.out_max, __float_as_uint(omax));
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
}

using FwdCfg = Cfg<64, 32, 0>;
using D1Cfg = Cfg<32, 64, 1>;

inline bool supported(int n1, int n2, int f1, int f2, int f3) {
  (void)f1; (void)f3;
  return n1 == 64 && n2 == 32 && f2 == F;
}

// the packed weight images of `w2`, cached per context while w2 is untouched (see
// srcnn_ctx::c5_*); `cacheable` as for the fused inference operand image
inline int prepare(srcnn_ctx* ctx, const float* w2, bool cacheable, const Images** out) {
  if (!ctx->c5_images) SRCNN_CUDA(cudaMalloc(&ctx->c5_images, sizeof(Images)));
  if (!(cacheable && ctx->c5_valid && ctx->c5_key == w2)) {
    prepare_kernel<<<16, 256, 0, ctx->stream>>>(w2, reinterpret_cast<Images*>(ctx->c5_images));
    ctx->launch_count++;
    ctx->c5_valid = cacheable;
    ctx->c5_key = w2;
  }
  *out = reinterpret_cast<const Images*>(ctx->c5_images);
  return SRCNN_OK;
}

// max |x| of n floats into *slot (zeroed here)
inline int absmax(srcnn_ctx* ctx, const float* x, size_t n, unsigned* slot) {
  SRCNN_CUDA(cudaMemsetAsync(slot, 0, sizeof(unsigned), ctx->stream));
  const size_t n4 = n / 4;
  const int blocks = (int)std::min<size_t>((n4 + 255) / 256, (size_t)ctx->sm_count * 8);
  absmax_kernel<<<blocks > 0 ? blocks : 1, 256, 0, ctx->stream>>>(x, n, slot);
  ctx->launch_count++;
  return SRCNN_OK;
}

template <class C>
inline int launch(srcnn_ctx* ctx, const Args& a) {
  SRCNN_TRY(ensure_func_setup(ctx, conv5_tc_kernel<C>, C::SMEM_BYTES));
  const long long vw = (long long)a.S * a.w1;
  const long long strips = (vw + C::M - 1) / C::M;
  if (strips > 0x7fffffffLL) return fail(SRCNN_EINVAL, "chunk too large for one conv5 launch");
  conv5_tc_kernel<C><<<(unsigned)strips, C::NT, C::SMEM_BYTES, ctx->stream>>>(a);
  return SRCNN_OK;
}

}  // namespace c5
}  // namespace srcnn
