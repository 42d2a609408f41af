// Fused SRCNN inference, FP16-split tensor-core version (9-1-5, n1=64, n2=32).
//
// Same structure as fused_forward_pl.cuh (plane operands, one MMA issuer per layer, in-place
// TMEM operands, every buffer double) but every operand is split into two HALVES instead of two
// TF32 terms:
//     x * s = hi + lo               hi = half(x*s), lo = half(x*s - hi)
// with s a power of two that puts the operand range at ~2^14: lo only becomes an FP16 subnormal
// for values below 2^-25 of that range, where its absolute error (2^-25) is 2^-39 of the range.
// (An earlier version kept lo * 2048 to stay clear of subnormals; the multiply and the
// rescaling FMA in the epilogues cost 7 % of the kernel: 0.982 -> 0.914 ms on C3.)  x.w is
// evaluated as hi.w_hi + (hi.w_lo + lo.w_hi): the first product accumulates in one half of the
// (stacked) accumulator, the two correction products in the other (one N = 2n MMA + one N = n
// MMA per K-step), and the epilogue adds them.  Accuracy is that of the 3xTF32 scheme (22
// mantissa bits per operand; probe/f16_probe.cu: 2.5e-7 max error on a 9x9x64 tile), but
//   * kind::f16 MMAs take K = 16 per instruction: 6 + 4 + 2 K-steps per tile instead of
//     11 + 8 + 4, i.e. 24 instructions instead of 46, ~1 050 pipe cycles instead of ~2 050;
//   * layer 1 reads "oct planes" O(s)[c] = rows s..s+7 of column c (8 halves = 16 bytes) and
//     H8(r)[c] = in[r][c..c+7]: one O and one H8 plane per tile;
//   * A2/A3 are packed half pairs: half the TMEM store traffic of the epilogues.
//
// Range.  The scales depend on the WEIGHTS only (computed on the device by hp_prepare_kernel;
// cached per context until a device-layer call writes device memory; data-independent, so a row-band partition of an image reproduces the
// single-launch result bit for bit) and assume |input| < 64, 64x the luma range:
//     sx = 2^9;  sw_l = 2^14 / pow2ceil(max|W_l|);  s_l = 2^14 / pow2ceil(bound on out_l)
// with bound(out1) = max_n(|b1| + sum|W1|) * 64 and bound(out2) likewise from bound(out1).
// The plane producers check every input pixel they load: the first |x| >= 64 (or NaN) clears the
// `ok` flag, and the TF32 kernel -- launched right behind this one with the flag as its gate --
// redoes the whole launch.  No result ever depends on an FP16 overflow.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstddef>

#include "context.cuh"
#include "fused_forward.cuh"
#include "fused_forward_pl.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace fused_hp {

struct Cfg {
  static constexpr int N1 = 64, N2 = 32, F1 = 9, F3 = 5;
  static constexpr int M = 128;
  static constexpr int OW3 = M - (F3 - 1);
  static constexpr int KS1 = 6, K1 = KS1 * 16;   // halves: 81 taps + 15 zero weights
  static constexpr int K2 = N1, K3 = N2, NT3 = 32, QP = F3 * F3;
  static constexpr int PW = 144;                 // plane entries (16 bytes = 8 halves each)
  static constexpr int PB = PW * 16;             // bytes per plane
  static constexpr int RO = 4, RH = 4;           // ring slots: oct planes, H8 planes
  // role -> warp ids.  Every E role needs warp % 4 = its TMEM lane quarter, so E blocks start at
  // multiples of 4.
  static constexpr int W_E1 = 0, N_E1 = 8, W_E2 = N_E1, W_E3 = W_E2 + 4, W_IM = W_E3 + 4,
                       N_IM = 5, W_I1 = W_IM + N_IM, W_I2 = W_I1 + 1, W_I3 = W_I2 + 1;
  static constexpr int NT = (W_I3 + 1) * 32;
  static constexpr int E1_CHUNKS = (N1 / 16) / (N_E1 / 4);   // 16-channel chunks per E1 warp
  static constexpr int IM_THREADS = N_IM * 32;
  // shared memory carve-up (bytes).  The H8 ring lies ABOVE the oct ring: one K-step pairs the
  // dx = 8 chunk of O with the first chunk of H8 through a positive leading-dimension offset.
  static constexpr int oOh = 0;
  static constexpr int oOl = oOh + RO * PB;
  static constexpr int oHh = oOl + RO * PB;
  static constexpr int oHl = oHh + RH * PB;
  static constexpr int oW1 = oHl + RH * PB;          // [128][K1] halves: rows 0..63 hi, 64.. lo
  static constexpr int oW2 = oW1 + 2 * N1 * K1 * 2;  // [64][K2]
  static constexpr int oW3 = oW2 + 2 * N2 * K2 * 2;  // [64][K3]: rows = taps (25 of 32), hi, lo
  static constexpr int oB1 = oW3 + 2 * NT3 * K3 * 2; // b1 * s1 (floats)
  static constexpr int oB2 = oB1 + N1 * 4;           // b2 * s2
  static constexpr int oQs = oB2 + N2 * 4;           // 2 staged Q rows [M][QP] floats
  static constexpr int TOTAL = oQs + 2 * M * QP * 4;
  static constexpr size_t SMEM_BYTES = (size_t)TOTAL;
  // training forward (out1 / out2 kept): each E1 / E2 warp stages its 32 pixels x 32 channels
  // of a tile in shared memory and writes them out as full 128-byte lines
  static constexpr int SP = 36;                        // floats per staged pixel (128 B + pad)
  static constexpr int oS1 = TOTAL;                    // E1: N_E1 warps x 32 px x SP
  static constexpr int oS2 = oS1 + N_E1 * 32 * SP * 4; // E2: 4 warps
  static constexpr size_t SMEM_BYTES_KEEP = (size_t)(oS2 + 4 * 32 * SP * 4);
  static_assert(E1_CHUNKS == 2 && N2 == 32, "staging assumes 32 channels per warp");
  // tensor memory columns (+ size * (b & 1)):
  //   D1: [0,64) hi.w_hi, [64,128) corrections  ->  A2: hi pairs of channels 16g..16g+15 at
  //       a2col(g) = 32*(g/2) + 8*(g%2), lo pairs at 64 + a2col(g): inside the columns the SAME
  //       E1 warp has already read
  //   D2: [0,32), [32,64)                       ->  A3: [0,16) hi pairs, [32,48) lo pairs
  //   D3: [0,32), [32,64) (25 taps of 32 used)
  static constexpr uint32_t cD1 = 0, cD2 = 256, cD3 = 384;
  // layers 2 and 3 with ONE accumulator: three N = n instructions per K-step (hi.w_hi, hi.w_lo,
  // lo.w_hi -- the low halves are unscaled, so the three products share a scale) instead of a
  // stacked N = 2n one + an N = n one.  The tensor pipe pays ~5 cycles more per K-step (A from
  // tensor memory: 20.5 cycles at N = 32, 36 at N = 64, tools/probe/ts_probe.cu); E2 / E3 lose
  // the addition of the two accumulator halves and half their tensor-memory loads.
#ifndef HP_ACC1_23
#define HP_ACC1_23 0
#endif
  static constexpr bool ACC1_23 = HP_ACC1_23 != 0;
  static constexpr uint32_t A3LO = ACC1_23 ? 16 : N2;   // column of A3's low half pairs
  // A2 in its OWN tensor-memory columns (needs the single-accumulator layers 2 / 3 to fit):
  // D1[b&1] is free again as soon as E1 has LOADED it, not after E1 has converted it and MMA-2
  // has read the result -- the loop MMA-1(b) -> E1(b) -> MMA-2(b) -> MMA-1(b+2) over the two D1
  // buffers was the tile period (tools/hp_prof.py: I1 waited 530 of 1 900 cycles per tile for it)
#ifndef HP_A2SEP
#define HP_A2SEP 0
#endif
  static constexpr bool A2SEP = HP_A2SEP != 0;
  static_assert(!A2SEP || ACC1_23, "separate A2 columns need the single-accumulator layers");
  static constexpr uint32_t cA2 = A2SEP ? 256 : cD1, sA2 = A2SEP ? 64 : 128;   // base, stride
  static constexpr uint32_t cD2x = A2SEP ? 384 : cD2, sD2 = A2SEP ? 32 : 64;
  static constexpr uint32_t cD3x = A2SEP ? 448 : cD3, sD3 = A2SEP ? 32 : 64;
  // column of chunk g's (16 channels) hi pairs inside an A2 buffer, and offset of the lo pairs
  __host__ __device__ static constexpr uint32_t a2col(uint32_t g) {
    return A2SEP ? 8u * g : 32u * (g >> 1) + 8u * (g & 1);
  }
  static constexpr uint32_t A2LO = A2SEP ? 32 : N1;
  static constexpr uint32_t TMEM_COLS = 512;
  static constexpr int BAR_E3 = 1;
};

struct ScaleVals {
  float sx, sw1, sw2, sw3, s1, s2;
  float c1s;      // s1 / (sx * sw1): D1 -> out1 * s1
  float c2s;      // s2 / (s1 * sw2): D2 -> out2 * s2
  float c3;       // 1 / (s2 * sw3):  D3 -> Q
  float inv_s1, inv_s2;
  int ok;         // 1: the input is inside the FP16 domain, this kernel runs; 0: the TF32 one
  float in_lim;   // |input| must stay below this (64 unless the scale was derived from the data)
};
// what hp_prepare_kernel leaves for the main kernel: the scales and the ready-made shared-memory
// image of the B operands (scaled, split, in the canonical K-major layout) and scaled biases, so
// that a CTA's prologue is a 37 KB copy instead of 24 576 scattered conversions -- the CTAs of a
// training chunk or of a multi-GPU row band only live for 25..130 tiles
struct Scales {
  ScaleVals v;
  int pad_[4 - (sizeof(ScaleVals) / 4) % 4];
  unsigned char wimg[Cfg::oQs - Cfg::oW1];
};
static_assert(offsetof(Scales, wimg) % 16 == 0 && sizeof(Scales) % 16 == 0, "uint4 copies");

// (K-step s, 16-byte chunk j, element e) of the layer-1 contraction -> filter tap, or -1.
// chunks 0..8: O at dx = chunk (taps dy = e); chunk 9: H8 at dx' = 0 (taps (8, e));
// chunk 10: H8 at dx' = 8 (tap (8,8) + 7 pads); chunk 11: pad
__host__ __device__ __forceinline__ int tap16(int s, int j, int e) {
  const int c = 2 * s + j;
  if (c < 9) return e * Cfg::F1 + c;
  if (c == 9) return 8 * Cfg::F1 + e;
  if (c == 10) return e == 0 ? 8 * Cfg::F1 + 8 : -1;
  return -1;
}

#ifdef PL_TRACE
using fused_pl::pl_trace;
#endif
using fused_pl::BatchExt;
using tc::mbar_arrive;
using tc::named_bar_sync;

#ifdef HP_PROF
// kernel-development aid: per-warp cycles spent blocked at each hand-off of CTA (1,1,0), read
// back with srcnn_debug_hp_prof (tools/hp_prof.py); no printf, no per-tile stores
__device__ unsigned hp_prof[32][4];
#define HPW(i, ...) { const unsigned _t = (unsigned)clock(); __VA_ARGS__; _hw[i] += (unsigned)clock() - _t; }
#else
#define HPW(i, ...) { __VA_ARGS__; }
#endif

// ---------------------------------------------------------------------------- prepare --------
// Derives the scales from the parameters (every CTA of a small grid, redundantly) and packs the
// operand image.  The domain check of the INPUT is done by
// the plane producers of the main kernel, which see every pixel anyway: the first |x| >= 64 (or
// NaN) clears `ok`, and the TF32 kernel launched behind redoes the launch.
constexpr float kInMax = 64.f;
// `in_max` (may be null): bit pattern of the largest |input| of the launch, measured on the
// device -- the input scale then follows the data (no domain restriction, no fallback); used by
// the layer-1-only launches, where a.pw2 / a.pw3 are null.
__global__ void __launch_bounds__(256) hp_prepare_kernel(fused::Args a, Scales* sc,
                                                         const unsigned* in_max = nullptr) {
  using namespace tc;
  // the parameters are staged in shared memory with coalesced loads first: the column sums
  // below would otherwise be chains of dependent global loads (13 us instead of ~3)
  __shared__ float sw1[Cfg::F1 * Cfg::F1 * Cfg::N1];   // |W1| [tap][n]
  __shared__ float sw2[Cfg::N1 * Cfg::N2];             // |W2| [k][n]
  __shared__ float red_f[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  auto block_max = [&](float v) -> float {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) red_f[warp] = v;
    __syncthreads();
    float r = red_f[0];
    for (int w = 1; w < 8; w++) r = fmaxf(r, red_f[w]);
    return r;
  };
  float v1 = 0.f, v2 = 0.f, v3 = 0.f;
  for (int i = tid; i < Cfg::F1 * Cfg::F1 * Cfg::N1; i += 256) {
    const float w = fabsf(__ldg(a.pw1 + i));
    sw1[i] = w;
    v1 = fmaxf(v1, w);
  }
  const bool l1only = a.pw2 == nullptr;
  for (int i = tid; i < Cfg::N1 * Cfg::N2; i += 256) {
    const float w = l1only ? 0.f : fabsf(__ldg(a.pw2 + i));
    sw2[i] = w;
    v2 = fmaxf(v2, w);
  }
  if (!l1only)
    for (int i = tid; i < Cfg::QP * Cfg::N2; i += 256) v3 = fmaxf(v3, fabsf(__ldg(a.pw3 + i)));
  const float b1v = tid < Cfg::N1 ? fabsf(__ldg(a.pb1 + tid)) : 0.f;
  const float b2v = (tid < Cfg::N2 && !l1only) ? fabsf(__ldg(a.pb2 + tid)) : 0.f;
  // input range: 64 (fixed: a row-band partition then reproduces the single launch bit for
  // bit), or the power of two above the measured maximum
  float in_lim = kInMax;
  if (in_max) {
    const float mx = __uint_as_float(__ldg(in_max));
    if (mx > 0.f && mx < 1e30f) {
      int e;
      frexpf(mx, &e);
      in_lim = ldexpf(1.f, e);      // > mx
    }
  }
  const float m1 = block_max(v1);
  const float m2 = block_max(v2);
  const float m3 = block_max(v3);
  // bound on |out1[n]| and, from it, on |out2[n]|
  float v = 0.f;
  if (tid < Cfg::N1) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int t = 0; t < Cfg::F1 * Cfg::F1; t += 3) {
      s0 += sw1[t * Cfg::N1 + tid];
      s1 += sw1[(t + 1) * Cfg::N1 + tid];
      s2 += sw1[(t + 2) * Cfg::N1 + tid];
    }
    v = (s0 + s1 + s2) * in_lim + b1v;
  }
  const float bound1 = block_max(v);
  v = 0.f;
  if (tid < Cfg::N2) {
    float s0 = 0.f, s1 = 0.f;
    for (int k = 0; k < Cfg::N1; k += 2) {
      s0 += sw2[k * Cfg::N2 + tid];
      s1 += sw2[(k + 1) * Cfg::N2 + tid];
    }
    v = (s0 + s1) * bound1 + b2v;
  }
  const float bound2 = block_max(v);
  __shared__ ScaleVals sv;
  if (tid == 0) {
    ScaleVals s;
    s.sx = 32768.f / in_lim;   // in_lim * sx = 2^15 (512 for the fixed range of 64)
    s.in_lim = in_lim;
    s.sw1 = pow2_scale(m1);
    s.sw2 = pow2_scale(m2);
    s.sw3 = pow2_scale(m3);
    s.s1 = pow2_scale(bound1);
    s.s2 = pow2_scale(bound2);
    s.c1s = s.s1 / (s.sx * s.sw1);
    s.c2s = s.s2 / (s.s1 * s.sw2);
    s.c3 = 1.f / (s.s2 * s.sw3);
    s.inv_s1 = 1.f / s.s1;
    s.inv_s2 = 1.f / s.s2;
    // non-finite parameters: leave the launch to the TF32 kernel
    s.ok = (bound2 < 1e30f && m3 < 1e30f) ? 1 : 0;
    sv = s;
    if (blockIdx.x == 0) sc->v = s;
  }
  __syncthreads();
  // ---- the shared-memory image of the B operands: every CTA of the grid packs its share ----
  using C = Cfg;
  __half* gW1 = reinterpret_cast<__half*>(sc->wimg);
  __half* gW2 = reinterpret_cast<__half*>(sc->wimg + (C::oW2 - C::oW1));
  __half* gW3 = reinterpret_cast<__half*>(sc->wimg + (C::oW3 - C::oW1));
  float* gB1 = reinterpret_cast<float*>(sc->wimg + (C::oB1 - C::oW1));
  float* gB2 = reinterpret_cast<float*>(sc->wimg + (C::oB2 - C::oW1));
  const int gtid = blockIdx.x * 256 + tid, gn = gridDim.x * 256;
  for (int i = gtid; i < 2 * C::N1 * C::K1; i += gn) {
    const int n = i / C::K1, k = i % C::K1;
    const int t = tap16(k >> 4, (k >> 3) & 1, k & 7);
    unsigned short hi, lo;
    split_h(t >= 0 ? __ldg(a.pw1 + t * C::N1 + (n & (C::N1 - 1))) * sv.sw1 : 0.f, hi, lo);
    gW1[kmajor16(n, k, C::K1)] = __ushort_as_half(n < C::N1 ? hi : lo);
  }
  if (l1only) {
    for (int i = gtid; i < C::N1; i += gn) gB1[i] = __ldg(a.pb1 + i) * sv.s1;
    return;
  }
  for (int i = gtid; i < 2 * C::N2 * C::K2; i += gn) {
    const int n = i / C::K2, k = i % C::K2;
    unsigned short hi, lo;
    split_h(__ldg(a.pw2 + k * C::N2 + (n & (C::N2 - 1))) * sv.sw2, hi, lo);
    gW2[kmajor16(n, k, C::K2)] = __ushort_as_half(n < C::N2 ? hi : lo);
  }
  for (int i = gtid; i < 2 * C::NT3 * C::K3; i += gn) {
    const int n = i / C::K3, k = i % C::K3;   // n & 31 = tap dy*5+dx, k = channel
    const int tap = n & (C::NT3 - 1);
    unsigned short hi, lo;
    split_h(tap < C::QP ? __ldg(a.pw3 + tap * C::N2 + k) * sv.sw3 : 0.f, hi, lo);
    gW3[kmajor16(n, k, C::K3)] = __ushort_as_half(n < C::NT3 ? hi : lo);
  }
  for (int i = gtid; i < C::N1; i += gn) gB1[i] = __ldg(a.pb1 + i) * sv.s1;
  for (int i = gtid; i < C::N2; i += gn) gB2[i] = __ldg(a.pb2 + i) * sv.s2;
}

// ---------------------------------------------------------------------------- main kernel ----
// L1ONLY (with BATCH): only layer 1 runs and out1 is its result -- the forward of the first
// layer of a 9-5-5 training chunk (a.w3 / a.h3 / rpc are those of the 9-1-5 geometry: one tile
// per out1 row).  The layer-2/3 roles idle; E1 releases D1 itself (bar2) and records max |out1|.
template <bool BATCH, bool L1ONLY = false>
__global__ void __launch_bounds__(Cfg::NT, 1) forward_fused_hp_kernel(fused::Args a, int rpc,
                                                                      BatchExt bx,
                                                                      const Scales* scales,
                                                                      int* fallback) {
  using C = Cfg;
  using namespace tc;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const ScaleVals sc = scales->v;
  if (!sc.ok) {         // non-finite parameters: the TF32 kernel behind us runs instead
    if (threadIdx.x == 0) *fallback = 1;
    return;
  }
  __half* sW1 = reinterpret_cast<__half*>(smem_raw + C::oW1);
  __half* sW2 = reinterpret_cast<__half*>(smem_raw + C::oW2);
  __half* sW3 = reinterpret_cast<__half*>(smem_raw + C::oW3);
  float* sB1 = reinterpret_cast<float*>(smem_raw + C::oB1);
  float* sB2 = reinterpret_cast<float*>(smem_raw + C::oB2);
  float* sQs = reinterpret_cast<float*>(smem_raw + C::oQs);
  __shared__ __align__(8) uint64_t p_full[4], p_free[4], bar1[2], a2_full[2], bar2[2], d1_free[2],
      a3_full[2], bar3[2], d3_free[2];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int X0 = blockIdx.x * C::OW3;
  // out1 / out2 kept (BATCH): a strip stores the columns of its OW3 output columns; the last one
  // also stores the halo columns to their right, which no strip after it covers
  const bool last_strip = X0 + C::OW3 >= a.w3;
  const int R0 = blockIdx.y * rpc;
  const float* img = BATCH ? a.in : a.in + (size_t)blockIdx.z * a.w * a.h;
  float* dst = BATCH ? a.out : a.out + (size_t)blockIdx.z * a.w3 * a.h3;

  // ---- B operands and scaled biases: the image hp_prepare_kernel packed ---------------------
  {
    const uint4* src = reinterpret_cast<const uint4*>(scales->wimg);
    uint4* dstw = reinterpret_cast<uint4*>(smem_raw + C::oW1);
    for (int i = tid; i < (C::oQs - C::oW1) / 16; i += C::NT) dstw[i] = __ldg(src + i);
  }
  // pad entries of the planes are read by the tensor core (times a zero weight): keep them finite
  for (int i = tid; i < 2 * (C::RO + C::RH) * C::PB / 4; i += C::NT)
    reinterpret_cast<uint32_t*>(smem_raw)[i] = 0u;
  const float b3 = L1ONLY ? 0.f : __ldg(a.pb3);

  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    if (smem_u32(smem_raw) & 127u) __trap();
    for (int i = 0; i < 4; i++) {
      mbar_init(&p_full[i], C::IM_THREADS);
      mbar_init(&p_free[i], 1);
    }
    for (int i = 0; i < 2; i++) {
      mbar_init(&bar1[i], 1);
      mbar_init(&a2_full[i], C::N_E1 * 32);
      mbar_init(&bar2[i], (L1ONLY && !C::A2SEP) ? C::N_E1 * 32 : 1);
      mbar_init(&d1_free[i], C::N_E1 * 32);
      mbar_init(&a3_full[i], 128);
      mbar_init(&bar3[i], 1);
      mbar_init(&d3_free[i], 128);
    }
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;

  const int rows_here = min(rpc, a.h3 - R0);
  const int n_tiles = rows_here + (C::F3 - 1);   // out2 rows R0 .. R0+rows_here+3
#ifdef HP_PROF
  unsigned _hw[3] = {0u, 0u, 0u};
  const unsigned _hstart = (unsigned)clock();
#endif

  const bool is_im = warp >= C::W_IM && warp < C::W_IM + C::N_IM;
  const bool is_e1 = warp >= C::W_E1 && warp < C::W_E1 + C::N_E1;
  const bool is_e2 = warp >= C::W_E2 && warp < C::W_E2 + 4;
  const bool is_e3 = warp >= C::W_E3 && warp < C::W_E3 + 4;
  if (is_im) {
    // ============================ IM: plane producers =====================================
    // thread c owns plane column c (image column X0+c): per input row r it writes
    // H8(r)[c] = in[r][c..c+7] and O(r-7)[c] = (in[r-7..r][c]); the 7 older rows of the column
    // live in registers as halves.
    const int c = tid - C::W_IM * 32;
    const bool active = c < C::PW;
    const int gx = X0 + c;
    uint8_t* pOh = smem_raw + C::oOh + c * 16;
    uint8_t* pOl = smem_raw + C::oOl + c * 16;
    uint8_t* pHh = smem_raw + C::oHh + c * 16;
    uint8_t* pHl = smem_raw + C::oHl + c * 16;
    long long boff[8];
    if (BATCH) {
#pragma unroll
      for (int e = 0; e < 8; e++) {
        const int vx = gx + e;
        const int smp = vx / bx.pw;
        boff[e] = (active && vx < a.w) ? (long long)smp * bx.pw * bx.ph + (vx - smp * bx.pw) : -1;
      }
    }
    auto ld = [&](int r, int e) -> float {
      const int gy = R0 + r;
      float v;
      if (BATCH)
        v = (boff[e] >= 0 && gy < a.h) ? __ldg(img + boff[e] + (long long)gy * bx.pw) : 0.f;
      else
        v = (active && gy < a.h && gx + e < a.w) ? __ldg(img + (size_t)gy * a.w + gx + e) : 0.f;
      return v;
    };
    // the domain check happens where a value is consumed, never where it is loaded: the loads
    // of the next two rows stay in flight across a tile (HBM latency > one tile period)
    const float in_lim = sc.in_lim * 0.999f;
    auto in_domain = [&](float x) {
      if (!(fabsf(x) < in_lim)) *fallback = 1;   // outside the FP16 domain (or NaN)
    };
    unsigned short hh[7], hl[7];   // rows r-7 .. r-1 of this column
    {
      float pv[C::F1 - 1];
#pragma unroll
      for (int r = 0; r < C::F1 - 1; r++) pv[r] = ld(r, 0);
      unsigned short h7, l7;
#pragma unroll
      for (int r = 0; r < C::F1 - 2; r++) {
        in_domain(pv[r]);
        split_h(pv[r] * sc.sx, hh[r], hl[r]);
      }
      in_domain(pv[C::F1 - 2]);
      split_h(pv[C::F1 - 2] * sc.sx, h7, l7);
      if (active) {   // O(0) = rows 0..7
        *reinterpret_cast<uint4*>(pOh) = make_uint4(pack2(hh[0], hh[1]), pack2(hh[2], hh[3]),
                                                    pack2(hh[4], hh[5]), pack2(hh[6], h7));
        *reinterpret_cast<uint4*>(pOl) = make_uint4(pack2(hl[0], hl[1]), pack2(hl[2], hl[3]),
                                                    pack2(hl[4], hl[5]), pack2(hl[6], l7));
      }
#pragma unroll
      for (int r = 0; r < 6; r++) { hh[r] = hh[r + 1]; hl[r] = hl[r + 1]; }
      hh[6] = h7; hl[6] = l7;
    }
    float v[8], nv[8];
#pragma unroll
    for (int e = 0; e < 8; e++) v[e] = ld(C::F1 - 1, e);
#pragma unroll
    for (int e = 0; e < 8; e++) nv[e] = n_tiles > 1 ? ld(C::F1, e) : 0.f;
    for (int b = 0; b < n_tiles; b++) {
      float nnv[8];
#pragma unroll
      for (int e = 0; e < 8; e++) nnv[e] = (b + 2 < n_tiles) ? ld(b + C::F1 + 1, e) : 0.f;
      uint32_t ph[4], pl[4];
#pragma unroll
      for (int e = 0; e < 8; e++) in_domain(v[e]);
#pragma unroll
      for (int e = 0; e < 4; e++)
        split_h2(v[2 * e] * sc.sx, v[2 * e + 1] * sc.sx, ph[e], pl[e]);
      const unsigned short nh = (unsigned short)(ph[0] & 0xffffu), nl = (unsigned short)(pl[0] & 0xffffu);
      // H8(b+8) replaces H8(b+4) (MMA-1(b-4)), O(b+1) replaces O(b-3) (MMA-1(b-3))
      if (b >= 3) HPW(0, mbar_wait(&p_free[(b - 3) & 3], (uint32_t)(((b - 3) >> 2) & 1)))
      if (active) {
        const int sh = b & (C::RH - 1), so = (b + 1) & (C::RO - 1);
        *reinterpret_cast<uint4*>(pHh + sh * C::PB) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
        *reinterpret_cast<uint4*>(pHl + sh * C::PB) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
        *reinterpret_cast<uint4*>(pOh + so * C::PB) = make_uint4(
            pack2(hh[0], hh[1]), pack2(hh[2], hh[3]), pack2(hh[4], hh[5]), pack2(hh[6], nh));
        *reinterpret_cast<uint4*>(pOl + so * C::PB) = make_uint4(
            pack2(hl[0], hl[1]), pack2(hl[2], hl[3]), pack2(hl[4], hl[5]), pack2(hl[6], nl));
      }
#pragma unroll
      for (int r = 0; r < 6; r++) { hh[r] = hh[r + 1]; hl[r] = hl[r + 1]; }
      hh[6] = nh; hl[6] = nl;
      fence_proxy_async();
      mbar_arrive(&p_full[b & 3]);
      if (warp == C::W_IM) PL_EV(b, 12)
#pragma unroll
      for (int e = 0; e < 8; e++) { v[e] = nv[e]; nv[e] = nnv[e]; }
    }
  } else if (warp == C::W_I1) {
    // ============================ I1: layer-1 MMA issuer ===================================
    const uint32_t idesc_hi = make_idesc_f16(C::M, 2 * C::N1);   // A_hi x [W_hi; W_lo]
    const uint32_t idesc_lo = make_idesc_f16(C::M, C::N1);       // A_lo x W_hi
    const uint64_t wdesc = make_desc_kmajor(sW1, 0, 128, 128 * (C::K1 / 8));
    const uint32_t aOh = smem_u32(smem_raw + C::oOh), aOl = smem_u32(smem_raw + C::oOl);
    const uint32_t aHh = smem_u32(smem_raw + C::oHh), aHl = smem_u32(smem_raw + C::oHl);
    auto adesc = [](uint32_t addr, uint32_t lbo) -> uint64_t {
      return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
             ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    };
    for (int t = 0; t < n_tiles; t++) {
      HPW(0, mbar_wait(&p_full[t & 3], (uint32_t)((t >> 2) & 1)))
      // D1[t&1] still holds A2(t-2) until MMA-2(t-2) has read it
      if (t >= 2) HPW(1, mbar_wait(C::A2SEP ? &d1_free[t & 1] : &bar2[t & 1], (uint32_t)(((t - 2) >> 1) & 1)))
      tcgen05_fence_after();
      const uint32_t d1 = tmem + C::cD1 + 128u * (uint32_t)(t & 1);
      const uint32_t so = (uint32_t)(t & (C::RO - 1)) * C::PB;
      const uint32_t sh = (uint32_t)(t & (C::RH - 1)) * C::PB;
      PL_EV(t, 0)
#ifdef HP_PROF
      const unsigned _tb = (unsigned)clock();
#endif
      if (elect_one()) {
#pragma unroll
        for (int s = 0; s < C::KS1; s++) {
          uint32_t ah, al, lbo_h, lbo_l;
          if (s < 4) { ah = aOh + so + 32 * s; al = aOl + so + 32 * s; lbo_h = lbo_l = 16; }
          else if (s == 4) {
            ah = aOh + so + 128; al = aOl + so + 128;
            lbo_h = (aHh + sh) - ah; lbo_l = (aHl + sh) - al;
          }
          else { ah = aHh + sh + 128; al = aHl + sh + 128; lbo_h = lbo_l = 16; }
          mma_f16_ss(d1, adesc(ah, lbo_h), wdesc + 16 * s, idesc_hi, s > 0);
          mma_f16_ss(d1 + C::N1, adesc(al, lbo_l), wdesc + 16 * s, idesc_lo, 1);
        }
        mma_commit(&bar1[t & 1]);
        mma_commit(&p_free[t & 3]);
      }
      __syncwarp();
#ifdef HP_PROF
      _hw[2] += (unsigned)clock() - _tb;
#endif
      PL_EV(t, 1)
    }
  } else if (L1ONLY && !is_e1) {
    // layer-1-only launch: the layer-2 / layer-3 roles have nothing to do
  } else if (warp == C::W_I2) {
    // ============================ I2: layer-2 MMA issuer (A2 in TMEM) ======================
    const uint32_t idesc_hi = make_idesc_f16(C::M, 2 * C::N2);
    const uint32_t idesc_lo = make_idesc_f16(C::M, C::N2);
    const uint64_t wdesc = make_desc_kmajor(sW2, 0, 128, 128 * (C::K2 / 8));
    for (int t = 0; t < n_tiles; t++) {
      HPW(0, mbar_wait(&a2_full[t & 1], (uint32_t)((t >> 1) & 1)))
      // D2[t&1] still holds A3(t-2) until MMA-3(t-2) has read it
      if (t >= 2) HPW(1, mbar_wait(&bar3[t & 1], (uint32_t)(((t - 2) >> 1) & 1)))
      tcgen05_fence_after();
      const uint32_t a2 = tmem + C::cA2 + C::sA2 * (uint32_t)(t & 1);
      const uint32_t d2 = tmem + C::cD2x + C::sD2 * (uint32_t)(t & 1);
      PL_EV(t, 4)
#ifdef HP_PROF
      const unsigned _tb = (unsigned)clock();
#endif
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::K2 / 16; ks++) {
          const uint32_t col = C::a2col((uint32_t)ks);
          if (C::ACC1_23) {
            // rows 32.. of sW2 (the low halves) start 4 row groups = 4 * 128 * K2/8 bytes in
            constexpr uint64_t kLo = (4 * 128 * (C::K2 / 8)) >> 4;
            mma_f16_ts(d2, a2 + col, wdesc + 16 * ks, idesc_lo, ks > 0);
            mma_f16_ts(d2, a2 + col, wdesc + kLo + 16 * ks, idesc_lo, 1);
            mma_f16_ts(d2, a2 + C::A2LO + col, wdesc + 16 * ks, idesc_lo, 1);
          } else {
            mma_f16_ts(d2, a2 + col, wdesc + 16 * ks, idesc_hi, ks > 0);
            mma_f16_ts(d2 + C::N2, a2 + C::A2LO + col, wdesc + 16 * ks, idesc_lo, 1);
          }
        }
        mma_commit(&bar2[t & 1]);
      }
      __syncwarp();
#ifdef HP_PROF
      _hw[2] += (unsigned)clock() - _tb;
#endif
      PL_EV(t, 5)
    }
  } else if (warp == C::W_I3) {
    // ============================ I3: layer-3 tap-GEMM issuer (A3 in TMEM) =================
    const uint32_t idesc_hi = make_idesc_f16(C::M, 2 * C::NT3);
    const uint32_t idesc_lo = make_idesc_f16(C::M, C::NT3);
    const uint64_t wdesc = make_desc_kmajor(sW3, 0, 128, 128 * (C::K3 / 8));
    for (int t = 0; t < n_tiles; t++) {
      HPW(0, mbar_wait(&a3_full[t & 1], (uint32_t)((t >> 1) & 1)))
      if (t >= 2) HPW(1, mbar_wait(&d3_free[t & 1], (uint32_t)(((t - 2) >> 1) & 1)))
      tcgen05_fence_after();
      const uint32_t a3 = tmem + C::cD2x + C::sD2 * (uint32_t)(t & 1);
      const uint32_t d3 = tmem + C::cD3x + C::sD3 * (uint32_t)(t & 1);
      PL_EV(t, 8)
#ifdef HP_PROF
      const unsigned _tb = (unsigned)clock();
#endif
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::K3 / 16; ks++) {
          if (C::ACC1_23) {
            constexpr uint64_t kLo = (4 * 128 * (C::K3 / 8)) >> 4;   // rows 32.. of sW3
            mma_f16_ts(d3, a3 + ks * 8, wdesc + 16 * ks, idesc_lo, ks > 0);
            mma_f16_ts(d3, a3 + ks * 8, wdesc + kLo + 16 * ks, idesc_lo, 1);
            mma_f16_ts(d3, a3 + C::A3LO + ks * 8, wdesc + 16 * ks, idesc_lo, 1);
          } else {
            mma_f16_ts(d3, a3 + ks * 8, wdesc + 16 * ks, idesc_hi, ks > 0);
            mma_f16_ts(d3 + C::NT3, a3 + C::N2 + ks * 8, wdesc + 16 * ks, idesc_lo, 1);
          }
        }
        mma_commit(&bar3[t & 1]);
      }
      __syncwarp();
#ifdef HP_PROF
      _hw[2] += (unsigned)clock() - _tb;
#endif
      PL_EV(t, 9)
    }
  } else if (is_e1) {
    // ============================ E1: A2 = split(relu(out1) * s1), in place ================
    // warp w: TMEM lane quarter w&3, chunks g0 .. g0+E1_CHUNKS-1 of 16 channels.  Chunk g reads
    // D1 columns [16g,16g+16) and [64+16g, ..), then writes its hi pairs to a2col(g) and its lo
    // pairs to 64 + a2col(g): columns this warp has consumed
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int g0 = ((warp - C::W_E1) >> 2) * C::E1_CHUNKS;
    // out1 (training): pixel index of this lane's pixel in tile 0, -1 = not an out1 pixel
    int pix1 = -1;
    const bool keep1 = BATCH && bx.out1 != nullptr;
    if (keep1) {
      const int m = (warp & 3) * 32 + lane, vx = X0 + m, smp = vx / bx.pw, px = vx - smp * bx.pw;
      const int w1 = bx.pw - (C::F1 - 1), h1 = bx.ph - (C::F1 - 1);
      if ((m < C::OW3 || last_strip) && vx < a.w && px < w1) pix1 = (smp * h1 + R0) * w1 + px;
    }
    const int w1_row = bx.pw - (C::F1 - 1);
    float* st1 = reinterpret_cast<float*>(smem_raw + C::oS1) + (warp - C::W_E1) * (32 * C::SP);
    float act_max = 0.f;   // L1ONLY: largest scaled activation this thread stored
    for (int b = 0; b < n_tiles; b++) {
      HPW(0, mbar_wait(&bar1[b & 1], (uint32_t)((b >> 1) & 1)))       // MMA-1(b) done
      if (warp == C::W_E1) PL_EV(b, 2)
      tcgen05_fence_after();
      const uint32_t d1 = tmem + lane_base + C::cD1 + 128u * (uint32_t)(b & 1);
      // all loads of this warp's chunks first (one TMEM round trip), then the conversions
      float va[C::E1_CHUNKS][16], vb[C::E1_CHUNKS][16];
#ifdef HP_PROF
      const unsigned _tl = (unsigned)clock();
#endif
#pragma unroll
      for (int gl = 0; gl < C::E1_CHUNKS; gl++) {
        tmem_ld16_nowait(d1 + (g0 + gl) * 16, va[gl]);
        tmem_ld16_nowait(d1 + C::N1 + (g0 + gl) * 16, vb[gl]);
      }
      tmem_ld_wait();
#ifdef HP_PROF
      _hw[1] += (unsigned)clock() - _tl;
#endif
      if (L1ONLY || C::A2SEP) {     // D1[b&1] may be overwritten by MMA-1(b+2)
        tcgen05_fence_before();
        mbar_arrive(C::A2SEP ? &d1_free[b & 1] : &bar2[b & 1]);
      }
      if (C::A2SEP && !L1ONLY && b >= 2) {   // A2[b&1] is still being read until MMA-2(b-2) is done
        mbar_wait(&bar2[b & 1], (uint32_t)(((b - 2) >> 1) & 1));
        tcgen05_fence_after();
      }
      const uint32_t a2w = tmem + lane_base + C::cA2 + C::sA2 * (uint32_t)(b & 1);
#pragma unroll
      for (int gl = 0; gl < C::E1_CHUNKS; gl++) {
        const int g = g0 + gl;
        uint32_t hi[8], lo[8];
        float act[16];
#pragma unroll
        for (int j = 0; j < 16; j++)
          act[j] = fmaxf(fmaf(va[gl][j] + vb[gl][j], sc.c1s, sB1[g * 16 + j]), 0.f);
        if (L1ONLY) {
          if (pix1 >= 0) {
#pragma unroll
            for (int j = 0; j < 16; j++) act_max = fmaxf(act_max, act[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; j++) split_h2(act[2 * j], act[2 * j + 1], hi[j], lo[j]);
          const uint32_t col = C::a2col((uint32_t)g);
          tmem_st8u(a2w + col, hi);
          tmem_st8u(a2w + C::A2LO + col, lo);
        }
        if (keep1) {
          float4* q = reinterpret_cast<float4*>(st1 + lane * C::SP + gl * 16);
#pragma unroll
          for (int j = 0; j < 4; j++)
            q[j] = make_float4(act[4 * j] * sc.inv_s1, act[4 * j + 1] * sc.inv_s1,
                               act[4 * j + 2] * sc.inv_s1, act[4 * j + 3] * sc.inv_s1);
        }
      }
      if (!L1ONLY) {
#ifdef HP_PROF
        const unsigned _ts = (unsigned)clock();
#endif
        tmem_st_wait();
#ifdef HP_PROF
        _hw[2] += (unsigned)clock() - _ts;
#endif
        tcgen05_fence_before();
        mbar_arrive(&a2_full[b & 1]);
      }
      if (keep1) {
        // 8 lanes per pixel: every store instruction writes four full 128-byte lines (one
        // 64-byte run per thread touched 32 lines per instruction and bound the whole kernel)
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; it++) {
          const int pp = it * 4 + (lane >> 3), ck = lane & 7;
          const int pidx = __shfl_sync(0xffffffffu, pix1, pp);
          const float4 v = *reinterpret_cast<const float4*>(st1 + pp * C::SP + ck * 4);
          if (pidx >= 0)
            *reinterpret_cast<float4*>(bx.out1 + ((size_t)pidx + (size_t)b * w1_row) * C::N1 +
                                       g0 * 16 + ck * 4) = v;
        }
        __syncwarp();
      }
      if (warp == C::W_E1) PL_EV(b, 3)
    }
    if (L1ONLY && bx.out1_max) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) act_max = fmaxf(act_max, __shfl_xor_sync(0xffffffffu, act_max, o));
      if (lane == 0 && act_max > 0.f) atomicMax(bx.out1_max, __float_as_uint(act_max * sc.inv_s1));
    }
  } else if (is_e2) {
    // ============================ E2: A3 = split(relu(out2) * s2), in place ================
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    int pix2 = -1;
    const bool keep2 = BATCH && bx.out2 != nullptr;
    if (keep2) {
      const int m = (warp & 3) * 32 + lane, vx = X0 + m, smp = vx / bx.pw, px = vx - smp * bx.pw;
      const int w2 = bx.pw - (C::F1 - 1), h2 = bx.ph - (C::F1 - 1);
      if ((m < C::OW3 || last_strip) && vx < a.w && px < w2) pix2 = (smp * h2 + R0) * w2 + px;
    }
    const int w2_row = bx.pw - (C::F1 - 1);
    float* st2 = reinterpret_cast<float*>(smem_raw + C::oS2) + (warp - C::W_E2) * (32 * C::SP);
    float act2_max = 0.f;   // largest scaled out2 value this thread stored
    for (int b = 0; b < n_tiles; b++) {
      HPW(0, mbar_wait(&bar2[b & 1], (uint32_t)((b >> 1) & 1)))       // MMA-2(b) done
      if (warp == C::W_E2) PL_EV(b, 6)
      tcgen05_fence_after();
      const uint32_t d2 = tmem + lane_base + C::cD2x + C::sD2 * (uint32_t)(b & 1);
      // all loads first (one TMEM round trip), then the conversions
      float va[2][16], vb[C::ACC1_23 ? 1 : 2][16];
#pragma unroll
      for (int g = 0; g < 2; g++) {
        tmem_ld16_nowait(d2 + g * 16, va[g]);
        if (!C::ACC1_23) tmem_ld16_nowait(d2 + C::N2 + g * 16, vb[C::ACC1_23 ? 0 : g]);
      }
      tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 2; g++) {
        uint32_t hi[8], lo[8];
        float act[16];
#pragma unroll
        for (int j = 0; j < 16; j++)
          act[j] = fmaxf(fmaf(C::ACC1_23 ? va[g][j] : va[g][j] + vb[C::ACC1_23 ? 0 : g][j], sc.c2s,
                              sB2[g * 16 + j]), 0.f);
#pragma unroll
        for (int j = 0; j < 8; j++) split_h2(act[2 * j], act[2 * j + 1], hi[j], lo[j]);
        tmem_st8u(d2 + g * 8, hi);
        tmem_st8u(d2 + C::A3LO + g * 8, lo);
        if (keep2) {
          if (pix2 >= 0) {
#pragma unroll
            for (int j = 0; j < 16; j++) act2_max = fmaxf(act2_max, act[j]);
          }
          float4* q = reinterpret_cast<float4*>(st2 + lane * C::SP + g * 16);
#pragma unroll
          for (int j = 0; j < 4; j++)
            q[j] = make_float4(act[4 * j] * sc.inv_s2, act[4 * j + 1] * sc.inv_s2,
                               act[4 * j + 2] * sc.inv_s2, act[4 * j + 3] * sc.inv_s2);
        }
      }
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive(&a3_full[b & 1]);
      if (keep2) {
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; it++) {
          const int pp = it * 4 + (lane >> 3), ck = lane & 7;
          const int pidx = __shfl_sync(0xffffffffu, pix2, pp);
          const float4 v = *reinterpret_cast<const float4*>(st2 + pp * C::SP + ck * 4);
          if (pidx >= 0)
            *reinterpret_cast<float4*>(bx.out2 + ((size_t)pidx + (size_t)b * w2_row) * C::N2 +
                                       ck * 4) = v;
        }
        __syncwarp();
      }
      if (warp == C::W_E2) PL_EV(b, 7)
    }
    if (keep2 && bx.out2_max) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) act2_max = fmaxf(act2_max, __shfl_xor_sync(0xffffffffu, act2_max, o));
      if (lane == 0 && act2_max > 0.f) atomicMax(bx.out2_max, __float_as_uint(act2_max * sc.inv_s2));
    }
  } else if (is_e3) {
    // ============================ E3: Q row -> smem, 25-term gather -> out3 ================
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int x = (warp & 3) * 32 + lane;
    bool live = x < C::OW3 && X0 + x < a.w3;
    size_t o3 = (size_t)R0 * a.w3 + X0 + x;   // output row 0 of this thread's column
    size_t o3_row = (size_t)a.w3;
    if (BATCH) {
      const int vx = X0 + x, smp = vx / bx.pw, px = vx - smp * bx.pw;
      const int w3 = bx.pw - (C::F1 + C::F3 - 2), h3 = bx.ph - (C::F1 + C::F3 - 2);
      live = live && px < w3;
      o3 = ((size_t)smp * h3 + R0) * w3 + px;
      o3_row = (size_t)w3;
    }
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
    for (int b = 0; b < n_tiles; b++) {
      HPW(0, mbar_wait(&bar3[b & 1], (uint32_t)((b >> 1) & 1)))       // MMA-3(b) done
      if (warp == C::W_E3) PL_EV(b, 10)
      tcgen05_fence_after();
      const uint32_t d3 = tmem + lane_base + C::cD3x + C::sD3 * (uint32_t)(b & 1);
      float v[32], w[C::ACC1_23 ? 1 : 32];
#ifdef HP_PROF
      const unsigned _tl3 = (unsigned)clock();
#endif
      tmem_ld16_nowait(d3, v);
      tmem_ld16_nowait(d3 + 16, v + 16);
      if (!C::ACC1_23) {
        tmem_ld16_nowait(d3 + 32, w);
        tmem_ld16_nowait(d3 + 48, w + (C::ACC1_23 ? 0 : 16));
      }
      tmem_ld_wait();
#ifdef HP_PROF
      _hw[2] += (unsigned)clock() - _tl3;
#endif
      tcgen05_fence_before();
      mbar_arrive(&d3_free[b & 1]);                            // D3[b&1] may be overwritten
      float* qs = sQs + (b & 1) * (C::M * C::QP);
#pragma unroll
      for (int j = 0; j < C::QP; j++) qs[x * C::QP + j] = C::ACC1_23 ? v[j] : v[j] + w[C::ACC1_23 ? 0 : j];
      HPW(1, named_bar_sync(C::BAR_E3, 128))                          // Q row visible to its neighbours
      float r[C::F3];
      if (x < C::OW3) {
#pragma unroll
        for (int dy = 0; dy < C::F3; dy++) {
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int dx = 0; dx < C::F3; dx++) {
            const float q = qs[(x + dx) * C::QP + dy * C::F3 + dx];
            if (dx & 1) s1 += q; else s0 += q;
          }
          r[dy] = s0 + s1;
        }
      } else {
#pragma unroll
        for (int dy = 0; dy < C::F3; dy++) r[dy] = 0.f;
      }
      const float done = acc0 + r[4];
      acc0 = acc1 + r[3];
      acc1 = acc2 + r[2];
      acc2 = acc3 + r[1];
      acc3 = r[0];
      if (b >= C::F3 - 1 && live)   // the scale of the tap GEMM is applied once, to the sum
        dst[o3 + (size_t)(b - (C::F3 - 1)) * o3_row] = fmaf(done, sc.c3, b3);
      if (warp == C::W_E3) PL_EV(b, 11)
    }
  }

#ifdef HP_PROF
  if (blockIdx.x == 1 && blockIdx.y == 1 && blockIdx.z == 0 && lane == 0) {
    hp_prof[warp][0] = (unsigned)clock() - _hstart;
    hp_prof[warp][1] = _hw[0];
    hp_prof[warp][2] = _hw[1];
    hp_prof[warp][3] = _hw[2];
  }
#endif
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
#ifdef PL_TRACE
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && tid == 0 && n_tiles >= PL_TRACE_BASE + 8) {
    const long long t0 = pl_trace[0][12];
    for (int t = 0; t < 8; t++)
      printf("tile %d: IM %6lld | I1 %6lld..%6lld | E1 %6lld..%6lld | I2 %6lld..%6lld | E2 %6lld..%6lld | I3 %6lld..%6lld | E3 %6lld..%6lld\n",
             PL_TRACE_BASE + t, pl_trace[t][12] - t0, pl_trace[t][0] - t0, pl_trace[t][1] - t0, pl_trace[t][2] - t0,
             pl_trace[t][3] - t0, pl_trace[t][4] - t0, pl_trace[t][5] - t0, pl_trace[t][6] - t0,
             pl_trace[t][7] - t0, pl_trace[t][8] - t0, pl_trace[t][9] - t0, pl_trace[t][10] - t0,
             pl_trace[t][11] - t0);
  }
#endif
}

inline int configure() {
  SRCNN_CUDA(cudaFuncSetAttribute(forward_fused_hp_kernel<false>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Cfg::SMEM_BYTES));
  SRCNN_CUDA(cudaFuncSetAttribute(forward_fused_hp_kernel<true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Cfg::SMEM_BYTES_KEEP));
  SRCNN_CUDA(cudaFuncSetAttribute(forward_fused_hp_kernel<true, true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Cfg::SMEM_BYTES_KEEP));
  return SRCNN_OK;
}

inline bool supported(int n1, int n2, int f1, int f2, int f3) {
  return n1 == 64 && n2 == 32 && f1 == 9 && f2 == 1 && f3 == 5;
}

// the per-context ring of scale blocks: launches on different streams (the pipelined
// host-buffer inference) must not share one
inline int scale_slot(srcnn_ctx* ctx, Scales** sc, unsigned** ws) {
  constexpr int kSlots = 128;   // three captured pipelines of 16-32 launches keep theirs
  if (!ctx->hp_scales) {
    SRCNN_CUDA(cudaMalloc(&ctx->hp_scales, kSlots * (sizeof(Scales) + 2 * sizeof(unsigned))));
    SRCNN_CUDA(cudaMemset(ctx->hp_scales, 0, kSlots * (sizeof(Scales) + 2 * sizeof(unsigned))));
  }
  const int i = (int)(ctx->hp_next++ % kSlots);
  *sc = reinterpret_cast<Scales*>(ctx->hp_scales) + i;
  *ws = reinterpret_cast<unsigned*>(reinterpret_cast<Scales*>(ctx->hp_scales) + kSlots) + 2 * i;
  return SRCNN_OK;
}

// the scales and operand image of a network, computed on the context stream into `block`
inline void prepare_into(srcnn_ctx* ctx, const fused::Args& a, void* block) {
  hp_prepare_kernel<<<8, 256, 0, ctx->stream>>>(a, reinterpret_cast<Scales*>(block));
}

// [prepare +] FP16 kernel + (gated) TF32 kernel; `S` images, or a batch as one virtual image.
// `shared` = scales already prepared for these parameters (the sub-bands of
// srcnn_infer_rows_host, or the context's cache); null = prepare here.  The scales are read-only
// for the kernels; "leave this launch to the TF32 kernel" is a per-launch word of the ring.
inline int launch(srcnn_ctx* ctx, const fused::Args& a, int S, bool batch, float* out1,
                  float* out2, const Scales* shared = nullptr, unsigned* out2_max = nullptr) {
  const Scales* sc = shared;
  Scales* slot;
  unsigned* ws;
  SRCNN_TRY(scale_slot(ctx, &slot, &ws));
  if (!sc) {
    hp_prepare_kernel<<<8, 256, 0, ctx->stream>>>(a, slot);
    sc = slot;
  }
  int* fallback = reinterpret_cast<int*>(ws);
  SRCNN_CUDA(cudaMemsetAsync(fallback, 0, sizeof(int), ctx->stream));
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  BatchExt bx{};
  bx.gate = fallback;
  if (batch) {
    fused::Args v = a;
    const int pad = Cfg::F1 + Cfg::F3 - 2;
    v.w = S * a.w;
    v.w3 = S * a.w - pad;
    const int rpc = fused_pl::rows_per_cta(v.w3, v.h3, 1, sms);
    dim3 grid((v.w3 + Cfg::OW3 - 1) / Cfg::OW3, (v.h3 + rpc - 1) / rpc, 1);
    bx.out1 = out1;
    bx.out2 = out2;
    bx.S = S;
    bx.pw = a.w;
    bx.ph = a.h;
    bx.out2_max = out2_max;
    if (out2_max) SRCNN_CUDA(cudaMemsetAsync(out2_max, 0, sizeof(unsigned), ctx->stream));
    forward_fused_hp_kernel<true>
        <<<grid, Cfg::NT, (out1 || out2) ? Cfg::SMEM_BYTES_KEEP : Cfg::SMEM_BYTES, ctx->stream>>>(
            v, rpc, bx, sc, fallback);
    fused_pl::forward_fused_pl_kernel<true>
        <<<grid, fused_pl::Cfg::NT, fused_pl::Cfg::SMEM_BYTES, ctx->stream>>>(v, rpc, bx);
  } else {
    const int rpc = fused_pl::rows_per_cta(a.w3, a.h3, S, sms);
    dim3 grid((a.w3 + Cfg::OW3 - 1) / Cfg::OW3, (a.h3 + rpc - 1) / rpc, S);
    forward_fused_hp_kernel<false>
        <<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(a, rpc, bx, sc, fallback);
    fused_pl::forward_fused_pl_kernel<false>
        <<<grid, fused_pl::Cfg::NT, fused_pl::Cfg::SMEM_BYTES, ctx->stream>>>(a, rpc, bx);
  }
  return SRCNN_OK;
}

// Layer 1 alone (9x9, 1 -> 64, ReLU) of a batch of S samples of pw x ph pixels, out1 kept: the
// first layer of a 9-5-5 training chunk.  `in_max` holds the measured max |input| (the operand
// scale follows it: no input-range restriction), `out1_max` receives max |out1| (zeroed here).
inline int launch_l1only(srcnn_ctx* ctx, const float* in, float* out1, const float* w1,
                         const float* b1, int pw, int ph, int S, const unsigned* in_max,
                         unsigned* out1_max) {
  Scales* slot;
  unsigned* ws;
  SRCNN_TRY(scale_slot(ctx, &slot, &ws));
  const int pad = Cfg::F1 + Cfg::F3 - 2;   // geometry of the 9-1-5 kernel: one tile per out1 row
  fused::Args v{in, nullptr, w1, b1, nullptr, nullptr, nullptr, nullptr, S * pw, ph, S * pw - pad, ph - pad};
  hp_prepare_kernel<<<8, 256, 0, ctx->stream>>>(v, slot, in_max);
  int* fallback = reinterpret_cast<int*>(ws);
  SRCNN_CUDA(cudaMemsetAsync(fallback, 0, sizeof(int), ctx->stream));
  SRCNN_CUDA(cudaMemsetAsync(out1_max, 0, sizeof(unsigned), ctx->stream));
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  BatchExt bx{};
  bx.out1 = out1;
  bx.S = S;
  bx.pw = pw;
  bx.ph = ph;
  bx.out1_max = out1_max;
  const int rpc = fused_pl::rows_per_cta(v.w3, v.h3, 1, sms);
  dim3 grid((v.w3 + Cfg::OW3 - 1) / Cfg::OW3, (v.h3 + rpc - 1) / rpc, 1);
  forward_fused_hp_kernel<true, true>
      <<<grid, Cfg::NT, Cfg::SMEM_BYTES_KEEP, ctx->stream>>>(v, rpc, bx, slot, fallback);
  return SRCNN_OK;
}

}  // namespace fused_hp
}  // namespace srcnn
