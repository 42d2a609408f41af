// Fused SRCNN inference, "plane" tensor-core version (9-1-5, n1=64, n2=32): all three layers
// of ConfigBasedDataPipeline::forward (src/ConfigBasedDataPipeline.cpp:200-241, three launches
// of src/kernel/layer_uber_kernel.cl:36-96) in one launch, as error-compensated TF32 tcgen05
// GEMMs on tiles of 128 pixels (one out2 row x 128 columns), accumulators and the layer-2/3 A
// operands in tensor memory.
//
// What is different from fused_forward_ws.cuh (measured, csrc/probe/plane_probe.cu):
//  * NO im2col.  Layer 1 has one input channel, so its im2col matrix is a Hankel matrix
//    A[x][(dy,dx)] = in[y+dy][x+dx].  A no-swizzle K-major shared-memory descriptor addresses
//    (row m, k) at base + (m/8)*SBO + (m%8)*16 + (k/4)*LBO + (k%4)*4; with SBO = 128 the rows
//    of a tile are consecutive 16-byte units, so a "plane" of vertically packed pixels
//        Qd(s)[c] = (in[s][c], in[s+1][c], in[s+2][c], in[s+3][c])
//    read at base = &Qd(s)[dx] IS the im2col block of taps (dy = s-y..s-y+3, dx) of 128 pixels.
//    Filter rows 0-3 and 4-7 come from Qd(y), Qd(y+4); row 8 from a plane of horizontally
//    packed pixels H(r)[c] = in[r][c..c+3].  Every input pixel is written 8 times (hi/lo x 4
//    quads... 2 planes) instead of 176 times, and the planes are shared by consecutive tiles.
//  * a tcgen05.mma costs its issuing thread ~57 cycles whatever its shape, and the tensor pipe
//    accepts instructions from several threads: each layer has its OWN issuer warp, and every
//    layer is issued as  A_hi x [W_hi; W_lo] (N doubled) + A_lo x W_hi: two instructions per
//    K-step instead of three (46 per tile instead of 69); the epilogue adds the two halves.
//  * the split A operand of the next layer is written in place over the accumulator it was
//    computed from, and every TMEM buffer exists twice, so no stage ever waits for the stage
//    behind it to release a buffer of the SAME tile parity before two tiles later.
//  * the operand split costs 3 instructions (tc_common.cuh) instead of 9.
//
//   role (warps)      per tile b (= out2 row R0+b of the strip)
//   IM   12..16       input row b+8 -> H(b+8), Qd(b+5) (hi/lo)                 -> p_full
//   I1   17           MMA-1(b): 11 K-steps x 2 -> D1[b&1]                      -> bar1, p_free
//   E1   0..3         D1 -> +b1, relu, split -> A2 (in place)                  -> a2_full
//   I2   18           MMA-2(b): 8 K-steps x 2 (A2 in TMEM) -> D2[b&1]          -> bar2
//   E2   4..7         D2 -> +b2, relu, split -> A3 (in place)                  -> a3_full
//   I3   19           MMA-3(b): tap GEMM Q[px][25] = out2[px][:] . W3[tap][:]  -> bar3
//   E3   8..11        D3 -> Q row in smem -> out3 row b-4 += 25-term gather    -> d3_free
#pragma once
#include <cuda_runtime.h>

#include "context.cuh"
#include "fused_forward.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace fused_pl {

struct Cfg {
  static constexpr int N1 = 64, N2 = 32, F1 = 9, F3 = 5;
  static constexpr int M = 128;                  // pixels (columns of one out2 row) per tile
  static constexpr int OW3 = M - (F3 - 1);       // 124 output columns per strip
  static constexpr int KS1 = 11, K1 = KS1 * 8;   // layer-1 K-steps (81 taps + 7 zero weights)
  static constexpr int K2 = N1, NT3 = 32, QP = F3 * F3;
  static constexpr int PW = 144;                 // plane entries (16 bytes each)
  static constexpr int PF = PW * 4;              // floats per plane
  static constexpr int RQ = 8, RH = 4;           // ring slots: quad planes, H planes
  static constexpr int W_E1 = 0, N_E1 = 4, W_E2 = N_E1, W_E3 = W_E2 + 4, W_IM = W_E3 + 4,
                       N_IM = 5, W_I1 = W_IM + N_IM, W_I2 = W_I1 + 1, W_I3 = W_I2 + 1;
  static constexpr int NT = (W_I3 + 1) * 32;
  static constexpr int E1_CH = N1 / (N_E1 / 4);  // channels per E1 warp
  static constexpr int IM_THREADS = N_IM * 32;
  // shared memory carve-up (floats).  The H ring lies BELOW the quad ring: one K-step pairs a
  // chunk of H with a chunk of Qd through a (positive) leading-dimension byte offset.
  static constexpr int oHh = 0;
  static constexpr int oHl = oHh + RH * PF;
  static constexpr int oQh = oHl + RH * PF;
  static constexpr int oQl = oQh + RQ * PF;
  static constexpr int oW1 = oQl + RQ * PF;      // [128][K1]: rows 0..63 W_hi, 64..127 W_lo
  static constexpr int oW2 = oW1 + 2 * N1 * K1;  // [64][K2]: rows 0..31 W_hi, 32..63 W_lo
  static constexpr int oW3 = oW2 + 2 * N2 * K2;  // [64][N2]: rows = taps (25 of 32), hi then lo
  static constexpr int oB1 = oW3 + 2 * NT3 * N2;
  static constexpr int oB2 = oB1 + N1;
  static constexpr int oQs = oB2 + N2;           // 2 staged Q rows [M][QP]
  static constexpr int TOTAL = oQs + 2 * M * QP;
  static constexpr size_t SMEM_BYTES = sizeof(float) * (size_t)TOTAL;
  // tensor memory columns, every buffer twice (+ its size * (b & 1)).  The split A operand of
  // the next layer is written IN PLACE over the accumulator it was computed from:
  //   D1: [0,64) A_hi.W_hi + A_lo.W_hi, [64,128) A_hi.W_lo   ->  A2: [0,64) hi, [64,128) lo
  //   D2: [0,32) + [32,64) likewise                          ->  A3: [0,32) hi, [32,64) lo
  //   D3: [0,32) + [32,64) (25 taps of 32 used)
  static constexpr uint32_t cD1 = 0, cD2 = 256, cD3 = 384;
  static constexpr uint32_t TMEM_COLS = 512;
  static constexpr int BAR_E3 = 1;
};

// (K-step s, 16-byte chunk j, element e) of the layer-1 contraction -> filter tap dy*9+dx, or
// -1 for the 7 padding positions (they read real pixels; their weights are zero)
__host__ __device__ __forceinline__ int tap_of(int s, int j, int e) {
  int dy, dx;
  if (s == 0) { dy = 8; dx = 4 * j + e; }                      // H[c], H[c+4]
  else if (s == 1) {
    if (j == 0) { if (e) return -1; dy = 8; dx = 8; }          // H[c+8]: tap (8,8) + 3 pads
    else { dy = e; dx = 8; }                                   // Qd(y)[c+8]
  }
  else if (s < 6) { dy = e; dx = 2 * (s - 2) + j; }            // Qd(y)[c+dx], dx = 0..7
  else if (s < 10) { dy = 4 + e; dx = 2 * (s - 6) + j; }       // Qd(y+4)[c+dx], dx = 0..7
  else { if (j) return -1; dy = 4 + e; dx = 8; }               // Qd(y+4)[c+8], [c+9] = pad
  return dy * Cfg::F1 + dx;
}

#ifdef PL_TRACE
// event timeline of tiles PL_TRACE_BASE .. +7 of CTA (0,0,0): PL_EV(tile, event id)
#ifndef PL_TRACE_BASE
#define PL_TRACE_BASE 100
#endif
__device__ long long pl_trace[8][16];
#define PL_EV(t, e) if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (t) >= PL_TRACE_BASE && (t) < PL_TRACE_BASE + 8 && lane == 0) \
    pl_trace[(t) - PL_TRACE_BASE][e] = clock64();
#else
#define PL_EV(t, e) {}
#endif

using tc::mbar_arrive;
using tc::named_bar_sync;

// BATCH = true: the input is a batch of S small samples [S][ph][pw] (training patches).  The
// kernel then works on the VIRTUAL image [ph][S*pw] made of the samples laid side by side, so
// that a 128-pixel tile is filled whatever the sample width; columns whose window straddles two
// samples are computed and dropped (pw-8 of every pw columns are kept: 76 % for 33x33).
// Optionally the n1- and n2-channel maps are written to HBM ([S][h1][w1][N1], [S][h2][w2][N2]):
// that is the forward pass of a training step (ConfigBasedDataPipeline.cpp:165-168), whose
// activations are needed again by backpropagate().
struct BatchExt {
  float* out1;   // may be null
  float* out2;   // may be null
  int S, pw, ph;
  // when set: run only if *gate != 0 (the FP16-split kernel of fused_forward_hp.cuh found the
  // input outside its domain and left the launch to this kernel)
  const int* gate;
  // layer-1-only launches of the FP16-split kernel (9-5-5 training forward): |out1| maximum,
  // as an unsigned bit pattern (atomicMax), for the layer-2 kernel's operand scale
  unsigned* out1_max;
  // training forward (out2 kept): |out2| maximum for the tensor-core backward of layer 3
  unsigned* out2_max;
};

template <bool BATCH>
__global__ void __launch_bounds__(Cfg::NT, 1) forward_fused_pl_kernel(fused::Args a, int rpc,
                                                                      BatchExt bx) {
  using C = Cfg;
  using namespace tc;
  extern __shared__ __align__(128) float smem[];
  if (bx.gate != nullptr && *bx.gate == 0) return;
  float* sW1 = smem + C::oW1;
  float* sW2 = smem + C::oW2;
  float* sW3 = smem + C::oW3;
  float* sB1 = smem + C::oB1;
  float* sB2 = smem + C::oB2;
  float* sQs = smem + C::oQs;
  // p_full[i]/p_free[i]: planes of tile b (i = b&3) written / no longer read by MMA-1(b);
  // barN[i]: MMA-N of a tile with b&1 == i done; aN_full[i]: A operand of layer N written;
  // d3_free[i]: D3 buffer i drained.  Every TMEM buffer exists twice (tile parity).
  __shared__ __align__(8) uint64_t p_full[4], p_free[4], bar1[2], a2_full[2], bar2[2],
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

  // ---- stage parameters (all threads): B operands [n][k] canonical, rows 0..N-1 the TF32 hi
  // parts, rows N..2N-1 the lo parts (one N=2N MMA evaluates A_hi.W_hi and A_hi.W_lo) ----------
  for (int i = tid; i < 2 * C::N1 * C::K1; i += C::NT) {
    const int n = i / C::K1, k = i % C::K1;
    const int t = tap_of(k >> 3, (k >> 2) & 1, k & 3);
    float hi, lo;
    split_tf32(t >= 0 ? __ldg(a.pw1 + t * C::N1 + (n & (C::N1 - 1))) : 0.f, hi, lo);
    sW1[kmajor_offset(n, k, C::K1)] = n < C::N1 ? hi : lo;
  }
  for (int i = tid; i < 2 * C::N2 * C::K2; i += C::NT) {
    const int n = i / C::K2, k = i % C::K2;
    float hi, lo;
    split_tf32(__ldg(a.pw2 + k * C::N2 + (n & (C::N2 - 1))), hi, lo);
    sW2[kmajor_offset(n, k, C::K2)] = n < C::N2 ? hi : lo;
  }
  for (int i = tid; i < 2 * C::NT3 * C::N2; i += C::NT) {
    const int n = i / C::N2, k = i % C::N2;   // n & 31 = tap dy*5+dx, k = channel
    const int tap = n & (C::NT3 - 1);
    float hi, lo;
    split_tf32(tap < C::QP ? __ldg(a.pw3 + tap * C::N2 + k) : 0.f, hi, lo);
    sW3[kmajor_offset(n, k, C::N2)] = n < C::NT3 ? hi : lo;
  }
  for (int i = tid; i < C::N1; i += C::NT) sB1[i] = __ldg(a.pb1 + i);
  for (int i = tid; i < C::N2; i += C::NT) sB2[i] = __ldg(a.pb2 + i);
  // pad entries of the planes are read by the tensor core (times a zero weight): keep them finite
  for (int i = tid; i < 2 * (C::RH + C::RQ) * C::PF; i += C::NT) smem[i] = 0.f;
  const float b3 = __ldg(a.pb3);

  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    if (smem_u32(smem) & 127u) __trap();
    for (int i = 0; i < 4; i++) {
      mbar_init(&p_full[i], C::IM_THREADS);
      mbar_init(&p_free[i], 1);
    }
    for (int i = 0; i < 2; i++) {
      mbar_init(&bar1[i], 1);
      mbar_init(&a2_full[i], C::N_E1 * 32);
      mbar_init(&bar2[i], 1);
      mbar_init(&a3_full[i], 128);
      mbar_init(&bar3[i], 1);
      mbar_init(&d3_free[i], 128);
    }
  }
  fence_proxy_async();   // the weight operands are read by the tensor core (async proxy)
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;

  const int rows_here = min(rpc, a.h3 - R0);
  const int n_tiles = rows_here + (C::F3 - 1);   // out2 rows R0 .. R0+rows_here+3

  if (warp >= C::W_IM && warp < C::W_IM + C::N_IM) {
    // ============================ IM: plane producers =====================================
    // thread c owns plane column c (image column X0+c).  The quad of the last four rows at
    // this column lives in registers, so each input row costs 4 loads, 4 splits and 4 STS.128.
    const int c = tid - C::W_IM * 32;
    const bool active = c < C::PW;
    const int gx = X0 + c;
    float* sHh = smem + C::oHh + c * 4;
    float* sHl = smem + C::oHl + c * 4;
    float* sQh = smem + C::oQh + c * 4;
    float* sQl = smem + C::oQl + c * 4;
    // BATCH: virtual column gx+e -> (sample, column) once; a row is then one add away
    long long boff[4];
    if (BATCH) {
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int vx = gx + e;
        const int smp = vx / bx.pw;
        boff[e] = (active && vx < a.w) ? (long long)smp * bx.pw * bx.ph + (vx - smp * bx.pw) : -1;
      }
    }
    auto ld = [&](int r, int e) -> float {
      const int gy = R0 + r;
      if (BATCH) return (boff[e] >= 0 && gy < a.h) ? __ldg(img + boff[e] + (long long)gy * bx.pw) : 0.f;
      return (active && gy < a.h && gx + e < a.w) ? __ldg(img + (size_t)gy * a.w + gx + e) : 0.f;
    };
    float qh0 = 0.f, qh1 = 0.f, qh2 = 0.f, ql0 = 0.f, ql1 = 0.f, ql2 = 0.f;
    {
      float pv[C::F1 - 1];
#pragma unroll
      for (int r = 0; r < C::F1 - 1; r++) pv[r] = ld(r, 0);
#pragma unroll
      for (int r = 0; r < C::F1 - 1; r++) {   // rows 0..7 -> Qd(0..4)
        float h, l;
        split_tf32(pv[r], h, l);
        if (r >= 3 && active) {
          const int slot = (r - 3) & (C::RQ - 1);
          *reinterpret_cast<float4*>(sQh + slot * C::PF) = make_float4(qh0, qh1, qh2, h);
          *reinterpret_cast<float4*>(sQl + slot * C::PF) = make_float4(ql0, ql1, ql2, l);
        }
        qh0 = qh1; qh1 = qh2; qh2 = h;
        ql0 = ql1; ql1 = ql2; ql2 = l;
      }
    }
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; e++) v[e] = ld(C::F1 - 1, e);
    for (int b = 0; b < n_tiles; b++) {
      float nv[4];
#pragma unroll
      for (int e = 0; e < 4; e++) nv[e] = (b + 1 < n_tiles) ? ld(b + C::F1, e) : 0.f;
      float h[4], l[4];
#pragma unroll
      for (int e = 0; e < 4; e++) split_tf32(v[e], h[e], l[e]);
      // H(b+8) replaces H(b+4) (last read by MMA-1(b-4)), Qd(b+5) replaces Qd(b-3) (MMA-1(b-3))
      if (b >= 3) mbar_wait(&p_free[(b - 3) & 3], (uint32_t)(((b - 3) >> 2) & 1));
      if (active) {
        const int sh = b & (C::RH - 1), sq = (b + 5) & (C::RQ - 1);
        *reinterpret_cast<float4*>(sHh + sh * C::PF) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(sHl + sh * C::PF) = make_float4(l[0], l[1], l[2], l[3]);
        *reinterpret_cast<float4*>(sQh + sq * C::PF) = make_float4(qh0, qh1, qh2, h[0]);
        *reinterpret_cast<float4*>(sQl + sq * C::PF) = make_float4(ql0, ql1, ql2, l[0]);
      }
      qh0 = qh1; qh1 = qh2; qh2 = h[0];
      ql0 = ql1; ql1 = ql2; ql2 = l[0];
      fence_proxy_async();
      mbar_arrive(&p_full[b & 3]);
      if (warp == C::W_IM) PL_EV(b, 12)
#pragma unroll
      for (int e = 0; e < 4; e++) v[e] = nv[e];
    }
  } else if (warp == C::W_I1) {
    // ============================ I1: layer-1 MMA issuer ===================================
    {
      const uint32_t idesc_hi = make_idesc_tf32(C::M, 2 * C::N1);   // A_hi x [W_hi; W_lo]
      const uint32_t idesc_lo = make_idesc_tf32(C::M, C::N1);       // A_lo x W_hi
      const uint64_t wdesc = make_desc_kmajor(sW1, 0, 128, 128 * (C::K1 / 4));
      const uint32_t aHh = smem_u32(smem + C::oHh), aHl = smem_u32(smem + C::oHl);
      const uint32_t aQh = smem_u32(smem + C::oQh), aQl = smem_u32(smem + C::oQl);
      constexpr uint32_t PB = C::PF * 4;   // bytes per plane
      // descriptor of a plane chunk pair: start address, LBO (second chunk), SBO = 128
      auto adesc = [](uint32_t addr, uint32_t lbo) -> uint64_t {
        return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
               ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
      };
      for (int t = 0; t < n_tiles; t++) {
        mbar_wait(&p_full[t & 3], (uint32_t)((t >> 2) & 1));
        // D1[t&1] still holds A2(t-2) until MMA-2(t-2) has read it
        if (t >= 2) mbar_wait(&bar2[t & 1], (uint32_t)(((t - 2) >> 1) & 1));
        tcgen05_fence_after();
        const uint32_t d1 = tmem + C::cD1 + 128u * (uint32_t)(t & 1);
        const uint32_t sh = (uint32_t)(t & (C::RH - 1)) * PB;
        const uint32_t s0 = (uint32_t)(t & (C::RQ - 1)) * PB;
        const uint32_t s4 = (uint32_t)((t + 4) & (C::RQ - 1)) * PB;
        PL_EV(t, 0)
        if (elect_one()) {
#pragma unroll
        for (int s = 0; s < C::KS1; s++) {
          uint32_t ah, al, lbo_h, lbo_l;
          if (s == 0) { ah = aHh + sh; al = aHl + sh; lbo_h = lbo_l = 64; }
          else if (s == 1) {
            ah = aHh + sh + 128; al = aHl + sh + 128;
            lbo_h = (aQh + s0 + 128) - ah; lbo_l = (aQl + s0 + 128) - al;
          }
          else if (s < 6) { ah = aQh + s0 + 32 * (s - 2); al = aQl + s0 + 32 * (s - 2); lbo_h = lbo_l = 16; }
          else if (s < 10) { ah = aQh + s4 + 32 * (s - 6); al = aQl + s4 + 32 * (s - 6); lbo_h = lbo_l = 16; }
          else { ah = aQh + s4 + 128; al = aQl + s4 + 128; lbo_h = lbo_l = 16; }
          mma_tf32(d1, adesc(ah, lbo_h), wdesc + 16 * s, idesc_hi, s > 0);
          mma_tf32(d1, adesc(al, lbo_l), wdesc + 16 * s, idesc_lo, 1);
        }
        mma_commit(&bar1[t & 1]);
        mma_commit(&p_free[t & 3]);
        }
        __syncwarp();
        PL_EV(t, 1)
      }
    }
  } else if (warp == C::W_I2) {
    // ============================ I2: layer-2 MMA issuer (A2 in TMEM) ======================
    {
      const uint32_t idesc_hi = make_idesc_tf32(C::M, 2 * C::N2);   // A2_hi x [W2_hi; W2_lo]
      const uint32_t idesc_lo = make_idesc_tf32(C::M, C::N2);       // A2_lo x W2_hi
      const uint64_t wdesc = make_desc_kmajor(sW2, 0, 128, 128 * (C::K2 / 4));
      for (int t = 0; t < n_tiles; t++) {
        mbar_wait(&a2_full[t & 1], (uint32_t)((t >> 1) & 1));
        // D2[t&1] still holds A3(t-2) until MMA-3(t-2) has read it
        if (t >= 2) mbar_wait(&bar3[t & 1], (uint32_t)(((t - 2) >> 1) & 1));
        tcgen05_fence_after();
        const uint32_t a2 = tmem + C::cD1 + 128u * (uint32_t)(t & 1);
        const uint32_t d2 = tmem + C::cD2 + 64u * (uint32_t)(t & 1);
        PL_EV(t, 4)
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < C::K2 / 8; ks++) {
            mma_tf32_ts(d2, a2 + ks * 8, wdesc + 16 * ks, idesc_hi, ks > 0);
            mma_tf32_ts(d2, a2 + C::N1 + ks * 8, wdesc + 16 * ks, idesc_lo, 1);
          }
          mma_commit(&bar2[t & 1]);
        }
        __syncwarp();
        PL_EV(t, 5)
      }
    }
  } else if (warp == C::W_I3) {
    // ============================ I3: layer-3 tap-GEMM issuer (A3 in TMEM) =================
    {
      const uint32_t idesc_hi = make_idesc_tf32(C::M, 2 * C::NT3);
      const uint32_t idesc_lo = make_idesc_tf32(C::M, C::NT3);
      const uint64_t wdesc = make_desc_kmajor(sW3, 0, 128, 128 * (C::N2 / 4));
      for (int t = 0; t < n_tiles; t++) {
        mbar_wait(&a3_full[t & 1], (uint32_t)((t >> 1) & 1));
        if (t >= 2) mbar_wait(&d3_free[t & 1], (uint32_t)(((t - 2) >> 1) & 1));
        tcgen05_fence_after();
        const uint32_t a3 = tmem + C::cD2 + 64u * (uint32_t)(t & 1);
        const uint32_t d3 = tmem + C::cD3 + 64u * (uint32_t)(t & 1);
        PL_EV(t, 8)
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < C::N2 / 8; ks++) {
            mma_tf32_ts(d3, a3 + ks * 8, wdesc + 16 * ks, idesc_hi, ks > 0);
            mma_tf32_ts(d3, a3 + C::N2 + ks * 8, wdesc + 16 * ks, idesc_lo, 1);
          }
          mma_commit(&bar3[t & 1]);
        }
        __syncwarp();
        PL_EV(t, 9)
      }
    }
  } else if (warp < C::W_E1 + C::N_E1) {
    // ============================ E1: A2 = split(relu(D1 + b1)), in place ==================
    // warp w works on TMEM lane quarter w&3 (the quarter a warp may access) and on channels
    // E1_CH*(w>>2) .. +E1_CH-1, 16 at a time.  Measured (probe/tmem_bw_probe.cu, and A/B runs of
    // this kernel): a tcgen05.ld/st round trip is ~125/~100 cycles, but TMEM traffic of the
    // epilogue warps disturbs the MMA stream, so neither 8 E1 warps (1.65 ms), nor fetching 32
    // channels ahead (1.53 ms), nor a software-pipelined chunk loop (1.56 ms) beats this plain
    // loop (1.49 ms on C3).
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int ch0 = (warp >> 2) * C::E1_CH;
    // BATCH: this thread's pixel of the n1-channel map (row 0), or null when not kept
    float* o1 = nullptr;
    if (BATCH && bx.out1) {
      const int m = (warp & 3) * 32 + lane, vx = X0 + m, smp = vx / bx.pw, px = vx - smp * bx.pw;
      const int w1 = bx.pw - (C::F1 - 1), h1 = bx.ph - (C::F1 - 1);
      if ((m < C::OW3 || last_strip) && vx < a.w && px < w1)
        o1 = bx.out1 + (((size_t)smp * h1 + R0) * w1 + px) * C::N1 + ch0;
    }
    const size_t o1_row = (size_t)(bx.pw - (C::F1 - 1)) * C::N1;
    for (int b = 0; b < n_tiles; b++) {
      mbar_wait(&bar1[b & 1], (uint32_t)((b >> 1) & 1));       // MMA-1(b) done
      if (warp == 0) PL_EV(b, 2)
      tcgen05_fence_after();
#pragma unroll 1
      for (int c16 = 0; c16 < C::E1_CH; c16 += 16) {
        const uint32_t d1 = tmem + lane_base + C::cD1 + 128u * (uint32_t)(b & 1) + ch0 + c16;
        float va[16], vb[16];
        tmem_ld16_nowait(d1, va);                       // A_hi.W_hi + A_lo.W_hi
        tmem_ld16_nowait(d1 + C::N1, vb);               // A_hi.W_lo
        tmem_ld_wait();
#pragma unroll
        for (int h8 = 0; h8 < 2; h8++) {
          float hi[8], lo[8];
          const float* bp = sB1 + ch0 + c16 + h8 * 8;
          const float4 ba = *reinterpret_cast<const float4*>(bp);
          const float4 bb = *reinterpret_cast<const float4*>(bp + 4);
          const float bias[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
          float act[8];
#pragma unroll
          for (int j = 0; j < 8; j++) {
            act[j] = fmaxf((va[h8 * 8 + j] + vb[h8 * 8 + j]) + bias[j], 0.f);
            split_tf32(act[j], hi[j], lo[j]);
          }
          tmem_st8(d1 + h8 * 8, hi);
          tmem_st8(d1 + C::N1 + h8 * 8, lo);
          if (BATCH && o1) {
            float4* q = reinterpret_cast<float4*>(o1 + (size_t)b * o1_row + c16 + h8 * 8);
            q[0] = make_float4(act[0], act[1], act[2], act[3]);
            q[1] = make_float4(act[4], act[5], act[6], act[7]);
          }
        }
      }
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive(&a2_full[b & 1]);
      if (warp == 0) PL_EV(b, 3)
    }
  } else if (warp < C::W_E3) {
    // ============================ E2: A3 = split(relu(D2 + b2)), in place ==================
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    float* o2 = nullptr;
    if (BATCH && bx.out2) {
      const int m = (warp & 3) * 32 + lane, vx = X0 + m, smp = vx / bx.pw, px = vx - smp * bx.pw;
      const int w2 = bx.pw - (C::F1 - 1), h2 = bx.ph - (C::F1 - 1);
      if ((m < C::OW3 || last_strip) && vx < a.w && px < w2)
        o2 = bx.out2 + (((size_t)smp * h2 + R0) * w2 + px) * C::N2;
    }
    const size_t o2_row = (size_t)(bx.pw - (C::F1 - 1)) * C::N2;
    float act2_max = 0.f;   // largest out2 value this thread stored (training forward)
    for (int b = 0; b < n_tiles; b++) {
      mbar_wait(&bar2[b & 1], (uint32_t)((b >> 1) & 1));       // MMA-2(b) done
      if (warp == C::W_E2) PL_EV(b, 6)
      tcgen05_fence_after();
      const uint32_t d2 = tmem + lane_base + C::cD2 + 64u * (uint32_t)(b & 1);
#pragma unroll
      for (int g = 0; g < 2; g++) {
        float va[16], vb[16];
        tmem_ld16_nowait(d2 + g * 16, va);
        tmem_ld16_nowait(d2 + C::N2 + g * 16, vb);
        tmem_ld_wait();
#pragma unroll
        for (int h8 = 0; h8 < 2; h8++) {
          float hi[8], lo[8];
          float act[8];
#pragma unroll
          for (int j = 0; j < 8; j++) {
            act[j] = fmaxf((va[h8 * 8 + j] + vb[h8 * 8 + j]) + sB2[g * 16 + h8 * 8 + j], 0.f);
            split_tf32(act[j], hi[j], lo[j]);
          }
          tmem_st8(d2 + g * 16 + h8 * 8, hi);
          tmem_st8(d2 + C::N2 + g * 16 + h8 * 8, lo);
          if (BATCH && o2) {
            float4* q = reinterpret_cast<float4*>(o2 + (size_t)b * o2_row + g * 16 + h8 * 8);
            q[0] = make_float4(act[0], act[1], act[2], act[3]);
            q[1] = make_float4(act[4], act[5], act[6], act[7]);
#pragma unroll
            for (int j = 0; j < 8; j++) act2_max = fmaxf(act2_max, act[j]);
          }
        }
      }
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive(&a3_full[b & 1]);
      if (warp == C::W_E2) PL_EV(b, 7)
    }
    if (BATCH && bx.out2 && bx.out2_max) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) act2_max = fmaxf(act2_max, __shfl_xor_sync(0xffffffffu, act2_max, o));
      if (lane == 0 && act2_max > 0.f) atomicMax(bx.out2_max, __float_as_uint(act2_max));
    }
  } else if (warp < C::W_IM) {
    // ============================ E3: Q row -> smem, 25-term gather -> out3 ================
    // thread x owns output column X0+x; the partial sums of the four output rows that still
    // miss out2 rows live in its registers (acc0 = oldest).
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
      mbar_wait(&bar3[b & 1], (uint32_t)((b >> 1) & 1));       // MMA-3(b) done
      if (warp == C::W_E3) PL_EV(b, 10)
      tcgen05_fence_after();
      const uint32_t d3 = tmem + lane_base + C::cD3 + 64u * (uint32_t)(b & 1);
      float v[32], w[32];
      tmem_ld16_nowait(d3, v);
      tmem_ld16_nowait(d3 + 16, v + 16);
      tmem_ld16_nowait(d3 + 32, w);
      tmem_ld16_nowait(d3 + 48, w + 16);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&d3_free[b & 1]);                            // D3[b&1] may be overwritten
      float* qs = sQs + (b & 1) * (C::M * C::QP);
#pragma unroll
      for (int j = 0; j < C::QP; j++) qs[x * C::QP + j] = v[j] + w[j];
      named_bar_sync(C::BAR_E3, 128);                          // Q row visible to its neighbours
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
      // out2 row b contributes its filter row dy to output row b-dy
      const float done = acc0 + r[4];
      acc0 = acc1 + r[3];
      acc1 = acc2 + r[2];
      acc2 = acc3 + r[1];
      acc3 = r[0];
      if (b >= C::F3 - 1 && live)
        dst[o3 + (size_t)(b - (C::F3 - 1)) * o3_row] = done + b3;
      if (warp == C::W_E3) PL_EV(b, 11)
    }
  }

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
  SRCNN_CUDA(cudaFuncSetAttribute(forward_fused_pl_kernel<false>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Cfg::SMEM_BYTES));
  SRCNN_CUDA(cudaFuncSetAttribute(forward_fused_pl_kernel<true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Cfg::SMEM_BYTES));
  return SRCNN_OK;
}

inline bool supported(int n1, int n2, int f1, int f2, int f3) {
  return n1 == 64 && n2 == 32 && f1 == 9 && f2 == 1 && f3 == 5;
}

// rows of a strip per CTA: the fewest full waves of (strips x bands x S) CTAs over the SMs,
// each CTA paying F3-1 halo tiles plus the pipeline fill
inline int rows_per_cta(int w3, int h3, int S, int sm_count) {
  const long strips = (w3 + Cfg::OW3 - 1) / Cfg::OW3;
  long best_cost = -1;
  int best_rpc = h3;
  for (int nb = 1; nb <= 512 && nb <= h3; nb++) {
    const int rpc = (h3 + nb - 1) / nb;
    const long ctas = strips * ((h3 + rpc - 1) / rpc) * S;
    const long waves = (ctas + sm_count - 1) / sm_count;
    const long cost = waves * (rpc + (Cfg::F3 - 1) + 8);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best_rpc = rpc;
    }
  }
  return best_rpc;
}

inline int launch(srcnn_ctx* ctx, const fused::Args& a, int S) {
  const int rpc = rows_per_cta(a.w3, a.h3, S, ctx->sm_count > 0 ? ctx->sm_count : 148);
  dim3 grid((a.w3 + Cfg::OW3 - 1) / Cfg::OW3, (a.h3 + rpc - 1) / rpc, S);
  forward_fused_pl_kernel<false><<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(a, rpc,
                                                                                 BatchExt{});
  return SRCNN_OK;
}

// a batch of S samples of pw x ph pixels as one virtual image; out1/out2 may be null
inline int launch_batch(srcnn_ctx* ctx, const fused::Args& a, int S, float* out1, float* out2,
                        unsigned* out2_max = nullptr) {
  fused::Args v = a;
  const int pad = Cfg::F1 + Cfg::F3 - 2;
  v.w = S * a.w;
  v.w3 = S * a.w - pad;
  const int rpc = rows_per_cta(v.w3, v.h3, 1, ctx->sm_count > 0 ? ctx->sm_count : 148);
  dim3 grid((v.w3 + Cfg::OW3 - 1) / Cfg::OW3, (v.h3 + rpc - 1) / rpc, 1);
  BatchExt bx{};
  bx.out1 = out1;
  bx.out2 = out2;
  bx.S = S;
  bx.pw = a.w;
  bx.ph = a.h;
  bx.out2_max = out2_max;
  if (out2_max) SRCNN_CUDA(cudaMemsetAsync(out2_max, 0, sizeof(unsigned), ctx->stream));
  forward_fused_pl_kernel<true><<<grid, Cfg::NT, Cfg::SMEM_BYTES, ctx->stream>>>(v, rpc, bx);
  return SRCNN_OK;
}

}  // namespace fused_pl
}  // namespace srcnn
