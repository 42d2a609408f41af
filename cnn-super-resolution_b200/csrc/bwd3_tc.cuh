// Backward of the last layer (f3 = 5, n2 = 32 channels -> 1) on the tensor cores, one launch:
//     d2[s][j][i][n] = [out2[s][j][i][n] > 0] * sum_{dy,dx} W3[dy][dx][n] * d3[s][j-dy][i-dx]
//     gW3[dy][dx][n] += sum_{s,y,x} d3[s][y][x] * out2[s][y+dy][x+dx][n],   gB3 += sum d3
// reference: src/kernel/layer_deltas.cl:42-127 (layer 2 <- layer 3) and
// src/kernel/backpropagate.cl:56-114 (layer 3), sequenced by
// src/ConfigBasedDataPipeline.cpp:258-295; d3 itself (last_layer_delta.cl:14-50) comes from
// d3_kernel below, which also measures its maximum.
//
// d3 has ONE channel, so both contractions see a Hankel matrix -- the structure the fused
// forward kernel uses for layer 1.  The samples of a chunk lie side by side as a virtual image
// (slot = out2's width: the w3-wide d3 row + 4 zero columns, which also are the next sample's
// left padding); a CTA owns 128 virtual columns and marches down out2's rows j.  Per row it
// builds ONE "oct plane" O_j[c] = (d3[j-7..j][c]) as 8 halves (hi and lo), kept from the running
// column history in registers.  Then
//   * d2 row j:  A = O_j read at base + (5 - dx) entries (K-major, rows = pixels, K = 8 rows of
//     the entry = taps dy = 7 - e; pairs of dx per K = 16 step), B = W3 packed [n][48]:
//     3 K-steps x 2 MMAs (A_hi x [W_hi; W_lo], A_lo x W_hi) -> D2[j & 1];
//   * gW3 += ...: the SAME plane as an MN-major A operand whose M groups OVERLAP (SBO = 16 bytes:
//     group g = the plane shifted by g entries = tap dx = 5 - g; tools/probe/mn16_probe.cu), M = 64
//     rows (g, e) = (dx, dy), K = the 128 pixels of the row in 8 steps, B = out2's row as
//     MN-major planes [hi 4 groups | lo 4 groups]: 8 x 2 MMAs into one persistent accumulator.
// out2 is read once (planes for the gradient; the epilogue re-reads its pixel from L2 for the
// ReLU' mask), d2 written once: 256 B per out2 pixel -- the kernel is HBM-bound (the FP32 SIMT
// kernel it replaces ran at 23 % of the HBM rate, FFMA-bound at 50 FFMA per element).
//
//   P  (5 warps)  d3 column history -> oct plane hi/lo of row j, bias sum     -> pfull[slot]
//   Q  (8 warps)  out2 row j -> MN-major planes hi/lo                          -> qfull[slot]
//   I0            d2 MMAs (6 per row)                                          -> d2_done[j&1]
//   I1            gW3 MMAs (16 per row)                                        -> pfree, qfree
//   E  (4 warps)  D2 -> scale, ReLU' mask -> d2 row j; at the end gW3 / gB3 -> per-CTA partial
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "context.cuh"
#include "conv5_tc.cuh"
#include "tc_common.cuh"

namespace srcnn {
namespace b3tc {

struct Cfg {
  static constexpr int F = 5, T = 25, N = 32;
  static constexpr int M = 128;                        // out2 pixels per strip row
  static constexpr int PW = 136, PB = PW * 16;         // oct plane: entries, bytes
  static constexpr int RP = 4, P_SLOT = 2 * PB;        // plane ring: hi plane + lo plane
  // one 8-channel group plane of out2: 128 entries of 16 bytes + 32 bytes of padding, so that the
  // four planes a quarter-warp of producers writes to start 8 banks apart
  static constexpr int GP = M * 16 + 32;
  static constexpr int RQ = 3, Q_SLOT = 8 * GP;        // out2 ring: hi groups 0..3, lo groups 4..7
  static constexpr int KW = 48;                        // K of the d2 GEMM (3 steps of 16)
  static constexpr int W_BYTES = 2 * N * KW * 2;       // [W_hi 32 rows; W_lo 32 rows][48] halves
  static constexpr int SP = 36;                        // floats per staged d2 pixel (128 B + pad)
  static constexpr int oP = 0, oQ = oP + RP * P_SLOT, oW = oQ + RQ * Q_SLOT;
  static constexpr int oMask = oW + W_BYTES;           // [RQ][M] ReLU' masks of the out2 rows
  static constexpr int oStage = oMask + RQ * M * 4;    // 4 epilogue warps x 32 pixels x SP floats
  static constexpr size_t SMEM_BYTES = (size_t)oStage + 4 * 32 * SP * 4;
  static constexpr int W_E = 0, W_P = 4, N_P = 5, W_Q = W_P + N_P, N_Q = 8, W_I = W_Q + N_Q,
                       NT = (W_I + 2) * 32;
  static constexpr uint32_t cD2 = 0, cGW = 128, TMEM_COLS = 256;
};

// d3 = (out3 - crop(gt)) * [out3 > 0] (quirk Q2 kept), and its |max| as a bit pattern
__global__ void __launch_bounds__(256) d3_kernel(const float* __restrict__ gt,
                                                 const float* __restrict__ out3,
                                                 float* __restrict__ d3, int gt_w, int gt_h, int w3,
                                                 int h3, long long total, unsigned* d3_max) {
  const int pad = (gt_w - w3) / 2;
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long s = i / ((long long)w3 * h3);
    const int rem = (int)(i - s * w3 * h3), y = rem / w3, x = rem - y * w3;
    const float o = __ldg(out3 + i);
    const float t = __ldg(gt + ((long long)s * gt_h + y + pad) * gt_w + pad + x);
    const float dv = o > 0.f ? o - t : 0.f;
    d3[i] = dv;
    m = fmaxf(m, fabsf(dv));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(d3_max, __float_as_uint(m));
}

struct Args {
  const float* d3;       // [S][h3][w3]
  const float* out2;     // [S][oh][ow][32]
  const float* W3;       // [25][32]
  float* d2;             // [S][oh][ow][32]
  float* partial;        // [grid][25*32 + 1]
  const unsigned* d3_max;
  const unsigned* out2_max;
  unsigned* d2_max;      // receives max |d2| (zeroed by the launcher)
  int S, ow, oh;         // out2 extent (w3 = ow - 4, h3 = oh - 4)
};

__global__ void __launch_bounds__(Cfg::NT, 1) bwd3_tc_kernel(Args a) {
  using C = Cfg;
  using namespace tc;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t pfull[C::RP], pfree[C::RP], qfull[C::RQ], qfree[C::RQ],
      d2_done[2], d2_free[2], gw_done;
  __shared__ uint32_t tmem_slot;
  __shared__ float s_wmax[8];
  __shared__ float s_gb[C::N_P];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ow = a.ow, oh = a.oh, w3 = ow - (C::F - 1), h3 = oh - (C::F - 1);
  const long long vw = (long long)a.S * ow;
  const long long X0 = (long long)blockIdx.x * C::M;

  // ---- W3 image: scale from max |W3| (800 values, every thread helps), packed K-major --------
  float wm = 0.f;
  for (int i = tid; i < C::T * C::N; i += C::NT) wm = fmaxf(wm, fabsf(__ldg(a.W3 + i)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
  if (warp < 8 && lane == 0) s_wmax[warp] = 0.f;
  __syncthreads();
  if (lane == 0 && wm > 0.f) atomicMax(reinterpret_cast<unsigned*>(&s_wmax[warp & 7]), __float_as_uint(wm));
  // the planes' pad entries are read by the tensor core (times zero weights / into rows nobody
  // stores): keep them finite
  for (int i = tid; i < (C::RP * C::P_SLOT + C::RQ * C::Q_SLOT) / 4; i += C::NT)
    reinterpret_cast<uint32_t*>(smem_raw)[i] = 0u;
  if (warp == 0) tmem_alloc(&tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    if (smem_u32(smem_raw) & 127u) __trap();
    for (int i = 0; i < C::RP; i++) {
      mbar_init(&pfull[i], C::N_P * 32);
      mbar_init(&pfree[i], 2);          // both issuers read the plane
    }
    for (int i = 0; i < C::RQ; i++) {
      mbar_init(&qfull[i], C::N_Q * 32);
      mbar_init(&qfree[i], 1 + 128);   // the gradient MMAs + the epilogue's mask readers
    }
    for (int i = 0; i < 2; i++) {
      mbar_init(&d2_done[i], 1);
      mbar_init(&d2_free[i], 128);
    }
    mbar_init(&gw_done, 1);
  }
  __syncthreads();
  float wmax = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) wmax = fmaxf(wmax, s_wmax[i]);
  const float s_w = c5::scale_for(wmax);
  {
    // element (row n | 32 + n, k = 16 s + 8 c + e): tap dx = (c == 0 ? 2 s + 1 : 2 s), dy = 7 - e
    __half* sW = reinterpret_cast<__half*>(smem_raw + C::oW);
    for (int i = tid; i < C::N * C::KW; i += C::NT) {
      const int n = i / C::KW, k = i % C::KW;
      const int s = k >> 4, c = (k >> 3) & 1, e = k & 7;
      const int dx = c == 0 ? 2 * s + 1 : 2 * s, dy = 7 - e;
      const float w = (dx < C::F && dy < C::F) ? __ldg(a.W3 + (dy * C::F + dx) * C::N + n) * s_w : 0.f;
      unsigned short hi, lo;
      split_h(w, hi, lo);
      sW[kmajor16(n, k, C::KW)] = __ushort_as_half(hi);
      sW[kmajor16(C::N + n, k, C::KW)] = __ushort_as_half(lo);
    }
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  const float s_d = c5::scale_for(__uint_as_float(__ldg(a.d3_max)));
  const float s_o = c5::scale_for(__uint_as_float(__ldg(a.out2_max)));
  float* part = a.partial + (size_t)blockIdx.x * (C::T * C::N + 1);

  if (warp >= C::W_P && warp < C::W_P + C::N_P) {
    // ============================ P: oct planes of d3 ==========================================
    // thread q owns plane entry q = d3 virtual column X0 + q - 5
    const int q = tid - C::W_P * 32;
    const long long vq = X0 + q - 5;
    long long base = -1;
    if (q < C::PW && vq >= 0 && vq < vw) {
      const int smp = (int)(vq / ow), x = (int)(vq - (long long)smp * ow);
      if (x < w3) base = ((long long)smp * h3) * w3 + x;
    }
    const bool own = q >= 5 && q < 5 + C::M;       // columns of this strip: counted in gB3 once
    float gb = 0.f;
    unsigned short hh[7], hl[7];                   // rows j-7 .. j-1
#pragma unroll
    for (int r = 0; r < 7; r++) hh[r] = hl[r] = 0;
    uint8_t* my = smem_raw + C::oP + q * 16;
    auto ld3 = [&](int j) -> float {
      return (base >= 0 && j < h3) ? __ldg(a.d3 + base + (long long)j * w3) : 0.f;
    };
    float v = ld3(0), v1 = ld3(1), v2 = ld3(2);   // three rows of d3 in flight
    for (int j = 0; j < oh; j++) {
      const int slot = j % C::RP;
      unsigned short nh, nl;
      split_h(v * s_d, nh, nl);
      if (own) gb += v;
      const float v3 = ld3(j + 3);
      if (j >= C::RP) mbar_wait(&pfree[slot], (uint32_t)(((j / C::RP) - 1) & 1));
      if (q < C::PW) {
        uint8_t* s = my + slot * C::P_SLOT;
        *reinterpret_cast<uint4*>(s) = make_uint4(pack2(hh[0], hh[1]), pack2(hh[2], hh[3]),
                                                  pack2(hh[4], hh[5]), pack2(hh[6], nh));
        *reinterpret_cast<uint4*>(s + C::PB) = make_uint4(pack2(hl[0], hl[1]), pack2(hl[2], hl[3]),
                                                          pack2(hl[4], hl[5]), pack2(hl[6], nl));
      }
#pragma unroll
      for (int r = 0; r < 6; r++) { hh[r] = hh[r + 1]; hl[r] = hl[r + 1]; }
      hh[6] = nh; hl[6] = nl;
      fence_proxy_async();
      mbar_arrive(&pfull[slot]);
      v = v1; v1 = v2; v2 = v3;
    }
    // bias gradient of this CTA: lanes, then the 5 producer warps in order
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gb += __shfl_xor_sync(0xffffffffu, gb, o);
    if (lane == 0) s_gb[warp - C::W_P] = gb;
  } else if (warp >= C::W_Q && warp < C::W_Q + C::N_Q) {
    // ============================ Q: out2 row -> MN-major planes ===============================
    // thread = (8-channel group g, pixels m0 and m0 + 64): a warp's lanes read consecutive
    // 32-byte pieces (8 pixels x 128 bytes per instruction pair; a thread-per-pixel mapping
    // touched 16-32 lines per load and kept the L1 pipe at 83 %, r2i)
    const int t = tid - C::W_Q * 32, g = t & 3, m0 = t >> 2;
    long long base[2];
#pragma unroll
    for (int it = 0; it < 2; it++) {
      const long long vm = X0 + m0 + 64 * it;
      base[it] = -1;
      if (vm < vw) {
        const int smp = (int)(vm / ow), x = (int)(vm - (long long)smp * ow);
        base[it] = (((long long)smp * oh) * ow + x) * C::N + g * 8;
      }
    }
    const long long row = (long long)ow * C::N;
    // three rows of loads in flight per thread (48 KB per SM): one row ahead left the HBM latency
    // exposed on every row
    constexpr int DEPTH = 3;
    float4 vq[DEPTH][4];
    auto load = [&](int j, float4 (&dst)[4]) {
#pragma unroll
      for (int it = 0; it < 2; it++) {
        if (base[it] >= 0 && j < oh) {
          const float4* p = reinterpret_cast<const float4*>(a.out2 + base[it] + j * row);
          dst[2 * it] = __ldg(p);
          dst[2 * it + 1] = __ldg(p + 1);
        } else {
          dst[2 * it] = dst[2 * it + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
#pragma unroll
    for (int d = 0; d < DEPTH; d++) load(d, vq[d]);
    uint8_t* my = smem_raw + C::oQ + g * C::GP + m0 * 16;
    uint32_t* smask = reinterpret_cast<uint32_t*>(smem_raw + C::oMask);
#pragma unroll 1
    for (int j0 = 0; j0 < oh; j0 += DEPTH) {
#pragma unroll
      for (int d = 0; d < DEPTH; d++) {
        const int j = j0 + d;
        if (j < oh) {
          const int slot = j % C::RQ;
          uint32_t hi[8], lo[8], bits[2];
#pragma unroll
          for (int c = 0; c < 4; c++) {
            const float4 v = vq[d][c];
            split_h2(v.x * s_o, v.y * s_o, hi[2 * c], lo[2 * c]);
            split_h2(v.z * s_o, v.w * s_o, hi[2 * c + 1], lo[2 * c + 1]);
          }
#pragma unroll
          for (int it = 0; it < 2; it++) {   // ReLU' mask bits of this thread's 8 channels
            const float4 p = vq[d][2 * it], q = vq[d][2 * it + 1];
            uint32_t b = (p.x > 0.f ? 1u : 0u) | (p.y > 0.f ? 2u : 0u) | (p.z > 0.f ? 4u : 0u) |
                         (p.w > 0.f ? 8u : 0u) | (q.x > 0.f ? 16u : 0u) | (q.y > 0.f ? 32u : 0u) |
                         (q.z > 0.f ? 64u : 0u) | (q.w > 0.f ? 128u : 0u);
            b <<= 8 * g;
            b |= __shfl_xor_sync(0xffffffffu, b, 1);
            b |= __shfl_xor_sync(0xffffffffu, b, 2);
            bits[it] = b;                       // all 32 channels of the pixel
          }
          load(j + DEPTH, vq[d]);
          if (j >= C::RQ) mbar_wait(&qfree[slot], (uint32_t)(((j / C::RQ) - 1) & 1));
          uint8_t* sq = my + slot * C::Q_SLOT;
          *reinterpret_cast<uint4*>(sq) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(sq + 4 * C::GP) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(sq + 64 * 16) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
          *reinterpret_cast<uint4*>(sq + 4 * C::GP + 64 * 16) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
          if (g == 0) {
            smask[slot * C::M + m0] = bits[0];
            smask[slot * C::M + m0 + 64] = bits[1];
          }
          fence_proxy_async();
          mbar_arrive(&qfull[slot]);
        }
      }
    }
  } else if (warp == C::W_I) {
    // ============================ I0: d2 = d3 (*) W3 ===========================================
    const uint32_t idesc2 = make_idesc_f16(C::M, 2 * C::N), idesc1 = make_idesc_f16(C::M, C::N);
    const uint32_t sP = smem_u32(smem_raw + C::oP), sW = smem_u32(smem_raw + C::oW);
    // A: K-major, the two 8-tap chunks of a K-step are neighbouring plane entries (LBO = 16)
    auto adesc = [](uint32_t addr) -> uint64_t {
      return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(16 >> 4) << 16) |
             ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    };
    const uint64_t wdesc = (uint64_t)((sW >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) |
                           ((uint64_t)((128 * (C::KW / 8)) >> 4) << 32) | ((uint64_t)1 << 46);
    for (int j = 0; j < oh; j++) {
      const int slot = j % C::RP;
      mbar_wait(&pfull[slot], (uint32_t)((j / C::RP) & 1));
      if (j >= 2) mbar_wait(&d2_free[j & 1], (uint32_t)(((j >> 1) - 1) & 1));
      tcgen05_fence_after();
      const uint32_t ph = sP + slot * C::P_SLOT, pl = ph + C::PB;
      const uint32_t d = tmem + C::cD2 + 64u * (uint32_t)(j & 1);
      if (elect_one()) {
#pragma unroll
        for (int s = 0; s < 3; s++) {
          // first chunk = tap dx = 2 s + 1 (5 = pad for s = 2) at entry 5 - dx = 4 - 2 s
          const uint32_t off = (uint32_t)(4 - 2 * s) * 16u;
          mma_f16_ss(d, adesc(ph + off), wdesc + 16 * s, idesc2, s > 0 ? 1u : 0u);
          mma_f16_ss(d, adesc(pl + off), wdesc + 16 * s, idesc1, 1u);
        }
        mma_commit(&d2_done[j & 1]);
        mma_commit(&pfree[slot]);
      }
      __syncwarp();
    }
  } else if (warp == C::W_I + 1) {
    // ============================ I1: gW3 += d3 (x) out2 =======================================
    const uint32_t idesc2 = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)((2 * C::N) >> 3) << 17) |
                            ((uint32_t)(64 >> 4) << 24);
    const uint32_t idesc1 = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(C::N >> 3) << 17) |
                            ((uint32_t)(64 >> 4) << 24);
    const uint32_t sP = smem_u32(smem_raw + C::oP), sQ = smem_u32(smem_raw + C::oQ);
    auto desc = [](uint32_t addr, uint32_t sbo) -> uint64_t {   // MN-major: LBO = 128, SBO = group
      return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) |
             ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
    };
    const uint32_t d = tmem + C::cGW;
    for (int j = 0; j < oh; j++) {
      const int ps = j % C::RP, qs = j % C::RQ;
      mbar_wait(&pfull[ps], (uint32_t)((j / C::RP) & 1));
      mbar_wait(&qfull[qs], (uint32_t)((j / C::RQ) & 1));
      tcgen05_fence_after();
      const uint32_t ph = sP + ps * C::P_SLOT, pl = ph + C::PB, qb = sQ + qs * C::Q_SLOT;
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::M / 16; ks++) {
          const uint32_t off = (uint32_t)ks * 256u;   // 16 pixels = 16 entries of 16 bytes
          mma_f16_ss(d, desc(ph + off, 16), desc(qb + off, C::GP), idesc2, (j > 0 || ks > 0) ? 1u : 0u);
          mma_f16_ss(d, desc(pl + off, 16), desc(qb + off, C::GP), idesc1, 1u);
        }
        mma_commit(&pfree[ps]);
        mma_commit(&qfree[qs]);
        if (j == oh - 1) mma_commit(&gw_done);
      }
      __syncwarp();
    }
  } else {
    // ============================ E: d2 rows, then the gradient ================================
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    const int m = warp * 32 + lane;
    const long long vm = X0 + m;
    long long obase = -1;
    if (vm < vw) {
      const int smp = (int)(vm / ow), x = (int)(vm - (long long)smp * ow);
      obase = (((long long)smp * oh) * ow + x) * C::N;
    }
    const long long row = (long long)ow * C::N;
    const float cs = 1.f / (s_d * s_w);
    float dmax = 0.f;
    const uint32_t* smask = reinterpret_cast<const uint32_t*>(smem_raw + C::oMask);
    float* st = reinterpret_cast<float*>(smem_raw + C::oStage) + warp * (32 * C::SP);
    for (int j = 0; j < oh; j++) {
      mbar_wait(&d2_done[j & 1], (uint32_t)((j >> 1) & 1));
      tcgen05_fence_after();
      const uint32_t d = tmem + lane_base + C::cD2 + 64u * (uint32_t)(j & 1);
      float v[32], w[32];
      tmem_ld16_nowait(d, v);
      tmem_ld16_nowait(d + 16, v + 16);
      tmem_ld16_nowait(d + 32, w);
      tmem_ld16_nowait(d + 48, w + 16);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&d2_free[j & 1]);
      // ReLU' mask of this pixel's out2 row (bit n = out2[n] > 0), written by the Q producers;
      // the accumulator can only be complete after the row's planes were full
      const int qs = j % C::RQ;
      mbar_wait(&qfull[qs], (uint32_t)((j / C::RQ) & 1));   // (the d2 MMAs do not depend on Q)
      const uint32_t bits = smask[qs * C::M + m];
      mbar_arrive(&qfree[qs]);
      // stage the 32 pixels of this warp, then 8 lanes per pixel: every store instruction writes
      // four full 128-byte lines
      float4* own = reinterpret_cast<float4*>(st + lane * C::SP);
#pragma unroll
      for (int c = 0; c < 8; c++) {
        float4 r;
        r.x = (bits >> (4 * c)) & 1u ? (v[4 * c] + w[4 * c]) * cs : 0.f;
        r.y = (bits >> (4 * c + 1)) & 1u ? (v[4 * c + 1] + w[4 * c + 1]) * cs : 0.f;
        r.z = (bits >> (4 * c + 2)) & 1u ? (v[4 * c + 2] + w[4 * c + 2]) * cs : 0.f;
        r.w = (bits >> (4 * c + 3)) & 1u ? (v[4 * c + 3] + w[4 * c + 3]) * cs : 0.f;
        own[c] = r;
        dmax = fmaxf(fmaxf(dmax, fmaxf(fabsf(r.x), fabsf(r.y))), fmaxf(fabsf(r.z), fabsf(r.w)));
      }
      __syncwarp();
#pragma unroll
      for (int it = 0; it < 8; it++) {
        const int pp = it * 4 + (lane >> 3), ck = lane & 7;
        const long long ob = __shfl_sync(0xffffffffu, obase, pp);
        const float4 r = *reinterpret_cast<const float4*>(st + pp * C::SP + ck * 4);
        if (ob >= 0) *reinterpret_cast<float4*>(a.d2 + ob + j * row + ck * 4) = r;
      }
      __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = fmaxf(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    if (lane == 0 && dmax > 0.f && a.d2_max) atomicMax(a.d2_max, __float_as_uint(dmax));
    // ---- gW3: accumulator rows (g, e) = (dx = 5 - g, dy = 7 - e); an M = 64 accumulator keeps row
    // r in TMEM lane 32 (r / 16) + r % 16
    mbar_wait(&gw_done, 0);
    tcgen05_fence_after();
    {
      // (the .sync.aligned loads are warp-wide: all 32 lanes take part, lanes 0..15 hold rows)
      float v[32], w[32];
      const uint32_t d = tmem + lane_base + C::cGW;
      tmem_ld16_nowait(d, v);
      tmem_ld16_nowait(d + 16, v + 16);
      tmem_ld16_nowait(d + 32, w);
      tmem_ld16_nowait(d + 48, w + 16);
      tmem_ld_wait();
      const int r = warp * 16 + lane, g = r >> 3, e = r & 7;
      const int dx = 5 - g, dy = 7 - e;
      if (lane < 16 && dx >= 0 && dx < C::F && dy >= 0 && dy < C::F) {
        const float cg = 1.f / (s_d * s_o);
        float* dst = part + (dy * C::F + dx) * C::N;
#pragma unroll
        for (int n = 0; n < C::N; n++) dst[n] = (v[n] + w[n]) * cg;
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (tid == 0) {
    float gb = 0.f;
#pragma unroll
    for (int i = 0; i < C::N_P; i++) gb += s_gb[i];
    part[C::T * C::N] = gb;
  }
  if (warp == 0) tmem_dealloc(tmem, C::TMEM_COLS);
}

inline bool supported(int k, int f) { return k == Cfg::N && f == Cfg::F; }
constexpr int MAX_ROWS = 64;   // out2 rows per sample (see fast::backward3_tc)

// d3 + d2 + gW3/gB3 partials; returns 1 when launched (partials in ctx->splitk_scratch, *count of
// them), 0 when the shape is not handled.  `mx`: the context's maxima block; out2's maximum must
// already be in mx->out2 when `out2_max_known`, else it is measured here.
inline int bwd3_tc(srcnn_ctx* ctx, const float* gt, const float* out3, const float* out2,
                   const float* W3, float* d3, float* d2, c5::Maxes* mx, bool out2_max_known, int k,
                   int f, int gt_w, int gt_h, int w3, int h3, int S, int* count) {
  using C = Cfg;
  if (!supported(k, f)) return 0;
  const int ow = w3 + f - 1, oh = h3 + f - 1;
  const long long vw = (long long)S * ow;
  const long long strips = (vw + C::M - 1) / C::M;
  if (strips > 0x7fffffffLL) return 0;
  SRCNN_TRY(ensure_func_setup(ctx, bwd3_tc_kernel, C::SMEM_BYTES));
  if (!out2_max_known) SRCNN_TRY(c5::absmax(ctx, out2, (size_t)S * ow * oh * k, &mx->out2));
  SRCNN_CUDA(cudaMemsetAsync(&mx->d3, 0, sizeof(unsigned), ctx->stream));
  SRCNN_CUDA(cudaMemsetAsync(&mx->d2, 0, sizeof(unsigned), ctx->stream));
  const long long total = (long long)S * w3 * h3;
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 8);
  d3_kernel<<<blocks > 0 ? blocks : 1, 256, 0, ctx->stream>>>(gt, out3, d3, gt_w, gt_h, w3, h3,
                                                              total, &mx->d3);
  *count = (int)strips;
  SRCNN_TRY(ensure_scratch(ctx, &ctx->splitk_scratch, &ctx->splitk_bytes,
                           sizeof(float) * (size_t)strips * (C::T * C::N + 1)));
  Args a{d3, out2, W3, d2, (float*)ctx->splitk_scratch, &mx->d3, &mx->out2, &mx->d2, S, ow, oh};
  bwd3_tc_kernel<<<(unsigned)strips, C::NT, C::SMEM_BYTES, ctx->stream>>>(a);
  ctx->launch_count += 1;
  return 1;
}

}  // namespace b3tc
}  // namespace srcnn
