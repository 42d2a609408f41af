// Any-shape FP32 SIMT kernels: correct for every (k, n, f) the reference accepts.  The
// specialised fast paths for the SRCNN shapes live in kernels_fast.cuh; these are what runs
// for the reference's own small test shapes (k1n3f3, k3n2f3, k3n3f1, ...).
//
// forward / deltas / backpropagate are all one contraction
//     C[M][N] = sum_K A[M][K] * B[K][N]
// with a gathered A operand, so they share one 64x64x16 register-tiled SIMT GEMM core
// (256 threads, 4x4 outputs per thread, operands staged through shared memory):
//   forward       M = pixels,        K = f*f*k (taps x in-channels), N = n     (implicit GEMM)
//   deltas        M = pixels,        K = f*f*n_next,                 N = n_curr (flipped taps,
//                                                                    zero outside d_next)
//   backpropagate M = f*f*k (+1 row of ones -> bias gradient), K = pixels of all samples,
//                 N = n; split-K over pixel ranges with a fixed-order second stage, so the
//                 result is deterministic (the reference races, backpropagate.cl:110).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace srcnn {
namespace generic {

constexpr int TM = 64, TN = 64, KC = 16, NT = 256;
constexpr int LDS_PAD = 4;

// acc[i][j] += As[kk][ty*4+i] * Bs[kk][tx*4+j]
__device__ __forceinline__ void tile_fma(const float (*As)[TM + LDS_PAD],
                                         const float (*Bs)[TN + LDS_PAD], int tx, int ty,
                                         float acc[4][4]) {
#pragma unroll
  for (int kk = 0; kk < KC; kk++) {
    const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
    const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
    const float av[4] = {a.x, a.y, a.z, a.w};
    const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }
}

// ------------------------------------------------------------------ forward ----------
// reference: src/kernel/layer_uber_kernel.cl:36-96
struct FwdArgs {
  const float* in;
  float* out;
  const float* W;
  const float* B;
  int k, n, f, relu, in_w, in_h, ow, oh, S;
};

__global__ void __launch_bounds__(NT) forward_gemm_kernel(FwdArgs a) {
  __shared__ __align__(16) float As[KC][TM + LDS_PAD];
  __shared__ __align__(16) float Bs[KC][TN + LDS_PAD];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const long long M = (long long)a.S * a.ow * a.oh;
  const int K = a.f * a.f * a.k;
  const long long m0 = (long long)blockIdx.x * TM;
  const int n0 = blockIdx.y * TN;

  // A-tile element e = tid + i*256 -> (kk = e % 16, mm = e / 16): mm is fixed per (thread,i)
  long long a_base[4];
  bool a_ok[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int mm = (tid + i * NT) / KC;
    const long long p = m0 + mm;
    a_ok[i] = p < M;
    long long s = 0, y = 0, x = 0;
    if (a_ok[i]) {
      s = p / ((long long)a.ow * a.oh);
      const long long r = p - s * a.ow * a.oh;
      y = r / a.ow;
      x = r - y * a.ow;
    }
    a_base[i] = ((s * a.in_h + y) * a.in_w + x) * a.k;
  }
  const int a_kk = tid % KC;

  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += KC) {
    // A: gathered input window
    const int kap = k0 + a_kk;
    int off = 0;
    const bool k_ok = kap < K;
    if (k_ok) {
      const int tap = kap / a.k, kk = kap - tap * a.k;
      const int dy = tap / a.f, dx = tap - dy * a.f;
      off = (dy * a.in_w + dx) * a.k + kk;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int mm = (tid + i * NT) / KC;
      As[a_kk][mm] = (k_ok && a_ok[i]) ? __ldg(a.in + a_base[i] + off) : 0.f;
    }
    // B: weights [kap][n], n contiguous.  e -> (nn = e % 64, kk = e / 64)
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int e = tid + i * NT;
      const int nn = e % TN, kk = e / TN;
      const int kq = k0 + kk, c = n0 + nn;
      Bs[kk][nn] = (kq < K && c < a.n) ? __ldg(a.W + (long long)kq * a.n + c) : 0.f;
    }
    __syncthreads();
    tile_fma(As, Bs, tx, ty, acc);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const long long p = m0 + ty * 4 + i;
    if (p >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = n0 + tx * 4 + j;
      if (c >= a.n) continue;
      float r = acc[i][j] + __ldg(a.B + c);
      if (a.relu) r = fmaxf(r, 0.f);
      a.out[p * a.n + c] = r;
    }
  }
}

// ------------------------------------------------------------------ deltas -----------
// reference: src/kernel/layer_deltas.cl:42-127
struct DeltaArgs {
  const float* dn;   // deltas of layer l      [S][nh][nw][n_next]
  const float* lo;   // output of layer l-1    [S][oh][ow][n_curr]
  float* target;     // deltas of layer l-1    [S][oh][ow][n_curr]
  const float* W;    // weights of layer l     [f][f][n_curr][n_next]
  int n_curr, f, n_next, ow, oh, nw, nh, S;
};

__global__ void __launch_bounds__(NT) deltas_gemm_kernel(DeltaArgs a) {
  __shared__ __align__(16) float As[KC][TM + LDS_PAD];
  __shared__ __align__(16) float Bs[KC][TN + LDS_PAD];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const long long M = (long long)a.S * a.ow * a.oh;
  const int K = a.f * a.f * a.n_next;
  const long long m0 = (long long)blockIdx.x * TM;
  const int n0 = blockIdx.y * TN;

  int ps[4], pj[4], pi[4];
  bool a_ok[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int mm = (tid + i * NT) / KC;
    const long long p = m0 + mm;
    a_ok[i] = p < M;
    ps[i] = pj[i] = pi[i] = 0;
    if (a_ok[i]) {
      const long long s = p / ((long long)a.ow * a.oh);
      const long long r = p - s * a.ow * a.oh;
      ps[i] = (int)s;
      pj[i] = (int)(r / a.ow);
      pi[i] = (int)(r - (long long)pj[i] * a.ow);
    }
  }
  const int a_kk = tid % KC;

  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += KC) {
    const int kap = k0 + a_kk;
    const bool k_ok = kap < K;
    int dy = 0, dx = 0, kk = 0;
    if (k_ok) {
      const int tap = kap / a.n_next;
      kk = kap - tap * a.n_next;
      dy = tap / a.f;
      dx = tap - dy * a.f;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int mm = (tid + i * NT) / KC;
      const int nj = pj[i] - dy, ni = pi[i] - dx;
      const bool ok = k_ok && a_ok[i] && nj >= 0 && nj < a.nh && ni >= 0 && ni < a.nw;
      As[a_kk][mm] =
          ok ? __ldg(a.dn + (((long long)ps[i] * a.nh + nj) * a.nw + ni) * a.n_next + kk) : 0.f;
    }
    // B[kap][n] = W[tap][n][k]  (k fastest in memory): e -> (kk = e % 16, nn = e / 16)
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int e = tid + i * NT;
      const int bk = e % KC, nn = e / KC;
      const int kq = k0 + bk, c = n0 + nn;
      float v = 0.f;
      if (kq < K && c < a.n_curr) {
        const int tap = kq / a.n_next, k2 = kq - tap * a.n_next;
        v = __ldg(a.W + ((long long)tap * a.n_curr + c) * a.n_next + k2);
      }
      Bs[bk][nn] = v;
    }
    __syncthreads();
    tile_fma(As, Bs, tx, ty, acc);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const long long p = m0 + ty * 4 + i;
    if (p >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = n0 + tx * 4 + j;
      if (c >= a.n_curr) continue;
      const float y = __ldg(a.lo + p * a.n_curr + c);
      a.target[p * a.n_curr + c] = y > 0.f ? acc[i][j] : 0.f;
    }
  }
}

// ------------------------------------------------------------------ backpropagate ----
// reference: src/kernel/backpropagate.cl:56-114
struct BpArgs {
  const float* d;    // deltas       [S][oh][ow][n]
  const float* in;   // layer input  [S][ih][iw][k]
  float* partial;    // [splits][M+1][n]
  int n, k, f, ow, oh, iw, ih, S;
  long long pix_per_split;
};

__global__ void __launch_bounds__(NT) backprop_gemm_kernel(BpArgs a) {
  __shared__ __align__(16) float As[KC][TM + LDS_PAD];  // As[pixel][m]
  __shared__ __align__(16) float Bs[KC][TN + LDS_PAD];  // Bs[pixel][n]
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int Mw = a.f * a.f * a.k;  // weight rows; row Mw = ones (bias gradient)
  const int M = Mw + 1;
  const long long P = (long long)a.S * a.ow * a.oh;
  const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
  const long long p_begin = (long long)blockIdx.z * a.pix_per_split;
  long long p_end = p_begin + a.pix_per_split;
  if (p_end > P) p_end = P;

  // A-tile element e -> (mm = e % 64, pp = e / 64): mm fixed per thread
  const int a_mm = tid % TM;
  const int m = m0 + a_mm;
  int a_off = 0;
  if (m < Mw) {
    const int tap = m / a.k, kk = m - tap * a.k;
    const int dy = tap / a.f, dx = tap - dy * a.f;
    a_off = (dy * a.iw + dx) * a.k + kk;
  }

  float acc[4][4] = {};
  for (long long p0 = p_begin; p0 < p_end; p0 += KC) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int pp = tid / TM + i * (NT / TM);
      const long long p = p0 + pp;
      float v = 0.f;
      if (p < p_end && m < M) {
        if (m == Mw) {
          v = 1.f;
        } else {
          const long long s = p / ((long long)a.ow * a.oh);
          const long long r = p - s * a.ow * a.oh;
          const long long y = r / a.ow, x = r - y * a.ow;
          v = __ldg(a.in + ((s * a.ih + y) * a.iw + x) * a.k + a_off);
        }
      }
      As[pp][a_mm] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int e = tid + i * NT;
      const int nn = e % TN, pp = e / TN;
      const long long p = p0 + pp;
      const int c = n0 + nn;
      Bs[pp][nn] = (p < p_end && c < a.n) ? __ldg(a.d + p * a.n + c) : 0.f;
    }
    __syncthreads();
    tile_fma(As, Bs, tx, ty, acc);
    __syncthreads();
  }
  float* dst = a.partial + (long long)blockIdx.z * M * a.n;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int mm = m0 + ty * 4 + i;
    if (mm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = n0 + tx * 4 + j;
      if (c < a.n) dst[(long long)mm * a.n + c] = acc[i][j];
    }
  }
}

// second stage: fixed-order sum over the splits, then `+=` into the accumulators
__global__ void backprop_reduce_kernel(const float* __restrict__ partial, float* grad_w,
                                       float* grad_b, int Mw, int n, int splits) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  const int total = (Mw + 1) * n;
  if (id >= total) return;
  float s = 0.f;
  for (int z = 0; z < splits; z++) s += partial[(long long)z * total + id];
  if (id < Mw * n)
    grad_w[id] += s;
  else
    grad_b[id - Mw * n] += s;
}

// ------------------------------------------------------------------ element-wise -----
// reference: src/kernel/last_layer_delta.cl:14-50
__global__ void last_layer_delta_kernel(const float* __restrict__ gt, const float* __restrict__ algo,
                                        float* __restrict__ target, int gt_w, int gt_h, int aw,
                                        int ah, int S) {
  const long long total = (long long)S * aw * ah;
  const int pad = (gt_w - aw) / 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long s = i / ((long long)aw * ah);
    const long long r = i - s * aw * ah;
    const int y = (int)(r / aw), x = (int)(r - (long long)y * aw);
    const float t = __ldg(gt + (s * gt_h + y + pad) * gt_w + pad + x);
    const float v = __ldg(algo + i);
    target[i] = v > 0.f ? v - t : 0.f;
  }
}

// reference: src/kernel/subtract_from_all.cl:1-8
__global__ void sub_from_all_kernel(float* data, float value, unsigned len) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < len;
       i += (size_t)gridDim.x * blockDim.x)
    data[i] = data[i] - value;
}

// sub_from_all_kernel with value = *sum / (float)len read on the device (the mean never goes
// through the host): the same float division and subtraction as the host route.  Frame
// blockIdx.y: data + blockIdx.y * len, its own sum[blockIdx.y].
__global__ void sub_mean_kernel(float* data, const float* __restrict__ sum, unsigned len) {
  data += blockIdx.y * (size_t)len;
  const float value = __fdiv_rn(sum[blockIdx.y], (float)len);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < len;
       i += (size_t)gridDim.x * blockDim.x)
    data[i] = data[i] - value;
}

__global__ void fill_kernel(float* data, float value, size_t len) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < len;
       i += (size_t)gridDim.x * blockDim.x)
    data[i] = value;
}

// reference: src/kernel/update_parameters.cl:1-33
__global__ void update_params_kernel(float* w, float* b, const float* __restrict__ gw,
                                     const float* __restrict__ gb, float* pdw, float* pdb,
                                     float momentum, float decay, float lr, unsigned batch,
                                     unsigned wsize, unsigned bsize) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  const float fb = (float)batch;
  if (i < wsize) {
    const float wv = w[i];
    const float dw = momentum * pdw[i] + lr * gw[i] + decay * wv;
    w[i] = wv - dw / fb;
    pdw[i] = dw;
  }
  if (i < bsize) {
    const float db = momentum * pdb[i] + lr * gb[i];
    b[i] -= db / fb;
    pdb[i] = db;
  }
}

// ------------------------------------------------------------------ reductions -------
// Deterministic two-stage sums in double (the oracle's definition: double sum of float32
// terms).  Stage 1: fixed grid, fixed per-thread element assignment, fixed-order tree;
// stage 2: one block folds the partials in index order.  Several equal-length arrays at once:
// stage 1 takes array blockIdx.y (data + blockIdx.y * len, partials blockIdx.y * gridDim.x on),
// stage 2 one block per array (partials blockIdx.x * count on, target[blockIdx.x]); each sum is
// the one a single-array launch gives.
constexpr int RED_THREADS = 256;
constexpr int RED_MAX_BLOCKS = 1024;

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  double r = 0.0;
  if (warp == 0) {
    r = lane < (int)(blockDim.x >> 5) ? sh[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
  }
  return r;  // valid in thread 0
}

// reference: src/kernel/squared_error.cl:36-92
__global__ void __launch_bounds__(RED_THREADS)
squared_error_stage1(const float* __restrict__ gt, const float* __restrict__ algo,
                     double* __restrict__ partial, int gt_w, int gt_h, int aw, int ah, int S) {
  __shared__ double sh[32];
  const long long total = (long long)S * aw * ah;
  const int pad = (gt_w - aw) / 2;
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long s = i / ((long long)aw * ah);
    const long long r = i - s * aw * ah;
    const int y = (int)(r / aw), x = (int)(r - (long long)y * aw);
    const float t = __ldg(gt + (s * gt_h + y + pad) * gt_w + pad + x);
    const float d = __ldg(algo + i) - t;
    acc += (double)(d * d);
  }
  const double r = block_sum(acc, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = r;
}

// reference: src/kernel/sum.cl:35-68
__global__ void __launch_bounds__(RED_THREADS)
sum_stage1(const float* __restrict__ data, double* __restrict__ partial, unsigned len,
           int squared) {
  __shared__ double sh[32];
  data += blockIdx.y * (size_t)len;
  partial += blockIdx.y * gridDim.x;
  double acc = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < len;
       i += (size_t)gridDim.x * blockDim.x) {
    float v = __ldg(data + i);
    if (squared) v = v * v;
    acc += (double)v;
  }
  const double r = block_sum(acc, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = r;
}

__global__ void __launch_bounds__(RED_THREADS)
reduce_stage2(const double* __restrict__ partial, int count, float* __restrict__ target) {
  __shared__ double sh[32];
  partial += blockIdx.x * (size_t)count;
  double acc = 0.0;
  for (int i = threadIdx.x; i < count; i += blockDim.x) acc += partial[i];
  const double r = block_sum(acc, sh);
  if (threadIdx.x == 0) target[blockIdx.x] = (float)r;
}

// batched sample gather: block (x, y) copies a slice of source y into slot y of dst
__global__ void gather_kernel(const float* const* __restrict__ src, float* __restrict__ dst,
                              size_t floats_each) {
  const float* s = src[blockIdx.y];
  float* d = dst + (size_t)blockIdx.y * floats_each;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < floats_each;
       i += (size_t)gridDim.x * blockDim.x)
    d[i] = __ldg(s + i);
}

// ------------------------------------------------------------------ luma -------------
// reference: src/kernel/extract_luma.cl:7-23
// the luma of one RGBA8 pixel; every kernel that produces luma from pixels calls this
__device__ __forceinline__ float luma_of(uchar4 p, int normalize) {
  // explicit round-to-nearest mul/add (never contracted to FMA) in the order of the
  // oracle's dot(): ((R*.299 + G*.587) + B*.114) + A*0
  float y = __fadd_rn(__fmul_rn((float)p.x, 0.299f), __fmul_rn((float)p.y, 0.587f));
  y = __fadd_rn(y, __fmul_rn((float)p.z, 0.114f));
  return normalize ? __fdiv_rn(y, 255.0f) : y;
}

__global__ void extract_luma_kernel(const uchar4* __restrict__ rgba, float* __restrict__ target,
                                    int count, int normalize) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  target[i] = luma_of(rgba[i], normalize);
}

// reference: src/kernel/swap_luma.cl:18-69.  Image rows [row0, row1) (the whole image is
// [0, gt_h)); the grid covers row1 - row0 rows.  Frame blockIdx.z of a set of gt_w x gt_h
// frames (rgba, target) and luma_w x luma_h results (luma), back to back.
__global__ void swap_luma_kernel(const uchar4* __restrict__ rgba, const float* __restrict__ luma,
                                 unsigned char* __restrict__ target, int gt_w, int gt_h, int row0,
                                 int row1, int luma_w, int luma_h) {
  rgba += blockIdx.z * (size_t)gt_w * gt_h;
  target += blockIdx.z * (size_t)gt_w * gt_h * 3;
  luma += blockIdx.z * (size_t)luma_w * luma_h;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = row0 + blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= gt_w || y >= row1) return;
  const int pad = (gt_w - luma_w) / 2;
  const size_t i = (size_t)y * gt_w + x;
  const uchar4 p = rgba[i];
  const int lx = x - pad, ly = y - pad;
  unsigned char o0 = p.x, o1 = p.y, o2 = p.z;
  if (lx >= 0 && lx < luma_w && ly >= 0 && ly < luma_h) {
    const float r = (float)p.x, g = (float)p.y, b = (float)p.z;
    // un-contracted arithmetic in the oracle's order so the 8-bit result is bit-exact
    const float Y = __fmul_rn(luma[(size_t)ly * luma_w + lx], 255.0f);
    const float Cb = __fadd_rn(__fadd_rn(__fmul_rn(r, -0.1687f), __fmul_rn(g, -0.3312f)),
                               __fmul_rn(b, 0.5f));
    const float Cr = __fadd_rn(__fadd_rn(__fmul_rn(r, 0.5f), __fmul_rn(g, -0.4186f)),
                               __fmul_rn(b, -0.0813f));
    const float R = fminf(fmaxf(__fadd_rn(Y, __fmul_rn(Cr, 1.4f)), 0.f), 255.f);
    const float G = fminf(
        fmaxf(__fadd_rn(__fadd_rn(Y, __fmul_rn(Cb, -0.343f)), __fmul_rn(Cr, -0.711f)), 0.f),
        255.f);
    const float Bv = fminf(fmaxf(__fadd_rn(Y, __fmul_rn(Cb, 1.765f)), 0.f), 255.f);
    o0 = (unsigned char)(unsigned int)R;
    o1 = (unsigned char)(unsigned int)G;
    o2 = (unsigned char)(unsigned int)Bv;
  }
  target[3 * i + 0] = o0;
  target[3 * i + 1] = o1;
  target[3 * i + 2] = o2;
}

// swap_luma_kernel for the Y plane of Y'CbCr 4:2:0 frames: the network's luma becomes the byte
// swap_luma_kernel writes for a pixel with zero chroma, clamp(luma * 255) truncated.  The grid
// covers the luma_w x luma_h interior, written (gt_w - luma_w) / 2 pixels in from the left and top
// edges of the gt_w-wide plane, whose rows are `pitch` bytes apart; the border keeps the enlarged
// Y.  Frame blockIdx.z: target + blockIdx.z * frame_bytes, luma + blockIdx.z * luma_w * luma_h.
// 10-bit planes (T = unsigned short, MAX = 1023) take the same rule with 1023 for 255, the value
// written at bit SHIFT of its word (I010: 0, P010: 6).
template <class T, int MAX, int SHIFT>
__global__ void swap_luma_plane_kernel(const float* __restrict__ luma,
                                       unsigned char* __restrict__ target, int gt_w, size_t pitch,
                                       size_t frame_bytes, int luma_w, int luma_h) {
  luma += blockIdx.z * (size_t)luma_w * luma_h;
  target += blockIdx.z * frame_bytes;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= luma_w || y >= luma_h) return;
  const int pad = (gt_w - luma_w) / 2;
  const float Y = __fmul_rn(luma[(size_t)y * luma_w + x], (float)MAX);
  *reinterpret_cast<T*>(target + (size_t)(y + pad) * pitch + x * sizeof(T) + pad * sizeof(T)) =
      (T)((unsigned int)fminf(fmaxf(Y, 0.f), (float)MAX) << SHIFT);
}

}  // namespace generic
}  // namespace srcnn
