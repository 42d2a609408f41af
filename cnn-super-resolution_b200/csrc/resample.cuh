// Image enlargement by Pillow's 8-bit RGB resampling (libImaging/Resample.c, ImagingResample
// with filterscale = 1), byte for byte: Image.fromarray(rgb, "RGB").resize((W, H), BICUBIC |
// LANCZOS).  It is the step before the reference's forward flow (src/Main_cl.cpp:217-239), whose
// input image is already enlarged; the reference's sample generator enlarged with PIL's
// ANTIALIAS (Lanczos) filter.
//
//   per axis: scale = in / out; output i takes the inputs [xmin, xmin + n) around
//   center = (i + 0.5) * scale with int32 weights of 22 fraction bits; each output is
//   clamp((2^21 + sum k * p) >> 22, 0, 255).  The horizontal pass runs first and rounds to an
//   8-bit intermediate; the vertical pass reads that intermediate.
//
// The weight tables are computed on the host in double, as Pillow does (a sin() that differs
// in its last bit on the device could flip a rounding), and cached in the context.  An axis whose
// size does not change gets the identity table (one tap of weight 2^22), which reproduces
// Pillow's "not resampled" exactly.
//
// One launch does both passes: a CTA owns kTY x kTX output pixels, runs the horizontal pass for
// the input rows its vertical taps need into shared memory, then the vertical pass from there,
// and writes the enlarged RGBA8 image (alpha 255) and, when asked, its normalized luma with the
// arithmetic of extract_luma_kernel (generic::luma_of).  Alpha of the input is ignored: this is
// Pillow's "RGB" path, not its premultiplying "RGBA" one.  A set of equal-sized frames is one
// launch with the frame in blockIdx.z (frame f reads in + f * in_frame, writes out / luma + f * W * H).
#pragma once
#include <cmath>
#include <cstring>
#include <vector>

#include "context.cuh"
#include "kernels_generic.cuh"

namespace srcnn {
namespace resample {

constexpr int kPrecisionBits = 22;
constexpr int kTX = 128, kTY = 16, kThreads = 256;

inline int support_of(int filter) { return filter == SRCNN_RESAMPLE_LANCZOS ? 3 : 2; }
inline int taps_of(int filter) { return 2 * support_of(filter) + 1; }

inline double bicubic(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}
inline double sinc(double x) {
  if (x == 0.0) return 1.0;
  x = x * M_PI;
  return std::sin(x) / x;
}
inline double lanczos(double x) {
  if (-3.0 <= x && x < 3.0) return sinc(x) * sinc(x / 3);
  return 0.0;
}

// one axis: bounds[n_out], counts[n_out], weights[n_out][taps] (int32, zero-padded)
inline void axis_table(int n_in, int n_out, int filter, std::vector<int>& t) {
  const int taps = taps_of(filter);
  const size_t base = t.size();
  t.resize(base + (size_t)n_out * (2 + taps), 0);
  int* bounds = t.data() + base;
  int* counts = bounds + n_out;
  int* w = counts + n_out;
  if (n_in == n_out) {   // not resampled
    for (int i = 0; i < n_out; i++) {
      bounds[i] = i;
      counts[i] = 1;
      w[(size_t)i * taps] = 1 << kPrecisionBits;
    }
    return;
  }
  const double support = support_of(filter), scale = (double)n_in / n_out;
  std::vector<double> k((size_t)taps);
  for (int i = 0; i < n_out; i++) {
    const double center = (i + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > n_in) xmax = n_in;
    const int n = xmax - xmin;
    double ww = 0.0;
    for (int j = 0; j < n; j++) {
      const double x = j + xmin - center + 0.5;
      k[j] = filter == SRCNN_RESAMPLE_LANCZOS ? lanczos(x) : bicubic(x);
      ww += k[j];
    }
    for (int j = 0; j < n; j++) {
      const double v = ww != 0.0 ? k[j] / ww : k[j];
      w[(size_t)i * taps + j] = v < 0 ? (int)(-0.5 + v * (1 << kPrecisionBits))
                                      : (int)(0.5 + v * (1 << kPrecisionBits));
    }
    bounds[i] = xmin;
    counts[i] = n;
  }
}

// the host tables of (w, h) -> (W, H): horizontal axis first, then vertical, plus the most
// input rows one CTA's vertical taps span
inline std::vector<int> tables(int w, int h, int W, int H, int filter, int* rows_max) {
  std::vector<int> t;
  axis_table(w, W, filter, t);
  axis_table(h, H, filter, t);
  const int* yb = t.data() + (size_t)W * (2 + taps_of(filter));
  const int* yn = yb + H;
  int m = 0;
  for (int y0 = 0; y0 < H; y0 += kTY) {
    const int y1 = std::min(y0 + kTY, H) - 1;
    m = std::max(m, yb[y1] + yn[y1] - yb[y0]);
  }
  *rows_max = m;
  return t;
}

template <int TAPS>
__global__ void __launch_bounds__(kThreads)
resample_kernel(const uchar4* __restrict__ in, int w, size_t in_frame, uchar4* __restrict__ out,
                float* __restrict__ luma, int W, int H, const int* __restrict__ tab) {
  extern __shared__ uchar4 mid[];   // [rows][kTX] horizontal-pass result, 8-bit
  in += blockIdx.z * in_frame;
  out += blockIdx.z * (size_t)W * H;
  if (luma) luma += blockIdx.z * (size_t)W * H;
  const int* xb = tab;
  const int* xn = xb + W;
  const int* xk = xn + W;
  const int* yb = tab + (size_t)W * (2 + TAPS);
  const int* yn = yb + H;
  const int* yk = yn + H;
  const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * kTY;
  const int ylast = min(y0 + kTY, H) - 1;
  const int row0 = __ldg(yb + y0);
  const int rows = __ldg(yb + ylast) + __ldg(yn + ylast) - row0;
  const int nx = min(kTX, W - x0);
  // horizontal pass: input rows [row0, row0 + rows) x output columns [x0, x0 + nx)
  for (int i = threadIdx.x; i < rows * kTX; i += kThreads) {
    const int r = i / kTX, c = i - r * kTX;
    if (c >= nx) continue;
    const int x = x0 + c;
    const int b = __ldg(xb + x), n = __ldg(xn + x);
    const uchar4* src = in + (size_t)(row0 + r) * w + b;
    int s0 = 1 << (kPrecisionBits - 1), s1 = s0, s2 = s0;
#pragma unroll
    for (int j = 0; j < TAPS; j++) {
      if (j < n) {
        const uchar4 p = src[j];
        const int k = __ldg(xk + (size_t)x * TAPS + j);
        s0 += (int)p.x * k;
        s1 += (int)p.y * k;
        s2 += (int)p.z * k;
      }
    }
    mid[i] = make_uchar4((unsigned char)min(max(s0 >> kPrecisionBits, 0), 255),
                         (unsigned char)min(max(s1 >> kPrecisionBits, 0), 255),
                         (unsigned char)min(max(s2 >> kPrecisionBits, 0), 255), 255);
  }
  __syncthreads();
  // vertical pass from shared memory
  const int ny = ylast - y0 + 1;
  for (int i = threadIdx.x; i < ny * kTX; i += kThreads) {
    const int r = i / kTX, c = i - r * kTX;
    if (c >= nx) continue;
    const int y = y0 + r, x = x0 + c;
    const int b = __ldg(yb + y) - row0, n = __ldg(yn + y);
    int s0 = 1 << (kPrecisionBits - 1), s1 = s0, s2 = s0;
#pragma unroll
    for (int j = 0; j < TAPS; j++) {
      if (j < n) {
        const uchar4 p = mid[(b + j) * kTX + c];
        const int k = __ldg(yk + (size_t)y * TAPS + j);
        s0 += (int)p.x * k;
        s1 += (int)p.y * k;
        s2 += (int)p.z * k;
      }
    }
    const uchar4 o = make_uchar4((unsigned char)min(max(s0 >> kPrecisionBits, 0), 255),
                                 (unsigned char)min(max(s1 >> kPrecisionBits, 0), 255),
                                 (unsigned char)min(max(s2 >> kPrecisionBits, 0), 255), 255);
    const size_t o_i = (size_t)y * W + x;
    out[o_i] = o;
    if (luma) luma[o_i] = generic::luma_of(o, 1);
  }
}

// the cached device tables of one shape and filter (uploaded on the context stream)
inline int table_for(srcnn_ctx* ctx, int w, int h, int W, int H, int filter, const int** dev,
                     int* rows_max) {
  const srcnn_ctx::ResampleKey key{w, h, W, H, filter};
  for (const srcnn_ctx::ResampleTable& t : ctx->resample_tables)
    if (std::memcmp(&t.key, &key, sizeof(key)) == 0) {
      *dev = t.dev;
      *rows_max = t.rows_max;
      return SRCNN_OK;
    }
  srcnn_ctx::ResampleTable t;
  t.key = key;
  t.host = tables(w, h, W, H, filter, &t.rows_max);
  void* p = nullptr;
  if (cudaMalloc(&p, t.host.size() * sizeof(int)) != cudaSuccess) {
    cudaGetLastError();
    return fail(SRCNN_ENOMEM, "resample table allocation failed");
  }
  t.dev = static_cast<int*>(p);
  // the host copy lives as long as the context, so the asynchronous copy may read it late
  ctx->resample_tables.push_back(std::move(t));
  srcnn_ctx::ResampleTable& s = ctx->resample_tables.back();
  SRCNN_CUDA(cudaMemcpyAsync(s.dev, s.host.data(), s.host.size() * sizeof(int),
                             cudaMemcpyHostToDevice, ctx->stream));
  *dev = s.dev;
  *rows_max = s.rows_max;
  return SRCNN_OK;
}

// `frames` frames of w x h (in) -> W x H (out, luma), back to back
inline int launch(srcnn_ctx* ctx, const uchar4* in, int w, int h, uchar4* out, float* luma, int W,
                  int H, int filter, const int* tab, int rows_max, int frames = 1) {
  const dim3 grid((unsigned)((W + kTX - 1) / kTX), (unsigned)((H + kTY - 1) / kTY), (unsigned)frames);
  const size_t in_frame = (size_t)w * h;
  const size_t smem = (size_t)rows_max * kTX * sizeof(uchar4);
  // at most (kTY - 1) + 2 * 3 + 1 rows for an enlargement: well under the default 48 KB
  if (filter == SRCNN_RESAMPLE_LANCZOS)
    resample_kernel<7><<<grid, kThreads, smem, ctx->stream>>>(in, w, in_frame, out, luma, W, H, tab);
  else
    resample_kernel<5><<<grid, kThreads, smem, ctx->stream>>>(in, w, in_frame, out, luma, W, H, tab);
  return SRCNN_OK;
}

}  // namespace resample
}  // namespace srcnn
