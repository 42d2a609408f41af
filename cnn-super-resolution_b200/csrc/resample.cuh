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
// The same kernel with one byte a pixel enlarges the planes of Y'CbCr 4:2:0 frames: Pillow's "L"
// path, and for the Y plane the luma Y' / 255; with two bytes a pixel NV12's interleaved CbCr plane,
// each byte as its own "L" plane.  Plane rows may be pitched (the luma stays dense).
//
// Chroma siting lives in the tables alone.  Pillow maps pixel centres onto pixel centres, which is
// right for centre-sited ("jpeg") chroma.  A chroma sample that sits at s (in chroma samples; 0.5
// centred, 0.25 co-sited with the even luma column or row) is a shift of the sample centres on that
// axis: the table of an axis from n_in samples sited at s_in to n_out sited at s_out is Pillow's
// with a box that starts at
//   in0 = (s_out - 0.5) * scale + (0.5 - s_in),  center = in0 + (i + 0.5) * scale,
// which is exactly 0.0 for centre to centre (Pillow's plain enlargement, bit for bit); an axis of
// ratio 1 whose in0 is not 0.0 is resampled, as Pillow resamples a box with a non-zero start.
//
// 10-bit planes (I010 and P010 frames: a 16-bit word a sample, the value v in [0, 1023]) take
// Pillow's 16-bit path ("I;16") on v: the same coefficients kept as doubles, each output the sum of
// v * k in double in tap order (no fused multiply-add), rounded half away from zero and clipped to
// [0, 65535], the horizontal pass into a 16-bit intermediate; only the final output is capped at
// 1023.  The kernel is the same template with `unsigned short` / `ushort2` pixels and a Words10
// load and store policy; the 8-bit instantiations are unchanged.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstring>
#include <type_traits>
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

// the offset of a siting inside its 2x2 luma cell, in chroma samples, per axis
inline double siting_x(int siting) { return siting == SRCNN_CHROMA_CENTER ? 0.5 : 0.25; }
inline double siting_y(int siting) { return siting == SRCNN_CHROMA_TOPLEFT ? 0.25 : 0.5; }
// the box start of an axis from n_in samples sited at s_in to n_out sited at s_out
inline double box_start(int n_in, int n_out, double s_in, double s_out) {
  const double scale = (double)n_in / n_out;
  return (s_out - 0.5) * scale + (0.5 - s_in);
}

// one axis from a box starting at in0: bounds[n_out], counts[n_out] (int32), then the weights
// [n_out][taps], zero-padded.  The coefficients are computed once in double; 8-bit tables hold them
// quantised as Pillow's 8-bit path does (int32, kPrecisionBits fraction bits), 10-bit ones
// (`exact`) hold the doubles themselves, as Pillow's 16-bit path uses them, two int32 words each
// (8-byte aligned when t's size and storage are)
inline void axis_table(int n_in, int n_out, int filter, double in0, bool exact, std::vector<int>& t) {
  const int taps = taps_of(filter), words = exact ? 2 : 1;
  const size_t base = t.size();
  t.resize(base + (size_t)n_out * (2 + words * taps), 0);
  int* bounds = t.data() + base;
  int* counts = bounds + n_out;
  int* w = counts + n_out;
  const auto put = [&](int i, int j, double v) {   // weight j of output i
    if (exact)
      std::memcpy(w + ((size_t)i * taps + j) * 2, &v, sizeof(v));
    else
      w[(size_t)i * taps + j] = v < 0 ? (int)(-0.5 + v * (1 << kPrecisionBits))
                                      : (int)(0.5 + v * (1 << kPrecisionBits));
  };
  if (n_in == n_out && in0 == 0.0) {   // not resampled
    for (int i = 0; i < n_out; i++) {
      bounds[i] = i;
      counts[i] = 1;
      put(i, 0, 1.0);
    }
    return;
  }
  const double support = support_of(filter), scale = (double)n_in / n_out;
  std::vector<double> k((size_t)taps);
  for (int i = 0; i < n_out; i++) {
    const double center = in0 + (i + 0.5) * scale;
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
    for (int j = 0; j < n; j++) put(i, j, ww != 0.0 ? k[j] / ww : k[j]);
    bounds[i] = xmin;
    counts[i] = n;
  }
}

// the host tables of (w, h) -> (W, H) with box starts x0 and y0: horizontal axis first, then
// vertical, plus the most input rows one CTA's vertical taps span
inline std::vector<int> tables(int w, int h, int W, int H, int filter, double x0, double y0,
                               bool exact, int* rows_max) {
  std::vector<int> t;
  axis_table(w, W, filter, x0, exact, t);
  axis_table(h, H, filter, y0, exact, t);
  const int* yb = t.data() + (size_t)W * (2 + (exact ? 2 : 1) * taps_of(filter));
  const int* yn = yb + H;
  int m = 0;
  for (int y0 = 0; y0 < H; y0 += kTY) {
    const int y1 = std::min(y0 + kTY, H) - 1;
    m = std::max(m, yb[y1] + yn[y1] - yb[y0]);
  }
  *rows_max = m;
  return t;
}

// one plane of a launch: frame f reads in + f * in_frame and writes out + f * out_frame (pixels),
// rows in_pitch and out_pitch pixels apart, and, with luma, the dense luma + f * W * H;
// tab = table_for(w, h, W, H, ...)
template <class Pix>
struct Plane {
  const Pix* in;
  int in_pitch;
  size_t in_frame;
  Pix* out;
  int out_pitch;
  size_t out_frame;
  float* luma;
  int W, H;
  const int* tab;
};
// up to three planes of every frame in one launch: blockIdx.z = frame * n + plane; a CTA past the
// edge of its (smaller) plane returns at once
template <class Pix>
struct Planes {
  Plane<Pix> p[3];
  int n;
};

// the per-tap sum of one output pixel: three channels of RGBA8 (alpha written as 255), or one
__device__ __forceinline__ unsigned char clip8(int s) {
  return (unsigned char)min(max(s >> kPrecisionBits, 0), 255);
}
template <class Pix>
struct Acc;
template <>
struct Acc<uchar4> {
  using Weight = int;
  int s0 = 1 << (kPrecisionBits - 1), s1 = s0, s2 = s0;
  __device__ __forceinline__ void add(uchar4 p, int k) {
    s0 += (int)p.x * k;
    s1 += (int)p.y * k;
    s2 += (int)p.z * k;
  }
  __device__ __forceinline__ uchar4 pixel() const {
    return make_uchar4(clip8(s0), clip8(s1), clip8(s2), 255);
  }
};
template <>
struct Acc<unsigned char> {
  using Weight = int;
  int s = 1 << (kPrecisionBits - 1);
  __device__ __forceinline__ void add(unsigned char p, int k) { s += (int)p * k; }
  __device__ __forceinline__ unsigned char pixel() const { return clip8(s); }
};
// two interleaved planes (NV12's CbCr): Acc<unsigned char> on each
template <>
struct Acc<uchar2> {
  using Weight = int;
  int s0 = 1 << (kPrecisionBits - 1), s1 = s0;
  __device__ __forceinline__ void add(uchar2 p, int k) {
    s0 += (int)p.x * k;
    s1 += (int)p.y * k;
  }
  __device__ __forceinline__ uchar2 pixel() const { return make_uchar2(clip8(s0), clip8(s1)); }
};
// Pillow's 16-bit arithmetic ("I;16") on one 10-bit sample a plane (the Y, Cb and Cr planes of
// I010 and P010 frames) or two (P010's interleaved CbCr): double weights, the sum of the taps in
// double in tap order with no fused multiply-add, rounded half away from zero and clipped to
// [0, 65535] -- the 16-bit intermediate of the horizontal pass
__device__ __forceinline__ double tap16(double s, unsigned short p, double k) {
  return __dadd_rn(s, __dmul_rn((double)p, k));
}
__device__ __forceinline__ unsigned short clip16(double s) {
  const int r = (int)(s >= 0.0 ? __dadd_rn(s, 0.5) : __dadd_rn(s, -0.5));
  return (unsigned short)min(max(r, 0), 65535);
}
template <>
struct Acc<unsigned short> {
  using Weight = double;
  double s = 0.0;
  __device__ __forceinline__ void add(unsigned short p, double k) { s = tap16(s, p, k); }
  __device__ __forceinline__ unsigned short pixel() const { return clip16(s); }
};
template <>
struct Acc<ushort2> {
  using Weight = double;
  double s0 = 0.0, s1 = 0.0;
  __device__ __forceinline__ void add(ushort2 p, double k) {
    s0 = tap16(s0, p.x, k);
    s1 = tap16(s1, p.y, k);
  }
  __device__ __forceinline__ ushort2 pixel() const { return make_ushort2(clip16(s0), clip16(s1)); }
};

// How a plane stores its samples.  8-bit samples are the bytes themselves.
struct Bytes {
  template <class P>
  static __device__ __forceinline__ P load(P p) { return p; }
  template <class P>
  static __device__ __forceinline__ P store(P p) { return p; }
};
// A 10-bit sample v in a 16-bit word at bit SHIFT: I010 (0) or P010 (6).  The other bits of a read
// word are ignored (I010 masks them off); a written word is min(v, 1023) << SHIFT, the other bits 0.
template <int SHIFT>
struct Words10 {
  static __device__ __forceinline__ unsigned short load(unsigned short w) {
    return (unsigned short)((w >> SHIFT) & 0x3FF);
  }
  static __device__ __forceinline__ ushort2 load(ushort2 w) {
    return make_ushort2(load(w.x), load(w.y));
  }
  static __device__ __forceinline__ unsigned short store(unsigned short v) {
    return (unsigned short)(min((unsigned)v, 1023u) << SHIFT);
  }
  static __device__ __forceinline__ ushort2 store(ushort2 v) {
    return make_ushort2(store(v.x), store(v.y));
  }
};

// the normalized luma of an enlarged pixel: extract_luma_kernel's of RGBA8, Y' / 255 of an 8-bit
// Y plane, v / 1023 of a 10-bit one (the stored v, capped at 1023)
__device__ __forceinline__ float luma_from(uchar4 p) { return generic::luma_of(p, 1); }
__device__ __forceinline__ float luma_from(unsigned char y) { return __fdiv_rn((float)y, 255.0f); }
__device__ __forceinline__ float luma_from(unsigned short v) {
  return __fdiv_rn((float)min((unsigned)v, 1023u), 1023.0f);
}

template <int TAPS, class Pix, class Io = Bytes>
__global__ void __launch_bounds__(kThreads) resample_kernel(const Planes<Pix> planes) {
  using Weight = typename Acc<Pix>::Weight;
  extern __shared__ __align__(16) unsigned char smem[];
  Pix* mid = reinterpret_cast<Pix*>(smem);   // [rows][kTX] horizontal-pass result, 8 or 16-bit
  const unsigned pl = blockIdx.z % planes.n, f = blockIdx.z / planes.n;
  // (selected, not indexed: a dynamic index would copy the parameters to local memory)
  const Plane<Pix>& P = pl == 0 ? planes.p[0] : pl == 1 ? planes.p[1] : planes.p[2];
  const int W = P.W, H = P.H;
  const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * kTY;
  if (x0 >= W || y0 >= H) return;
  const Pix* __restrict__ in = P.in + f * P.in_frame;
  Pix* __restrict__ out = P.out + f * P.out_frame;
  float* __restrict__ luma = P.luma ? P.luma + f * (size_t)W * H : nullptr;
  const int* xb = P.tab;
  const int* xn = xb + W;
  const Weight* xk = reinterpret_cast<const Weight*>(xn + W);
  const int* yb = P.tab + (size_t)W * (2 + TAPS * (sizeof(Weight) / sizeof(int)));
  const int* yn = yb + H;
  const Weight* yk = reinterpret_cast<const Weight*>(yn + H);
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
    const Pix* src = in + (size_t)(row0 + r) * P.in_pitch + b;
    Acc<Pix> acc;
#pragma unroll
    for (int j = 0; j < TAPS; j++)
      if (j < n) acc.add(Io::load(src[j]), __ldg(xk + (size_t)x * TAPS + j));
    mid[i] = acc.pixel();
  }
  __syncthreads();
  // vertical pass from shared memory
  const int ny = ylast - y0 + 1;
  for (int i = threadIdx.x; i < ny * kTX; i += kThreads) {
    const int r = i / kTX, c = i - r * kTX;
    if (c >= nx) continue;
    const int y = y0 + r, x = x0 + c;
    const int b = __ldg(yb + y) - row0, n = __ldg(yn + y);
    Acc<Pix> acc;
#pragma unroll
    for (int j = 0; j < TAPS; j++)
      if (j < n) acc.add(mid[(b + j) * kTX + c], __ldg(yk + (size_t)y * TAPS + j));
    const Pix o = acc.pixel();
    out[(size_t)y * P.out_pitch + x] = Io::store(o);
    if constexpr (!std::is_same<Pix, uchar2>::value && !std::is_same<Pix, ushort2>::value)
      if (luma) luma[(size_t)y * W + x] = luma_from(o);
  }
}

// the cached device tables of one shape, filter, pair of chroma sitings (SRCNN_CHROMA_*; both
// SRCNN_CHROMA_CENTER for RGBA8 and Y) and sample bit depth (8: 22-bit weights, 10: double ones),
// uploaded on the context stream on first use
inline int table_for(srcnn_ctx* ctx, int w, int h, int W, int H, int filter, int siting_in,
                     int siting_out, const int** dev, int* rows_max, int bit_depth = 8) {
  const srcnn_ctx::ResampleKey key{w, h, W, H, filter, siting_in, siting_out, bit_depth};
  for (const srcnn_ctx::ResampleTable& t : ctx->resample_tables)
    if (std::memcmp(&t.key, &key, sizeof(key)) == 0) {
      *dev = t.dev;
      *rows_max = t.rows_max;
      return SRCNN_OK;
    }
  srcnn_ctx::ResampleTable t;
  t.key = key;
  t.host = tables(w, h, W, H, filter, box_start(w, W, siting_x(siting_in), siting_x(siting_out)),
                  box_start(h, H, siting_y(siting_in), siting_y(siting_out)), bit_depth == 10,
                  &t.rows_max);
  void* p = nullptr;
  if (cudaMalloc(&p, t.host.size() * sizeof(int)) != cudaSuccess) {
    cudaGetLastError();
    return fail(SRCNN_ENOMEM, "resample table allocation failed");
  }
  t.dev = static_cast<int*>(p);
  // cudaMalloc's alignment keeps double weights 8-byte aligned; the host copy lives as long as the
  // context, so the asynchronous copy may read it late
  ctx->resample_tables.push_back(std::move(t));
  srcnn_ctx::ResampleTable& s = ctx->resample_tables.back();
  SRCNN_CUDA(cudaMemcpyAsync(s.dev, s.host.data(), s.host.size() * sizeof(int),
                             cudaMemcpyHostToDevice, ctx->stream));
  *dev = s.dev;
  *rows_max = s.rows_max;
  return SRCNN_OK;
}

// `frames` frames of every plane in one launch; rows_max: the most of the planes' table_for
template <class Pix, class Io = Bytes>
inline int launch_planes(srcnn_ctx* ctx, const Planes<Pix>& planes, int filter, int rows_max,
                         int frames) {
  int W = 0, H = 0;
  for (int i = 0; i < planes.n; i++) {
    W = std::max(W, planes.p[i].W);
    H = std::max(H, planes.p[i].H);
  }
  const dim3 grid((unsigned)((W + kTX - 1) / kTX), (unsigned)((H + kTY - 1) / kTY),
                  (unsigned)(frames * planes.n));
  const size_t smem = (size_t)rows_max * kTX * sizeof(Pix);
  // at most (kTY - 1) + 2 * 3 + 1 rows for an enlargement: well under the default 48 KB.  A siting
  // shifts a CTA's centres but not their spread, at most (kTY - 1) * scale <= kTY - 1 rows, and each
  // output spans at most 2 * 3 + 1 taps (a conversion at ratio 1: 15 + 7 = 22 rows)
  if (filter == SRCNN_RESAMPLE_LANCZOS)
    resample_kernel<7, Pix, Io><<<grid, kThreads, smem, ctx->stream>>>(planes);
  else
    resample_kernel<5, Pix, Io><<<grid, kThreads, smem, ctx->stream>>>(planes);
  return SRCNN_OK;
}

// `frames` RGBA8 frames of w x h (in) -> W x H (out, luma), back to back
inline int launch(srcnn_ctx* ctx, const uchar4* in, int w, int h, uchar4* out, float* luma, int W,
                  int H, int filter, const int* tab, int rows_max, int frames = 1) {
  Planes<uchar4> p{};
  p.p[0] = Plane<uchar4>{in, w, (size_t)w * h, out, W, (size_t)W * H, luma, W, H, tab};
  p.n = 1;
  return launch_planes(ctx, p, filter, rows_max, frames);
}

// `frames` Y'CbCr 4:2:0 frames of w x h (in, layout li) -> W x H (out, layout lo), I420 (or I010:
// T = unsigned short, Io = Words10<0>): Y through tab_y (w x h -> W x H, its luma into the dense
// `luma`), Cb and Cr through tab_c (w/2 x h/2 -> W/2 x H/2), one launch.  w, h, W and H are even;
// the layouts are I420 and hold the planes, and their pitches, offsets and strides (in bytes) are
// multiples of sizeof(T) (the entries check all of it).
template <class T, class Io>
inline int launch_yuv420(srcnn_ctx* ctx, const unsigned char* in, const srcnn_yuv420_layout& li,
                         int w, int h, unsigned char* out, const srcnn_yuv420_layout& lo,
                         float* luma, int W, int H, int filter, const int* tab_y, int rows_y,
                         const int* tab_c, int rows_c, int frames) {
  constexpr size_t b = sizeof(T);
  const T* pi = reinterpret_cast<const T*>(in);
  T* po = reinterpret_cast<T*>(out);
  Planes<T> p{};
  p.p[0] = Plane<T>{pi, (int)(li.y_pitch / b), li.frame_stride / b, po, (int)(lo.y_pitch / b),
                    lo.frame_stride / b, luma, W, H, tab_y};
  p.p[1] = Plane<T>{pi + li.cb_offset / b, (int)(li.c_pitch / b), li.frame_stride / b,
                    po + lo.cb_offset / b, (int)(lo.c_pitch / b), lo.frame_stride / b, nullptr,
                    W / 2, H / 2, tab_c};
  p.p[2] = Plane<T>{pi + li.cr_offset / b, (int)(li.c_pitch / b), li.frame_stride / b,
                    po + lo.cr_offset / b, (int)(lo.c_pitch / b), lo.frame_stride / b, nullptr,
                    W / 2, H / 2, tab_c};
  p.n = 3;
  return launch_planes<T, Io>(ctx, p, filter, std::max(rows_y, rows_c), frames);
}

// launch_yuv420 for NV12 (or P010: T = unsigned short, Io = Words10<6>) layouts, whose chroma is
// one plane of interleaved Cb, Cr pairs: the Y plane, then the CbCr plane as (w/2 x h/2 pairs),
// each sample of a pair as launch_yuv420 computes its plane.  Two launches (a launch has one pixel
// type).  The CbCr planes, their pitches and the frame strides are multiples of 2 * sizeof(T)
// (the entries check them).
template <class T, class Io>
inline int launch_nv12(srcnn_ctx* ctx, const unsigned char* in, const srcnn_yuv420_layout& li,
                       int w, int h, unsigned char* out, const srcnn_yuv420_layout& lo,
                       float* luma, int W, int H, int filter, const int* tab_y, int rows_y,
                       const int* tab_c, int rows_c, int frames) {
  using T2 = typename std::conditional<sizeof(T) == 1, uchar2, ushort2>::type;
  constexpr size_t b = sizeof(T), b2 = sizeof(T2);
  Planes<T> y{};
  y.p[0] = Plane<T>{reinterpret_cast<const T*>(in), (int)(li.y_pitch / b), li.frame_stride / b,
                    reinterpret_cast<T*>(out), (int)(lo.y_pitch / b), lo.frame_stride / b, luma,
                    W, H, tab_y};
  y.n = 1;
  SRCNN_TRY((launch_planes<T, Io>(ctx, y, filter, rows_y, frames)));
  Planes<T2> c{};
  c.p[0] = Plane<T2>{reinterpret_cast<const T2*>(in + li.cb_offset), (int)(li.c_pitch / b2),
                     li.frame_stride / b2,
                     reinterpret_cast<T2*>(out + lo.cb_offset), (int)(lo.c_pitch / b2),
                     lo.frame_stride / b2, nullptr, W / 2, H / 2, tab_c};
  c.n = 1;
  return launch_planes<T2, Io>(ctx, c, filter, rows_c, frames);
}

}  // namespace resample
}  // namespace srcnn
