// Enlargement quality: PSNR / SSIM inputs of S image pairs (a result against its reference).
//
// Both metrics are taken on the network's own luma (generic::luma_of, normalize = 1: data range
// L = 1) over the region [border, w - border) x [border, h - border):
//   mse  = mean over the region of d^2, d = Y_result - Y_ref in float, d^2 and the sum in double;
//   ssim = Wang et al. 2004 (their reference `ssim_index`): the mean, over every 11 x 11 window
//          lying wholly inside the region ("valid" windows, no padding), of
//          ((2 mx my + C1)(2 sxy + C2)) / ((mx^2 + my^2 + C1)(sx^2 + sy^2 + C2)), C1 = 0.01^2,
//          C2 = 0.03^2, with the window statistics weighted by a Gaussian of sigma 1.5 normalised
//          to sum 1, in population form (sx^2 = E[x^2] - mx^2, sxy = E[xy] - mx my).
// The window statistics are accumulated in double: E[x^2] - mx^2 cancels, and in float the
// cancellation error of a flat window is a sizeable fraction of C2.
//
// Two launches.  Stage 1: a CTA owns kTY x kTX region pixels of one frame (blockIdx.z) and the
// windows whose top-left corner is one of them.  It loads its tile plus the 10 rows / columns
// those windows reach beyond it (a 5-pixel halo around the window centres) of both images as
// luma, runs the separable Gaussian horizontally over the five maps x, y, x^2, y^2, xy into
// shared memory, then vertically, and reduces the SSIM values and squared differences to one
// double pair per CTA.  Stage 2: one block per frame folds that frame's pairs in index order.
// The partition depends on the frame's size only, so a frame's result is the same whatever else
// shares the launch, and bit-identical between calls.
#pragma once
#include <cmath>

#include "context.cuh"
#include "kernels_generic.cuh"

namespace srcnn {
namespace quality {

constexpr int kWin = 11;                       // SSIM window (Gaussian, sigma 1.5)
constexpr int kTX = 32, kTY = 16, kThreads = 256;
constexpr int kRows = kTY + kWin - 1, kCols = kTX + kWin - 1;
constexpr double kC1 = 0.01 * 0.01, kC2 = 0.03 * 0.03;

// the 1-D Gaussian, normalised to sum 1: the 2-D window is its outer product with itself
struct Window {
  double g[kWin];
};

inline Window gaussian_window() {
  Window w;
  double s = 0.0;
  for (int i = 0; i < kWin; i++) {
    const double x = i - kWin / 2;
    w.g[i] = std::exp(-(x * x) / (2.0 * 1.5 * 1.5));
    s += w.g[i];
  }
  for (int i = 0; i < kWin; i++) w.g[i] /= s;
  return w;
}

// the CTAs of one frame's stage 1
inline int tiles_x(int w, int border) { return (w - 2 * border + kTX - 1) / kTX; }
inline int tiles_y(int h, int border) { return (h - 2 * border + kTY - 1) / kTY; }

// result: w*h*bpp bytes a frame (RGB8 or RGBA8), ref: w*h RGBA8 a frame; partial: one
// {sum of d^2, sum of SSIM} per CTA, frame by frame
__global__ void __launch_bounds__(kThreads)
quality_stage1(const unsigned char* __restrict__ result, int bpp, const uchar4* __restrict__ ref,
               int w, int h, int border, Window win, double2* __restrict__ partial) {
  __shared__ float lx[kRows][kCols], ly[kRows][kCols];
  __shared__ double hsum[5][kRows][kTX];        // x, y, x^2, y^2, xy after the horizontal pass
  __shared__ double sh_a[32], sh_b[32];
  const size_t npx = (size_t)w * h;
  result += blockIdx.z * npx * bpp;
  ref += blockIdx.z * npx;
  const int x1 = w - border, y1 = h - border;   // region end (exclusive)
  const int tx0 = border + blockIdx.x * kTX, ty0 = border + blockIdx.y * kTY;
  // tile + halo as luma; outside the region 0 (no valid window reads it)
  double sse = 0.0;
  for (int i = threadIdx.x; i < kRows * kCols; i += kThreads) {
    const int r = i / kCols, c = i - r * kCols;
    const int y = ty0 + r, x = tx0 + c;
    float a = 0.f, b = 0.f;
    if (x < x1 && y < y1) {
      const size_t p = (size_t)y * w + x;
      const unsigned char* q = result + p * bpp;
      a = generic::luma_of(make_uchar4(q[0], q[1], q[2], 0), 1);
      b = generic::luma_of(ref[p], 1);
      if (r < kTY && c < kTX) {
        const double d = (double)__fsub_rn(a, b);
        sse += d * d;
      }
    }
    lx[r][c] = a;
    ly[r][c] = b;
  }
  __syncthreads();
  // horizontal pass: every tile + halo row, the window columns of the kTX window corners
  for (int i = threadIdx.x; i < kRows * kTX; i += kThreads) {
    const int r = i / kTX, c = i - r * kTX;
    double sx = 0.0, sy = 0.0, sxx = 0.0, syy = 0.0, sxy = 0.0;
#pragma unroll
    for (int j = 0; j < kWin; j++) {
      const double a = lx[r][c + j], b = ly[r][c + j], g = win.g[j];
      sx += g * a;
      sy += g * b;
      sxx += g * (a * a);
      syy += g * (b * b);
      sxy += g * (a * b);
    }
    hsum[0][r][c] = sx;
    hsum[1][r][c] = sy;
    hsum[2][r][c] = sxx;
    hsum[3][r][c] = syy;
    hsum[4][r][c] = sxy;
  }
  __syncthreads();
  // vertical pass and SSIM of every valid window whose top-left corner is in the tile
  double ssim = 0.0;
  for (int i = threadIdx.x; i < kTY * kTX; i += kThreads) {
    const int r = i / kTX, c = i - r * kTX;
    if (tx0 + c + kWin > x1 || ty0 + r + kWin > y1) continue;
    double m[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int j = 0; j < kWin; j++) {
      const double g = win.g[j];
#pragma unroll
      for (int k = 0; k < 5; k++) m[k] += g * hsum[k][r + j][c];
    }
    const double mx = m[0], my = m[1];
    const double vx = m[2] - mx * mx, vy = m[3] - my * my, cxy = m[4] - mx * my;
    ssim += ((2.0 * mx * my + kC1) * (2.0 * cxy + kC2)) /
            ((mx * mx + my * my + kC1) * (vx + vy + kC2));
  }
  const double a = generic::block_sum(sse, sh_a);
  const double b = generic::block_sum(ssim, sh_b);
  if (threadIdx.x == 0)
    partial[((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = make_double2(a, b);
}

// frame blockIdx.x: folds its `count` pairs in index order; out[blockIdx.x * stride + {0, 1}] =
// {mse, mean SSIM}
__global__ void __launch_bounds__(generic::RED_THREADS)
quality_stage2(const double2* __restrict__ partial, int count, double n_px, double n_win,
               double* __restrict__ out, int stride) {
  __shared__ double sh_a[32], sh_b[32];
  partial += (size_t)blockIdx.x * count;
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < count; i += blockDim.x) {
    const double2 p = partial[i];
    a += p.x;
    b += p.y;
  }
  a = generic::block_sum(a, sh_a);
  b = generic::block_sum(b, sh_b);
  if (threadIdx.x == 0) {
    out[(size_t)blockIdx.x * stride] = a / n_px;
    out[(size_t)blockIdx.x * stride + 1] = b / n_win;
  }
}

// doubles of stage-1 partials for S frames of w x h
inline size_t partial_bytes(int w, int h, int border, int S) {
  return sizeof(double2) * (size_t)tiles_x(w, border) * tiles_y(h, border) * S;
}

// both stages for S frames on the context stream (the caller validated the arguments and sized
// `partial` with partial_bytes): frame s's {mse, ssim} land at out[s * stride], out[s * stride + 1]
inline void launch(srcnn_ctx* ctx, const unsigned char* result, int bpp, const uchar4* ref, int w,
                   int h, int S, int border, double2* partial, double* out, int stride) {
  static const Window win = gaussian_window();
  const int gx = tiles_x(w, border), gy = tiles_y(h, border);
  const int rw = w - 2 * border, rh = h - 2 * border;
  quality_stage1<<<dim3(gx, gy, S), kThreads, 0, ctx->stream>>>(result, bpp, ref, w, h, border,
                                                               win, partial);
  quality_stage2<<<S, generic::RED_THREADS, 0, ctx->stream>>>(
      partial, gx * gy, (double)rw * rh, (double)(rw - kWin + 1) * (rh - kWin + 1), out, stride);
}

}  // namespace quality
}  // namespace srcnn
