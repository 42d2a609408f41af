// Shape-specialised sm_100a kernels for the SRCNN configurations (9-1-5 / 9-5-5, n1/n2 =
// 64/32, 128/64, 32/16) and the fused launches of the hot path.  Every entry returns
// "not handled" for shapes it has no instantiation for; the caller then uses the any-shape
// kernels of kernels_generic.cuh.
#pragma once
#include <cuda_runtime.h>

#include "context.cuh"
#include "fused_forward.cuh"
#include "fused_forward_pl.cuh"
#include "fused_forward_hp.cuh"
#include "fused_forward_hpw.cuh"
#include "train_kernels.cuh"
#include "deltas_tc.cuh"
#include "wgrad_tc.cuh"
#include "wgrad1_fused_tc.cuh"
#include "conv5_tc.cuh"
#include "wgrad5_tc.cuh"
#include "bwd3_tc.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace srcnn {
namespace fast {

// ------------------------------------------------------------------ fused update -----
// ConfigBasedDataPipeline::update_parameters (src/ConfigBasedDataPipeline.cpp:325-361) in
// one launch: update_params (src/kernel/update_parameters.cl:1-33) for the three layers
// with their own learning rates, then the six gradient accumulators are zeroed
// (ConfigBasedDataPipeline.cpp:353-358) by the same thread that consumed them.
struct UpdateAllArgs {
  float *w[3], *b[3], *gw[3], *gb[3], *pw[3], *pb[3];
  unsigned ws[3], bs[3];
  float lr[3];
  float momentum, decay, batch;
};

__global__ void update_all_kernel(UpdateAllArgs a) {
  unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
  for (int l = 0; l < 3; l++) {
    if (i < a.ws[l]) {
      const float wv = a.w[l][i];
      const float dw = a.momentum * a.pw[l][i] + a.lr[l] * a.gw[l][i] + a.decay * wv;
      a.w[l][i] = wv - dw / a.batch;
      a.pw[l][i] = dw;
      a.gw[l][i] = 0.f;
      return;
    }
    i -= a.ws[l];
    if (i < a.bs[l]) {
      const float db = a.momentum * a.pb[l][i] + a.lr[l] * a.gb[l][i];
      a.b[l][i] -= db / a.batch;
      a.pb[l][i] = db;
      a.gb[l][i] = 0.f;
      return;
    }
    i -= a.bs[l];
  }
}

// one-time per-context setup (opt-in shared memory sizes etc.)
inline int configure(srcnn_ctx* ctx) {
  SRCNN_TRY(fused::configure());
  SRCNN_TRY(fused_pl::configure());
  SRCNN_TRY(fused_hp::configure());
  SRCNN_TRY(fused_hpw::configure());
  // A/B switch between the generations of the fused kernel (default: the newest)
  const char* impl = std::getenv("SRCNN_FUSED_IMPL");
  ctx->fused_impl = 4;                                           // "hp": planes, FP16 split
  if (impl && std::strcmp(impl, "pl") == 0) ctx->fused_impl = 3;  // planes, 3xTF32
  if (impl && std::strcmp(impl, "simt") == 0) ctx->fused_impl = 0;
  const char* d1 = std::getenv("SRCNN_D1_IMPL");   // "simt": FP32 kernel for the f=1 deltas
  ctx->deltas_tc = !(d1 && std::strcmp(d1, "simt") == 0);
  const char* gw = std::getenv("SRCNN_GW_IMPL");   // "simt": FP32 kernel for the layer-1 gradient
  ctx->wgrad_tc = !(gw && std::strcmp(gw, "simt") == 0);
  // "separate" (or "simt"): the layer-1 deltas are materialised by their own launch; default:
  // they only exist inside the layer-1 gradient kernel (wgrad1_fused_tc.cuh)
  ctx->d1_fused = ctx->deltas_tc && ctx->wgrad_tc && !(d1 && std::strcmp(d1, "separate") == 0);
  return SRCNN_OK;
}

// returns true when it launched
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// returns true when it launched
inline bool forward_layer(srcnn_ctx* ctx, const float* in, float* out, const float* W,
                          const float* B, int k, int n, int f, bool relu, int in_w, int in_h,
                          int S) {
  return train::n1_forward(ctx, in, out, W, B, k, n, f, relu, in_w, in_h, S);
}

// ---- backward of the last layer on the tensor cores (bwd3_tc.cuh) ------------------------------
// d3, d2 and the layer-3 gradient partials of a chunk of patch-sized samples; returns 1 when
// launched (then max |d2| is in the context's maxima block), 0 when left to the FP32 kernel
inline int conv5_maxes(srcnn_ctx* ctx, c5::Maxes** out);
inline int backward3_tc(srcnn_ctx* ctx, const float* gt, const float* out3, const float* out2,
                        const float* W3, float* d3, float* d2, float* gw, float* gb, int k, int f,
                        int gt_w, int gt_h, int w3, int h3, int S) {
  static const bool off = std::getenv("SRCNN_B3_IMPL") && std::strcmp(std::getenv("SRCNN_B3_IMPL"), "simt") == 0;
  if (off || !ctx->wgrad_tc || !b3tc::supported(k, f)) return 0;
  const int ow = w3 + f - 1, oh = h3 + f - 1;
  // batches of patches.  gW3 sums 16 MMAs per out2 row into one FP32 tensor-memory accumulator,
  // whose rounding error grows with the row count (1.5e-4 relative at 396 rows, measured on a
  // B200): taller samples go to the FP32 kernel
  if ((long long)S * ow < 32 * 128 || ow > 1024 || oh > b3tc::MAX_ROWS) return 0;
  if (!aligned16(out2) || !aligned16(d2)) return 0;
  c5::Maxes* mx;
  SRCNN_TRY(conv5_maxes(ctx, &mx));
  int count = 0;
  const int rc = b3tc::bwd3_tc(ctx, gt, out3, out2, W3, d3, d2, mx, ctx->c5_fresh_out2 == out2, k, f,
                               gt_w, gt_h, w3, h3, S, &count);
  if (rc != 1) return rc;
  ctx->c5_fresh_d2 = d2;
  const int Mw = f * f * k;
  train::partial_reduce_kernel<<<(Mw + 1 + train::RED_OUT - 1) / train::RED_OUT,
                                 train::RED_OUT * train::RED_WARPS, 0, ctx->stream>>>(
      (const float*)ctx->splitk_scratch, gw, gb, Mw, 1, count);
  return 1;
}

// ---- 9-5-5 layer 2 on the tensor cores (conv5_tc.cuh) ----------------------------------------
// The virtual-image kernels want enough strips of 128 columns to fill the GPU: batches of
// patch-sized samples (training / validation chunks).  Returns 1 when launched, 0 when the
// shape is left to the other kernels, < 0 on error.
inline bool conv5_shape_ok(srcnn_ctx* ctx, int w1, int h1, int S) {
  static const bool off = std::getenv("SRCNN_C5_IMPL") && std::strcmp(std::getenv("SRCNN_C5_IMPL"), "simt") == 0;
  if (off || !ctx->wgrad_tc) return false;
  const long long vw = (long long)S * w1;
  return w1 >= c5::F && h1 >= c5::F && w1 <= 1024 && h1 <= 4096 && vw >= 32 * 128 &&
         (long long)S * w1 * h1 * 64 < (1LL << 40);
}
inline int conv5_maxes(srcnn_ctx* ctx, c5::Maxes** out) {
  if (!ctx->c5_maxes) SRCNN_CUDA(cudaMalloc(&ctx->c5_maxes, sizeof(c5::Maxes)));
  *out = reinterpret_cast<c5::Maxes*>(ctx->c5_maxes);
  return SRCNN_OK;
}
inline int conv5_forward(srcnn_ctx* ctx, const float* in, float* out, const float* W, const float* B,
                         int k, int n, int f, bool relu, int in_w, int in_h, int S, srcnn_mem wh,
                         bool cacheable, bool max_known = false) {
  if (!(k == 64 && n == 32 && f == c5::F && relu) || !conv5_shape_ok(ctx, in_w, in_h, S)) return 0;
  if (!aligned16(in) || !aligned16(out)) return 0;
  const c5::Images* img;
  ctx->c5_h = wh;
  SRCNN_TRY(c5::prepare(ctx, W, cacheable, &img));
  c5::Maxes* mx;
  SRCNN_TRY(conv5_maxes(ctx, &mx));
  if (!max_known) SRCNN_TRY(c5::absmax(ctx, in, (size_t)S * in_w * in_h * 64, &mx->out1));
  ctx->c5_max_out1_of = in;
  SRCNN_CUDA(cudaMemsetAsync(&mx->out2, 0, sizeof(unsigned), ctx->stream));
  c5::Args a{in, B, out, img->fwd, &img->sw, &mx->out1, S, in_w, in_h, &mx->out2};
  SRCNN_TRY(c5::launch<c5::FwdCfg>(ctx, a));
  ctx->c5_fresh_out2 = out;   // max |out2| recorded by the epilogue
  return 1;
}
// layer 1 of a 9-5-5 training chunk through the FP16-split tensor-core kernel in its
// layer-1-only mode; leaves max |out1| in the context's c5::Maxes.  Returns 1 when launched.
inline int conv5_layer1(srcnn_ctx* ctx, const float* in, float* out1, const float* w1,
                        const float* b1, int n1, int f1, int w, int h, int S) {
  if (ctx->fused_impl != 4 || n1 != fused_hp::Cfg::N1 || f1 != fused_hp::Cfg::F1) return 0;
  if (!conv5_shape_ok(ctx, w - f1 + 1, h - f1 + 1, S)) return 0;
  if (w > 512 || (long long)S * w >= (1LL << 30) || (long long)S * w * h >= (1LL << 31)) return 0;
  if (!aligned16(out1)) return 0;   // (the one-channel input is read float by float)
  c5::Maxes* mx;
  SRCNN_TRY(conv5_maxes(ctx, &mx));
  SRCNN_TRY(c5::absmax(ctx, in, (size_t)S * w * h, &mx->in));
  SRCNN_TRY(fused_hp::launch_l1only(ctx, in, out1, w1, b1, w, h, S, &mx->in, &mx->out1));
  ctx->launch_count += 2;
  return 1;
}

// layer-1 deltas below the 5x5 layer 2: target / layer_output are out1-shaped [S][oh][ow][64]
inline int conv5_deltas(srcnn_ctx* ctx, const float* dn, const float* lo, float* target,
                        const float* W, int n_curr, int f_next, int n_next, int ow, int oh, int S,
                        srcnn_mem wh, bool cacheable) {
  if (!(n_curr == 64 && n_next == 32 && f_next == c5::F) || !conv5_shape_ok(ctx, ow, oh, S)) return 0;
  if (!aligned16(dn) || !aligned16(lo) || !aligned16(target)) return 0;
  const c5::Images* img;
  ctx->c5_h = wh;
  SRCNN_TRY(c5::prepare(ctx, W, cacheable, &img));
  c5::Maxes* mx;
  SRCNN_TRY(conv5_maxes(ctx, &mx));
  if (ctx->c5_fresh_d2 != dn)   // (the tensor-core backward of layer 3 records it)
    SRCNN_TRY(c5::absmax(ctx, dn, (size_t)S * (ow - 4) * (oh - 4) * 32, &mx->d2));
  ctx->c5_max_d2_of = dn;
  c5::Args a{dn, lo, target, img->d1, &img->sw, &mx->d2, S, ow, oh, nullptr};
  SRCNN_TRY(c5::launch<c5::D1Cfg>(ctx, a));
  return 1;
}

inline bool deltas(srcnn_ctx* ctx, const float* dn, const float* lo, float* target,
                   const float* W, int n_curr, int f_next, int n_next, int ow, int oh, int S) {
  if (ctx->deltas_tc &&
      d1tc::f1_deltas_tc(ctx, dn, lo, target, W, n_curr, f_next, n_next, ow, oh, S))
    return true;
  if (train::f1_deltas(ctx, dn, lo, target, W, n_curr, f_next, n_next, ow, oh, S)) return true;
  return train::n1_deltas(ctx, dn, lo, target, W, n_curr, f_next, n_next, ow, oh, S);
}

// returns 1 when it launched, 0 when not handled, <0 on error.  `maxes_known`: the |x| maxima of
// `in` (an out1) and `d` (a d2) are already in the context's c5::Maxes (the chunk entries compute
// them for the layer-2 forward / layer-1 deltas of the same tensors)
inline int backpropagate(srcnn_ctx* ctx, const float* d, const float* in, float* gw, float* gb,
                         int n, int k, int f, int ow, int oh, int S, bool maxes_known = false) {
  // the register-tiled kernels use LDG.128 (a one-channel layer input is read float by float:
  // sample sets whose size is not a multiple of 4 leave later chunks float-aligned only)
  if (!aligned16(d) || (k != 1 && !aligned16(in))) return 0;
  if (ctx->wgrad_tc) {   // layer-1 / layer-2 gradients on the tensor cores
    int count = 0;
    int rc = wgtc::wgrad1_tc(ctx, d, in, n, k, f, ow, oh, S, &count);
    if (rc == 0) rc = wgtc::wgrad2_tc(ctx, d, in, n, k, f, ow, oh, S, &count);
    if (rc == 0 && n == wg5::Cfg::N && k == wg5::Cfg::K && f == wg5::Cfg::F &&
        conv5_shape_ok(ctx, ow + f - 1, oh + f - 1, S)) {   // the 5x5 layer 2 of 9-5-5
      c5::Maxes* mx;
      SRCNN_TRY(conv5_maxes(ctx, &mx));
      if (!maxes_known) {
        SRCNN_TRY(c5::absmax(ctx, in, (size_t)S * (ow + f - 1) * (oh + f - 1) * k, &mx->out1));
        SRCNN_TRY(c5::absmax(ctx, d, (size_t)S * ow * oh * n, &mx->d2));
      }
      rc = wg5::wgrad5_tc(ctx, d, in, mx, n, k, f, ow, oh, S, &count);
    }
    if (rc < 0) return rc;
    if (rc == 1) {
      const int Mw = f * f * k, total = (Mw + 1) * n;
      train::partial_reduce_kernel<<<(total + train::RED_OUT - 1) / train::RED_OUT,
                                     train::RED_OUT * train::RED_WARPS, 0, ctx->stream>>>(
          (const float*)ctx->splitk_scratch, gw, gb, Mw, n, count);
      return 1;
    }
  }
  if (!aligned16(in)) return 0;   // the FP32 split-K kernels stage the input with LDG.128
  return train::gradw(ctx, d, in, gw, gb, n, k, f, ow, oh, S);
}

// layer-1 deltas + layer-1 gradients in one launch (+ the fixed-order reduce of the per-CTA
// partials).  returns 1 when it launched, 0 when not handled, <0 on error
inline bool backward1_fused_supported(srcnn_ctx* ctx, int n1, int n2, int f1, int f2) {
  return ctx->d1_fused && f1 == wgf::Cfg::F && f2 == 1 && n1 == wgf::Cfg::N && n2 == wgf::Cfg::K2;
}
inline int backward1_fused(srcnn_ctx* ctx, const float* d2, const float* out1, const float* W2,
                           const float* in, float* gw, float* gb, int n1, int n2, int f1, int f2,
                           int ow, int oh, int S) {
  if (!backward1_fused_supported(ctx, n1, n2, f1, f2)) return 0;
  if (!aligned16(d2) || !aligned16(out1)) return 0;
  int count = 0;
  const int rc = wgf::wgrad1_fused_tc(ctx, d2, out1, W2, in, n1, n2, f1, f2, ow, oh, S, &count);
  if (rc != 1) return rc;
  const int Mw = f1 * f1, total = (Mw + 1) * n1;
  train::partial_reduce_kernel<<<(total + train::RED_OUT - 1) / train::RED_OUT,
                                 train::RED_OUT * train::RED_WARPS, 0, ctx->stream>>>(
      (const float*)ctx->splitk_scratch, gw, gb, Mw, n1, count);
  return 1;
}

inline bool fused_supported(int n1, int n2, int f1, int f2, int f3) {
  return fused::supported(n1, n2, f1, f2, f3);
}

// a network with a fused forward: its shape, its six parameter buffers and the operand image
// fused_prepare returned for them (null when the selected kernel needs none, or not prepared)
struct FusedNet {
  int n1, n2, f1, f2, f3;
  const float *w1, *b1, *w2, *b2, *w3, *b3;
  const void* scales;
};

// prepared operand image for forward_fused launches with these parameters (null when the
// selected kernel needs none).  `cacheable`: the six buffers are context-owned allocations, so
// nothing outside the device layer can have changed them since ctx->write_gen was recorded.
inline int fused_prepare(srcnn_ctx* ctx, const FusedNet& net, bool cacheable, const void** out) {
  *out = nullptr;
  const int n1 = net.n1, n2 = net.n2, f1 = net.f1, f2 = net.f2, f3 = net.f3;
  const bool wide = fused_hpw::supported(n1, n2, f1, f2, f3);
  if (ctx->fused_impl != 4 || !(wide || fused_hp::supported(n1, n2, f1, f2, f3))) return SRCNN_OK;
  const void* key[6] = {net.w1, net.b1, net.w2, net.b2, net.w3, net.b3};
  if (cacheable && ctx->hp_cache_valid && ctx->hp_cache_gen == ctx->write_gen &&
      ctx->hp_cache_n1 == n1 && std::memcmp(key, ctx->hp_cache_key, sizeof(key)) == 0) {
    *out = ctx->hp_cache;
    return SRCNN_OK;
  }
  // the image is about to be rewritten: calls srcnn_infer_rows_host_async still has in flight
  // (for other parameters) read it
  SRCNN_CUDA(ctx->drain_lanes());
  if (!ctx->hp_cache) {
    constexpr size_t bytes = sizeof(fused_hpw::Scales) > sizeof(fused_hp::Scales)
                                 ? sizeof(fused_hpw::Scales) : sizeof(fused_hp::Scales);
    SRCNN_CUDA(cudaMalloc(&ctx->hp_cache, bytes));
  }
  fused::Args a{nullptr, nullptr, net.w1, net.b1, net.w2, net.b2, net.w3, net.b3, 0, 0, 0, 0};
  if (wide)
    fused_hpw::prepare(ctx, a, ctx->hp_cache);
  else
    fused_hp::prepare_into(ctx, a, ctx->hp_cache);
  ctx->launch_count += 1;
  ctx->stats[SRCNN_K_FORWARD_FUSED].launches += 1;
  *out = ctx->hp_cache;
  ctx->hp_cache_valid = cacheable;
  ctx->hp_cache_gen = ctx->write_gen;
  ctx->hp_cache_n1 = n1;
  std::memcpy(ctx->hp_cache_key, key, sizeof(key));
  return SRCNN_OK;
}

// one fused forward of `net` (its `scales` shared by a series of launches, or null)
inline int forward_fused(srcnn_ctx* ctx, const FusedNet& net, const float* in, float* out, int in_w,
                         int in_h, int S) {
  const int n1 = net.n1, n2 = net.n2, f1 = net.f1, f2 = net.f2, f3 = net.f3;
  if (!fused::supported(n1, n2, f1, f2, f3))
    return fail(SRCNN_EINVAL, "no fused forward instantiation");
  // the per-image launches put the sample index in gridDim.z (at most 65 535): larger sample
  // counts that do not take the virtual-image path go out in slices
  constexpr int kMaxZ = 65535;
  const bool virtual_image = S > 1 && in_w <= 512 && (long long)S * in_w < (1LL << 30) &&
                             ctx->fused_impl >= 3 && fused_pl::supported(n1, n2, f1, f2, f3);
  const bool virtual_wide = S > 1 && in_w <= 512 && (long long)S * in_w < (1LL << 30) &&
                            ctx->fused_impl == 4 && fused_hpw::supported(n1, n2, f1, f2, f3);
  if (S > kMaxZ && !virtual_image && !virtual_wide) {
    const int pad = f1 + f2 + f3 - 3;
    const size_t in_px = (size_t)in_w * in_h, out_px = (size_t)(in_w - pad) * (in_h - pad);
    for (int s0 = 0; s0 < S; s0 += kMaxZ)
      SRCNN_TRY(forward_fused(ctx, net, in + s0 * in_px, out + s0 * out_px, in_w, in_h,
                              std::min(kMaxZ, S - s0)));
    return SRCNN_OK;
  }
  fused::Args a{in, out, net.w1, net.b1, net.w2, net.b2, net.w3, net.b3, in_w, in_h,
                in_w - (f1 + f2 + f3 - 3), in_h - (f1 + f2 + f3 - 3)};
  const void* scales = net.scales;
  if (ctx->fused_impl == 4 && fused_hpw::supported(n1, n2, f1, f2, f3)) {
    // the wide network (n1 = 128, n2 = 64)
    const bool as_batch = S > 1 && in_w <= 512 && (long long)S * in_w < (1LL << 30);
    if (!scales) SRCNN_TRY(fused_prepare(ctx, net, false, &scales));
    fused_hp::Scales* unused;
    unsigned* ws;
    SRCNN_TRY(fused_hp::scale_slot(ctx, &unused, &ws));
    return fused_hpw::launch(ctx, a, S, as_batch, static_cast<const fused_hpw::Scales*>(scales),
                             reinterpret_cast<int*>(ws));
  }
  if (ctx->fused_impl >= 3 && fused_pl::supported(n1, n2, f1, f2, f3)) {
    // batches of small samples (validation patches) go through the virtual-image variant
    const bool as_batch = S > 1 && in_w <= 512 && (long long)S * in_w < (1LL << 30);
    if (ctx->fused_impl == 4)
      return fused_hp::launch(ctx, a, S, as_batch, nullptr, nullptr,
                              static_cast<const fused_hp::Scales*>(scales));
    if (as_batch) return fused_pl::launch_batch(ctx, a, S, nullptr, nullptr);
    return fused_pl::launch(ctx, a, S);
  }
  return fused::launch(ctx, n1, n2, a, S);
}

// kernels one fused forward call launches: the FP16-split path is prepare + main + gated TF32
inline int fused_launches(srcnn_ctx* ctx, const FusedNet& net) {
  if (ctx->fused_impl != 4) return 1;
  // FP16 kernel + gated fallback kernel, + the prepare kernel when the launch packs its own
  // operand image (fused_prepare counts the ones it launches itself)
  if (fused_hp::supported(net.n1, net.n2, net.f1, net.f2, net.f3) ||
      fused_hpw::supported(net.n1, net.n2, net.f1, net.f2, net.f3))
    return net.scales ? 2 : 3;
  return 1;
}

inline bool fused_train_supported(srcnn_ctx* ctx, int n1, int n2, int f1, int f2, int f3) {
  return ctx->fused_impl >= 3 && fused_pl::supported(n1, n2, f1, f2, f3);
}

// forward pass of a training chunk: all three layers in one launch, n1/n2-channel maps kept.
// returns 1 when it launched, 0 when there is no instantiation for the shape
inline int forward_train_fused(srcnn_ctx* ctx, const FusedNet& net, const float* in, float* out1,
                               float* out2, float* out3, int in_w, int in_h, int S,
                               unsigned* out2_max) {
  const int pad = net.f1 + net.f2 + net.f3 - 3;
  if (ctx->fused_impl < 3 || !fused_pl::supported(net.n1, net.n2, net.f1, net.f2, net.f3)) return 0;
  if ((long long)S * in_w >= (1LL << 30)) return 0;
  if ((long long)S * in_w * in_h >= (1LL << 31)) return 0;   // 32-bit pixel indices of out1 / out2
  fused::Args a{in, out3, net.w1, net.b1, net.w2, net.b2, net.w3, net.b3, in_w, in_h, in_w - pad,
                in_h - pad};
  const int rc = ctx->fused_impl == 4
                     ? fused_hp::launch(ctx, a, S, true, out1, out2,
                                        static_cast<const fused_hp::Scales*>(net.scales), out2_max)
                     : fused_pl::launch_batch(ctx, a, S, out1, out2, out2_max);
  return rc == SRCNN_OK ? 1 : rc;
}

}  // namespace fast
}  // namespace srcnn
