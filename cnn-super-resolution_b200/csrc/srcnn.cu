// C-ABI entry points of the B200 SRCNN device layer (include/srcnn_b200.h).
// Built for sm_100a only.  There is no CPU fallback anywhere in this file: every entry
// either launches CUDA kernels on the context's stream or fails with an error code.
#include "../../include/srcnn_b200.h"


#include <algorithm>
#include <functional>
#include <new>
#include <vector>

#include "comm.cuh"
#include "context.cuh"
#include "kernels_fast.cuh"
#include "kernels_generic.cuh"
#include "quality.cuh"
#include "resample.cuh"

using namespace srcnn;

namespace {

inline int grid_1d(size_t work, int threads, int cap) {
  size_t b = (work + threads - 1) / threads;
  if (b < 1) b = 1;
  if ((size_t)cap < b) b = cap;
  return (int)b;
}

struct Dims {
  int w1, h1, w2, h2, w3, h3;
};
inline Dims net_dims(const srcnn_net* net, int w, int h) {
  Dims d;
  d.w1 = w - net->f1 + 1;
  d.h1 = h - net->f1 + 1;
  d.w2 = d.w1 - net->f2 + 1;
  d.h2 = d.h1 - net->f2 + 1;
  d.w3 = d.w2 - net->f3 + 1;
  d.h3 = d.h2 - net->f3 + 1;
  return d;
}

inline size_t align256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// the enlargements srcnn_resample accepts
inline int check_resample(int w, int h, int out_w, int out_h, int filter) {
  SRCNN_REQUIRE(w > 0 && h > 0 && out_w > 0 && out_h > 0, "bad resample size %dx%d -> %dx%d", w, h,
                out_w, out_h);
  SRCNN_REQUIRE(out_w >= w && out_h >= h, "resample %dx%d -> %dx%d: only enlargements are supported",
                w, h, out_w, out_h);
  SRCNN_REQUIRE((size_t)out_w * out_h < ((size_t)1 << 31), "output of %dx%d pixels is too large",
                out_w, out_h);
  SRCNN_REQUIRE(filter == SRCNN_RESAMPLE_BICUBIC || filter == SRCNN_RESAMPLE_LANCZOS,
                "unknown resample filter %d", filter);
  return SRCNN_OK;
}

// the region srcnn_image_quality measures: at least one SSIM window
inline int check_quality_region(int w, int h, int border) {
  SRCNN_REQUIRE(border >= 0 && w - 2 * (long long)border >= quality::kWin &&
                    h - 2 * (long long)border >= quality::kWin,
                "border %d leaves less than %dx%d pixels of a %dx%d image", border, quality::kWin,
                quality::kWin, w, h);
  return SRCNN_OK;
}

inline int check_net(const srcnn_net* net) {
  SRCNN_REQUIRE(net != nullptr, "net is null");
  SRCNN_REQUIRE(net->n1 > 0 && net->n2 > 0, "n1/n2 must be > 0");
  SRCNN_REQUIRE(net->f1 > 0 && net->f2 > 0 && net->f3 > 0, "f1/f2/f3 must be > 0");
  return SRCNN_OK;
}

// fills `key` with the call arguments (pointers and integers) a captured pipeline depends on
inline unsigned long long key_word(const void* p) { return (unsigned long long)(uintptr_t)p; }
inline unsigned long long key_word(long long v) { return (unsigned long long)v; }
template <class... T>
void graph_key(unsigned long long (&key)[srcnn_ctx::kGraphKey], T... args) {
  static_assert(sizeof...(T) <= srcnn_ctx::kGraphKey, "graph key too long");
  const unsigned long long words[] = {key_word(args)...};
  std::copy(words, words + sizeof...(T), key);
}

}  // namespace

extern "C" {

// ======================================================================= context =====

const char* srcnn_last_error(void) { return last_error_ref().c_str(); }

int srcnn_ctx_create_on_stream(int device, void* cuda_stream, int profile, srcnn_ctx** out) {
  SRCNN_REQUIRE(out != nullptr, "out is null");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(SRCNN_ECUDA,
                "no CUDA device available (%s) -- this library has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  SRCNN_REQUIRE(device >= 0 && device < count, "device %d out of range (have %d)", device, count);
  SRCNN_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SRCNN_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(SRCNN_ECUDA, "device %d is sm_%d%d; this library is built for sm_100a only",
                device, prop.major, prop.minor);
  srcnn_ctx* ctx = new (std::nothrow) srcnn_ctx();
  if (!ctx) return fail(SRCNN_ENOMEM, "out of host memory");
  ctx->device = device;
  ctx->profile = profile != 0;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  if (cuda_stream) {
    ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    ctx->own_stream = false;
  } else {
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      delete ctx;
      return fail(SRCNN_ECUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e));
    }
    ctx->own_stream = true;
  }
  cudaEventCreate(&ctx->ev_start);
  cudaEventCreate(&ctx->ev_stop);
  e = cudaMalloc(&ctx->red_scratch, srcnn_ctx::kRedScratchBytes);
  if (e != cudaSuccess) {
    delete ctx;
    return fail(SRCNN_ENOMEM, "scratch allocation failed: %s", cudaGetErrorString(e));
  }
  ctx->allocs.reserve(256);
  int rc = fast::configure(ctx);
  if (rc != SRCNN_OK) {
    srcnn_ctx_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return SRCNN_OK;
}

int srcnn_ctx_create(int device, int profile, srcnn_ctx** out) {
  return srcnn_ctx_create_on_stream(device, nullptr, profile, out);
}

int srcnn_ctx_destroy(srcnn_ctx* ctx) {
  if (!ctx) return SRCNN_OK;
  cudaSetDevice(ctx->device);
  ctx->drain_lanes();
  cudaStreamSynchronize(ctx->stream);
  for (srcnn_ctx::RowsLane& l : ctx->lanes) {
    if (l.graph) cudaGraphExecDestroy(l.graph);
    if (l.in) cudaFree(l.in);
    if (l.out) cudaFree(l.out);
    if (l.stream) cudaStreamDestroy(l.stream);
  }
  if (ctx->lane_ev) cudaEventDestroy(ctx->lane_ev);
  {
    srcnn_ctx::UpscaleStaging& u = ctx->up;
    if (u.graph) cudaGraphExecDestroy(u.graph);
    for (void* p : {u.small, u.rgba, u.luma, u.out, u.rgb, u.s1, u.s2})
      if (p) cudaFree(p);
  }
  for (srcnn_ctx::FramesStaging* f : {&ctx->frames, &ctx->eval, &ctx->yuv, &ctx->yuv_dev})
    for (void* p : {f->small, f->rgba, f->luma, f->out, f->rgb, f->red, f->s1, f->s2, f->ref,
                    f->qred, f->metrics})
      if (p) cudaFree(p);
  if (ctx->quality_red) cudaFree(ctx->quality_red);
  for (srcnn_ctx::ResampleTable& t : ctx->resample_tables) cudaFree(t.dev);
  if (ctx->nccl_comm && comm::api()) comm::api()->CommDestroy(ctx->nccl_comm);
  ctx->nccl_comm = nullptr;
  for (Allocation& a : ctx->allocs)
    if (a.owned && !a.released && a.ptr) cudaFree(a.ptr);
  if (ctx->red_scratch) cudaFree(ctx->red_scratch);
  if (ctx->splitk_scratch) cudaFree(ctx->splitk_scratch);
  if (ctx->gather_tab) cudaFree(ctx->gather_tab);
  if (ctx->c5_images) cudaFree(ctx->c5_images);
  if (ctx->c5_maxes) cudaFree(ctx->c5_maxes);
  if (ctx->band_in) cudaFree(ctx->band_in);
  if (ctx->band_out) cudaFree(ctx->band_out);
  for (int i = 0; i < 2; i++) {
    if (ctx->stage_in[i]) cudaFree(ctx->stage_in[i]);
    if (ctx->stage_gt[i]) cudaFree(ctx->stage_gt[i]);
  }
  if (ctx->packed_params) cudaFree(ctx->packed_params);
  if (ctx->hp_scales) cudaFree(ctx->hp_scales);
  if (ctx->hp_cache) cudaFree(ctx->hp_cache);
  if (ctx->copy_in) {
    cudaStreamDestroy(ctx->copy_in);
    cudaStreamDestroy(ctx->copy_out);
    if (ctx->compute2) cudaStreamDestroy(ctx->compute2);
    if (ctx->e2e_graph) cudaGraphExecDestroy(ctx->e2e_graph);
    for (int i = 0; i < 2; i++)
      if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
    for (int i = 0; i < srcnn_ctx::kEvents; i++) {
      cudaEventDestroy(ctx->ev_in[i]);
      cudaEventDestroy(ctx->ev_k[i]);
    }
    for (int i = 0; i < 4; i++)
      if (ctx->ev_d[i]) cudaEventDestroy(ctx->ev_d[i]);
  }
  if (ctx->ev_start) cudaEventDestroy(ctx->ev_start);
  if (ctx->ev_stop) cudaEventDestroy(ctx->ev_stop);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return SRCNN_OK;
}

int srcnn_block(srcnn_ctx* ctx) {
  SRCNN_ENTER(ctx);
  SRCNN_CUDA(ctx->drain_lanes());
  SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  return SRCNN_OK;
}

int srcnn_device_info(srcnn_ctx* ctx, char* name, size_t name_len, int* sm_count,
                      size_t* global_mem_bytes) {
  SRCNN_ENTER(ctx);
  cudaDeviceProp prop;
  SRCNN_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
  if (name && name_len) {
    strncpy(name, prop.name, name_len - 1);
    name[name_len - 1] = 0;
  }
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (global_mem_bytes) *global_mem_bytes = prop.totalGlobalMem;
  return SRCNN_OK;
}

int srcnn_profile_get(srcnn_ctx* ctx, int kernel_id, uint64_t* total_ns, uint64_t* launches) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(kernel_id >= 0 && kernel_id < SRCNN_K_COUNT, "bad kernel id %d", kernel_id);
  if (total_ns) *total_ns = ctx->stats[kernel_id].total_ns;
  if (launches) *launches = ctx->stats[kernel_id].launches;
  return SRCNN_OK;
}

int srcnn_launch_count(srcnn_ctx* ctx, uint64_t* launches) {
  SRCNN_REQUIRE(ctx && launches, "null argument");
  *launches = ctx->launch_count;
  return SRCNN_OK;
}

int srcnn_stream(srcnn_ctx* ctx, void** cuda_stream) {
  SRCNN_REQUIRE(ctx && cuda_stream, "null argument");
  *cuda_stream = reinterpret_cast<void*>(ctx->stream);
  return SRCNN_OK;
}

// ======================================================================= memory ======

int srcnn_alloc(srcnn_ctx* ctx, size_t bytes, srcnn_mem* out) {
  SRCNN_REQUIRE(ctx && out, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(bytes > 0, "cannot allocate 0 bytes");
  SRCNN_REQUIRE(ctx->allocs.size() < (size_t)SRCNN_NULL_MEM, "handle table full");
  Allocation a;
  cudaError_t e = cudaMalloc(&a.ptr, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(SRCNN_ENOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  }
  a.bytes = bytes;
  ctx->allocs.push_back(a);
  *out = (srcnn_mem)(ctx->allocs.size() - 1);
  return SRCNN_OK;
}

int srcnn_wrap(srcnn_ctx* ctx, void* device_ptr, size_t bytes, srcnn_mem* out) {
  SRCNN_REQUIRE(ctx && out && device_ptr, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(bytes > 0, "cannot wrap 0 bytes");
  SRCNN_REQUIRE(ctx->allocs.size() < (size_t)SRCNN_NULL_MEM, "handle table full");
  Allocation a;
  a.ptr = device_ptr;
  a.bytes = bytes;
  a.owned = false;
  ctx->allocs.push_back(a);
  *out = (srcnn_mem)(ctx->allocs.size() - 1);
  return SRCNN_OK;
}

int srcnn_release(srcnn_ctx* ctx, srcnn_mem mem) {
  SRCNN_ENTER(ctx);
  if (mem >= ctx->allocs.size()) return fail(SRCNN_EHANDLE, "invalid memory handle");
  ctx->note_write(mem);
  Allocation& a = ctx->allocs[mem];
  if (!a.released && a.ptr && a.owned) {
    SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
    SRCNN_CUDA(cudaFree(a.ptr));
  }
  a.released = true;
  a.ptr = nullptr;
  return SRCNN_OK;
}

int srcnn_mem_size(srcnn_ctx* ctx, srcnn_mem mem, size_t* bytes) {
  SRCNN_REQUIRE(ctx && bytes, "null argument");
  if (mem >= ctx->allocs.size())
    return fail(SRCNN_EHANDLE, "Invalid memory handle.Could not get RawMemoryHandle object");
  *bytes = ctx->allocs[mem].bytes;
  return SRCNN_OK;
}

int srcnn_mem_ptr(srcnn_ctx* ctx, srcnn_mem mem, void** device_ptr) {
  SRCNN_REQUIRE(ctx && device_ptr, "null argument");
  Allocation* a = ctx->get(mem);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle");
  // the raw pointer leaves the device layer: writes through it are invisible to note_write, so
  // nothing derived from this allocation is cached any more (see srcnn_invalidate_params)
  a->exposed = true;
  ctx->note_write(mem);
  *device_ptr = a->ptr;
  return SRCNN_OK;
}

int srcnn_mem_usage(srcnn_ctx* ctx, size_t* buffer_bytes) {
  SRCNN_REQUIRE(ctx && buffer_bytes, "null argument");
  size_t t = 0;
  for (const Allocation& a : ctx->allocs)
    if (!a.released && a.owned) t += a.bytes;
  *buffer_bytes = t;
  return SRCNN_OK;
}

int srcnn_write(srcnn_ctx* ctx, srcnn_mem mem, size_t offset, size_t bytes, const void* src,
                int block) {
  SRCNN_REQUIRE(ctx && src, "null argument");
  SRCNN_ENTER(ctx);
  Allocation* a = ctx->get(mem);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle in write");
  if (bytes > a->bytes || offset > a->bytes - bytes)
    return fail(SRCNN_ERANGE, "Tried to write more then is allocated (%zu+%zu > %zu)", offset,
                bytes, a->bytes);
  ctx->note_write(mem);
  SRCNN_CUDA(cudaMemcpyAsync((char*)a->ptr + offset, src, bytes, cudaMemcpyHostToDevice,
                             ctx->stream));
  if (block) SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  return SRCNN_OK;
}

int srcnn_read(srcnn_ctx* ctx, srcnn_mem mem, size_t offset, size_t bytes, void* dst,
               int block) {
  SRCNN_REQUIRE(ctx && dst, "null argument");
  SRCNN_ENTER(ctx);
  Allocation* a = ctx->get(mem);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle in read");
  if (bytes > a->bytes || offset > a->bytes - bytes)
    return fail(SRCNN_ERANGE, "Tried to read more then is allocated (%zu+%zu > %zu)", offset,
                bytes, a->bytes);
  SRCNN_CUDA(cudaMemcpyAsync(dst, (const char*)a->ptr + offset, bytes, cudaMemcpyDeviceToHost,
                             ctx->stream));
  if (block) SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  return SRCNN_OK;
}

int srcnn_copy_region(srcnn_ctx* ctx, srcnn_mem src, size_t src_offset, srcnn_mem dst,
                      size_t dst_offset, size_t bytes) {
  SRCNN_ENTER(ctx);
  Allocation* s = ctx->get(src);
  Allocation* d = ctx->get(dst);
  if (!s || !d) return fail(SRCNN_EHANDLE, "invalid memory handle in copy");
  if (bytes > s->bytes || src_offset > s->bytes - bytes)
    return fail(SRCNN_ERANGE, "buffer copy would read after src end");
  if (bytes > d->bytes || dst_offset > d->bytes - bytes)
    return fail(SRCNN_ERANGE, "When performing buffer copy, would write after dst end");
  ctx->note_write(dst);
  SRCNN_CUDA(cudaMemcpyAsync((char*)d->ptr + dst_offset, (const char*)s->ptr + src_offset, bytes,
                             cudaMemcpyDeviceToDevice, ctx->stream));
  return SRCNN_OK;
}

int srcnn_copy(srcnn_ctx* ctx, srcnn_mem src, srcnn_mem dst, size_t dst_offset) {
  SRCNN_ENTER(ctx);
  Allocation* s = ctx->get(src);
  if (!s) return fail(SRCNN_EHANDLE, "invalid memory handle in copy");
  return srcnn_copy_region(ctx, src, 0, dst, dst_offset, s->bytes);
}

int srcnn_gather(srcnn_ctx* ctx, const srcnn_mem* src, int n, size_t bytes_each, srcnn_mem dst) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(src != nullptr && n > 0, "nothing to gather");
  SRCNN_REQUIRE(bytes_each > 0 && bytes_each % sizeof(float) == 0, "bytes_each must be a multiple of 4");
  SRCNN_REQUIRE(n <= 65535 * 64, "too many buffers in one gather");
  float* pd;
  SRCNN_TRY(resolve(ctx, dst, bytes_each * (size_t)n, &pd, "gather destination"));
  ctx->note_write(dst);
  std::vector<const float*> tab((size_t)n);
  for (int i = 0; i < n; i++)
    SRCNN_TRY(resolve(ctx, src[i], bytes_each, &tab[(size_t)i], "gather source"));
  SRCNN_TRY(ensure_scratch(ctx, &ctx->gather_tab, &ctx->gather_tab_bytes, sizeof(void*) * (size_t)n));
  // pageable source: the runtime stages the table before the call returns, so `tab` may go
  SRCNN_CUDA(cudaMemcpyAsync(ctx->gather_tab, tab.data(), sizeof(void*) * (size_t)n,
                             cudaMemcpyHostToDevice, ctx->stream));
  const size_t floats_each = bytes_each / sizeof(float);
  for (int y0 = 0; y0 < n; y0 += 65535) {
    const int ny = std::min(65535, n - y0);
    dim3 grid((unsigned)std::min<size_t>(64, (floats_each + 255) / 256), (unsigned)ny);
    generic::gather_kernel<<<grid, 256, 0, ctx->stream>>>(
        reinterpret_cast<const float* const*>(ctx->gather_tab) + y0, pd + (size_t)y0 * floats_each,
        floats_each);
    ctx->launch_count++;
  }
  return check_launch("gather");
}

int srcnn_fill_float(srcnn_ctx* ctx, srcnn_mem mem, float value) {
  SRCNN_ENTER(ctx);
  Allocation* a = ctx->get(mem);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle in fill");
  ctx->note_write(mem);
  const size_t len = a->bytes / sizeof(float);
  if (len == 0) return SRCNN_OK;
  if (value == 0.f) {
    SRCNN_CUDA(cudaMemsetAsync(a->ptr, 0, len * sizeof(float), ctx->stream));
    return SRCNN_OK;
  }
  generic::fill_kernel<<<grid_1d(len, 256, 4 * ctx->sm_count), 256, 0, ctx->stream>>>(
      (float*)a->ptr, value, len);
  ctx->launch_count++;
  return check_launch("fill");
}

int srcnn_host_alloc(size_t bytes, void** host_ptr) {
  SRCNN_REQUIRE(host_ptr && bytes > 0, "bad argument");
  SRCNN_CUDA(cudaHostAlloc(host_ptr, bytes, cudaHostAllocDefault));
  return SRCNN_OK;
}

int srcnn_host_free(void* host_ptr) {
  if (host_ptr) SRCNN_CUDA(cudaFreeHost(host_ptr));
  return SRCNN_OK;
}

// ======================================================================= kernels =====

int srcnn_forward_layer(srcnn_ctx* ctx, srcnn_mem in, srcnn_mem out, srcnn_mem W, srcnn_mem B,
                        int k, int n, int f, int skip_relu, int in_w, int in_h, int S) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(k > 0 && n > 0 && f > 0 && S > 0, "bad layer shape k=%d n=%d f=%d S=%d", k, n, f, S);
  SRCNN_REQUIRE(in_w >= f && in_h >= f, "input %dx%d smaller than filter %d", in_w, in_h, f);
  const int ow = in_w - f + 1, oh = in_h - f + 1;
  const float *pin, *pW, *pB;
  float* pout;
  SRCNN_TRY(resolve(ctx, in, sizeof(float) * (size_t)S * in_w * in_h * k, &pin, "layer input"));
  SRCNN_TRY(resolve(ctx, out, sizeof(float) * (size_t)S * ow * oh * n, &pout, "layer output"));
  ctx->note_write(out);
  SRCNN_TRY(resolve(ctx, W, sizeof(float) * (size_t)f * f * k * n, &pW, "weights"));
  SRCNN_TRY(resolve(ctx, B, sizeof(float) * (size_t)n, &pB, "bias"));
  LaunchScope scope(ctx, SRCNN_K_FORWARD);
  {
    const Allocation* wa = ctx->get(W);
    const int rc5 = fast::conv5_forward(ctx, pin, pout, pW, pB, k, n, f, !skip_relu, in_w, in_h, S,
                                        W, wa && wa->owned && !wa->exposed,
                                        ctx->c5_l1_max_of == pin);
    if (rc5 < 0) return rc5;
    if (rc5 > 0) {
      return check_launch("forward(conv5 tc)");   // (absmax / image kernels count themselves)
    }
  }
  if (fast::forward_layer(ctx, pin, pout, pW, pB, k, n, f, !skip_relu, in_w, in_h, S))
    return check_launch("forward(fast)");
  generic::FwdArgs a{pin, pout, pW, pB, k, n, f, skip_relu ? 0 : 1, in_w, in_h, ow, oh, S};
  const long long M = (long long)S * ow * oh;
  dim3 grid((unsigned)((M + generic::TM - 1) / generic::TM), (n + generic::TN - 1) / generic::TN);
  generic::forward_gemm_kernel<<<grid, generic::NT, 0, ctx->stream>>>(a);
  return check_launch("forward");
}

int srcnn_squared_error(srcnn_ctx* ctx, srcnn_mem gt, srcnn_mem algo, srcnn_mem target,
                        int gt_w, int gt_h, int algo_w, int algo_h, int S) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(S > 0 && algo_w > 0 && algo_h > 0 && gt_w >= algo_w && gt_h >= algo_h,
                "bad squared_error dimensions");
  const float *pgt, *palgo;
  float* pt;
  SRCNN_TRY(resolve(ctx, gt, sizeof(float) * (size_t)S * gt_w * gt_h, &pgt, "ground truth"));
  SRCNN_TRY(resolve(ctx, algo, sizeof(float) * (size_t)S * algo_w * algo_h, &palgo, "algo result"));
  SRCNN_TRY(resolve(ctx, target, sizeof(float), &pt, "squared error target"));
  ctx->note_write(target);
  const size_t total = (size_t)S * algo_w * algo_h;
  const int blocks = grid_1d(total, generic::RED_THREADS, generic::RED_MAX_BLOCKS);
  LaunchScope scope(ctx, SRCNN_K_SQUARED_ERR, 2);
  generic::squared_error_stage1<<<blocks, generic::RED_THREADS, 0, ctx->stream>>>(
      pgt, palgo, (double*)ctx->red_scratch, gt_w, gt_h, algo_w, algo_h, S);
  generic::reduce_stage2<<<1, generic::RED_THREADS, 0, ctx->stream>>>(
      (const double*)ctx->red_scratch, blocks, pt);
  return check_launch("squared_err");
}

int srcnn_last_layer_delta(srcnn_ctx* ctx, srcnn_mem gt, srcnn_mem algo, srcnn_mem target,
                           int gt_w, int gt_h, int algo_w, int algo_h, int S) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(S > 0 && algo_w > 0 && algo_h > 0 && gt_w >= algo_w && gt_h >= algo_h,
                "bad last_layer_delta dimensions");
  const float *pgt, *palgo;
  float* pt;
  const size_t total = (size_t)S * algo_w * algo_h;
  SRCNN_TRY(resolve(ctx, gt, sizeof(float) * (size_t)S * gt_w * gt_h, &pgt, "ground truth"));
  SRCNN_TRY(resolve(ctx, algo, sizeof(float) * total, &palgo, "algo result"));
  SRCNN_TRY(resolve(ctx, target, sizeof(float) * total, &pt, "last layer delta target"));
  ctx->note_write(target);
  LaunchScope scope(ctx, SRCNN_K_LAST_LAYER_DELTA);
  generic::last_layer_delta_kernel<<<grid_1d(total, 256, 8 * ctx->sm_count), 256, 0, ctx->stream>>>(
      pgt, palgo, pt, gt_w, gt_h, algo_w, algo_h, S);
  return check_launch("last_layer_delta");
}

int srcnn_deltas(srcnn_ctx* ctx, srcnn_mem deltas_next, srcnn_mem layer_output,
                 srcnn_mem target, srcnn_mem W, int n_curr, int f_next, int n_next, int out_w,
                 int out_h, int S) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(n_curr > 0 && f_next > 0 && n_next > 0 && S > 0, "bad deltas shape");
  SRCNN_REQUIRE(out_w >= f_next && out_h >= f_next, "layer output smaller than next filter");
  const int nw = out_w - f_next + 1, nh = out_h - f_next + 1;
  const float *pdn, *plo, *pW;
  float* pt;
  const size_t cur = (size_t)S * out_w * out_h * n_curr;
  SRCNN_TRY(resolve(ctx, deltas_next, sizeof(float) * (size_t)S * nw * nh * n_next, &pdn, "next layer deltas"));
  SRCNN_TRY(resolve(ctx, layer_output, sizeof(float) * cur, &plo, "layer output"));
  SRCNN_TRY(resolve(ctx, target, sizeof(float) * cur, &pt, "deltas target"));
  ctx->note_write(target);
  SRCNN_TRY(resolve(ctx, W, sizeof(float) * (size_t)f_next * f_next * n_curr * n_next, &pW, "next layer weights"));
  LaunchScope scope(ctx, SRCNN_K_DELTAS);
  {
    const Allocation* wa = ctx->get(W);
    const int rc5 = fast::conv5_deltas(ctx, pdn, plo, pt, pW, n_curr, f_next, n_next, out_w, out_h,
                                       S, W, wa && wa->owned && !wa->exposed);
    if (rc5 < 0) return rc5;
    if (rc5 > 0) return check_launch("deltas(conv5 tc)");
  }
  if (fast::deltas(ctx, pdn, plo, pt, pW, n_curr, f_next, n_next, out_w, out_h, S))
    return check_launch("deltas(fast)");
  generic::DeltaArgs a{pdn, plo, pt, pW, n_curr, f_next, n_next, out_w, out_h, nw, nh, S};
  const long long M = (long long)S * out_w * out_h;
  dim3 grid((unsigned)((M + generic::TM - 1) / generic::TM), (n_curr + generic::TN - 1) / generic::TN);
  generic::deltas_gemm_kernel<<<grid, generic::NT, 0, ctx->stream>>>(a);
  return check_launch("deltas");
}

int srcnn_backpropagate(srcnn_ctx* ctx, srcnn_mem deltas, srcnn_mem layer_input,
                        srcnn_mem grad_w, srcnn_mem grad_b, int n, int k, int f, int out_w,
                        int out_h, int S) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(n > 0 && k > 0 && f > 0 && S > 0 && out_w > 0 && out_h > 0, "bad backpropagate shape");
  const int iw = out_w + f - 1, ih = out_h + f - 1;
  const float *pd, *pin;
  float *pgw, *pgb;
  SRCNN_TRY(resolve(ctx, deltas, sizeof(float) * (size_t)S * out_w * out_h * n, &pd, "layer deltas"));
  SRCNN_TRY(resolve(ctx, layer_input, sizeof(float) * (size_t)S * iw * ih * k, &pin, "layer input"));
  SRCNN_TRY(resolve(ctx, grad_w, sizeof(float) * (size_t)f * f * k * n, &pgw, "grad_w"));
  SRCNN_TRY(resolve(ctx, grad_b, sizeof(float) * (size_t)n, &pgb, "grad_b"));
  ctx->note_write(grad_w);
  ctx->note_write(grad_b);
  LaunchScope scope(ctx, SRCNN_K_BACKPROPAGATE, 2);
  int rc_fast = fast::backpropagate(ctx, pd, pin, pgw, pgb, n, k, f, out_w, out_h, S,
                                    ctx->c5_maxes_known && ctx->c5_max_out1_of == pin &&
                                        ctx->c5_max_d2_of == pd);
  if (rc_fast < 0) return rc_fast;
  if (rc_fast > 0) return check_launch("backpropagate(fast)");
  const int Mw = f * f * k, M = Mw + 1;
  const long long P = (long long)S * out_w * out_h;
  const int mt = (M + generic::TM - 1) / generic::TM, nt = (n + generic::TN - 1) / generic::TN;
  // split the pixel (reduction) dimension so the grid fills the GPU ~2x, at least 256
  // pixels per split
  long long splits = std::max<long long>(1, (2LL * ctx->sm_count) / std::max(1, mt * nt));
  splits = std::min<long long>(splits, std::max<long long>(1, P / 256));
  long long pps = (P + splits - 1) / splits;
  pps = (pps + generic::KC - 1) / generic::KC * generic::KC;
  splits = (P + pps - 1) / pps;
  SRCNN_TRY(ensure_scratch(ctx, &ctx->splitk_scratch, &ctx->splitk_bytes,
                           sizeof(float) * (size_t)splits * M * n));
  generic::BpArgs a{pd, pin, (float*)ctx->splitk_scratch, n, k, f, out_w, out_h, iw, ih, S, pps};
  dim3 grid(mt, nt, (unsigned)splits);
  generic::backprop_gemm_kernel<<<grid, generic::NT, 0, ctx->stream>>>(a);
  generic::backprop_reduce_kernel<<<(M * n + 255) / 256, 256, 0, ctx->stream>>>(
      (const float*)ctx->splitk_scratch, pgw, pgb, Mw, n, (int)splits);
  return check_launch("backpropagate");
}

int srcnn_update_params(srcnn_ctx* ctx, srcnn_mem w, srcnn_mem b, srcnn_mem grad_w,
                        srcnn_mem grad_b, srcnn_mem prev_dw, srcnn_mem prev_db, float momentum,
                        float weight_decay, float learning_rate, unsigned batch_size,
                        unsigned weights_size, unsigned bias_size) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(batch_size > 0, "batch_size must be > 0");
  float *pw, *pb, *ppw, *ppb;
  const float *pgw, *pgb;
  const size_t wb = sizeof(float) * (size_t)weights_size, bb = sizeof(float) * (size_t)bias_size;
  SRCNN_TRY(resolve(ctx, w, wb, &pw, "weights"));
  SRCNN_TRY(resolve(ctx, b, bb, &pb, "bias"));
  SRCNN_TRY(resolve(ctx, grad_w, wb, &pgw, "grad_w"));
  SRCNN_TRY(resolve(ctx, grad_b, bb, &pgb, "grad_b"));
  SRCNN_TRY(resolve(ctx, prev_dw, wb, &ppw, "previous delta w"));
  SRCNN_TRY(resolve(ctx, prev_db, bb, &ppb, "previous delta b"));
  ctx->note_write(w);
  ctx->note_write(b);
  ctx->note_write(prev_dw);
  ctx->note_write(prev_db);
  if (weights_size == 0 && bias_size == 0) return SRCNN_OK;   // nothing to update
  const unsigned total = std::max(weights_size, bias_size);
  LaunchScope scope(ctx, SRCNN_K_UPDATE_PARAMS);
  generic::update_params_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(
      pw, pb, pgw, pgb, ppw, ppb, momentum, weight_decay, learning_rate, batch_size,
      weights_size, bias_size);
  return check_launch("update_params");
}

int srcnn_sum(srcnn_ctx* ctx, srcnn_mem data, unsigned len, int squared, srcnn_mem target) {
  SRCNN_ENTER(ctx);
  const float* pd;
  float* pt;
  SRCNN_TRY(resolve(ctx, data, sizeof(float) * (size_t)len, &pd, "sum data"));
  SRCNN_TRY(resolve(ctx, target, sizeof(float), &pt, "sum target"));
  ctx->note_write(target);
  const int blocks = grid_1d(len, generic::RED_THREADS, generic::RED_MAX_BLOCKS);
  LaunchScope scope(ctx, SRCNN_K_SUM, 2);
  generic::sum_stage1<<<blocks, generic::RED_THREADS, 0, ctx->stream>>>(
      pd, (double*)ctx->red_scratch, len, squared);
  generic::reduce_stage2<<<1, generic::RED_THREADS, 0, ctx->stream>>>(
      (const double*)ctx->red_scratch, blocks, pt);
  return check_launch("sum");
}

int srcnn_sub_from_all(srcnn_ctx* ctx, srcnn_mem data, float value, unsigned len) {
  SRCNN_ENTER(ctx);
  float* pd;
  SRCNN_TRY(resolve(ctx, data, sizeof(float) * (size_t)len, &pd, "sub_from_all data"));
  ctx->note_write(data);
  if (len == 0) return SRCNN_OK;
  LaunchScope scope(ctx, SRCNN_K_SUB_FROM_ALL);
  generic::sub_from_all_kernel<<<grid_1d(len, 256, 8 * ctx->sm_count), 256, 0, ctx->stream>>>(
      pd, value, len);
  return check_launch("sub_from_all");
}

int srcnn_extract_luma(srcnn_ctx* ctx, srcnn_mem rgba, srcnn_mem target, int w, int h,
                       int normalize) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(w > 0 && h > 0, "bad image size");
  const uchar4* pi;
  float* pt;
  SRCNN_TRY(resolve(ctx, rgba, (size_t)w * h * 4, &pi, "rgba image"));
  SRCNN_TRY(resolve(ctx, target, sizeof(float) * (size_t)w * h, &pt, "luma target"));
  ctx->note_write(target);
  LaunchScope scope(ctx, SRCNN_K_EXTRACT_LUMA);
  const size_t npx = (size_t)w * h;
  SRCNN_REQUIRE(npx < ((size_t)1 << 31), "image of %dx%d pixels is too large for one launch", w, h);
  generic::extract_luma_kernel<<<(unsigned)((npx + 255) / 256), 256, 0, ctx->stream>>>(
      pi, pt, (int)npx, normalize);
  return check_launch("extract_luma");
}

int srcnn_swap_luma(srcnn_ctx* ctx, srcnn_mem rgba, srcnn_mem new_luma, srcnn_mem target,
                    int gt_w, int gt_h, int luma_w, int luma_h) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(gt_w > 0 && gt_h > 0 && luma_w > 0 && luma_h > 0 && luma_w <= gt_w && luma_h <= gt_h,
                "bad swap_luma dimensions");
  const uchar4* pi;
  const float* pl;
  unsigned char* pt;
  SRCNN_TRY(resolve(ctx, rgba, (size_t)gt_w * gt_h * 4, &pi, "rgba image"));
  SRCNN_TRY(resolve(ctx, new_luma, sizeof(float) * (size_t)luma_w * luma_h, &pl, "new luma"));
  SRCNN_TRY(resolve(ctx, target, (size_t)gt_w * gt_h * 3, &pt, "rgb target"));
  ctx->note_write(target);
  LaunchScope scope(ctx, SRCNN_K_SWAP_LUMA);
  dim3 block(32, 8), grid((gt_w + 31) / 32, (gt_h + 7) / 8);
  generic::swap_luma_kernel<<<grid, block, 0, ctx->stream>>>(pi, pl, pt, gt_w, gt_h, 0, gt_h,
                                                             luma_w, luma_h);
  return check_launch("swap_luma");
}

int srcnn_resample(srcnn_ctx* ctx, srcnn_mem rgba_in, int w, int h, srcnn_mem rgba_out,
                   srcnn_mem luma_out, int out_w, int out_h, int filter) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_resample(w, h, out_w, out_h, filter));
  const uchar4* pi;
  uchar4* po;
  float* pl = nullptr;
  const size_t npx = (size_t)out_w * out_h;
  SRCNN_TRY(resolve(ctx, rgba_in, (size_t)w * h * 4, &pi, "rgba input"));
  SRCNN_TRY(resolve(ctx, rgba_out, npx * 4, &po, "rgba output"));
  if (luma_out != SRCNN_NULL_MEM) {
    SRCNN_TRY(resolve(ctx, luma_out, sizeof(float) * npx, &pl, "luma output"));
    ctx->note_write(luma_out);
  }
  ctx->note_write(rgba_out);
  const int* tab;
  int rows_max;
  SRCNN_TRY(resample::table_for(ctx, w, h, out_w, out_h, filter, SRCNN_CHROMA_CENTER,
                                SRCNN_CHROMA_CENTER, &tab, &rows_max));
  LaunchScope scope(ctx, SRCNN_K_RESAMPLE);
  SRCNN_TRY(resample::launch(ctx, pi, w, h, po, pl, out_w, out_h, filter, tab, rows_max));
  return check_launch("resample");
}

int srcnn_image_quality(srcnn_ctx* ctx, srcnn_mem result, int result_bpp, srcnn_mem reference,
                        int w, int h, int S, int border, srcnn_mem out) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(w > 0 && h > 0 && S > 0 && S <= 65535, "bad image set: %d frames of %dx%d", S, w, h);
  SRCNN_REQUIRE(result_bpp == 3 || result_bpp == 4, "result_bpp must be 3 or 4, got %d", result_bpp);
  SRCNN_TRY(check_quality_region(w, h, border));
  const size_t npx = (size_t)w * h * S;
  const unsigned char* pr;
  const uchar4* pref;
  double* po;
  SRCNN_TRY(resolve(ctx, result, npx * result_bpp, &pr, "result images"));
  SRCNN_TRY(resolve(ctx, reference, npx * 4, &pref, "reference images"));
  SRCNN_TRY(resolve(ctx, out, sizeof(double) * 2 * (size_t)S, &po, "quality output"));
  ctx->note_write(out);
  SRCNN_TRY(ensure_scratch(ctx, &ctx->quality_red, &ctx->quality_red_bytes,
                           quality::partial_bytes(w, h, border, S)));
  LaunchScope scope(ctx, SRCNN_K_QUALITY, 2);
  quality::launch(ctx, pr, result_bpp, pref, w, h, S, border, (double2*)ctx->quality_red, po, 2);
  return check_launch("image_quality");
}

// ======================================================================= fused hot path

namespace {
// true when the six parameter buffers are context-owned allocations (nothing outside this
// library can write them, so ctx->write_gen tells whether they may have changed)
bool params_owned(srcnn_ctx* ctx, const srcnn_net* net) {
  for (int l = 0; l < 3; l++) {
    const Allocation* w = ctx->get(net->w[l]);
    const Allocation* b = ctx->get(net->b[l]);
    if (!w || !b || !w->owned || !b->owned || w->exposed || b->exposed) return false;
  }
  return true;
}

// `net` for the fused kernels: its six parameter buffers resolved and, when it has a fused
// forward, their prepared operand image (from the context's cache while the six buffers are
// untouched, context-owned and never exposed; else packed afresh)
int fused_net(srcnn_ctx* ctx, const srcnn_net* net, fast::FusedNet* fn) {
  *fn = fast::FusedNet{net->n1, net->n2, net->f1, net->f2, net->f3};
  SRCNN_TRY(resolve(ctx, net->w[0], sizeof(float) * (size_t)net->f1 * net->f1 * net->n1, &fn->w1, "w1"));
  SRCNN_TRY(resolve(ctx, net->b[0], sizeof(float) * (size_t)net->n1, &fn->b1, "b1"));
  SRCNN_TRY(resolve(ctx, net->w[1], sizeof(float) * (size_t)net->f2 * net->f2 * net->n1 * net->n2, &fn->w2, "w2"));
  SRCNN_TRY(resolve(ctx, net->b[1], sizeof(float) * (size_t)net->n2, &fn->b2, "b2"));
  SRCNN_TRY(resolve(ctx, net->w[2], sizeof(float) * (size_t)net->f3 * net->f3 * net->n2, &fn->w3, "w3"));
  SRCNN_TRY(resolve(ctx, net->b[2], sizeof(float), &fn->b3, "b3"));
  if (!fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3)) return SRCNN_OK;
  SRCNN_TRY(fast::fused_prepare(ctx, *fn, params_owned(ctx, net), &fn->scales));
  for (int l = 0; l < 3; l++) {
    ctx->hp_cache_h[2 * l] = net->w[l];
    ctx->hp_cache_h[2 * l + 1] = net->b[l];
  }
  return SRCNN_OK;
}

// one fused forward on the context stream
int launch_fused(srcnn_ctx* ctx, const fast::FusedNet& fn, const float* in, float* out, int in_w,
                 int in_h, int S) {
  LaunchScope scope(ctx, SRCNN_K_FORWARD_FUSED, fast::fused_launches(ctx, fn));
  SRCNN_TRY(fast::forward_fused(ctx, fn, in, out, in_w, in_h, S));
  return check_launch("forward_fused");
}

// points the context stream (which the launch helpers and the profile timers use) at `s` for the
// lifetime of the object
struct StreamSwap {
  srcnn_ctx* ctx;
  cudaStream_t saved;
  StreamSwap(srcnn_ctx* c, cudaStream_t s) : ctx(c), saved(c->stream) { c->stream = s; }
  ~StreamSwap() { ctx->stream = saved; }
};

// the copy-in / copy-out / second compute stream and the events of the pipelined host-buffer
// entries (created on first use)
int ensure_side_streams(srcnn_ctx* ctx) {
  if (ctx->copy_in) return SRCNN_OK;
  SRCNN_CUDA(cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
  SRCNN_CUDA(cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
  SRCNN_CUDA(cudaStreamCreateWithFlags(&ctx->compute2, cudaStreamNonBlocking));
  for (int i = 0; i < srcnn_ctx::kEvents; i++) {
    SRCNN_CUDA(cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming));
    SRCNN_CUDA(cudaEventCreateWithFlags(&ctx->ev_k[i], cudaEventDisableTiming));
  }
  for (int i = 0; i < 4; i++)
    SRCNN_CUDA(cudaEventCreateWithFlags(&ctx->ev_d[i], cudaEventDisableTiming));
  return SRCNN_OK;
}

// drops the handles a scope appended to the table (wrapped views of a workspace, staging
// buffers) on EVERY exit path, so that errors do not grow the table
struct TableScope {
  srcnn_ctx* ctx;
  size_t size;
  explicit TableScope(srcnn_ctx* c) : ctx(c), size(c->allocs.size()) {}
  ~TableScope() {
    if (ctx->allocs.size() > size) ctx->allocs.resize(size);
  }
};
}  // namespace

#ifdef HP_PROF
// kernel-development aid (never in the product build): the hand-off wait counters of the fused
// inference kernel, [32 warps][total, wait0, wait1, tiles]
int srcnn_debug_hp_prof(unsigned* out) {
  return cudaMemcpyFromSymbol(out, srcnn::fused_hp::hp_prof, 32 * 4 * sizeof(unsigned)) == cudaSuccess
             ? SRCNN_OK : SRCNN_ECUDA;
}
#endif

int srcnn_invalidate_params(srcnn_ctx* ctx) {
  SRCNN_ENTER(ctx);
  ctx->write_gen++;
  ctx->hp_cache_valid = false;
  ctx->c5_valid = false;
  return SRCNN_OK;
}

int srcnn_forward_fused_supported(const srcnn_net* net) {
  if (!net) return 0;
  return fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3) ? 1 : 0;
}

int srcnn_forward_fused(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem out,
                        int in_w, int in_h, int S, srcnn_mem scratch1, srcnn_mem scratch2) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, in_w, in_h);
  SRCNN_REQUIRE(S > 0 && d.w3 > 0 && d.h3 > 0, "image %dx%d too small for the network", in_w, in_h);
  if (fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3)) {
    const float* pin;
    float* pout;
    SRCNN_TRY(resolve(ctx, in, sizeof(float) * (size_t)S * in_w * in_h, &pin, "input luma"));
    SRCNN_TRY(resolve(ctx, out, sizeof(float) * (size_t)S * d.w3 * d.h3, &pout, "output luma"));
    ctx->note_write(out);   // before the operand image: `out` may be a parameter buffer
    fast::FusedNet fn;
    SRCNN_TRY(fused_net(ctx, net, &fn));
    return launch_fused(ctx, fn, pin, pout, in_w, in_h, S);
  }
  SRCNN_REQUIRE(scratch1 != SRCNN_NULL_MEM && scratch2 != SRCNN_NULL_MEM,
                "no fused kernel for %d-%d-%d n1=%d n2=%d and no scratch buffers for the "
                "three-launch path", net->f1, net->f2, net->f3, net->n1, net->n2);
  SRCNN_TRY(srcnn_forward_layer(ctx, in, scratch1, net->w[0], net->b[0], 1, net->n1, net->f1, 0,
                                in_w, in_h, S));
  SRCNN_TRY(srcnn_forward_layer(ctx, scratch1, scratch2, net->w[1], net->b[1], net->n1, net->n2,
                                net->f2, 0, d.w1, d.h1, S));
  return srcnn_forward_layer(ctx, scratch2, out, net->w[2], net->b[2], net->n2, 1, net->f3, 1,
                             d.w2, d.h2, S);
}

namespace {
constexpr int kMaxSub = srcnn_ctx::kEvents;

// The sub-band cut of a band of `band_out_h` output rows: sub-band i is the band-relative output
// rows [sub_r0[i], sub_r0[i + 1]); returns the count (1 below 256 rows).
int subband_rows(int band_out_h, int sub_r0[kMaxSub + 1]) {
  // SRCNN_E2E_SUBBANDS=n (2..32) / SRCNN_E2E_RAMPCAP=c override the defaults for experiments.
  // Measured on C3 (PCIe gen5 x16, 55 GB/s each way, 47.6 with both directions busy), wall
  // clock of the call with the 0.9 ms kernel: 12 sub-bands 1.84-1.88 ms, 14: 1.78, 16: 1.73-1.78,
  // 18: 1.78, 20 (cap 3): 1.79, 24: 1.83, 32: 1.96; ramp cap 3 / 5 / 6 at 16: 1.78 / 1.83 / 1.79.
  static const int kSubDefault = std::getenv("SRCNN_E2E_SUBBANDS") ? std::atoi(std::getenv("SRCNN_E2E_SUBBANDS")) : 16;
  // bands of a multi-GPU partition are pipelined too (an 8-way split of C3 leaves 511 rows per
  // rank, and with 8 ranks copying at once each gets ~18 GB/s of the host's pinned-copy rate, so
  // the copies dominate even more): about one sub-band per 64 output rows, at most the default
  const int n_sub = band_out_h >= 256
                  ? std::min(std::min(std::max(kSubDefault, 2), kMaxSub), std::max(2, band_out_h / 64))
                  : 1;
  sub_r0[0] = 0;
  {
    // shares ramp up from a small first sub-band and down to a small last one: 1,2,3,..,3,2,1
    // capped at 2 units (round-2 sweep, profiles/r2g_e2e_subband_sweep.txt: cap 2 / 4 / 8 at 16
    // sub-bands: 1.69 / 1.77 / 1.86 ms); the exposed head upload / tail download shrink with them
    float unit[kMaxSub], total = 0.f;
    for (int i = 0; i < n_sub; i++) {
      static const int kRampCap = std::getenv("SRCNN_E2E_RAMPCAP") ? std::atoi(std::getenv("SRCNN_E2E_RAMPCAP")) : 2;
      unit[i] = (float)std::min(std::min(i + 1, n_sub - i), std::max(kRampCap, 1));
      total += unit[i];
    }
    float acc = 0.f;
    for (int i = 0; i < n_sub; i++) {
      acc += unit[i];
      sub_r0[i + 1] = i + 1 == n_sub ? band_out_h : std::min((int)(acc / total * band_out_h + 0.5f), band_out_h);
    }
    if (n_sub == 1) sub_r0[1] = band_out_h;
  }
  return n_sub;
}

// ---- the captured sub-band pipelines (srcnn_infer_rows_host, srcnn_upscale_image_host) -------
// The pipelines are ~10 runtime calls per sub-band; issued one by one the host only just stays
// ahead of the GPU (and falls behind when another thread competes for the CPU), so each is
// captured once into a CUDA graph and replayed with one launch while the arguments repeat
// (SRCNN_E2E_GRAPH=0 disables; profile mode times individual launches and never captures).
bool graphs_enabled(const srcnn_ctx* ctx) {
  static const bool kGraphs = !(std::getenv("SRCNN_E2E_GRAPH") && std::atoi(std::getenv("SRCNN_E2E_GRAPH")) == 0);
  return kGraphs && !ctx->profile;
}

// one route's graph, the arguments it was captured for, and its launches per kernel id
struct GraphSlot {
  cudaGraphExec_t* graph;
  unsigned long long* key;   // [srcnn_ctx::kGraphKey]
  unsigned* launches;        // [SRCNN_K_COUNT]
};

// drops the slot's old graph and starts capturing the context stream
int graph_begin(srcnn_ctx* ctx, const GraphSlot& g) {
  if (*g.graph) {
    SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));   // the old graph may still be running
    cudaGraphExecDestroy(*g.graph);
    *g.graph = nullptr;
  }
  if (!ctx->ev_join[0])
    for (int i = 0; i < 2; i++)
      SRCNN_CUDA(cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming));
  {   // everything the launches allocate lazily must exist before the capture starts
    fused_hp::Scales* s_;
    unsigned* w_;
    SRCNN_TRY(fused_hp::scale_slot(ctx, &s_, &w_));
  }
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(ctx->stream, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
    cudaGraph_t stale = nullptr;   // a capture an earlier failed call left open
    cudaStreamEndCapture(ctx->stream, &stale);
    if (stale) cudaGraphDestroy(stale);
    cudaGetLastError();
  }
  SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  SRCNN_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed));
  return SRCNN_OK;
}

// ends (and discards) an open capture on every early exit, so that a failed call never leaves
// the context stream and the side streams capturing
struct CaptureGuard {
  cudaStream_t s;
  bool active;
  ~CaptureGuard() {
    if (!active) return;
    cudaGraph_t g = nullptr;
    cudaStreamEndCapture(s, &g);
    if (g) cudaGraphDestroy(g);
    cudaGetLastError();
  }
};

// One call of a sub-band pipeline (srcnn_infer_rows_host, srcnn_upscale_image_host): `head`
// (optional) on the context stream; then for every sub-band i of output rows
// [sub_r0[i], sub_r0[i + 1]), `upload` (optional) on the copy-in stream, `work` on the context
// stream or the second compute stream (alternately, so that the tail wave of one sub-band overlaps
// the head of the next) and `download` on the copy-out stream.  Captured into `slot`'s graph and
// replayed while `key` repeats.  `block`: return when the downloads are complete (the route
// without graphs always does: its side streams and events are shared).
int run_subbands(srcnn_ctx* ctx, const GraphSlot& slot, const unsigned long long* key,
                 const int* sub_r0, int n_sub, bool block, const std::function<int()>& head,
                 const std::function<cudaError_t(int i, int r0, int r1)>& upload,
                 const std::function<int(int i, int r0, int r1)>& work,
                 const std::function<cudaError_t(int i, int r0, int r1)>& download) {
  SRCNN_TRY(ensure_side_streams(ctx));
  const bool use_graph = graphs_enabled(ctx);
  const size_t key_bytes = sizeof(unsigned long long) * srcnn_ctx::kGraphKey;
  if (use_graph && *slot.graph && std::memcmp(key, slot.key, key_bytes) == 0) {
    for (int i = 0; i < SRCNN_K_COUNT; i++) {
      ctx->launch_count += slot.launches[i];
      ctx->stats[i].launches += slot.launches[i];
    }
    SRCNN_CUDA(cudaGraphLaunch(*slot.graph, ctx->stream));
    if (block) SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
    return SRCNN_OK;
  }
  if (use_graph) SRCNN_TRY(graph_begin(ctx, slot));
  CaptureGuard capture{ctx->stream, use_graph};
  uint64_t before[SRCNN_K_COUNT];   // the launch counters when the capture started
  for (int i = 0; i < SRCNN_K_COUNT; i++) before[i] = ctx->stats[i].launches;
  cudaStream_t main_stream = ctx->stream;
  int rc = head ? head() : SRCNN_OK;
  if (rc == SRCNN_OK) {
    // order the side streams after whatever the context stream was doing with the buffers (the
    // copy-in stream only when it has work: the capture joins back the other two only)
    SRCNN_CUDA(cudaEventRecord(ctx->ev_k[0], main_stream));
    if (upload) SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[0], 0));
    SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[0], 0));
    SRCNN_CUDA(cudaStreamWaitEvent(ctx->compute2, ctx->ev_k[0], 0));
  }
  for (int i = 0; i < n_sub && rc == SRCNN_OK; i++) {
    const int r0 = sub_r0[i], r1 = sub_r0[i + 1];
    if (r1 <= r0) continue;
    cudaStream_t cs = (i & 1) ? ctx->compute2 : main_stream;
    if (upload) {
      SRCNN_CUDA(upload(i, r0, r1));
      SRCNN_CUDA(cudaEventRecord(ctx->ev_in[i], ctx->copy_in));
      SRCNN_CUDA(cudaStreamWaitEvent(cs, ctx->ev_in[i], 0));
    }
    {
      StreamSwap on(ctx, cs);
      rc = work(i, r0, r1);
    }
    if (rc != SRCNN_OK) break;
    SRCNN_CUDA(cudaEventRecord(ctx->ev_k[i], cs));
    SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[i], 0));
    SRCNN_CUDA(download(i, r0, r1));
  }
  if (!use_graph) {
    SRCNN_CUDA(cudaStreamSynchronize(ctx->copy_out));
    SRCNN_CUDA(cudaStreamSynchronize(ctx->compute2));
    SRCNN_CUDA(cudaStreamSynchronize(main_stream));
    return rc;
  }
  // join the side streams back into the capturing stream, instantiate the graph into the slot
  // and launch it once
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaEventRecord(ctx->ev_join[0], ctx->copy_out);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(main_stream, ctx->ev_join[0], 0);
  if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_join[1], ctx->compute2);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(main_stream, ctx->ev_join[1], 0);
  const cudaError_t e2 = cudaStreamEndCapture(main_stream, &graph);
  capture.active = false;
  if (e == cudaSuccess) e = e2;
  if (rc == SRCNN_OK && e == cudaSuccess) e = cudaGraphInstantiate(slot.graph, graph, 0);
  if (graph) cudaGraphDestroy(graph);
  if (rc != SRCNN_OK) return rc;
  if (e != cudaSuccess) {
    *slot.graph = nullptr;
    return fail(SRCNN_ECUDA, "capturing the sub-band pipeline failed: %s", cudaGetErrorString(e));
  }
  std::memcpy(slot.key, key, key_bytes);
  for (int i = 0; i < SRCNN_K_COUNT; i++)
    slot.launches[i] = (unsigned)(ctx->stats[i].launches - before[i]);
  SRCNN_CUDA(cudaGraphLaunch(*slot.graph, main_stream));
  if (block) SRCNN_CUDA(cudaStreamSynchronize(main_stream));
  return SRCNN_OK;
}

// lane < 0: the blocking call (context stream, returns when host_out is complete);
// lane 0 / 1: srcnn_infer_rows_host_async (that lane's stream, staging and graph; no wait)
int infer_rows_host_impl(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in, int in_w,
                         int in_h, int out_row0, int out_row1, float* host_out, int lane) {
  SRCNN_REQUIRE(ctx && host_in && host_out, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, in_w, in_h);
  SRCNN_REQUIRE(d.w3 > 0 && d.h3 > 0, "image %dx%d too small for the network", in_w, in_h);
  SRCNN_REQUIRE(out_row0 >= 0 && out_row0 < out_row1 && out_row1 <= d.h3,
                "bad output row band [%d,%d) of %d", out_row0, out_row1, d.h3);
  const int halo = net->f1 + net->f2 + net->f3 - 3;
  const int band_out_h = out_row1 - out_row0, band_in_h = band_out_h + halo;
  const size_t in_bytes = sizeof(float) * (size_t)band_in_h * in_w;
  const size_t out_bytes = sizeof(float) * (size_t)band_out_h * d.w3;
  // the state of this call's route: the blocking call's staging / graph, or a lane's
  const bool async = lane >= 0;
  srcnn_ctx::RowsLane* ln = async ? &ctx->lanes[lane] : nullptr;
  void** st_in = async ? &ln->in : &ctx->band_in;
  void** st_out = async ? &ln->out : &ctx->band_out;
  const GraphSlot slot = async ? GraphSlot{&ln->graph, ln->key, ln->graph_launches}
                               : GraphSlot{&ctx->e2e_graph, ctx->e2e_key, ctx->e2e_graph_launches};
  if (!async) SRCNN_CUDA(ctx->drain_lanes());   // "returns when done" covers earlier async calls
  SRCNN_TRY(ensure_scratch(ctx, st_in, async ? &ln->in_bytes : &ctx->band_in_bytes, in_bytes));
  SRCNN_TRY(ensure_scratch(ctx, st_out, async ? &ln->out_bytes : &ctx->band_out_bytes, out_bytes));
  // one set of operand scales for all sub-bands (computed on the context stream, before the
  // event the side streams wait for)
  fast::FusedNet fn;
  SRCNN_TRY(fused_net(ctx, net, &fn));
  SRCNN_REQUIRE(fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3),
                "srcnn_infer_rows_host needs a fused instantiation for %d-%d-%d n1=%d n2=%d",
                net->f1, net->f2, net->f3, net->n1, net->n2);
  // The band is cut into sub-bands; upload, fused forward and download of consecutive sub-bands
  // overlap, so a large image costs ~max(H2D, compute, D2H) + a short head and tail instead of
  // their sum: the first and the last sub-band are small because their upload / download is
  // exposed.  Every sub-band is the same valid-convolution problem with a halo, so the result is
  // bit-identical to a single launch.
  int sub_r0[kMaxSub + 1];
  const int n_sub = subband_rows(band_out_h, sub_r0);
  float* din = (float*)*st_in;
  float* dout = (float*)*st_out;
  // an asynchronous call runs on its lane's stream, behind whatever the context stream has
  // queued so far (the operand image above, parameter updates)
  if (async) {
    if (!ln->stream) SRCNN_CUDA(cudaStreamCreateWithFlags(&ln->stream, cudaStreamNonBlocking));
    if (!ctx->lane_ev) SRCNN_CUDA(cudaEventCreateWithFlags(&ctx->lane_ev, cudaEventDisableTiming));
    SRCNN_CUDA(cudaEventRecord(ctx->lane_ev, ctx->stream));
    SRCNN_CUDA(cudaStreamWaitEvent(ln->stream, ctx->lane_ev, 0));
    // (Ordering the two calls stage by stage -- this call's uploads behind the other lane's last
    // upload, through an external event-record node in the graph -- was measured SLOWER than
    // letting them share the copy engines: 1.83 vs 1.67 ms per 4096x4096 image.)
    ctx->lanes_busy = true;
    for (int l = 0; l < 3; l++) {
      ln->params[2 * l] = net->w[l];
      ln->params[2 * l + 1] = net->b[l];
    }
  }
  StreamSwap on_lane(ctx, async ? ln->stream : ctx->stream);
  if (n_sub == 1) {
    SRCNN_CUDA(cudaMemcpyAsync(din, host_in + (size_t)out_row0 * in_w, in_bytes,
                               cudaMemcpyHostToDevice, ctx->stream));
    SRCNN_TRY(launch_fused(ctx, fn, din, dout, in_w, band_in_h, 1));
    SRCNN_CUDA(cudaMemcpyAsync(host_out, dout, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (!async) SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
    return SRCNN_OK;
  }
  unsigned long long key[srcnn_ctx::kGraphKey] = {};
  graph_key(key, host_in, host_out, din, dout, in_w, in_h, out_row0, out_row1, n_sub, fn.w1, fn.b1,
            fn.w2, fn.b2, fn.w3, fn.b3, fn.scales, ctx->fused_impl, net->n1, net->n2, ctx->stream);
  return run_subbands(
      ctx, slot, key, sub_r0, n_sub, !async, nullptr,
      [&](int i, int r0, int r1) {
        // input rows [r0 + (i ? halo : 0), r1 + halo): disjoint pieces that tile the band
        const int in0 = r0 + (i ? halo : 0), in1 = r1 + halo;
        return cudaMemcpyAsync(din + (size_t)in0 * in_w, host_in + ((size_t)out_row0 + in0) * in_w,
                               sizeof(float) * (size_t)(in1 - in0) * in_w, cudaMemcpyHostToDevice,
                               ctx->copy_in);
      },
      [&](int, int r0, int r1) {
        return launch_fused(ctx, fn, din + (size_t)r0 * in_w, dout + (size_t)r0 * d.w3, in_w,
                            r1 - r0 + halo, 1);
      },
      [&](int, int r0, int r1) {
        return cudaMemcpyAsync(host_out + (size_t)r0 * d.w3, dout + (size_t)r0 * d.w3,
                               sizeof(float) * (size_t)(r1 - r0) * d.w3, cudaMemcpyDeviceToHost,
                               ctx->copy_out);
      });
}
}  // namespace

int srcnn_infer_rows_host(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in, int in_w,
                          int in_h, int out_row0, int out_row1, float* host_out) {
  return infer_rows_host_impl(ctx, net, host_in, in_w, in_h, out_row0, out_row1, host_out, -1);
}

int srcnn_infer_rows_host_async(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in,
                                int in_w, int in_h, int out_row0, int out_row1, float* host_out) {
  SRCNN_REQUIRE(ctx, "null context");
  const int lane = (int)(ctx->lane_next++ & 1u);
  return infer_rows_host_impl(ctx, net, host_in, in_w, in_h, out_row0, out_row1, host_out, lane);
}


namespace {
// wraps context-owned staging under a handle for the handle-based entries (dropped by TableScope)
srcnn_mem stage_handle(srcnn_ctx* ctx, void* ptr, size_t bytes) {
  Allocation a;
  a.ptr = ptr;
  a.bytes = bytes;
  a.owned = false;
  ctx->allocs.push_back(a);
  return (srcnn_mem)(ctx->allocs.size() - 1);
}

// the arguments srcnn_upscale_image_host and srcnn_upscale_frames_host accept
int check_upscale(const srcnn_net* net, int w, int h, int out_w, int out_h, int filter) {
  SRCNN_TRY(check_net(net));
  SRCNN_TRY(check_resample(w, h, out_w, out_h, filter));
  const int pad = net->f1 + net->f2 + net->f3 - 3;
  SRCNN_REQUIRE(out_w > pad && out_h > pad, "output %dx%d too small for the network (padding %d)",
                out_w, out_h, pad);
  return SRCNN_OK;
}

// One enlargement job: `frames` equal frames back to back in each device buffer, enlarged from
// w x h to out_w x out_h (network output d.w3 x d.h3).
struct Upscale {
  int w, h, out_w, out_h, filter, frames;
  Dims d;
  const int* tab;             // resample::table_for
  int rows_max;
  const uchar4* small;        // input RGBA8
  uchar4* rgba;               // enlarged RGBA8
  float* luma;                // enlarged luma, then minus its Q1 mean
  float* out3;                // network output
  unsigned char* rgb;         // result RGB8
  double* partial;            // Q1 reduction partials: red_blocks() per frame
  float* sums;                // Q1 sums, one per frame
  size_t npx() const { return (size_t)out_w * out_h; }
  int red_blocks() const { return grid_1d(npx(), generic::RED_THREADS, generic::RED_MAX_BLOCKS); }
  // the Q1 reduction bytes of one frame: its partials and its sum
  size_t red_frame() const { return sizeof(double) * red_blocks() + sizeof(float); }
};

// the Q1 "mean" of every frame's u.luma (sum of squares / count, subtracted on the device:
// DataPipeline::subtract_mean).  3 launches.  Each frame's sum takes the block partition a
// single-frame sum takes, so its float is the same.
int q1_mean(srcnn_ctx* ctx, const Upscale& u) {
  const size_t npx = u.npx();
  const int blocks = u.red_blocks();
  {
    LaunchScope scope(ctx, SRCNN_K_SUM, 2);
    generic::sum_stage1<<<dim3(blocks, u.frames), generic::RED_THREADS, 0, ctx->stream>>>(
        u.luma, u.partial, (unsigned)npx, 1);
    generic::reduce_stage2<<<u.frames, generic::RED_THREADS, 0, ctx->stream>>>(u.partial, blocks,
                                                                               u.sums);
    SRCNN_TRY(check_launch("sum"));
  }
  LaunchScope scope(ctx, SRCNN_K_SUB_FROM_ALL);
  generic::sub_mean_kernel<<<dim3(grid_1d(npx, 256, 8 * ctx->sm_count), u.frames), 256, 0,
                             ctx->stream>>>(u.luma, u.sums, (unsigned)npx);
  return check_launch("sub_from_all");
}

// the device work the forward waits for: enlargement + luma, the Q1 mean.  4 launches.
int upscale_head(srcnn_ctx* ctx, const Upscale& u) {
  {
    LaunchScope scope(ctx, SRCNN_K_RESAMPLE);
    SRCNN_TRY(resample::launch(ctx, u.small, u.w, u.h, u.rgba, u.luma, u.out_w, u.out_h, u.filter,
                               u.tab, u.rows_max, u.frames));
    SRCNN_TRY(check_launch("resample"));
  }
  return q1_mean(ctx, u);
}

// swap_luma over image rows [y0, y1) of every frame.  1 launch.
int upscale_swap(srcnn_ctx* ctx, const Upscale& u, int y0, int y1) {
  LaunchScope scope(ctx, SRCNN_K_SWAP_LUMA);
  dim3 block(32, 8), grid((u.out_w + 31) / 32, (y1 - y0 + 7) / 8, u.frames);
  generic::swap_luma_kernel<<<grid, block, 0, ctx->stream>>>(u.rgba, u.out3, u.rgb, u.out_w,
                                                             u.out_h, y0, y1, u.d.w3, u.d.h3);
  return check_launch("swap_luma");
}

// The forward of one image (u.frames == 1) on the three-launch path, u.luma -> u.out3 through the
// layer activations s1 and s2.  L launches.  conv5_tc takes its FP16 operand scale from the
// measured maximum of its whole input, so a sub-band -- or a batch of frames -- could get another
// scale (and result) than the image alone.
int forward_three_launch(srcnn_ctx* ctx, const srcnn_net* net, const Upscale& u, void* s1, void* s2) {
  const Dims& d = u.d;
  TableScope handles(ctx);
  const srcnn_mem m_luma = stage_handle(ctx, u.luma, sizeof(float) * u.npx());
  const srcnn_mem m_out = stage_handle(ctx, u.out3, sizeof(float) * (size_t)d.w3 * d.h3);
  const srcnn_mem m_s1 = stage_handle(ctx, s1, sizeof(float) * (size_t)d.w1 * d.h1 * net->n1);
  const srcnn_mem m_s2 = stage_handle(ctx, s2, sizeof(float) * (size_t)d.w2 * d.h2 * net->n2);
  return srcnn_forward_fused(ctx, net, m_luma, m_out, u.out_w, u.out_h, 1, m_s1, m_s2);
}

// One image (u.frames == 1) through the three-launch path, on the context stream, synchronous:
// upload, head, forward, swap_luma, download.
int upscale_three_launch(srcnn_ctx* ctx, const srcnn_net* net, const Upscale& u, void* s1,
                         void* s2, const unsigned char* host_rgba, unsigned char* host_rgb) {
  SRCNN_CUDA(cudaMemcpyAsync((void*)u.small, host_rgba, (size_t)u.w * u.h * 4,
                             cudaMemcpyHostToDevice, ctx->stream));
  SRCNN_TRY(upscale_head(ctx, u));
  SRCNN_TRY(forward_three_launch(ctx, net, u, s1, s2));
  SRCNN_TRY(upscale_swap(ctx, u, 0, u.out_h));
  SRCNN_CUDA(cudaMemcpyAsync(host_rgb, u.rgb, u.npx() * 3, cudaMemcpyDeviceToHost, ctx->stream));
  SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  return SRCNN_OK;
}
}  // namespace

int srcnn_upscale_image_host(srcnn_ctx* ctx, const srcnn_net* net, const unsigned char* host_rgba,
                             int w, int h, int out_w, int out_h, int filter,
                             unsigned char* host_rgb) {
  SRCNN_REQUIRE(ctx && host_rgba && host_rgb, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_upscale(net, w, h, out_w, out_h, filter));
  const int pad = net->f1 + net->f2 + net->f3 - 3;
  const Dims d = net_dims(net, out_w, out_h);
  const size_t npx = (size_t)out_w * out_h;
  SRCNN_CUDA(ctx->drain_lanes());
  srcnn_ctx::UpscaleStaging& st = ctx->up;
  SRCNN_TRY(ensure_scratch(ctx, &st.small, &st.small_bytes, (size_t)w * h * 4));
  SRCNN_TRY(ensure_scratch(ctx, &st.rgba, &st.rgba_bytes, npx * 4));
  SRCNN_TRY(ensure_scratch(ctx, &st.luma, &st.luma_bytes, npx * sizeof(float)));
  SRCNN_TRY(ensure_scratch(ctx, &st.out, &st.out_bytes, sizeof(float) * (size_t)d.w3 * d.h3));
  SRCNN_TRY(ensure_scratch(ctx, &st.rgb, &st.rgb_bytes, npx * 3));
  const bool fused = fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3);
  if (!fused) {
    SRCNN_TRY(ensure_scratch(ctx, &st.s1, &st.s1_bytes, sizeof(float) * (size_t)d.w1 * d.h1 * net->n1));
    SRCNN_TRY(ensure_scratch(ctx, &st.s2, &st.s2_bytes, sizeof(float) * (size_t)d.w2 * d.h2 * net->n2));
  }
  Upscale u{w, h, out_w, out_h, filter, 1, d, nullptr, 0};
  SRCNN_TRY(resample::table_for(ctx, w, h, out_w, out_h, filter, SRCNN_CHROMA_CENTER,
                                SRCNN_CHROMA_CENTER, &u.tab, &u.rows_max));
  fast::FusedNet fn;
  SRCNN_TRY(fused_net(ctx, net, &fn));
  u.small = (const uchar4*)st.small;
  u.rgba = (uchar4*)st.rgba;
  u.luma = (float*)st.luma;
  u.out3 = (float*)st.out;
  u.rgb = (unsigned char*)st.rgb;
  // the partials take at most RED_MAX_BLOCKS doubles at the start of the reduction scratch, the
  // sum its last word
  u.partial = (double*)ctx->red_scratch;
  u.sums = (float*)ctx->red_scratch + srcnn_ctx::kRedScratchBytes / sizeof(float) - 1;
  if (!fused) return upscale_three_launch(ctx, net, u, st.s1, st.s2, host_rgba, host_rgb);
  // The sub-band pipeline of srcnn_infer_rows_host over the network's output rows, behind the
  // upload and the head: the forward of each sub-band, then swap_luma over its image rows, then
  // their download.  The first sub-band also writes the top border rows, the last one the bottom
  // border rows.
  int sub_r0[kMaxSub + 1];
  const int n_sub = subband_rows(d.h3, sub_r0);
  const auto image_rows = [&](int i, int r0, int r1) {
    return std::make_pair(i == 0 ? 0 : pad / 2 + r0, i + 1 == n_sub ? out_h : pad / 2 + r1);
  };
  unsigned long long key[srcnn_ctx::kGraphKey] = {};
  graph_key(key, host_rgba, host_rgb, st.small, st.rgba, st.luma, st.out, st.rgb, u.tab, w, h, out_w,
            out_h, filter, n_sub, fn.w1, fn.b1, fn.w2, fn.b2, fn.w3, fn.b3, fn.scales, ctx->fused_impl,
            net->n1, net->n2, net->f1, net->f2, net->f3, ctx->stream);
  return run_subbands(
      ctx, GraphSlot{&st.graph, st.key, st.graph_launches}, key, sub_r0, n_sub, true,
      [&] {
        SRCNN_CUDA(cudaMemcpyAsync(st.small, host_rgba, (size_t)w * h * 4, cudaMemcpyHostToDevice,
                                   ctx->stream));
        return upscale_head(ctx, u);
      },
      nullptr,
      [&](int i, int r0, int r1) {
        SRCNN_TRY(launch_fused(ctx, fn, u.luma + (size_t)r0 * out_w, u.out3 + (size_t)r0 * d.w3,
                               out_w, r1 - r0 + pad, 1));
        const auto y = image_rows(i, r0, r1);
        return upscale_swap(ctx, u, y.first, y.second);
      },
      [&](int i, int r0, int r1) {
        const auto y = image_rows(i, r0, r1);
        return cudaMemcpyAsync(host_rgb + (size_t)y.first * out_w * 3,
                               u.rgb + (size_t)y.first * out_w * 3,
                               (size_t)(y.second - y.first) * out_w * 3, cudaMemcpyDeviceToHost,
                               ctx->copy_out);
      });
}

namespace {
// the frame entries' ring of device slots: the upload of group g+1 and the download of group g-1
// overlap the device work of group g
constexpr int kFrameRing = 3;

// frames per group: SRCNN_FRAMES_GROUP=n when set (read once per process), else as many as fit
// `target_bytes` of device staging at `frame_bytes` each (at least 1); never more than n_frames
int frames_group(size_t frame_bytes, size_t target_bytes, int n_frames) {
  static const int kGroupEnv = std::getenv("SRCNN_FRAMES_GROUP") ? std::atoi(std::getenv("SRCNN_FRAMES_GROUP")) : 0;
  const size_t g = kGroupEnv > 0 ? (size_t)kGroupEnv : std::max<size_t>(1, target_bytes / frame_bytes);
  return (int)std::min<size_t>(g, (size_t)n_frames);
}

// Runs n_frames frames in groups of `group` through the ring: the upload of a group's frames
// (`in_frame` bytes each) from host_in into device slot r of dev_in (copy-in stream), then
// work(S frames, r) on the context stream, then the download of the slot's results (`out_frame`
// bytes each) from dev_out to host_out (copy-out stream).  Returns when the downloads are done.
// With host_in2, a second input (`in2_frame` bytes a frame) goes up the same way into slot r of
// dev_in2, right behind the first.
int run_frame_ring(srcnn_ctx* ctx, int n_frames, int group, const void* host_in, void* dev_in,
                   size_t in_frame, void* host_out, const void* dev_out, size_t out_frame,
                   const std::function<int(int S, int r)>& work, const void* host_in2 = nullptr,
                   void* dev_in2 = nullptr, size_t in2_frame = 0) {
  SRCNN_TRY(ensure_side_streams(ctx));
  // the side streams start behind whatever the context stream was doing with the staging
  SRCNN_CUDA(cudaEventRecord(ctx->ev_k[kFrameRing], ctx->stream));
  SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[kFrameRing], 0));
  SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[kFrameRing], 0));
  for (int g = 0, f0 = 0; f0 < n_frames; g++, f0 += group) {
    const int S = std::min(group, n_frames - f0), r = g % kFrameRing;
    // input slot r was last read by the device work of group g - kFrameRing
    if (g >= kFrameRing) SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[r], 0));
    SRCNN_CUDA(cudaMemcpyAsync((char*)dev_in + in_frame * group * r, (const char*)host_in + in_frame * f0,
                               in_frame * S, cudaMemcpyHostToDevice, ctx->copy_in));
    if (host_in2)
      SRCNN_CUDA(cudaMemcpyAsync((char*)dev_in2 + in2_frame * group * r,
                                 (const char*)host_in2 + in2_frame * f0, in2_frame * S,
                                 cudaMemcpyHostToDevice, ctx->copy_in));
    SRCNN_CUDA(cudaEventRecord(ctx->ev_in[r], ctx->copy_in));
    SRCNN_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[r], 0));
    // output slot r was last downloaded for group g - kFrameRing
    if (g >= kFrameRing) SRCNN_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_d[r], 0));
    SRCNN_TRY(work(S, r));
    SRCNN_CUDA(cudaEventRecord(ctx->ev_k[r], ctx->stream));
    SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[r], 0));
    SRCNN_CUDA(cudaMemcpyAsync((char*)host_out + out_frame * f0, (const char*)dev_out + out_frame * group * r,
                               out_frame * S, cudaMemcpyDeviceToHost, ctx->copy_out));
    SRCNN_CUDA(cudaEventRecord(ctx->ev_d[r], ctx->copy_out));
  }
  SRCNN_CUDA(cudaStreamSynchronize(ctx->copy_out));
  SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  return SRCNN_OK;
}
}  // namespace

namespace {
// A call of the frames entries: its enlargement job (u.frames, u.small and u.rgb are set per
// group), its network, its group size and where the ring of inputs and results lives.
struct FramesCall {
  Upscale u;
  fast::FusedNet fn;
  int group;
  bool fused;
  uchar4* small;          // ring of input groups (one frame without a fused kernel)
  unsigned char* rgb;     // ring of result groups
};

// A frames call's bytes a frame: its input (`in`, ring slots `small`), its enlarged RGBA8 (`rgba`,
// 0 when the call has none) and its result (`out`, ring slots `rgb`); `group` of them a frame set
// the group size, `max_group` caps it (the frame is a grid dimension of the group's launches).
struct FrameBytes {
  size_t in, rgba, out, group;
  int max_group;
};

// the RGBA8-in, RGB8-out frame of srcnn_upscale_frames_host, plus `extra` device bytes a frame
// that enter the group size (the caller allocates them): ~128 MB of device staging per group
// (input, enlarged RGBA8 + luma + RGB8, network output; 960x540 -> 1920x1080: 4 frames) --
// launches long enough to fill the GPU, a first upload and a last download short next to a whole
// call
FrameBytes rgba_frame_bytes(const srcnn_net* net, int w, int h, int out_w, int out_h, size_t extra) {
  const Dims d = net_dims(net, out_w, out_h);
  const size_t in_px = (size_t)w * h, npx = (size_t)out_w * out_h, out_px = (size_t)d.w3 * d.h3;
  return FrameBytes{in_px * 4, npx * 4, npx * 3, in_px * 4 + npx * (4 + 4 + 3) + out_px * 4 + extra,
                    65535};
}

// staging in `st`, the resample table and the prepared network of a frames call whose arguments
// have been checked
// (`bit_depth` selects the resample table: 8, or 10 for the Y plane of 10-bit frames)
int frames_prepare(srcnn_ctx* ctx, const srcnn_net* net, srcnn_ctx::FramesStaging& st, int w, int h,
                   int n_frames, int out_w, int out_h, int filter, const FrameBytes& fb,
                   FramesCall* fc, int bit_depth = 8) {
  const Dims d = net_dims(net, out_w, out_h);
  const size_t npx = (size_t)out_w * out_h, out_px = (size_t)d.w3 * d.h3;
  SRCNN_CUDA(ctx->drain_lanes());
  const bool fused = fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3);
  Upscale u{w, h, out_w, out_h, filter, 1, d, nullptr, 0};
  const int group =
      fused ? std::min(frames_group(fb.group, (size_t)128 << 20, n_frames), fb.max_group) : 1;
  const int ring = fused ? kFrameRing : 1;
  SRCNN_TRY(ensure_scratch(ctx, &st.small, &st.small_bytes, fb.in * group * ring));
  if (fb.rgba) SRCNN_TRY(ensure_scratch(ctx, &st.rgba, &st.rgba_bytes, fb.rgba * group));
  SRCNN_TRY(ensure_scratch(ctx, &st.luma, &st.luma_bytes, npx * sizeof(float) * group));
  SRCNN_TRY(ensure_scratch(ctx, &st.out, &st.out_bytes, out_px * sizeof(float) * group));
  SRCNN_TRY(ensure_scratch(ctx, &st.rgb, &st.rgb_bytes, fb.out * group * ring));
  SRCNN_TRY(ensure_scratch(ctx, &st.red, &st.red_bytes, u.red_frame() * group));
  if (!fused) {
    SRCNN_TRY(ensure_scratch(ctx, &st.s1, &st.s1_bytes, sizeof(float) * (size_t)d.w1 * d.h1 * net->n1));
    SRCNN_TRY(ensure_scratch(ctx, &st.s2, &st.s2_bytes, sizeof(float) * (size_t)d.w2 * d.h2 * net->n2));
  }
  SRCNN_TRY(resample::table_for(ctx, w, h, out_w, out_h, filter, SRCNN_CHROMA_CENTER,
                                SRCNN_CHROMA_CENTER, &u.tab, &u.rows_max, bit_depth));
  SRCNN_TRY(fused_net(ctx, net, &fc->fn));
  u.rgba = (uchar4*)st.rgba;
  u.luma = (float*)st.luma;
  u.out3 = (float*)st.out;
  u.partial = (double*)st.red;
  u.sums = (float*)(u.partial + (size_t)u.red_blocks() * group);
  u.small = (uchar4*)st.small;
  u.rgb = (unsigned char*)st.rgb;
  fc->u = u;
  fc->group = group;
  fc->fused = fused;
  fc->small = (uchar4*)st.small;
  fc->rgb = (unsigned char*)st.rgb;
  return SRCNN_OK;
}

// the device work of one group of the frames entry in ring slot r: enlargement, Q1 mean, fused
// forward, swap_luma.  5 + F launches.
int frames_group_work(srcnn_ctx* ctx, FramesCall& fc, int S, int r) {
  Upscale& u = fc.u;
  const size_t in_px = (size_t)u.w * u.h, npx = u.npx();
  u.frames = S;
  u.small = fc.small + (size_t)r * fc.group * in_px;
  u.rgb = fc.rgb + (size_t)r * fc.group * npx * 3;
  SRCNN_TRY(upscale_head(ctx, u));
  SRCNN_TRY(launch_fused(ctx, fc.fn, u.luma, u.out3, u.out_w, u.out_h, S));
  return upscale_swap(ctx, u, 0, u.out_h);
}

// the quality of u's frames against `ref`: the RGB8 result into m[4 s + 0, 1], the enlarged
// RGBA8 into m[4 s + 2, 3].  4 launches.
int quality_pair(srcnn_ctx* ctx, const Upscale& u, const uchar4* ref, int border, double2* partial,
                 double* m) {
  LaunchScope scope(ctx, SRCNN_K_QUALITY, 4);
  quality::launch(ctx, u.rgb, 3, ref, u.out_w, u.out_h, u.frames, border, partial, m, 4);
  quality::launch(ctx, (const unsigned char*)u.rgba, 4, ref, u.out_w, u.out_h, u.frames, border,
                  partial, m + 2, 4);
  return check_launch("image_quality");
}
}  // namespace

int srcnn_upscale_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const unsigned char* host_rgba,
                              int w, int h, int n_frames, int out_w, int out_h, int filter,
                              unsigned char* host_rgb) {
  SRCNN_REQUIRE(ctx && host_rgba && host_rgb, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_upscale(net, w, h, out_w, out_h, filter));
  SRCNN_REQUIRE(n_frames > 0, "bad frame count %d", n_frames);
  srcnn_ctx::FramesStaging& st = ctx->frames;
  FramesCall fc;
  SRCNN_TRY(frames_prepare(ctx, net, st, w, h, n_frames, out_w, out_h, filter,
                           rgba_frame_bytes(net, w, h, out_w, out_h, 0), &fc));
  const size_t in_px = (size_t)w * h, npx = (size_t)out_w * out_h;
  if (!fc.fused) {
    // frame by frame, each as the image entry runs it
    for (int f = 0; f < n_frames; f++)
      SRCNN_TRY(upscale_three_launch(ctx, net, fc.u, st.s1, st.s2, host_rgba + (size_t)f * in_px * 4,
                                     host_rgb + (size_t)f * npx * 3));
    return SRCNN_OK;
  }
  return run_frame_ring(ctx, n_frames, fc.group, host_rgba, fc.small, in_px * 4, host_rgb, fc.rgb,
                        npx * 3, [&](int S, int r) { return frames_group_work(ctx, fc, S, r); });
}

int srcnn_evaluate_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const unsigned char* host_rgba,
                               int w, int h, int n_frames, int out_w, int out_h, int filter,
                               const unsigned char* host_ref, int border, unsigned char* host_rgb,
                               double* host_metrics) {
  SRCNN_REQUIRE(ctx && host_rgba && host_rgb && host_ref && host_metrics, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_upscale(net, w, h, out_w, out_h, filter));
  SRCNN_REQUIRE(n_frames > 0, "bad frame count %d", n_frames);
  if (border < 0) border = (net->f1 + net->f2 + net->f3 - 3) / 2;
  SRCNN_TRY(check_quality_region(out_w, out_h, border));
  srcnn_ctx::FramesStaging& st = ctx->eval;
  const size_t in_px = (size_t)w * h, npx = (size_t)out_w * out_h;
  FramesCall fc;
  SRCNN_TRY(frames_prepare(ctx, net, st, w, h, n_frames, out_w, out_h, filter,
                           rgba_frame_bytes(net, w, h, out_w, out_h, npx * 4), &fc));
  const int ring = fc.fused ? kFrameRing : 1;
  SRCNN_TRY(ensure_scratch(ctx, &st.ref, &st.ref_bytes, npx * 4 * fc.group * ring));
  SRCNN_TRY(ensure_scratch(ctx, &st.qred, &st.qred_bytes,
                           quality::partial_bytes(out_w, out_h, border, fc.group)));
  SRCNN_TRY(ensure_scratch(ctx, &st.metrics, &st.metrics_bytes, sizeof(double) * 4 * (size_t)n_frames));
  uchar4* refs = (uchar4*)st.ref;
  double2* qred = (double2*)st.qred;
  double* metrics = (double*)st.metrics;
  if (!fc.fused) {
    // frame by frame through the image entry's route, the reference uploaded ahead of it and the
    // quality measured behind it on the context stream
    for (int f = 0; f < n_frames; f++) {
      SRCNN_CUDA(cudaMemcpyAsync(refs, host_ref + (size_t)f * npx * 4, npx * 4,
                                 cudaMemcpyHostToDevice, ctx->stream));
      SRCNN_TRY(upscale_three_launch(ctx, net, fc.u, st.s1, st.s2, host_rgba + (size_t)f * in_px * 4,
                                     host_rgb + (size_t)f * npx * 3));
      SRCNN_TRY(quality_pair(ctx, fc.u, refs, border, qred, metrics + (size_t)f * 4));
    }
  } else {
    int f0 = 0;   // first frame of the group the ring hands out next (groups come in order)
    SRCNN_TRY(run_frame_ring(
        ctx, n_frames, fc.group, host_rgba, fc.small, in_px * 4, host_rgb, fc.rgb, npx * 3,
        [&](int S, int r) {
          SRCNN_TRY(frames_group_work(ctx, fc, S, r));
          const uchar4* ref = refs + (size_t)r * fc.group * npx;
          double* m = metrics + (size_t)f0 * 4;
          f0 += S;
          return quality_pair(ctx, fc.u, ref, border, qred, m);
        },
        host_ref, refs, npx * 4));
  }
  SRCNN_CUDA(cudaMemcpyAsync(host_metrics, metrics, sizeof(double) * 4 * (size_t)n_frames,
                             cudaMemcpyDeviceToHost, ctx->stream));
  SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
  return SRCNN_OK;
}

namespace {
// the arguments srcnn_upscale_yuv420_frames_host and srcnn_upscale_yuv420_frames accept
int check_yuv420(const srcnn_net* net, int w, int h, int n_frames, int out_w, int out_h,
                 int filter) {
  SRCNN_TRY(check_upscale(net, w, h, out_w, out_h, filter));
  SRCNN_REQUIRE(w % 2 == 0 && h % 2 == 0 && out_w % 2 == 0 && out_h % 2 == 0,
                "4:2:0 frames need even sizes, got %dx%d -> %dx%d", w, h, out_w, out_h);
  SRCNN_REQUIRE(n_frames > 0, "bad frame count %d", n_frames);
  return SRCNN_OK;
}

int check_sitings(int siting_in, int siting_out) {
  for (int s : {siting_in, siting_out})
    SRCNN_REQUIRE(s == SRCNN_CHROMA_CENTER || s == SRCNN_CHROMA_LEFT || s == SRCNN_CHROMA_TOPLEFT,
                  "unknown chroma siting %d", s);
  return SRCNN_OK;
}

// whole I420 (bit_depth 10: I010) frames of w x h back to back: the frames of
// srcnn_upscale_yuv420_frames_host (srcnn_upscale_yuv420p10_frames_host)
srcnn_yuv420_layout i420_dense(int w, int h, int bit_depth = 8) {
  const size_t b = bit_depth == 10 ? 2 : 1, y = (size_t)w * h * b, c = y / 4;
  return srcnn_yuv420_layout{SRCNN_YUV_I420, y + 2 * c, (size_t)w * b, (size_t)w / 2 * b, y, y + c,
                             SRCNN_CHROMA_CENTER, bit_depth};
}

// the layout of n_frames frames of w x h (w, h even and > 0) holds them: *need = the bytes from
// the first frame's start to the end of the last frame's last plane.  Its bit_depth is 0, 8 or 10.
int check_layout(const srcnn_yuv420_layout& l, int w, int h, int n_frames, size_t* need,
                 const char* what) {
  const bool nv12 = l.format == SRCNN_YUV_NV12;
  SRCNN_REQUIRE(l.bit_depth == 0 || l.bit_depth == 8 || l.bit_depth == 10,
                "%s layout: bit depth %d is not 8 or 10", what, l.bit_depth);
  const bool ten = l.bit_depth == 10;
  const size_t big = (size_t)1 << 31, b = ten ? 2 : 1, y_row = (size_t)w * b,
               c_row = (nv12 ? (size_t)w : (size_t)w / 2) * b;
  SRCNN_REQUIRE(l.frame_stride < big && l.y_pitch < big && l.c_pitch < big && l.cb_offset < big &&
                    l.cr_offset < big,
                "%s layout: a pitch, offset or stride of 2^31 bytes or more", what);
  SRCNN_REQUIRE(l.y_pitch >= y_row && l.c_pitch >= c_row,
                "%s layout: pitches %zu (Y) and %zu (chroma) below the rows' %zu and %zu bytes", what,
                l.y_pitch, l.c_pitch, y_row, c_row);
  if (ten) {
    // every sample is a 16-bit word, every P010 CbCr pair a 32-bit one
    SRCNN_REQUIRE(l.y_pitch % 2 == 0 && l.c_pitch % 2 == 0 && l.cb_offset % 2 == 0 &&
                      l.cr_offset % 2 == 0 && (n_frames == 1 || l.frame_stride % 2 == 0),
                  "%s layout: 10-bit samples need even pitches, offsets and frame_stride", what);
    SRCNN_REQUIRE(!nv12 || (l.c_pitch % 4 == 0 && (n_frames == 1 || l.frame_stride % 4 == 0)),
                  "%s layout: P010 needs a c_pitch and frame_stride that are multiples of 4, got "
                  "%zu and %zu", what, l.c_pitch, l.frame_stride);
  }
  // the planes' byte ranges from the frame start: Y [0, y_end), chroma [offset, offset + c_len)
  const size_t y_end = (size_t)(h - 1) * l.y_pitch + y_row;
  const size_t c_len = (size_t)(h / 2 - 1) * l.c_pitch + c_row;
  size_t extent = std::max(y_end, l.cb_offset + c_len);
  SRCNN_REQUIRE(l.cb_offset >= y_end, "%s layout: the %s plane at %zu intersects the Y plane [0, %zu)",
                what, nv12 ? "CbCr" : "Cb", l.cb_offset, y_end);
  if (nv12) {
    SRCNN_REQUIRE(l.cr_offset == 0, "%s layout: NV12 needs cr_offset 0, got %zu", what, l.cr_offset);
    SRCNN_REQUIRE(l.c_pitch % 2 == 0, "%s layout: NV12 needs an even c_pitch, got %zu", what,
                  l.c_pitch);
  } else {
    SRCNN_REQUIRE(l.cr_offset >= y_end &&
                      (l.cr_offset >= l.cb_offset + c_len || l.cb_offset >= l.cr_offset + c_len),
                  "%s layout: the Cr plane at %zu intersects the Y plane [0, %zu) or the Cb plane "
                  "[%zu, %zu)", what, l.cr_offset, y_end, l.cb_offset, l.cb_offset + c_len);
    extent = std::max(extent, l.cr_offset + c_len);
  }
  SRCNN_REQUIRE(n_frames == 1 || l.frame_stride >= extent,
                "%s layout: frame_stride %zu below the frame's extent %zu", what, l.frame_stride,
                extent);
  *need = (size_t)(n_frames - 1) * l.frame_stride + extent;
  return SRCNN_OK;
}

// A group of Y'CbCr 4:2:0 frames of an Upscale job (its u.small, u.rgba and u.rgb unused): frame
// f at in + f * li.frame_stride and out + f * lo.frame_stride, the chroma planes enlarged through
// tab_c.
struct Yuv420 {
  const int* tab_c;
  int rows_max_c;
  const unsigned char* in;
  unsigned char* out;
  srcnn_yuv420_layout li, lo;
};

// the device work the forward waits for: the planes enlarged straight into the result frames,
// the luma of the Y plane, its Q1 mean.  4 launches (I420), 5 (NV12).
int yuv420_head(srcnn_ctx* ctx, const Upscale& u, const Yuv420& y) {
  {
    using namespace resample;
    const bool nv12 = y.li.format == SRCNN_YUV_NV12;
    LaunchScope scope(ctx, SRCNN_K_RESAMPLE, nv12 ? 2 : 1);
    const auto launch =
        y.li.bit_depth == 10
            ? (nv12 ? launch_nv12<unsigned short, Words10<6>>
                    : launch_yuv420<unsigned short, Words10<0>>)
            : (nv12 ? launch_nv12<unsigned char, Bytes> : launch_yuv420<unsigned char, Bytes>);
    SRCNN_TRY(launch(ctx, y.in, y.li, u.w, u.h, y.out, y.lo, u.luma, u.out_w, u.out_h, u.filter,
                     u.tab, u.rows_max, y.tab_c, y.rows_max_c, u.frames));
    SRCNN_TRY(check_launch("resample"));
  }
  return q1_mean(ctx, u);
}

// the network's luma over the interior of every frame's Y plane.  1 launch.
int yuv420_swap(srcnn_ctx* ctx, const Upscale& u, const Yuv420& y) {
  LaunchScope scope(ctx, SRCNN_K_SWAP_LUMA);
  dim3 block(32, 8), grid((u.d.w3 + 31) / 32, (u.d.h3 + 7) / 8, u.frames);
  const auto kernel = y.lo.bit_depth != 10 ? generic::swap_luma_plane_kernel<unsigned char, 255, 0>
                      : y.lo.format == SRCNN_YUV_NV12
                          ? generic::swap_luma_plane_kernel<unsigned short, 1023, 6>
                          : generic::swap_luma_plane_kernel<unsigned short, 1023, 0>;
  kernel<<<grid, block, 0, ctx->stream>>>(u.out3, y.out, u.out_w, y.lo.y_pitch, y.lo.frame_stride,
                                          u.d.w3, u.d.h3);
  return check_launch("swap_luma");
}
}  // namespace

int srcnn_upscale_yuv420_frames_host(srcnn_ctx* ctx, const srcnn_net* net,
                                     const unsigned char* host_in, int w, int h, int n_frames,
                                     int out_w, int out_h, int filter, unsigned char* host_out) {
  return srcnn_upscale_yuv420_frames_host_sited(ctx, net, host_in, w, h, n_frames, out_w, out_h,
                                                filter, SRCNN_CHROMA_CENTER, SRCNN_CHROMA_CENTER,
                                                host_out);
}

namespace {
// srcnn_upscale_yuv420_frames_host_sited (bit_depth 8) and srcnn_upscale_yuv420p10_frames_host
// (bit_depth 10) on dense frames
int yuv420_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const void* host_in_v, int w, int h,
                       int n_frames, int out_w, int out_h, int filter, int in_siting,
                       int out_siting, int bit_depth, void* host_out_v) {
  SRCNN_REQUIRE(ctx && host_in_v && host_out_v, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_yuv420(net, w, h, n_frames, out_w, out_h, filter));
  SRCNN_TRY(check_sitings(in_siting, out_siting));
  const unsigned char* host_in = static_cast<const unsigned char*>(host_in_v);
  unsigned char* host_out = static_cast<unsigned char*>(host_out_v);
  srcnn_ctx::FramesStaging& st = ctx->yuv;
  const Dims d = net_dims(net, out_w, out_h);
  Yuv420 y{nullptr, 0, nullptr, nullptr, i420_dense(w, h, bit_depth),
           i420_dense(out_w, out_h, bit_depth)};
  const size_t in_frame = y.li.frame_stride, out_frame = y.lo.frame_stride;
  // the device bytes a frame of a group holds: its input and result in each ring slot, its luma
  // and its network output (960x540 -> 1920x1080: 4 frames in ~128 MB, 3 with 10-bit samples);
  // the frame and the plane share the grid dimension of the resampling launch
  const FrameBytes fb{in_frame, 0, out_frame,
                      (in_frame + out_frame) * kFrameRing + (size_t)out_w * out_h * 4 +
                          (size_t)d.w3 * d.h3 * 4,
                      65535 / 3};
  FramesCall fc;
  SRCNN_TRY(frames_prepare(ctx, net, st, w, h, n_frames, out_w, out_h, filter, fb, &fc, bit_depth));
  SRCNN_TRY(resample::table_for(ctx, w / 2, h / 2, out_w / 2, out_h / 2, filter, in_siting,
                                out_siting, &y.tab_c, &y.rows_max_c, bit_depth));
  unsigned char* ring_in = (unsigned char*)st.small;
  unsigned char* ring_out = (unsigned char*)st.rgb;
  Upscale& u = fc.u;
  if (!fc.fused) {
    // frame by frame, for the reason forward_three_launch gives
    y.in = ring_in;
    y.out = ring_out;
    for (int f = 0; f < n_frames; f++) {
      SRCNN_CUDA(cudaMemcpyAsync(ring_in, host_in + (size_t)f * in_frame, in_frame,
                                 cudaMemcpyHostToDevice, ctx->stream));
      SRCNN_TRY(yuv420_head(ctx, u, y));
      SRCNN_TRY(forward_three_launch(ctx, net, u, st.s1, st.s2));
      SRCNN_TRY(yuv420_swap(ctx, u, y));
      SRCNN_CUDA(cudaMemcpyAsync(host_out + (size_t)f * out_frame, ring_out, out_frame,
                                 cudaMemcpyDeviceToHost, ctx->stream));
      SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return SRCNN_OK;
  }
  // a group's device work: enlargement + luma, Q1 mean, fused forward, Y write.  5 + F launches.
  return run_frame_ring(ctx, n_frames, fc.group, host_in, ring_in, in_frame, host_out, ring_out,
                        out_frame, [&](int S, int r) {
                          u.frames = S;
                          y.in = ring_in + (size_t)r * fc.group * in_frame;
                          y.out = ring_out + (size_t)r * fc.group * out_frame;
                          SRCNN_TRY(yuv420_head(ctx, u, y));
                          SRCNN_TRY(launch_fused(ctx, fc.fn, u.luma, u.out3, u.out_w, u.out_h, S));
                          return yuv420_swap(ctx, u, y);
                        });
}
}  // namespace

int srcnn_upscale_yuv420_frames_host_sited(srcnn_ctx* ctx, const srcnn_net* net,
                                           const unsigned char* host_in, int w, int h, int n_frames,
                                           int out_w, int out_h, int filter, int in_siting,
                                           int out_siting, unsigned char* host_out) {
  return yuv420_frames_host(ctx, net, host_in, w, h, n_frames, out_w, out_h, filter, in_siting,
                            out_siting, 8, host_out);
}

int srcnn_upscale_yuv420p10_frames_host(srcnn_ctx* ctx, const srcnn_net* net,
                                        const uint16_t* host_in, int w, int h, int n_frames,
                                        int out_w, int out_h, int filter, int in_siting,
                                        int out_siting, uint16_t* host_out) {
  return yuv420_frames_host(ctx, net, host_in, w, h, n_frames, out_w, out_h, filter, in_siting,
                            out_siting, 10, host_out);
}

int srcnn_upscale_yuv420_frames(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in,
                                const srcnn_yuv420_layout* in_layout, int w, int h, int n_frames,
                                srcnn_mem out, const srcnn_yuv420_layout* out_layout, int out_w,
                                int out_h, int filter) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_yuv420(net, w, h, n_frames, out_w, out_h, filter));
  SRCNN_REQUIRE(in_layout && out_layout, "null layout");
  const int format = in_layout->format;
  SRCNN_REQUIRE(format == SRCNN_YUV_I420 || format == SRCNN_YUV_NV12, "unknown 4:2:0 format %d",
                format);
  SRCNN_REQUIRE(out_layout->format == format, "input format %d and output format %d differ", format,
                out_layout->format);
  SRCNN_TRY(check_sitings(in_layout->chroma_siting, out_layout->chroma_siting));
  const int bits = in_layout->bit_depth == 10 ? 10 : 8;
  SRCNN_REQUIRE(bits == (out_layout->bit_depth == 10 ? 10 : 8),
                "input bit depth %d and output bit depth %d differ", in_layout->bit_depth,
                out_layout->bit_depth);
  size_t in_need, out_need;
  SRCNN_TRY(check_layout(*in_layout, w, h, n_frames, &in_need, "input"));
  SRCNN_TRY(check_layout(*out_layout, out_w, out_h, n_frames, &out_need, "output"));
  const unsigned char* pi;
  unsigned char* po;
  SRCNN_TRY(resolve(ctx, in, in_need, &pi, "input frames"));
  SRCNN_TRY(resolve(ctx, out, out_need, &po, "output frames"));
  const bool nv12 = format == SRCNN_YUV_NV12;
  if (nv12) {
    // the CbCr plane is read and written as uchar2: every frame's must start at an even address
    SRCNN_REQUIRE(((uintptr_t)pi + in_layout->cb_offset) % 2 == 0 &&
                      (n_frames == 1 || in_layout->frame_stride % 2 == 0),
                  "input NV12 CbCr plane at an odd address");
    SRCNN_REQUIRE(((uintptr_t)po + out_layout->cb_offset) % 2 == 0 &&
                      (n_frames == 1 || out_layout->frame_stride % 2 == 0),
                  "output NV12 CbCr plane at an odd address");
  }
  if (bits == 10) {
    // 16-bit words, and P010 CbCr pairs read and written as 32-bit words (the strides and
    // pitches are checked with the layouts)
    const size_t a = nv12 ? 4 : 2;
    SRCNN_REQUIRE((uintptr_t)pi % 2 == 0 && ((uintptr_t)pi + in_layout->cb_offset) % a == 0,
                  "input 10-bit frames at an odd address, or a P010 CbCr plane off 4 bytes");
    SRCNN_REQUIRE((uintptr_t)po % 2 == 0 && ((uintptr_t)po + out_layout->cb_offset) % a == 0,
                  "output 10-bit frames at an odd address, or a P010 CbCr plane off 4 bytes");
  }
  SRCNN_REQUIRE(pi + in_need <= po || po + out_need <= pi, "input and output bytes overlap");
  ctx->note_write(out);
  const Upscale job{w, h, out_w, out_h, filter, 1, net_dims(net, out_w, out_h), nullptr, 0};
  // the scratch a frame of a group needs: its luma, its network output, its Q1 partials and sum;
  // the frame (times the planes, I420) is a grid dimension of the group's launches
  const FrameBytes fb{0, 0, 0,
                      job.npx() * 4 + (size_t)job.d.w3 * job.d.h3 * 4 + job.red_frame(),
                      nv12 ? 65535 : 65535 / 3};
  FramesCall fc;
  SRCNN_TRY(frames_prepare(ctx, net, ctx->yuv_dev, w, h, n_frames, out_w, out_h, filter, fb, &fc,
                           bits));
  Yuv420 y{nullptr, 0, pi, po, *in_layout, *out_layout};
  SRCNN_TRY(resample::table_for(ctx, w / 2, h / 2, out_w / 2, out_h / 2, filter,
                                in_layout->chroma_siting, out_layout->chroma_siting, &y.tab_c,
                                &y.rows_max_c, bits));
  // groups of frames (one frame without a fused kernel, for the reason forward_three_launch
  // gives): enlargement + luma, Q1 mean, forward, Y write
  Upscale& u = fc.u;
  for (int f0 = 0; f0 < n_frames; f0 += fc.group) {
    u.frames = std::min(fc.group, n_frames - f0);
    y.in = pi + (size_t)f0 * y.li.frame_stride;
    y.out = po + (size_t)f0 * y.lo.frame_stride;
    SRCNN_TRY(yuv420_head(ctx, u, y));
    if (fc.fused)
      SRCNN_TRY(launch_fused(ctx, fc.fn, u.luma, u.out3, u.out_w, u.out_h, u.frames));
    else
      SRCNN_TRY(forward_three_launch(ctx, net, u, ctx->yuv_dev.s1, ctx->yuv_dev.s2));
    SRCNN_TRY(yuv420_swap(ctx, u, y));
  }
  return SRCNN_OK;
}

int srcnn_infer_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in, int w,
                            int h, int n_frames, float* host_out) {
  SRCNN_REQUIRE(ctx && host_in && host_out, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, w, h);
  SRCNN_REQUIRE(n_frames > 0 && d.w3 > 0 && d.h3 > 0, "bad frame set: %d frames of %dx%d", n_frames, w, h);
  SRCNN_REQUIRE(fast::fused_supported(net->n1, net->n2, net->f1, net->f2, net->f3),
                "srcnn_infer_frames_host needs a fused instantiation for %d-%d-%d n1=%d n2=%d",
                net->f1, net->f2, net->f3, net->n1, net->n2);
  fast::FusedNet fn;
  SRCNN_TRY(fused_net(ctx, net, &fn));
  // groups of frames go through the ring (one fused forward per group, frame = gridDim.z)
  const size_t in_px = (size_t)w * h, out_px = (size_t)d.w3 * d.h3;
  // ~16 MB of input per group: long enough launches to fill the GPU, short enough that the
  // exposed first upload / last download stay small
  const int group = frames_group(in_px * sizeof(float), (size_t)16 << 20, n_frames);
  SRCNN_TRY(ensure_scratch(ctx, &ctx->band_in, &ctx->band_in_bytes, sizeof(float) * in_px * group * kFrameRing));
  SRCNN_TRY(ensure_scratch(ctx, &ctx->band_out, &ctx->band_out_bytes, sizeof(float) * out_px * group * kFrameRing));
  float* din = (float*)ctx->band_in;
  float* dout = (float*)ctx->band_out;
  return run_frame_ring(ctx, n_frames, group, host_in, din, sizeof(float) * in_px, host_out, dout,
                        sizeof(float) * out_px, [&](int S, int r) {
                          return launch_fused(ctx, fn, din + (size_t)r * group * in_px,
                                              dout + (size_t)r * group * out_px, w, h, S);
                        });
}

size_t srcnn_train_workspace_bytes(const srcnn_net* net, int w, int h, int S) {
  if (!net || S <= 0) return 0;
  const Dims d = net_dims(net, w, h);
  if (d.w3 <= 0 || d.h3 <= 0) return 0;
  const size_t e1 = align256(sizeof(float) * (size_t)d.w1 * d.h1 * net->n1 * S),
               e2 = align256(sizeof(float) * (size_t)d.w2 * d.h2 * net->n2 * S),
               e3 = align256(sizeof(float) * (size_t)d.w3 * d.h3 * S);
  return 2 * (e1 + e2 + e3);
}

namespace {
struct Work {
  srcnn_mem out1, out2, out3, d1, d2, d3;
};
// carve the chunk workspace into six wrapped sub-buffers (handles are cheap table entries)
int carve(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem work, int w, int h, int S, Work* wk) {
  const Dims d = net_dims(net, w, h);
  // every sub-buffer starts 256-byte aligned (vectorised loads in the training kernels)
  const size_t e1 = align256(sizeof(float) * (size_t)d.w1 * d.h1 * net->n1 * S),
               e2 = align256(sizeof(float) * (size_t)d.w2 * d.h2 * net->n2 * S),
               e3 = align256(sizeof(float) * (size_t)d.w3 * d.h3 * S);
  char* base;
  SRCNN_TRY(resolve(ctx, work, 2 * (e1 + e2 + e3), &base, "training workspace"));
  SRCNN_TRY(srcnn_wrap(ctx, base, e1, &wk->out1));
  SRCNN_TRY(srcnn_wrap(ctx, base + e1, e2, &wk->out2));
  SRCNN_TRY(srcnn_wrap(ctx, base + e1 + e2, e3, &wk->out3));
  SRCNN_TRY(srcnn_wrap(ctx, base + e1 + e2 + e3, e1, &wk->d1));
  SRCNN_TRY(srcnn_wrap(ctx, base + 2 * e1 + e2 + e3, e2, &wk->d2));
  SRCNN_TRY(srcnn_wrap(ctx, base + 2 * e1 + 2 * e2 + e3, e3, &wk->d3));
  return SRCNN_OK;
}

// last_layer_delta + deltas(layer 2) + backpropagate(layer 3) in one launch (+ the reduce)
int backward3_fused_entry(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem gt, const Work& wk,
                          int w, int h, int S, int* launched) {
  const Dims d = net_dims(net, w, h);
  const float *pgt, *o3, *o2, *w3;
  float *pd3, *pd2, *gw, *gb;
  SRCNN_TRY(resolve(ctx, gt, sizeof(float) * (size_t)S * w * h, &pgt, "ground truth"));
  SRCNN_TRY(resolve(ctx, wk.out3, sizeof(float) * (size_t)S * d.w3 * d.h3, &o3, "out3"));
  SRCNN_TRY(resolve(ctx, wk.out2, sizeof(float) * (size_t)S * d.w2 * d.h2 * net->n2, &o2, "out2"));
  SRCNN_TRY(resolve(ctx, wk.d3, sizeof(float) * (size_t)S * d.w3 * d.h3, &pd3, "d3"));
  SRCNN_TRY(resolve(ctx, wk.d2, sizeof(float) * (size_t)S * d.w2 * d.h2 * net->n2, &pd2, "d2"));
  SRCNN_TRY(resolve(ctx, net->w[2], sizeof(float) * (size_t)net->f3 * net->f3 * net->n2, &w3, "w3"));
  SRCNN_TRY(resolve(ctx, net->grad_w[2], sizeof(float) * (size_t)net->f3 * net->f3 * net->n2, &gw, "grad_w3"));
  SRCNN_TRY(resolve(ctx, net->grad_b[2], sizeof(float), &gb, "grad_b3"));
  LaunchScope scope(ctx, SRCNN_K_BACKPROPAGATE, 2);
  {   // tensor cores first (batches of patches, 32 channels); 3 launches: d3, main, reduce
    const int rtc = fast::backward3_tc(ctx, pgt, o3, o2, w3, pd3, pd2, gw, gb, net->n2, net->f3, w, h,
                                       d.w3, d.h3, S);
    if (rtc < 0) return rtc;
    if (rtc > 0) {
      *launched = 1;
      return check_launch("bwd3_tc");
    }
  }
  const int rc = train::bwd3_fused(ctx, pgt, o3, o2, w3, pd3, pd2, gw, gb, net->n2, net->f3, w, h,
                                   d.w3, d.h3, S);
  if (rc < 0) return rc;
  *launched = rc;
  if (!rc) scope.n_launches = 0;
  return rc ? check_launch("bwd3_fused") : SRCNN_OK;
}

// layer-1 deltas + layer-1 gradients in one launch: d1 is never materialised
// (replaces `deltas` + `backpropagate` of ConfigBasedDataPipeline.cpp:265-270, 300-320)
int backward1_fused_entry(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, const Work& wk,
                          int w, int h, int S, int* launched) {
  const Dims d = net_dims(net, w, h);
  const float *pin, *o1, *pd2, *w2;
  float *gw, *gb;
  SRCNN_TRY(resolve(ctx, in, sizeof(float) * (size_t)S * w * h, &pin, "input luma"));
  SRCNN_TRY(resolve(ctx, wk.out1, sizeof(float) * (size_t)S * d.w1 * d.h1 * net->n1, &o1, "out1"));
  SRCNN_TRY(resolve(ctx, wk.d2, sizeof(float) * (size_t)S * d.w2 * d.h2 * net->n2, &pd2, "d2"));
  SRCNN_TRY(resolve(ctx, net->w[1], sizeof(float) * (size_t)net->n1 * net->n2, &w2, "w2"));
  SRCNN_TRY(resolve(ctx, net->grad_w[0], sizeof(float) * (size_t)net->f1 * net->f1 * net->n1, &gw, "grad_w1"));
  SRCNN_TRY(resolve(ctx, net->grad_b[0], sizeof(float) * (size_t)net->n1, &gb, "grad_b1"));
  LaunchScope scope(ctx, SRCNN_K_TRAIN_FUSED, 2);
  const int rc = fast::backward1_fused(ctx, pd2, o1, w2, pin, gw, gb, net->n1, net->n2, net->f1,
                                       net->f2, d.w1, d.h1, S);
  if (rc < 0) return rc;
  *launched = rc;
  if (!rc) scope.n_launches = 0;
  return rc ? check_launch("backward1_fused") : SRCNN_OK;
}

// forward of a training chunk through the fused tensor-core kernel, activations kept
// (replaces the three execute_layer calls of ConfigBasedDataPipeline.cpp:200-241)
int forward_train_fused_entry(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, const Work& wk,
                              int w, int h, int S, int* launched) {
  const Dims d = net_dims(net, w, h);
  const float* pin;
  float *o1, *o2, *o3;
  SRCNN_TRY(resolve(ctx, in, sizeof(float) * (size_t)S * w * h, &pin, "input luma"));
  SRCNN_TRY(resolve(ctx, wk.out1, sizeof(float) * (size_t)S * d.w1 * d.h1 * net->n1, &o1, "out1"));
  SRCNN_TRY(resolve(ctx, wk.out2, sizeof(float) * (size_t)S * d.w2 * d.h2 * net->n2, &o2, "out2"));
  SRCNN_TRY(resolve(ctx, wk.out3, sizeof(float) * (size_t)S * d.w3 * d.h3, &o3, "out3"));
  // the operand image only changes when the parameters do (srcnn_update_all, srcnn_write ...):
  // the chunks of an epoch share the context's cached copy
  fast::FusedNet fn;
  SRCNN_TRY(fused_net(ctx, net, &fn));
  LaunchScope scope(ctx, SRCNN_K_FORWARD_FUSED, fast::fused_launches(ctx, fn));
  c5::Maxes* mx;
  SRCNN_TRY(fast::conv5_maxes(ctx, &mx));
  const int rc = fast::forward_train_fused(ctx, fn, pin, o1, o2, o3, w, h, S, &mx->out2);
  if (rc < 0) return rc;
  if (rc > 0) ctx->c5_fresh_out2 = o2;   // max |out2| recorded for the layer-3 backward
  *launched = rc;
  if (!rc) scope.n_launches = 0;
  return rc ? check_launch("forward_train_fused") : SRCNN_OK;
}
}  // namespace

namespace {
// forward (keeping the activations), deltas and gradients of one chunk on six given buffers
int train_chunk_on(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt, int w, int h,
                   int S, const Work& wk) {
  const Dims d = net_dims(net, w, h);
  int rc = SRCNN_OK;
  // 9-5-5: the maxima the layer-2 forward and the layer-1 deltas measure (conv5_tc.cuh) stay
  // valid for the layer-2 gradient of the same chunk
  ctx->c5_max_out1_of = ctx->c5_max_d2_of = nullptr;
  ctx->c5_fresh_out2 = ctx->c5_fresh_d2 = nullptr;
  // the maxima this chunk's producers record describe its buffers only until it returns: a later
  // standalone call on the same buffers (after new data was written into them, or after another
  // call overwrote the context's c5::Maxes) must measure them again
  struct KnownScope {
    srcnn_ctx* c;
    ~KnownScope() {
      c->c5_maxes_known = false;
      c->c5_fresh_out2 = c->c5_fresh_d2 = c->c5_l1_max_of = nullptr;
    }
  } known_scope{ctx};
  // forward, keeping the activations (ConfigBasedDataPipeline.cpp:200-241)
  int fused_fwd = 0;
  if (fast::fused_train_supported(ctx, net->n1, net->n2, net->f1, net->f2, net->f3))
    rc = forward_train_fused_entry(ctx, net, in, wk, w, h, S, &fused_fwd);
  if (!fused_fwd) {
    // 9-5-5: layer 1 through the FP16-split tensor-core kernel in its layer-1-only mode (it also
    // records max |out1| for the layer-2 kernel), layer 2 through conv5_tc
    int l1_tc = 0;
    ctx->c5_l1_max_of = nullptr;
    if (rc == SRCNN_OK && c5::supported(net->n1, net->n2, net->f1, net->f2, net->f3)) {
      const float *pin, *w1, *b1;
      float* o1;
      rc = resolve(ctx, in, sizeof(float) * (size_t)S * w * h, &pin, "input luma");
      if (rc == SRCNN_OK) rc = resolve(ctx, wk.out1, sizeof(float) * (size_t)S * d.w1 * d.h1 * net->n1, &o1, "out1");
      if (rc == SRCNN_OK) rc = resolve(ctx, net->w[0], sizeof(float) * (size_t)net->f1 * net->f1 * net->n1, &w1, "w1");
      if (rc == SRCNN_OK) rc = resolve(ctx, net->b[0], sizeof(float) * (size_t)net->n1, &b1, "b1");
      if (rc == SRCNN_OK) {
        LaunchScope scope(ctx, SRCNN_K_FORWARD, 2);
        l1_tc = fast::conv5_layer1(ctx, pin, o1, w1, b1, net->n1, net->f1, w, h, S);
        if (l1_tc < 0) rc = l1_tc;
        if (l1_tc <= 0) scope.n_launches = 0;
        if (l1_tc > 0) {
          rc = check_launch("forward(layer 1, tc)");
          ctx->c5_l1_max_of = o1;
        }
      }
    }
    if (l1_tc <= 0 && rc == SRCNN_OK) rc = srcnn_forward_layer(ctx, in, wk.out1, net->w[0], net->b[0], 1, net->n1, net->f1, 0, w, h, S);
    if (rc == SRCNN_OK) rc = srcnn_forward_layer(ctx, wk.out1, wk.out2, net->w[1], net->b[1], net->n1, net->n2, net->f2, 0, d.w1, d.h1, S);
    ctx->c5_l1_max_of = nullptr;
    if (rc == SRCNN_OK) rc = srcnn_forward_layer(ctx, wk.out2, wk.out3, net->w[2], net->b[2], net->n2, 1, net->f3, 1, d.w2, d.h2, S);
  }
  // last-layer delta, layer-2 deltas and layer-3 gradients share one pass over out2 when the
  // samples are patch-sized (ConfigBasedDataPipeline.cpp:258-270, 287-295)
  int fused_b3 = 0;
  if (rc == SRCNN_OK) rc = backward3_fused_entry(ctx, net, gt, wk, w, h, S, &fused_b3);
  if (!fused_b3) {
    if (rc == SRCNN_OK) rc = srcnn_last_layer_delta(ctx, gt, wk.out3, wk.d3, w, h, d.w3, d.h3, S);
    if (rc == SRCNN_OK) rc = srcnn_deltas(ctx, wk.d3, wk.out2, wk.d2, net->w[2], net->n2, net->f3, 1, d.w2, d.h2, S);
  }
  // layer-1 deltas and gradients in one launch where instantiated: d1 is then NOT written
  int fused_b1 = 0;
  if (rc == SRCNN_OK) rc = backward1_fused_entry(ctx, net, in, wk, w, h, S, &fused_b1);
  if (!fused_b1 && rc == SRCNN_OK) rc = srcnn_deltas(ctx, wk.d2, wk.out1, wk.d1, net->w[1], net->n1, net->f2, net->n2, d.w1, d.h1, S);
  // gradients (ConfigBasedDataPipeline.cpp:287-320)
  if (!fused_b3 && rc == SRCNN_OK) rc = srcnn_backpropagate(ctx, wk.d3, wk.out2, net->grad_w[2], net->grad_b[2], 1, net->n2, net->f3, d.w3, d.h3, S);
  ctx->c5_maxes_known = ctx->c5_max_out1_of != nullptr && ctx->c5_max_d2_of != nullptr;
  if (rc == SRCNN_OK) rc = srcnn_backpropagate(ctx, wk.d2, wk.out1, net->grad_w[1], net->grad_b[1], net->n2, net->n1, net->f2, d.w2, d.h2, S);
  ctx->c5_maxes_known = false;
  if (!fused_b1 && rc == SRCNN_OK) rc = srcnn_backpropagate(ctx, wk.d1, in, net->grad_w[0], net->grad_b[0], net->n1, 1, net->f1, d.w1, d.h1, S);
  return rc;
}
}  // namespace

int srcnn_train_materializes_d1(srcnn_ctx* ctx, const srcnn_net* net) {
  if (!ctx || !net) return 1;
  return fast::backward1_fused_supported(ctx, net->n1, net->n2, net->f1, net->f2) ? 0 : 1;
}

int srcnn_train_chunk(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt, int w,
                      int h, int S, srcnn_mem work) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, w, h);
  SRCNN_REQUIRE(S > 0 && d.w3 > 0 && d.h3 > 0, "sample %dx%d too small for the network", w, h);
  TableScope views(ctx);   // the six wrapped views of `work` leave the table on every exit path
  Work wk;
  SRCNN_TRY(carve(ctx, net, work, w, h, S, &wk));
  return train_chunk_on(ctx, net, in, gt, w, h, S, wk);
}

int srcnn_train_chunk_buffers(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt,
                              int w, int h, int S, srcnn_mem out1, srcnn_mem out2,
                              srcnn_mem out3, srcnn_mem d1, srcnn_mem d2, srcnn_mem d3) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, w, h);
  SRCNN_REQUIRE(S > 0 && d.w3 > 0 && d.h3 > 0, "sample %dx%d too small for the network", w, h);
  Work wk{out1, out2, out3, d1, d2, d3};
  return train_chunk_on(ctx, net, in, gt, w, h, S, wk);
}

int srcnn_train_chunks_host(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in,
                            const float* host_gt, int w, int h, int n_samples, int chunk,
                            srcnn_mem work) {
  SRCNN_REQUIRE(ctx && host_in && host_gt, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, w, h);
  SRCNN_REQUIRE(n_samples > 0 && chunk > 0 && d.w3 > 0 && d.h3 > 0,
                "bad sample set: %d samples of %dx%d, chunk %d", n_samples, w, h, chunk);
  const size_t per = sizeof(float) * (size_t)w * h;
  const size_t need = per * (size_t)std::min(chunk, n_samples);
  for (int b = 0; b < 2; b++) {
    SRCNN_TRY(ensure_scratch(ctx, &ctx->stage_in[b], &ctx->stage_in_bytes[b], need));
    SRCNN_TRY(ensure_scratch(ctx, &ctx->stage_gt[b], &ctx->stage_gt_bytes[b], need));
  }
  SRCNN_TRY(ensure_side_streams(ctx));
  // the copy stream starts behind whatever the context stream was doing with the staging
  SRCNN_CUDA(cudaEventRecord(ctx->ev_k[2], ctx->stream));
  SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[2], 0));
  int rc = SRCNN_OK;
  // The upload of the FIRST chunk is exposed (nothing to train yet): when there is more than one
  // chunk's worth of samples it is cut to half a chunk (SRCNN_TRAIN_HEAD=0 keeps it whole)
  static const bool kHead = !(std::getenv("SRCNN_TRAIN_HEAD") && std::atoi(std::getenv("SRCNN_TRAIN_HEAD")) == 0);
  const int head = (kHead && n_samples > chunk && chunk >= 512) ? chunk / 2 : chunk;
  for (int i = 0, s0 = 0, S = 0; s0 < n_samples && rc == SRCNN_OK; i++, s0 += S) {
    S = std::min(i == 0 ? head : chunk, n_samples - s0);
    const int b = i & 1;
    // staging b was last read by the training of chunk i-2
    if (i >= 2) SRCNN_CUDA(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[b], 0));
    SRCNN_CUDA(cudaMemcpyAsync(ctx->stage_in[b], host_in + (size_t)s0 * w * h, per * S,
                               cudaMemcpyHostToDevice, ctx->copy_in));
    SRCNN_CUDA(cudaMemcpyAsync(ctx->stage_gt[b], host_gt + (size_t)s0 * w * h, per * S,
                               cudaMemcpyHostToDevice, ctx->copy_in));
    SRCNN_CUDA(cudaEventRecord(ctx->ev_in[b], ctx->copy_in));
    SRCNN_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[b], 0));
    TableScope views(ctx);   // staging + workspace views leave the table on every exit path
    srcnn_mem mi, mg;
    SRCNN_TRY(srcnn_wrap(ctx, ctx->stage_in[b], per * S, &mi));
    SRCNN_TRY(srcnn_wrap(ctx, ctx->stage_gt[b], per * S, &mg));
    Work wk;
    SRCNN_TRY(carve(ctx, net, work, w, h, S, &wk));
    rc = train_chunk_on(ctx, net, mi, mg, w, h, S, wk);
    if (rc == SRCNN_OK) SRCNN_CUDA(cudaEventRecord(ctx->ev_k[b], ctx->stream));
  }
  SRCNN_CUDA(cudaStreamSynchronize(ctx->copy_in));   // the host buffers may be reused
  return rc;
}

int srcnn_update_all(srcnn_ctx* ctx, const srcnn_net* net, unsigned batch_size, float momentum,
                     float weight_decay, const float lr[3]) {
  SRCNN_REQUIRE(ctx && lr, "null argument");
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  SRCNN_REQUIRE(batch_size > 0, "batch_size must be > 0");
  fast::UpdateAllArgs a;
  const int ks[3] = {1, net->n1, net->n2}, ns[3] = {net->n1, net->n2, 1},
            fs[3] = {net->f1, net->f2, net->f3};
  unsigned total = 0;
  for (int l = 0; l < 3; l++) {
    const unsigned ws = (unsigned)(fs[l] * fs[l] * ks[l] * ns[l]), bs = (unsigned)ns[l];
    SRCNN_TRY(resolve(ctx, net->w[l], sizeof(float) * ws, &a.w[l], "weights"));
    SRCNN_TRY(resolve(ctx, net->b[l], sizeof(float) * bs, &a.b[l], "bias"));
    SRCNN_TRY(resolve(ctx, net->grad_w[l], sizeof(float) * ws, &a.gw[l], "grad_w"));
    SRCNN_TRY(resolve(ctx, net->grad_b[l], sizeof(float) * bs, &a.gb[l], "grad_b"));
    SRCNN_TRY(resolve(ctx, net->prev_dw[l], sizeof(float) * ws, &a.pw[l], "previous delta w"));
    SRCNN_TRY(resolve(ctx, net->prev_db[l], sizeof(float) * bs, &a.pb[l], "previous delta b"));
    ctx->note_write(net->w[l]);
    ctx->note_write(net->b[l]);
    a.ws[l] = ws;
    a.bs[l] = bs;
    a.lr[l] = lr[l];
    total += ws + bs;
  }
  a.momentum = momentum;
  a.decay = weight_decay;
  a.batch = (float)batch_size;
  LaunchScope scope(ctx, SRCNN_K_UPDATE_PARAMS);
  fast::update_all_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(a);
  return check_launch("update_all");
}

int srcnn_validate_chunk(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt,
                         int w, int h, int S, srcnn_mem work, srcnn_mem target) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  const Dims d = net_dims(net, w, h);
  SRCNN_REQUIRE(S > 0 && d.w3 > 0 && d.h3 > 0, "sample %dx%d too small for the network", w, h);
  TableScope views(ctx);
  Work wk;
  SRCNN_TRY(carve(ctx, net, work, w, h, S, &wk));
  SRCNN_TRY(srcnn_forward_fused(ctx, net, in, wk.out3, w, h, S, wk.out1, wk.out2));
  return srcnn_squared_error(ctx, gt, wk.out3, target, w, h, d.w3, d.h3, S);
}

// ======================================================================= multi-GPU ====

int srcnn_comm_unique_id(unsigned char id[SRCNN_COMM_ID_BYTES]) {
  SRCNN_REQUIRE(id != nullptr, "id is null");
  comm::Api* api = comm::api();
  if (!api) return fail(SRCNN_ECUDA, "libnccl.so.2 could not be loaded: %s", dlerror());
  static_assert(sizeof(comm::UniqueId) == SRCNN_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  comm::UniqueId u;
  SRCNN_NCCL(api->GetUniqueId(&u), "ncclGetUniqueId");
  std::memcpy(id, &u, sizeof(u));
  return SRCNN_OK;
}

int srcnn_comm_init(srcnn_ctx* ctx, int rank, int world,
                    const unsigned char id[SRCNN_COMM_ID_BYTES]) {
  SRCNN_ENTER(ctx);
  SRCNN_REQUIRE(id != nullptr, "id is null");
  SRCNN_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank %d of %d", rank, world);
  SRCNN_REQUIRE(ctx->nccl_comm == nullptr, "this context already has a communicator");
  comm::Api* api = comm::api();
  if (!api) return fail(SRCNN_ECUDA, "libnccl.so.2 could not be loaded: %s", dlerror());
  comm::UniqueId u;
  std::memcpy(&u, id, sizeof(u));
  comm::ncclComm_t c = nullptr;
  SRCNN_NCCL(api->CommInitRank(&c, world, u, rank), "ncclCommInitRank");
  ctx->nccl_comm = c;
  ctx->comm_rank = rank;
  ctx->comm_world = world;
  return SRCNN_OK;
}

int srcnn_comm_destroy(srcnn_ctx* ctx) {
  SRCNN_ENTER(ctx);
  if (ctx->nccl_comm) {
    SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
    SRCNN_NCCL(comm::api()->CommDestroy(ctx->nccl_comm), "ncclCommDestroy");
  }
  ctx->nccl_comm = nullptr;
  ctx->comm_rank = 0;
  ctx->comm_world = 1;
  return SRCNN_OK;
}

int srcnn_comm_info(srcnn_ctx* ctx, int* rank, int* world) {
  SRCNN_ENTER(ctx);
  if (rank) *rank = ctx->comm_rank;
  if (world) *world = ctx->comm_world;
  return SRCNN_OK;
}

int srcnn_allreduce_sum(srcnn_ctx* ctx, srcnn_mem buf, size_t offset_floats, size_t count) {
  SRCNN_ENTER(ctx);
  Allocation* a = ctx->get(buf);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle in allreduce");
  const size_t total = a->bytes / sizeof(float);
  if (count > total || offset_floats > total - count)
    return fail(SRCNN_ERANGE, "allreduce of %zu floats at %zu outside a buffer of %zu", count,
                offset_floats, total);
  if (!ctx->nccl_comm || ctx->comm_world == 1 || count == 0) return SRCNN_OK;   // sum over one rank
  ctx->note_write(buf);
  float* p = reinterpret_cast<float*>(a->ptr) + offset_floats;
  SRCNN_NCCL(comm::api()->AllReduce(p, p, count, comm::kNcclFloat, comm::kNcclSum, ctx->nccl_comm,
                                    ctx->stream),
             "ncclAllReduce");
  return SRCNN_OK;
}

int srcnn_broadcast(srcnn_ctx* ctx, srcnn_mem buf, size_t count, int root) {
  SRCNN_ENTER(ctx);
  Allocation* a = ctx->get(buf);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle in broadcast");
  if (count > a->bytes / sizeof(float))
    return fail(SRCNN_ERANGE, "broadcast of %zu floats outside a buffer of %zu bytes", count, a->bytes);
  SRCNN_REQUIRE(root >= 0 && root < ctx->comm_world, "bad broadcast root %d", root);
  if (!ctx->nccl_comm || ctx->comm_world == 1 || count == 0) return SRCNN_OK;
  ctx->note_write(buf);
  SRCNN_NCCL(comm::api()->Broadcast(a->ptr, a->ptr, count, comm::kNcclFloat, root, ctx->nccl_comm,
                                    ctx->stream),
             "ncclBroadcast");
  return SRCNN_OK;
}

int srcnn_allreduce_grads(srcnn_ctx* ctx, const srcnn_net* net) {
  SRCNN_ENTER(ctx);
  SRCNN_TRY(check_net(net));
  if (!ctx->nccl_comm || ctx->comm_world == 1) return SRCNN_OK;
  const int ks[3] = {1, net->n1, net->n2}, ns[3] = {net->n1, net->n2, 1},
            fs[3] = {net->f1, net->f2, net->f3};
  float* p[6];
  size_t cnt[6];
  for (int l = 0; l < 3; l++) {
    cnt[2 * l] = (size_t)fs[l] * fs[l] * ks[l] * ns[l];
    cnt[2 * l + 1] = (size_t)ns[l];
    SRCNN_TRY(resolve(ctx, net->grad_w[l], sizeof(float) * cnt[2 * l], &p[2 * l], "grad_w"));
    SRCNN_TRY(resolve(ctx, net->grad_b[l], sizeof(float) * cnt[2 * l + 1], &p[2 * l + 1], "grad_b"));
  }
  // the six accumulators normally are views of ONE flat buffer (gw1 | gb1 | gw2 | gb2 | gw3 |
  // gb3): then the exchange step of the path is a single all-reduce (SURVEY 8e)
  bool flat = true;
  size_t total = cnt[0];
  for (int i = 1; i < 6; i++) {
    flat = flat && p[i] == p[i - 1] + cnt[i - 1];
    total += cnt[i];
  }
  comm::Api* api = comm::api();
  if (flat) {
    SRCNN_NCCL(api->AllReduce(p[0], p[0], total, comm::kNcclFloat, comm::kNcclSum, ctx->nccl_comm,
                              ctx->stream),
               "ncclAllReduce(gradients)");
    return SRCNN_OK;
  }
  SRCNN_NCCL(api->GroupStart(), "ncclGroupStart");
  for (int i = 0; i < 6; i++)
    SRCNN_NCCL(api->AllReduce(p[i], p[i], cnt[i], comm::kNcclFloat, comm::kNcclSum, ctx->nccl_comm,
                              ctx->stream),
               "ncclAllReduce(gradient tensor)");
  SRCNN_NCCL(api->GroupEnd(), "ncclGroupEnd");
  return SRCNN_OK;
}

}  // extern "C"
