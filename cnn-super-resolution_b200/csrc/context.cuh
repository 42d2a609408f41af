// Context, handle table and launch bookkeeping of the C-ABI device layer.
// Replaces the reference's opencl::Context / RawMemoryHandle
// (src/opencl/Context.hpp:53-66,72-299, src/opencl/Context.cpp).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/srcnn_b200.h"

namespace srcnn {

// thread-local last-error text (srcnn_last_error)
inline std::string& last_error_ref() {
  static thread_local std::string s;
  return s;
}

inline int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  last_error_ref() = buf;
  return code;
}

#define SRCNN_CUDA(expr)                                                                   \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return ::srcnn::fail(SRCNN_ECUDA, "CUDA error %s (%d) in `%s` at %s:%d",             \
                           cudaGetErrorString(_e), (int)_e, #expr, __FILE__, __LINE__);    \
  } while (0)

#define SRCNN_REQUIRE(cond, ...)                                      \
  do {                                                                \
    if (!(cond)) return ::srcnn::fail(SRCNN_EINVAL, __VA_ARGS__);     \
  } while (0)

#define SRCNN_TRY(expr)          \
  do {                           \
    int _rc = (expr);            \
    if (_rc != SRCNN_OK) return _rc; \
  } while (0)

struct Allocation {
  void* ptr = nullptr;
  size_t bytes = 0;
  bool released = false;
  bool owned = true;  // false: wrapped caller memory (srcnn_wrap)
  // srcnn_mem_ptr has handed the raw device pointer out: anything (an NCCL broadcast, a torch
  // copy, a kernel on another stream) may write it behind the device layer's back, so derived
  // data (the packed operand image of the fused kernels) is never cached for it
  bool exposed = false;
};

struct KernelStat {
  uint64_t total_ns = 0;
  uint64_t launches = 0;
};

}  // namespace srcnn

struct srcnn_ctx {
  int device = 0;
  bool profile = false;
  bool own_stream = true;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  int sm_count = 0;
  size_t smem_optin = 0;
  std::vector<srcnn::Allocation> allocs;
  srcnn::KernelStat stats[SRCNN_K_COUNT];
  uint64_t launch_count = 0;
  // fused inference implementation: tensor cores (tcgen05, 3xTF32) where instantiated, unless
  // SRCNN_FUSED_IMPL=simt asks for the FP32 SIMT kernel (A/B measurements)
  // 0 simt, 3 planes (3xTF32), 4 planes (FP16 split); the two earlier generations are in the
  // git history (tools/superseded/ at 99b7bf0)
  int fused_impl = 4;
  bool deltas_tc = true;              // f=1 deltas on the tensor cores (deltas_tc.cuh)
  bool wgrad_tc = true;               // layer-1 weight gradient on the tensor cores (wgrad_tc.cuh)
  bool d1_fused = true;               // layer-1 deltas inside the layer-1 gradient kernel
  void* hp_scales = nullptr;          // ring of fused_hp::Scales blocks + their work words
  unsigned long long hp_next = 0;
  // cache of the prepared operand image: valid while the six parameter buffers are the same
  // owned allocations and no device-layer call has written device memory since (write_gen)
  void* hp_cache = nullptr;
  bool hp_cache_valid = false;
  const void* hp_cache_key[6] = {};
  unsigned long long hp_cache_gen = 0;
  int hp_cache_n1 = 0;
  // bumped whenever one of the six buffers the cached image was packed from is written through
  // the device layer (note_write) or by srcnn_invalidate_params
  unsigned long long write_gen = 0;
  srcnn_mem hp_cache_h[6] = {};
  // 9-5-5 layer 2 on the tensor cores (conv5_tc.cuh): packed FP16 hi/lo images of W2, valid
  // while the allocation behind c5_h is untouched; per-chunk maxima of the split operands
  void* c5_images = nullptr;
  bool c5_valid = false;
  const void* c5_key = nullptr;
  srcnn_mem c5_h = SRCNN_NULL_MEM;
  void* c5_maxes = nullptr;
  // tensors whose maxima are in c5_maxes (set by the conv5 launches of the current training
  // chunk, so that its layer-2 gradient does not measure them again)
  const void* c5_max_out1_of = nullptr;
  const void* c5_max_d2_of = nullptr;
  bool c5_maxes_known = false;
  const void* c5_l1_max_of = nullptr;   // out1 whose maximum the layer-1-only kernel recorded
  const void* c5_fresh_out2 = nullptr;  // out2 whose maximum the forward of this chunk recorded
  const void* c5_fresh_d2 = nullptr;    // d2 whose maximum the layer-3 backward recorded
  // (the three pointers above hold inside one training chunk only: cleared when it returns)
  // per-context (= per-device) one-time kernel setup: opt-in dynamic shared memory sizes and
  // occupancy queries, keyed by the kernel's address.  cudaFuncSetAttribute is per DEVICE, so a
  // process-wide flag would leave a second context on another GPU unconfigured.
  std::unordered_map<const void*, std::pair<size_t, int>> func_setup;
  // context-owned scratch: reduction partials, split-K partial tiles, row-band staging
  void* red_scratch = nullptr;      // fixed: kRedScratchBytes
  void* splitk_scratch = nullptr;   // grown on demand
  void* gather_tab = nullptr;       // pointer table of srcnn_gather
  size_t gather_tab_bytes = 0;
  size_t splitk_bytes = 0;
  void* band_in = nullptr;          // srcnn_infer_rows_host staging (device)
  void* band_out = nullptr;
  size_t band_in_bytes = 0, band_out_bytes = 0;
  void* stage_in[2] = {nullptr, nullptr};   // srcnn_train_chunks_host staging (device)
  void* stage_gt[2] = {nullptr, nullptr};
  size_t stage_in_bytes[2] = {0, 0}, stage_gt_bytes[2] = {0, 0};
  // side streams + events of the pipelined host-buffer inference (created on first use)
  cudaStream_t copy_in = nullptr, copy_out = nullptr, compute2 = nullptr;
  // the sub-band pipeline of srcnn_infer_rows_host as an instantiated CUDA graph, replayed while
  // the call's arguments (host / device pointers, shape, band, parameters) stay the same
  // (the sub-band pipelines, srcnn_infer_rows_host and srcnn_upscale_image_host, key their
  // graphs by kGraphKey words of call arguments)
  static constexpr int kGraphKey = 32;
  cudaGraphExec_t e2e_graph = nullptr;
  unsigned long long e2e_key[kGraphKey] = {};
  unsigned e2e_graph_launches[SRCNN_K_COUNT] = {};   // launches per kernel id of one replay
  cudaEvent_t ev_join[2] = {};
  // srcnn_infer_rows_host_async: two lanes, each with its own stream, staging and graph, used
  // alternately, so that the tail (download) of one call overlaps the head (upload, first
  // launches) of the next.  lanes_busy: work may be in flight on a lane stream.
  struct RowsLane {
    cudaStream_t stream = nullptr;
    void* in = nullptr;
    void* out = nullptr;
    size_t in_bytes = 0, out_bytes = 0;
    cudaGraphExec_t graph = nullptr;
    unsigned long long key[kGraphKey] = {};
    unsigned graph_launches[SRCNN_K_COUNT] = {};
    srcnn_mem params[6] = {};   // the parameter buffers the lane's call in flight reads
  } lanes[2];
  unsigned lane_next = 0;
  bool lanes_busy = false;

  cudaEvent_t lane_ev = nullptr;
  // srcnn_resample weight tables, one per (w, h, W, H, filter, input and output chroma siting,
  // sample bit depth); the host copy stays alive because the upload that reads it is asynchronous
  struct ResampleKey {
    int w, h, W, H, filter, siting_in, siting_out, bit_depth;
  };
  struct ResampleTable {
    ResampleKey key;
    std::vector<int> host;
    int* dev = nullptr;
    int rows_max = 0;
  };
  std::vector<ResampleTable> resample_tables;
  // srcnn_upscale_image_host: device staging (grown on demand) and its captured pipeline
  struct UpscaleStaging {
    void* small = nullptr;   // input RGBA8
    void* rgba = nullptr;    // enlarged RGBA8
    void* luma = nullptr;    // enlarged luma, then minus its Q1 mean
    void* out = nullptr;     // network output
    void* rgb = nullptr;     // result RGB8
    void* s1 = nullptr;      // layer 1 / 2 activations of the three-launch route
    void* s2 = nullptr;
    size_t small_bytes = 0, rgba_bytes = 0, luma_bytes = 0, out_bytes = 0, rgb_bytes = 0,
           s1_bytes = 0, s2_bytes = 0;
    cudaGraphExec_t graph = nullptr;
    unsigned long long key[kGraphKey] = {};
    unsigned graph_launches[SRCNN_K_COUNT] = {};
  } up;
  // srcnn_upscale_frames_host (`frames`), srcnn_evaluate_frames_host (`eval`),
  // srcnn_upscale_yuv420_frames_host (`yuv`) and srcnn_upscale_yuv420_frames (`yuv_dev`, which
  // uses luma / out / red / s1 / s2 only): device staging (grown on demand), apart from `up` and
  // from each other so that the entries do not resize (and so re-capture) each other's buffers.
  // small / rgb / ref hold a ring of frame groups, rgba / luma / out / red / qred one group.
  struct FramesStaging {
    void* small = nullptr;   // input RGBA8 (yuv: input I420)
    void* rgba = nullptr;    // enlarged RGBA8 (not used by yuv)
    void* luma = nullptr;    // enlarged luma, then minus its Q1 mean
    void* out = nullptr;     // network output
    void* rgb = nullptr;     // result RGB8 (yuv: result I420)
    void* red = nullptr;     // Q1 reduction partials, then one sum per frame
    void* s1 = nullptr;      // layer 1 / 2 activations of the three-launch route
    void* s2 = nullptr;
    void* ref = nullptr;     // reference RGBA8 (evaluate entry)
    void* qred = nullptr;    // quality reduction partials (evaluate entry)
    void* metrics = nullptr; // 4 doubles a frame of the whole call (evaluate entry)
    size_t small_bytes = 0, rgba_bytes = 0, luma_bytes = 0, out_bytes = 0, rgb_bytes = 0,
           red_bytes = 0, s1_bytes = 0, s2_bytes = 0, ref_bytes = 0, qred_bytes = 0,
           metrics_bytes = 0;
  } frames, eval, yuv, yuv_dev;
  // srcnn_image_quality's reduction partials (grown on demand)
  void* quality_red = nullptr;
  size_t quality_red_bytes = 0;
  static constexpr int kEvents = 32;
  cudaEvent_t ev_in[kEvents] = {}, ev_k[kEvents] = {};
  cudaEvent_t ev_d[4] = {};   // download-finished events of the frame entries' rings
  // data-parallel communicator (NCCL, loaded at run time: comm.cuh); null = single GPU
  void* nccl_comm = nullptr;
  int comm_rank = 0, comm_world = 1;
  // last srcnn_net whose derived (repacked) parameters are cached; see fused kernels
  void* packed_params = nullptr;
  size_t packed_bytes = 0;

  static constexpr size_t kRedScratchBytes = 64 * 1024;

  // a device-layer call is about to write the allocation behind `h`
  // waits for the calls srcnn_infer_rows_host_async has in flight
  cudaError_t drain_lanes() {
    if (!lanes_busy) return cudaSuccess;
    lanes_busy = false;
    for (RowsLane& l : lanes)
      if (l.stream) {
        const cudaError_t e = cudaStreamSynchronize(l.stream);
        if (e != cudaSuccess) return e;
      }
    return cudaSuccess;
  }

  void note_write(srcnn_mem h) {
    if (lanes_busy)
      for (int i = 0; i < 12; i++)
        if (lanes[i / 6].params[i % 6] == h) {
          drain_lanes();   // an asynchronous inference is still reading these parameters
          break;
        }
    for (int i = 0; i < 6; i++)
      if (hp_cache_valid && hp_cache_h[i] == h) write_gen++;
    if (c5_valid && c5_h == h) c5_valid = false;
  }

  srcnn::Allocation* get(srcnn_mem h) {
    if (h >= allocs.size()) return nullptr;
    srcnn::Allocation* a = &allocs[h];
    if (a->released || a->ptr == nullptr) return nullptr;
    return a;
  }
};

namespace srcnn {

// RAII bracket around one kernel launch: counts it and, in profile mode, times it with a
// cudaEvent pair and blocks (reference: src/opencl/Kernel.cpp:108-116).
struct LaunchScope {
  srcnn_ctx* ctx;
  int id;
  int n_launches;
  LaunchScope(srcnn_ctx* c, int kernel_id, int launches = 1)
      : ctx(c), id(kernel_id), n_launches(launches) {
    if (ctx->profile) cudaEventRecord(ctx->ev_start, ctx->stream);
  }
  ~LaunchScope() {
    ctx->launch_count += (uint64_t)n_launches;
    ctx->stats[id].launches += (uint64_t)n_launches;
    if (ctx->profile) {
      cudaEventRecord(ctx->ev_stop, ctx->stream);
      cudaEventSynchronize(ctx->ev_stop);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop);
      ctx->stats[id].total_ns += (uint64_t)((double)ms * 1e6);
    }
  }
};

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    return fail(SRCNN_ECUDA, "kernel launch `%s` failed: %s (%d)", what, cudaGetErrorString(e),
                (int)e);
  return SRCNN_OK;
}

// resolve a handle to a typed device pointer, checking it holds at least `need` bytes
template <class T>
inline int resolve(srcnn_ctx* ctx, srcnn_mem h, size_t need, T** out, const char* what) {
  Allocation* a = ctx->get(h);
  if (!a) return fail(SRCNN_EHANDLE, "invalid memory handle for `%s` (%llu)", what,
                      (unsigned long long)h);
  if (a->bytes < need)
    return fail(SRCNN_ERANGE, "buffer `%s` too small: %zu bytes allocated, %zu needed", what,
                a->bytes, need);
  *out = reinterpret_cast<T*>(a->ptr);
  return SRCNN_OK;
}

// Opt-in dynamic shared memory of `kernel` on this context's device, once per context and size;
// with `occ` also the resident CTAs per SM at `threads` threads.
template <class Kernel>
inline int ensure_func_setup(srcnn_ctx* ctx, Kernel kernel, size_t smem, int threads = 0,
                             int* occ = nullptr) {
  const void* key = reinterpret_cast<const void*>(kernel);
  auto it = ctx->func_setup.find(key);
  if (it == ctx->func_setup.end() || it->second.first != smem || (occ && it->second.second < 0)) {
    SRCNN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int q = -1;
    if (occ) SRCNN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kernel, threads, smem));
    ctx->func_setup[key] = std::make_pair(smem, q);
    it = ctx->func_setup.find(key);
  }
  if (occ) *occ = it->second.second;
  return SRCNN_OK;
}

// every C-ABI entry starts here: the context must exist and its device must be current (a
// caller thread, or torch, may have switched devices since the context was created)
#define SRCNN_ENTER(ctx)                                                    \
  do {                                                                      \
    if (!(ctx)) return ::srcnn::fail(SRCNN_EINVAL, "ctx is null");          \
    int _dev = -1;                                                          \
    if (cudaGetDevice(&_dev) != cudaSuccess || _dev != (ctx)->device)       \
      SRCNN_CUDA(cudaSetDevice((ctx)->device));                             \
  } while (0)

inline int ensure_scratch(srcnn_ctx* ctx, void** ptr, size_t* have, size_t need) {
  if (*have >= need) return SRCNN_OK;
  if (*ptr) {
    SRCNN_CUDA(cudaStreamSynchronize(ctx->stream));
    SRCNN_CUDA(cudaFree(*ptr));
    *ptr = nullptr;
    *have = 0;
  }
  cudaError_t e = cudaMalloc(ptr, need);
  if (e != cudaSuccess) return fail(SRCNN_ENOMEM, "scratch allocation of %zu bytes failed", need);
  *have = need;
  return SRCNN_OK;
}

}  // namespace srcnn
