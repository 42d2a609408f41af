/*
 * srcnn_b200.h -- C-ABI of the B200 (sm_100a) SRCNN device layer.
 *
 * This is the drop-in boundary: it replaces the reference's OpenCL runtime wrapper
 * (src/opencl/{Context,Kernel,UtilsOpenCL}.{hpp,cpp}) and its ten OpenCL kernels
 * (src/kernel/ *.cl).  The C++ host classes that keep the reference's API
 * (cnn-super-resolution_b200/host: DataPipeline, ConfigBasedDataPipeline, LayerData,
 * Config, `cnn` CLI) call ONLY these functions; so do tests/ (through ctypes) and bench.py.
 * Plain pointers and sizes only -- no C++ or torch types.  Every entry cites the reference
 * interface it replaces (paths relative to the reference repository root).
 *
 * Conventions
 *   - every function returns 0 on success, a negative SRCNN_E* code on failure; the message
 *     is available from srcnn_last_error() (thread-local).  The reference prints
 *     "[OPENCL ERROR] ..." and throws std::runtime_error (src/opencl/Context.cpp:111-123);
 *     the C++ host shim re-throws from the status code.
 *   - one context = one device + one in-order stream (reference: one in-order command queue,
 *     src/opencl/Context.cpp:70-73).  Not thread-safe, like the reference.
 *   - memory handles are indices into a context-owned table, never reused; the context owns
 *     all device memory until it is destroyed (src/opencl/Context.cpp:164-176, 98-101).
 *   - layouts: activations [S][H][W][C] (C fastest), weights [f][f][C_in][C_out] (C_out
 *     fastest), ground truth [S][H][W]  (src/kernel/layer_uber_kernel.cl:1-34).
 *   - all launches are asynchronous on the context's stream; srcnn_block() waits.
 *   - there is NO CPU fallback: without a CUDA device srcnn_ctx_create fails.
 */
#ifndef SRCNN_B200_H
#define SRCNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRCNN_OK 0
#define SRCNN_EINVAL (-1)   /* bad argument / failed validation                         */
#define SRCNN_ECUDA (-2)    /* a CUDA runtime call failed                               */
#define SRCNN_ENOMEM (-3)   /* device allocation failed                                 */
#define SRCNN_EHANDLE (-4)  /* unknown / released memory handle                         */
#define SRCNN_ERANGE (-5)   /* read/write/copy outside an allocation                    */

typedef struct srcnn_ctx srcnn_ctx; /* replaces opencl::Context (src/opencl/Context.hpp:72) */
typedef uint64_t srcnn_mem;         /* replaces opencl::MemoryHandle (Context.hpp:48)       */
/* replaces gpu_nullptr (src/DataPipeline.hpp:7) */
#define SRCNN_NULL_MEM ((srcnn_mem)1 << 30)

/* kernel ids, for per-kernel profiling totals (reference: one opencl::Kernel object per
 * .cl entry point, src/DataPipeline.cpp:121-180) */
enum srcnn_kernel_id {
  SRCNN_K_FORWARD = 0,       /* layer_uber_kernel.cl  `forward`            */
  SRCNN_K_SQUARED_ERR,       /* squared_error.cl      `squared_err`        */
  SRCNN_K_LAST_LAYER_DELTA,  /* last_layer_delta.cl   `last_layer_delta`   */
  SRCNN_K_DELTAS,            /* layer_deltas.cl       `deltas`             */
  SRCNN_K_BACKPROPAGATE,     /* backpropagate.cl      `backpropagate`      */
  SRCNN_K_UPDATE_PARAMS,     /* update_parameters.cl  `update_params`      */
  SRCNN_K_SUM,               /* sum.cl                `sum`                */
  SRCNN_K_SUB_FROM_ALL,      /* subtract_from_all.cl  `sub_from_all`       */
  SRCNN_K_EXTRACT_LUMA,      /* extract_luma.cl       `extract_luma`       */
  SRCNN_K_SWAP_LUMA,         /* swap_luma.cl          `swap_luma`          */
  SRCNN_K_FORWARD_FUSED,     /* (new) layers 1-3 in one launch, inference  */
  SRCNN_K_TRAIN_FUSED,       /* (new) fused pieces of the training step    */
  SRCNN_K_RESAMPLE,          /* (new) Pillow-exact enlargement             */
  SRCNN_K_QUALITY,           /* (new) PSNR / SSIM of image pairs           */
  SRCNN_K_COUNT
};

/* ---------------------------------------------------------------- context ---------- */

/* Context::init(bool profile)  (src/opencl/Context.cpp:45-79).  `device` = CUDA ordinal.
 * `profile` != 0 times every launch with a cudaEvent pair and blocks on it, like
 * CL_QUEUE_PROFILING_ENABLE + clWaitForEvents (src/opencl/Kernel.cpp:108-116). */
int srcnn_ctx_create(int device, int profile, srcnn_ctx** out);
/* Same, but enqueue on a caller-owned cudaStream_t (e.g. a torch.cuda.Stream()) so that
 * launches order with the caller's own work (NCCL all-reduce of the gradient).  A null
 * cuda_stream -- which is also what the legacy default stream, e.g. torch's current stream in a
 * process that never switched streams, reports as its handle -- is not that stream: the context
 * then creates a non-blocking stream of its own, which does not order with the default stream. */
int srcnn_ctx_create_on_stream(int device, void* cuda_stream, int profile, srcnn_ctx** out);
/* Context::~Context / _cleanup (src/opencl/Context.cpp:81-109): waits, frees everything. */
int srcnn_ctx_destroy(srcnn_ctx* ctx);
/* message of the last failed call on this thread */
const char* srcnn_last_error(void);
/* Context::block()  (src/opencl/Context.cpp:153-162): flush + finish. */
int srcnn_block(srcnn_ctx* ctx);
/* device name / SM count / global memory, for the "DEVICE:" line (Context.cpp:62) */
int srcnn_device_info(srcnn_ctx* ctx, char* name, size_t name_len, int* sm_count,
                      size_t* global_mem_bytes);
/* accumulated device time (ns) and launch count of one kernel id while profiling
 * (Kernel::get_total_execution_time, src/opencl/Kernel.hpp:64-66) */
int srcnn_profile_get(srcnn_ctx* ctx, int kernel_id, uint64_t* total_ns, uint64_t* launches);
/* number of kernel launches this context has issued (all ids); bench.py's gpu_launches */
int srcnn_launch_count(srcnn_ctx* ctx, uint64_t* launches);
/* the cudaStream_t this context enqueues on */
int srcnn_stream(srcnn_ctx* ctx, void** cuda_stream);

/* ---------------------------------------------------------------- memory ----------- */

/* Context::allocate(flags,size)  (src/opencl/Context.cpp:164-176) */
int srcnn_alloc(srcnn_ctx* ctx, size_t bytes, srcnn_mem* out);
/* register caller-owned device memory (a torch tensor's data_ptr) under a handle; the
 * context never frees it */
int srcnn_wrap(srcnn_ctx* ctx, void* device_ptr, size_t bytes, srcnn_mem* out);
/* RawMemoryHandle::release()  (src/opencl/Context.cpp:26-33); the handle stays invalid */
int srcnn_release(srcnn_ctx* ctx, srcnn_mem mem);
/* RawMemoryHandle::size via Context::raw_memory  (src/opencl/Context.cpp:125-130) */
int srcnn_mem_size(srcnn_ctx* ctx, srcnn_mem mem, size_t* bytes);
int srcnn_mem_ptr(srcnn_ctx* ctx, srcnn_mem mem, void** device_ptr);
/* Context::print_app_memory_usage (src/opencl/Context.cpp:132-149): bytes currently held */
int srcnn_mem_usage(srcnn_ctx* ctx, size_t* buffer_bytes);
/* Context::write_buffer(handle, offset, size, src, block)  (Context.cpp:262-294) */
int srcnn_write(srcnn_ctx* ctx, srcnn_mem mem, size_t offset, size_t bytes, const void* src,
                int block);
/* Context::read_buffer(handle, offset, size, dst, block)  (Context.cpp:235-260) */
int srcnn_read(srcnn_ctx* ctx, srcnn_mem mem, size_t offset, size_t bytes, void* dst,
               int block);
/* Context::copy_buffer(src, dst, dst_offset)  (Context.cpp:312-341): copies ALL of src */
int srcnn_copy(srcnn_ctx* ctx, srcnn_mem src, srcnn_mem dst, size_t dst_offset);
/* partial device-to-device copy (new; used by the batched sample gather) */
int srcnn_copy_region(srcnn_ctx* ctx, srcnn_mem src, size_t src_offset, srcnn_mem dst,
                      size_t dst_offset, size_t bytes);
/* the sample gather of ConfigBasedDataPipeline::execute_batch
 * (src/ConfigBasedDataPipeline.cpp:149-161: one clEnqueueCopyBuffer per sample and tensor) as
 * ONE launch: `n` buffers of `bytes_each` bytes (a multiple of 4) land in consecutive slots of
 * dst */
int srcnn_gather(srcnn_ctx* ctx, const srcnn_mem* src, int n, size_t bytes_each, srcnn_mem dst);
/* Context::fill_float / zeros_float  (Context.cpp:296-310): whole buffer, on the device */
int srcnn_fill_float(srcnn_ctx* ctx, srcnn_mem mem, float value);
/* pinned host staging memory for the e2e path (new) */
int srcnn_host_alloc(size_t bytes, void** host_ptr);
int srcnn_host_free(void* host_ptr);

/* ---------------------------------------------------------------- kernels ---------- */

/* kernel `forward` + DataPipeline::execute_layer's launch
 * (src/kernel/layer_uber_kernel.cl:36-96, src/DataPipeline.cpp:392-409):
 *   out[s][y][x][n] = act(B[n] + sum_{dy,dx,k} W[dy][dx][k][n] * in[s][y+dy][x+dx][k])
 * k = PREVIOUS_FILTER_COUNT, n = CURRENT_FILTER_COUNT, f = F_SPATIAL_SIZE, skip_relu =
 * SKIP_RELU.  Sizes are validated against the allocations. */
int srcnn_forward_layer(srcnn_ctx* ctx, srcnn_mem in, srcnn_mem out, srcnn_mem W, srcnn_mem B,
                        int k, int n, int f, int skip_relu, int in_w, int in_h, int S);

/* kernel `squared_err` (src/kernel/squared_error.cl:36-92, DataPipeline.cpp:416-472):
 * *target = sum_{s,y,x} (algo[s][y][x] - gt[s][y+p][x+p])^2, p = (gt_w - algo_w)/2.
 * `target` is a 1-float buffer; it is zeroed first (DataPipeline.cpp:441-444).  The
 * reduction is deterministic (fixed-order two-stage), unlike the reference's CAS atomics. */
int srcnn_squared_error(srcnn_ctx* ctx, srcnn_mem gt, srcnn_mem algo, srcnn_mem target,
                        int gt_w, int gt_h, int algo_w, int algo_h, int S);

/* kernel `last_layer_delta` (src/kernel/last_layer_delta.cl:14-50):
 * target[s][y][x] = (y - t) * [y > 0]   (quirk Q2 kept). */
int srcnn_last_layer_delta(srcnn_ctx* ctx, srcnn_mem gt, srcnn_mem algo, srcnn_mem target,
                           int gt_w, int gt_h, int algo_w, int algo_h, int S);

/* kernel `deltas` (src/kernel/layer_deltas.cl:42-127, DataPipeline.cpp:522-594):
 * target[s][j][i][n] = [layer_output>0] * sum_{dy,dx,k} W[dy][dx][n][k]*deltas_next[s][j-dy][i-dx][k]
 * n_curr = CURRENT_FILTER_COUNT (layer l-1), f_next/n_next = layer l, out_w/out_h = extent of
 * layer l-1's output. */
int srcnn_deltas(srcnn_ctx* ctx, srcnn_mem deltas_next, srcnn_mem layer_output,
                 srcnn_mem target, srcnn_mem W, int n_curr, int f_next, int n_next, int out_w,
                 int out_h, int S);

/* kernel `backpropagate` (src/kernel/backpropagate.cl:56-114, DataPipeline.cpp:596-663):
 * grad_w[dy][dx][k][n] += sum_{s,row,col} deltas[s][row][col][n]*layer_input[s][row+dy][col+dx][k]
 * grad_b[n]            += sum deltas[..][n].   ACCUMULATES; deterministic order. */
int srcnn_backpropagate(srcnn_ctx* ctx, srcnn_mem deltas, srcnn_mem layer_input,
                        srcnn_mem grad_w, srcnn_mem grad_b, int n, int k, int f, int out_w,
                        int out_h, int S);

/* kernel `update_params` (src/kernel/update_parameters.cl:1-33, DataPipeline.cpp:665-729),
 * quirk Q3 kept: dw = m*prev + lr*g + decay*w; w -= dw/batch; prev = dw (bias: no decay). */
int srcnn_update_params(srcnn_ctx* ctx, srcnn_mem w, srcnn_mem b, srcnn_mem grad_w,
                        srcnn_mem grad_b, srcnn_mem prev_dw, srcnn_mem prev_db, float momentum,
                        float weight_decay, float learning_rate, unsigned batch_size,
                        unsigned weights_size, unsigned bias_size);

/* kernel `sum` (src/kernel/sum.cl:35-68, DataPipeline.cpp:282-313): *target = sum data[i]
 * or sum data[i]^2 over the first `len` floats; target is zeroed first. */
int srcnn_sum(srcnn_ctx* ctx, srcnn_mem data, unsigned len, int squared, srcnn_mem target);

/* kernel `sub_from_all` (src/kernel/subtract_from_all.cl:1-8) */
int srcnn_sub_from_all(srcnn_ctx* ctx, srcnn_mem data, float value, unsigned len);

/* kernel `extract_luma` (src/kernel/extract_luma.cl:7-23, DataPipeline.cpp:186-220):
 * rgba = w*h*4 bytes (RGBA8, the reference's image2d_t), target = w*h floats. */
int srcnn_extract_luma(srcnn_ctx* ctx, srcnn_mem rgba, srcnn_mem target, int w, int h,
                       int normalize);

/* kernel `swap_luma` (src/kernel/swap_luma.cl:18-69, DataPipeline.cpp:222-266):
 * target = gt_w*gt_h*3 bytes RGB8. */
int srcnn_swap_luma(srcnn_ctx* ctx, srcnn_mem rgba, srcnn_mem new_luma, srcnn_mem target,
                    int gt_w, int gt_h, int luma_w, int luma_h);

/* Image enlargement, byte for byte Pillow's Image.fromarray(rgb, "RGB").resize((out_w, out_h),
 * BICUBIC | LANCZOS) (libImaging/Resample.c): the step before the reference's forward flow
 * (src/Main_cl.cpp:217-239), whose input is an already-enlarged image.  rgba_in = w*h*4 bytes
 * RGBA8 (alpha ignored), rgba_out = out_w*out_h*4 bytes (alpha 255), luma_out = out_w*out_h
 * floats: the luma of rgba_out exactly as srcnn_extract_luma(normalize = 1) computes it, or
 * SRCNN_NULL_MEM for none.  Enlargements only (out_w >= w, out_h >= h); an axis whose size does
 * not change is copied.  One launch. */
enum { SRCNN_RESAMPLE_BICUBIC = 0, SRCNN_RESAMPLE_LANCZOS = 1 };
int srcnn_resample(srcnn_ctx* ctx, srcnn_mem rgba_in, int w, int h, srcnn_mem rgba_out,
                   srcnn_mem luma_out, int out_w, int out_h, int filter);

/* Enlargement quality: the PSNR / SSIM inputs of S image pairs on the device.  result holds S
 * frames of w*h*result_bpp bytes (result_bpp = 3: RGB8 as srcnn_swap_luma writes it, 4: RGBA8),
 * reference S frames of w*h RGBA8; out receives 2*S doubles, {mse, ssim} per frame, over the
 * region [border, w-border) x [border, h-border).  Both are taken on the luma srcnn_extract_luma
 * computes with normalize = 1 (data range 1):
 *   mse  = mean over the region of d^2, d = Y_result - Y_reference in float, d^2 and the sum in
 *          double; PSNR = 10 log10(1 / mse) (+inf for mse = 0) is the caller's;
 *   ssim = Wang et al. 2004 (`ssim_index`): the mean over every 11x11 window wholly inside the
 *          region of the SSIM of the window, Gaussian weights (sigma 1.5, sum 1), C1 = 0.01^2,
 *          C2 = 0.03^2, population (co)variances E[xy] - mx*my.
 * A frame's result does not depend on S or on the other frames, and repeats bit for bit.  A
 * region smaller than 11x11, a negative border, S outside [1, 65535] or result_bpp other than 3
 * or 4: SRCNN_EINVAL.  2 launches. */
int srcnn_image_quality(srcnn_ctx* ctx, srcnn_mem result, int result_bpp, srcnn_mem reference,
                        int w, int h, int S, int border, srcnn_mem out);

/* ---------------------------------------------------------------- fused hot path --- */

typedef struct srcnn_net {
  int n1, n2, f1, f2, f3;        /* Config n1,n2,f1,f2,f3 (src/Config.hpp:27-29)          */
  srcnn_mem w[3], b[3];          /* LayerAllocationPool::weights / bias                    */
  srcnn_mem grad_w[3], grad_b[3];/* accumulating_grad_w / _b   (DataPipeline.hpp:11-29)   */
  srcnn_mem prev_dw[3], prev_db[3]; /* previous_batch_delta_w / _b                         */
} srcnn_net;

/* ConfigBasedDataPipeline::forward(w,h,S) for INFERENCE
 * (src/ConfigBasedDataPipeline.cpp:200-241) as ONE launch: layers 1-3 fused, the n1- and
 * n2-channel maps live in shared memory only.  in = [S][h][w] luma, out = [S][h3][w3].
 * Falls back to three srcnn_forward_layer launches through `scratch1/scratch2` for shapes the
 * fused kernel is not instantiated for (pass SRCNN_NULL_MEM to forbid the fallback). */
int srcnn_forward_fused(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem out,
                        int in_w, int in_h, int S, srcnn_mem scratch1, srcnn_mem scratch2);
/* 1 when srcnn_forward_fused has a fused instantiation for this shape */
int srcnn_forward_fused_supported(const srcnn_net* net);

/* Row-band inference on HOST buffers (the reference-facing e2e call): uploads input rows
 * [row0 - halo .. row1 + halo) of a [h][w] luma image, runs the fused forward, downloads
 * output rows [row0,row1) of the [h3][w3] result into host_out (which points at row row0).
 * halo = f1+f2+f3-3 input rows per band (SURVEY 8e).  Used by bench.py e2e and by the
 * multi-GPU row-band sharding: rank g calls it with its own [row0,row1).
 * Bands of >= 256 output rows are cut into sub-bands whose upload, compute and download
 * overlap on separate streams; that pipeline is captured into a CUDA graph owned by the
 * context and replayed while the call's arguments (both host pointers, shape, band, network
 * buffers) repeat -- the buffers' CONTENTS are read afresh on every call.  Synchronous: the
 * result is in host_out on return.  Pinned host buffers give the PCIe rate; pageable ones work. */
int srcnn_infer_rows_host(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in, int in_w,
                          int in_h, int out_row0, int out_row1, float* host_out);
/* The same call, NON-BLOCKING: the reference's read_buffer(..., block = false) followed by
 * Context::block() (src/opencl/Context.cpp:255-276, 120-126).  Returns once the work is queued;
 * host_out is complete (and host_in may be rewritten) after srcnn_block(ctx) or after the next
 * blocking device-layer call on the parameters.  Two calls can be in flight: consecutive calls
 * alternate between two lanes (stream + staging + graph each), so that for a STREAM of images
 * the download of image i overlaps the upload and the first launches of image i+1 -- the
 * throughput tends to max(H2D, compute, D2H) per image instead of one call's head + tail on top.
 * Calls in flight must not share host_out.  Pinned host buffers are required for the overlap.
 * A device-layer write to the network's parameters, or a call with other parameters, first waits
 * for the calls in flight; in profile mode (and with SRCNN_E2E_GRAPH=0) the call is blocking. */
int srcnn_infer_rows_host_async(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in,
                                int in_w, int in_h, int out_row0, int out_row1, float* host_out);

/* The `cnn` forward mode for an image that must first be enlarged, on HOST buffers: host_rgba
 * (w*h*4 bytes RGBA8) is enlarged to out_w x out_h by srcnn_resample, and host_rgb receives
 * out_w*out_h*3 bytes: exactly what the forward mode (src/Main_cl.cpp:217-239) returns for the
 * enlarged image -- luma/255, minus the Q1 "mean" (the mean of the SQUARES, computed and
 * subtracted on the device), the three layers, swap_luma.  Synchronous; pageable buffers work.
 * Networks with a fused kernel run the sub-band pipeline of srcnn_infer_rows_host (forward,
 * swap_luma and download of consecutive sub-bands overlap; captured into a CUDA graph and replayed
 * while the arguments repeat); the others run the whole image through the three-launch path.
 * Launches per call: 4 + n_sub * (F + 1) with a fused kernel (F = launches of one
 * srcnn_forward_fused call with the packed operand image cached, n_sub = 1 below 256 network
 * output rows, else min(max(S, 2), 32, max(2, h3 / 64)) with h3 = out_h - padding and S = 16 or
 * SRCNN_E2E_SUBBANDS), 4 + L + 1 without (L = launches of srcnn_forward_fused on the three-launch path),
 * plus 1 when the network's packed operand image has to be rebuilt (first call, new parameters).
 * Out of range sizes, an output smaller than padding + 1 or an unknown filter: SRCNN_EINVAL. */
int srcnn_upscale_image_host(srcnn_ctx* ctx, const srcnn_net* net, const unsigned char* host_rgba,
                             int w, int h, int out_w, int out_h, int filter,
                             unsigned char* host_rgb);

/* srcnn_upscale_image_host for MANY equal-sized frames (a folder of photos, the frames of a
 * video): host_rgba holds n_frames frames of w*h*4 bytes RGBA8, host_rgb receives n_frames frames
 * of out_w*out_h*3 bytes RGB8.  Frame i of the result is byte for byte what
 * srcnn_upscale_image_host returns for frame i alone.  Synchronous; pageable buffers work, pinned
 * ones give the overlap.  Waits for srcnn_infer_rows_host_async calls in flight first.
 * Networks with a fused kernel run groups of frames through a ring of device slots: the upload of
 * group g+1 (copy-in stream) and the download of group g-1 (copy-out stream) overlap the device
 * work of group g, which is one launch per step with every frame of the group in the grid:
 * enlargement + luma, the Q1 sum (per frame, with the block partition of a single frame), minus
 * the mean, the fused forward, swap_luma.  A group holds as many frames as fit ~128 MB of device
 * staging (w*h*4 + out_w*out_h*11 + h3*w3*4 bytes a frame; 4 frames of 960x540 -> 1920x1080), or
 * SRCNN_FRAMES_GROUP frames when that is set (at most 65535).  Networks without a fused kernel run
 * frame by frame through the image entry's three-launch route: conv5_tc takes its operand scale
 * from its whole input, so a batch of frames could change a frame's result.
 * Launches per call: n_groups * (5 + F) with a fused kernel (n_groups = ceil(n_frames / group),
 * F = launches of one srcnn_forward_fused call with the packed operand image cached),
 * n_frames * (4 + L + 1) without (L as for srcnn_upscale_image_host), plus 1 when the network's
 * packed operand image has to be rebuilt.  Everything srcnn_upscale_image_host rejects, n_frames
 * <= 0 and null pointers: SRCNN_EINVAL before any host buffer is read or written. */
int srcnn_upscale_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const unsigned char* host_rgba,
                              int w, int h, int n_frames, int out_w, int out_h, int filter,
                              unsigned char* host_rgb);

/* srcnn_upscale_frames_host for video as decoders hand it out and encoders take it: planar
 * Y'CbCr 4:2:0 (I420, `yuv420p`, the frames of a Y4M file) in and out.  A frame is its Y plane
 * (w*h bytes), then Cb, then Cr ((w/2)*(h/2) bytes each): host_in holds n_frames frames of
 * w*h*3/2 bytes, host_out receives n_frames frames of out_w*out_h*3/2 bytes.  Per frame:
 *   - Y is enlarged to out_w x out_h with Pillow's 8-bit filter (its "L" mode, the arithmetic of
 *     srcnn_resample on one channel); its luma Y'/255, minus the Q1 "mean" (the mean of the
 *     squares), goes through the three layers; inside the network's output region the result is
 *     clamp(luma * 255, 0, 255) truncated -- the byte swap_luma writes for a pixel with zero
 *     chroma -- and the border of (f1+f2+f3-3)/2 rows and columns keeps the enlarged Y, as
 *     swap_luma leaves it.
 *   - Cb and Cr are each enlarged (w/2, h/2) -> (out_w/2, out_h/2) with the same filter, for
 *     centre-sited chroma (SRCNN_CHROMA_CENTER; srcnn_upscale_yuv420_frames_host_sited takes
 *     others): Pillow's enlargement, which maps pixel centres onto pixel centres.
 *   - The network sees the Y plane as stored: there is no range conversion, full or limited.
 * A frame's bytes do not depend on the other frames of the call or on the group size.
 * Synchronous; pageable buffers work, pinned ones give the overlap.  Waits for
 * srcnn_infer_rows_host_async calls in flight first.  Staging is the context's and apart from the
 * other entries'.  Networks with a fused kernel run groups of frames through the ring of
 * srcnn_upscale_frames_host; the device work of a group is one launch per step with every frame
 * in the grid: the enlargement of all three planes straight into the result slot + the luma, the
 * Q1 sum (2), minus the mean, the fused forward, the Y write.  A group holds as many frames as fit
 * ~128 MB of device staging (3 * (w*h*3/2 + out_w*out_h*3/2) + out_w*out_h*4 + h3*w3*4 bytes a
 * frame: input and result in each of the 3 ring slots, luma, network output; 4 frames of 960x540
 * -> 1920x1080), or SRCNN_FRAMES_GROUP frames when that is set (at most 21845).  Networks without
 * a fused kernel run frame by frame (upload, head, forward, Y write, download), for the reason
 * srcnn_upscale_frames_host gives.
 * Launches per call: n_groups * (5 + F) with a fused kernel, n_frames * (4 + L + 1) without (F, L
 * as for srcnn_upscale_frames_host), plus 1 when the network's packed operand image has to be
 * rebuilt.  Everything srcnn_upscale_image_host rejects, an odd w, h, out_w or out_h, n_frames <= 0
 * and null pointers: SRCNN_EINVAL before any host buffer is read or written.
 * It is srcnn_upscale_yuv420_frames_host_sited with both sitings SRCNN_CHROMA_CENTER. */
int srcnn_upscale_yuv420_frames_host(srcnn_ctx* ctx, const srcnn_net* net,
                                     const unsigned char* host_in, int w, int h, int n_frames,
                                     int out_w, int out_h, int filter, unsigned char* host_out);

/* Where a 4:2:0 chroma sample sits inside its 2x2 luma cell, per axis in chroma samples: s = 0.5
 * is centred, s = 0.25 co-sited with the even luma column or row.
 *
 *   siting                 s_x   s_y   Y4M tag (ffmpeg)   H.273 chroma_sample_loc_type
 *   SRCNN_CHROMA_CENTER    0.5   0.5   C420jpeg, C420     1 (JPEG)
 *   SRCNN_CHROMA_LEFT      0.25  0.5   C420mpeg2          0 (H.264 / HEVC without a signal)
 *   SRCNN_CHROMA_TOPLEFT   0.25  0.25  C420paldv          2 (UHD / BT.2020, AV1 "colocated")
 *
 * A chroma axis from n_in samples sited at s_in to n_out samples sited at s_out is Pillow's
 * enlargement of a box that starts at in0, computed in double in this order:
 *   scale = (double)n_in / n_out;  in0 = (s_out - 0.5) * scale + (0.5 - s_in);
 *   output i takes the taps around center = in0 + (i + 0.5) * scale
 * (then the taps, weights, normalisation and 22-bit rounding of srcnn_resample).  Centre to centre
 * gives in0 = 0.0 exactly, Pillow's plain enlargement.  An axis is copied only when n_in == n_out
 * and in0 == 0.0; a siting conversion on an axis whose size does not change is resampled, as
 * Pillow resamples a box with a non-zero start.  Luma is never affected. */
enum { SRCNN_CHROMA_CENTER = 0, SRCNN_CHROMA_LEFT = 1, SRCNN_CHROMA_TOPLEFT = 2 };

/* srcnn_upscale_yuv420_frames_host for chroma sited at in_siting in host_in, written sited at
 * out_siting in host_out (SRCNN_CHROMA_*; they may differ, which converts the siting): Cb and Cr
 * are enlarged as the definition above gives; Y, the launches, copies and groups are those of
 * srcnn_upscale_yuv420_frames_host.  A siting pair's chroma table is built and uploaded on the
 * pair's first call.  Everything srcnn_upscale_yuv420_frames_host rejects, and a siting outside
 * SRCNN_CHROMA_*: SRCNN_EINVAL before any host buffer is read or written. */
int srcnn_upscale_yuv420_frames_host_sited(srcnn_ctx* ctx, const srcnn_net* net,
                                           const unsigned char* host_in, int w, int h, int n_frames,
                                           int out_w, int out_h, int filter, int in_siting,
                                           int out_siting, unsigned char* host_out);

/* Where the planes of 4:2:0 frames lie in a device buffer.  A frame's Y plane starts at the frame's
 * first byte; every offset, pitch and stride is in bytes.  SRCNN_YUV_I420: Y, Cb and Cr planes
 * (`yuv420p`); SRCNN_YUV_NV12: Y, then one plane of interleaved Cb, Cr pairs, Cb first (what
 * hardware video decoders hand out and encoders take).  The dense I420 layout of
 * srcnn_upscale_yuv420_frames_host is {I420, w*h*3/2, w, w/2, w*h, w*h*5/4, 0}, the dense NV12 one
 * {NV12, w*h*3/2, w, w, w*h, 0, 0}.
 * chroma_siting was appended as the last field so that the fields before it keep their offsets
 * and a zero-initialised layout keeps its meaning (centre-sited chroma); a caller that declares
 * the struct itself (a language binding) adds the field too.
 * bit_depth was appended after it for the same reason: 0 or 8 is 8-bit samples, one byte each;
 * 10 is 10-bit samples v in [0, 1023], one little-endian 16-bit word each, and then
 * SRCNN_YUV_I420 means I010 (`yuv420p10le`, the frames of a C420p10 Y4M file: v in the low 10
 * bits) and SRCNN_YUV_NV12 means P010 (what hardware decoders hand out for 10-bit streams: v in the
 * high 10 bits, word = v << 6).  The other 6 bits of an input word never affect a result and are
 * written as 0.  A 10-bit row is twice the bytes of an 8-bit one: the dense I010 layout is {I420,
 * w*h*3, 2*w, w, 2*w*h, 2*w*h*5/4, 0, 10}, the dense P010 one {NV12, w*h*3, 2*w, 2*w, 2*w*h, 0, 0,
 * 10}. */
enum { SRCNN_YUV_I420 = 0, SRCNN_YUV_NV12 = 1 };
typedef struct srcnn_yuv420_layout {
  int format;           /* SRCNN_YUV_I420 or SRCNN_YUV_NV12 */
  size_t frame_stride;  /* from one frame's start to the next's */
  size_t y_pitch;       /* from one Y row to the next, >= width */
  size_t c_pitch;       /* from one chroma row to the next, >= width/2 (I420) or width (NV12) */
  size_t cb_offset;     /* of the Cb plane (NV12: the CbCr plane) from the frame start */
  size_t cr_offset;     /* I420: of the Cr plane; NV12: must be 0 */
  int chroma_siting;    /* SRCNN_CHROMA_*: where the frames' chroma samples sit; 0 = centre */
  int bit_depth;        /* 0 or 8: 8-bit samples; 10: 10-bit samples in 16-bit words (I010, P010) */
} srcnn_yuv420_layout;

/* srcnn_upscale_yuv420_frames_host on frames that are already in device memory, in I420 or NV12
 * with pitched rows: `in` holds n_frames frames of w x h in in_layout, `out` receives n_frames
 * frames of out_w x out_h in out_layout, of the same format.  The Y, Cb and Cr bytes of a frame are
 * those srcnn_upscale_yuv420_frames_host_sited writes for it with in_layout's chroma_siting as the
 * input's and out_layout's as the output's (NV12: the same Cb and Cr bytes, interleaved).  With
 * bit_depth 10 in both layouts the frames are I010 or P010, and a frame's samples are those
 * srcnn_upscale_yuv420p10_frames_host writes for it (P010: the same Cb and Cr, interleaved, each
 * value at bit 6 of its word); the groups, scratch and launches are those of 8-bit frames.  Bytes of `out` outside the planes' rows (pitch padding, gaps between planes or
 * frames) are never written; bytes of `in` outside them never affect the result.
 * Stream-ordered, like srcnn_forward_fused: the work is enqueued on the context stream and the
 * call returns, without a copy or a host synchronisation (the caller orders its own work on that
 * stream: create the context with srcnn_ctx_create_on_stream on a non-default stream, e.g. a
 * torch.cuda.Stream(), and fill `in` and read `out` on it).  Once a call with the same sizes,
 * layouts' formats, pair of chroma sitings and network has run, a call allocates nothing, so it can
 * be captured into a CUDA graph on the context stream.  (A new siting pair is a new chroma table,
 * allocated and uploaded on its first call: capture only a call whose pair has run before.)  Such a graph reads the entry's scratch, which grows on
 * demand: a later call on the context that needs more of it (larger frames, or more frames a
 * group) reallocates it, and the graph must then be captured again.  It waits for
 * srcnn_infer_rows_host_async calls in flight first; in profile mode every launch blocks.  Staging
 * is the context's and apart from the other entries'.
 * Networks with a fused kernel run groups of frames, one launch per step with every frame of the
 * group in the grid: the enlargement of the planes straight into `out` + the luma of Y, the Q1 sum
 * (2), minus the mean, the fused forward, the Y write.  A group holds as many frames as fit
 * ~128 MB of device scratch (out_w*out_h*4 + h3*w3*4 bytes and the Q1 partials a frame: 8 frames
 * of 1920x1080 with a 9-1-5 network), or SRCNN_FRAMES_GROUP frames when that is set (at most
 * 21845 for I420, 65535 for NV12).  Networks without a fused kernel run frame by frame, for the
 * reason srcnn_upscale_frames_host gives.
 * Launches per call: n_groups * (5 + F) for I420 and n_groups * (6 + F) for NV12 (whose Y plane and
 * CbCr plane are one enlargement launch each) with a fused kernel, n_frames * (4 + L + 1) without
 * (plus n_frames for NV12), plus 1 when the network's packed operand image has to be rebuilt (F, L
 * as for srcnn_upscale_frames_host).
 * Errors, all before any launch (the output and the launch count stay untouched):
 *   SRCNN_EINVAL: everything srcnn_upscale_yuv420_frames_host rejects; a null layout; an unknown
 *     format, or formats that differ; a chroma_siting outside SRCNN_CHROMA_* in either layout; a
 *     bit_depth other than 0, 8 or 10, or input and output bit depths that differ; 10-bit with an
 *     odd pitch, offset, buffer start or (n_frames > 1) frame_stride, or P010 with a CbCr plane
 *     or c_pitch that is not a multiple of 4 bytes in any frame; a pitch below its row's bytes
 *     (10-bit: 2*w for Y and P010 CbCr, w for I010 chroma); a pitch, offset or stride of
 *     2^31 bytes or more; planes of one frame whose byte ranges intersect; with n_frames > 1, a
 *     frame_stride below the frame's extent (the end of its last plane's last row); NV12 with
 *     cr_offset != 0, an odd c_pitch, or a CbCr plane at an odd address in any frame; input and
 *     output byte ranges that overlap.
 *   SRCNN_EHANDLE / SRCNN_ERANGE: an unknown buffer, or one smaller than
 *     (n_frames - 1) * frame_stride + the frame's extent. */
int srcnn_upscale_yuv420_frames(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in,
                                const srcnn_yuv420_layout* in_layout, int w, int h, int n_frames,
                                srcnn_mem out, const srcnn_yuv420_layout* out_layout, int out_w,
                                int out_h, int filter);

/* srcnn_upscale_yuv420_frames_host_sited for 10-bit frames: host_in holds n_frames dense I010
 * frames of w x h (Y, then Cb, then Cr, one little-endian 16-bit word a sample with the value v in
 * its low 10 bits: w*h*3 bytes a frame, the frames of a C420p10 Y4M file), host_out receives
 * n_frames frames of out_w*out_h*3 bytes.  The bits above the low 10 of an input word never
 * affect a result; every output word is v in [0, 1023], its upper bits 0.  Per frame:
 *   - every plane is enlarged with Pillow's 16-bit path (Image.fromarray(plane, "I;16").resize):
 *     the coefficients of the 8-bit path kept as normalised doubles (not rounded to 22 bits), each
 *     output the sum of v * k in double in tap order, rounded half away from zero and clipped to
 *     [0, 65535]; the horizontal pass first into a 16-bit intermediate, an axis copied when its
 *     size does not change and its box starts at 0.0.  The final samples are capped at 1023.  The
 *     chroma planes take the box starts of the sitings as in the 8-bit entry.
 *   - the luma v / 1023 of the enlarged Y, minus the Q1 mean, goes through the three layers;
 *     inside the network's output region the Y sample is clamp(luma * 1023, 0, 1023) truncated,
 *     and the border keeps the enlarged Y.
 * A frame's words do not depend on the other frames of the call or on the group size.  The ring,
 * groups and launches are those of srcnn_upscale_yuv420_frames_host with every frame twice the
 * bytes (3 frames a group for 960x540 -> 1920x1080 with a 9-1-5 network).  Everything
 * srcnn_upscale_yuv420_frames_host_sited rejects: SRCNN_EINVAL before any host buffer is read or
 * written. */
int srcnn_upscale_yuv420p10_frames_host(srcnn_ctx* ctx, const srcnn_net* net,
                                        const uint16_t* host_in, int w, int h, int n_frames,
                                        int out_w, int out_h, int filter, int in_siting,
                                        int out_siting, uint16_t* host_out);

/* srcnn_upscale_frames_host plus the quality of its results: host_ref holds n_frames reference
 * frames of out_w*out_h*4 bytes RGBA8 (the ground truth the small frames were made from).
 * host_rgb receives what srcnn_upscale_frames_host returns for the same arguments, byte for byte;
 * host_metrics receives 4 doubles a frame: {mse, ssim} of the network's result and {mse, ssim}
 * of the plain enlargement (the resampled RGBA8 alone, the baseline the network starts from),
 * both against the reference as srcnn_image_quality measures them, over the region border from
 * each edge (border < 0: (f1+f2+f3-3)/2, the rows and columns swap_luma leaves as enlarged).
 * Synchronous; pinned host buffers give the overlap.  The reference frames go up on the copy-in
 * stream into ring slots of their own; the metrics of all frames stay on the device and come
 * down once, after the last group.  Staging is the context's and apart from the frames entry's.
 * Groups hold as many frames as fit ~128 MB (the frames entry's bytes + out_w*out_h*4 a frame),
 * or SRCNN_FRAMES_GROUP frames.
 * Launches per call: n_groups * (5 + F + 4) with a fused kernel, n_frames * (4 + L + 1 + 4)
 * without (F, L as for srcnn_upscale_frames_host), plus 1 when the network's packed operand image
 * has to be rebuilt.  Everything srcnn_upscale_frames_host rejects, a null host_ref or
 * host_metrics and a border that leaves less than 11x11 pixels: SRCNN_EINVAL before any host
 * buffer is read or written. */
int srcnn_evaluate_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const unsigned char* host_rgba,
                               int w, int h, int n_frames, int out_w, int out_h, int filter,
                               const unsigned char* host_ref, int border, unsigned char* host_rgb,
                               double* host_metrics);

/* ConfigBasedDataPipeline::forward(sample) for MANY frames (src/ConfigBasedDataPipeline.cpp:
 * 114-126 is called once per image by src/Main_cl.cpp:217-239): `n_frames` luma frames of
 * w x h floats in host memory -> n_frames results of w3 x h3 floats in host_out.  Groups of
 * frames go through a ring of device slots so that the upload of the next group and the download
 * of the previous one overlap the fused forward of the current one.  Synchronous.  Frames are
 * independent: a multi-GPU caller gives each rank its own slice of the frame set (SURVEY 8e,
 * BASELINE config C5). */
int srcnn_infer_frames_host(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in, int w,
                            int h, int n_frames, float* host_out);

/* One training chunk on device-resident samples: forward (keeping out1/out2), last-layer
 * delta, deltas 2<-3 and 1<-2, the three weight/bias gradients accumulated into
 * net->grad_*  (= ConfigBasedDataPipeline::forward + ::backpropagate,
 * src/ConfigBasedDataPipeline.cpp:165-176,243-323).  `work` holds the activations and deltas
 * of the chunk; size it with srcnn_train_workspace_bytes(). */
int srcnn_train_chunk(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt,
                      int w, int h, int S, srcnn_mem work);
size_t srcnn_train_workspace_bytes(const srcnn_net* net, int w, int h, int S);
/* The layer-1 deltas are an intermediate of the layer-1 gradients only
 * (ConfigBasedDataPipeline.cpp:265-270 -> 300-320).  For f2 = 1, n1 = 64, n2 = 32 networks the
 * training-chunk entries compute them inside the layer-1 gradient kernel and leave the d1
 * buffer untouched; returns 1 when the chunk entries write d1 for this network on this
 * context, 0 when they do not (SRCNN_D1_IMPL=separate in the environment restores the
 * separate launch; srcnn_deltas itself always materialises its target). */
int srcnn_train_materializes_d1(srcnn_ctx* ctx, const srcnn_net* net);

/* Same chunk, with the six activation / delta buffers owned by the caller -- the buffers
 * ConfigBasedDataPipeline allocates itself (_out_1.._out_3, _delta_1.._delta_3,
 * src/ConfigBasedDataPipeline.cpp:82-108), so that its forward() + backpropagate() pair for a
 * training chunk is one call.  Every buffer must start 16-byte aligned. */
int srcnn_train_chunk_buffers(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt,
                              int w, int h, int S, srcnn_mem out1, srcnn_mem out2,
                              srcnn_mem out3, srcnn_mem d1, srcnn_mem d2, srcnn_mem d3);

/* ConfigBasedDataPipeline::execute_batch(backpropagate = true, ...)
 * (src/ConfigBasedDataPipeline.cpp:128-195) on HOST-resident samples: `n_samples` inputs and
 * ground truths of w x h floats each are cut into chunks of at most `chunk` samples; the upload
 * of chunk i+1 (copy stream, double-buffered staging owned by the context) overlaps the
 * forward + backward of chunk i (srcnn_train_chunk); the first chunk, whose upload nothing can
 * hide, is half a chunk when there is more than one chunk of samples.  Gradients accumulate in net->grad_*;
 * the caller all-reduces them (multi-GPU) and calls srcnn_update_all.  `work` must hold
 * srcnn_train_workspace_bytes(net, w, h, chunk).  Returns once the host buffers may be reused;
 * the last chunk may still be training on the context stream. */
int srcnn_train_chunks_host(srcnn_ctx* ctx, const srcnn_net* net, const float* host_in,
                            const float* host_gt, int w, int h, int n_samples, int chunk,
                            srcnn_mem work);

/* ConfigBasedDataPipeline::update_parameters (src/ConfigBasedDataPipeline.cpp:325-361) in
 * ONE launch: the three layers with lr[0..2], then the six accumulators are zeroed. */
int srcnn_update_all(srcnn_ctx* ctx, const srcnn_net* net, unsigned batch_size, float momentum,
                     float weight_decay, const float lr[3]);

/* Validation pass of execute_batch (src/ConfigBasedDataPipeline.cpp:177-187): forward +
 * squared error of S device-resident samples; the SSE lands in the 1-float `target`. */
int srcnn_validate_chunk(srcnn_ctx* ctx, const srcnn_net* net, srcnn_mem in, srcnn_mem gt,
                         int w, int h, int S, srcnn_mem work, srcnn_mem target);

/* The fused kernels cache a packed copy of a network's parameters per context while the six
 * parameter buffers are context-owned, were never handed out by srcnn_mem_ptr, and no call of
 * this layer has written them.  A buffer whose raw pointer was obtained with srcnn_mem_ptr is
 * never cached (anything may write through it).  Call this after writing parameters by any
 * other route (a kernel of your own on the context stream, a peer copy ...). */
int srcnn_invalidate_params(srcnn_ctx* ctx);

/* ---------------------------------------------------------------- multi-GPU -------- */
/* New (the reference is single-device: src/opencl/Context.cpp:52-60).  One context per GPU /
 * process; the communicator enqueues on the context stream, so collectives order with the
 * launches around them.  NCCL (libnccl.so.2) is loaded on first use.  Partitioning (SURVEY 8e):
 * inference = row bands, no collective; training = patches split across ranks, replicated
 * parameters, ONE sum all-reduce of the gradient accumulators before each
 * srcnn_update_all(batch_size = GLOBAL sample count); validation = 1-float all-reduce of the
 * squared error (src/ConfigBasedDataPipeline.cpp:177-187, src/Main_cl.cpp:174-192). */
#define SRCNN_COMM_ID_BYTES 128
/* rank 0 creates the id and hands it to the other ranks (file, pipe, launcher ...) */
int srcnn_comm_unique_id(unsigned char id[SRCNN_COMM_ID_BYTES]);
/* collective over all ranks: joins this context to the communicator */
int srcnn_comm_init(srcnn_ctx* ctx, int rank, int world,
                    const unsigned char id[SRCNN_COMM_ID_BYTES]);
int srcnn_comm_destroy(srcnn_ctx* ctx);
/* rank / world of the context (0 / 1 without a communicator) */
int srcnn_comm_info(srcnn_ctx* ctx, int* rank, int* world);
/* in-place sum over ranks of `count` floats at buf[offset_floats..]; no-op on one rank */
int srcnn_allreduce_sum(srcnn_ctx* ctx, srcnn_mem buf, size_t offset_floats, size_t count);
/* in-place sum over ranks of the six gradient accumulators of `net`: one all-reduce when they
 * are consecutive views of one flat buffer, a grouped call otherwise */
int srcnn_allreduce_grads(srcnn_ctx* ctx, const srcnn_net* net);
/* the first `count` floats of `buf` on rank `root` replace everybody's (parameter sync) */
int srcnn_broadcast(srcnn_ctx* ctx, srcnn_mem buf, size_t count, int root);

#ifdef __cplusplus
}
#endif
#endif /* SRCNN_B200_H */
