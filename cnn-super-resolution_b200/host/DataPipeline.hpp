// Per-kernel host wrappers: validate sizes, lazily allocate, launch.  Same public methods,
// argument meaning and error behaviour as the reference's cnn_sr::DataPipeline
// (src/DataPipeline.hpp:39-222); the bodies call the CUDA C-ABI instead of pushing OpenCL
// kernel arguments.
#ifndef CNN_SR_DATA_PIPELINE_H
#define CNN_SR_DATA_PIPELINE_H

#include "Context.hpp"
#include "LayerData.hpp"
#include "pch.hpp"

/** "no allocation yet": wrappers allocate lazily when they see it (src/DataPipeline.hpp:7) */
const opencl::MemoryHandle gpu_nullptr = 1 << 30;

namespace cnn_sr {

/** device buffers of one layer (reference: src/DataPipeline.hpp:11-29) */
struct LayerAllocationPool {
  opencl::MemoryHandle weights = gpu_nullptr;                 // f*f*k*n
  opencl::MemoryHandle bias = gpu_nullptr;                    // n
  opencl::MemoryHandle accumulating_grad_w = gpu_nullptr;     // summed over the whole epoch
  opencl::MemoryHandle accumulating_grad_b = gpu_nullptr;
  opencl::MemoryHandle previous_batch_delta_w = gpu_nullptr;  // momentum state
  opencl::MemoryHandle previous_batch_delta_b = gpu_nullptr;
};

class DataPipeline {
 public:
  static int LOAD_KERNEL_LUMA;
  static int LOAD_KERNEL_LAYERS;
  static int LOAD_KERNEL_BACKPROPAGATE;
  static int LOAD_KERNEL_MISC;
  static int LOAD_KERNEL_NONE;
  static int LOAD_KERNEL_ALL;

  DataPipeline(opencl::Context*);
  virtual ~DataPipeline() {}
  virtual void init(int load_flags = DataPipeline::LOAD_KERNEL_ALL);
  opencl::Context* context();

  /** uploads the RGBA image and writes its luma (optionally /255) to gpu_buf_luma */
  cl_event extract_luma(opencl::utils::ImageData&, opencl::MemoryHandle& gpu_buf_raw_img,
                        opencl::MemoryHandle& gpu_buf_luma, bool normalize,
                        cl_event* ev = nullptr);

  /** uploads the RGBA image and enlarges it to out_w x out_h (Pillow-exact, `filter` =
   * SRCNN_RESAMPLE_*) into the RGBA8 gpu_buf_out, with its normalized luma in gpu_buf_luma */
  cl_event resample(opencl::utils::ImageData&, opencl::MemoryHandle& gpu_buf_raw_img,
                    size_t out_w, size_t out_h, int filter, opencl::MemoryHandle& gpu_buf_out,
                    opencl::MemoryHandle& gpu_buf_luma);

  /** new luma (x255) + chroma of the original image -> RGB8 in `target` */
  cl_event swap_luma(opencl::utils::ImageData&, opencl::MemoryHandle& gpu_buf_org_img,
                     opencl::MemoryHandle gpu_buf_new_luma, opencl::MemoryHandle& target,
                     size_t new_luma_w, size_t new_luma_h, cl_event* ev = nullptr);

  /** forward propagation of one layer for `sample_count` images of input_w x input_h */
  cl_event execute_layer(opencl::Kernel&, const LayerData&, cnn_sr::LayerAllocationPool&,
                         opencl::MemoryHandle& gpu_buf_in, size_t input_w, size_t input_h,
                         size_t sample_count, opencl::MemoryHandle& gpu_buf_out,
                         cl_event* ev = nullptr);

  /** sum of squared differences to the centre crop of the ground truth; the result arrives in
   * `target` once the returned event has been waited for */
  cl_event squared_error(opencl::MemoryHandle gpu_buf_ground_truth, size_t ground_truth_w,
                         size_t ground_truth_h, size_t sample_count,
                         opencl::MemoryHandle gpu_buf_algo_res, opencl::MemoryHandle tmp_buffer,
                         float& target, size_t total_padding, cl_event* ev = nullptr);

  cl_event last_layer_delta(opencl::MemoryHandle gpu_buf_ground_truth, size_t ground_truth_w,
                            size_t ground_truth_h, size_t sample_count,
                            opencl::MemoryHandle gpu_buf_algo_res,
                            opencl::MemoryHandle& gpu_buf_target, size_t total_padding,
                            cl_event* ev = nullptr);

  /** deltas of `curr_layer` from the deltas of `next_layer` */
  cl_event calculate_deltas(opencl::Kernel&, const LayerData& curr_layer,
                            const LayerData& next_layer, cnn_sr::LayerAllocationPool& next_alloc,
                            opencl::MemoryHandle curr_deltas, opencl::MemoryHandle next_deltas,
                            size_t next_layer_out_w, size_t next_layer_out_h, size_t sample_count,
                            opencl::MemoryHandle curr_output, cl_event* ev = nullptr);

  /** weight / bias gradients, accumulated into the pool's accumulating_grad_* */
  cl_event backpropagate(LayerData&, opencl::MemoryHandle layer_input,
                         opencl::MemoryHandle layer_deltas, LayerAllocationPool&,
                         size_t layer_out_w, size_t layer_out_h, size_t sample_count,
                         cl_event* ev = nullptr, size_t ev_cnt = 0);

  cl_event update_parameters(LayerData&, LayerAllocationPool&, size_t batch_size, float momentum,
                             float w_decay, float learning_rate, cl_event* ev = nullptr);

  /** NOTE quirk Q1: passes `ev` to sum()'s `squared` parameter exactly like the reference
   * (src/DataPipeline.cpp:274), so a non-null event subtracts the mean of SQUARES */
  cl_event subtract_mean(opencl::MemoryHandle, float* mean = nullptr, cl_event* ev = nullptr);
  float sum(opencl::MemoryHandle, bool squared = false, cl_event* ev = nullptr);
  cl_event subtract_from_all(opencl::MemoryHandle, float, cl_event* ev = nullptr);

  opencl::Kernel* create_layer_kernel(const LayerData&, bool skip_relu);
  opencl::Kernel* create_deltas_kernel(const LayerData&);

  void print_buffer(opencl::MemoryHandle, const char* const name, size_t lines);

 protected:
  void check_initialized(int kernel_load_flags);
  virtual void load_kernels(int load_flags);
  /** true: allocation exists and is big enough; false: gpu_nullptr; throws when it exists but
   * is too small (src/DataPipeline.cpp:66-86) */
  bool allocation_has_right_size__(opencl::MemoryHandle, size_t bytes, size_t line,
                                   const char* variable_name);

 private:
  void pre_execute_layer_validation(const LayerData&, opencl::MemoryHandle, size_t, size_t);
  size_t element_count(opencl::MemoryHandle, size_t el_size);

 protected:
  opencl::Context* const _context;
  bool _initialized;
  opencl::MemoryHandle _tmp_gpu_float = gpu_nullptr;

  opencl::Kernel* _luma_kernel_norm = nullptr;
  opencl::Kernel* _luma_kernel_raw = nullptr;
  opencl::Kernel* _swap_luma_kernel = nullptr;
  opencl::Kernel* _resample_kernel = nullptr;   // see resample_kernel()
  opencl::Kernel* resample_kernel();
  opencl::Kernel* _squared_error_kernel = nullptr;
  opencl::Kernel* _sum_kernel = nullptr;
  opencl::Kernel* _sum_squared_kernel = nullptr;
  opencl::Kernel* _subtract_from_all_kernel = nullptr;
  opencl::Kernel* _last_layer_delta_kernel = nullptr;
  opencl::Kernel* _update_parameters_kernel = nullptr;
  opencl::Kernel* _backpropagate_kernel = nullptr;
};

}  // namespace cnn_sr
#endif
