// The SRCNN model: three LayerData, the batch / activation / delta buffers, forward,
// execute_batch, backpropagate, update_parameters, parameter file I/O, result image.
// Same public surface as the reference's cnn_sr::ConfigBasedDataPipeline
// (src/ConfigBasedDataPipeline.hpp:45-156).
#ifndef CNN_SR_CONFIG_BASED_DATA_PIPELINE_H
#define CNN_SR_CONFIG_BASED_DATA_PIPELINE_H

#include "Config.hpp"
#include "DataPipeline.hpp"
#include "LayerData.hpp"

namespace cnn_sr {

/** device buffers of one image / training sample (src/ConfigBasedDataPipeline.hpp:12-31) */
struct SampleAllocationPool {
  opencl::MemoryHandle input_data = gpu_nullptr;   // RGBA image
  opencl::MemoryHandle input_luma = gpu_nullptr;   // input_w * input_h floats
  size_t input_w = 0, input_h = 0;
  opencl::MemoryHandle expected_data = gpu_nullptr;  // training: RGBA ground truth
  opencl::MemoryHandle expected_luma = gpu_nullptr;  // training: luma to compare with
};

struct GpuAllocationPool {
  LayerAllocationPool layer_1, layer_2, layer_3;
  std::vector<SampleAllocationPool> samples;
};

class ConfigBasedDataPipeline : public DataPipeline {
 public:
  ConfigBasedDataPipeline(Config&, opencl::Context*);

  /** loads kernels, then parameters: from config.parameters_file when set, else random */
  void init(int load_flags);
  void set_mini_batch_size(size_t);

  /** Processes the sample set in chunks of mini_batch_size: forward, then either
   * backpropagation (gradients ACCUMULATE until update_parameters) or the squared error.
   * Returns the summed squared error (0 when backpropagating). */
  float execute_batch(bool backpropagate, GpuAllocationPool&, std::vector<SampleAllocationPool*>&);

  /** inference of one image; the result stays in the layer-3 output buffer */
  cl_event forward(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                   SampleAllocationPool& sample);

  /** momentum + weight-decay step of all three layers with batch_size, then zeroes the six
   * gradient accumulators and counts one epoch */
  void update_parameters(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                         size_t batch_size, cl_event* ev_to_wait_for = nullptr);

  void write_params_to_file(const char* const file_path, LayerAllocationPool, LayerAllocationPool,
                            LayerAllocationPool);
  void write_result_image(const char* const, opencl::utils::ImageData&, SampleAllocationPool&);

  /** the forward mode for an image that must first be enlarged: `in` (RGBA8) is enlarged to
   * out_w x out_h with `filter` (SRCNN_RESAMPLE_*), its luma goes through the three layers and is
   * swapped back; `out` receives the RGB8 result (out_w * out_h * 3 bytes, owned by the caller) */
  void upscale_image(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                     opencl::utils::ImageData& in, size_t out_w, size_t out_h, int filter,
                     opencl::utils::ImageData& out);
  /** upscale_image for n_frames frames of w x h RGBA8, back to back in `in_rgba`; `out_rgb`
   * receives n_frames results of out_w * out_h * 3 bytes (srcnn_upscale_frames_host) */
  void upscale_frames(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                      const unsigned char* in_rgba, size_t w, size_t h, size_t n_frames,
                      size_t out_w, size_t out_h, int filter, unsigned char* out_rgb);
  /** upscale_frames for n_frames planar Y'CbCr 4:2:0 (I420) frames of w x h, back to back in
   * `in_yuv`; `out_yuv` receives n_frames I420 frames of out_w x out_h: Y enlarged and its
   * interior replaced by the network's luma, Cb and Cr enlarged from chroma sited at in_siting to
   * chroma sited at out_siting (SRCNN_CHROMA_*; srcnn_upscale_yuv420_frames_host_sited) */
  void upscale_yuv420_frames(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                             const unsigned char* in_yuv, size_t w, size_t h, size_t n_frames,
                             size_t out_w, size_t out_h, int filter, unsigned char* out_yuv,
                             int in_siting = SRCNN_CHROMA_CENTER,
                             int out_siting = SRCNN_CHROMA_CENTER);
  /** upscale_yuv420_frames for 10-bit I010 frames (a little-endian 16-bit word a sample, the
   * value in its low 10 bits): `out_yuv` receives n_frames I010 frames of out_w x out_h
   * (srcnn_upscale_yuv420p10_frames_host) */
  void upscale_yuv420p10_frames(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                                const uint16_t* in_yuv, size_t w, size_t h, size_t n_frames,
                                size_t out_w, size_t out_h, int filter, uint16_t* out_yuv,
                                int in_siting = SRCNN_CHROMA_CENTER,
                                int out_siting = SRCNN_CHROMA_CENTER);
  /** upscale_frames plus the quality of every result against its reference (n_frames frames of
   * out_w x out_h RGBA8 in `ref_rgba`): `metrics` receives 4 doubles a frame, {mse, ssim} of the
   * network's result and of the plain enlargement, over the region `border` pixels in from each
   * edge (< 0: half the network's padding) (srcnn_evaluate_frames_host) */
  void evaluate_frames(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                       const unsigned char* in_rgba, size_t w, size_t h, size_t n_frames,
                       size_t out_w, size_t out_h, int filter, const unsigned char* ref_rgba,
                       int border, unsigned char* out_rgb, double* metrics);

  inline const Config* config() { return _config; }
  inline const LayerData* layer_1() { return &layer_data_1; }
  inline const LayerData* layer_2() { return &layer_data_2; }
  inline const LayerData* layer_3() { return &layer_data_3; }
  /** layer-3 output of the last forward pass (device) */
  inline opencl::MemoryHandle result_buffer() const { return _out_3_gpu_buf; }

 protected:
  void load_kernels(int load_flags);

 private:
  void allocate_buffers(size_t w, size_t h, bool training);
  cl_event forward(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&, size_t w,
                   size_t h, size_t sample_count);
  cl_event backpropagate(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                         size_t w, size_t h, size_t sample_count, cl_event* ev = nullptr);
  void ensure_parameters_on_device(LayerData&, LayerAllocationPool&);
  void ensure_gradients_on_device(LayerData&, LayerAllocationPool&);
  /** forward() + backpropagate() of one training chunk in one device-layer call */
  void train_chunk(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&, size_t w,
                   size_t h, size_t sample_count);
  /** the three layers' device buffers as the C-ABI's srcnn_net */
  srcnn_net device_net(LayerAllocationPool&, LayerAllocationPool&, LayerAllocationPool&,
                       bool with_gradients, bool with_momentum);
  void ensure_momentum_on_device(int layer, LayerData&, LayerAllocationPool&);
  void fill_random_parameters(LayerData&, ParametersDistribution&);
  size_t load_parameters_file(const char* const);

  /** momentum state read from the optional "resume" key of a parameters file (uploaded when the
   * previous_batch_delta buffers are first needed) */
  std::vector<float> _resume_prev_w[3], _resume_prev_b[3];
  std::vector<opencl::MemoryHandle> _gather_in, _gather_gt;
  Config* const _config;
  LayerData layer_data_1, layer_data_2, layer_data_3;
  size_t epochs = 0;
  size_t _mini_batch_size = 0;
  size_t _alloc_w = 0, _alloc_h = 0, _alloc_batch = 0;
  bool _alloc_training = false;

  opencl::MemoryHandle _ground_truth_gpu_buf = gpu_nullptr;
  opencl::MemoryHandle _forward_gpu_buf = gpu_nullptr;
  opencl::MemoryHandle _out_1_gpu_buf = gpu_nullptr, _out_2_gpu_buf = gpu_nullptr,
                       _out_3_gpu_buf = gpu_nullptr;
  opencl::MemoryHandle _delta_1_gpu_buf = gpu_nullptr, _delta_2_gpu_buf = gpu_nullptr,
                       _delta_3_gpu_buf = gpu_nullptr;

  opencl::Kernel* _layer_1_kernel = nullptr;
  opencl::Kernel* _layer_2_kernel = nullptr;
  opencl::Kernel* _layer_3_kernel = nullptr;
  opencl::Kernel* _layer_1_deltas_kernel = nullptr;
  opencl::Kernel* _layer_2_deltas_kernel = nullptr;
};

}  // namespace cnn_sr
#endif
