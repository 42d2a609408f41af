#include "DataPipeline.hpp"

#include <sstream>
#include <stdexcept>

using opencl::MemoryHandle;
using opencl::ProfiledLaunch;

namespace {
// logical kernel "files": kept so that `profile` output (and profile.py) reads like the
// reference's (src/DataPipeline.cpp:12-25)
const std::string kernel_folder = "src/kernel/";
const char* const luma_kernel_file = "extract_luma.cl";
const char* const swap_luma_kernel_file = "swap_luma.cl";
const char* const resample_kernel_file = "resample.cu";   // (new: no reference kernel)
const char* const squared_error_kernel_file = "squared_error.cl";
const char* const sum_kernel_file = "sum.cl";
const char* const layer_kernel_file = "layer_uber_kernel.cl";
const char* const deltas_kernel_file = "layer_deltas.cl";
const char* const last_layer_delta_kernel_file = "last_layer_delta.cl";
const char* const backpropagate_kernel_file = "backpropagate.cl";
const char* const subtract_from_all_kernel_file = "subtract_from_all.cl";
const char* const update_parameters_kernel_file = "update_parameters.cl";
}  // namespace

namespace cnn_sr {

int DataPipeline::LOAD_KERNEL_LUMA = 1;
int DataPipeline::LOAD_KERNEL_LAYERS = 2;
int DataPipeline::LOAD_KERNEL_MISC = 4;
int DataPipeline::LOAD_KERNEL_BACKPROPAGATE = 8;
int DataPipeline::LOAD_KERNEL_NONE = 0;
int DataPipeline::LOAD_KERNEL_ALL = 1 | 2 | 4 | 8;

#define ALLOCATION_HAS_RIGHT_SIZE(VAR, BYTES) \
  (this->allocation_has_right_size__(VAR, BYTES, __LINE__, STRINGIFY(VAR)))

DataPipeline::DataPipeline(opencl::Context* context) : _context(context), _initialized(false) {}

void DataPipeline::init(int load_flags) {
  load_kernels(load_flags);
  _initialized = true;
}

void DataPipeline::check_initialized(int kernel_load_flags) {
  if (!_initialized) throw std::runtime_error("Tried to use DataPipeline before it was initialized");
  this->load_kernels(kernel_load_flags);
}

opencl::Context* DataPipeline::context() { return _context; }

bool DataPipeline::allocation_has_right_size__(MemoryHandle alloc, size_t size, size_t line,
                                               const char* variable_name) {
  if (alloc == gpu_nullptr) return false;
  const size_t have = _context->raw_memory(alloc)->size;
  if (have >= size) return true;
  std::cout << "Was forced to realocate gpu buffer. This is not optimal and may be a bug. In "
               "many cases DataPipeline is able to allocate buffer of right size, so You only "
               "need to explictly set MemoryHandle to gpu_nullptr. Expected: "
            << size << ", got: " << have << ". Code line: " << line << ", variable: '"
            << variable_name << "'" << std::endl;
  throw std::runtime_error("Was forced to realocate gpu buffer due too difference in sizes.");
}

size_t DataPipeline::element_count(MemoryHandle alloc, size_t el_size) {
  return _context->raw_memory(alloc)->size / el_size;
}

void DataPipeline::print_buffer(MemoryHandle mh, const char* const name, size_t lines) {
  const size_t len = _context->raw_memory(mh)->size / sizeof(float);
  std::vector<float> data(len);
  _context->block();
  _context->read_buffer(mh, data.data(), true);
  std::cout << name << ": [" << std::endl;
  utils::dump_vector(std::cout, data, "", lines ? len / lines : 0, true);
  std::cout << "]" << std::endl << std::endl << std::endl;
}

// ------------------------------------------------------------------ kernel objects -----
void DataPipeline::load_kernels(int load_flags) {
  auto make = [&](const char* file, const char* opts, const char* entry) {
    return _context->create_kernel((kernel_folder + file).c_str(), opts, entry);
  };
  if (load_flags & LOAD_KERNEL_LUMA) {
    if (!_luma_kernel_norm) _luma_kernel_norm = make(luma_kernel_file, "-D NORMALIZE", "extract_luma");
    if (!_luma_kernel_raw) _luma_kernel_raw = make(luma_kernel_file, nullptr, "extract_luma");
    if (!_swap_luma_kernel) _swap_luma_kernel = make(swap_luma_kernel_file, nullptr, "swap_luma");
  }
  if (load_flags & LOAD_KERNEL_MISC) {
    if (!_squared_error_kernel) _squared_error_kernel = make(squared_error_kernel_file, nullptr, "squared_err");
    if (!_sum_kernel) _sum_kernel = make(sum_kernel_file, nullptr, "sum");
    if (!_sum_squared_kernel) _sum_squared_kernel = make(sum_kernel_file, "-D SUM_SQUARED", "sum");
    if (!_subtract_from_all_kernel) _subtract_from_all_kernel = make(subtract_from_all_kernel_file, nullptr, "sub_from_all");
  }
  if (load_flags & LOAD_KERNEL_BACKPROPAGATE) {
    if (!_last_layer_delta_kernel) _last_layer_delta_kernel = make(last_layer_delta_kernel_file, nullptr, "last_layer_delta");
    if (!_update_parameters_kernel) _update_parameters_kernel = make(update_parameters_kernel_file, nullptr, "update_params");
    if (!_backpropagate_kernel) _backpropagate_kernel = make(backpropagate_kernel_file, nullptr, "backpropagate");
  }
}

opencl::Kernel* DataPipeline::create_layer_kernel(const LayerData& d, bool skip_relu) {
  std::ostringstream opts;
  opts << "-D CURRENT_FILTER_COUNT=" << d.current_filter_count
       << " -D PREVIOUS_FILTER_COUNT=" << d.n_prev_filter_cnt
       << " -D F_SPATIAL_SIZE=" << d.f_spatial_size;
  if (skip_relu) opts << " -D SKIP_RELU";
  return _context->create_kernel((kernel_folder + layer_kernel_file).c_str(), opts.str().c_str(),
                                 "forward");
}

opencl::Kernel* DataPipeline::create_deltas_kernel(const LayerData& d) {
  std::ostringstream opts;
  opts << "-D CURRENT_FILTER_COUNT=" << d.current_filter_count;
  return _context->create_kernel((kernel_folder + deltas_kernel_file).c_str(),
                                 opts.str().c_str(), "deltas");
}

// ------------------------------------------------------------------ luma / misc --------
cl_event DataPipeline::extract_luma(opencl::utils::ImageData& img, MemoryHandle& gpu_buf_raw_img,
                                    MemoryHandle& gpu_buf_luma, bool normalize, cl_event*) {
  check_initialized(LOAD_KERNEL_LUMA);
  const size_t px = (size_t)img.w * img.h;
  opencl::Kernel* kernel = normalize ? _luma_kernel_norm : _luma_kernel_raw;
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_raw_img, px))
    gpu_buf_raw_img = _context->create_image(CL_MEM_READ_WRITE, CL_RGBA, CL_UNSIGNED_INT8, img.w, img.h);
  _context->write_image(gpu_buf_raw_img, img, true);
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_luma, px))
    gpu_buf_luma = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * px);
  ProfiledLaunch pl(*kernel);
  _context->check_status(srcnn_extract_luma(_context->c_ctx(), _context->mem(gpu_buf_raw_img),
                                            _context->mem(gpu_buf_luma), img.w, img.h,
                                            normalize ? 1 : 0),
                         "extract_luma");
  return _context->ticket();
}

// created on first use, so that `profile` output lists it only for runs that enlarge
opencl::Kernel* DataPipeline::resample_kernel() {
  if (!_resample_kernel)
    _resample_kernel = _context->create_kernel((kernel_folder + resample_kernel_file).c_str(),
                                               nullptr, "resample");
  return _resample_kernel;
}

cl_event DataPipeline::resample(opencl::utils::ImageData& img, MemoryHandle& gpu_buf_raw_img,
                                size_t out_w, size_t out_h, int filter, MemoryHandle& gpu_buf_out,
                                MemoryHandle& gpu_buf_luma) {
  check_initialized(LOAD_KERNEL_LUMA);
  const size_t px = (size_t)img.w * img.h, out_px = out_w * out_h;
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_raw_img, px * 4))
    gpu_buf_raw_img = _context->create_image(CL_MEM_READ_WRITE, CL_RGBA, CL_UNSIGNED_INT8, img.w, img.h);
  _context->write_image(gpu_buf_raw_img, img, true);
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_out, out_px * 4))
    gpu_buf_out = _context->create_image(CL_MEM_READ_WRITE, CL_RGBA, CL_UNSIGNED_INT8, out_w, out_h);
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_luma, sizeof(float) * out_px))
    gpu_buf_luma = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * out_px);
  ProfiledLaunch pl(*resample_kernel());
  _context->check_status(srcnn_resample(_context->c_ctx(), _context->mem(gpu_buf_raw_img), img.w,
                                        img.h, _context->mem(gpu_buf_out),
                                        _context->mem(gpu_buf_luma), (int)out_w, (int)out_h, filter),
                         "resample");
  return _context->ticket();
}

cl_event DataPipeline::swap_luma(opencl::utils::ImageData& img, MemoryHandle& gpu_buf_org_img,
                                 MemoryHandle gpu_buf_new_luma, MemoryHandle& target,
                                 size_t new_luma_w, size_t new_luma_h, cl_event*) {
  check_initialized(LOAD_KERNEL_LUMA);
  const size_t px = (size_t)img.w * img.h;
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_new_luma, new_luma_w * new_luma_h * sizeof(float)))
    throw std::runtime_error("Invalid size of new luma buffer");
  if (!ALLOCATION_HAS_RIGHT_SIZE(target, px * 3)) target = _context->allocate(CL_MEM_READ_WRITE, px * 3);
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_org_img, px * 4))
    gpu_buf_org_img = _context->create_image(CL_MEM_READ_WRITE, CL_RGBA, CL_UNSIGNED_INT8, img.w, img.h);
  _context->write_image(gpu_buf_org_img, img, true);
  ProfiledLaunch pl(*_swap_luma_kernel);
  _context->check_status(
      srcnn_swap_luma(_context->c_ctx(), _context->mem(gpu_buf_org_img),
                      _context->mem(gpu_buf_new_luma), _context->mem(target), img.w, img.h,
                      (int)new_luma_w, (int)new_luma_h),
      "swap_luma");
  return _context->ticket();
}

cl_event DataPipeline::subtract_mean(MemoryHandle data, float* mean, cl_event* ev_to_wait_for) {
  check_initialized(LOAD_KERNEL_MISC);
  const size_t len = element_count(data, sizeof(float));
  // Quirk Q1, kept on purpose: the event POINTER converts to sum()'s `bool squared`
  // (reference: src/DataPipeline.cpp:274 vs src/DataPipeline.hpp:171).
  const float buf_sum = sum(data, ev_to_wait_for);
  const float mean_v = buf_sum / len;
  if (mean) *mean = mean_v;
  return subtract_from_all(data, mean_v);
}

float DataPipeline::sum(MemoryHandle data, bool squared, cl_event*) {
  if (cnn_sr::warn_about_blocking_operation) std::cout << "BLOCK: sum" << std::endl;
  check_initialized(LOAD_KERNEL_MISC);
  const size_t len = element_count(data, sizeof(float));
  opencl::Kernel* kernel = squared ? _sum_squared_kernel : _sum_kernel;
  if (!ALLOCATION_HAS_RIGHT_SIZE(_tmp_gpu_float, sizeof(float)))
    _tmp_gpu_float = _context->allocate(CL_MEM_READ_WRITE, sizeof(float));
  float result = 0.f;
  {
    ProfiledLaunch pl(*kernel);
    _context->check_status(srcnn_sum(_context->c_ctx(), _context->mem(data), (unsigned)len,
                                     squared ? 1 : 0, _context->mem(_tmp_gpu_float)),
                           "sum");
  }
  _context->read_buffer(_tmp_gpu_float, &result, true);
  return result;
}

cl_event DataPipeline::subtract_from_all(MemoryHandle data, float val, cl_event*) {
  check_initialized(LOAD_KERNEL_MISC);
  const size_t len = element_count(data, sizeof(float));
  ProfiledLaunch pl(*_subtract_from_all_kernel);
  _context->check_status(
      srcnn_sub_from_all(_context->c_ctx(), _context->mem(data), val, (unsigned)len),
      "sub_from_all");
  return _context->ticket();
}

// ------------------------------------------------------------------ forward ------------
void DataPipeline::pre_execute_layer_validation(const LayerData& data, MemoryHandle input,
                                                size_t input_w, size_t input_h) {
  LayerData::validate(data);
  const size_t expected = data.input_size(input_w, input_h);
  const size_t cnt = element_count(input, sizeof(float));
  if (expected > cnt) {
    std::ostringstream os;
    os << "Declared input_w(" << input_w << ")*input_h(" << input_h << ")*n_prev_filter_cnt("
       << data.n_prev_filter_cnt << ")=" << expected
       << " is bigger then allocated gpu memory (" << cnt << " elements).";
    throw std::runtime_error(os.str());
  }
}

cl_event DataPipeline::execute_layer(opencl::Kernel& kernel, const LayerData& data,
                                     LayerAllocationPool& gpu_alloc, MemoryHandle& gpu_buf_in,
                                     size_t input_w, size_t input_h, size_t sample_count,
                                     MemoryHandle& gpu_buf_out, cl_event*) {
  pre_execute_layer_validation(data, gpu_buf_in, input_w, input_h);
  size_t out[2];
  data.get_output_dimensions(out, input_w, input_h);
  const size_t out_bytes = sizeof(float) * out[0] * out[1] * data.current_filter_count * sample_count;
  const size_t w_bytes = sizeof(float) * data.weight_size(), b_bytes = sizeof(float) * data.bias_size();
  // parameters are uploaded once; afterwards the device copy is authoritative
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.weights, w_bytes)) {
    gpu_alloc.weights = _context->allocate(CL_MEM_READ_WRITE, w_bytes);
    _context->write_buffer(gpu_alloc.weights, (void*)data.weights_ptr(), true);
  }
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.bias, b_bytes)) {
    gpu_alloc.bias = _context->allocate(CL_MEM_READ_WRITE, b_bytes);
    _context->write_buffer(gpu_alloc.bias, (void*)data.bias_ptr(), true);
  }
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_out, out_bytes))
    gpu_buf_out = _context->allocate(CL_MEM_READ_WRITE, out_bytes);
  // the Kernel object carries the "-D" specialisation: it must describe this layer
  if (kernel.kind() != opencl::Kernel::Kind::Forward ||
      kernel.current_filter_count != data.current_filter_count ||
      kernel.previous_filter_count != data.n_prev_filter_cnt ||
      kernel.f_spatial_size != data.f_spatial_size)
    throw std::runtime_error("execute_layer: kernel was created for a different layer shape");
  ProfiledLaunch pl(kernel);
  _context->check_status(
      srcnn_forward_layer(_context->c_ctx(), _context->mem(gpu_buf_in), _context->mem(gpu_buf_out),
                          _context->mem(gpu_alloc.weights), _context->mem(gpu_alloc.bias),
                          (int)data.n_prev_filter_cnt, (int)data.current_filter_count,
                          (int)data.f_spatial_size, kernel.skip_relu ? 1 : 0, (int)input_w,
                          (int)input_h, (int)sample_count),
      "forward");
  return _context->ticket();
}

// ------------------------------------------------------------------ backward -----------
cl_event DataPipeline::squared_error(MemoryHandle gpu_buf_ground_truth, size_t ground_truth_w,
                                     size_t ground_truth_h, size_t sample_count,
                                     MemoryHandle gpu_buf_algo_res, MemoryHandle tmp_buffer,
                                     float& target, size_t total_padding, cl_event*) {
  check_initialized(LOAD_KERNEL_MISC);
  const size_t algo_w = ground_truth_w - total_padding, algo_h = ground_truth_h - total_padding;
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_algo_res, sizeof(float) * algo_w * algo_h))
    throw std::runtime_error("Allocated gpu_buf_algo_res buffer size did not match calculated size");
  if (tmp_buffer == gpu_nullptr) {
    if (!ALLOCATION_HAS_RIGHT_SIZE(_tmp_gpu_float, sizeof(float)))
      _tmp_gpu_float = _context->allocate(CL_MEM_READ_WRITE, sizeof(float));
    tmp_buffer = _tmp_gpu_float;
  }
  {
    ProfiledLaunch pl(*_squared_error_kernel);
    _context->check_status(
        srcnn_squared_error(_context->c_ctx(), _context->mem(gpu_buf_ground_truth),
                            _context->mem(gpu_buf_algo_res), _context->mem(tmp_buffer),
                            (int)ground_truth_w, (int)ground_truth_h, (int)algo_w, (int)algo_h,
                            (int)sample_count),
        "squared_err");
  }
  // non-blocking read: `target` is valid after the event / Context::block()
  return _context->read_buffer(tmp_buffer, 0, sizeof(float), &target, false);
}

cl_event DataPipeline::last_layer_delta(MemoryHandle gpu_buf_ground_truth, size_t ground_truth_w,
                                        size_t ground_truth_h, size_t sample_count,
                                        MemoryHandle gpu_buf_algo_res, MemoryHandle& gpu_buf_target,
                                        size_t total_padding, cl_event*) {
  check_initialized(LOAD_KERNEL_BACKPROPAGATE);
  const size_t algo_w = ground_truth_w - total_padding, algo_h = ground_truth_h - total_padding;
  const size_t bytes = sizeof(float) * algo_w * algo_h * sample_count;
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_algo_res, sizeof(float) * algo_w * algo_h))
    throw std::runtime_error("Allocated gpu_buf_algo_res buffer size did not match calculated size");
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_buf_target, bytes))
    gpu_buf_target = _context->allocate(CL_MEM_READ_WRITE, bytes);
  ProfiledLaunch pl(*_last_layer_delta_kernel);
  _context->check_status(
      srcnn_last_layer_delta(_context->c_ctx(), _context->mem(gpu_buf_ground_truth),
                             _context->mem(gpu_buf_algo_res), _context->mem(gpu_buf_target),
                             (int)ground_truth_w, (int)ground_truth_h, (int)algo_w, (int)algo_h,
                             (int)sample_count),
      "last_layer_delta");
  return _context->ticket();
}

cl_event DataPipeline::calculate_deltas(opencl::Kernel& kernel, const LayerData& curr_layer,
                                        const LayerData& next_layer,
                                        LayerAllocationPool& next_gpu_alloc,
                                        MemoryHandle curr_deltas, MemoryHandle next_deltas,
                                        size_t next_layer_out_w, size_t next_layer_out_h,
                                        size_t sample_count, MemoryHandle curr_output, cl_event*) {
  LayerData::validate(next_layer);
  if (curr_layer.current_filter_count != next_layer.n_prev_filter_cnt)
    throw std::runtime_error(
        "When calculating deltas for layer it's filter count should be equal to next layer's "
        "previous filter count");
  const size_t out_w = next_layer_out_w + next_layer.f_spatial_size - 1,
               out_h = next_layer_out_h + next_layer.f_spatial_size - 1;
  const size_t out_bytes = sizeof(float) * out_w * out_h * next_layer.n_prev_filter_cnt * sample_count;
  const size_t w_bytes = sizeof(float) * next_layer.weight_size();
  if (!ALLOCATION_HAS_RIGHT_SIZE(next_gpu_alloc.weights, w_bytes)) {
    next_gpu_alloc.weights = _context->allocate(CL_MEM_READ_WRITE, w_bytes);
    _context->write_buffer(next_gpu_alloc.weights, (void*)next_layer.weights_ptr(), true);
  }
  if (!ALLOCATION_HAS_RIGHT_SIZE(curr_output, out_bytes))
    throw std::runtime_error(
        "Tried to calculate deltas for previous layer, but there are no previous layer output "
        "values.They are normally allocated during forward step.");
  if (kernel.kind() != opencl::Kernel::Kind::Deltas ||
      kernel.current_filter_count != curr_layer.current_filter_count)
    throw std::runtime_error("calculate_deltas: kernel was created for a different filter count");
  ProfiledLaunch pl(kernel);
  _context->check_status(
      srcnn_deltas(_context->c_ctx(), _context->mem(next_deltas), _context->mem(curr_output),
                   _context->mem(curr_deltas), _context->mem(next_gpu_alloc.weights),
                   (int)curr_layer.current_filter_count, (int)next_layer.f_spatial_size,
                   (int)next_layer.current_filter_count, (int)out_w, (int)out_h,
                   (int)sample_count),
      "deltas");
  return _context->ticket();
}

cl_event DataPipeline::backpropagate(LayerData& layer_data, MemoryHandle layer_input,
                                     MemoryHandle layer_deltas, LayerAllocationPool& gpu_alloc,
                                     size_t layer_out_w, size_t layer_out_h, size_t sample_count,
                                     cl_event*, size_t) {
  LayerData::validate(layer_data);
  check_initialized(LOAD_KERNEL_BACKPROPAGATE);
  const size_t input_w = layer_out_w + layer_data.f_spatial_size - 1,
               input_h = layer_out_h + layer_data.f_spatial_size - 1;
  const size_t in_bytes = sizeof(float) * input_w * input_h * layer_data.n_prev_filter_cnt * sample_count;
  const size_t gw_bytes = sizeof(float) * layer_data.weight_size(),
               gb_bytes = sizeof(float) * layer_data.bias_size();
  if (!ALLOCATION_HAS_RIGHT_SIZE(layer_input, in_bytes))
    throw std::runtime_error(
        "Tried to calculate gradients, but there are no previous layer output values.They are "
        "normally allocated during forward step.");
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.accumulating_grad_w, gw_bytes)) {
    gpu_alloc.accumulating_grad_w = _context->allocate(CL_MEM_READ_WRITE, gw_bytes);
    _context->zeros_float(gpu_alloc.accumulating_grad_w, true);
  }
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.accumulating_grad_b, gb_bytes)) {
    gpu_alloc.accumulating_grad_b = _context->allocate(CL_MEM_READ_WRITE, gb_bytes);
    _context->zeros_float(gpu_alloc.accumulating_grad_b, true);
  }
  ProfiledLaunch pl(*_backpropagate_kernel);
  _context->check_status(
      srcnn_backpropagate(_context->c_ctx(), _context->mem(layer_deltas), _context->mem(layer_input),
                          _context->mem(gpu_alloc.accumulating_grad_w),
                          _context->mem(gpu_alloc.accumulating_grad_b),
                          (int)layer_data.current_filter_count, (int)layer_data.n_prev_filter_cnt,
                          (int)layer_data.f_spatial_size, (int)layer_out_w, (int)layer_out_h,
                          (int)sample_count),
      "backpropagate");
  return _context->ticket();
}

cl_event DataPipeline::update_parameters(LayerData& layer_data, LayerAllocationPool& gpu_alloc,
                                         size_t batch_size, float momentum, float w_decay,
                                         float learning_rate, cl_event*) {
  LayerData::validate(layer_data);
  check_initialized(LOAD_KERNEL_BACKPROPAGATE);
  const size_t ws = layer_data.weight_size(), bs = layer_data.bias_size();
  const size_t w_bytes = sizeof(float) * ws, b_bytes = sizeof(float) * bs;
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.weights, w_bytes))
    throw std::runtime_error("Tried to update weights, but old values are not valid. Impossible if forward pass was completed");
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.bias, b_bytes))
    throw std::runtime_error("Tried to update bias, but old values are not valid. Impossible if forward pass was completed");
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.accumulating_grad_w, w_bytes))
    throw std::runtime_error("Tried to update weights, but gradient values are not valid. Impossible if backpropagation was completed");
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.accumulating_grad_b, b_bytes))
    throw std::runtime_error("Tried to update bias, but gradient values are not valid. Impossible if backpropagation was completed");
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.previous_batch_delta_w, w_bytes)) {
    gpu_alloc.previous_batch_delta_w = _context->allocate(CL_MEM_READ_WRITE, w_bytes);
    _context->zeros_float(gpu_alloc.previous_batch_delta_w, true);
  }
  if (!ALLOCATION_HAS_RIGHT_SIZE(gpu_alloc.previous_batch_delta_b, b_bytes)) {
    gpu_alloc.previous_batch_delta_b = _context->allocate(CL_MEM_READ_WRITE, b_bytes);
    _context->zeros_float(gpu_alloc.previous_batch_delta_b, true);
  }
  ProfiledLaunch pl(*_update_parameters_kernel);
  _context->check_status(
      srcnn_update_params(_context->c_ctx(), _context->mem(gpu_alloc.weights),
                          _context->mem(gpu_alloc.bias), _context->mem(gpu_alloc.accumulating_grad_w),
                          _context->mem(gpu_alloc.accumulating_grad_b),
                          _context->mem(gpu_alloc.previous_batch_delta_w),
                          _context->mem(gpu_alloc.previous_batch_delta_b), momentum, w_decay,
                          learning_rate, (unsigned)batch_size, (unsigned)ws, (unsigned)bs),
      "update_params");
  return _context->ticket();
}

}  // namespace cnn_sr
