#include "ConfigBasedDataPipeline.hpp"

#include <chrono>
#include <cstdlib>
#include <fstream>
#include <random>
#include <stdexcept>

#include "json.hpp"

using opencl::MemoryHandle;

namespace {
const bool print_steps = false;
const char* const layer_keys[3] = {"layer1", "layer2", "layer3"};
}  // namespace

namespace cnn_sr {

ConfigBasedDataPipeline::ConfigBasedDataPipeline(Config& cfg, opencl::Context* context)
    : DataPipeline(context),
      _config(&cfg),
      layer_data_1(1, cfg.n1, cfg.f1),
      layer_data_2(cfg.n1, cfg.n2, cfg.f2),
      layer_data_3(cfg.n2, 1, cfg.f3) {}

void ConfigBasedDataPipeline::init(int load_flags) {
  DataPipeline::init(load_flags);
  if (!_config->parameters_file.empty()) {
    std::cout << "Loading layer parameters from: '" << _config->parameters_file << "'" << std::endl;
    this->epochs = load_parameters_file(_config->parameters_file.c_str());
    std::cout << "Previous epochs:  " << this->epochs << std::endl;
  } else {
    std::cout << "No parameters file provided, initializing random weights and biases"
              << std::endl;
    fill_random_parameters(layer_data_1, _config->params_distr_1);
    fill_random_parameters(layer_data_2, _config->params_distr_2);
    fill_random_parameters(layer_data_3, _config->params_distr_3);
  }
  LayerData::validate(layer_data_1);
  LayerData::validate(layer_data_2);
  LayerData::validate(layer_data_3);
}

void ConfigBasedDataPipeline::load_kernels(int load_flags) {
  DataPipeline::load_kernels(load_flags);
  if (load_flags & DataPipeline::LOAD_KERNEL_LAYERS) {
    if (!_layer_1_kernel) _layer_1_kernel = create_layer_kernel(layer_data_1, false);
    if (!_layer_2_kernel) _layer_2_kernel = create_layer_kernel(layer_data_2, false);
    if (!_layer_3_kernel) _layer_3_kernel = create_layer_kernel(layer_data_3, true);
  }
  if (load_flags & DataPipeline::LOAD_KERNEL_BACKPROPAGATE) {
    if (!_layer_1_deltas_kernel) _layer_1_deltas_kernel = create_deltas_kernel(layer_data_1);
    if (!_layer_2_deltas_kernel) _layer_2_deltas_kernel = create_deltas_kernel(layer_data_2);
  }
}

void ConfigBasedDataPipeline::set_mini_batch_size(size_t mini_batch_size) {
  _mini_batch_size = mini_batch_size;
  std::cout << "mini-batch size: " << _mini_batch_size << std::endl;
}

// The reference allocates all eight batch buffers -- deltas included -- even for inference
// (src/ConfigBasedDataPipeline.cpp:82-108; 13 GB for a 4096x4096 image) and leaks the old
// ones on every forward(sample).  Here inference through the fused launch needs only the
// input and the layer-3 output; old buffers are released when the shape changes.
void ConfigBasedDataPipeline::allocate_buffers(size_t w, size_t h, bool training) {
  if (_out_3_gpu_buf != gpu_nullptr && _alloc_w == w && _alloc_h == h &&
      _alloc_batch >= _mini_batch_size && (_alloc_training || !training))
    return;
  for (MemoryHandle* m : {&_ground_truth_gpu_buf, &_forward_gpu_buf, &_out_1_gpu_buf,
                          &_out_2_gpu_buf, &_out_3_gpu_buf, &_delta_1_gpu_buf,
                          &_delta_2_gpu_buf, &_delta_3_gpu_buf}) {
    if (*m != gpu_nullptr) _context->raw_memory(*m)->release();
    *m = gpu_nullptr;
  }
  size_t d1[2], d2[2], d3[2];
  layer_data_1.get_output_dimensions(d1, w, h);
  layer_data_2.get_output_dimensions(d2, d1[0], d1[1]);
  layer_data_3.get_output_dimensions(d3, d2[0], d2[1]);
  if (w < _config->total_padding() + 1 || h < _config->total_padding() + 1)
    throw std::runtime_error("Image is smaller than the network's total padding");
  const size_t S = _mini_batch_size * sizeof(float);
  const size_t per0 = w * h, per1 = d1[0] * d1[1] * layer_data_1.current_filter_count,
               per2 = d2[0] * d2[1] * layer_data_2.current_filter_count, per3 = d3[0] * d3[1];
  srcnn_net probe{};
  probe.n1 = (int)_config->n1; probe.n2 = (int)_config->n2;
  probe.f1 = (int)_config->f1; probe.f2 = (int)_config->f2; probe.f3 = (int)_config->f3;
  const bool fused = !training && !_context->is_running_profile_mode() &&
                     srcnn_forward_fused_supported(&probe);
  _forward_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per0);
  _out_3_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per3);
  if (!fused) {
    _out_1_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per1);
    _out_2_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per2);
  }
  if (training) {
    _ground_truth_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per0);
    _delta_1_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per1);
    _delta_2_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per2);
    _delta_3_gpu_buf = _context->allocate(CL_MEM_READ_WRITE, S * per3);
  }
  _alloc_w = w;
  _alloc_h = h;
  _alloc_batch = _mini_batch_size;
  _alloc_training = training;
}

void ConfigBasedDataPipeline::ensure_parameters_on_device(LayerData& data, LayerAllocationPool& pool) {
  // data parallel: every rank starts from rank 0's values (random initialisation is time-seeded
  // per process); srcnn_broadcast is a no-op without a communicator
  if (pool.weights == gpu_nullptr) {
    pool.weights = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * data.weight_size());
    _context->write_buffer(pool.weights, (void*)data.weights_ptr(), true);
    _context->check_status(srcnn_broadcast(_context->c_ctx(), _context->mem(pool.weights),
                                           data.weight_size(), 0), "broadcast of the weights");
  }
  if (pool.bias == gpu_nullptr) {
    pool.bias = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * data.bias_size());
    _context->write_buffer(pool.bias, (void*)data.bias_ptr(), true);
    _context->check_status(srcnn_broadcast(_context->c_ctx(), _context->mem(pool.bias),
                                           data.bias_size(), 0), "broadcast of the bias");
  }
}

srcnn_net ConfigBasedDataPipeline::device_net(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                              LayerAllocationPool& l3, bool with_gradients,
                                              bool with_momentum) {
  srcnn_net net{};
  net.n1 = (int)_config->n1; net.n2 = (int)_config->n2;
  net.f1 = (int)_config->f1; net.f2 = (int)_config->f2; net.f3 = (int)_config->f3;
  LayerData* layers[3] = {&layer_data_1, &layer_data_2, &layer_data_3};
  LayerAllocationPool* pools[3] = {&l1, &l2, &l3};
  for (int i = 0; i < 3; i++) {
    ensure_parameters_on_device(*layers[i], *pools[i]);
    net.w[i] = _context->mem(pools[i]->weights);
    net.b[i] = _context->mem(pools[i]->bias);
    net.grad_w[i] = net.grad_b[i] = net.prev_dw[i] = net.prev_db[i] = SRCNN_NULL_MEM;
    if (with_gradients) {
      ensure_gradients_on_device(*layers[i], *pools[i]);
      net.grad_w[i] = _context->mem(pools[i]->accumulating_grad_w);
      net.grad_b[i] = _context->mem(pools[i]->accumulating_grad_b);
    }
    if (with_momentum) {
      ensure_momentum_on_device(i, *layers[i], *pools[i]);
      net.prev_dw[i] = _context->mem(pools[i]->previous_batch_delta_w);
      net.prev_db[i] = _context->mem(pools[i]->previous_batch_delta_b);
    }
  }
  return net;
}

// momentum state: zero, or what the "resume" key of the parameters file held
void ConfigBasedDataPipeline::ensure_momentum_on_device(int layer, LayerData& data,
                                                        LayerAllocationPool& pool) {
  if (pool.previous_batch_delta_w == gpu_nullptr) {
    pool.previous_batch_delta_w = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * data.weight_size());
    if (_resume_prev_w[layer].size() == data.weight_size())
      _context->write_buffer(pool.previous_batch_delta_w, _resume_prev_w[layer].data(), true);
    else
      _context->zeros_float(pool.previous_batch_delta_w, true);
  }
  if (pool.previous_batch_delta_b == gpu_nullptr) {
    pool.previous_batch_delta_b = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * data.bias_size());
    if (_resume_prev_b[layer].size() == data.bias_size())
      _context->write_buffer(pool.previous_batch_delta_b, _resume_prev_b[layer].data(), true);
    else
      _context->zeros_float(pool.previous_batch_delta_b, true);
  }
}

// ------------------------------------------------------------------ forward ------------
cl_event ConfigBasedDataPipeline::forward(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                          LayerAllocationPool& l3, SampleAllocationPool& sample) {
  set_mini_batch_size(1);
  allocate_buffers(sample.input_w, sample.input_h, false);
  _context->copy_buffer(sample.input_luma, _forward_gpu_buf);
  return forward(l1, l2, l3, sample.input_w, sample.input_h, 1);
}

cl_event ConfigBasedDataPipeline::forward(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                          LayerAllocationPool& l3, size_t w, size_t h,
                                          size_t sample_count) {
  check_initialized(DataPipeline::LOAD_KERNEL_LAYERS);
  if (sample_count > _mini_batch_size)
    throw std::runtime_error("Allocation pool out of bounds exception");
  size_t d1[2], d2[2];
  layer_data_1.get_output_dimensions(d1, w, h);
  layer_data_2.get_output_dimensions(d2, d1[0], d1[1]);

  srcnn_net probe = device_net(l1, l2, l3, false, false);
  if (_out_1_gpu_buf == gpu_nullptr ||
      (!_context->is_running_profile_mode() && srcnn_forward_fused_supported(&probe))) {
    // inference / validation through the single fused launch: the n1/n2-channel maps stay on
    // chip (the `profile` mode keeps the per-kernel sequence so its totals stay meaningful)
    const srcnn_net& net = probe;
    _context->check_status(
        srcnn_forward_fused(_context->c_ctx(), &net, _context->mem(_forward_gpu_buf),
                            _context->mem(_out_3_gpu_buf), (int)w, (int)h, (int)sample_count,
                            SRCNN_NULL_MEM, SRCNN_NULL_MEM),
        "forward (fused)");
    return _context->ticket();
  }

  if (print_steps) std::cout << "### Executing layer 1" << std::endl;
  cl_event e1 = execute_layer(*_layer_1_kernel, layer_data_1, l1, _forward_gpu_buf, w, h,
                              sample_count, _out_1_gpu_buf);
  if (print_steps) std::cout << "### Executing layer 2" << std::endl;
  cl_event e2 = execute_layer(*_layer_2_kernel, layer_data_2, l2, _out_1_gpu_buf, d1[0], d1[1],
                              sample_count, _out_2_gpu_buf, &e1);
  if (print_steps) std::cout << "### Executing layer 3" << std::endl;
  return execute_layer(*_layer_3_kernel, layer_data_3, l3, _out_2_gpu_buf, d2[0], d2[1],
                       sample_count, _out_3_gpu_buf, &e2);
}

// ------------------------------------------------------------------ batches ------------
float ConfigBasedDataPipeline::execute_batch(bool backpropagate__, GpuAllocationPool& gpu_alloc,
                                             std::vector<SampleAllocationPool*>& sample_set) {
  if (sample_set.empty() || _mini_batch_size == 0)
    throw std::runtime_error("Batch cannot be empty");
  const size_t w = sample_set[0]->input_w, h = sample_set[0]->input_h;
  allocate_buffers(w, h, true);

  float validation_error = 0.0f;
  size_t i = 0;
  while (i < sample_set.size()) {
    // gather the chunk's samples into contiguous [S][h][w] buffers: ONE launch per tensor (the
    // reference enqueues 2 copies per sample, src/ConfigBasedDataPipeline.cpp:149-161)
    size_t in_batch = 0;
    std::vector<srcnn_mem> src_in, src_gt;
    for (size_t j = i; in_batch < _mini_batch_size && j < sample_set.size(); ++j, ++in_batch) {
      SampleAllocationPool& s = *sample_set[j];
      if (s.input_w != w || s.input_h != h)
        throw std::runtime_error("All samples of a batch must have the same dimensions");
      src_in.push_back(_context->mem(s.input_luma));
      src_gt.push_back(_context->mem(s.expected_luma));
    }
    _context->check_status(srcnn_gather(_context->c_ctx(), src_in.data(), (int)in_batch,
                                        w * h * sizeof(float), _context->mem(_forward_gpu_buf)),
                           "gather input luma");
    _context->check_status(srcnn_gather(_context->c_ctx(), src_gt.data(), (int)in_batch,
                                        w * h * sizeof(float), _context->mem(_ground_truth_gpu_buf)),
                           "gather expected luma");
    if (backpropagate__ && !_context->is_running_profile_mode()) {
      // forward() + backpropagate() of the chunk as ONE call into the device layer (fused
      // tensor-core forward that keeps out1/out2, fused backward of the last layer); the
      // `profile` mode keeps the per-kernel sequence so that its per-kernel totals stay
      // meaningful (src/opencl/Kernel.cpp:108-116)
      train_chunk(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, w, h, in_batch);
      _context->block();
      i += in_batch;
      continue;
    }
    cl_event forward_ev =
        forward(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, w, h, in_batch);
    if (backpropagate__) {
      backpropagate(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, w, h, in_batch,
                    &forward_ev);
    } else {
      float chunk_error = 0.0f;
      cl_event e = squared_error(_ground_truth_gpu_buf, w, h, in_batch, _out_3_gpu_buf,
                                 _tmp_gpu_float, chunk_error, _config->total_padding(), &forward_ev);
      clWaitForEvents(1, &e);
      validation_error += chunk_error;
    }
    _context->block();
    i += in_batch;
  }
  return validation_error;
}

void ConfigBasedDataPipeline::ensure_gradients_on_device(LayerData& data, LayerAllocationPool& pool) {
  if (pool.accumulating_grad_w == gpu_nullptr) {
    pool.accumulating_grad_w = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * data.weight_size());
    _context->zeros_float(pool.accumulating_grad_w, true);
  }
  if (pool.accumulating_grad_b == gpu_nullptr) {
    pool.accumulating_grad_b = _context->allocate(CL_MEM_READ_WRITE, sizeof(float) * data.bias_size());
    _context->zeros_float(pool.accumulating_grad_b, true);
  }
}

void ConfigBasedDataPipeline::train_chunk(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                          LayerAllocationPool& l3, size_t w, size_t h,
                                          size_t sample_count) {
  check_initialized(DataPipeline::LOAD_KERNEL_LAYERS);
  if (sample_count > _mini_batch_size)
    throw std::runtime_error("Allocation pool out of bounds exception");
  const srcnn_net net = device_net(l1, l2, l3, true, false);
  _context->check_status(
      srcnn_train_chunk_buffers(_context->c_ctx(), &net, _context->mem(_forward_gpu_buf),
                                _context->mem(_ground_truth_gpu_buf), (int)w, (int)h,
                                (int)sample_count, _context->mem(_out_1_gpu_buf),
                                _context->mem(_out_2_gpu_buf), _context->mem(_out_3_gpu_buf),
                                _context->mem(_delta_1_gpu_buf), _context->mem(_delta_2_gpu_buf),
                                _context->mem(_delta_3_gpu_buf)),
      "train chunk");
}

cl_event ConfigBasedDataPipeline::backpropagate(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                                LayerAllocationPool& l3, size_t w, size_t h,
                                                size_t sample_count, cl_event* ev) {
  size_t d1[2], d2[2], d3[2];
  layer_data_1.get_output_dimensions(d1, w, h);
  layer_data_2.get_output_dimensions(d2, d1[0], d1[1]);
  layer_data_3.get_output_dimensions(d3, d2[0], d2[1]);
  const size_t padding = _config->total_padding();
  // deltas, last layer first
  cl_event e_d3 = last_layer_delta(_ground_truth_gpu_buf, w, h, sample_count, _out_3_gpu_buf,
                                   _delta_3_gpu_buf, padding, ev);
  cl_event e_d2 = calculate_deltas(*_layer_2_deltas_kernel, layer_data_2, layer_data_3, l3,
                                   _delta_2_gpu_buf, _delta_3_gpu_buf, d3[0], d3[1],
                                   sample_count, _out_2_gpu_buf, &e_d3);
  cl_event e_d1 = calculate_deltas(*_layer_1_deltas_kernel, layer_data_1, layer_data_2, l2,
                                   _delta_1_gpu_buf, _delta_2_gpu_buf, d2[0], d2[1],
                                   sample_count, _out_1_gpu_buf, &e_d2);
  // weight / bias gradients
  cl_event e_g3 = DataPipeline::backpropagate(layer_data_3, _out_2_gpu_buf, _delta_3_gpu_buf, l3,
                                              d3[0], d3[1], sample_count, &e_d3);
  cl_event e_g2 = DataPipeline::backpropagate(layer_data_2, _out_1_gpu_buf, _delta_2_gpu_buf, l2,
                                              d2[0], d2[1], sample_count, &e_d2);
  cl_event evs[3] = {e_d1, e_g3, e_g2};
  return DataPipeline::backpropagate(layer_data_1, _forward_gpu_buf, _delta_1_gpu_buf, l1, d1[0],
                                     d1[1], sample_count, evs, 3);
}

void ConfigBasedDataPipeline::update_parameters(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                                LayerAllocationPool& l3, size_t batch_size,
                                                cl_event* ev) {
  if (!_context->is_running_profile_mode()) {
    // ONE launch for the three layers + the zeroing of the six accumulators; with a
    // communicator, the gradients of all ranks are summed first and `batch_size` is the GLOBAL
    // sample count, so the rule (quirk Q3) is unchanged
    const srcnn_net net = device_net(l1, l2, l3, true, true);
    _context->check_status(srcnn_allreduce_grads(_context->c_ctx(), &net), "all-reduce of the gradients");
    const float lr[3] = {_config->learning_rate[0], _config->learning_rate[1], _config->learning_rate[2]};
    _context->check_status(srcnn_update_all(_context->c_ctx(), &net, (unsigned)batch_size,
                                            _config->momentum, _config->weight_decay_parameter, lr),
                           "update_parameters");
    _context->block();
    ++epochs;
    return;
  }
  DataPipeline::update_parameters(layer_data_3, l3, batch_size, _config->momentum,
                                  _config->weight_decay_parameter, _config->learning_rate[2], ev);
  DataPipeline::update_parameters(layer_data_2, l2, batch_size, _config->momentum,
                                  _config->weight_decay_parameter, _config->learning_rate[1], ev);
  DataPipeline::update_parameters(layer_data_1, l1, batch_size, _config->momentum,
                                  _config->weight_decay_parameter, _config->learning_rate[0], ev);
  // device-side fills; the reference uploads host zeros six times (Context.cpp:301-310)
  for (LayerAllocationPool* p : {&l1, &l2, &l3}) {
    _context->zeros_float(p->accumulating_grad_w, false);
    _context->zeros_float(p->accumulating_grad_b, false);
  }
  _context->block();
  ++epochs;
}

// ------------------------------------------------------------------ parameters ---------
void ConfigBasedDataPipeline::fill_random_parameters(LayerData& data, ParametersDistribution& d) {
  // time-seeded like the reference; CNN_SR_SEED makes a run reproducible
  unsigned seed = (unsigned)std::chrono::system_clock::now().time_since_epoch().count();
  if (const char* s = std::getenv("CNN_SR_SEED")) seed = (unsigned)std::strtoul(s, nullptr, 10) + (unsigned)data.weight_size();
  std::default_random_engine generator(seed);
  std::normal_distribution<float> rand_w(d.mean_w, d.sd_w);
  std::normal_distribution<float> rand_b(d.mean_b, d.sd_b);
  for (size_t i = 0; i < data.weight_size(); i++) data.weights.push_back(rand_w(generator));
  for (size_t i = 0; i < data.bias_size(); i++)
    data.bias.push_back(d.sd_b > 0 ? rand_b(generator) : d.mean_b);
}

size_t ConfigBasedDataPipeline::load_parameters_file(const char* const file_path) {
  const json::Value root = json::parse_file(file_path);
  if (!root.is(json::Type::Object))
    throw std::runtime_error("Expected root of JSON file had invalid type");
  size_t file_epochs = 0;
  LayerData* layers[3] = {&layer_data_1, &layer_data_2, &layer_data_3};
  std::vector<float> resume_w[3], resume_b[3];
  for (const auto& kv : root.object) {
    if (kv.first == "epochs" && kv.second.is(json::Type::Number)) {
      file_epochs = (size_t)(unsigned int)kv.second.number;
      continue;
    }
    if (kv.first == "resume" && kv.second.is(json::Type::Object)) {
      // optional extra the reference's reader skips with a warning
      // (src/ConfigBasedDataPipeline.cpp:408-410): full-precision parameters + momentum state
      for (const auto& lk : kv.second.object) {
        int l = -1;
        for (int i = 0; i < 3; i++)
          if (lk.first == layer_keys[i]) l = i;
        if (l < 0 || !lk.second.is(json::Type::Object)) continue;
        for (const auto& sub : lk.second.object) {
          if (!sub.second.is(json::Type::Array)) continue;
          std::vector<float>* target = sub.first == "weights" ? &resume_w[l]
                                       : sub.first == "bias" ? &resume_b[l]
                                       : sub.first == "previous_delta_w" ? &_resume_prev_w[l]
                                       : sub.first == "previous_delta_b" ? &_resume_prev_b[l]
                                                                         : nullptr;
          if (!target) continue;
          target->clear();
          for (const json::Value& v : sub.second.array) target->push_back((float)v.number);
        }
      }
      continue;
    }
    int which = -1;
    for (int l = 0; l < 3; l++)
      if (kv.first == layer_keys[l]) which = l;
    if (which < 0) {
      std::cout << "[Warning] Unknown key '" << kv.first << "' in parameters file" << std::endl;
      continue;
    }
    if (!kv.second.is(json::Type::Object)) continue;
    for (const auto& sub : kv.second.object) {
      if (!sub.second.is(json::Type::Array)) continue;
      std::vector<float>* target = sub.first == "weights" ? &layers[which]->weights
                                   : sub.first == "bias"  ? &layers[which]->bias
                                                          : nullptr;
      if (!target) continue;
      for (const json::Value& v : sub.second.array) target->push_back((float)v.number);
    }
  }
  // the 9-digit copies of "resume" supersede the 6-digit ones (quirk Q6) when they fit
  bool resumed = false;
  for (int l = 0; l < 3; l++) {
    if (resume_w[l].size() == layers[l]->weight_size() && resume_b[l].size() == layers[l]->bias_size()) {
      layers[l]->weights = resume_w[l];
      layers[l]->bias = resume_b[l];
      resumed = true;
    }
  }
  if (resumed)
    std::cout << "Resume state found: full-precision parameters"
              << (_resume_prev_w[0].empty() ? "" : " and momentum") << " restored" << std::endl;
  return file_epochs;
}

static void dump_layer(std::ostream& os, const char* key, std::vector<float>& weights,
                       std::vector<float>& bias) {
  os << "  \"" << key << "\":{" << std::endl << "    \"weights\": [";
  utils::dump_vector(os, weights);
  os << "]," << std::endl << "    \"bias\": [";
  utils::dump_vector(os, bias);
  os << "]" << std::endl << "  }";
}

void ConfigBasedDataPipeline::write_params_to_file(const char* const file_path,
                                                   LayerAllocationPool l1, LayerAllocationPool l2,
                                                   LayerAllocationPool l3) {
  std::cout << "Saving parameters to: '" << file_path << "'" << std::endl;
  LayerData* layers[3] = {&layer_data_1, &layer_data_2, &layer_data_3};
  LayerAllocationPool* pools[3] = {&l1, &l2, &l3};
  for (int l = 0; l < 3; l++) {
    layers[l]->weights.resize(layers[l]->weight_size());
    layers[l]->bias.resize(layers[l]->bias_size());
    if (pools[l]->weights != gpu_nullptr)
      _context->read_buffer(pools[l]->weights, 0, sizeof(float) * layers[l]->weight_size(),
                            layers[l]->weights.data(), true);
    if (pools[l]->bias != gpu_nullptr)
      _context->read_buffer(pools[l]->bias, 0, sizeof(float) * layers[l]->bias_size(),
                            layers[l]->bias.data(), true);
  }
  std::ofstream f(file_path);
  if (!f.is_open()) throw std::ios_base::failure("Could not open parameters file for writing");
  f << "{" << std::endl << "  \"epochs\": " << this->epochs << "," << std::endl << std::endl;
  for (int l = 0; l < 3; l++) {
    dump_layer(f, layer_keys[l], layers[l]->weights, layers[l]->bias);
    if (l < 2) f << "," << std::endl;
  }
  // Resume state (new, optional): the reference restarts momentum at zero and keeps 6 digits
  // (SURVEY 5 "Checkpoint / resume").  Written as ONE extra top-level key, which the reference's
  // reader reports as unknown and skips; CNN_SR_RESUME_STATE=0 leaves it out.
  const char* rs = std::getenv("CNN_SR_RESUME_STATE");
  if (!(rs && std::atoi(rs) == 0)) {
    auto dump9 = [&](const std::vector<float>& v) {
      const std::streamsize old = f.precision(9);
      for (size_t i = 0; i < v.size(); i++) f << (i ? ", " : "") << v[i];
      f.precision(old);
    };
    f << "," << std::endl << "  \"resume\":{" << std::endl;
    for (int l = 0; l < 3; l++) {
      std::vector<float> pw(layers[l]->weight_size(), 0.f), pb(layers[l]->bias_size(), 0.f);
      if (pools[l]->previous_batch_delta_w != gpu_nullptr)
        _context->read_buffer(pools[l]->previous_batch_delta_w, 0, sizeof(float) * pw.size(), pw.data(), true);
      if (pools[l]->previous_batch_delta_b != gpu_nullptr)
        _context->read_buffer(pools[l]->previous_batch_delta_b, 0, sizeof(float) * pb.size(), pb.data(), true);
      f << "    \"" << layer_keys[l] << "\":{" << std::endl << "      \"weights\": [";
      dump9(layers[l]->weights);
      f << "]," << std::endl << "      \"bias\": [";
      dump9(layers[l]->bias);
      f << "]," << std::endl << "      \"previous_delta_w\": [";
      dump9(pw);
      f << "]," << std::endl << "      \"previous_delta_b\": [";
      dump9(pb);
      f << "]" << std::endl << "    }" << (l < 2 ? "," : "") << std::endl;
    }
    f << "  }";
  }
  f << std::endl << "}";
}

void ConfigBasedDataPipeline::write_result_image(const char* const out_path,
                                                 opencl::utils::ImageData& input_img,
                                                 SampleAllocationPool& sample) {
  std::cout << "Saving result image to: '" << out_path << "'" << std::endl;
  const size_t luma_w = input_img.w - _config->total_padding(),
               luma_h = input_img.h - _config->total_padding();
  MemoryHandle gpu_buf_target = gpu_nullptr;
  swap_luma(input_img, sample.input_data, _out_3_gpu_buf, gpu_buf_target, luma_w, luma_h);
  std::vector<unsigned char> result((size_t)input_img.w * input_img.h * 3);
  _context->read_buffer(gpu_buf_target, result.data(), true);
  opencl::utils::ImageData res_img(input_img.w, input_img.h, 3, result.data());
  opencl::utils::write_image(out_path, res_img);
}

void ConfigBasedDataPipeline::upscale_image(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                            LayerAllocationPool& l3, opencl::utils::ImageData& in,
                                            size_t out_w, size_t out_h, int filter,
                                            opencl::utils::ImageData& out) {
  if (in.bpp != 4 || out.bpp != 3 || (size_t)out.w != out_w || (size_t)out.h != out_h)
    throw std::runtime_error("upscale_image: RGBA8 input and an RGB8 output of out_w x out_h expected");
  check_initialized(DataPipeline::LOAD_KERNEL_LUMA | DataPipeline::LOAD_KERNEL_MISC);
  const srcnn_net net = device_net(l1, l2, l3, false, false);
  // `profile`: the per-kernel totals of the steps the call runs besides the forward
  opencl::ProfiledLaunch p1(*resample_kernel()), p2(*_sum_squared_kernel),
      p3(*_subtract_from_all_kernel), p4(*_swap_luma_kernel);
  _context->check_status(srcnn_upscale_image_host(_context->c_ctx(), &net, in.data, in.w, in.h,
                                                  (int)out_w, (int)out_h, filter, out.data),
                         "upscale_image");
}

void ConfigBasedDataPipeline::upscale_frames(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                             LayerAllocationPool& l3, const unsigned char* in_rgba,
                                             size_t w, size_t h, size_t n_frames, size_t out_w,
                                             size_t out_h, int filter, unsigned char* out_rgb) {
  check_initialized(DataPipeline::LOAD_KERNEL_LUMA | DataPipeline::LOAD_KERNEL_MISC);
  const srcnn_net net = device_net(l1, l2, l3, false, false);
  // `profile`: the per-kernel totals of the steps the call runs besides the forward
  opencl::ProfiledLaunch p1(*resample_kernel()), p2(*_sum_squared_kernel),
      p3(*_subtract_from_all_kernel), p4(*_swap_luma_kernel);
  _context->check_status(srcnn_upscale_frames_host(_context->c_ctx(), &net, in_rgba, (int)w, (int)h,
                                                   (int)n_frames, (int)out_w, (int)out_h, filter,
                                                   out_rgb),
                         "upscale_frames");
}

void ConfigBasedDataPipeline::upscale_yuv420_frames(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                                    LayerAllocationPool& l3,
                                                    const unsigned char* in_yuv, size_t w, size_t h,
                                                    size_t n_frames, size_t out_w, size_t out_h,
                                                    int filter, unsigned char* out_yuv,
                                                    int in_siting, int out_siting) {
  check_initialized(DataPipeline::LOAD_KERNEL_LUMA | DataPipeline::LOAD_KERNEL_MISC);
  const srcnn_net net = device_net(l1, l2, l3, false, false);
  opencl::ProfiledLaunch p1(*resample_kernel()), p2(*_sum_squared_kernel),
      p3(*_subtract_from_all_kernel), p4(*_swap_luma_kernel);
  _context->check_status(
      srcnn_upscale_yuv420_frames_host_sited(_context->c_ctx(), &net, in_yuv, (int)w, (int)h,
                                             (int)n_frames, (int)out_w, (int)out_h, filter,
                                             in_siting, out_siting, out_yuv),
      "upscale_yuv420_frames");
}

void ConfigBasedDataPipeline::upscale_yuv420p10_frames(LayerAllocationPool& l1,
                                                       LayerAllocationPool& l2,
                                                       LayerAllocationPool& l3,
                                                       const uint16_t* in_yuv, size_t w, size_t h,
                                                       size_t n_frames, size_t out_w, size_t out_h,
                                                       int filter, uint16_t* out_yuv,
                                                       int in_siting, int out_siting) {
  check_initialized(DataPipeline::LOAD_KERNEL_LUMA | DataPipeline::LOAD_KERNEL_MISC);
  const srcnn_net net = device_net(l1, l2, l3, false, false);
  opencl::ProfiledLaunch p1(*resample_kernel()), p2(*_sum_squared_kernel),
      p3(*_subtract_from_all_kernel), p4(*_swap_luma_kernel);
  _context->check_status(
      srcnn_upscale_yuv420p10_frames_host(_context->c_ctx(), &net, in_yuv, (int)w, (int)h,
                                          (int)n_frames, (int)out_w, (int)out_h, filter, in_siting,
                                          out_siting, out_yuv),
      "upscale_yuv420p10_frames");
}

void ConfigBasedDataPipeline::evaluate_frames(LayerAllocationPool& l1, LayerAllocationPool& l2,
                                              LayerAllocationPool& l3, const unsigned char* in_rgba,
                                              size_t w, size_t h, size_t n_frames, size_t out_w,
                                              size_t out_h, int filter, const unsigned char* ref_rgba,
                                              int border, unsigned char* out_rgb, double* metrics) {
  check_initialized(DataPipeline::LOAD_KERNEL_LUMA | DataPipeline::LOAD_KERNEL_MISC);
  const srcnn_net net = device_net(l1, l2, l3, false, false);
  opencl::ProfiledLaunch p1(*resample_kernel()), p2(*_sum_squared_kernel),
      p3(*_subtract_from_all_kernel), p4(*_swap_luma_kernel);
  _context->check_status(srcnn_evaluate_frames_host(_context->c_ctx(), &net, in_rgba, (int)w, (int)h,
                                                    (int)n_frames, (int)out_w, (int)out_h, filter,
                                                    ref_rgba, border, out_rgb, metrics),
                         "evaluate_frames");
}

}  // namespace cnn_sr
