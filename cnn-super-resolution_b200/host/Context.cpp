#include "Context.hpp"

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <ctime>
#include <fstream>
#include <sstream>
#include <stdexcept>

namespace gpu {

// ------------------------------------------------------------------ images (PPM/PGM) ---
namespace utils {

ImageData::ImageData() : w(0), h(0), bpp(0), data(nullptr) {}
ImageData::ImageData(int w_, int h_, int bpp_, unsigned char* d)
    : w(w_), h(h_), bpp(bpp_), data(d), owned(false) {}
ImageData::~ImageData() {
  if (owned && data) delete[] data;
}

static int read_header_int(std::istream& f) {
  // skips whitespace and '#' comments
  while (true) {
    int c = f.peek();
    if (c == '#') {
      std::string line;
      std::getline(f, line);
    } else if (c == ' ' || c == '\n' || c == '\r' || c == '\t') {
      f.get();
    } else {
      break;
    }
  }
  int v = 0;
  f >> v;
  return v;
}

void load_image(const char* path, ImageData& img) {
  std::ifstream f(path, std::ios::binary);
  if (!f.is_open()) throw std::ios_base::failure(std::string("Could not open image: ") + path);
  std::string magic;
  f >> magic;
  if (magic != "P6" && magic != "P5")
    throw std::ios_base::failure(std::string("Only binary PPM/PGM images are supported "
                                             "(convert with tools/img2ppm.py): ") + path);
  const int channels = magic == "P6" ? 3 : 1;
  const int w = read_header_int(f), h = read_header_int(f), maxv = read_header_int(f);
  f.get();  // single whitespace after maxval
  if (w <= 0 || h <= 0 || maxv != 255)
    throw std::ios_base::failure(std::string("Unsupported PPM header in: ") + path);
  std::vector<unsigned char> raw((size_t)w * h * channels);
  f.read(reinterpret_cast<char*>(raw.data()), (std::streamsize)raw.size());
  if ((size_t)f.gcount() != raw.size())
    throw std::ios_base::failure(std::string("Truncated image: ") + path);
  if (img.owned && img.data) delete[] img.data;
  img.w = w;
  img.h = h;
  img.bpp = 4;  // always RGBA, like stbi_load(.., 4)
  img.data = new unsigned char[(size_t)w * h * 4];
  img.owned = true;
  for (size_t i = 0; i < (size_t)w * h; i++) {
    for (int c = 0; c < 3; c++) img.data[4 * i + c] = raw[channels * i + (channels == 3 ? c : 0)];
    img.data[4 * i + 3] = 255;
  }
}

int write_image(const char* path, ImageData& img) {
  std::ofstream f(path, std::ios::binary);
  if (!f.is_open()) return 0;
  f << "P6\n" << img.w << " " << img.h << "\n255\n";
  if (img.bpp == 3) {
    f.write(reinterpret_cast<const char*>(img.data), (std::streamsize)((size_t)img.w * img.h * 3));
  } else {
    for (size_t i = 0; i < (size_t)img.w * img.h; i++)
      f.write(reinterpret_cast<const char*>(img.data + (size_t)img.bpp * i), 3);
  }
  return f.good() ? 1 : 0;
}

void write_image(const char* path, float* luma, size_t w, size_t h) {
  std::ofstream f(path, std::ios::binary);
  if (!f.is_open()) throw std::ios_base::failure(std::string("Could not write image: ") + path);
  f << "P5\n" << w << " " << h << "\n255\n";
  for (size_t i = 0; i < w * h; i++) {
    float v = luma[i] * 255.0f;
    v = v < 0.f ? 0.f : (v > 255.f ? 255.f : v);
    f.put((char)(unsigned char)v);
  }
}

// ------------------------------------------------------------------ video (Y4M) ---------
static std::runtime_error y4m_error(const std::string& path, const std::string& what) {
  return std::runtime_error("Y4M '" + path + "': " + what);
}

// the colourspace tag (after 'C') and the XYSCSS= value of each SRCNN_CHROMA_* siting
static const char* const kY4mSiting[3] = {"420jpeg", "420mpeg2", "420paldv"};
static const char* const kY4mXyscss[3] = {"420JPEG", "420MPEG2", "420PALDV"};

Y4mReader::Y4mReader(const char* path, bool any_siting, bool ten_bit)
    : _path(path), _f(path, std::ios::binary) {
  if (!_f.is_open()) throw y4m_error(_path, "could not open");
  std::string line;
  if (!std::getline(_f, line) || line.compare(0, 10, "YUV4MPEG2 ") != 0)
    throw y4m_error(_path, "not a YUV4MPEG2 stream");
  std::istringstream tags(line.substr(10));
  std::string t;
  bool has_w = false, has_h = false;
  while (std::getline(tags, t, ' ')) {
    if (t.empty()) continue;
    const std::string v = t.substr(1);
    switch (t[0]) {
      case 'W':
      case 'H': {
        char* end = nullptr;
        const long n = std::strtol(v.c_str(), &end, 10);
        if (v.empty() || *end != '\0' || n <= 0 || n > 65535)
          throw y4m_error(_path, "bad frame size tag '" + t + "'");
        (t[0] == 'W' ? _header.w : _header.h) = (int)n;
        (t[0] == 'W' ? has_w : has_h) = true;
        break;
      }
      case 'C':
        if (v == "420mpeg2" || v == "420paldv") {
          if (!any_siting)
            throw y4m_error(_path, "chroma siting '" + t + "' is left-sited; only centre-sited 4:2:0 "
                                   "(C420jpeg, C420) is supported; --chroma-siting keep enlarges it "
                                   "at its own siting");
          _header.chroma_siting = v == "420mpeg2" ? SRCNN_CHROMA_LEFT : SRCNN_CHROMA_TOPLEFT;
        } else if (v == "420p10" && ten_bit) {
          _header.bit_depth = 10;
        } else if (v != "420jpeg" && v != "420")
          throw y4m_error(_path, "colourspace '" + t + "' is not supported; only 8-bit 4:2:0 "
                                 "(C420jpeg, C420) is" +
                                 (v == "420p10" ? "; --bit-depth 10 reads 10-bit 4:2:0" : ""));
        break;
      case 'I':
        if (v != "p")
          throw y4m_error(_path, "interlacing '" + t + "' is not supported; only progressive "
                                 "frames (Ip) are");
        break;
      case 'F':
      case 'A':
      case 'X':
        break;
      default:
        throw y4m_error(_path, "unknown header tag '" + t + "'");
    }
    _header.tags.push_back(t);
  }
  if (!has_w || !has_h) throw y4m_error(_path, "the header gives no W or no H");
  if (_header.w % 2 || _header.h % 2)
    throw y4m_error(_path, "frame size " + std::to_string(_header.w) + "x" +
                               std::to_string(_header.h) + " is odd; 4:2:0 needs even sizes");
  _first = _f.tellg();
}

// reads "FRAME[ params]\n"; false at the end of the stream
bool Y4mReader::read_marker(size_t frame) {
  if (_f.peek() == std::char_traits<char>::eof()) return false;
  std::string line;
  const bool full = (bool)std::getline(_f, line) && !_f.eof();
  if (line.compare(0, 5, "FRAME") != 0 || (line.size() > 5 && line[5] != ' '))
    throw y4m_error(_path, "frame " + std::to_string(frame) + " does not start with FRAME");
  if (!full) throw y4m_error(_path, "frame " + std::to_string(frame) + " is truncated");
  return true;
}

size_t Y4mReader::check_frames() {
  _f.clear();
  _f.seekg(0, std::ios::end);
  const std::streamoff size = _f.tellg();
  _f.seekg(_first);
  size_t n = 0;
  while (read_marker(n)) {
    if (size - (std::streamoff)_f.tellg() < (std::streamoff)_header.frame_bytes())
      throw y4m_error(_path, "frame " + std::to_string(n) + " is truncated");
    _f.seekg((std::streamoff)_header.frame_bytes(), std::ios::cur);
    n++;
  }
  _f.clear();
  _f.seekg(_first);
  _next = 0;
  return n;
}

size_t Y4mReader::read_frames(size_t max, std::vector<unsigned char>& out) {
  const size_t bytes = _header.frame_bytes();
  size_t n = 0;
  while (n < max && read_marker(_next)) {
    const size_t at = out.size();
    out.resize(at + bytes);
    _f.read(reinterpret_cast<char*>(out.data() + at), (std::streamsize)bytes);
    if ((size_t)_f.gcount() != bytes)
      throw y4m_error(_path, "frame " + std::to_string(_next) + " is truncated");
    n++;
    _next++;
  }
  return n;
}

void write_y4m_header(std::ostream& f, const Y4mHeader& in, int out_w, int out_h, int out_siting) {
  const bool resite = out_siting != in.chroma_siting;
  bool has_c = false;
  f << "YUV4MPEG2";
  for (const std::string& t : in.tags) {
    if (t[0] == 'W')
      f << " W" << out_w;
    else if (t[0] == 'H')
      f << " H" << out_h;
    else if (resite && t[0] == 'C')
      f << " C" << kY4mSiting[out_siting];
    else if (resite && t.compare(0, 7, "XYSCSS=") == 0)
      f << " XYSCSS=" << kY4mXyscss[out_siting];
    else
      f << " " << t;
    has_c = has_c || t[0] == 'C';
  }
  if (resite && !has_c) f << " C" << kY4mSiting[out_siting];
  f << "\n";
}

void write_y4m_frames(std::ostream& f, const unsigned char* frames, size_t n, size_t frame_bytes) {
  for (size_t i = 0; i < n; i++) {
    f << "FRAME\n";
    f.write(reinterpret_cast<const char*>(frames + i * frame_bytes), (std::streamsize)frame_bytes);
  }
}

}  // namespace utils

// ------------------------------------------------------------------ RawMemoryHandle ----
void RawMemoryHandle::release() {
  if (!released && context && mem != SRCNN_NULL_MEM) srcnn_release(context->c_ctx(), mem);
  released = true;
}

// ------------------------------------------------------------------ ProfiledLaunch -----
ProfiledLaunch::ProfiledLaunch(Kernel& k) : _k(k) {
  if (_k._context->is_running_profile_mode())
    srcnn_profile_get(_k._context->c_ctx(), _k._kernel_id, &_before, nullptr);
}
ProfiledLaunch::~ProfiledLaunch() {
  if (_k._context->is_running_profile_mode()) {
    uint64_t after = 0;
    srcnn_profile_get(_k._context->c_ctx(), _k._kernel_id, &after, nullptr);
    _k._execution_time_ns += after - _before;
  }
}

// ------------------------------------------------------------------ Context ------------
Context::Context() {}
Context::~Context() { cleanup(); }

// rank 0 publishes the 128-byte NCCL id through a file (written under a temporary name and
// renamed, so that readers never see a partial id); the other ranks poll for it
static void exchange_comm_id(int rank, const char* path, unsigned char id[SRCNN_COMM_ID_BYTES]) {
  if (rank == 0) {
    if (srcnn_comm_unique_id(id) != SRCNN_OK) throw std::runtime_error(srcnn_last_error());
    const std::string tmp = std::string(path) + ".tmp";
    {
      std::ofstream f(tmp, std::ios::binary);
      if (!f.is_open()) throw std::ios_base::failure("Could not write CNN_SR_COMM_FILE");
      f.write(reinterpret_cast<const char*>(id), SRCNN_COMM_ID_BYTES);
    }
    if (std::rename(tmp.c_str(), path) != 0)
      throw std::ios_base::failure("Could not publish CNN_SR_COMM_FILE");
    return;
  }
  for (int tries = 0; tries < 3000; tries++) {   // up to ~5 minutes
    std::ifstream f(path, std::ios::binary);
    if (f.is_open()) {
      f.read(reinterpret_cast<char*>(id), SRCNN_COMM_ID_BYTES);
      if (f.gcount() == SRCNN_COMM_ID_BYTES) return;
    }
    struct timespec ts = {0, 100 * 1000 * 1000};
    nanosleep(&ts, nullptr);
  }
  throw std::runtime_error("Timed out waiting for rank 0 to publish CNN_SR_COMM_FILE");
}

void Context::init(bool profile) {
  _profiling = profile;
  const char* world_env = std::getenv("CNN_SR_WORLD");
  const char* rank_env = std::getenv("CNN_SR_RANK");
  _world = world_env ? std::max(1, std::atoi(world_env)) : 1;
  _rank = rank_env ? std::atoi(rank_env) : 0;
  if (_rank < 0 || _rank >= _world) throw std::runtime_error("CNN_SR_RANK outside CNN_SR_WORLD");
  const char* dev_env = std::getenv("CNN_SR_DEVICE");
  const int device = dev_env ? std::atoi(dev_env) : _rank;
  const int rc = srcnn_ctx_create(device, profile ? 1 : 0, &_ctx);
  if (rc != SRCNN_OK) {
    std::cout << "[GPU ERROR] (" << rc << ") : " << srcnn_last_error() << std::endl;
    throw std::runtime_error(srcnn_last_error());
  }
  char name[256];
  int sms = 0;
  srcnn_device_info(_ctx, name, sizeof(name), &sms, &_device_mem);
  _device_name = name;
  std::cout << "PLATFORM: CUDA (sm_100a C-ABI layer)" << std::endl;
  std::cout << "DEVICE:" << name << ", " << sms << " SMs, " << (_device_mem >> 20) << " MB"
            << std::endl;
  _initialized = true;
  if (_world > 1) {
    const char* file = std::getenv("CNN_SR_COMM_FILE");
    if (!file) throw std::runtime_error("CNN_SR_WORLD > 1 needs CNN_SR_COMM_FILE (a path all ranks can reach)");
    unsigned char id[SRCNN_COMM_ID_BYTES];
    exchange_comm_id(_rank, file, id);
    check_status(srcnn_comm_init(_ctx, _rank, _world, id), "joining the communicator");
    std::cout << "DATA PARALLEL: rank " << _rank << " of " << _world << " (NCCL)" << std::endl;
  }
}

void Context::allreduce_sum(MemoryHandle h, size_t count) {
  check_status(srcnn_allreduce_sum(_ctx, mem(h), 0, count), "all-reduce");
}

float Context::allreduce_scalar(float value) {
  if (_world == 1) return value;
  if (_scalar_buf == ((MemoryHandle)1 << 30)) _scalar_buf = allocate(CL_MEM_READ_WRITE, sizeof(float));
  write_buffer(_scalar_buf, &value, true);
  allreduce_sum(_scalar_buf, 1);
  read_buffer(_scalar_buf, &value, true);
  return value;
}

void Context::cleanup() {
  if (!_initialized) return;
  _initialized = false;
  srcnn_block(_ctx);
  if (_profiling) {
    // same line format the reference prints (src/opencl/Context.cpp:88-96); profile.py parses it
    for (const Kernel& k : _kernels) {
      const unsigned long long t = k.get_total_execution_time();
      std::cout << "Kernel " << k.get_human_identifier() << " total execution time: " << t
                << "ns = " << (t / 1000000000.0) << "s" << std::endl;
    }
  }
  srcnn_ctx_destroy(_ctx);
  _ctx = nullptr;
}

void Context::check_error(bool ok, char const* msg) {
  if (ok) return;
  std::cout << "[GPU ERROR] (-100) : " << msg << std::endl;
  cleanup();
  throw std::runtime_error(msg);
}

void Context::check_status(int status, char const* what) {
  if (status == SRCNN_OK) return;
  const std::string detail = srcnn_last_error();
  std::cout << "[GPU ERROR] (" << status << ") : " << what << ": " << detail << std::endl;
  throw std::runtime_error(detail.empty() ? what : detail);
}

void Context::print_app_memory_usage() {
  size_t image_memory = 0, buffer_memory = 0;
  for (const RawMemoryHandle& m : _allocations) {
    if (!m.is_usable()) continue;
    (m.is_image() ? image_memory : buffer_memory) += m.size;
  }
  const size_t unit = 1024 * 1024;
  std::cout << "Memory usage: " << (image_memory + buffer_memory) / unit << "/"
            << _device_mem / unit << " MB ("
            << (image_memory + buffer_memory) * 100.0 / (double)_device_mem << "%), "
            << buffer_memory / unit << "MB of raw buffers and " << image_memory / unit
            << "MB for images" << std::endl;
}

void Context::block() {
  if (cnn_sr_warn_blocking()) std::cout << "BLOCK explicit Context::block()" << std::endl;
  check_status(srcnn_block(_ctx), "Context::block()");
}

MemoryHandle Context::allocate(cl_mem_flags_t, size_t bytes) {
  check_error(_initialized, "Context was not initialized");
  srcnn_mem m = SRCNN_NULL_MEM;
  check_status(srcnn_alloc(_ctx, bytes, &m), "Context::allocate");
  RawMemoryHandle h;
  h.context = this;
  h.mem = m;
  h.size = bytes;
  _allocations.push_back(h);
  return _allocations.size() - 1;
}

RawMemoryHandle* Context::raw_memory(MemoryHandle handle) {
  check_error(handle < _allocations.size(),
              "Invalid memory handle.Could not get RawMemoryHandle object");
  return &_allocations[handle];
}

srcnn_mem Context::mem(MemoryHandle handle) {
  RawMemoryHandle* r = raw_memory(handle);
  check_error(r->is_usable(), "Memory handle was already released");
  return r->mem;
}

Event Context::ticket() {
  Event e;
  e.context = this;
  e.ticket = ++_ticket;
  return e;
}

void Context::wait(const Event&) { check_status(srcnn_block(_ctx), "wait for event"); }

void wait_for_events(int count, Event* events) {
  for (int i = 0; i < count; i++)
    if (events[i].context) events[i].context->wait(events[i]);
}

static bool parse_macro(const std::string& opts, const char* name, size_t* value) {
  const std::string key = std::string("-D ") + name;
  size_t pos = opts.find(key);
  while (pos != std::string::npos) {
    const size_t end = pos + key.size();
    if (end == opts.size() || opts[end] == ' ') {  // flag macro
      if (value) *value = 1;
      return true;
    }
    if (opts[end] == '=') {
      if (value) *value = (size_t)std::strtoull(opts.c_str() + end + 1, nullptr, 10);
      return true;
    }
    pos = opts.find(key, end);
  }
  return false;
}

Kernel* Context::create_kernel(char const* file_path, char const* cmp_opt, char const* main_f) {
  check_error(_initialized, "Context was not initialized");
  struct Entry {
    const char* name;
    Kernel::Kind kind;
    int id;
  };
  static const Entry entries[] = {
      {"forward", Kernel::Kind::Forward, SRCNN_K_FORWARD},
      {"squared_err", Kernel::Kind::SquaredErr, SRCNN_K_SQUARED_ERR},
      {"last_layer_delta", Kernel::Kind::LastLayerDelta, SRCNN_K_LAST_LAYER_DELTA},
      {"deltas", Kernel::Kind::Deltas, SRCNN_K_DELTAS},
      {"backpropagate", Kernel::Kind::Backpropagate, SRCNN_K_BACKPROPAGATE},
      {"update_params", Kernel::Kind::UpdateParams, SRCNN_K_UPDATE_PARAMS},
      {"sum", Kernel::Kind::Sum, SRCNN_K_SUM},
      {"sub_from_all", Kernel::Kind::SubFromAll, SRCNN_K_SUB_FROM_ALL},
      {"extract_luma", Kernel::Kind::ExtractLuma, SRCNN_K_EXTRACT_LUMA},
      {"swap_luma", Kernel::Kind::SwapLuma, SRCNN_K_SWAP_LUMA},
      {"resample", Kernel::Kind::Resample, SRCNN_K_RESAMPLE},
  };
  const Entry* found = nullptr;
  for (const Entry& e : entries)
    if (std::strcmp(e.name, main_f) == 0) found = &e;
  if (!found) {
    std::string msg = std::string("Unknown kernel entry point '") + main_f + "' (" +
                      (file_path ? file_path : "??") + ")";
    check_error(false, msg.c_str());
  }
  Kernel k;
  k._kind = found->kind;
  k._kernel_id = found->id;
  k._context = this;
  const std::string opts = cmp_opt ? cmp_opt : "";
  parse_macro(opts, "CURRENT_FILTER_COUNT", &k.current_filter_count);
  parse_macro(opts, "PREVIOUS_FILTER_COUNT", &k.previous_filter_count);
  parse_macro(opts, "F_SPATIAL_SIZE", &k.f_spatial_size);
  k.skip_relu = parse_macro(opts, "SKIP_RELU", nullptr);
  k.normalize = parse_macro(opts, "NORMALIZE", nullptr);
  k.sum_squared = parse_macro(opts, "SUM_SQUARED", nullptr);
  k._identifier = std::string("'") + (file_path ? file_path : "??") + "'[" +
                  (cmp_opt ? cmp_opt : "--") + "]";
  _kernels.push_back(k);
  return &_kernels.back();
}

Event Context::read_buffer(MemoryHandle h, size_t offset, size_t size, void* dst, bool block,
                           Event*, int) {
  if (cnn_sr_warn_blocking() && block) std::cout << "BLOCK: read_buffer" << std::endl;
  check_error(_initialized, "Context was not initialized");
  check_error(size <= raw_memory(h)->size, "Tried to read more then is allocated");
  check_status(srcnn_read(_ctx, mem(h), offset, size, dst, block ? 1 : 0), "Error in read buffer");
  return ticket();
}

Event Context::read_buffer(MemoryHandle h, void* dst, bool block, Event* es, int n) {
  return read_buffer(h, 0, raw_memory(h)->size, dst, block, es, n);
}

Event Context::write_buffer(MemoryHandle h, size_t offset, size_t size, void* src, bool block,
                            Event*, int) {
  if (cnn_sr_warn_blocking() && block) std::cout << "BLOCK: write_buffer" << std::endl;
  check_error(_initialized, "Context was not initialized");
  check_error(size <= raw_memory(h)->size, "Tried to write more then is allocated");
  check_status(srcnn_write(_ctx, mem(h), offset, size, src, block ? 1 : 0),
               "Error in write buffer");
  return ticket();
}

Event Context::write_buffer(MemoryHandle h, void* src, bool block, Event* es, int n) {
  return write_buffer(h, 0, raw_memory(h)->size, src, block, es, n);
}

Event Context::zeros_float(MemoryHandle h, bool block, Event* es, int n) {
  return fill_float(h, 0.0f, block, es, n);
}

Event Context::fill_float(MemoryHandle h, float v, bool block, Event*, int) {
  // the reference uploads a host vector of `v` (Context.cpp:301-310); here it is a device fill
  check_status(srcnn_fill_float(_ctx, mem(h), v), "Error in fill_float");
  if (block) this->block();
  return ticket();
}

Event Context::copy_buffer(MemoryHandle src, MemoryHandle dst, Event* es, int n) {
  check_error(raw_memory(src)->size == raw_memory(dst)->size,
              "When performing buffer copy, both buffers should have equal length");
  return copy_buffer(src, dst, 0, es, n);
}

Event Context::copy_buffer(MemoryHandle src, MemoryHandle dst, size_t dst_offset, Event*, int) {
  check_error(_initialized, "Context was not initialized");
  check_error(raw_memory(src)->size + dst_offset <= raw_memory(dst)->size,
              "When performing buffer copy, would write after dst end");
  check_status(srcnn_copy(_ctx, mem(src), mem(dst), dst_offset), "Error in copy buffer");
  return ticket();
}

MemoryHandle Context::create_image(cl_mem_flags_t flags, int, int, size_t w, size_t h) {
  const MemoryHandle idx = allocate(flags, w * h * 4);
  _allocations[idx].bpp = 4;
  return idx;
}

Event Context::write_image(MemoryHandle h, utils::ImageData& data, bool block, Event*, int) {
  RawMemoryHandle* r = raw_memory(h);
  const size_t bytes = (size_t)data.w * data.h * r->bpp;
  check_error(data.bpp == (int)r->bpp, "Image has a different pixel format than the gpu image");
  check_error(bytes <= r->size, "Tried to write more then is allocated");
  check_status(srcnn_write(_ctx, mem(h), 0, bytes, data.data, block ? 1 : 0),
               "Error in write_image");
  return ticket();
}

}  // namespace gpu

std::ostream& operator<<(std::ostream& os, const gpu::Kernel& k) {
  os << "Kernel " << k.get_human_identifier();
  return os;
}
