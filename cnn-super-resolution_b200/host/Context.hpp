// C++ face of the CUDA device layer: the drop-in for the reference's opencl::Context /
// opencl::Kernel / opencl::utils (src/opencl/Context.hpp:72-299, Kernel.hpp:15-95,
// UtilsOpenCL.hpp:27-87).  Everything here is a thin wrapper over the C-ABI of
// include/srcnn_b200.h: status codes become std::runtime_error, like check_error does in the
// reference (src/opencl/Context.cpp:111-123).
//
// `namespace opencl` is an alias of `namespace gpu`, and cl_event / CL_MEM_* are provided, so
// code written against the reference's host API (Main_cl.cpp, the test specs) keeps compiling.
#ifndef CNN_SR_GPU_CONTEXT_H
#define CNN_SR_GPU_CONTEXT_H

#include <cstddef>
#include <cstdint>
#include <deque>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "../../include/srcnn_b200.h"
#include "pch.hpp"

inline bool cnn_sr_warn_blocking() { return cnn_sr::warn_about_blocking_operation; }

namespace gpu {

class Context;
typedef size_t MemoryHandle;

/** Stand-in for cl_event.  The context has ONE in-order stream, so an event is just the
 * ticket number of the enqueued operation; waiting on it drains the stream. */
struct Event {
  Context* context = nullptr;
  uint64_t ticket = 0;
};

typedef int cl_mem_flags_t;

namespace utils {
/** decoded image, RGBA8 when loaded with 4 channels (reference: UtilsOpenCL.hpp:27-38) */
struct ImageData {
  ImageData();
  ImageData(int w, int h, int bpp, unsigned char* data);  // borrows `data`
  ~ImageData();
  ImageData(const ImageData&) = delete;
  ImageData& operator=(const ImageData&) = delete;
  int w, h;
  int bpp;  // bytes per pixel
  unsigned char* data;

 private:
  bool owned = false;
  friend void load_image(const char*, ImageData&);
};
/** Binary PPM (P6) / PGM (P5) in, always expanded to RGBA8.  The reference decodes JPEG/PNG
 * with the vendored stb_image; the codecs are outside the hot path (SURVEY 2.1 #11) --
 * tools/img2ppm.py converts other formats. */
void load_image(const char* path, ImageData&);
/** 3-channel RGB8 -> binary PPM; returns non-zero on success like stbi_write_png */
int write_image(const char* path, ImageData&);
/** luma in [0,1] -> 8-bit binary PGM (reference: UtilsOpenCL.cpp write_image(float*)) */
void write_image(const char* path, float* luma, size_t w, size_t h);

/** The header of a YUV4MPEG2 (Y4M) stream: "YUV4MPEG2" and space-separated tags.  Only
 * progressive 4:2:0 of even size is accepted: 8-bit, or 10-bit (C420p10, ffmpeg's yuv420p10le:
 * a little-endian 16-bit word a sample) when asked for.  Its chroma siting is read as ffmpeg's
 * reader maps the colourspace tag: C420jpeg (the format's default), C420 and C420p10 centre-sited,
 * C420mpeg2 left-sited, C420paldv top-left-sited. */
struct Y4mHeader {
  int w = 0, h = 0;
  int chroma_siting = SRCNN_CHROMA_CENTER;   // SRCNN_CHROMA_*
  int bit_depth = 8;                         // 8, or 10 for C420p10
  std::vector<std::string> tags;   // every tag as read, in order ("W960", "F30000:1001", ...)
  size_t frame_bytes() const { return (size_t)w * h * 3 / 2 * (bit_depth == 10 ? 2 : 1); }
};
/** Reads the frames of a Y4M file.  Every check throws std::runtime_error with a one-line
 * message: the constructor checks the header, check_frames() every frame marker and frame size. */
class Y4mReader {
 public:
  /** any_siting: accept chroma that is not centre-sited; ten_bit: accept C420p10 (each refused
   * otherwise) */
  explicit Y4mReader(const char* path, bool any_siting = false, bool ten_bit = false);
  const Y4mHeader& header() const { return _header; }
  /** the number of frames; every frame starts with "FRAME[ params]\n" and is complete.  Leaves
   * the reader at the first frame. */
  size_t check_frames();
  /** up to `max` next frames (I420 or I010 bytes, their parameters dropped) into `out`; returns
   * how many */
  size_t read_frames(size_t max, std::vector<unsigned char>& out);

 private:
  bool read_marker(size_t frame);
  std::string _path;
  std::ifstream _f;
  std::streampos _first;
  size_t _next = 0;
  Y4mHeader _header;
};
/** `in`'s header with W and H set to out_w x out_h and every other tag copied; for an out_siting
 * (SRCNN_CHROMA_*) other than in's, the C tag names it (appended when `in` has none) and an
 * XYSCSS= tag matches it */
void write_y4m_header(std::ostream&, const Y4mHeader& in, int out_w, int out_h, int out_siting);
/** n frames of `frame_bytes` bytes, each behind a bare "FRAME\n" (10-bit frames as the
 * little-endian words of a little-endian host, as they were read) */
void write_y4m_frames(std::ostream&, const unsigned char* frames, size_t n, size_t frame_bytes);
}  // namespace utils

/** One allocation of the context (reference: RawMemoryHandle, Context.hpp:53-66) */
struct RawMemoryHandle {
  void release();
  bool is_usable() const { return !released; }
  bool is_image() const { return bpp != 0; }
  size_t size = 0;
  size_t bpp = 0;

 private:
  friend class Context;
  Context* context = nullptr;
  srcnn_mem mem = SRCNN_NULL_MEM;
  bool released = false;
};

/**
 * A launchable kernel *descriptor*: which entry point, which compile-time specialisation.
 * The reference JIT-compiles a .cl file with "-D" macros per Kernel object
 * (src/opencl/Context.cpp:178-230); here the CUDA kernels are precompiled and the macros only
 * select / validate the specialisation.  Keeps per-object execution time for `profile` mode.
 */
class Kernel {
 public:
  enum class Kind {
    Forward, SquaredErr, LastLayerDelta, Deltas, Backpropagate, UpdateParams, Sum, SubFromAll,
    ExtractLuma, SwapLuma, Resample
  };
  Kind kind() const { return _kind; }
  Context* get_context() const { return _context; }
  size_t get_max_work_group_size() const { return 1024; }
  unsigned long long get_total_execution_time() const { return _execution_time_ns; }
  const char* get_human_identifier() const { return _identifier.c_str(); }
  // "-D" macros (0 / false when absent)
  size_t current_filter_count = 0, previous_filter_count = 0, f_spatial_size = 0;
  bool skip_relu = false, normalize = false, sum_squared = false;

 private:
  friend class Context;
  friend class ProfiledLaunch;
  Kind _kind = Kind::Forward;
  Context* _context = nullptr;
  int _kernel_id = 0;
  unsigned long long _execution_time_ns = 0;
  std::string _identifier;
};

/** Brackets one launch: adds the device time the C-ABI measured to the Kernel object. */
class ProfiledLaunch {
 public:
  explicit ProfiledLaunch(Kernel& k);
  ~ProfiledLaunch();

 private:
  Kernel& _k;
  uint64_t _before = 0;
};

class Context {
 public:
  Context();
  ~Context();
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;

  /** picks CUDA device `CNN_SR_DEVICE` (default 0), one in-order stream.  `profile` times
   * every launch and blocks on it (reference: Context::init, Context.cpp:45-79) */
  void init(bool profile = false);
  void check_error(bool ok, char const* msg);
  /** throws when a C-ABI call returned non-zero, after printing "[GPU ERROR] ..." */
  void check_status(int status, char const* what);
  void print_app_memory_usage();

  void block();
  MemoryHandle allocate(cl_mem_flags_t flags, size_t bytes);
  Kernel* create_kernel(char const* file_path, char const* cmp_opt = nullptr,
                        char const* main_f = "main");

  Event read_buffer(MemoryHandle, size_t offset, size_t size, void* dst, bool block,
                    Event* es = nullptr, int event_count = 0);
  Event read_buffer(MemoryHandle, void* dst, bool block, Event* es = nullptr,
                    int event_count = 0);
  Event write_buffer(MemoryHandle, size_t offset, size_t size, void* src, bool block,
                     Event* es = nullptr, int event_count = 0);
  Event write_buffer(MemoryHandle, void* src, bool block, Event* es = nullptr,
                     int event_count = 0);
  Event zeros_float(MemoryHandle, bool block, Event* es = nullptr, int event_count = 0);
  Event fill_float(MemoryHandle, float, bool block, Event* es = nullptr, int event_count = 0);
  Event copy_buffer(MemoryHandle src, MemoryHandle dst, Event* es = nullptr,
                    int event_count = 0);
  Event copy_buffer(MemoryHandle src, MemoryHandle dst, size_t dst_offset, Event* es = nullptr,
                    int event_count = 0);
  /** RGBA8 "image" = a w*h*4 byte buffer (the CUDA kernels index it directly) */
  MemoryHandle create_image(cl_mem_flags_t, int channel_order, int channel_type, size_t w,
                            size_t h);
  Event write_image(MemoryHandle, utils::ImageData&, bool block, Event* es = nullptr,
                    int event_count = 0);

  // --- data parallel (new; the reference is single-device) ----------------------------
  /** rank / world of this process: CNN_SR_RANK / CNN_SR_WORLD in the environment of init().
   * With CNN_SR_WORLD > 1 init() joins the NCCL communicator of the device layer; the id is
   * handed over through the file CNN_SR_COMM_FILE (rank 0 writes it, the others wait for it). */
  int rank() const { return _rank; }
  int world() const { return _world; }
  /** in-place sum over all ranks of the first `count` floats of the buffer (no-op on 1 rank) */
  void allreduce_sum(MemoryHandle, size_t count);
  /** sum of one host float over all ranks (validation squared error) */
  float allreduce_scalar(float value);

  bool is_initialized() const { return _initialized; }
  bool is_running_profile_mode() const { return _profiling; }
  RawMemoryHandle* raw_memory(MemoryHandle);
  std::string device_name() const { return _device_name; }

  // --- used by DataPipeline -----------------------------------------------------------
  srcnn_ctx* c_ctx() { return _ctx; }
  /** C-ABI handle behind a MemoryHandle; throws on an invalid / released handle */
  srcnn_mem mem(MemoryHandle);
  Event ticket();
  void wait(const Event&);

 private:
  void cleanup();
  bool _initialized = false;
  bool _profiling = false;
  srcnn_ctx* _ctx = nullptr;
  uint64_t _ticket = 0;
  int _rank = 0, _world = 1;
  MemoryHandle _scalar_buf = (MemoryHandle)1 << 30;
  std::string _device_name;
  size_t _device_mem = 0;
  std::deque<Kernel> _kernels;               // stable addresses
  std::deque<RawMemoryHandle> _allocations;  // stable addresses
};

/** clWaitForEvents */
void wait_for_events(int count, Event* events);

}  // namespace gpu

// ---- names the reference's callers use ---------------------------------------------------
namespace opencl = gpu;
typedef gpu::Event cl_event;
typedef float cl_float;
typedef unsigned int cl_uint;
typedef unsigned char cl_char;
enum {
  CL_MEM_READ_WRITE = 1, CL_MEM_WRITE_ONLY = 2, CL_MEM_READ_ONLY = 4,
  CL_RGBA = 0x10B5, CL_UNSIGNED_INT8 = 0x10DA
};
inline void clWaitForEvents(int n, cl_event* e) { gpu::wait_for_events(n, e); }

std::ostream& operator<<(std::ostream&, const gpu::Kernel&);

#endif
