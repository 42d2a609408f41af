// `cnn [train | eval] [dry] [profile] --config CFG --in PATH [--out PATH] [--epochs N]
//      [--scale N [--resample lanczos|bicubic]] [--chroma-siting keep|420jpeg|420mpeg2|420paldv]
//      [--bit-depth 8|10]`
// Same grammar, flow and console output as the reference CLI (src/Main_cl.cpp:40-318):
// forward mode = one image through the three layers, luma swapped back into the image (or every
// image of a directory, see below);
// training mode = samples `*_large.*` (ground truth) / `*_small.*` (input) from a directory,
// 80/20 train/validation split re-drawn every epoch, ONE parameter update per epoch.
// --scale N (forward mode, N >= 2) first enlarges the input N times with Pillow's filter (Lanczos by
// default, as the reference's sample generator did; bicubic is Pillow's and the SRCNN paper's
// default), all on the device (srcnn_upscale_image_host); N = 1 is the plain forward mode.
// -i DIR (forward mode) runs every `.ppm` / `.pgm` file of DIR, in sorted name order, into
// OUT_DIR/<stem>.ppm (-o OUT_DIR): consecutive files of equal size go through
// srcnn_upscale_frames_host together, at most kDirBatch at a time; other files are skipped.
// -i IN.y4m (forward mode) enlarges every frame of a YUV4MPEG2 video, 8-bit progressive 4:2:0 with
// centre-sited chroma (C420jpeg / C420), into OUT.y4m (-o OUT.y4m): the header's W and H times
// --scale, its other tags copied, kDirBatch frames per srcnn_upscale_yuv420_frames_host_sited call;
// the network replaces the luma, the chroma is only enlarged.  The header and every frame marker are
// checked before any device work.  Left- and top-left-sited chroma (C420mpeg2, C420paldv) is refused
// unless --chroma-siting names the output's siting: `keep` (the input's, every tag copied) or a
// colourspace tag, to which the chroma is converted (the C tag, and an XYSCSS= tag, then name it).
// 10-bit video (C420p10, ffmpeg's yuv420p10le; centre-sited) is refused unless --bit-depth 10 asks
// for it, and then goes through srcnn_upscale_yuv420p10_frames_host; --bit-depth 10 needs a
// C420p10 header, and its output is centre-sited (--chroma-siting keep or 420jpeg), because a
// C420p10 tag cannot state another siting.
// eval -i SAMPLES_DIR measures the network on the training mode's sample pairs: every `_small`
// image, enlarged N times (--scale, default 1: the reference's `_small` images are already
// enlarged), against its `_large` image, which must be exactly N times its size.  One line a pair
// (PSNR / SSIM of the network's result and of the plain enlargement, and the PSNR gain), then
// their means; -o OUT_DIR also writes OUT_DIR/<name>.ppm (srcnn_evaluate_frames_host).
// Images are binary PPM/PGM (see Context.hpp); `_large.ppm/_small.ppm` as well as the
// reference's `.jpg` suffix pattern are recognised by name.
#include <sys/stat.h>

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <memory>
#include <random>
#include <stdexcept>
#include <unordered_map>
#include <utility>

#include "Config.hpp"
#include "ConfigBasedDataPipeline.hpp"
#include "Context.hpp"
#include "LayerData.hpp"
#include "pch.hpp"

using namespace opencl::utils;
using namespace cnn_sr;

typedef std::pair<std::string, std::string> TrainSampleFiles;  // (large, small)

static cl_event prepare_image(DataPipeline* pipeline, const char* file_path, ImageData& img,
                              opencl::MemoryHandle& gpu_data, opencl::MemoryHandle& gpu_luma) {
  load_image(file_path, img);
  return pipeline->extract_luma(img, gpu_data, gpu_luma, /*normalize=*/true);
}

static void execute_forward(ConfigBasedDataPipeline& pipeline, GpuAllocationPool& gpu_alloc,
                            const char* in_path, const char* out_path) {
  opencl::Context* context = pipeline.context();
  ImageData input_img;
  SampleAllocationPool sample;
  cl_event ev = prepare_image(&pipeline, in_path, input_img, sample.input_data, sample.input_luma);
  pipeline.subtract_mean(sample.input_luma, nullptr, &ev);  // (quirk Q1 applies)
  sample.input_w = (size_t)input_img.w;
  sample.input_h = (size_t)input_img.h;
  context->block();
  pipeline.forward(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, sample);
  if (out_path) pipeline.write_result_image(out_path, input_img, sample);
}

static void execute_upscale(ConfigBasedDataPipeline& pipeline, GpuAllocationPool& gpu_alloc,
                            const char* in_path, const char* out_path, size_t scale, int filter) {
  ImageData input_img;
  load_image(in_path, input_img);
  const size_t out_w = scale * (size_t)input_img.w, out_h = scale * (size_t)input_img.h;
  std::vector<unsigned char> result(out_w * out_h * 3);
  ImageData res_img((int)out_w, (int)out_h, 3, result.data());
  pipeline.upscale_image(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, input_img, out_w,
                         out_h, filter, res_img);
  if (out_path) {
    std::cout << "Saving result image to: '" << out_path << "'" << std::endl;
    write_image(out_path, res_img);
  }
}

// --scale: a whole number >= 1
static bool parse_scale(const char* text, size_t* scale) {
  if (!text) return true;
  char* end = nullptr;
  errno = 0;
  const long v = std::strtol(text, &end, 10);
  if (end == text || *end != '\0' || errno != 0 || v < 1 || v > 65535) return false;
  *scale = (size_t)v;
  return true;
}

static bool ends_with(const std::string& s, const std::string& suffix, size_t* stem_len) {
  if (s.size() < suffix.size() || s.compare(s.size() - suffix.size(), suffix.size(), suffix) != 0)
    return false;
  *stem_len = s.size() - suffix.size();
  return true;
}

static bool is_directory(const char* path) {
  struct stat st;
  return path && stat(path, &st) == 0 && S_ISDIR(st.st_mode);
}

// frames per srcnn_upscale_frames_host call in directory mode: bounds the host memory a batch
// holds (its input RGBA8 and its result RGB8; 64 frames of 960x540 -> 1920x1080: 531 MB)
static const size_t kDirBatch = 64;

struct DirImage {
  std::string path, stem;
};

// the `.ppm` / `.pgm` files of `dir`, in sorted name order; the others are skipped with a message
static std::vector<DirImage> get_directory_images(const std::string& dir) {
  std::vector<std::string> files;
  cnn_sr::utils::list_files(dir.c_str(), files);
  std::sort(files.begin(), files.end());
  std::vector<DirImage> images;
  for (const std::string& f : files) {
    size_t stem = 0;
    if (ends_with(f, ".ppm", &stem) || ends_with(f, ".pgm", &stem)) {
      if (is_directory((dir + "/" + f).c_str()))
        std::cout << "'" << f << "' is a directory. Skipping" << std::endl;
      else
        images.push_back({dir + "/" + f, f.substr(0, stem)});
    } else if (f != "." && f != "..") {
      std::cout << "'" << f << "' is not a .ppm/.pgm image. Skipping" << std::endl;
    }
  }
  return images;
}

// every image of the directory through the frames entry, `scale` times enlarged (1: at its own
// size); results go to out_dir/<stem>.ppm unless out_dir is null (dry run)
static void execute_directory(ConfigBasedDataPipeline& pipeline, GpuAllocationPool& gpu_alloc,
                              const std::vector<DirImage>& images, const char* out_dir,
                              size_t scale, int filter) {
  std::vector<unsigned char> in, out;
  std::vector<const DirImage*> batch;
  size_t w = 0, h = 0;
  auto flush = [&]() {
    if (batch.empty()) return;
    const size_t out_w = scale * w, out_h = scale * h, out_bytes = out_w * out_h * 3;
    out.resize(batch.size() * out_bytes);
    pipeline.upscale_frames(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, in.data(), w,
                            h, batch.size(), out_w, out_h, filter, out.data());
    for (size_t i = 0; i < batch.size() && out_dir; i++) {
      const std::string path = std::string(out_dir) + "/" + batch[i]->stem + ".ppm";
      std::cout << "Saving result image to: '" << path << "'" << std::endl;
      ImageData res_img((int)out_w, (int)out_h, 3, out.data() + i * out_bytes);
      if (!write_image(path.c_str(), res_img))
        throw std::runtime_error("Could not write image: " + path);
    }
    batch.clear();
    in.clear();
  };
  for (const DirImage& image : images) {
    ImageData img;
    load_image(image.path.c_str(), img);
    if (!batch.empty() && ((size_t)img.w != w || (size_t)img.h != h || batch.size() == kDirBatch))
      flush();
    w = (size_t)img.w;
    h = (size_t)img.h;
    in.insert(in.end(), img.data, img.data + w * h * 4);
    batch.push_back(&image);
  }
  flush();
}

// every frame of a Y4M video through the I420 (10-bit: I010) frames entry, `scale` times enlarged,
// kDirBatch frames at a time; the result goes to out_path unless it is null (dry run)
static void execute_y4m(ConfigBasedDataPipeline& pipeline, GpuAllocationPool& gpu_alloc,
                        Y4mReader& video, const char* out_path, size_t scale, int filter,
                        int out_siting) {
  const Y4mHeader& hd = video.header();
  const size_t w = (size_t)hd.w, h = (size_t)hd.h, out_w = scale * w, out_h = scale * h;
  const bool ten = hd.bit_depth == 10;
  const size_t out_bytes = out_w * out_h * 3 / 2 * (ten ? 2 : 1);
  std::ofstream out;
  if (out_path) {
    std::cout << "Saving result video to: '" << out_path << "'" << std::endl;
    out.open(out_path, std::ios::binary);
    if (!out.is_open()) throw std::runtime_error(std::string("Could not write video: ") + out_path);
    write_y4m_header(out, hd, (int)out_w, (int)out_h, out_siting);
  }
  std::vector<unsigned char> in, result;
  size_t n;
  while ((n = video.read_frames(kDirBatch, in)) > 0) {
    result.resize(n * out_bytes);
    // a 10-bit frame's bytes are its little-endian words; vector storage is aligned for them
    if (ten)
      pipeline.upscale_yuv420p10_frames(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3,
                                        reinterpret_cast<const uint16_t*>(in.data()), w, h, n,
                                        out_w, out_h, filter,
                                        reinterpret_cast<uint16_t*>(result.data()),
                                        hd.chroma_siting, out_siting);
    else
      pipeline.upscale_yuv420_frames(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3,
                                     in.data(), w, h, n, out_w, out_h, filter, result.data(),
                                     hd.chroma_siting, out_siting);
    if (out_path) write_y4m_frames(out, result.data(), n, out_bytes);
    in.clear();
  }
  if (out_path && !out.good()) throw std::runtime_error(std::string("Could not write video: ") + out_path);
}

static void get_training_samples(const std::string& dir, std::vector<TrainSampleFiles>& target) {
  std::vector<std::string> files;
  cnn_sr::utils::list_files(dir.c_str(), files);
  std::sort(files.begin(), files.end());  // deterministic order (readdir's is not)
  std::unordered_map<std::string, TrainSampleFiles> by_base;
  std::vector<std::string> order;
  for (const std::string& f : files) {
    size_t stem = 0;
    bool large = false, small = false;
    for (const char* ext : {".ppm", ".pgm", ".jpg"}) {
      if (ends_with(f, std::string("_large") + ext, &stem)) large = true;
      else if (ends_with(f, std::string("_small") + ext, &stem)) small = true;
      if (large || small) break;
    }
    if (!large && !small) {
      if (f != "." && f != "..")
        std::cout << "'" << f << "' is not a sample image. Skipping sample" << std::endl;
      continue;
    }
    const std::string base = f.substr(0, stem);
    if (!by_base.count(base)) order.push_back(base);
    (large ? by_base[base].first : by_base[base].second) = dir + "/" + f;
  }
  for (const std::string& base : order) {
    const TrainSampleFiles& p = by_base[base];
    if (p.first.empty() || p.second.empty())
      std::cout << "Only 1 image for pair with name '" << base << "'. Skipping sample" << std::endl;
    else
      target.push_back(p);
  }
}

// PSNR for data range 1 (+inf for identical images)
static double psnr_db(double mse) { return mse > 0.0 ? 10.0 * std::log10(1.0 / mse) : INFINITY; }

static std::string quality_line(double net_mse, double net_ssim, double base_mse, double base_ssim) {
  char buf[256];
  const double net = psnr_db(net_mse), base = psnr_db(base_mse);
  std::snprintf(buf, sizeof(buf),
                "network PSNR %.4f dB SSIM %.6f | baseline PSNR %.4f dB SSIM %.6f | gain %.4f dB",
                net, net_ssim, base, base_ssim, net - base);
  return buf;
}

// `eval`: every sample pair through the evaluate entry, consecutive pairs of equal size together
// (at most kDirBatch); per pair and mean PSNR / SSIM lines, results to out_dir/<name>.ppm unless
// out_dir is null (dry run)
static void execute_eval(ConfigBasedDataPipeline& pipeline, GpuAllocationPool& gpu_alloc,
                         const std::vector<TrainSampleFiles>& files, const char* out_dir,
                         size_t scale, int filter) {
  const int border = (int)pipeline.config()->total_padding() / 2;
  std::vector<unsigned char> in, ref, out;
  std::vector<double> metrics;
  std::vector<std::string> batch;
  double sum[5] = {};
  size_t n_done = 0, w = 0, h = 0;
  auto flush = [&]() {
    if (batch.empty()) return;
    const size_t out_w = scale * w, out_h = scale * h, out_bytes = out_w * out_h * 3;
    out.resize(batch.size() * out_bytes);
    metrics.resize(batch.size() * 4);
    pipeline.evaluate_frames(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3, in.data(), w,
                             h, batch.size(), out_w, out_h, filter, ref.data(), border, out.data(),
                             metrics.data());
    for (size_t i = 0; i < batch.size(); i++) {
      const double* m = metrics.data() + 4 * i;
      std::cout << batch[i] << ": " << quality_line(m[0], m[1], m[2], m[3]) << std::endl;
      const double v[5] = {psnr_db(m[0]), m[1], psnr_db(m[2]), m[3], psnr_db(m[0]) - psnr_db(m[2])};
      for (int k = 0; k < 5; k++) sum[k] += v[k];
      n_done++;
      if (!out_dir) continue;
      const std::string path = std::string(out_dir) + "/" + batch[i] + ".ppm";
      std::cout << "Saving result image to: '" << path << "'" << std::endl;
      ImageData res_img((int)out_w, (int)out_h, 3, out.data() + i * out_bytes);
      if (!write_image(path.c_str(), res_img))
        throw std::runtime_error("Could not write image: " + path);
    }
    batch.clear();
    in.clear();
    ref.clear();
  };
  for (const TrainSampleFiles& pair : files) {
    // the pair's name: the file name of its small image before "_small"
    const size_t slash = pair.second.find_last_of('/');
    std::string name = pair.second.substr(slash == std::string::npos ? 0 : slash + 1);
    name = name.substr(0, name.rfind("_small"));
    ImageData small, large;
    load_image(pair.second.c_str(), small);
    load_image(pair.first.c_str(), large);
    if ((size_t)large.w != scale * small.w || (size_t)large.h != scale * small.h) {
      std::cout << "'" << name << "': reference is " << large.w << "x" << large.h << ", not " << scale
                << " x " << small.w << "x" << small.h << ". Skipping sample" << std::endl;
      continue;
    }
    if (large.w - 2 * border < 11 || large.h - 2 * border < 11) {
      std::cout << "'" << name << "': " << large.w << "x" << large.h
                << " leaves less than 11x11 pixels inside the border of " << border
                << ". Skipping sample" << std::endl;
      continue;
    }
    if (!batch.empty() && ((size_t)small.w != w || (size_t)small.h != h || batch.size() == kDirBatch))
      flush();
    w = (size_t)small.w;
    h = (size_t)small.h;
    in.insert(in.end(), small.data, small.data + w * h * 4);
    ref.insert(ref.end(), large.data, large.data + (size_t)large.w * large.h * 4);
    batch.push_back(name);
  }
  flush();
  if (n_done == 0) throw std::runtime_error("No sample pairs of matching sizes found");
  const double n = (double)n_done;
  char buf[256];
  std::snprintf(buf, sizeof(buf),
                "mean over %zu pairs: network PSNR %.4f dB SSIM %.6f | baseline PSNR %.4f dB SSIM "
                "%.6f | gain %.4f dB",
                n_done, sum[0] / n, sum[1] / n, sum[2] / n, sum[3] / n, sum[4] / n);
  std::cout << buf << std::endl;
}

static void divide_samples(size_t validation_set_size, GpuAllocationPool& pool,
                           std::vector<SampleAllocationPool*>& train_set,
                           std::vector<SampleAllocationPool*>& validation_set, std::mt19937& rng) {
  train_set.clear();
  validation_set.clear();
  std::shuffle(pool.samples.begin(), pool.samples.end(), rng);
  for (size_t i = 0; i < pool.samples.size(); i++)
    (i < validation_set_size ? validation_set : train_set).push_back(&pool.samples[i]);
}

// contiguous even split of a sample set across the ranks
static std::vector<SampleAllocationPool*> shard(const std::vector<SampleAllocationPool*>& set,
                                                int rank, int world) {
  const size_t base = set.size() / (size_t)world, rem = set.size() % (size_t)world;
  const size_t begin = (size_t)rank * base + std::min<size_t>((size_t)rank, rem);
  const size_t count = base + ((size_t)rank < rem ? 1 : 0);
  return std::vector<SampleAllocationPool*>(set.begin() + (long)begin, set.begin() + (long)(begin + count));
}

int main(int argc, char** argv) {
  cnn_sr::utils::Argparse argparse("cnn", "SRCNN super-resolution (B200 CUDA build)");
  argparse.add_argument("train").help("Train mode");
  argparse.add_argument("eval").help("Measure PSNR / SSIM of the samples of a directory against their references");
  argparse.add_argument("dry").help("Do not store result");
  argparse.add_argument("profile").help("Print kernel execution times");
  argparse.add_argument("-c", "--config").required().help("CNN configuration");
  argparse.add_argument("-i", "--in").required().help("Image (or directory of images) during forward, samples directory during training");
  argparse.add_argument("-o", "--out").help("Output file path (either result image or new parameters)");
  argparse.add_argument("-e", "--epochs").help("Number of epochs during training");
  argparse.add_argument("-s", "--scale").help("Forward mode: enlarge the image N times first (default 1)");
  argparse.add_argument("-r", "--resample").help("Enlargement filter: lanczos (default) or bicubic");
  argparse.add_argument("--chroma-siting").help("A .y4m input: the output's chroma siting, keep (the input's), 420jpeg, 420mpeg2 or 420paldv; accepts every siting the input may have");
  argparse.add_argument("--bit-depth").help("A .y4m input: 8 (default) or 10, which reads 10-bit 4:2:0 (C420p10)");
  try {
    if (!argparse.parse((size_t)argc, argv)) return EXIT_SUCCESS;
  } catch (const std::exception& e) {
    std::cout << e.what() << std::endl;
    return EXIT_FAILURE;
  }

  const bool train = argparse.has_arg("train"), eval = argparse.has_arg("eval"),
             dry = argparse.has_arg("dry"), profile = argparse.has_arg("profile");
  const char* config_path = argparse.value("config");
  const char* in_path = argparse.value("in");
  const char* out_path = dry ? nullptr : argparse.value("out");
  size_t epochs = 0;
  argparse.value("epochs", epochs);
  if (!dry && !out_path) {
    std::cout << "Either provide out path or do the dry run" << std::endl;
    return EXIT_FAILURE;
  }
  size_t scale = 1;
  if (!parse_scale(argparse.value("scale"), &scale)) {
    std::cout << "--scale must be a whole number >= 1, got '" << argparse.value("scale") << "'"
              << std::endl;
    return EXIT_FAILURE;
  }
  const char* resample_name = argparse.value("resample") ? argparse.value("resample") : "lanczos";
  int filter = SRCNN_RESAMPLE_LANCZOS;
  if (std::strcmp(resample_name, "bicubic") == 0) {
    filter = SRCNN_RESAMPLE_BICUBIC;
  } else if (std::strcmp(resample_name, "lanczos") != 0) {
    std::cout << "--resample must be lanczos or bicubic, got '" << resample_name << "'" << std::endl;
    return EXIT_FAILURE;
  }
  if (train && eval) {
    std::cout << "eval and train exclude each other" << std::endl;
    return EXIT_FAILURE;
  }
  if (train && argparse.value("scale")) {
    std::cout << "--scale applies to the forward mode only" << std::endl;
    return EXIT_FAILURE;
  }
  size_t stem_len = 0;
  const bool in_y4m = ends_with(in_path, ".y4m", &stem_len);
  if ((train || eval) && in_y4m) {
    std::cout << "A .y4m input applies to the forward mode only" << std::endl;
    return EXIT_FAILURE;
  }
  // --chroma-siting: -1 = keep, else SRCNN_CHROMA_*
  const char* siting_name = argparse.value("chroma-siting");
  int out_siting = -1;
  if (siting_name) {
    const char* names[] = {"420jpeg", "420mpeg2", "420paldv"};
    for (int s = 0; s < 3; s++)
      if (std::strcmp(siting_name, names[s]) == 0) out_siting = s;
    if (out_siting < 0 && std::strcmp(siting_name, "keep") != 0) {
      std::cout << "--chroma-siting must be keep, 420jpeg, 420mpeg2 or 420paldv, got '"
                << siting_name << "'" << std::endl;
      return EXIT_FAILURE;
    }
    if (!in_y4m || train || eval) {
      std::cout << "--chroma-siting applies to a .y4m input in the forward mode only" << std::endl;
      return EXIT_FAILURE;
    }
  }
  const char* depth_name = argparse.value("bit-depth");
  int bit_depth = 8;
  if (depth_name) {
    if (std::strcmp(depth_name, "8") != 0 && std::strcmp(depth_name, "10") != 0) {
      std::cout << "--bit-depth must be 8 or 10, got '" << depth_name << "'" << std::endl;
      return EXIT_FAILURE;
    }
    bit_depth = std::atoi(depth_name);
    if (!in_y4m || train || eval) {
      std::cout << "--bit-depth applies to a .y4m input in the forward mode only" << std::endl;
      return EXIT_FAILURE;
    }
  }
  const bool in_dir = !train && !eval && !in_y4m && is_directory(in_path);
  if ((in_dir || eval) && out_path && !is_directory(out_path)) {
    std::cout << "Output directory '" << out_path << "' does not exist or is not a directory"
              << std::endl;
    return EXIT_FAILURE;
  }
  if (profile)
    std::cout << "!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!" << std::endl
              << "!!! RUNNING IN PROFILING MODE !!!" << std::endl
              << "!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!!" << std::endl;
  if (train)
    std::cout << "Training mode, epochs: " << epochs << std::endl
              << "Training samples directory: " << in_path << std::endl
              << "Output: " << (out_path ? out_path : "-") << std::endl;
  else if (eval)
    std::cout << "Evaluation mode" << std::endl
              << "Samples directory: " << in_path << std::endl
              << "Output: " << (out_path ? out_path : "-") << std::endl;
  else
    std::cout << "Forward mode" << std::endl
              << (in_dir ? "Input directory: " : in_y4m ? "Input video: " : "Input image: ")
              << in_path << std::endl
              << "Output: " << (out_path ? out_path : "-") << std::endl;
  if (!train && scale > 1)
    std::cout << "Scale: " << scale << "x, resample: " << resample_name << std::endl;

  const size_t validation_set_percent = 20, mini_batch_count = 2;
  bool error = false;
  try {
    ConfigReader reader;
    Config cfg = reader.read(config_path);
    std::cout << cfg << std::endl;
    // a video is checked whole before the context exists
    std::unique_ptr<Y4mReader> video;
    if (in_y4m) {
      video.reset(new Y4mReader(in_path, siting_name != nullptr, bit_depth == 10));
      if (video->header().bit_depth != bit_depth)
        throw std::runtime_error("--bit-depth 10 needs a 10-bit (C420p10) input; '" +
                                 std::string(in_path) + "' is 8-bit");
      if (bit_depth == 10 && out_siting > SRCNN_CHROMA_CENTER)
        throw std::runtime_error("--chroma-siting must be keep or 420jpeg for a 10-bit input: a "
                                 "C420p10 tag cannot state another siting");
      const size_t n_frames = video->check_frames();
      std::cout << "Video: " << video->header().w << "x" << video->header().h << ", " << n_frames
                << " frames" << std::endl;
    }

    opencl::Context context;
    context.init(profile);
    ConfigBasedDataPipeline data_pipeline(cfg, &context);
    data_pipeline.init(DataPipeline::LOAD_KERNEL_ALL);
    GpuAllocationPool gpu_alloc;

    if (eval) {
      std::vector<TrainSampleFiles> files;
      get_training_samples(in_path, files);
      if (files.empty()) throw std::runtime_error("No samples found");
      execute_eval(data_pipeline, gpu_alloc, files, out_path, scale, filter);
      context.block();
      return EXIT_SUCCESS;
    }
    if (video) {
      execute_y4m(data_pipeline, gpu_alloc, *video, out_path, scale, filter,
                  out_siting < 0 ? video->header().chroma_siting : out_siting);
      context.block();
      return EXIT_SUCCESS;
    }
    if (in_dir) {
      const std::vector<DirImage> images = get_directory_images(in_path);
      if (images.empty()) throw std::runtime_error("No .ppm/.pgm images found");
      execute_directory(data_pipeline, gpu_alloc, images, out_path, scale, filter);
      context.block();
      return EXIT_SUCCESS;
    }
    if (!train) {
      if (scale > 1)
        execute_upscale(data_pipeline, gpu_alloc, in_path, out_path, scale, filter);
      else
        execute_forward(data_pipeline, gpu_alloc, in_path, out_path);
      context.block();
      return EXIT_SUCCESS;
    }

    std::vector<TrainSampleFiles> files;
    get_training_samples(in_path, files);
    if (files.empty()) throw std::runtime_error("No training samples found");
    const size_t validation_set_size = (size_t)(files.size() * validation_set_percent / 100.0f),
                 train_set_size = files.size() - validation_set_size;
    if (validation_set_size == 0)
      std::cout << "[WARNING] Validation set is empty" << std::endl;
    else
      std::cout << "validation_set_size: " << validation_set_size << "/" << files.size() << " = "
                << (validation_set_size * 100.0f / files.size()) << "%" << std::endl;
    data_pipeline.set_mini_batch_size((train_set_size / mini_batch_count) + mini_batch_count);

    for (auto& pair : files) {
      ImageData expected_img, input_img;
      SampleAllocationPool s;
      prepare_image(&data_pipeline, pair.first.c_str(), expected_img, s.expected_data, s.expected_luma);
      cl_event ev = prepare_image(&data_pipeline, pair.second.c_str(), input_img, s.input_data, s.input_luma);
      data_pipeline.subtract_mean(s.input_luma, nullptr, &ev);
      s.input_w = (size_t)input_img.w;
      s.input_h = (size_t)input_img.h;
      context.block();
      context.raw_memory(s.input_data)->release();     // RGBA copies are no longer needed
      context.raw_memory(s.expected_data)->release();
      gpu_alloc.samples.push_back(s);
    }
    const size_t per_sample_px = gpu_alloc.samples[0].input_w * gpu_alloc.samples[0].input_h;
    context.block();

    // the reference shuffles with an unseeded std::random_shuffle; CNN_SR_SEED pins it
    std::mt19937 rng(std::getenv("CNN_SR_SEED") ? (unsigned)std::atoi(std::getenv("CNN_SR_SEED")) : 5489u);
    std::vector<SampleAllocationPool*> train_set, validation_set;
    const int rank = context.rank(), world = context.world();
    if (world > 1 && !std::getenv("CNN_SR_SEED"))
      std::cout << "[WARNING] data parallel run without CNN_SR_SEED: the ranks share the default "
                   "shuffle seed" << std::endl;
    for (size_t epoch_id = 0; epoch_id < epochs; epoch_id++) {
      divide_samples(validation_set_size, gpu_alloc, train_set, validation_set, rng);
      // data parallel (CNN_SR_WORLD > 1): every rank draws the SAME split (same seed), trains its
      // contiguous share of it, and update_parameters sums the gradients over the ranks before
      // the one update with the GLOBAL batch size (SURVEY 8e)
      const size_t global_train = train_set.size(), global_val = validation_set.size();
      if (world > 1) {
        train_set = shard(train_set, rank, world);
        validation_set = shard(validation_set, rank, world);
      }
      if (!train_set.empty()) data_pipeline.execute_batch(true, gpu_alloc, train_set);
      data_pipeline.update_parameters(gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3,
                                      global_train);
      if (((epoch_id % 25) == 0 || epoch_id == epochs - 1) && global_val != 0) {
        float sq_err = validation_set.empty()
                           ? 0.0f
                           : data_pipeline.execute_batch(false, gpu_alloc, validation_set);
        sq_err = context.allreduce_scalar(sq_err);   // 1-float all-reduce (no-op on one rank)
        if (std::isnan(sq_err)) {
          std::cout << "Error: squared error is NAN, after " << epoch_id << "/" << epochs
                    << " epochs" << std::endl;
          error = true;
          break;
        }
        const float mean_err = sq_err / global_val;
        if (rank == 0)
          std::cout << "[" << epoch_id << "] mean validation error: " << mean_err << " ("
                    << (mean_err / per_sample_px) << " per px)" << std::endl;
      }
      context.block();
    }
    if (out_path && rank == 0)   // replicas are identical: rank 0 writes
      data_pipeline.write_params_to_file(out_path, gpu_alloc.layer_1, gpu_alloc.layer_2, gpu_alloc.layer_3);
    context.block();
    std::cout << "DONE" << std::endl;
  } catch (const std::exception& e) {
    std::cout << "[ERROR] " << e.what() << std::endl;
    return EXIT_FAILURE;
  }
  return error ? EXIT_FAILURE : EXIT_SUCCESS;
}
