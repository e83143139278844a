// OptixHello <xml> <rays_per_pixel> [options] — headless stand-in for the reference executable.
//
// Keeps the reference's command line (optixHello.cpp:81-102): two positional arguments, the same usage
// message and exit code 1 when they are missing, the xml path taken relative to the current directory,
// rays per pixel through atoi; and its two timing lines ("Setup took : N ms", :1157;
// "Average frame time  : X ms", :1263). There is no window: the frame loop (:1163-1259) runs --frames
// times and the last frame is written to --out. Everything after the positionals is new surface
// (SURVEY.md Appendix E).
#include <cuda_runtime.h>

#include <unistd.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <string>
#include <utility>
#include <vector>

#include "../../include/params.h"
#include "../../include/rdc_b200.h"

#define CALL_CHECK(call)                                                                                       \
  do {                                                                                                         \
    int rc__ = (call);                                                                                         \
    if (rc__ != 0) {                                                                                           \
      std::cerr << "call (" << #call << ") failed with code " << rc__ << " (line " << __LINE__ << " in " << __FILE__ \
                << "): " << rdc_last_error_string() << std::endl;                                            \
      return 2;                                                                                                \
    }                                                                                                          \
  } while (0)

static void usage_options() {
  std::cout << "options: --width W --height H --frames N --out file.ppm|file.png|file.jpg --dump-f32 file --save-cache scene.rdc\n"
               "         --zoom Z --offset-x X --offset-y Y --seed S --max-depth D --tolerance T --curve-width R --endcap-size E\n"
               "         --weight-degree G --native (not an Orzan save) --no-blur --no-aa --denoiser (ignored) --brute-force\n"
               "         --device I --gpus N (the frame is split over N GPUs of this box, device I onwards)\n"
               "         --units-per-tile U (1, 2, 4, 8; pins the summation order: the same pixels bit for bit on any number of GPUs)\n"
               "         --accumulate (running mean over frames, restarted when the view changes)\n"
               "         --scroll-at F:Y / --drag-at F:DX:DY (before frame F: the scroll / drag callbacks of glfw_events.cpp:105-130)\n"
               "         --pick IX:IY (repeatable; after the last frame: the curve under pixel IX:IY of the final view)\n";
}

int main(int argc, char* argv[]) {
  if (argc < 3) {
    std::cout << "Please provide a path to a diffusion curve xml and the number of rays per pixel" << std::endl;
    return 1;
  }
  const int number_of_rays = std::atoi(argv[2]);
  std::string file_name = argv[1];
  if (file_name.empty() || file_name[0] != '/') {
    char cwd[4096];
    if (!getcwd(cwd, sizeof cwd)) return 2;
    file_name = std::string(cwd) + "/" + file_name;
  }

  rdc_ingest_options ingest;
  rdc_default_ingest_options(&ingest);
  ingest.use_diffusion_curve_save = USE_DIFFUSION_CURVE_SAVE;
  ingest.default_weight_degree = RDC_DEFAULT_WEIGHT_DEGREE;
  ingest.endcap_size = RDC_DEFAULT_ENDCAP_SIZE;
  rdc_accel_options accel;
  rdc_default_accel_options(&accel);
  accel.curve_width = RDC_DEFAULT_CURVE_WIDTH;
  bool use_blur = USE_BLUR, use_aa = USE_AA, brute = false;
  int max_depth = MAX_TRACE_DEPTH, frames = 1, device = 0;
  int out_w = 0, out_h = 0;
  float zoom = -1.0f, off_x = RDC_DEFAULT_OFFSET_X, off_y = RDC_DEFAULT_OFFSET_Y;
  unsigned seed = 0;
  int gpus = 1;
  unsigned units_per_tile = 0;  // rdc_frame_params::units_per_tile: 0 = chosen per launch
  bool accumulate = false;
  struct ViewEvent {
    int frame;
    bool scroll;
    double a, b;
  };
  std::vector<ViewEvent> events;
  std::vector<std::pair<unsigned, unsigned>> picks;
  std::string out_path, cache_path, dump_path;
  for (int i = 3; i < argc; ++i) {
    std::string a = argv[i];
    auto value = [&]() -> const char* {
      if (i + 1 >= argc) {
        std::cerr << "missing value for " << a << std::endl;
        std::exit(1);
      }
      return argv[++i];
    };
    if (a == "--width") out_w = std::atoi(value());
    else if (a == "--height") out_h = std::atoi(value());
    else if (a == "--frames") frames = std::atoi(value());
    else if (a == "--out") out_path = value();
    else if (a == "--save-cache") cache_path = value();
    else if (a == "--zoom") zoom = (float)std::atof(value());
    else if (a == "--offset-x") off_x = (float)std::atof(value());
    else if (a == "--offset-y") off_y = (float)std::atof(value());
    else if (a == "--seed") seed = (unsigned)std::strtoul(value(), nullptr, 0);
    else if (a == "--max-depth") max_depth = std::atoi(value());
    else if (a == "--tolerance") accel.flatness_tolerance = (float)std::atof(value());
    else if (a == "--curve-width") accel.curve_width = (float)std::atof(value());
    else if (a == "--endcap-size") ingest.endcap_size = (float)std::atof(value());
    else if (a == "--weight-degree") ingest.default_weight_degree = (float)std::atof(value());
    else if (a == "--native") ingest.use_diffusion_curve_save = 0;
    else if (a == "--no-blur") use_blur = false;
    else if (a == "--no-aa") use_aa = false;
    else if (a == "--denoiser") {}  // USE_DENOISER: accepted, ignored (closed OptiX model)
    else if (a == "--brute-force") brute = true;
    else if (a == "--device") device = std::atoi(value());
    else if (a == "--gpus") gpus = std::atoi(value());
    else if (a == "--units-per-tile") units_per_tile = (unsigned)std::atoi(value());
    else if (a == "--dump-f32") dump_path = value();
    else if (a == "--accumulate") accumulate = true;
    else if (a == "--scroll-at" || a == "--drag-at") {
      ViewEvent e{0, a == "--scroll-at", 0.0, 0.0};
      const char* v = value();
      const int got = e.scroll ? std::sscanf(v, "%d:%lf", &e.frame, &e.a) : std::sscanf(v, "%d:%lf:%lf", &e.frame, &e.a, &e.b);
      if (got != (e.scroll ? 2 : 3)) {
        std::cerr << "bad value for " << a << ": " << v << std::endl;
        return 1;
      }
      events.push_back(e);
    }
    else if (a == "--pick") {
      const char* v = value();
      unsigned ix = 0, iy = 0;
      if (std::sscanf(v, "%u:%u", &ix, &iy) != 2) {
        std::cerr << "bad value for --pick: " << v << std::endl;
        return 1;
      }
      picks.emplace_back(ix, iy);
    }
    else if (a == "--help") { usage_options(); return 0; }
    else {
      std::cerr << "unknown option " << a << std::endl;
      usage_options();
      return 1;
    }
  }
  if (frames < 1) frames = 1;

  if (gpus < 1 || gpus > RDC_MAX_FRAME_TARGETS) {
    std::cerr << "--gpus must be between 1 and " << RDC_MAX_FRAME_TARGETS << std::endl;
    return 1;
  }
  if (gpus > 1 && accumulate) {
    std::cerr << "--accumulate works on one GPU" << std::endl;
    return 1;
  }

  auto start_time = std::chrono::high_resolution_clock::now();
  int n_devices = 0;
  if (cudaGetDeviceCount(&n_devices) != cudaSuccess || n_devices < 1 || cudaSetDevice(device % (n_devices > 0 ? n_devices : 1)) != cudaSuccess) {
    std::cerr << "no usable CUDA device " << device << " (this program has no CPU path)" << std::endl;
    return 2;
  }
  rdc_host_scene* host = nullptr;
  // a ".rdc" path names a binary scene cache written by --save-cache (skips the XML parse)
  const bool cached = file_name.size() > 4 && file_name.compare(file_name.size() - 4, 4, ".rdc") == 0;
  auto t_ingest = std::chrono::high_resolution_clock::now();
  if (cached) CALL_CHECK(rdc_host_scene_load(file_name.c_str(), &host));
  else CALL_CHECK(rdc_ingest_xml_file(file_name.c_str(), &ingest, &host));
  const double ingest_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t_ingest).count();
  if (!cache_path.empty()) CALL_CHECK(rdc_host_scene_save(host, cache_path.c_str()));
  rdc_scene_arrays arrays;
  CALL_CHECK(rdc_host_scene_arrays(host, &arrays));

  // resolution comes from the XML unless overridden; the default zoom keeps the XML frame visible
  const int width = out_w > 0 ? out_w : arrays.image_width;
  const int height = out_h > 0 ? out_h : arrays.image_height;
  if (zoom <= 0.0f) zoom = (out_h > 0 && out_h != arrays.image_height) ? (float)arrays.image_height / (float)height : RDC_DEFAULT_ZOOM_FACTOR;
  rdc_frame_params params;
  rdc_default_frame_params(&params, (uint32_t)width, (uint32_t)height, (float)number_of_rays);
  params.zoom_factor = zoom;
  params.offset_x = off_x;
  params.offset_y = off_y;
  params.seed = seed;
  params.use_diffusion_curve_save = ingest.use_diffusion_curve_save;
  params.use_aa = use_aa;
  params.max_trace_depth = max_depth;
  params.traversal = brute ? RDC_TRAVERSAL_BRUTE_FORCE : RDC_TRAVERSAL_LBVH;
  params.units_per_tile = units_per_tile;
  int halo_rows = 0;
  CALL_CHECK(rdc_host_scene_halo_rows(host, max_depth, &halo_rows));

  // one rank per GPU: stream, device-resident scene + tree (replicated), and — with several GPUs — the shared frames
  std::vector<int> rank_device(gpus);
  std::vector<cudaStream_t> streams(gpus);
  std::vector<rdc_scene*> scenes(gpus, nullptr);
  std::vector<rdc_peer_frames*> peers(gpus, nullptr);
  auto t_build = std::chrono::high_resolution_clock::now();
  for (int r = 0; r < gpus; ++r) {
    rank_device[r] = (device + r) % n_devices;
    CALL_CHECK((int)cudaSetDevice(rank_device[r]));
    CALL_CHECK((int)cudaStreamCreate(&streams[r]));
    CALL_CHECK(rdc_accel_build(&arrays, &accel, streams[r], &scenes[r]));
    CALL_CHECK(rdc_scene_reserve(scenes[r], &params, gpus == 1 ? 1 : 0, streams[r]));
    if (gpus > 1) CALL_CHECK(rdc_peer_frames_create((uint32_t)width, (uint32_t)height, r, gpus, &peers[r]));
  }
  if (gpus > 1) CALL_CHECK(rdc_peer_frames_connect_local(peers.data(), gpus));
  for (int r = 0; r < gpus; ++r) CALL_CHECK((int)cudaStreamSynchronize(streams[r]));
  const double build_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t_build).count();
  CALL_CHECK((int)cudaSetDevice(rank_device[0]));
  rdc_scene* scene = scenes[0];
  cudaStream_t stream = streams[0];
  rdc_scene_info info;
  CALL_CHECK(rdc_scene_get_info(scene, &info));

  const size_t n_pixels = (size_t)width * height;
  float* host_image = nullptr;
  CALL_CHECK((int)cudaHostAlloc((void**)&host_image, sizeof(float) * 4 * n_pixels, cudaHostAllocPortable));
  // --accumulate: the running mean stands where the reference's temporal denoiser stands in the frame loop
  // (optixHello.cpp:1186-1235); frame, sigma, blur scratch and mean live on the device
  float *d_image = nullptr, *d_sigma = nullptr, *d_scratch = nullptr, *d_mean = nullptr;
  if (accumulate) {
    CALL_CHECK((int)cudaMalloc((void**)&d_image, sizeof(float) * 4 * n_pixels));
    CALL_CHECK((int)cudaMalloc((void**)&d_sigma, sizeof(float) * n_pixels));
    CALL_CHECK((int)cudaMalloc((void**)&d_scratch, sizeof(float) * 4 * n_pixels));
    CALL_CHECK((int)cudaMalloc((void**)&d_mean, sizeof(float) * 4 * n_pixels));
  }
  auto setup_ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::high_resolution_clock::now() - start_time);
  std::cout << "Setup took : " << setup_ms.count() << " ms" << std::endl;
  std::cout << "Setup parts : ingest " << ingest_ms << " ms, upload + tree build on " << gpus << " GPU(s) " << build_ms << " ms" << std::endl;
  std::cout << "Scene : " << info.n_curves << " curves, " << info.n_segments << " segments, " << info.n_chords
            << " chords, tree depth " << info.bvh_depth << std::endl;

  double total_ms = 0.0;
  uint32_t frames_in_mean = 0;
  for (int f = 0; f < frames; ++f) {
    auto t0 = std::chrono::high_resolution_clock::now();
    // the callbacks run between frames and mutate the view (glfw_events.cpp:105-130); a changed view restarts the mean
    for (const ViewEvent& e : events)
      if (e.frame == f) {
        if (e.scroll) rdc_view_scroll(&params, e.a);
        else rdc_view_drag(&params, e.a, e.b);
        frames_in_mean = 0;
      }
    params.frame = (uint32_t)f;
    if (accumulate) {
      CALL_CHECK(rdc_render(scene, &params, d_image, d_sigma, stream));
      if (use_blur) CALL_CHECK(rdc_gaussian_blur(d_image, d_image, d_sigma, d_scratch, width, height, 0, height, nullptr, stream));
      CALL_CHECK(rdc_accumulate(d_mean, d_image, n_pixels, frames_in_mean, stream));
      frames_in_mean++;
      CALL_CHECK((int)cudaMemcpyAsync(host_image, d_mean, sizeof(float) * 4 * n_pixels, cudaMemcpyDeviceToHost, stream));
      CALL_CHECK((int)cudaStreamSynchronize(stream));
    } else if (gpus == 1) {
      CALL_CHECK(rdc_render_frame_to_host(scene, &params, use_blur ? 1 : 0, host_image, stream));
    } else {
      // every rank renders its strips and copies its rows of the finished frame over its own PCIe link
      for (int r = 0; r < gpus; ++r) {
        CALL_CHECK((int)cudaSetDevice(rank_device[r]));
        CALL_CHECK(rdc_peer_frame_to_host(scenes[r], peers[r], &params, use_blur ? 1 : 0, halo_rows, host_image, streams[r]));
      }
      for (int r = 0; r < gpus; ++r) CALL_CHECK(rdc_peer_frames_wait(peers[r]));
    }
    printf("\rframe : %d", f + 1);
    fflush(stdout);
    total_ms += std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
  }
  std::cout << std::endl;
  const double avg_ms = total_ms / frames;
  std::cout << "Average frame time  : " << avg_ms << " ms" << std::endl;
  std::cout << "Throughput : " << (double)width * height * number_of_rays / (avg_ms * 1e-3) / 1e9 << " Grays/s" << std::endl;
  if (accumulate) std::cout << "Frames in the mean : " << frames_in_mean << std::endl;

  if (!picks.empty()) {  // the editor's click: pixel -> scene point -> nearest curve, on the view of the last frame
    const uint32_t n = (uint32_t)picks.size();
    std::vector<float> pts(2 * n);
    for (uint32_t k = 0; k < n; ++k)
      CALL_CHECK(rdc_view_pixel_to_scene(&params, picks[k].first, picks[k].second, &pts[2 * k], &pts[2 * k + 1]));
    std::vector<rdc_pick> got(n);
    float* d_pts = nullptr;
    rdc_pick* d_out = nullptr;
    CALL_CHECK((int)cudaMalloc((void**)&d_pts, sizeof(float) * 2 * n));
    CALL_CHECK((int)cudaMalloc((void**)&d_out, sizeof(rdc_pick) * n));
    CALL_CHECK((int)cudaMemcpyAsync(d_pts, pts.data(), sizeof(float) * 2 * n, cudaMemcpyHostToDevice, stream));
    CALL_CHECK(rdc_scene_pick(scene, d_pts, n, INFINITY, params.use_diffusion_curve_save, d_out, nullptr, stream));
    CALL_CHECK((int)cudaMemcpyAsync(got.data(), d_out, sizeof(rdc_pick) * n, cudaMemcpyDeviceToHost, stream));
    CALL_CHECK((int)cudaStreamSynchronize(stream));
    cudaFree(d_pts);
    cudaFree(d_out);
    for (uint32_t k = 0; k < n; ++k) {
      const rdc_pick& q = got[k];
      if (q.chord == RDC_PICK_NONE) {
        printf("Pick %u:%u : scene (%g, %g) nothing\n", picks[k].first, picks[k].second, pts[2 * k], pts[2 * k + 1]);
        continue;
      }
      printf("Pick %u:%u : scene (%g, %g) curve %u segment %u u %.6g side %s%s distance %g\n", picks[k].first, picks[k].second,
             pts[2 * k], pts[2 * k + 1], q.curve, q.segment, q.u, (q.flags & RDC_PICK_RIGHT) ? "right" : "left",
             (q.flags & RDC_PICK_PORTAL) ? " (portal)" : "", q.distance);
    }
  }

  if (!dump_path.empty()) {  // the float image as rendered (row 0 first, RGBA float32, no flip): input of tools/rdc_diff.py
    FILE* fp = std::fopen(dump_path.c_str(), "wb");
    if (!fp || std::fwrite(host_image, sizeof(float) * 4, n_pixels, fp) != n_pixels) {
      std::cerr << "cannot write " << dump_path << std::endl;
      return 2;
    }
    std::fclose(fp);
    std::cout << "Wrote " << dump_path << " (" << width << "x" << height << " float4)" << std::endl;
  }
  if (!out_path.empty()) {
    std::vector<uint8_t> rgba((size_t)4 * width * height);
    // Orzan saves are rendered bottom-up (DeviceCode.cu:104-105) and shown with glDrawPixels; the
    // screenshot flips them into a top-down file (glfw_events.cpp:92). Same rule here.
    CALL_CHECK(rdc_image_to_rgba8(host_image, width, height, ingest.use_diffusion_curve_save ? 1 : 0, rgba.data()));
    auto ends_with = [&](const char* ext) {
      const size_t n = std::strlen(ext);
      return out_path.size() > n && out_path.compare(out_path.size() - n, n, ext) == 0;
    };
    if (ends_with(".png")) CALL_CHECK(rdc_write_png(out_path.c_str(), rgba.data(), width, height));
    else if (ends_with(".jpg") || ends_with(".jpeg"))  // the screenshot's format; its quality argument ends up as 100
      CALL_CHECK(rdc_write_jpg(out_path.c_str(), rgba.data(), width, height, 100));
    else CALL_CHECK(rdc_write_ppm(out_path.c_str(), rgba.data(), width, height));
    std::cout << "Wrote " << out_path << std::endl;
  }
  cudaFreeHost(host_image);
  cudaFree(d_image);
  cudaFree(d_sigma);
  cudaFree(d_scratch);
  cudaFree(d_mean);
  for (int r = 0; r < gpus; ++r) {
    cudaSetDevice(rank_device[r]);
    if (peers[r]) rdc_peer_frames_destroy(peers[r]);
    rdc_scene_destroy(scenes[r]);
    cudaStreamDestroy(streams[r]);
  }
  rdc_host_scene_destroy(host);
  return 0;
}
