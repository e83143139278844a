// capi.cu — the extern "C" surface declared in include/rdc_b200.h. No C++ exception crosses it.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>

#include "device_scene.h"
#include "host_scene.h"
#include "xml_dom.h"

namespace rdc {
const char* last_error();
}

namespace {

template <class F>
int guarded(int parse_code, F&& body) {
  try {
    return body();
  } catch (const rdc::XmlError& e) {
    rdc::set_error("%s", e.what());
    return RDC_E_PARSE;
  } catch (const std::bad_alloc&) {
    rdc::set_error("out of host memory");
    return RDC_E_LIMIT;
  } catch (const std::exception& e) {
    rdc::set_error("%s", e.what());
    return parse_code;
  } catch (...) {
    rdc::set_error("unknown failure");
    return RDC_E_INVALID;
  }
}

}  // namespace

// ---- binary scene cache (SURVEY.md 8f rank 4): the ingested arrays, little-endian, versioned ----
namespace {
const char kCacheMagic[8] = {'R', 'D', 'C', 'S', 'C', 'N', '0', '1'};

template <class T>
bool put_vec(std::FILE* f, const std::vector<T>& v) {
  const uint64_t n = v.size();
  return std::fwrite(&n, sizeof n, 1, f) == 1 && (n == 0 || std::fwrite(v.data(), sizeof(T), n, f) == n);
}
// bytes between the read position and the end of the file: no element count of an untrusted header may ask for more
uint64_t bytes_left(std::FILE* f) {
  const long here = std::ftell(f);
  if (here < 0 || std::fseek(f, 0, SEEK_END) != 0) return 0;
  const long end = std::ftell(f);
  std::fseek(f, here, SEEK_SET);
  return end > here ? (uint64_t)(end - here) : 0;
}
template <class T>
bool get_vec(std::FILE* f, std::vector<T>& v) {
  uint64_t n = 0;
  if (std::fread(&n, sizeof n, 1, f) != 1 || n > bytes_left(f) / sizeof(T)) return false;
  v.resize(n);
  return n == 0 || std::fread(v.data(), sizeof(T), n, f) == n;
}
struct FileCloser {
  std::FILE* f;
  ~FileCloser() {
    if (f) std::fclose(f);
  }
};
template <class Op>
bool stop_list_io(std::FILE* f, rdc_host_scene::StopList& l, Op&& io) {
  return io(f, l.index) && io(f, l.value) && io(f, l.u);
}
}  // namespace

extern "C" {

const char* rdc_last_error_string(void) { return rdc::last_error(); }
const char* rdc_version(void) { return "rdc_b200 0.1 (sm_100a)"; }
void rdc_free(void* p) { std::free(p); }

void rdc_default_ingest_options(rdc_ingest_options* o) {
  if (!o) return;
  o->use_diffusion_curve_save = 1;  // params.h:24
  o->default_weight_degree = 0.5f;  // optixHello.cpp:94
  o->endcap_size = 8.0f;            // optixHello.cpp:96
}

int rdc_ingest_xml_file(const char* path, const rdc_ingest_options* opts, rdc_host_scene** out) {
  if (!path || !out) {
    rdc::set_error("ingest: null argument");
    return RDC_E_INVALID;
  }
  rdc_ingest_options o;
  rdc_default_ingest_options(&o);
  if (opts) o = *opts;
  return guarded(RDC_E_PARSE, [&]() {
    std::FILE* f = std::fopen(path, "rb");
    if (!f) {
      rdc::set_error("ingest: cannot open %s", path);
      return RDC_E_IO;
    }
    std::fclose(f);
    auto* s = new rdc_host_scene();
    try {
      rdc::ingest_xml_file(path, o, *s);
    } catch (...) {
      delete s;
      throw;
    }
    *out = s;
    return 0;
  });
}

int rdc_ingest_xml_memory(const char* text, size_t len, const rdc_ingest_options* opts, rdc_host_scene** out) {
  if (!text || !out) {
    rdc::set_error("ingest: null argument");
    return RDC_E_INVALID;
  }
  rdc_ingest_options o;
  rdc_default_ingest_options(&o);
  if (opts) o = *opts;
  return guarded(RDC_E_PARSE, [&]() {
    auto* s = new rdc_host_scene();
    try {
      rdc::ingest_xml_text(text, len, o, *s);
    } catch (...) {
      delete s;
      throw;
    }
    *out = s;
    return 0;
  });
}

int rdc_host_scene_arrays(const rdc_host_scene* scene, rdc_scene_arrays* out) {
  if (!scene || !out) {
    rdc::set_error("scene arrays: null argument");
    return RDC_E_INVALID;
  }
  scene->view(out);
  return 0;
}

void rdc_host_scene_destroy(rdc_host_scene* scene) { delete scene; }

int rdc_host_scene_halo_rows(const rdc_host_scene* scene, int max_trace_depth, int* halo_rows) {
  if (!scene || !halo_rows || max_trace_depth < 0) {
    rdc::set_error("halo rows: bad argument");
    return RDC_E_INVALID;
  }
  float m = 0.0f;
  for (uint32_t i = 0; i < scene->n_true[2]; ++i) m = std::fmax(m, scene->blur.value[i]);
  bool portals = false;
  for (int32_t c : scene->curve_connect) portals |= c >= 0;
  double reach = m;
  if (portals && m > 1.0f) reach = std::pow((double)m, max_trace_depth + 1);
  const double rows = std::ceil(3.0 * reach);
  *halo_rows = rows > 1e6 ? 1000000 : (int)rows;
  return 0;
}

int rdc_host_scene_save(const rdc_host_scene* scene, const char* path) {
  if (!scene || !path) {
    rdc::set_error("scene save: null argument");
    return RDC_E_INVALID;
  }
  std::FILE* f = std::fopen(path, "wb");
  if (!f) {
    rdc::set_error("scene save: cannot open %s", path);
    return RDC_E_IO;
  }
  rdc_host_scene& s = const_cast<rdc_host_scene&>(*scene);
  const int32_t dims[2] = {s.image_width, s.image_height};
  auto put = [](std::FILE* fp, auto& v) { return put_vec(fp, v); };
  bool ok = std::fwrite(kCacheMagic, 1, 8, f) == 8 && std::fwrite(dims, sizeof dims, 1, f) == 1 &&
            std::fwrite(s.n_true, sizeof s.n_true, 1, f) == 1 && put_vec(f, s.vertices) && put_vec(f, s.segment_indices) &&
            put_vec(f, s.curve_map) && put_vec(f, s.curve_index) && put_vec(f, s.curve_map_inverse) && put_vec(f, s.curve_connect);
  for (rdc_host_scene::StopList* l : {&s.color_left, &s.color_right, &s.blur, &s.weight, &s.weight_degree}) ok = ok && stop_list_io(f, *l, put);
  ok = (std::fclose(f) == 0) && ok;
  if (!ok) {
    rdc::set_error("scene save: write failed for %s", path);
    return RDC_E_IO;
  }
  return 0;
}

int rdc_host_scene_load(const char* path, rdc_host_scene** out) {
  if (!path || !out) {
    rdc::set_error("scene load: null argument");
    return RDC_E_INVALID;
  }
  std::FILE* f = std::fopen(path, "rb");
  if (!f) {
    rdc::set_error("scene load: cannot open %s", path);
    return RDC_E_IO;
  }
  FileCloser closer{f};  // closed on every path, exceptions included
  return guarded(RDC_E_PARSE, [&]() {
    std::unique_ptr<rdc_host_scene> s(new rdc_host_scene());
    char magic[8];
    int32_t dims[2] = {0, 0};
    auto get = [](std::FILE* fp, auto& v) { return get_vec(fp, v); };
    bool ok = std::fread(magic, 1, 8, f) == 8 && std::memcmp(magic, kCacheMagic, 8) == 0 && std::fread(dims, sizeof dims, 1, f) == 1 &&
              std::fread(s->n_true, sizeof s->n_true, 1, f) == 1 && get_vec(f, s->vertices) && get_vec(f, s->segment_indices) &&
              get_vec(f, s->curve_map) && get_vec(f, s->curve_index) && get_vec(f, s->curve_map_inverse) && get_vec(f, s->curve_connect);
    for (rdc_host_scene::StopList* l : {&s->color_left, &s->color_right, &s->blur, &s->weight, &s->weight_degree}) ok = ok && stop_list_io(f, *l, get);
    // structural checks: the arrays must describe a consistent scene (rdc_accel_build checks the cross references)
    const size_t nseg = s->segment_indices.size(), ncurves = s->curve_connect.size();
    ok = ok && dims[0] > 0 && dims[1] > 0 && nseg > 0 && ncurves > 0 && s->vertices.size() % 3 == 0 && s->curve_map.size() == nseg &&
         s->curve_index.size() == nseg && s->curve_map_inverse.size() == ncurves;
    const rdc_host_scene::StopList* lists[5] = {&s->color_left, &s->color_right, &s->blur, &s->weight, &s->weight_degree};
    for (int k = 0; ok && k < 5; ++k) {
      const rdc_host_scene::StopList* l = lists[k];
      ok = l->index.size() == 2 * ncurves && l->value.size() == l->u.size() * (size_t)l->stride && l->u.size() >= 2 &&
           (size_t)s->n_true[k] + 2 <= l->u.size();
    }
    if (!ok) {
      rdc::set_error("scene load: %s is not a scene cache of this version", path);
      return RDC_E_PARSE;
    }
    s->image_width = dims[0];
    s->image_height = dims[1];
    s->sealed = true;
    *out = s.release();
    return 0;
  });
}

int rdc_xml_dump_file(const char* path, char** out_text) {
  if (!path || !out_text) {
    rdc::set_error("xml dump: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_PARSE, [&]() {
    auto doc = rdc::xml_parse_file(path);
    std::string s;
    rdc::xml_dump(*doc->root, 0, s);
    char* buf = (char*)std::malloc(s.size() + 1);
    if (!buf) throw std::bad_alloc();
    std::memcpy(buf, s.c_str(), s.size() + 1);
    *out_text = buf;
    return 0;
  });
}

void rdc_default_accel_options(rdc_accel_options* o) {
  if (!o) return;
  o->curve_width = 1e-3f;  // optixHello.cpp:95
  o->flatness_tolerance = 0.05f;
  o->max_chords_per_segment = 1024;
  o->run_length = 0;
  o->shading_records = 0;
  o->tree = RDC_TREE_AUTO;
}

int rdc_accel_build(const rdc_scene_arrays* arrays, const rdc_accel_options* opts, rdc_stream stream, rdc_scene** out) {
  if (!arrays || !out) {
    rdc::set_error("accel: null argument");
    return RDC_E_INVALID;
  }
  rdc_accel_options o;
  rdc_default_accel_options(&o);
  if (opts) o = *opts;
  return guarded(RDC_E_INVALID, [&]() { return rdc::build_scene(*arrays, o, (cudaStream_t)stream, out); });
}

int rdc_scene_get_info(const rdc_scene* scene, rdc_scene_info* out) {
  if (!scene || !out) {
    rdc::set_error("scene info: null argument");
    return RDC_E_INVALID;
  }
  *out = scene->info;
  return 0;
}

int rdc_scene_download_chords(const rdc_scene* scene, float* geom, uint32_t* ids) {
  if (!scene || !geom || !ids) {
    rdc::set_error("download chords: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() { return rdc::download_chords(scene, geom, ids); });
}

int rdc_scene_update_stops(rdc_scene* scene, const rdc_scene_arrays* arrays, rdc_stream stream) {
  if (!scene || !arrays) {
    rdc::set_error("update stops: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() { return rdc::update_stops(scene, *arrays, (cudaStream_t)stream); });
}

int rdc_scene_download_stop_tables(const rdc_scene* scene, void* seg_walk, void* chord_walk, void* chord_records) {
  if (!scene || !seg_walk || !chord_walk) {
    rdc::set_error("download stop tables: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() { return rdc::download_stop_tables(scene, seg_walk, chord_walk, chord_records); });
}

void rdc_scene_destroy(rdc_scene* scene) { rdc::destroy_scene(scene); }

void rdc_default_frame_params(rdc_frame_params* p, uint32_t width, uint32_t height, float rays_per_pixel) {
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->image_width = width;
  p->image_height = height;
  p->number_of_rays_per_pixel = rays_per_pixel;
  p->zoom_factor = 1.0f;  // optixHello.cpp:89-91
  p->offset_x = 0.0f;
  p->offset_y = 0.0f;
  p->frame = 0;
  p->seed = 0;
  p->row_begin = 0;
  p->row_end = height;
  p->strip_stride = 0;
  p->strip_offset = 0;
  p->use_diffusion_curve_save = 1;  // params.h:24
  p->use_aa = 1;                    // params.h:28
  p->max_trace_depth = 2;           // params.h:32
  p->traversal = RDC_TRAVERSAL_LBVH;
  p->hit_ids = nullptr;
  p->max_sigma = nullptr;
  p->stats = nullptr;
  p->route = RDC_ROUTE_AUTO;
  p->units_per_tile = 0;
  p->local_radius = 0.0f;
}

int rdc_render(rdc_scene* scene, const rdc_frame_params* params, float* image, float* blur_map, rdc_stream stream) {
  if (!scene || !params) {
    rdc::set_error("render: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    return rdc::render(scene, *params, reinterpret_cast<float4*>(image), blur_map, (cudaStream_t)stream);
  });
}

int rdc_render_to_frames(rdc_scene* scene, const rdc_frame_params* params, uint32_t n_targets, float* const* images,
                         float* const* blur_maps, rdc_stream stream) {
  if (!scene || !params || n_targets == 0) {
    rdc::set_error("render_to_frames: null argument or no target frame");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    return rdc::render(scene, *params, nullptr, nullptr, (cudaStream_t)stream, n_targets, images, blur_maps);
  });
}

int rdc_render_color_adjoint(rdc_scene* scene, const rdc_frame_params* params, const float* image_grad,
                             double* grad_color_left, double* grad_color_right, rdc_stream stream) {
  if (!params) {
    rdc::set_error("color adjoint: null params");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    return rdc::color_adjoint(scene, *params, reinterpret_cast<const float4*>(image_grad), grad_color_left, grad_color_right,
                              (cudaStream_t)stream);
  });
}

int rdc_render_blur_adjoint(rdc_scene* scene, const rdc_frame_params* params, const float* sigma_grad, double* grad_blur,
                            rdc_stream stream) {
  if (!params) {
    rdc::set_error("render blur adjoint: null params");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    return rdc::blur_adjoint(scene, *params, sigma_grad, grad_blur, (cudaStream_t)stream);
  });
}

int rdc_render_weight_adjoint(rdc_scene* scene, const rdc_frame_params* params, const float* image_grad, const float* sigma_grad,
                              double* grad_weight, double* grad_weight_degree, rdc_stream stream) {
  if (!params) {
    rdc::set_error("render weight adjoint: null params");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    return rdc::weight_adjoint(scene, *params, reinterpret_cast<const float4*>(image_grad), sigma_grad, grad_weight,
                               grad_weight_degree, (cudaStream_t)stream);
  });
}

int rdc_scene_pick(rdc_scene* scene, const float* points, uint32_t n, float max_distance, int use_diffusion_curve_save,
                   rdc_pick* out, float* stops, rdc_stream stream) {
  return guarded(RDC_E_INVALID, [&]() {
    return rdc::pick(scene, points, n, max_distance, use_diffusion_curve_save, out, stops, (cudaStream_t)stream);
  });
}

int rdc_scene_pick_frame(rdc_scene* scene, const rdc_frame_params* params, float max_distance, rdc_pick* out, float* stops,
                         rdc_stream stream) {
  return guarded(RDC_E_INVALID, [&]() { return rdc::pick_frame(scene, params, max_distance, out, stops, (cudaStream_t)stream); });
}

int rdc_view_pixel_to_scene(const rdc_frame_params* params, uint32_t ix, uint32_t iy, float* x, float* y) {
  if (!params || !x || !y) {
    rdc::set_error("view pixel to scene: null argument");
    return RDC_E_INVALID;
  }
  if (ix >= params->image_width || iy >= params->image_height) {
    rdc::set_error("view pixel to scene: pixel (%u, %u) is outside the %ux%u frame", ix, iy, params->image_width, params->image_height);
    return RDC_E_INVALID;
  }
  *x = rdc_pixel_centre_x(params->image_width, params->zoom_factor, params->offset_x, ix);
  *y = rdc_pixel_centre_y(params->image_height, params->zoom_factor, params->offset_y, params->use_diffusion_curve_save != 0, iy);
  return 0;
}

int rdc_gaussian_blur(void* dest, const void* source, const float* sigma, void* scratch, int width, int height,
                      int row_begin, int row_end, const float* max_sigma, rdc_stream stream) {
  return rdc::gaussian_blur(static_cast<float4*>(dest), static_cast<const float4*>(source), sigma,
                            static_cast<float4*>(scratch), width, height, row_begin, row_end, max_sigma,
                            (cudaStream_t)stream);
}

int rdc_gaussian_blur_band(void* dest, const void* source, const float* sigma, void* scratch, int width, int height,
                           int row_begin, int row_end, int halo_rows, const float* max_sigma, rdc_stream stream) {
  return rdc::gaussian_blur(static_cast<float4*>(dest), static_cast<const float4*>(source), sigma,
                            static_cast<float4*>(scratch), width, height, row_begin, row_end, max_sigma,
                            (cudaStream_t)stream, halo_rows);
}

int rdc_gaussian_blur_adjoint(void* grad_source, const void* grad_dest, const float* sigma, void* scratch, int width, int height,
                              int row_begin, int row_end, const float* max_sigma, rdc_stream stream) {
  return rdc::gaussian_blur_adjoint(static_cast<float4*>(grad_source), static_cast<const float4*>(grad_dest), sigma,
                                    static_cast<float4*>(scratch), width, height, row_begin, row_end, max_sigma,
                                    (cudaStream_t)stream);
}

int rdc_gaussian_blur_sigma_adjoint(float* grad_sigma, const void* grad_dest, const void* source, const float* sigma,
                                    void* scratch, int width, int height, int row_begin, int row_end,
                                    const float* max_sigma, rdc_stream stream) {
  return rdc::gaussian_blur_sigma_adjoint(grad_sigma, static_cast<const float4*>(grad_dest), static_cast<const float4*>(source),
                                          sigma, static_cast<float4*>(scratch), width, height, row_begin, row_end, max_sigma,
                                          (cudaStream_t)stream);
}

// Reference-named helpers. They return void like the originals; failures are readable through
// rdc_last_error_string() and, being CUDA errors, through cudaGetLastError().
void gaussianBlur(void* dest, void* source, float* sigma, int width, int height, rdc_stream stream) {
  if (width <= 0 || height <= 0) {
    rdc::set_error("gaussianBlur: bad size");
    return;
  }
  cudaStream_t st = (cudaStream_t)stream;
  void* scratch = nullptr;
  cudaError_t e = cudaMallocAsync(&scratch, sizeof(float4) * (size_t)width * height, st);
  if (e != cudaSuccess) {
    rdc::cuda_fail(e, "cudaMallocAsync(blur scratch)");
    return;
  }
  rdc::gaussian_blur(static_cast<float4*>(dest), static_cast<const float4*>(source), sigma, static_cast<float4*>(scratch),
                     width, height, 0, height, nullptr, st);
  e = cudaFreeAsync(scratch, st);
  if (e != cudaSuccess) rdc::cuda_fail(e, "cudaFreeAsync(blur scratch)");
}

void setFloatDevice(float* dest, unsigned int n, float src, rdc_stream stream) {
  rdc::set_float(dest, n, src, (cudaStream_t)stream);
}

void setupCurand(void* states, int width, int height, rdc_stream stream) {
  (void)states;
  (void)stream;
  if (width <= 0 || height <= 0) rdc::set_error("setupCurand: bad size");
}

namespace {
// copy stream, events and the grow-only device frames of rdc_render_frame_to_host(_async)
int ensure_frame_buffers(rdc_scene* scene, size_t n, cudaStream_t st) {
  if (!scene->copy_stream) {
    RDC_CUDA(cudaStreamCreateWithFlags(&scene->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      RDC_CUDA(cudaEventCreateWithFlags(&scene->rendered[k], cudaEventDisableTiming));
      RDC_CUDA(cudaEventCreateWithFlags(&scene->copied[k], cudaEventDisableTiming));
    }
  }
  if (n > scene->frame_pixels) {
    RDC_CUDA(cudaStreamSynchronize(st));
    RDC_CUDA(cudaStreamSynchronize(scene->copy_stream));
    cudaFree(scene->frame_image[0]);
    cudaFree(scene->frame_image[1]);
    cudaFree(scene->frame_scratch);
    cudaFree(scene->frame_sigma);
    scene->frame_image[0] = scene->frame_image[1] = scene->frame_scratch = nullptr;
    scene->frame_sigma = nullptr;
    scene->frame_pixels = 0;
    RDC_CUDA(cudaMalloc((void**)&scene->frame_image[0], n * sizeof(float4)));
    RDC_CUDA(cudaMalloc((void**)&scene->frame_image[1], n * sizeof(float4)));
    RDC_CUDA(cudaMalloc((void**)&scene->frame_scratch, n * sizeof(float4)));
    RDC_CUDA(cudaMalloc((void**)&scene->frame_sigma, (n + 1) * sizeof(float)));
    scene->frame_pixels = n;
  }
  return 0;
}
}  // namespace

int rdc_scene_reserve(rdc_scene* scene, const rdc_frame_params* params, int host_frames, rdc_stream stream) {
  if (!scene || !params) {
    rdc::set_error("reserve: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    int rc = rdc::reserve(scene, *params, (cudaStream_t)stream);
    if (rc == 0 && host_frames)
      rc = ensure_frame_buffers(scene, (size_t)(params->row_end - params->row_begin) * params->image_width, (cudaStream_t)stream);
    return rc;
  });
}

int rdc_scene_launch_plan(const rdc_scene* scene, const rdc_frame_params* params, rdc_launch_plan* out) {
  if (!scene || !params || !out) {
    rdc::set_error("launch plan: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() { return rdc::launch_plan(scene, *params, out); });
}

// Enqueue-only frame: render -> [blur] on `stream`, then the copy to host memory on the handle's own copy
// stream, so that the copy of frame f overlaps the rendering of frame f+1 (two device images, used in turn).
int rdc_render_frame_to_host_async(rdc_scene* scene, const rdc_frame_params* params, int use_blur, float* host_image,
                                   rdc_stream stream) {
  if (!scene || !params || !host_image) {
    rdc::set_error("render frame: null argument");
    return RDC_E_INVALID;
  }
  return guarded(RDC_E_INVALID, [&]() {
    cudaStream_t st = (cudaStream_t)stream;
    if (params->row_begin >= params->row_end || params->row_end > params->image_height) {
      rdc::set_error("render frame: bad row band");
      return RDC_E_INVALID;
    }
    const size_t rows = params->row_end - params->row_begin;
    const size_t n = rows * params->image_width;
    if (int rc = ensure_frame_buffers(scene, n, st)) return rc;  // grow-only; rdc_scene_reserve does it ahead of time
    const int slot = scene->frame_slot ^= 1;
    float4* image = scene->frame_image[slot];
    float* sigma = scene->frame_sigma;
    float* flag = sigma + scene->frame_pixels;
    rdc_frame_params p = *params;
    // the copy that last read this image must be over before it is rendered into again
    RDC_CUDA(cudaStreamWaitEvent(st, scene->copied[slot], 0));
    if (use_blur) {
      RDC_CUDA(cudaMemsetAsync(flag, 0, sizeof(float), st));
      p.max_sigma = flag;
    }
    int rc = rdc::render(scene, p, image, sigma, st);
    if (rc == 0 && use_blur)
      rc = rdc::gaussian_blur(image, image, sigma, scene->frame_scratch, (int)params->image_width, (int)rows, 0, (int)rows, flag, st);
    if (rc != 0) return rc;
    RDC_CUDA(cudaEventRecord(scene->rendered[slot], st));
    RDC_CUDA(cudaStreamWaitEvent(scene->copy_stream, scene->rendered[slot], 0));
    RDC_CUDA(cudaMemcpyAsync(host_image, image, n * sizeof(float4), cudaMemcpyDeviceToHost, scene->copy_stream));
    RDC_CUDA(cudaEventRecord(scene->copied[slot], scene->copy_stream));
    return 0;
  });
}

// Blocks until every frame enqueued with rdc_render_frame_to_host_async has reached host memory.
int rdc_frame_wait(rdc_scene* scene) {
  if (!scene) {
    rdc::set_error("frame wait: null argument");
    return RDC_E_INVALID;
  }
  if (scene->copy_stream) RDC_CUDA(cudaStreamSynchronize(scene->copy_stream));
  return 0;
}

int rdc_render_frame_to_host(rdc_scene* scene, const rdc_frame_params* params, int use_blur, float* host_image,
                             rdc_stream stream) {
  int rc = rdc_render_frame_to_host_async(scene, params, use_blur, host_image, stream);
  if (rc != 0) return rc;
  return rdc_frame_wait(scene);
}

int rdc_image_to_rgba8(const float* image, int width, int height, int flip, uint8_t* out) {
  if (!image || !out || width <= 0 || height <= 0) {
    rdc::set_error("image_to_rgba8: bad argument");
    return RDC_E_INVALID;
  }
  // glfw_events.cpp:73-94: min(v*255, 255) stored to an unsigned char, rows flipped for Orzan saves.
  for (int y = 0; y < height; ++y) {
    const float* src = image + (size_t)4 * width * y;
    uint8_t* dst = out + (size_t)4 * width * (flip ? height - 1 - y : y);
    for (int i = 0; i < 4 * width; ++i) {
      float v = src[i] * 255;
      if (v > 255.0f) v = 255.0f;
      dst[i] = (v == v && v > 0.0f) ? (uint8_t)v : 0;  // NaN (all rays missed) and negatives -> 0
    }
  }
  return 0;
}

int rdc_write_ppm(const char* path, const uint8_t* rgba, int width, int height) {
  if (!path || !rgba || width <= 0 || height <= 0) {
    rdc::set_error("write_ppm: bad argument");
    return RDC_E_INVALID;
  }
  std::FILE* f = std::fopen(path, "wb");
  if (!f) {
    rdc::set_error("write_ppm: cannot open %s", path);
    return RDC_E_IO;
  }
  std::fprintf(f, "P6\n%d %d\n255\n", width, height);
  for (size_t i = 0; i < (size_t)width * height; ++i) std::fwrite(rgba + 4 * i, 1, 3, f);
  bool ok = std::fclose(f) == 0;
  if (!ok) {
    rdc::set_error("write_ppm: write failed for %s", path);
    return RDC_E_IO;
  }
  return 0;
}

}  // extern "C"
