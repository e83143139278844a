// oracle_port.cpp — TEST INFRASTRUCTURE: CPU restatement ("port") of the reference's device logic.
//
// Parity status: PINNED against oracle/_ref (the reference's own DeviceCode.cu compiled for the host through
// oracle/shim/, see ref_glue.cpp) for the switch set the reference ships with; the reference itself holds
// no golden vectors or tests (SURVEY.md §4, §8c). Ray/curve intersection parity with the closed OptiX
// intersector is unpinned by construction — see DESIGN.md.
//
// Follows, function by function (paths relative to /root/reference/optixHello):
//   render_pixel      __raygen__rg       DeviceCode.cu:85-182
//   trace (miss)      __miss__ms         DeviceCode.cu:185-192
//   trace (hit)       __closesthit__ch   DeviceCode.cu:194-342, RECURSIVE like the reference (:267-280)
//   oracle_blur       gaussHorizontal / gaussVertical / gaussianBlur   helperKernels.cu:48-148
// Substitutions shared with the product (SURVEY.md §8c): Philox4x32-10 for the per-pixel XORWOW state,
// chord intersection for OptiX's curve intersector — here by brute force over all chords.
// Unlike the reference build (--use_fast_math, CMakeLists.txt:172) everything is IEEE fp32 in source order.
#include <omp.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "oracle_common.h"

namespace {

using oracle::ChordSet;
using oracle::Hit;

struct Ctx {
  const rdc_scene_arrays& a;
  const rdc_frame_params& p;
  const ChordSet& cs;
};

struct Payload {
  float r = 0, g = 0, b = 0, w = 0, blur = 0;
};

struct Stops {
  const uint32_t* index;
  const float* value;
  const float* u;
};

// What a primary ray decided (oracle_ray_records): the closest chord and where on it, the curve, the side. Layout mirrored
// by pyoracle.RAY_RECORD.
struct RayRecord {
  uint32_t id;        // chord id, 0xFFFFFFFF for a miss
  float t;            // ray parameter of the hit (+inf for a miss)
  float segment_u;    // rdc_hit_u of the hit
  uint32_t curve;
  float curve_u;      // segment_u + the segment's ordinal in its curve: the u the stop walks compare
  int32_t right;      // rdc_is_ray_right
  int32_t portal;     // the hit curve connects to another (at depth 0 it shades nothing)
};

float scalar_at(const uint32_t* index, const float* value, const float* us, uint32_t curve, float cu) {
  float ratio;
  int ind = rdc_interp(index[2 * curve], index[2 * curve + 1], cu, us, &ratio);
  return rdc_lerp_stop(value[ind], value[ind + 1], ratio);
}

void colour_at(const uint32_t* index, const float* rgb, const float* us, uint32_t curve, float cu, float out[3]) {
  float ratio;
  int ind = rdc_interp(index[2 * curve], index[2 * curve + 1], cu, us, &ratio);
  for (int c = 0; c < 3; ++c) out[c] = rdc_lerp_color(rgb[3 * ind + c], rgb[3 * (ind + 1) + c], ratio);
}

// optixTrace + closest-hit / miss programs. `depth` is payload p5.
Payload trace(const Ctx& c, float ox, float oy, float dx, float dy, unsigned depth, uint32_t skip_lo, uint32_t skip_hi,
              RayRecord* rec) {
  const rdc_scene_arrays& a = c.a;
  Hit h = oracle::closest_hit(c.cs, ox, oy, dx, dy, depth == 0, skip_lo, skip_hi);
  if (rec) *rec = RayRecord{h.id, h.t, 0.0f, 0u, 0.0f, 0, 0};
  Payload out;
  if (!h.valid()) return out;  // miss: all zero
  const oracle::Chord& ch = c.cs.chords[h.id];
  const uint32_t seg = ch.seg;
  const float segment_u = rdc_hit_u(ch.k, ch.K, h.s);
  const float rt = h.t;
  const uint32_t curve = a.curve_map[seg];
  const float curve_u = segment_u + a.curve_index[seg];

  const float blur = scalar_at(a.blur_index, a.blur, a.blur_u, curve, curve_u);
  const float weight_multiplier = scalar_at(a.weight_index, a.weight, a.weight_u, curve, curve_u);
  const float weight_degree = scalar_at(a.weight_degree_index, a.weight_degree, a.weight_degree_u, curve, curve_u);
  rdc_f2 v[4];
  oracle::control_points(a, seg, v);
  const bool right = rdc_is_ray_right(segment_u, dx, dy, v[0], v[1], v[2], v[3], c.p.use_diffusion_curve_save != 0);
  if (rec) *rec = RayRecord{h.id, rt, segment_u, curve, curve_u, right ? 1 : 0, a.curve_connect[curve] >= 0 ? 1 : 0};

  if (a.curve_connect[curve] >= 0) {
    const unsigned next_depth = depth + 1;
    if (next_depth > (unsigned)c.p.max_trace_depth) return out;  // depth cap = miss
    const uint32_t target = a.curve_map_inverse[a.curve_connect[curve]] + a.curve_index[seg];
    rdc_f2 tv[4];
    oracle::control_points(a, target, tv);
    const rdc_f2 origin = rdc_spline_point(segment_u, tv[0], tv[1], tv[2], tv[3]);
    rdc_f2 n = rdc_spline_normal(segment_u, v[0], v[1], v[2], v[3]);
    const float n_len = sqrtf(n.x * n.x + n.y * n.y);
    n.x /= n_len;
    n.y /= n_len;
    const float ray_cos = n.x * dx + n.y * dy;
    const float ray_sin = n.x * dy + n.y * dx;  // the reference's expression, not a cross product (:243)
    rdc_f2 m = rdc_spline_normal(segment_u, tv[0], tv[1], tv[2], tv[3]);
    const float m_len = sqrtf(m.x * m.x + m.y * m.y);
    m.x /= m_len;
    m.y /= m_len;
    const float ndx = m.x * ray_cos - m.y * ray_sin;
    const float ndy = m.y * ray_cos + m.x * ray_sin;
    int klo, khi;
    rdc_portal_skip(segment_u, (int)(c.cs.seg_base[target + 1] - c.cs.seg_base[target]), &klo, &khi);
    Payload in = trace(c, origin.x, origin.y, ndx, ndy, next_depth, c.cs.seg_base[target] + (uint32_t)klo,
                       c.cs.seg_base[target] + (uint32_t)khi, nullptr);
    float filter[3];
    if (right) colour_at(a.color_right_index, a.color_right, a.color_right_u, curve, curve_u, filter);
    else colour_at(a.color_right_index, a.color_left, a.color_left_u, curve, curve_u, filter);  // :297 uses the right index
    out.r = filter[0] * in.r;
    out.g = filter[1] * in.g;
    out.b = filter[2] * in.b;
    out.w = 1 / ((1 / in.w) + 1 / (weight_multiplier * powf(rt, -weight_degree)));
    out.blur = blur * in.blur;
    return out;
  }
  out.w = weight_multiplier * powf(rt, -weight_degree);
  out.blur = blur;
  float rgb[3];
  if (right) colour_at(a.color_right_index, a.color_right, a.color_right_u, curve, curve_u, rgb);
  else colour_at(a.color_left_index, a.color_left, a.color_left_u, curve, curve_u, rgb);
  out.r = rgb[0];
  out.g = rgb[1];
  out.b = rgb[2];
  return out;
}

void render_pixel(const Ctx& c, uint32_t ix, uint32_t iy, uint32_t local_row, float* image, float* blur_map,
                  uint32_t* hit_ids, RayRecord* records) {
  const rdc_frame_params& p = c.p;
  const float N = p.number_of_rays_per_pixel;
  float rot_sin, rot_cos;
  rdc_sincospi(2 / N, &rot_sin, &rot_cos);
  const float origin_x = ((int)(ix - (p.image_width / 2))) * p.zoom_factor + p.offset_x;
  const float origin_y = p.use_diffusion_curve_save
                             ? ((int)((p.image_height - iy) - (p.image_height / 2))) * p.zoom_factor + p.offset_y
                             : ((int)(iy - (p.image_height / 2))) * p.zoom_factor + p.offset_y;
  float dir_x = 1, dir_y = 0;
  float color[3] = {0, 0, 0}, blur = 0, weight_total = 0;
  const uint32_t pixel = iy * p.image_width + ix;
  const size_t local = (size_t)local_row * p.image_width + ix;
  const int n_iter = (int)ceilf(N);
  for (int i = 0; i < N; i++) {
    const rdc_u4 rnd = rdc_philox4x32_10(pixel, (uint32_t)i, 0u, 0u, p.seed, p.frame);
    float rs, rc;
    rdc_sincospi((2 / N) * rdc_u01(rnd.x), &rs, &rc);
    const float jx = dir_x * rc - dir_y * rs;
    const float jy = dir_x * rs + dir_y * rc;
    const float ox = origin_x + (p.use_aa ? (rdc_u01(rnd.y) * p.zoom_factor) : 0);
    const float oy = origin_y + (p.use_aa ? (rdc_u01(rnd.z) * p.zoom_factor) : 0);
    RayRecord rec;
    Payload s = trace(c, ox, oy, p.use_aa ? jx : dir_x, p.use_aa ? jy : dir_y, 0, 1, 0, &rec);
    if (hit_ids) hit_ids[local * n_iter + i] = rec.id;
    if (records) records[local * n_iter + i] = rec;
    weight_total += s.w;
    color[0] += s.r * s.w;
    color[1] += s.g * s.w;
    color[2] += s.b * s.w;
    blur += s.blur * s.w;
    const float nx = dir_x * rot_cos - dir_y * rot_sin;
    const float ny = dir_x * rot_sin + dir_y * rot_cos;
    dir_x = nx;
    dir_y = ny;
  }
  image[4 * local + 0] = color[0] / weight_total;
  image[4 * local + 1] = color[1] / weight_total;
  image[4 * local + 2] = color[2] / weight_total;
  image[4 * local + 3] = 1.0f;  // the reference leaves .w unwritten (DeviceCode.cu:176-178)
  blur_map[local] = blur / weight_total;
}

}  // namespace

namespace {
int g_search = 0;  // 0: every chord per ray; 1: through the uniform grid of oracle_common.h (same answer, checked in tests/)

// rows of the band, or (strip_stride > 1) the strips t % stride == offset of it, packed (rdc_b200.h)
std::vector<uint32_t> band_rows(const rdc_frame_params& p) {
  const uint32_t stride = p.strip_stride > 1 ? p.strip_stride : 1, offset = p.strip_stride > 1 ? p.strip_offset : 0;
  std::vector<uint32_t> rows;
  for (uint32_t iy = p.row_begin; iy < p.row_end; ++iy)
    if (((iy - p.row_begin) / RDC_STRIP_ROWS) % stride == offset) rows.push_back(iy);
  return rows;
}

void render_band(const rdc_scene_arrays* a, const rdc_accel_options* o, const rdc_frame_params* p, float* image,
                 float* blur_map, uint32_t* hit_ids, RayRecord* records, int threads) {
  ChordSet cs = oracle::build_chords(*a, *o);
  if (g_search == 1) oracle::build_grid(cs);
  Ctx c{*a, *p, cs};
  if (threads <= 0) threads = omp_get_max_threads();
  const uint32_t stride = p->strip_stride > 1 ? p->strip_stride : 1;
  const std::vector<uint32_t> rows = band_rows(*p);
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads)
  for (size_t r = 0; r < rows.size(); ++r) {
    const uint32_t iy = rows[r];
    const uint32_t rel = iy - p->row_begin;
    const uint32_t local_row = (rel / RDC_STRIP_ROWS / stride) * RDC_STRIP_ROWS + rel % RDC_STRIP_ROWS;
    for (uint32_t ix = 0; ix < p->image_width; ++ix) render_pixel(c, ix, iy, local_row, image, blur_map, hit_ids, records);
  }
}
}  // namespace

extern "C" {

int oracle_threads(void) { return omp_get_max_threads(); }
void oracle_set_search(int mode) { g_search = mode; }

// chord list in original order; geom = 4 floats, ids = 3 uint32 (segment, k, K) per chord.
// Call with geom == NULL to get the count.
int oracle_chords(const rdc_scene_arrays* a, const rdc_accel_options* o, float* geom, uint32_t* ids, uint32_t* n) {
  ChordSet cs = oracle::build_chords(*a, *o);
  *n = (uint32_t)cs.chords.size();
  if (!geom) return 0;
  for (size_t i = 0; i < cs.chords.size(); ++i) {
    const oracle::Chord& c = cs.chords[i];
    geom[4 * i] = c.ax; geom[4 * i + 1] = c.ay; geom[4 * i + 2] = c.bx; geom[4 * i + 3] = c.by;
    ids[3 * i] = c.seg; ids[3 * i + 1] = (uint32_t)c.k; ids[3 * i + 2] = (uint32_t)c.K;
  }
  return 0;
}

// image = float4[rows*W], blur_map = float[rows*W], hit_ids optional [rows*W*ceil(N)]; rows = band of params
int oracle_render(const rdc_scene_arrays* a, const rdc_accel_options* o, const rdc_frame_params* p, float* image,
                  float* blur_map, uint32_t* hit_ids, int threads) {
  render_band(a, o, p, image, blur_map, hit_ids, nullptr, threads);
  return 0;
}

// The frame's primary rays as render_pixel traces them (same draws, rotation, jitter and closest hit): records =
// RayRecord[rows*W*ceil(N)], laid out like hit_ids. A portal hit is recorded as the primary ray's hit, whatever lies
// behind the portal.
int oracle_ray_records(const rdc_scene_arrays* a, const rdc_accel_options* o, const rdc_frame_params* p, void* records,
                       int threads) {
  const size_t pixels = band_rows(*p).size() * (size_t)p->image_width;
  std::vector<float> image(4 * pixels), blur_map(pixels);
  render_band(a, o, p, image.data(), blur_map.data(), nullptr, static_cast<RayRecord*>(records), threads);
  return 0;
}

// Closest hit of arbitrary primary rays (rays = n x {ox, oy, dx, dy}); id = chord id or 0xFFFFFFFF, t = ray
// parameter, u = segment parameter of the hit ((k + s) / K). Feeds the geometry check of the chord intersector
// against a double-precision ray/B-spline root (tests/test_intersector_geometry_cpu.py).
int oracle_trace_rays(const rdc_scene_arrays* a, const rdc_accel_options* o, const float* rays, uint32_t n, uint32_t* id,
                      float* t, float* u) {
  ChordSet cs = oracle::build_chords(*a, *o);
  if (g_search == 1) oracle::build_grid(cs);
#pragma omp parallel for schedule(dynamic, 256)
  for (uint32_t i = 0; i < n; ++i) {
    const Hit h = oracle::closest_hit(cs, rays[4 * i], rays[4 * i + 1], rays[4 * i + 2], rays[4 * i + 3], true, 1u, 0u);
    id[i] = h.id;
    t[i] = h.t;
    u[i] = h.valid() ? rdc_hit_u(cs.chords[h.id].k, cs.chords[h.id].K, h.s) : 0.0f;
  }
  return 0;
}

// helperKernels.cu:48-148, in-place capable. image = float4[w*h].
int oracle_blur(float* dest, const float* source, const float* sigma, int width, int height, int threads) {
  const float MINUM_SIGMA = 1e-6f;
  std::vector<float> tmp((size_t)4 * width * height);
  if (threads <= 0) threads = omp_get_max_threads();
  for (int pass = 0; pass < 2; ++pass) {
    const float* src = pass == 0 ? source : tmp.data();
    float* dst = pass == 0 ? tmp.data() : dest;
#pragma omp parallel for schedule(dynamic, 4) num_threads(threads)
    for (int y = 0; y < height; ++y)
      for (int x = 0; x < width; ++x) {
        const int i = y * width + x;
        float accum = 0;
        const float k_size = 2 * ceilf(3 * sigma[i]) + 1;
        const float sig_square = (sigma[i] + MINUM_SIGMA) * (sigma[i] + MINUM_SIGMA);
        float d[4] = {0, 0, 0, 0};
        if (k_size == k_size && k_size < 65536.0f) {  // NaN sigma: no tap runs in the reference either
          for (int k_i = -k_size / 2; k_i <= (k_size / 2); k_i++) {
            const int loc = pass == 0 ? std::max(0, std::min(i % width + k_i, width - 1)) + (i / width) * width
                                      : std::max(i % width, std::min(i + k_i * width, (height - 1) * width + (i % width)));
            const float g = expf(-(k_i * k_i) / sig_square);
            accum += g;
            for (int ch = 0; ch < 4; ++ch) d[ch] += src[4 * loc + ch] * g;
          }
        }
        for (int ch = 0; ch < 4; ++ch) dst[4 * i + ch] = d[ch] / accum;
      }
  }
  return 0;
}

}  // extern "C"
