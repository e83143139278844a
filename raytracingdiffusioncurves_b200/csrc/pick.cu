// pick.cu — the curve under a point: nearest chord by a best-first walk of the render's tree (rdc_scene_pick,
// rdc_scene_pick_frame). Read-only over what the build made: chords in leaf runs, the tree over them and the stop tables.
//
// Mapping. The points form gives every point one thread, in the caller's order. The frame form gives every warp one
// 8 x 4 tile of the band (the render kernel's warp tile): the lanes are neighbouring pixels and walk nearly the same
// subtrees. Nothing is persistent and there are no global counters.
//
// Traversal: ordered depth-first search in the shape of render.cu's closest_chord. One node fetch gives both children's
// padded boxes; the child whose box is nearer is entered first and the other goes on a per-thread stack with its box
// distance, so a subtree that a chord found in the meantime has put out of reach is dropped when it is popped. Leaves
// test the up to RDC_RUN chords of a run from its shared end points: chord j joins points j and j + 1, its id is
// first_id + j.
//
// Exactness: the answer is the brute force's lexicographic minimum of (d2, id) over the chords with d2 <= max_distance^2,
// whatever the tree. The best so far starts as (max_distance^2, RDC_PICK_NONE), so rdc_pick_closer accepts exactly
// the chords in range, and a subtree is entered when its box's fp32 squared distance rdc_point_box_d2 is <= the best d2
// (ties are visited). A subtree is dropped only if box_d2 > best, and that never loses a chord that would win or tie:
//   * the point c = a + s e that rdc_point_chord computes for a chord of the subtree lies inside the subtree's padded box.
//     Exactly, c lies on the chord, inside the run's tight box; in fp32 e = b - a, s e and a + s e round once each, which
//     moves c by at most ~5 ulp of the scene's largest coordinate (3e-7 x extent), and the box padding is
//     curve_width + 4e-6 x extent (accel.cu). Inner boxes are unions of padded child boxes (fmin / fmax, exact);
//   * for c inside the box, per axis the true distance from p to the box is at most |cx - px|, and IEEE rounding is
//     monotone: fl(xmin - px) <= fl(cx - px), the same for the squares and their sum. rdc_point_box_d2 is written with
//     the same operations as d2, so box_d2 <= d2 for every chord of the subtree, in fp32, with no further slack;
//   * so box_d2 > best implies d2 > best for all of them: none ties or wins.
// The single-leaf tree's empty right box {+inf, +inf, -inf, -inf} has box_d2 = +inf and is only entered when the bound is
// +inf; it names the same leaf again, and a chord seen twice cannot displace itself.
#include <cmath>

#include "device_scene.h"
#include "rdc_math.h"

namespace rdc {
namespace {

constexpr int kPickBlock = 128;
constexpr int kTileW = 8, kTileH = 4;  // render.cu's warp tile
constexpr int kStack = 64;             // the tree is at most 62 deep (accel.cu)
constexpr uint32_t kNone = RDC_PICK_NONE;
constexpr int kRunVec = sizeof(RunRecord) / 16;
static_assert(sizeof(rdc_pick) == 32, "rdc_pick must stay 32 bytes");

struct PickArgs {
  DevScene sc;
  const float2* points;
  uint32_t n;          // points form: points; frame form: pixels of the band
  rdc_pick* out;
  float4* stops;
  float bound;         // max_distance^2
  int orzan;
  uint32_t width, height, row_begin, rows, tiles_x;  // frame form
  float zoom, off_x, off_y;
};

struct Nearest {
  float d2, s, x, y;
  uint32_t id;
  int run, j;
};

__device__ __forceinline__ void test_chord(float px, float py, float ax, float ay, float bx, float by, uint32_t id, int run, int j,
                                           Nearest& best) {
  float s, x, y, d2;
  rdc_point_chord(px, py, ax, ay, bx, by, &s, &x, &y, &d2);
  if (rdc_pick_closer(d2, id, best.d2, best.id)) best = Nearest{d2, s, x, y, id, run, j};
}

// every chord of run `run` against the point, reading the record two points at a time and only as far as the run is long
__device__ __forceinline__ void test_run(const DevScene& sc, int run, float px, float py, Nearest& best) {
  const float4* rp = reinterpret_cast<const float4*>(sc.runs + run);
  const float4 head = __ldg(rp);
  const uint32_t first_id = __float_as_uint(head.x);
  const int count = (int)__float_as_uint(head.y);
  float ax = head.z, ay = head.w;
#pragma unroll
  for (int v = 1; v < kRunVec; ++v) {
    if (2 * v - 2 >= count) break;
    const float4 q = __ldg(rp + v);
    test_chord(px, py, ax, ay, q.x, q.y, first_id + (uint32_t)(2 * v - 2), run, 2 * v - 2, best);
    if (2 * v - 1 < count) test_chord(px, py, q.x, q.y, q.z, q.w, first_id + (uint32_t)(2 * v - 1), run, 2 * v - 1, best);
    ax = q.z;
    ay = q.w;
  }
}

__device__ __forceinline__ Nearest nearest_chord(const DevScene& sc, float px, float py, float bound) {
  Nearest best{bound, 0.0f, 0.0f, 0.0f, kNone, -1, 0};
  int2 stack[kStack];  // (node, box d2 bits)
  int sp = 0;
  int node = 0;
  constexpr int kDone = 0x7fffffff;
  for (;;) {
    while (node >= 0 && node != kDone) {
      const float4* np = reinterpret_cast<const float4*>(sc.nodes + node);
      const float4 lb = __ldg(np), rb = __ldg(np + 1), ch = __ldg(np + 2);
      const int left = __float_as_int(ch.x), right = __float_as_int(ch.y);
      const float ld = rdc_point_box_d2(px, py, lb.x, lb.y, lb.z, lb.w);
      const float rd = rdc_point_box_d2(px, py, rb.x, rb.y, rb.z, rb.w);
      const bool hl = ld <= best.d2, hr = rd <= best.d2;
      if (hl && hr) {
        const bool left_first = ld <= rd;
        stack[sp++] = make_int2(left_first ? right : left, __float_as_int(left_first ? rd : ld));
        node = left_first ? left : right;
      } else if (hl || hr) {
        node = hl ? left : right;
      } else {
        node = kDone;
      }
      if (node == kDone) {
        while (sp > 0) {  // the nearest pending subtree that is still in reach
          const int2 e = stack[--sp];
          if (__int_as_float(e.y) <= best.d2) {
            node = e.x;
            break;
          }
        }
      }
    }
    if (node == kDone) return best;
    test_run(sc, ~node, px, py, best);
    node = kDone;
    while (sp > 0) {
      const int2 e = stack[--sp];
      if (__int_as_float(e.y) <= best.d2) {
        node = e.x;
        break;
      }
    }
    if (node == kDone) return best;
  }
}

__device__ __forceinline__ float scalar_stop(const DevStops& st, uint32_t first, uint32_t end, float cu) {
  float ratio;
  const int ind = rdc_interp_from(first, end, cu, st.u, &ratio);
  return rdc_lerp_stop(__ldg(st.value + ind), __ldg(st.value + ind + 1), ratio);
}

__device__ __forceinline__ float3 colour_stop(const DevStops& st, uint32_t first, uint32_t end, float cu) {
  float ratio;
  const int ind = rdc_interp_from(first, end, cu, st.u, &ratio);
  const float4 c0 = __ldg(st.rgb + ind), c1 = __ldg(st.rgb + ind + 1);
  return make_float3(rdc_lerp_color(c0.x, c1.x, ratio), rdc_lerp_color(c0.y, c1.y, ratio), rdc_lerp_color(c0.z, c1.z, ratio));
}

// colour of a shading record's two stops {rgb0, u0} {rgb1, u1} at cu (render.cu trace_from, same operations)
__device__ __forceinline__ float3 record_colour(float4 c0, float4 c1, float cu) {
  const float ratio = rdc_ratio(cu - c0.w, c1.w - c0.w);
  return make_float3(rdc_lerp_color(c0.x, c1.x, ratio), rdc_lerp_color(c0.y, c1.y, ratio), rdc_lerp_color(c0.z, c1.z, ratio));
}
__device__ __forceinline__ float record_scalar(float4 r, float cu) { return rdc_lerp_stop(r.z, r.w, rdc_ratio(cu - r.x, r.y - r.x)); }

template <bool STOPS>
__device__ __forceinline__ void pick_point(const PickArgs& a, float px, float py, size_t i) {
  const DevScene& sc = a.sc;
  rdc_pick r;
  const float nan = __int_as_float(0x7fffffff);
  const bool finite = isfinite(px) && isfinite(py);
  const Nearest b = finite ? nearest_chord(sc, px, py, a.bound) : Nearest{0.0f, 0.0f, 0.0f, 0.0f, kNone, -1, 0};
  if (b.id == kNone) {
    r = rdc_pick{kNone, kNone, kNone, 0u, nan, __int_as_float(0x7f800000), nan, nan};
    a.out[i] = r;
    if (STOPS) {
      const float4 m = make_float4(nan, nan, nan, nan);
      a.stops[3 * i] = m;
      a.stops[3 * i + 1] = m;
      a.stops[3 * i + 2] = m;
    }
    return;
  }
  const uint4 id = __ldg(sc.run_ids + b.run);  // first chord id, segment, k of the first chord, K
  const uint32_t seg = id.y;
  const float u = rdc_hit_u((int)id.z + b.j, (int)id.w, b.s);
  const uint4* wp = reinterpret_cast<const uint4*>(sc.seg_walk + seg);
  const uint4 wd = __ldg(wp + 2);
  const uint32_t curve = wd.z, ordinal = wd.w;
  const float cu = u + ordinal;
  const float4* vp = reinterpret_cast<const float4*>(sc.vertices + __ldg(sc.segment_indices + seg));
  const float4 va = __ldg(vp), vb = __ldg(vp + 1);
  const bool right = rdc_is_ray_right(u, b.x - px, b.y - py, rdc_f2{va.x, va.y}, rdc_f2{va.z, va.w}, rdc_f2{vb.x, vb.y},
                                      rdc_f2{vb.z, vb.w}, a.orzan != 0);
  const uint32_t flags = (right ? RDC_PICK_RIGHT : 0u) | (__ldg(sc.curve_connect + curve) >= 0 ? RDC_PICK_PORTAL : 0u);
  r = rdc_pick{b.id, seg, curve, flags, cu, sqrtf(b.d2), b.x, b.y};
  a.out[i] = r;
  if (!STOPS) return;
  float3 left_rgb, right_rgb;
  float blur, weight, degree;
  const float4* rec = sc.chord_records ? sc.chord_records + 8 * (size_t)b.id : nullptr;
  if (rec && (__float_as_uint(__ldg(rec + 7).w) >> 27) == 0x1Fu) {
    // every family stays inside one stop interval over the whole chord: the record holds the two stops (device_scene.h)
    blur = record_scalar(__ldg(rec), cu);
    weight = record_scalar(__ldg(rec + 1), cu);
    degree = record_scalar(__ldg(rec + 2), cu);
    left_rgb = record_colour(__ldg(rec + 3), __ldg(rec + 4), cu);
    right_rgb = record_colour(__ldg(rec + 5), __ldg(rec + 6), cu);
  } else {
    const uint4 wc = __ldg(wp), ws = __ldg(wp + 1);
    const uint4 cw = __ldg(sc.chord_walk + 2 * (size_t)b.id), cw2 = __ldg(sc.chord_walk + 2 * (size_t)b.id + 1);
    left_rgb = colour_stop(sc.color_left, cw.x, wc.y, cu);
    right_rgb = colour_stop(sc.color_right, cw.y, wc.w, cu);
    blur = scalar_stop(sc.blur, cw.z, ws.y, cu);
    weight = scalar_stop(sc.weight, cw.w, ws.w, cu);
    degree = scalar_stop(sc.weight_degree, cw2.x, wd.y, cu);
  }
  a.stops[3 * i] = make_float4(left_rgb.x, left_rgb.y, left_rgb.z, blur);
  a.stops[3 * i + 1] = make_float4(right_rgb.x, right_rgb.y, right_rgb.z, weight);
  a.stops[3 * i + 2] = make_float4(degree, 0.0f, 0.0f, 0.0f);
}

template <bool FRAME, bool STOPS>
__global__ void __launch_bounds__(kPickBlock) k_pick(const PickArgs a) {
  if (!FRAME) {
    const size_t i = (size_t)blockIdx.x * kPickBlock + threadIdx.x;
    if (i >= a.n) return;
    const float2 p = a.points[i];
    pick_point<STOPS>(a, p.x, p.y, i);
    return;
  }
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t tile = blockIdx.x * (kPickBlock / 32) + threadIdx.x / 32u;
  const uint32_t ix = (tile % a.tiles_x) * kTileW + lane % kTileW;
  const uint32_t vy = (tile / a.tiles_x) * kTileH + lane / kTileW;  // row of the band
  if (ix >= a.width || vy >= a.rows) return;
  const uint32_t iy = a.row_begin + vy;
  pick_point<STOPS>(a, rdc_pixel_centre_x(a.width, a.zoom, a.off_x, ix), rdc_pixel_centre_y(a.height, a.zoom, a.off_y, a.orzan != 0, iy),
                    (size_t)vy * a.width + ix);
}

int check_max_distance(float max_distance, const char* who) {
  if (!(max_distance > 0.0f)) {
    set_error("%s: max_distance must be positive (+INF: no limit), got %g", who, (double)max_distance);
    return RDC_E_INVALID;
  }
  return 0;
}

// like a launch: behind the handle's previous launch or update, whatever stream that was on; the next launch waits for it
int launch(rdc_scene* s, PickArgs& a, bool frame, size_t threads, cudaStream_t stream) {
  if (int rc = wait_previous_launch(s, stream)) return rc;
  a.sc = s->dev;
  const unsigned grid = (unsigned)((threads + kPickBlock - 1) / kPickBlock);
  if (frame) {
    if (a.stops) k_pick<true, true><<<grid, kPickBlock, 0, stream>>>(a);
    else k_pick<true, false><<<grid, kPickBlock, 0, stream>>>(a);
  } else {
    if (a.stops) k_pick<false, true><<<grid, kPickBlock, 0, stream>>>(a);
    else k_pick<false, false><<<grid, kPickBlock, 0, stream>>>(a);
  }
  RDC_CUDA(cudaGetLastError());
  return record_launch(s, stream);
}

}  // namespace

int pick(rdc_scene* s, const float* points, uint32_t n, float max_distance, int orzan, rdc_pick* out, float* stops,
         cudaStream_t stream) {
  if (!out || (!points && n > 0)) {
    set_error("pick: null %s", !out ? "out" : "points");
    return RDC_E_INVALID;
  }
  if (int rc = check_max_distance(max_distance, "pick")) return rc;
  if (!s) {
    set_error("pick: null scene");
    return RDC_E_INVALID;
  }
  if (n == 0) return 0;
  PickArgs a{};
  a.points = reinterpret_cast<const float2*>(points);
  a.n = n;
  a.out = out;
  a.stops = reinterpret_cast<float4*>(stops);
  a.bound = max_distance * max_distance;
  a.orzan = orzan;
  return launch(s, a, false, n, stream);
}

int pick_frame(rdc_scene* s, const rdc_frame_params* p, float max_distance, rdc_pick* out, float* stops, cudaStream_t stream) {
  if (!p || !out) {
    set_error("pick frame: null %s", !p ? "params" : "out");
    return RDC_E_INVALID;
  }
  if (int rc = check_max_distance(max_distance, "pick frame")) return rc;
  if (p->image_width == 0 || p->row_begin >= p->row_end || p->row_end > p->image_height) {
    set_error("pick frame: rows [%u,%u) of a %ux%u frame are not a band to pick", p->row_begin, p->row_end, p->image_width,
              p->image_height);
    return RDC_E_INVALID;
  }
  if (p->strip_stride > 1) {
    set_error("pick frame: strips (strip_stride %u) are not supported; pick a contiguous row band", p->strip_stride);
    return RDC_E_INVALID;
  }
  if (!s) {
    set_error("pick frame: null scene");
    return RDC_E_INVALID;
  }
  PickArgs a{};
  a.out = out;
  a.stops = reinterpret_cast<float4*>(stops);
  a.bound = max_distance * max_distance;
  a.orzan = p->use_diffusion_curve_save;
  a.width = p->image_width;
  a.height = p->image_height;
  a.row_begin = p->row_begin;
  a.rows = p->row_end - p->row_begin;
  a.tiles_x = (a.width + kTileW - 1) / kTileW;
  a.n = a.rows * a.width;
  a.zoom = p->zoom_factor;
  a.off_x = p->offset_x;
  a.off_y = p->offset_y;
  const size_t tiles = (size_t)a.tiles_x * ((a.rows + kTileH - 1) / kTileH);
  return launch(s, a, true, tiles * 32, stream);
}

}  // namespace rdc
