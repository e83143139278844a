// accel.cu — scene upload + on-GPU acceleration structure.
//
// Replaces the reference's per-array uploads (optixHello.cpp:524-762) and the closed
// optixAccelBuild over round cubic B-spline primitives (optixHello.cpp:765-830):
//   1. every spline segment is cut into K parameter-uniform chords, K from a flatness bound
//      (rdc_chord_count), end points evaluated with the bit-exact spline of rdc_math.h;
//   2. consecutive chords of a segment are grouped into runs of up to RDC_RUN chords (RDC_RUN+1 points:
//      shared end points are stored once); a run is the tree's leaf primitive;
//   3. runs are ordered by the 32-bit Morton code of their box centre (cub radix sort);
//   4. a binary radix tree is built over the sorted codes (Karras 2012), boxes are fitted bottom-up with
//      one atomic counter per inner node, each node ends up holding both children's padded boxes.
// The chord's ORIGINAL id (segment order, then k) is what hit parity is defined on; runs and Morton order
// are only a memory layout.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <limits>
#include <algorithm>
#include <vector>

#include "device_scene.h"
#include "rdc_math.h"

namespace rdc {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof g_error, fmt, ap);
  va_end(ap);
}
const char* last_error() { return g_error; }

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return (int)e;
}

namespace {

constexpr int kThreads = 256;
inline unsigned blocks_for(size_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

struct Bounds {
  float xmin, ymin, xmax, ymax;
};

__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
  if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  if (v >= 0.0f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__device__ __forceinline__ void load_segment(const float2* vertices, uint32_t first, rdc_f2 v[4]) {
  const float4* p = reinterpret_cast<const float4*>(vertices + first);  // first % 4 == 0 -> 32-byte aligned
  float4 a = __ldg(p), b = __ldg(p + 1);
  v[0] = {a.x, a.y};
  v[1] = {a.z, a.w};
  v[2] = {b.x, b.y};
  v[3] = {b.z, b.w};
}

__global__ void k_chord_counts(const float2* vertices, const uint32_t* segment_indices, uint32_t n_segments, float tol,
                               int kmax, uint32_t* counts) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segments) return;
  rdc_f2 v[4];
  load_segment(vertices, segment_indices[s], v);
  counts[s] = (uint32_t)rdc_chord_count(v[0], v[1], v[2], v[3], tol, kmax);
}

__global__ void k_emit_chords(const float2* vertices, const uint32_t* segment_indices, const uint32_t* base,
                              uint32_t n_segments, uint32_t n_chords, float4* geom, uint4* ids, Bounds* bounds) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_chords) return;
  // segment = last s with base[s] <= c
  uint32_t lo = 0, hi = n_segments;
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (base[mid] <= c) lo = mid; else hi = mid;
  }
  uint32_t seg = lo;
  int k = (int)(c - base[seg]);
  int K = (int)(base[seg + 1] - base[seg]);
  rdc_f2 v[4];
  load_segment(vertices, segment_indices[seg], v);
  rdc_f2 a = rdc_spline_point(rdc_chord_u(k, K), v[0], v[1], v[2], v[3]);
  rdc_f2 b = rdc_spline_point(rdc_chord_u(k + 1, K), v[0], v[1], v[2], v[3]);
  geom[c] = make_float4(a.x, a.y, b.x, b.y);
  ids[c] = make_uint4(c, seg, (uint32_t)k, (uint32_t)K);
  atomic_min_float(&bounds->xmin, fminf(a.x, b.x));
  atomic_min_float(&bounds->ymin, fminf(a.y, b.y));
  atomic_max_float(&bounds->xmax, fmaxf(a.x, b.x));
  atomic_max_float(&bounds->ymax, fmaxf(a.y, b.y));
}

__device__ __forceinline__ uint32_t spread16(uint32_t x) {
  x &= 0xFFFFu;
  x = (x | (x << 8)) & 0x00FF00FFu;
  x = (x | (x << 4)) & 0x0F0F0F0Fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}

__global__ void k_run_counts(const uint32_t* chord_counts, uint32_t n_segments, uint32_t run_len, uint32_t* run_counts) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_segments) run_counts[s] = (chord_counts[s] + run_len - 1) / run_len;
}

// one thread per run (original order): points, ids, tight box, Morton code of the box centre
__global__ void k_emit_runs(const float4* chord_geom, const uint32_t* chord_base, const uint32_t* run_base,
                            uint32_t n_segments, uint32_t n_runs, uint32_t run_len, Bounds b, RunRecord* runs, uint4* run_ids,
                            float4* run_box, uint32_t* codes, uint32_t* order) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_runs) return;
  uint32_t lo = 0, hi = n_segments;
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (run_base[mid] <= r) lo = mid; else hi = mid;
  }
  const uint32_t seg = lo;
  const uint32_t K = chord_base[seg + 1] - chord_base[seg];
  const uint32_t k_first = (r - run_base[seg]) * run_len;
  const uint32_t count = min(run_len, K - k_first);
  const uint32_t first = chord_base[seg] + k_first;
  RunRecord rec;
  float4 g = chord_geom[first];
  float xmin = g.x, xmax = g.x, ymin = g.y, ymax = g.y;
  rec.pts[0] = g.x;
  rec.pts[1] = g.y;
  float lx = g.x, ly = g.y;
#pragma unroll
  for (uint32_t j = 0; j < RDC_RUN; ++j) {
    if (j < count) {
      g = chord_geom[first + j];
      lx = g.z;
      ly = g.w;
      xmin = fminf(xmin, lx); xmax = fmaxf(xmax, lx);
      ymin = fminf(ymin, ly); ymax = fmaxf(ymax, ly);
    }
    rec.pts[2 * j + 2] = lx;  // unused slots repeat the last point
    rec.pts[2 * j + 3] = ly;
  }
  rec.first_id = first;
  rec.count = count;
  runs[r] = rec;
  run_ids[r] = make_uint4(first, seg, k_first, K);
  run_box[r] = make_float4(xmin, ymin, xmax, ymax);
  float cx = 0.5f * (xmin + xmax), cy = 0.5f * (ymin + ymax);
  float ex = fmaxf(b.xmax - b.xmin, 1e-20f), ey = fmaxf(b.ymax - b.ymin, 1e-20f);
  float nx = fminf(fmaxf((cx - b.xmin) / ex, 0.0f), 1.0f);
  float ny = fminf(fmaxf((cy - b.ymin) / ey, 0.0f), 1.0f);
  codes[r] = spread16((uint32_t)(nx * 65535.0f)) | (spread16((uint32_t)(ny * 65535.0f)) << 1);
  order[r] = r;
}

__global__ void k_gather_runs(const uint32_t* order, const RunRecord* runs_in, const uint4* ids_in, const float4* box_in,
                              uint32_t n, RunRecord* runs, uint4* ids, float4* box) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t src = order[i];
  runs[i] = runs_in[src];
  ids[i] = ids_in[src];
  box[i] = box_in[src];
}

// length of the common prefix of the (code, position) keys i and j; -1 outside the array
__device__ __forceinline__ int prefix_len(const uint32_t* codes, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  uint32_t a = codes[i], b = codes[j];
  if (a == b) return 32 + __clz((uint32_t)i ^ (uint32_t)j);
  return __clz(a ^ b);
}

__global__ void k_radix_tree(const uint32_t* codes, int n, BvhNode* nodes, int* leaf_parent) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  int d = (prefix_len(codes, n, i, i + 1) - prefix_len(codes, n, i, i - 1)) >= 0 ? 1 : -1;
  int dmin = prefix_len(codes, n, i, i - d);
  int lmax = 2;
  while (prefix_len(codes, n, i, i + lmax * d) > dmin) lmax <<= 1;
  int l = 0;
  for (int t = lmax >> 1; t >= 1; t >>= 1)
    if (prefix_len(codes, n, i, i + (l + t) * d) > dmin) l += t;
  int j = i + l * d;
  int dnode = prefix_len(codes, n, i, j);
  int s = 0;
  for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
    if (prefix_len(codes, n, i, i + (s + t) * d) > dnode) s += t;
    if (t == 1) break;
  }
  int gamma = i + s * d + min(d, 0);
  int lo = min(i, j), hi = max(i, j);
  int left = (lo == gamma) ? ~gamma : gamma;
  int right = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
  nodes[i].left = left;
  nodes[i].right = right;
  nodes[i].pad = 0;
  if (i == 0) nodes[i].parent = -1;
  if (left < 0) leaf_parent[gamma] = i; else nodes[left].parent = i;
  if (right < 0) leaf_parent[gamma + 1] = i; else nodes[right].parent = i;
}

__device__ __forceinline__ float4 padded(float4 b, float pad) {
  return make_float4(b.x - pad, b.y - pad, b.z + pad, b.w + pad);
}
__device__ __forceinline__ float4 box_union(float4 a, float4 b) {
  return make_float4(fminf(a.x, b.x), fminf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}

// Bottom-up fit. The second thread to reach a node owns it: both children are complete by then.
__global__ void k_fit_boxes(const float4* leaf_box, int n, float pad, const int* leaf_parent, BvhNode* nodes,
                            float4* node_box, unsigned int* arrivals) {
  int leaf = blockIdx.x * blockDim.x + threadIdx.x;
  if (leaf >= n) return;
  int node = leaf_parent[leaf];
  while (node >= 0) {
    __threadfence();
    if (atomicAdd(&arrivals[node], 1u) == 0u) return;
    __threadfence();
    int l = nodes[node].left, r = nodes[node].right;
    float4 lb = l < 0 ? padded(leaf_box[~l], pad) : __ldcg(&node_box[l]);  // L2: written by another SM
    float4 rb = r < 0 ? padded(leaf_box[~r], pad) : __ldcg(&node_box[r]);
    nodes[node].lbox = lb;
    nodes[node].rbox = rb;
    node_box[node] = box_union(lb, rb);
    node = nodes[node].parent;
  }
}

// Also sums the padded boxes' widths and heights (fixed point, 1/1024: integer atomics keep the sums — and
// everything derived from them — independent of the order of arrival) for the render's local-table radius.
__global__ void k_pad_boxes(const float4* leaf_box, uint32_t n, float pad, float4* out, unsigned long long* extent_sums) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long w = 0, h = 0;
  if (i < n) {
    const float4 b = padded(leaf_box[i], pad);
    out[i] = b;
    w = (unsigned long long)fminf((b.z - b.x) * 1024.0f, 4e18f);
    h = (unsigned long long)fminf((b.w - b.y) * 1024.0f, 4e18f);
  }
  for (int o = 16; o > 0; o >>= 1) {
    w += __shfl_down_sync(0xFFFFFFFFu, w, o);
    h += __shfl_down_sync(0xFFFFFFFFu, h, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(extent_sums, w);
    atomicAdd(extent_sums + 1, h);
  }
}

__global__ void k_single_leaf_root(const float4* leaf_box, float pad, BvhNode* nodes) {
  const float inf = __int_as_float(0x7f800000);
  nodes[0].lbox = padded(leaf_box[0], pad);
  nodes[0].rbox = make_float4(inf, inf, -inf, -inf);  // a placeholder: pick's box distance is +inf; the render's fused slab
                                                      // test would enter it, so closest_chord tests the one run directly
  nodes[0].left = ~0;
  nodes[0].right = ~0;
  nodes[0].parent = -1;
  nodes[0].pad = 0;
}

__global__ void k_depth(const int* leaf_parent, const BvhNode* nodes, int n, unsigned int* max_depth) {
  int leaf = blockIdx.x * blockDim.x + threadIdx.x;
  if (leaf >= n) return;
  unsigned int depth = 0;
  for (int node = leaf_parent[leaf]; node >= 0; node = nodes[node].parent) ++depth;
  atomicMax(max_depth, depth);
}

__global__ void k_fill(float* dest, unsigned int n, float v) {
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += blockDim.x * gridDim.x) dest[i] = v;
}

// ---- stop tables (device_scene.h: SegWalk, chord_walk, chord_records) from the stop lists on the device ------------------
// Threads [0, n_segments) write one segment's SegWalk each; the next n_chords threads one chord's walk starts and, when
// `records` is set, its shading record.
//
// A walk over a list [start, end) of parameters u stands at W(x) = the first j >= start with j == end || !(u[j+1] < x)
// once it has consumed every stop below x. A scan that starts anywhere in [start, W(x)] ends at W(x): no j before W(x)
// stops it. For x <= y, every j that stops the walk at y also stops it at x, so W is non-decreasing in x, whether or not
// u is sorted. A chord's walks stand at W(cu_min), cu_min = rdc_hit_u(k, K, 0) + ordinal, which is non-decreasing in k
// (IEEE rounding is monotone) and at least the ordinal, where the segment's hint W(ordinal) stands. So a scan from the
// list's start, from the segment's hint or from the previous chord's result all end at the same j: each chord scans from
// the list's start on its own thread and finds what a sequential loop continuing from the previous chord finds.
constexpr int kWalks = 6;  // chord_walk order: left, right, blur, weight, exponent, portal-left

struct Walks {
  const uint2* index[kWalks];
  const float* u[kWalks];
};

__device__ __forceinline__ Walks walks_of(const DevScene& d) {
  // the portal-left walk takes the right list's range on the LEFT u array (DeviceCode.cu:297)
  return Walks{{d.color_left.index, d.color_right.index, d.blur.index, d.weight.index, d.weight_degree.index, d.color_right.index},
               {d.color_left.u, d.color_right.u, d.blur.u, d.weight.u, d.weight_degree.u, d.color_left.u}};
}

__global__ void __launch_bounds__(kThreads) k_stop_tables(const DevScene d, uint4* seg_walk, uint4* chord_walk, uint4* records) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const Walks w = walks_of(d);
  if (i < d.n_segments) {
    const uint32_t c = __ldg(d.curve_map + i), ordinal = __ldg(d.curve_index + i);
    uint32_t first[kWalks], end[kWalks];
#pragma unroll
    for (int f = 0; f < kWalks; ++f) {
      const uint2 r = __ldg(w.index[f] + c);
      first[f] = rdc_walk_hint(r.x, r.y, (float)ordinal, w.u[f]);
      end[f] = r.x + r.y;
    }
    uint4* out = seg_walk + 4 * (size_t)i;  // SegWalk field order; the pad words are zero
    out[0] = make_uint4(first[0], end[0], first[1], end[1]);
    out[1] = make_uint4(first[2], end[2], first[3], end[3]);
    out[2] = make_uint4(first[4], end[4], c, ordinal);
    out[3] = make_uint4(first[5], end[5], 0u, 0u);
    return;
  }
  const uint32_t ch = i - d.n_segments;
  if (ch >= d.n_chords) return;
  const uint4 id = __ldg(d.chord_ids + ch);  // chord id, segment, k, K
  const uint32_t sg = id.y, c = __ldg(d.curve_map + sg), ordinal = __ldg(d.curve_index + sg);
  const int k = (int)id.z, K = (int)id.w;
  const float cu_min = rdc_hit_u(k, K, 0.0f) + ordinal;
  uint32_t f[kWalks];
#pragma unroll
  for (int fam = 0; fam < kWalks; ++fam) {
    const uint2 r = __ldg(w.index[fam] + c);
    f[fam] = rdc_walk_hint(r.x, r.y, cu_min, w.u[fam]);
  }
  chord_walk[2 * (size_t)ch] = make_uint4(f[0], f[1], f[2], f[3]);
  chord_walk[2 * (size_t)ch + 1] = make_uint4(f[4], f[5], 0u, 0u);
  if (!records) return;
  // the largest parameter a hit on this chord can have: s = 1 (rounding is monotone, so every hit lies in between)
  const float cu_max = rdc_hit_u(k, K, 1.0f) + ordinal;
  uint32_t flags = 0;
#pragma unroll
  for (int fam = 0; fam < 5; ++fam) {  // family `fam` is simple when the walk would not step even at cu_max
    const uint2 r = __ldg(w.index[fam] + c);
    if (!(f[fam] < r.x + r.y && __ldg(w.u[fam] + f[fam] + 1) < cu_max)) flags |= 1u << fam;
  }
  float4* rec = reinterpret_cast<float4*>(records) + 8 * (size_t)ch;
  const float* scalar_v[3] = {d.blur.value, d.weight.value, d.weight_degree.value};
#pragma unroll
  for (int sf = 0; sf < 3; ++sf) {  // blur, weight, exponent: families 2, 3, 4
    const uint32_t j = f[2 + sf];
    const float* us = w.u[2 + sf];
    rec[sf] = make_float4(__ldg(us + j), __ldg(us + j + 1), __ldg(scalar_v[sf] + j), __ldg(scalar_v[sf] + j + 1));
  }
  const float4* rgb[2] = {d.color_left.rgb, d.color_right.rgb};
#pragma unroll
  for (int side = 0; side < 2; ++side) {  // left, right colour: families 0, 1
    const uint32_t j = f[side];
    const float4 c0 = __ldg(rgb[side] + j), c1 = __ldg(rgb[side] + j + 1);
    rec[3 + 2 * side] = make_float4(c0.x, c0.y, c0.z, __ldg(w.u[side] + j));
    rec[4 + 2 * side] = make_float4(c1.x, c1.y, c1.z, __ldg(w.u[side] + j + 1));
  }
  uint4 meta = make_uint4(sg, ordinal, (uint32_t)k | ((uint32_t)K << 16), (c & 0x07FFFFFFu) | (flags << 27));
  if (K > 0xFFFF || c > 0x07FFFFFFu) meta.w &= 0x07FFFFFFu;  // does not fit the packing: never simple
  records[8 * (size_t)ch + 7] = meta;
}

// Where each stop array sits in the stop block (rdc_scene::stops). Per family: the {start,count} pairs, the parameters
// and the values (colours widened to float4 with w = 0), each at a 128-byte boundary. Both colour families hold
// max(n_color_left, n_color_right) + 2 stops, the scalar families n + 2 (the sentinels of rdc_scene_arrays).
struct StopLayout {
  size_t index[5], u[5], value[5], len[5];
  size_t bytes;
};

StopLayout stop_layout(const rdc_scene_arrays& a) {
  const uint32_t n[5] = {a.n_color_left, a.n_color_right, a.n_blur, a.n_weight, a.n_weight_degree};
  StopLayout L{};
  size_t at = 0;
  auto place = [&](size_t bytes) {
    const size_t here = at;
    at = (at + bytes + 127) & ~(size_t)127;
    return here;
  };
  for (int f = 0; f < 5; ++f) {
    const bool colour = f < 2;
    L.len[f] = colour ? (size_t)std::max(a.n_color_left, a.n_color_right) + 2 : (size_t)n[f] + 2;
    L.index[f] = place((size_t)2 * a.n_curves * sizeof(uint32_t));
    L.u[f] = place(L.len[f] * sizeof(float));
    L.value[f] = place(L.len[f] * (colour ? sizeof(float4) : sizeof(float)));
  }
  L.bytes = at;
  return L;
}

void pack_stops(const rdc_scene_arrays& a, const StopLayout& L, void* dst) {
  char* base = static_cast<char*>(dst);
  const uint32_t* index[5] = {a.color_left_index, a.color_right_index, a.blur_index, a.weight_index, a.weight_degree_index};
  const float* value[5] = {a.color_left, a.color_right, a.blur, a.weight, a.weight_degree};
  const float* u[5] = {a.color_left_u, a.color_right_u, a.blur_u, a.weight_u, a.weight_degree_u};
  for (int f = 0; f < 5; ++f) {
    std::memcpy(base + L.index[f], index[f], (size_t)2 * a.n_curves * sizeof(uint32_t));
    std::memcpy(base + L.u[f], u[f], L.len[f] * sizeof(float));
    if (f < 2) {
      float4* c4 = reinterpret_cast<float4*>(base + L.value[f]);
      for (size_t i = 0; i < L.len[f]; ++i) c4[i] = make_float4(value[f][3 * i], value[f][3 * i + 1], value[f][3 * i + 2], 0.0f);
    } else {
      std::memcpy(base + L.value[f], value[f], L.len[f] * sizeof(float));
    }
  }
}

void point_stops(DevScene& d, void* block, const StopLayout& L) {
  const char* base = static_cast<const char*>(block);
  DevStops* st[5] = {&d.color_left, &d.color_right, &d.blur, &d.weight, &d.weight_degree};
  for (int f = 0; f < 5; ++f) {
    *st[f] = DevStops{};
    st[f]->index = reinterpret_cast<const uint2*>(base + L.index[f]);
    st[f]->u = reinterpret_cast<const float*>(base + L.u[f]);
    if (f < 2) st[f]->rgb = reinterpret_cast<const float4*>(base + L.value[f]);
    else st[f]->value = reinterpret_cast<const float*>(base + L.value[f]);
  }
}

// The checks every stop list passes before it reaches the device, in rdc_accel_build and rdc_scene_update_stops alike.
int check_stops(const rdc_scene_arrays& a, const char* who) {
  const uint32_t* idx[5] = {a.color_left_index, a.color_right_index, a.blur_index, a.weight_index, a.weight_degree_index};
  const float* value[5] = {a.color_left, a.color_right, a.blur, a.weight, a.weight_degree};
  const float* u[5] = {a.color_left_u, a.color_right_u, a.blur_u, a.weight_u, a.weight_degree_u};
  const uint32_t cnt[5] = {a.n_color_left, a.n_color_right, a.n_blur, a.n_weight, a.n_weight_degree};
  for (int f = 0; f < 5; ++f) {
    if (!idx[f] || !value[f] || !u[f]) {
      set_error("%s: stop list %d has a null array", who, f);
      return RDC_E_INVALID;
    }
    for (uint32_t c = 0; c < a.n_curves; ++c)
      if ((uint64_t)idx[f][2 * c] + idx[f][2 * c + 1] > cnt[f]) {
        set_error("%s: stop list %d of curve %u runs past its array", who, f, c);
        return RDC_E_INVALID;
      }
  }
  return 0;
}

int launch_stop_tables(const rdc_scene* s, cudaStream_t stream) {
  const DevScene& d = s->dev;
  k_stop_tables<<<blocks_for((size_t)d.n_segments + d.n_chords), kThreads, 0, stream>>>(
      d, const_cast<uint4*>(reinterpret_cast<const uint4*>(d.seg_walk)), const_cast<uint4*>(d.chord_walk),
      const_cast<uint4*>(reinterpret_cast<const uint4*>(d.chord_records)));
  RDC_CUDA(cudaGetLastError());
  return 0;
}

struct Uploader {
  rdc_scene* s;
  cudaStream_t stream;
  int status = 0;

  template <class T>
  T* alloc(size_t count) {
    if (status) return nullptr;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (count ? count : 1) * sizeof(T));
    if (e != cudaSuccess) {
      status = cuda_fail(e, "cudaMalloc");
      return nullptr;
    }
    s->allocations.push_back(p);
    s->info.device_bytes += (count ? count : 1) * sizeof(T);
    return static_cast<T*>(p);
  }
  template <class T>
  T* upload(const T* host, size_t count) {
    T* d = alloc<T>(count);
    if (status || !count) return d;
    cudaError_t e = cudaMemcpyAsync(d, host, count * sizeof(T), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) status = cuda_fail(e, "cudaMemcpyAsync(H2D)");
    return d;
  }
};

}  // namespace

int set_float(float* dest, unsigned n, float v, cudaStream_t stream) {
  if (n == 0) return 0;
  unsigned grid = blocks_for(n);
  if (grid > 148u * 8u) grid = 148u * 8u;
  k_fill<<<grid, kThreads, 0, stream>>>(dest, n, v);
  RDC_CUDA(cudaGetLastError());
  return 0;
}

void destroy_scene(rdc_scene* s) {
  if (!s) return;
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(s->device);
  for (void* p : s->allocations) cudaFree(p);
  cudaFree(s->frame_image[0]);
  cudaFree(s->frame_image[1]);
  if (s->copy_stream) {
    cudaStreamSynchronize(s->copy_stream);
    cudaStreamDestroy(s->copy_stream);
    for (int k = 0; k < 2; ++k) {
      cudaEventDestroy(s->rendered[k]);
      cudaEventDestroy(s->copied[k]);
    }
  }
  if (s->launched) cudaEventDestroy(s->launched);
  cudaFree(s->stops);
  if (s->staged) {
    cudaEventSynchronize(s->staged);  // the last update's copy has read the staging buffer
    cudaEventDestroy(s->staged);
  }
  cudaFreeHost(s->staging);
  cudaFree(s->frame_scratch);
  cudaFree(s->frame_sigma);
  cudaFree(s->part_rgbw);
  cudaFree(s->part_blur);
  cudaFree(s->tile_arrivals);
  cudaSetDevice(prev);
  delete s;
}

// ---- binned surface-area-heuristic tree over the runs' boxes, built on the host -------------------------------------
// The Morton radix tree (k_radix_tree) splits where the codes' bits say; this one splits where the expected number of box
// tests says: in 2-D a random line meets a convex shape with probability proportional to its perimeter, so a split costs
// perimeter(left) * count(left) + perimeter(right) * count(right). Top-down, 16 bins per axis, both axes tried. Same leaves
// (runs in Morton order), same node layout, so traversal, table queries and every result are untouched — only the number
// of nodes and leaves a ray has to look at changes. Scenes up to kSahMaxRuns runs (the build is O(n log n) on one core).
constexpr uint32_t kSahMaxRuns = 1u << 16;

namespace {
struct HostBox {
  float x0, y0, x1, y1;
  void grow(const HostBox& b) {
    x0 = std::fmin(x0, b.x0); y0 = std::fmin(y0, b.y0); x1 = std::fmax(x1, b.x1); y1 = std::fmax(y1, b.y1);
  }
  float perimeter() const { return (x1 - x0) + (y1 - y0); }
};

inline HostBox empty_box() {
  const float inf = std::numeric_limits<float>::infinity();
  return HostBox{inf, inf, -inf, -inf};
}

// Returns the depth of the tree (leaves at depth >= 1), or 0 when it grew deeper than `max_depth`.
unsigned sah_build(const std::vector<float4>& leaf, float pad, std::vector<BvhNode>& nodes, unsigned max_depth) {
  const int n = (int)leaf.size();
  std::vector<int> order(n);
  for (int i = 0; i < n; ++i) order[i] = i;
  nodes.assign((size_t)n - 1, BvhNode{});
  struct Task {
    int lo, hi, node, parent;
    unsigned depth;
  };
  auto bounds_of = [&](int lo, int hi) {
    HostBox b = empty_box();
    for (int i = lo; i < hi; ++i) b.grow(HostBox{leaf[order[i]].x, leaf[order[i]].y, leaf[order[i]].z, leaf[order[i]].w});
    return b;
  };
  auto padded_box = [&](const HostBox& b) { return make_float4(b.x0 - pad, b.y0 - pad, b.x1 + pad, b.y1 + pad); };
  int next_node = 1;
  unsigned depth = 1;
  std::vector<Task> stack{Task{0, n, 0, -1, 1}};
  constexpr int kBins = 16;
  while (!stack.empty()) {
    const Task t = stack.back();
    stack.pop_back();
    if (t.depth + 1 > max_depth) return 0;
    depth = std::max(depth, t.depth + 1);
    const int count = t.hi - t.lo;
    // centroid bounds of the range
    float cx0 = INFINITY, cy0 = INFINITY, cx1 = -INFINITY, cy1 = -INFINITY;
    for (int i = t.lo; i < t.hi; ++i) {
      const float4 b = leaf[order[i]];
      const float cx = 0.5f * (b.x + b.z), cy = 0.5f * (b.y + b.w);
      cx0 = std::fmin(cx0, cx); cx1 = std::fmax(cx1, cx); cy0 = std::fmin(cy0, cy); cy1 = std::fmax(cy1, cy);
    }
    int best_axis = -1, best_bin = -1;
    float best_cost = INFINITY;
    for (int axis = 0; axis < 2 && count > 2; ++axis) {
      const float lo = axis ? cy0 : cx0, hi = axis ? cy1 : cx1;
      if (!(hi > lo)) continue;
      const float scale = kBins / (hi - lo);
      HostBox bin_box[kBins];
      int bin_count[kBins] = {};
      for (int b = 0; b < kBins; ++b) bin_box[b] = empty_box();
      for (int i = t.lo; i < t.hi; ++i) {
        const float4 b = leaf[order[i]];
        const float c = axis ? 0.5f * (b.y + b.w) : 0.5f * (b.x + b.z);
        const int k = std::min(kBins - 1, std::max(0, (int)((c - lo) * scale)));
        bin_box[k].grow(HostBox{b.x, b.y, b.z, b.w});
        bin_count[k]++;
      }
      float right_cost[kBins];
      HostBox acc = empty_box();
      int cnt = 0;
      for (int k = kBins - 1; k > 0; --k) {
        if (bin_count[k]) acc.grow(bin_box[k]);
        cnt += bin_count[k];
        right_cost[k] = cnt ? acc.perimeter() * (float)cnt : INFINITY;
      }
      acc = empty_box();
      cnt = 0;
      for (int k = 0; k < kBins - 1; ++k) {
        if (bin_count[k]) acc.grow(bin_box[k]);
        cnt += bin_count[k];
        if (cnt == 0 || cnt == count) continue;
        const float cost = acc.perimeter() * (float)cnt + right_cost[k + 1];
        if (cost < best_cost) {
          best_cost = cost;
          best_axis = axis;
          best_bin = k;
        }
      }
    }
    int mid;
    if (best_axis < 0) {
      mid = t.lo + count / 2;  // two leaves, or all centroids in one place: split the (Morton-ordered) range in the middle
    } else {
      const float lo = best_axis ? cy0 : cx0, hi = best_axis ? cy1 : cx1;
      const float scale = kBins / (hi - lo);
      auto in_left = [&](int r) {
        const float4 b = leaf[r];
        const float c = best_axis ? 0.5f * (b.y + b.w) : 0.5f * (b.x + b.z);
        return std::min(kBins - 1, std::max(0, (int)((c - lo) * scale))) <= best_bin;
      };
      mid = (int)(std::stable_partition(order.begin() + t.lo, order.begin() + t.hi, in_left) - order.begin());
      if (mid == t.lo || mid == t.hi) mid = t.lo + count / 2;
    }
    BvhNode& node = nodes[t.node];
    node.parent = t.parent;
    node.pad = 0;
    node.lbox = padded_box(bounds_of(t.lo, mid));
    node.rbox = padded_box(bounds_of(mid, t.hi));
    if (mid - t.lo == 1) node.left = ~order[t.lo];
    else {
      node.left = next_node++;
      stack.push_back(Task{t.lo, mid, node.left, t.node, t.depth + 1});
    }
    if (t.hi - mid == 1) node.right = ~order[mid];
    else {
      node.right = next_node++;
      stack.push_back(Task{mid, t.hi, node.right, t.node, t.depth + 1});
    }
  }
  return depth;
}

// A cut through the tree for the per-tile table of mid-size scenes: start from the root's two children and keep opening
// the entry that costs most — perimeter of its box times the runs below it — until there are `max_entries` of them or only
// leaves are left. Entries: node index (subtree) or ~run (leaf); boxes are the padded child boxes the nodes carry.
void tree_cut(const std::vector<BvhNode>& nodes, int n_runs, int max_entries, std::vector<int>& entry, std::vector<float4>& box) {
  // runs below every inner node (children are created after their parents: a reverse sweep sees children first)
  std::vector<int> below(nodes.size(), 0);
  for (int i = (int)nodes.size() - 1; i >= 0; --i) {
    const BvhNode& nd = nodes[i];
    below[i] = (nd.left < 0 ? 1 : below[nd.left]) + (nd.right < 0 ? 1 : below[nd.right]);
  }
  (void)n_runs;
  entry = {nodes[0].left, nodes[0].right};
  box = {nodes[0].lbox, nodes[0].rbox};
  while ((int)entry.size() < max_entries) {
    int pick = -1;
    float worst = -1.0f;
    for (size_t e = 0; e < entry.size(); ++e) {
      if (entry[e] < 0) continue;
      const float cost = ((box[e].z - box[e].x) + (box[e].w - box[e].y)) * (float)below[entry[e]];
      if (cost > worst) {
        worst = cost;
        pick = (int)e;
      }
    }
    if (pick < 0) break;
    const BvhNode& nd = nodes[entry[pick]];
    entry[pick] = nd.left;
    box[pick] = nd.lbox;
    entry.push_back(nd.right);
    box.push_back(nd.rbox);
  }
}
}  // namespace

int build_scene(const rdc_scene_arrays& a, const rdc_accel_options& o, cudaStream_t stream, rdc_scene** out) {
  if (a.n_segments == 0 || a.n_curves == 0 || a.n_vertices < 4) {
    set_error("accel: empty scene");
    return RDC_E_INVALID;
  }
  if (!(o.flatness_tolerance > 0.0f) || o.max_chords_per_segment < 1 || !(o.curve_width >= 0.0f) || o.run_length < 0 ||
      o.run_length > RDC_RUN || o.tree < RDC_TREE_AUTO || o.tree > RDC_TREE_SAH) {
    set_error("accel: bad options");
    return RDC_E_INVALID;
  }
  for (uint32_t i = 0; i < a.n_segments; ++i)
    if (a.segment_indices[i] % 4 != 0 || a.segment_indices[i] + 4 > a.n_vertices) {
      set_error("accel: segment %u does not address four aligned control points", i);
      return RDC_E_INVALID;
    }
  if (int rc = check_stops(a, "accel")) return rc;
  {
    // segments of a curve are consecutive: curve c owns [curve_map_inverse[c], next curve's first segment)
    std::vector<uint32_t> seg_count(a.n_curves, 0u);
    for (uint32_t sg = 0; sg < a.n_segments; ++sg) {
      const uint32_t c = a.curve_map[sg];
      if (c >= a.n_curves || a.curve_map_inverse[c] > sg || a.curve_index[sg] != sg - a.curve_map_inverse[c]) {
        set_error("accel: segment %u does not sit at its ordinal inside its curve (curve_map / curve_index / curve_map_inverse disagree)", sg);
        return RDC_E_INVALID;
      }
      seg_count[c]++;
    }
    for (uint32_t c = 0; c < a.n_curves; ++c) {
      if (a.curve_map_inverse[c] >= a.n_segments) {
        set_error("accel: curve %u starts past the last segment", c);
        return RDC_E_INVALID;
      }
      const int32_t target = a.curve_connect[c];
      if (target >= (int32_t)a.n_curves) {
        set_error("accel: curve %u connects to a missing curve", c);
        return RDC_E_INVALID;
      }
      // a portal hit on ordinal k continues from ordinal k of the target curve (DeviceCode.cu:228)
      if (target >= 0 && seg_count[target] < seg_count[c]) {
        set_error("accel: curve %u connects to curve %d, which has fewer segments", c, target);
        return RDC_E_INVALID;
      }
    }
  }
  rdc_scene* s = new rdc_scene();
  cudaGetDevice(&s->device);
  cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, s->device);
  Uploader up{s, stream};
  DevScene& d = s->dev;
  bool portals = false;
  for (uint32_t c = 0; c < a.n_curves; ++c) portals |= a.curve_connect[c] >= 0;

  // ---- scene arrays ------------------------------------------------------------------------------
  {
    std::vector<float2> v2(a.n_vertices);
    for (uint32_t i = 0; i < a.n_vertices; ++i) v2[i] = make_float2(a.vertices[3 * i], a.vertices[3 * i + 1]);
    d.vertices = up.upload(v2.data(), v2.size());
  }
  d.segment_indices = up.upload(a.segment_indices, a.n_segments);
  d.curve_map = up.upload(a.curve_map, a.n_segments);
  d.curve_index = up.upload(a.curve_index, a.n_segments);
  d.curve_connect = up.upload(a.curve_connect, a.n_curves);
  d.curve_map_inverse = up.upload(a.curve_map_inverse, a.n_curves);
  s->n_vertices = a.n_vertices;
  // the stop lists, packed into one block of their own (rdc_scene_update_stops may replace it); the build reads back and
  // synchronises anyway, so it copies from pageable memory and leaves the pinned staging buffer to the first update
  const StopLayout stop_at = stop_layout(a);
  std::vector<char> packed(stop_at.bytes);
  pack_stops(a, stop_at, packed.data());
  if (!up.status) {
    cudaError_t e = cudaMalloc(&s->stops, stop_at.bytes);
    if (e == cudaSuccess) {
      s->stops_capacity = stop_at.bytes;
      s->info.device_bytes += stop_at.bytes;
      e = cudaMemcpyAsync(s->stops, packed.data(), stop_at.bytes, cudaMemcpyHostToDevice, stream);
    }
    if (e != cudaSuccess) up.status = cuda_fail(e, "stop lists");
  }
  point_stops(d, s->stops, stop_at);
  s->colour_stops = (uint32_t)stop_at.len[0];
  s->blur_stops = (uint32_t)stop_at.len[2];
  s->weight_stops = (uint32_t)stop_at.len[3];
  s->degree_stops = (uint32_t)stop_at.len[4];
  d.n_segments = a.n_segments;
  d.n_curves = a.n_curves;
  d.seg_walk = up.alloc<SegWalk>(a.n_segments);

  // ---- chords ------------------------------------------------------------------------------------
  const uint32_t nseg = a.n_segments;
  uint32_t* counts = up.alloc<uint32_t>(nseg + 1);
  uint32_t* base = up.alloc<uint32_t>(nseg + 1);
  Bounds* bounds = up.alloc<Bounds>(1);
  s->zero_sigma = up.alloc<float>(1);
  s->work_counters = up.alloc<unsigned int>(2);
  auto fail = [&](int code) {
    destroy_scene(s);
    return code;
  };
  if (up.status) return fail(up.status);
#define BUILD_CUDA(call)                                              \
  do {                                                                \
    cudaError_t e__ = (call);                                         \
    if (e__ != cudaSuccess) return fail(cuda_fail(e__, #call));       \
  } while (0)
  BUILD_CUDA(cudaMemsetAsync(counts, 0, (nseg + 1) * sizeof(uint32_t), stream));
  BUILD_CUDA(cudaMemsetAsync(s->zero_sigma, 0, sizeof(float), stream));
  BUILD_CUDA(cudaMemsetAsync(s->work_counters, 0, 2 * sizeof(unsigned int), stream));
  k_chord_counts<<<blocks_for(nseg), kThreads, 0, stream>>>(d.vertices, d.segment_indices, nseg, o.flatness_tolerance,
                                                            o.max_chords_per_segment, counts);
  BUILD_CUDA(cudaGetLastError());
  size_t temp_bytes = 0;
  BUILD_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, counts, base, (int)(nseg + 1), stream));
  void* scan_temp = nullptr;
  BUILD_CUDA(cudaMalloc(&scan_temp, temp_bytes ? temp_bytes : 1));
  cudaError_t scan_err = cub::DeviceScan::ExclusiveSum(scan_temp, temp_bytes, counts, base, (int)(nseg + 1), stream);
  uint32_t n_chords = 0;
  if (scan_err == cudaSuccess)
    scan_err = cudaMemcpyAsync(&n_chords, base + nseg, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
  if (scan_err == cudaSuccess) scan_err = cudaStreamSynchronize(stream);
  cudaFree(scan_temp);
  BUILD_CUDA(scan_err);
  if (n_chords == 0 || n_chords > (1u << 30)) {
    set_error("accel: %u chords", n_chords);
    return fail(RDC_E_LIMIT);
  }

  // chords stay in original order (hit ids, download hook); runs + tree are what rays touch
  float4* chord_geom = up.alloc<float4>(n_chords);
  uint4* chord_ids = up.alloc<uint4>(n_chords);
  // Per-chord walk starts: where each stop walk stands once it has consumed every stop below the chord's smallest curve
  // parameter. Hits on the chord start their walks there (usually zero steps) instead of at the segment's hint.
  d.chord_walk = up.alloc<uint4>(2 * (size_t)n_chords);
  // the shading records only pay while they stay in L2 next to everything else: 32 MB at most (250 k chords)
  const bool with_records = (size_t)n_chords * 128 <= (32u << 20) && o.shading_records >= 0;
  d.chord_records = with_records ? up.alloc<float4>(8 * (size_t)n_chords) : nullptr;
  uint32_t* run_counts = up.alloc<uint32_t>(nseg + 1);
  uint32_t* run_base = up.alloc<uint32_t>(nseg + 1);
  unsigned int* max_depth = up.alloc<unsigned int>(1);
  unsigned long long* extent_sums = up.alloc<unsigned long long>(2);
  if (up.status) return fail(up.status);
  const float inf = std::numeric_limits<float>::infinity();
  Bounds init{inf, inf, -inf, -inf};
  BUILD_CUDA(cudaMemcpyAsync(bounds, &init, sizeof init, cudaMemcpyHostToDevice, stream));
  k_emit_chords<<<blocks_for(n_chords), kThreads, 0, stream>>>(d.vertices, d.segment_indices, base, nseg, n_chords,
                                                               chord_geom, chord_ids, bounds);
  BUILD_CUDA(cudaGetLastError());
  d.chord_ids = chord_ids;
  d.n_chords = n_chords;
  if (int rc = launch_stop_tables(s, stream)) return fail(rc);
  BUILD_CUDA(cudaMemsetAsync(run_counts, 0, (nseg + 1) * sizeof(uint32_t), stream));
  // Leaf size: long runs make a shallow tree (good when curves are sparse: few boxes overlap), short runs
  // keep leaf boxes tight (good when curves are dense). Mean chord spacing ~ extent / sqrt(#chords).
  uint32_t run_len = (uint32_t)o.run_length;
  if (o.run_length <= 0) run_len = n_chords <= 4096 ? 8 : 4;
  if (run_len > RDC_RUN) run_len = RDC_RUN;
  k_run_counts<<<blocks_for(nseg), kThreads, 0, stream>>>(counts, nseg, run_len, run_counts);
  BUILD_CUDA(cudaGetLastError());
  BUILD_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, run_counts, run_base, (int)(nseg + 1), stream));
  BUILD_CUDA(cudaMalloc(&scan_temp, temp_bytes ? temp_bytes : 1));
  scan_err = cub::DeviceScan::ExclusiveSum(scan_temp, temp_bytes, run_counts, run_base, (int)(nseg + 1), stream);
  uint32_t n_runs = 0;
  Bounds hb{};
  if (scan_err == cudaSuccess) scan_err = cudaMemcpyAsync(&n_runs, run_base + nseg, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
  if (scan_err == cudaSuccess) scan_err = cudaMemcpyAsync(&hb, bounds, sizeof hb, cudaMemcpyDeviceToHost, stream);
  if (scan_err == cudaSuccess) scan_err = cudaStreamSynchronize(stream);
  cudaFree(scan_temp);
  BUILD_CUDA(scan_err);
  if (n_runs == 0 || !(std::isfinite(hb.xmin) && std::isfinite(hb.ymin) && std::isfinite(hb.xmax) && std::isfinite(hb.ymax))) {
    set_error("accel: control points are not finite");
    return fail(RDC_E_INVALID);
  }
  float extent = std::fmax(std::fmax(std::fabs(hb.xmin), std::fabs(hb.xmax)), std::fmax(std::fabs(hb.ymin), std::fabs(hb.ymax)));
  // curve_width thickens every leaf box; the relative term keeps the padding above the rounding of the
  // chord test (a few ulp of the largest coordinate), which is what makes culling exact.
  const float pad = o.curve_width + 4e-6f * extent;

  RunRecord* runs_in = nullptr;
  uint4* ids_in = nullptr;
  float4 *box_in = nullptr, *leaf_box = nullptr, *node_box = nullptr;
  uint32_t *codes_in = nullptr, *codes = nullptr, *order_in = nullptr, *order = nullptr;
  void* sort_temp = nullptr;
  unsigned int* arrivals = nullptr;
  int* leaf_parent = nullptr;
  auto free_temps = [&]() {
    cudaFree(runs_in); cudaFree(ids_in); cudaFree(box_in); cudaFree(leaf_box); cudaFree(node_box); cudaFree(codes_in);
    cudaFree(codes); cudaFree(order_in); cudaFree(order); cudaFree(sort_temp); cudaFree(arrivals); cudaFree(leaf_parent);
  };
#define TEMP_CUDA(call)                                         \
  do {                                                          \
    cudaError_t e__ = (call);                                   \
    if (e__ != cudaSuccess) {                                   \
      free_temps();                                             \
      return fail(cuda_fail(e__, #call));                       \
    }                                                           \
  } while (0)
  const uint32_t n_nodes = n_runs > 1 ? n_runs - 1 : 1;
  TEMP_CUDA(cudaMalloc(&runs_in, n_runs * sizeof(RunRecord)));
  TEMP_CUDA(cudaMalloc(&ids_in, n_runs * sizeof(uint4)));
  TEMP_CUDA(cudaMalloc(&box_in, n_runs * sizeof(float4)));
  TEMP_CUDA(cudaMalloc(&leaf_box, n_runs * sizeof(float4)));
  TEMP_CUDA(cudaMalloc(&node_box, n_nodes * sizeof(float4)));
  TEMP_CUDA(cudaMalloc(&codes_in, n_runs * sizeof(uint32_t)));
  TEMP_CUDA(cudaMalloc(&codes, n_runs * sizeof(uint32_t)));
  TEMP_CUDA(cudaMalloc(&order_in, n_runs * sizeof(uint32_t)));
  TEMP_CUDA(cudaMalloc(&order, n_runs * sizeof(uint32_t)));
  TEMP_CUDA(cudaMalloc(&arrivals, n_nodes * sizeof(unsigned int)));
  TEMP_CUDA(cudaMalloc(&leaf_parent, n_runs * sizeof(int)));
  RunRecord* runs = up.alloc<RunRecord>(n_runs);
  uint4* run_ids = up.alloc<uint4>(n_runs);
  float4* run_box = up.alloc<float4>(n_runs);
  BvhNode* nodes = up.alloc<BvhNode>(n_nodes);
  if (up.status) {
    free_temps();
    return fail(up.status);
  }

  k_emit_runs<<<blocks_for(n_runs), kThreads, 0, stream>>>(chord_geom, base, run_base, nseg, n_runs, run_len, hb, runs_in, ids_in,
                                                           box_in, codes_in, order_in);
  TEMP_CUDA(cudaGetLastError());
  size_t sort_bytes = 0;
  TEMP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, codes_in, codes, order_in, order, (int)n_runs, 0, 32, stream));
  TEMP_CUDA(cudaMalloc(&sort_temp, sort_bytes ? sort_bytes : 1));
  TEMP_CUDA(cub::DeviceRadixSort::SortPairs(sort_temp, sort_bytes, codes_in, codes, order_in, order, (int)n_runs, 0, 32, stream));
  k_gather_runs<<<blocks_for(n_runs), kThreads, 0, stream>>>(order, runs_in, ids_in, box_in, n_runs, runs, run_ids, leaf_box);
  TEMP_CUDA(cudaGetLastError());

  TEMP_CUDA(cudaMemsetAsync(extent_sums, 0, 2 * sizeof(unsigned long long), stream));
  k_pad_boxes<<<blocks_for(n_runs), kThreads, 0, stream>>>(leaf_box, n_runs, pad, run_box, extent_sums);
  TEMP_CUDA(cudaGetLastError());
  TEMP_CUDA(cudaMemsetAsync(max_depth, 0, sizeof(unsigned int), stream));
  unsigned int sah_depth = 0;
  if (n_runs == 1) {
    k_single_leaf_root<<<1, 1, 0, stream>>>(leaf_box, pad, nodes);
    TEMP_CUDA(cudaGetLastError());
  } else {
    // tree over the runs: surface-area heuristic on the host for scenes it handles in milliseconds, Morton radix tree on
    // the device otherwise (or when the SAH tree comes out deeper than the traversal stack)
    const bool want_sah = o.tree == RDC_TREE_SAH || (o.tree == RDC_TREE_AUTO && n_runs <= kSahMaxRuns);
    if (want_sah) {
      std::vector<float4> h_leaf(n_runs);
      TEMP_CUDA(cudaMemcpyAsync(h_leaf.data(), leaf_box, n_runs * sizeof(float4), cudaMemcpyDeviceToHost, stream));
      TEMP_CUDA(cudaStreamSynchronize(stream));
      std::vector<BvhNode> h_nodes;
      sah_depth = sah_build(h_leaf, pad, h_nodes, 62);
      if (sah_depth) {
        TEMP_CUDA(cudaMemcpyAsync(nodes, h_nodes.data(), h_nodes.size() * sizeof(BvhNode), cudaMemcpyHostToDevice, stream));
        std::vector<int> cut_entry;
        std::vector<float4> cut_boxes;
        tree_cut(h_nodes, (int)n_runs, RDC_CUT_SEED, cut_entry, cut_boxes);
        d.cut_node = up.upload(cut_entry.data(), cut_entry.size());
        d.cut_box = up.upload(cut_boxes.data(), cut_boxes.size());
        d.n_cut = (uint32_t)cut_entry.size();
        TEMP_CUDA(cudaStreamSynchronize(stream));  // h_nodes and the cut leave scope
        if (up.status) {
          free_temps();
          return fail(up.status);
        }
      }
    }
    if (!sah_depth) {
      TEMP_CUDA(cudaMemsetAsync(arrivals, 0, n_nodes * sizeof(unsigned int), stream));
      k_radix_tree<<<blocks_for(n_runs - 1), kThreads, 0, stream>>>(codes, (int)n_runs, nodes, leaf_parent);
      TEMP_CUDA(cudaGetLastError());
      k_fit_boxes<<<blocks_for(n_runs), kThreads, 0, stream>>>(leaf_box, (int)n_runs, pad, leaf_parent, nodes, node_box, arrivals);
      TEMP_CUDA(cudaGetLastError());
      k_depth<<<blocks_for(n_runs), kThreads, 0, stream>>>(leaf_parent, nodes, (int)n_runs, max_depth);
      TEMP_CUDA(cudaGetLastError());
    }
  }
  unsigned int depth = 0;
  unsigned long long h_extent[2] = {0, 0};
  TEMP_CUDA(cudaMemcpyAsync(h_extent, extent_sums, sizeof h_extent, cudaMemcpyDeviceToHost, stream));
  TEMP_CUDA(cudaMemcpyAsync(&depth, max_depth, sizeof depth, cudaMemcpyDeviceToHost, stream));
  TEMP_CUDA(cudaStreamSynchronize(stream));
  free_temps();
  if (sah_depth) depth = sah_depth;
  if (depth > 62) {
    set_error("accel: tree depth %u exceeds the traversal stack", depth);
    return fail(RDC_E_LIMIT);
  }

  d.chord_geom = chord_geom;
  d.seg_chord_base = base;
  d.seg_chord_count = counts;
  d.runs = runs;
  d.run_ids = run_ids;
  d.run_box = run_box;
  d.nodes = nodes;
  d.n_runs = n_runs;
  d.n_nodes = n_nodes;
  d.root_box = make_float4(hb.xmin - pad, hb.ymin - pad, hb.xmax + pad, hb.ymax + pad);
  s->info.n_segments = a.n_segments;
  s->info.n_curves = a.n_curves;
  s->info.n_chords = n_chords;
  s->info.n_runs = n_runs;
  s->info.n_nodes = n_nodes;
  s->info.bvh_depth = depth ? depth : 1;
  s->info.has_portals = portals ? 1 : 0;
  s->info.traversal_bytes = (uint64_t)n_nodes * sizeof(BvhNode) + (uint64_t)n_runs * sizeof(RunRecord);
  s->info.pad = pad;
  s->mean_run_w = (float)((double)h_extent[0] / 1024.0 / n_runs);
  s->mean_run_h = (float)((double)h_extent[1] / 1024.0 / n_runs);
  *out = s;
  return 0;
#undef BUILD_CUDA
#undef TEMP_CUDA
}

int download_chords(const rdc_scene* s, float* geom, uint32_t* ids) {
  const uint32_t n = s->dev.n_chords;
  std::vector<uint4> id(n);
  RDC_CUDA(cudaMemcpy(geom, s->dev.chord_geom, n * sizeof(float4), cudaMemcpyDeviceToHost));
  RDC_CUDA(cudaMemcpy(id.data(), s->dev.chord_ids, n * sizeof(uint4), cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < n; ++i) {
    if (id[i].x != i) {
      set_error("chord table is corrupt");
      return RDC_E_INVALID;
    }
    ids[3 * i + 0] = id[i].y; ids[3 * i + 1] = id[i].z; ids[3 * i + 2] = id[i].w;
  }
  return 0;
}

// New stop lists on a built handle: validate everything first (a rejection leaves the handle as it was), make room, then
// pack into the pinned staging buffer and enqueue copy + k_stop_tables behind the handle's previous launch or update.
int update_stops(rdc_scene* s, const rdc_scene_arrays& a, cudaStream_t stream) {
  if (a.n_vertices != s->n_vertices || a.n_segments != s->dev.n_segments || a.n_curves != s->dev.n_curves) {
    set_error("update stops: the arrays have %u vertices, %u segments and %u curves, the scene was built from %u, %u and %u",
              a.n_vertices, a.n_segments, a.n_curves, s->n_vertices, s->dev.n_segments, s->dev.n_curves);
    return RDC_E_INVALID;
  }
  if (int rc = check_stops(a, "update stops")) return rc;
  const StopLayout L = stop_layout(a);
  const bool grow = L.bytes > s->stops_capacity;
  const size_t capacity = grow ? L.bytes : s->stops_capacity;
  if (s->staging_capacity < capacity) {  // the handle's first update, or lists larger than any it has held
    void* fresh = nullptr;
    RDC_CUDA(cudaMallocHost(&fresh, capacity));
    if (s->staged) {
      cudaError_t e = cudaEventSynchronize(s->staged);
      if (e != cudaSuccess) {
        cudaFreeHost(fresh);
        return cuda_fail(e, "cudaEventSynchronize(staged)");
      }
    } else {
      cudaError_t e = cudaEventCreateWithFlags(&s->staged, cudaEventDisableTiming);
      if (e != cudaSuccess) {
        cudaFreeHost(fresh);
        return cuda_fail(e, "cudaEventCreate(staged)");
      }
    }
    cudaFreeHost(s->staging);
    s->staging = fresh;
    s->staging_capacity = capacity;
  } else {
    RDC_CUDA(cudaEventSynchronize(s->staged));  // the previous update's copy has left the staging buffer
  }
  if (grow) {  // the old block may still be read by the handle's last launch: wait for it, then replace the block
    void* fresh = nullptr;
    RDC_CUDA(cudaMalloc(&fresh, capacity));
    if (s->launched_any) {
      cudaError_t e = cudaEventSynchronize(s->launched);
      if (e != cudaSuccess) {
        cudaFree(fresh);
        return cuda_fail(e, "cudaEventSynchronize(launched)");
      }
    }
    cudaFree(s->stops);
    s->info.device_bytes += capacity - s->stops_capacity;
    s->stops = fresh;
    s->stops_capacity = capacity;
  }
  pack_stops(a, L, s->staging);
  // like a launch: the device work waits for the handle's previous launch or update, whatever stream that was on
  if (int rc = wait_previous_launch(s, stream)) return rc;
  RDC_CUDA(cudaMemcpyAsync(s->stops, s->staging, L.bytes, cudaMemcpyHostToDevice, stream));
  RDC_CUDA(cudaEventRecord(s->staged, stream));
  point_stops(s->dev, s->stops, L);
  s->colour_stops = (uint32_t)L.len[0];
  s->blur_stops = (uint32_t)L.len[2];
  s->weight_stops = (uint32_t)L.len[3];
  s->degree_stops = (uint32_t)L.len[4];
  if (int rc = launch_stop_tables(s, stream)) return rc;
  return record_launch(s, stream);
}

int wait_previous_launch(rdc_scene* s, cudaStream_t stream) {
  if (!s->launched) RDC_CUDA(cudaEventCreateWithFlags(&s->launched, cudaEventDisableTiming));
  if (s->launched_any && s->launched_on != stream) RDC_CUDA(cudaStreamWaitEvent(stream, s->launched, 0));
  return 0;
}

int record_launch(rdc_scene* s, cudaStream_t stream) {
  RDC_CUDA(cudaEventRecord(s->launched, stream));
  s->launched_on = stream;
  s->launched_any = true;
  return 0;
}

int download_stop_tables(const rdc_scene* s, void* seg_walk, void* chord_walk, void* chord_records) {
  const DevScene& d = s->dev;
  if (chord_records && !d.chord_records) {
    set_error("download stop tables: the scene has no shading records");
    return RDC_E_INVALID;
  }
  if (s->launched_any) RDC_CUDA(cudaEventSynchronize(s->launched));
  RDC_CUDA(cudaMemcpy(seg_walk, d.seg_walk, d.n_segments * sizeof(SegWalk), cudaMemcpyDeviceToHost));
  RDC_CUDA(cudaMemcpy(chord_walk, d.chord_walk, 2 * (size_t)d.n_chords * sizeof(uint4), cudaMemcpyDeviceToHost));
  if (chord_records) RDC_CUDA(cudaMemcpy(chord_records, d.chord_records, 8 * (size_t)d.n_chords * sizeof(float4), cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace rdc
