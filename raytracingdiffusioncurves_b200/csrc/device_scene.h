// device_scene.h — device-resident scene layout shared by the accel build, the render kernels and the
// C ABI glue. Everything a kernel needs travels by value in DevScene (kernel parameter space).
#ifndef RDC_DEVICE_SCENE_H
#define RDC_DEVICE_SCENE_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/rdc_b200.h"
#include "rdc_math.h"

// One LBVH node, 48 bytes = three 128-bit loads. A node stores the padded boxes of BOTH children, so a
// ray decides which children to visit from one node fetch. child >= 0: inner node index; child < 0:
// leaf, ~child is the chord's position in Morton order.
struct __align__(16) BvhNode {
  float4 lbox;  // xmin, ymin, xmax, ymax of the left child
  float4 rbox;
  int left, right;
  int parent;  // -1 for the root
  int pad;
};

// Leaf primitive: up to RDC_RUN consecutive chords of one spline segment = RDC_RUN+1 points, 80 bytes =
// five 128-bit loads. Chord j of the run joins points j and j+1; its original id is first_id + j.
struct __align__(16) RunRecord {
  uint32_t first_id;
  uint32_t count;
  float pts[2 * (RDC_RUN + 1)];  // vector 0 = {first_id, count, P0}, vectors 1..4 = two points each
};
static_assert(sizeof(RunRecord) == 80, "RunRecord must be five float4");

// Per spline segment: where each stop-list walk may start (rdc_walk_hint with u_min = the segment's
// ordinal) and where it ends, plus the two per-segment lookups shading needs. 64 bytes = four 128-bit loads.
struct __align__(16) SegWalk {
  uint32_t left_first, left_end, right_first, right_end;
  uint32_t blur_first, blur_end, weight_first, weight_end;
  uint32_t degree_first, degree_end, curve, ordinal;
  uint32_t portal_left_first, portal_left_end;  // right list's range walked on the LEFT u array (DeviceCode.cu:297)
  uint32_t pad0, pad1;
};

// entries of the scene-wide seed cut through the tree (cut_node / cut_box below); the render kernel opens it further per tile
#define RDC_CUT_SEED 32

struct DevStops {
  const uint2* index;  // {start,count} per curve
  const float* u;      // flat stop parameters (+INF sentinels at the end)
  const float* value;  // scalar families
  const float4* rgb;   // colour families (rgb, 0)
};

struct DevScene {
  // spline segments (reference Params: vertices, segmentIndices, curve_map, curve_index, curve_connect,
  // curve_map_inverse). Control points are float2 (z == 0 always); segment s owns points [4s,4s+4).
  const float2* vertices;
  const uint32_t* segment_indices;
  const uint32_t* curve_map;
  const uint32_t* curve_index;
  const int32_t* curve_connect;
  const uint32_t* curve_map_inverse;
  DevStops color_left, color_right, blur, weight, weight_degree;
  // chords, original order (segment by segment, k ascending): parity ids, download hook
  const float4* chord_geom;        // [n_chords] ax, ay, bx, by
  const uint4* chord_ids;          // [n_chords] chord id, segment, k, K
  const uint32_t* seg_chord_base;  // [n_segments+1] id of chord 0 of each segment
  const uint32_t* seg_chord_count; // [n_segments]   K
  const SegWalk* seg_walk;         // [n_segments]
  const uint4* chord_walk;         // [2*n_chords] per chord: walk start of left, right, blur, weight | degree, portal-left
  // Shading records: per chord, the two stops of every family its hits interpolate between — 8 x 16 bytes: blur, weight,
  // exponent {u0,u1,v0,v1}; left colour {rgb0,u0} {rgb1,u1}; right colour likewise; {segment, ordinal, k | K << 16,
  // curve | flags << 27}. flags 0x1F: every family stays inside one stop interval over the whole chord, and the record
  // replaces the walks. nullptr: no table (rdc_accel_options::shading_records = -1 turns it off, to measure the difference).
  const float4* chord_records;
  // acceleration structure: what rays touch
  const RunRecord* runs;           // [n_runs] Morton order
  const uint4* run_ids;            // [n_runs] Morton order: first chord id, segment, k of the first chord, K
  const float4* run_box;           // [n_runs] Morton order: padded box of each run (per-tile run table)
  const BvhNode* nodes;            // [max(n_runs-1,1)]
  // seed cut through the tree: at most RDC_CUT_SEED subtrees (node index) or leaves (~run) that together hold every run, with
  // their padded boxes — what the per-tile cut table starts from (render.cu, kModeCut). n_cut == 0: no cut (Morton trees).
  const int* cut_node;
  const float4* cut_box;
  uint32_t n_cut;
  float4 root_box;                 // padded box of the whole scene (per-pixel angular culling)
  uint32_t n_segments, n_curves, n_chords, n_runs, n_nodes;
};

struct rdc_scene {
  int device = 0;
  int sm_count = 0;  // multiprocessors of `device`
  DevScene dev{};
  rdc_scene_info info{};
  uint32_t n_vertices = 0;         // of the arrays the handle was built from (rdc_scene_update_stops checks it)
  std::vector<void*> allocations;  // everything to cudaFree on destroy
  // the five stop families in one device block (accel.cu, StopLayout), grown by rdc_scene_update_stops and never shrunk;
  // updates pack the caller's lists into the pinned staging buffer, which `staged` guards until the copy has read it
  void* stops = nullptr;
  size_t stops_capacity = 0;
  void* staging = nullptr;
  size_t staging_capacity = 0;
  cudaEvent_t staged = nullptr;
  uint32_t colour_stops = 0;  // stops per colour family in the block: max(n_color_left, n_color_right) + 2
  // per-N table of the iterated base directions (DeviceCode.cu:110-112,167-171)
  float2* base_dirs = nullptr;
  float base_dirs_n = -1.0f;
  uint32_t base_dirs_capacity = 0;
  float* zero_sigma = nullptr;  // device float used when the caller passes no max_sigma
  unsigned int* work_counters = nullptr;  // k_render's tile counter pair (one render in flight per handle)
  // the handle's launches are serialised: a launch on another stream waits for this event first
  cudaEvent_t launched = nullptr;
  cudaStream_t launched_on = nullptr;
  bool launched_any = false;
  uint32_t grid_blocks[32] = {};  // SM-filling grid size per k_render variant (render.cu, variant_index) ...
  size_t grid_dyn[32] = {};       // ... at this much dynamic shared memory
  float mean_run_w = 0.0f, mean_run_h = 0.0f;  // mean padded run box (local-table radius estimate)
  // partial sums of k_render's work units (a tile's rays are dealt to several units), grown on demand
  float4* part_rgbw = nullptr;
  float* part_blur = nullptr;
  unsigned int* tile_arrivals = nullptr;
  size_t part_capacity = 0, tile_capacity = 0;
  // frame buffers of rdc_render_frame_to_host, grown on demand and kept (no per-frame allocation)
  float4* frame_image[2] = {nullptr, nullptr};  // used in turn: the copy of one overlaps the rendering of the other
  float4* frame_scratch = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t rendered[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
  int frame_slot = 0;
  float* frame_sigma = nullptr;  // pixels + 1: the extra float is the max-sigma flag
  size_t frame_pixels = 0;
};

namespace rdc {
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
// accel.cu
int build_scene(const rdc_scene_arrays& a, const rdc_accel_options& o, cudaStream_t stream, rdc_scene** out);
void destroy_scene(rdc_scene* s);
int download_chords(const rdc_scene* s, float* geom, uint32_t* ids);
int update_stops(rdc_scene* s, const rdc_scene_arrays& a, cudaStream_t stream);
int download_stop_tables(const rdc_scene* s, void* seg_walk, void* chord_walk, void* chord_records);
// render.cu
int render(rdc_scene* s, const rdc_frame_params& p, float4* image, float* blur_map, cudaStream_t stream, uint32_t n_targets = 0,
           float* const* target_images = nullptr, float* const* target_blur_maps = nullptr);
int reserve(rdc_scene* s, const rdc_frame_params& p, cudaStream_t stream);
int launch_plan(const rdc_scene* s, const rdc_frame_params& p, rdc_launch_plan* out);
int color_adjoint(rdc_scene* s, const rdc_frame_params& p, const float4* image_grad, double* grad_left, double* grad_right,
                  cudaStream_t stream);
// pick.cu
int pick(rdc_scene* s, const float* points, uint32_t n, float max_distance, int orzan, rdc_pick* out, float* stops,
         cudaStream_t stream);
int pick_frame(rdc_scene* s, const rdc_frame_params* p, float max_distance, rdc_pick* out, float* stops, cudaStream_t stream);
// blur.cu
int gaussian_blur(float4* dest, const float4* src, const float* sigma, float4* scratch, int width, int height,
                  int row_begin, int row_end, const float* max_sigma, cudaStream_t stream, int halo_rows = -1);
int set_float(float* dest, unsigned n, float v, cudaStream_t stream);
int blur_preload();
}  // namespace rdc

#define RDC_CUDA(call)                                            \
  do {                                                            \
    cudaError_t e__ = (call);                                     \
    if (e__ != cudaSuccess) return rdc::cuda_fail(e__, #call);    \
  } while (0)

#endif
