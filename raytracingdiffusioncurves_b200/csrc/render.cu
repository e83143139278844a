// render.cu — per-frame ray generation, closest-chord traversal, shading, weighted normalisation.
//
// Replaces optixLaunch(...) of DeviceCode.cu's three programs (optixHello.cpp:1184):
//   __raygen__rg      DeviceCode.cu:85-182   -> k_render's pixel loop (gen_ray, accumulate)
//   __closesthit__ch  DeviceCode.cu:194-342  -> trace_from (terminal :328-340, portal :220-320 as an
//                                               iterative re-trace loop, shape of DeviceCodeIt.cu:151-170)
//   __miss__ms        DeviceCode.cu:185-192  -> zero contribution
//   RT-core traversal + built-in curve intersector (closed) -> closest chord by one of three routes:
//       table_closest over a whole-scene run table (at most 64 runs), table_closest over a per-tile table of
//       the nearest runs with the far rays deferred to the tree (1024 runs or more, gather_local), or
//       closest_chord over the LBVH of accel.cu (everything else, portal continuations, deferred rays)
// Compiled with -fmad=false: plain expressions keep the reference's operation order and rounding; fused
// operations appear only through rdc_fma (rdc_math.h).
//
// Work that cannot change the result is skipped, never approximated:
//   * a ray whose angular stratum cannot reach the scene's box from anywhere inside its pixel is a miss
//     (contributes zero, DeviceCode.cu:185-192) and is not generated at all (pixel_cull);
//   * tree and table culling only use conservative tests (padded boxes, widened angular intervals, shrunk
//     distances); the accepted hit is the lexicographic minimum of (t, chord id) over all chords, the same
//     rule the brute-force oracle applies.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <utility>

#include "device_scene.h"
#include "rdc_math.h"

namespace rdc {
namespace {

constexpr int kBlock = 256;
constexpr int kWarpTileW = 8, kWarpTileH = 4;   // a tile: 8x4 pixels, one lane per pixel, all lanes on the same ray index
constexpr int kMaxSplit = 8;                    // a tile's rays may be dealt to up to 8 work units (RenderArgs::split)
constexpr int kAutoSplit = 8;                   // (the automatic choice may use all of them: a rank of 8 at 1080p does)
constexpr uint32_t kTableRuns = 64;             // scenes with at most this many runs use the whole-scene run table
constexpr int kStripRows = RDC_STRIP_ROWS;       // multi-GPU strips (rdc_frame_params::strip_stride)
static_assert(kStripRows % kWarpTileH == 0, "a warp tile must not straddle two strips");
constexpr int kStack = 64;
constexpr uint32_t kMiss = 0xFFFFFFFFu;
constexpr size_t kSmemSceneLimit = 56 * 1024;  // stage nodes + runs in shared memory below this (4 blocks per SM still fit;
                                               // measured: 40 -> 56 KB buys 4-7 % on the scenes it adds, 72 KB loses 8 % on the next ones)
constexpr int kRunVec = sizeof(RunRecord) / 16;
constexpr int kMinBlocks = 4;                   // resident blocks per SM the register allocation aims for
// local run table (scenes too large for the whole-scene table): per warp, the runs around the tile
constexpr int kTableWords = 2;                    // whole-scene table: 64 slots, two per lane
constexpr int kLocalWords = 2;                    // local table: 32 slots per word, one slot of each word per lane
constexpr int kLocalSlots = 32 * kLocalWords;
constexpr int kGatherCap = 2 * kLocalSlots;       // runs a neighbourhood query may return / nodes pending in it (at most 256)
constexpr int kGatherAttempts = 6;                // radius adjustments per work unit
constexpr int kDeferCap = 64;                     // deferred rays a warp can hold (a batch of 32 leaves when 32 are waiting)
constexpr int kRingWords = kGatherCap > 2 * kDeferCap ? kGatherCap : 2 * kDeferCap;
static_assert(kGatherCap <= 256, "candidate keys carry the position in their low 8 bits");
enum { kModeTree = 0, kModeTable = 1, kModeLocal = 2, kModeCut = 3 };

struct __align__(16) WarpLocal {
  float4 box[kLocalSlots];        // padded box of the run in each slot; slots are sorted by distance from the tile
  uint32_t run[kLocalSlots];      // its position in Morton order
  float dist[kLocalSlots];        // lower bound of its distance from any origin in the tile
  uint32_t cand_run[kGatherCap];  // neighbourhood query: runs found ...
  uint32_t cand_key[kGatherCap];  // ... and their sort keys: distance bits with the position in the low byte
  uint32_t ring[kRingWords];      // query: nodes pending; ray loop: queue of deferred rays {lane << 16 | ray, bound}
  // (copying the slots' run records in here as well was measured: 10-15 % slower — fewer resident blocks)
  // per-lane state that is only touched once per 32 iterations or per batch of deferred rays: kept out of registers
  int first[kLocalWords][32], span[kLocalWords][32];  // ray-index interval of the slots the lane looks after
  float deferred[5][32];                              // running sums of the lane's deferred samples: w, r*w, g*w, b*w, blur*w
  int root_first, root_span;                          // the rays of the tile that can reach the scene at all
};

// whole-scene run table: the order in which a tile looks at the scene's runs — nearest first, so that a ray's candidate
// scan can stop at the first run that lies beyond the hit found so far (per warp, rebuilt per work unit)
struct __align__(16) WarpOrder {
  uint32_t run[kTableRuns];   // slot -> run
  float dist[kTableRuns];     // lower bound of the run's distance from any origin in the tile (shrunk like WarpLocal::dist)
  uint32_t key[kTableRuns];   // sort keys: distance bits with the run in the low six bits
};
static_assert(kTableRuns <= 64, "sort keys carry the run in their low six bits");

// cut table: the warp's own cut through the tree for the tile in work — the scene's seed cut (accel.cu) with the subtrees
// nearest the tile opened until the table is full — followed by its WarpOrder
struct __align__(16) WarpCut {
  float4 box[kTableRuns];  // padded box of each entry
  int node[kTableRuns];    // what the entry is: node index (subtree) or ~run (leaf)
  WarpOrder order;
};
static_assert(RDC_CUT_SEED <= kTableRuns, "the seed cut must fit the table");

// group mode (table launches with more than one unit per tile): the G warps that take a tile's G units together share ...
struct __align__(16) GroupTable {
  int first[kTableRuns], span[kTableRuns];  // ray-index interval of every table slot (computed once, by the group's first warp)
  uint32_t tile;
};
// ... and a block (8 / G groups) holds
struct __align__(16) GroupShared {
  float4 part_rgbw[kBlock / 32][32];  // every warp's partial sums, added up by its group's first warp in unit order
  float part_blur[kBlock / 32][32];
  GroupTable table[kBlock / 64];      // one per group (at most four groups of two warps)
};

struct RenderArgs {
  DevScene sc;
  float4* image;
  float* blur_map;
  const float2* base_dirs;
  uint32_t* hit_ids;
  float* max_sigma;
  unsigned long long* stats;
  uint32_t width, height, row_begin, row_end;
  uint32_t strip_stride, strip_offset;  // rows are dealt out in strips of kStripRows: strip t belongs to t % stride == offset
  uint32_t local_rows;                  // rows of the output buffers this launch covers
  uint32_t row_skew;                    // row_begin % 4 of a contiguous band: tiles stay aligned to the full frame's
  uint32_t split;                       // work units per tile: unit q traces rays i = q (mod split)
  int group;                            // table launches with split > 1: G = split warps of a block take the units of ONE tile
                                        // together (one table per tile instead of one per unit, partial sums in shared memory); 0 = off
  uint32_t mid_tx, mid_ty;              // the tile (column, local tile row) nearest the scene's centre: units are handed out
                                        // centre-out from it
  float4* part_rgbw;                    // [split][local pixels] partial sums of units (split > 1)
  float* part_blur;
  unsigned int* tile_arrivals;          // [tiles] units of the tile that have finished (self-rewinding)
  unsigned int* work;                   // [0] next warp tile, [1] warps finished (self-rewinding)
  int n_iter;         // number of loop trips: ceil(number_of_rays_per_pixel)
  float n_rays;       // number_of_rays_per_pixel
  float two_over_n;   // 2 / number_of_rays_per_pixel  (DeviceCode.cu:99,120)
  float zoom, off_x, off_y;
  uint32_t frame, seed;
  int orzan, use_aa, max_depth, brute, cull;
  float local_r0;  // local table: first radius tried around a tile
  // rdc_render_to_frames: finished pixels go to their place in up to RDC_MAX_FRAME_TARGETS FULL frames (peer memory)
  uint32_t n_targets;
  float4* target_image[RDC_MAX_FRAME_TARGETS];
  float* target_blur[RDC_MAX_FRAME_TARGETS];
};

struct Hit {
  float t, s;
  int leaf;      // run position in Morton order, -1 = miss
  int j;         // chord inside the run
  uint32_t id;   // original chord id (tie-break, parity)
};

// no hit closer than `bound`
__device__ __forceinline__ Hit miss_hit(float bound) { return Hit{bound, 0.0f, -1, 0, kMiss}; }

struct Accel {
  const BvhNode* nodes;
  const float4* runs;     // kRunVec float4 per run
  const float4* run_box;  // padded box per run
  uint32_t n_runs;
  // per-tile table (kModeTable, kModeCut): padded box per table entry and, in cut mode, what the entry is — a subtree
  // (node index) or a leaf (~run); kModeTable: entry = run, slot_node stays null
  const float4* slot_box;
  const int* slot_node;
};

// per-thread work counters of the counting build (rdc_frame_params::stats)
struct Counters {
  unsigned int rays = 0, nodes = 0, chords = 0, shaded = 0, deferred = 0, gathered = 0;
};

template <bool SMEM>
__device__ __forceinline__ float4 load16(const float4* p) {
  if (SMEM) return *p;
  return __ldg(p);
}

// reciprocal for the slab test only (never decides a hit): one MUFU.RCP, |d| kept away from 0
__device__ __forceinline__ float slab_rcp(float d) {
  float a = fabsf(d) < 1e-30f ? copysignf(1e-30f, d) : d;
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
  return r;
}

// Slab test of a padded box in fused form: t = x * (1/d) - o * (1/d), the second product computed once per ray.
// Culling only — never decides a hit. Against exact arithmetic, the fused test, the approximate reciprocal and the chord
// test's own differences p - o move the box as the ray sees it by a few ulp of the coordinates involved: up to ~6 x 2^-23
// x max(M, extent), M the largest origin coordinate. So the rounding scales with the ORIGINS, not with the scene: the
// boxes' padding (curve_width + 4e-6 x extent, accel.cu) alone covers it only while M stays within about twice the
// extent. A launch whose origins lie farther out reads boxes widened by w (slab_widening, widened_boxes), which makes the
// padding and w together >= 16 x 2^-23 x max(M, extent), more than twice the displacement, for any view; views near the
// scene read the scene's own boxes. 12 operations per box instead of 16: lady_bug.xml 1080p 8.92 -> 8.49 ms, the 21-scene
// 4K sweep 834 -> 805 ms (profiles/r02b/variants.log).
struct SlabRay {
  float idx, idy, nox, noy;  // 1/dx, 1/dy, -ox/dx, -oy/dy
};
__device__ __forceinline__ SlabRay slab_ray(float ox, float oy, float dx, float dy) {
  SlabRay r;
  r.idx = slab_rcp(dx);
  r.idy = slab_rcp(dy);
  r.nox = -(ox * r.idx);
  r.noy = -(oy * r.idy);
  return r;
}
__device__ __forceinline__ float slab_enter(const SlabRay& r, float4 b, float* exit) {
  const float tx1 = fmaf(b.x, r.idx, r.nox), tx2 = fmaf(b.z, r.idx, r.nox);
  const float ty1 = fmaf(b.y, r.idy, r.noy), ty2 = fmaf(b.w, r.idy, r.noy);
  *exit = fminf(fmaxf(tx1, tx2), fmaxf(ty1, ty2));
  return fmaxf(fmaxf(fminf(tx1, tx2), fminf(ty1, ty2)), 0.0f);
}

// All chords of one run against the ray. Edge values of the shared end points are computed once; the
// record is read two points at a time and only as far as the run is long. The unrolled pass only marks
// the chords whose end points lie on different sides of the ray; the (rare) marked ones are then resolved
// in a rolled loop that re-reads their two points — same inputs, same operations, same bits.
template <bool SMEM, bool PORTALS>
__device__ __forceinline__ int test_run(const float4* rp, int leaf, float ox, float oy, float dx, float dy, float inv_dd,
                                        uint32_t skip_lo, uint32_t skip_hi, Hit& h) {
  const float4 head = load16<SMEM>(rp);
  const int count = (int)__float_as_uint(head.y);
  // bit k of `above`: point k lies on the positive side of the ray's supporting line
  uint32_t above = rdc_edge(dx, dy, head.z - ox, head.w - oy) > 0.0f ? 1u : 0u;
#pragma unroll
  for (int v = 1; v < kRunVec; ++v) {
    if (2 * v - 2 >= count) break;
    const float4 q = load16<SMEM>(rp + v);
    if (rdc_edge(dx, dy, q.x - ox, q.y - oy) > 0.0f) above |= 1u << (2 * v - 1);
    if (rdc_edge(dx, dy, q.z - ox, q.w - oy) > 0.0f) above |= 1u << (2 * v);
  }
  // chord j joins points j and j+1: crossed where their sides differ
  uint32_t crossed = (above ^ (above >> 1)) & ((1u << count) - 1u);
  if (crossed == 0) return count;
  const uint32_t first_id = __float_as_uint(head.x);
  const float2* pts = reinterpret_cast<const float2*>(rp) + 1;  // P0 follows the two header words
  while (crossed) {
    const int j = __ffs(crossed) - 1;
    crossed &= crossed - 1;
    const float2 pa = SMEM ? pts[j] : __ldg(pts + j), pb = SMEM ? pts[j + 1] : __ldg(pts + j + 1);
    const float wax = pa.x - ox, way = pa.y - oy, wbx = pb.x - ox, wby = pb.y - oy;
    float t, s;
    if (rdc_chord_hit(dx, dy, inv_dd, wax, way, wbx, wby, rdc_edge(dx, dy, wax, way), rdc_edge(dx, dy, wbx, wby), &t, &s)) {
      const uint32_t id = first_id + (uint32_t)j;
      if (!(PORTALS && id >= skip_lo && id <= skip_hi) && rdc_hit_closer(t, id, h.t, h.id)) {
        h.t = t; h.s = s; h.leaf = leaf; h.j = j; h.id = id;
      }
    }
  }
  return count;  // chords looked at
}

// Every run against the ray: the kernel behind RDC_TRAVERSAL_BRUTE_FORCE (validation only, kept out of line).
template <bool SMEM, bool PORTALS>
__device__ __noinline__ void brute_force(const Accel& ac, float ox, float oy, float dx, float dy, float inv_dd,
                                         uint32_t skip_lo, uint32_t skip_hi, Hit& h) {
  for (uint32_t r = 0; r < ac.n_runs; ++r) test_run<SMEM, PORTALS>(ac.runs + (size_t)r * kRunVec, (int)r, ox, oy, dx, dy, inv_dd, skip_lo, skip_hi, h);
}

template <int W>
__device__ __forceinline__ uint32_t pick_word(const uint32_t (&m)[W], int w) {
  uint32_t v = m[0];
#pragma unroll
  for (int k = 1; k < W; ++k) v = w == k ? m[k] : v;
  return v;
}

// slot -> run, distance bound and (local table only) padded box of the table in work
struct Slots {
  const uint32_t* run;
  const float* dist;
  const float4* box;  // nullptr: the whole-scene table reads ac.run_box[run]
};

template <bool SMEM, bool PORTALS, bool STATS>
__device__ __forceinline__ Hit closest_chord(const Accel& ac, bool brute, float ox, float oy, float dx, float dy, bool primary,
                                             uint32_t skip_lo, uint32_t skip_hi, float bound, Counters& cnt, int root = 0,
                                             bool whole_ray = true);

// One table entry against the ray: a run (test_run), or — cut mode — everything below a node of the tree, walked with the
// best hit so far as the bound. Returns true when the entry produced the new best hit.
template <bool SMEM, bool PORTALS, bool STATS, bool CUT>
__device__ __forceinline__ bool test_entry(const Accel& ac, int entry, float ox, float oy, float dx, float dy, Hit& h, Counters& cnt) {
  const int ref = CUT ? ac.slot_node[entry] : ~entry;
  if (!CUT || ref < 0) {
    const int run = ~ref;
    const uint32_t before = h.id;
    const int looked = test_run<SMEM, PORTALS>(ac.runs + (size_t)run * kRunVec, run, ox, oy, dx, dy, 1.0f, 1u, 0u, h);
    if (STATS) cnt.chords += looked;
    return h.id != before;
  }
  const Hit sub = closest_chord<SMEM, PORTALS, STATS>(ac, false, ox, oy, dx, dy, true, 1u, 0u, h.t, cnt, ref, false);
  if (sub.leaf >= 0 && rdc_hit_closer(sub.t, sub.id, h.t, h.id)) {
    h = sub;
    return true;
  }
  return false;
}

// Closest chord among the table slots named by two bit masks (slots 0..31 and 32..63): the replacement for
// the tree walk of primary rays. Whole-scene table (small scenes): slot = run. Local table: slot -> run
// through the warp's WarpLocal. The slot that the lane's previous ray hit goes first — neighbouring
// strata mostly hit the same run — which gives a tight bound early; every other candidate first has to
// pass the slab test of its padded box against that bound (the same conservative test the tree applies
// to a leaf's box), and most do not. Returns the hit with leaf = run.
template <bool SMEM, bool PORTALS, bool STATS, bool LOCAL, bool CUT, int W>
__device__ __forceinline__ Hit table_closest(const Accel& ac, const Slots& sl, uint32_t (&m)[W], int& last_slot, float ox,
                                             float oy, float dx, float dy, Counters& cnt) {
  if (STATS) cnt.rays++;
  Hit h = miss_hit(__int_as_float(0x7f800000));
  int best_slot = -1;
  uint32_t rest = 0u;
  if (last_slot >= 0) {
    const uint32_t bit = 1u << (last_slot & 31);
    const int word = last_slot >> 5;
    bool there = false;
#pragma unroll
    for (int k = 0; k < W; ++k)
      if (word == k && (m[k] & bit)) {
        m[k] &= ~bit;
        there = true;
      }
    if (there && test_entry<SMEM, PORTALS, STATS, CUT>(ac, (int)sl.run[last_slot], ox, oy, dx, dy, h, cnt)) best_slot = last_slot;
  }
#pragma unroll
  for (int k = 0; k < W; ++k) rest |= m[k];
  if (rest != 0u) {
    const SlabRay sr = slab_ray(ox, oy, dx, dy);
    bool open = true;  // slots come in order of distance — once one lies beyond the hit, all the rest do
#pragma unroll 1
    for (int w = 0; w < W && open; ++w) {
      uint32_t mw = pick_word<W>(m, w);
      while (mw) {
        const int slot = __ffs(mw) - 1 + 32 * w;
        mw &= mw - 1;
        if (sl.dist[slot] > h.t) {
          open = false;
          break;
        }
        const int entry = (int)sl.run[slot];
        const float4 b = LOCAL ? sl.box[slot] : ac.slot_box[entry];
        float te;
        const float tn = slab_enter(sr, b, &te);
        if (STATS) cnt.nodes++;
        if (tn <= te && tn <= h.t * RDC_CULL_SLACK && test_entry<SMEM, PORTALS, STATS, CUT>(ac, entry, ox, oy, dx, dy, h, cnt)) best_slot = slot;
      }
    }
  }
  if (best_slot >= 0) last_slot = best_slot;
  return h;
}

// Closest chord along the ray. Ordered depth-first traversal: the nearer child first, the farther one on
// a per-thread stack together with its entry distance, so that a subtree that lies behind a hit found in
// the meantime is dropped when it is popped, without fetching it. A child is entered when the ray's
// interval inside its box starts before the best hit so far (with RDC_CULL_SLACK). Leaves go through the
// same loop (one leaf-test site keeps the kernel inside the instruction cache). `bound`: nothing farther
// than this can be the answer (a deferred ray of the local table already has a candidate).
template <bool SMEM, bool PORTALS, bool STATS>
__device__ __forceinline__ Hit closest_chord(const Accel& ac, bool brute, float ox, float oy, float dx, float dy,
                                             bool primary, uint32_t skip_lo, uint32_t skip_hi, float bound, Counters& cnt,
                                             int root, bool whole_ray) {
  if (STATS && whole_ray) cnt.rays++;  // (a walk below one table entry is part of a ray the table already counted)
  Hit h = miss_hit(bound);  // +inf, or the distance of a hit already known (that hit is found again: ties go to the smaller id)
  const float inv_dd = PORTALS ? rdc_inv_dd(dx, dy, primary) : 1.0f;
  if (brute) {
    brute_force<SMEM, PORTALS>(ac, ox, oy, dx, dy, inv_dd, skip_lo, skip_hi, h);
    if (STATS) cnt.chords += ac.n_runs * RDC_RUN;  // upper bound
    return h;
  }
  const SlabRay sr = slab_ray(ox, oy, dx, dy);
  int2 stack[kStack];  // (node, entry distance bits)
  int sp = 0;
  // a scene of one run: its root's second child is a placeholder, and the run is tested without a box test at all
  int node = ac.n_runs == 1 ? ~0 : root;
  // while-while form (Aila & Laine 2009): every lane first walks inner nodes until it stands on a leaf (or has nothing
  // left), then the warp tests leaves together — a lane on a leaf no longer waits out its neighbours' node steps one
  // iteration at a time, and vice versa. Same visits in the same order per lane as the single if/else loop it replaces:
  // same bits; lady_bug.xml 1080p 8.49 -> 7.70 ms, dolphin.xml 4K 114.5 -> 109.4 ms on top of the fused slab test
  // (profiles/r02b/variants.log).
  constexpr int kDone = 0x7fffffff;
  for (;;) {
    while (node >= 0 && node != kDone) {
      if (STATS) cnt.nodes++;
      const float4* np = reinterpret_cast<const float4*>(ac.nodes + node);
      const float4 lb = load16<SMEM>(np), rb = load16<SMEM>(np + 1);
      const float4 ch = load16<SMEM>(np + 2);
      const int left = __float_as_int(ch.x), right = __float_as_int(ch.y);
      float le, re;
      const float ln = slab_enter(sr, lb, &le);
      const float rn = slab_enter(sr, rb, &re);
      const float lim = h.t * RDC_CULL_SLACK;
      const bool hl = ln <= le && ln <= lim;
      const bool hr = rn <= re && rn <= lim;
      if (hl && hr) {
        const bool left_first = ln <= rn;
        stack[sp++] = make_int2(left_first ? right : left, __float_as_int(left_first ? rn : ln));
        node = left_first ? left : right;
      } else if (hl || hr) {
        node = hl ? left : right;
      } else {
        node = kDone;
        while (sp > 0) {  // the nearest pending subtree that still starts before the best hit
          const int2 e = stack[--sp];
          if (__int_as_float(e.y) <= lim) {
            node = e.x;
            break;
          }
        }
      }
    }
    if (node == kDone) return h;
    const int looked = test_run<SMEM, PORTALS>(ac.runs + (size_t)(~node) * kRunVec, ~node, ox, oy, dx, dy, inv_dd, skip_lo, skip_hi, h);
    if (STATS) cnt.chords += looked;
    node = kDone;
    while (sp > 0) {
      const int2 e = stack[--sp];
      if (__int_as_float(e.y) <= h.t * RDC_CULL_SLACK) {
        node = e.x;
        break;
      }
    }
    if (node == kDone) return h;
  }
}

__device__ __forceinline__ void load_control_points(const DevScene& sc, uint32_t seg, rdc_f2 v[4]) {
  const float4* p = reinterpret_cast<const float4*>(sc.vertices + __ldg(sc.segment_indices + seg));
  float4 a = __ldg(p), b = __ldg(p + 1);
  v[0] = {a.x, a.y};
  v[1] = {a.z, a.w};
  v[2] = {b.x, b.y};
  v[3] = {b.z, b.w};
}

// A hit's walk data: the segment and u from the run's ids, the walk ranges of the segment (SegWalk: the stop walks start
// where the segment starts) and, finer, where this chord starts (chord_walk: the walks then rarely take a step); cu = u + ordinal.
struct HitWalks {
  uint32_t seg;
  float u, cu;
  uint4 wc, ws, wd, cw, cw2;
};

__device__ __forceinline__ HitWalks hit_walks(const DevScene& sc, const Hit& h) {
  HitWalks w;
  const uint4 id = __ldg(sc.run_ids + h.leaf);  // first chord id, segment, k of the first chord, K
  w.seg = id.y;
  w.u = rdc_hit_u((int)id.z + h.j, (int)id.w, h.s);
  const uint4* wp = reinterpret_cast<const uint4*>(sc.seg_walk + w.seg);
  w.wc = __ldg(wp), w.ws = __ldg(wp + 1), w.wd = __ldg(wp + 2);
  w.cw = __ldg(sc.chord_walk + 2 * (size_t)h.id), w.cw2 = __ldg(sc.chord_walk + 2 * (size_t)h.id + 1);
  w.cu = w.u + w.wd.w;
  return w;
}

// The stop cu interpolates from on a walk over [first,end) of a family's u list, the ratio, and the lerped value
struct ScalarStop {
  int ind;
  float ratio, value;
};

__device__ __forceinline__ ScalarStop stop_walk(const DevStops& st, uint32_t first, uint32_t end, float cu) {
  ScalarStop s;
  s.ind = rdc_interp_from(first, end, cu, st.u, &s.ratio);
  s.value = rdc_lerp_stop(__ldg(st.value + s.ind), __ldg(st.value + s.ind + 1), s.ratio);
  return s;
}

__device__ __forceinline__ float scalar_stop(const DevStops& st, uint32_t first, uint32_t end, float cu) {
  return stop_walk(st, first, end, cu).value;
}

// [first,end) selects the walk range, `us`/`rgb` the arrays (the portal filter mixes families, DeviceCode.cu:297); returns
// the index of the stop cu interpolates from
__device__ __forceinline__ int colour_stop(uint32_t first, uint32_t end, const float* us, const float4* rgb, float cu,
                                          float& ratio, float& r, float& g, float& b) {
  int ind = rdc_interp_from(first, end, cu, us, &ratio);
  float4 c0 = __ldg(rgb + ind), c1 = __ldg(rgb + ind + 1);
  r = rdc_lerp_color(c0.x, c1.x, ratio);
  g = rdc_lerp_color(c0.y, c1.y, ratio);
  b = rdc_lerp_color(c0.z, c1.z, ratio);
  return ind;
}

// The colour walk of a terminal hit: the right family's for a ray on the curve's right, the left one's otherwise
__device__ __forceinline__ int terminal_colour(const DevScene& sc, const HitWalks& w, bool right, float& ratio, float& r, float& g,
                                               float& b) {
  if (right) return colour_stop(w.cw.y, w.wc.w, sc.color_right.u, sc.color_right.rgb, w.cu, ratio, r, g, b);
  else return colour_stop(w.cw.x, w.wc.y, sc.color_left.u, sc.color_left.rgb, w.cu, ratio, r, g, b);
}

struct Sample {
  float r, g, b, w, blur;
};

// Shades a primary ray whose closest hit `h` is known and follows it through any number of portals
// (DeviceCode.cu:194-342, iteratively; continuation rays use the tree).
// Carried state: F = product of portal filters, Bp = product of portal blurs, S = sum of 1/w_portal;
// terminal hit: rgb = F*rgb_T, blur = Bp*blur_T, w = 1/(1/w_T + S) — the closed form of the reference's
// recursion w = 1/(1/w' + 1/w_here) (:310).
template <bool SMEM, bool PORTALS, bool STATS>
__device__ __forceinline__ Sample trace_from(const RenderArgs& a, const Accel& ac, Hit h, float ox, float oy, float dx, float dy,
                                             Counters& cnt) {
  const DevScene& sc = a.sc;
  Sample out{0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
  float Fr = 1.0f, Fg = 1.0f, Fb = 1.0f, Bp = 1.0f, S = 0.0f;
  int depth = 0;
  for (;;) {
    if (h.leaf < 0) return out;  // miss: contributes nothing (DeviceCode.cu:185-192)
    if (STATS) cnt.shaded++;
    // Shading records (device_scene.h): one 128-byte record instead of run ids -> walk hints -> stop parameters -> stop
    // values. Same operands, same operations, same bits as the walks below for a chord whose hits all interpolate
    // between the same two stops of every family (1.879 -> 1.762 ms on the headline frame).
    if (!PORTALS && sc.chord_records) {
      const float4* rec = sc.chord_records + 8 * (size_t)h.id;
      const float4 m4 = __ldg(rec + 7);
      if ((__float_as_uint(m4.w) >> 27) == 0x1Fu) {
        const uint32_t seg = __float_as_uint(m4.x), ordinal = __float_as_uint(m4.y), kk = __float_as_uint(m4.z);
        const float u = rdc_hit_u((int)(kk & 0xFFFFu), (int)(kk >> 16), h.s);
        const float cu = u + ordinal;
        const float4 sb = __ldg(rec), sw = __ldg(rec + 1), sd = __ldg(rec + 2);
        const float blur_here = rdc_lerp_stop(sb.z, sb.w, rdc_ratio(cu - sb.x, sb.y - sb.x));
        const float wm = rdc_lerp_stop(sw.z, sw.w, rdc_ratio(cu - sw.x, sw.y - sw.x));
        const float e = rdc_lerp_stop(sd.z, sd.w, rdc_ratio(cu - sd.x, sd.y - sd.x));
        rdc_f2 v[4];
        load_control_points(sc, seg, v);
        const bool right = rdc_is_ray_right(u, dx, dy, v[0], v[1], v[2], v[3], a.orzan != 0);
        const float4 c0 = __ldg(rec + (right ? 5 : 3)), c1 = __ldg(rec + (right ? 6 : 4));
        const float ratio = rdc_ratio(cu - c0.w, c1.w - c0.w);
        out.r = rdc_lerp_color(c0.x, c1.x, ratio);
        out.g = rdc_lerp_color(c0.y, c1.y, ratio);
        out.b = rdc_lerp_color(c0.z, c1.z, ratio);
        out.blur = blur_here;
        out.w = wm * rdc_weight_falloff(h.t, e);
        return out;
      }
    }
    const HitWalks hw = hit_walks(sc, h);
    const uint4* wp = reinterpret_cast<const uint4*>(sc.seg_walk + hw.seg);  // the portal filter's walk range: wp[3]
    const float u = hw.u, cu = hw.cu;
    const float blur_here = scalar_stop(sc.blur, hw.cw.z, hw.ws.y, cu);
    const float wm = scalar_stop(sc.weight, hw.cw.w, hw.ws.w, cu);
    const float e = scalar_stop(sc.weight_degree, hw.cw2.x, hw.wd.y, cu);
    const float w_here = wm * rdc_weight_falloff(h.t, e);
    rdc_f2 v[4];
    load_control_points(sc, hw.seg, v);
    const bool right = rdc_is_ray_right(u, dx, dy, v[0], v[1], v[2], v[3], a.orzan != 0);

    if (PORTALS) {
      const int target_curve = __ldg(sc.curve_connect + hw.wd.z);
      if (target_curve >= 0) {
        if (++depth > a.max_depth) return out;  // depth cap: regarded as a miss (:313-320)
        const uint32_t tseg = __ldg(sc.curve_map_inverse + target_curve) + hw.wd.w;
        rdc_f2 tv[4];
        load_control_points(sc, tseg, tv);
        rdc_f2 o2 = rdc_spline_point(u, tv[0], tv[1], tv[2], tv[3]);
        rdc_f2 n = rdc_spline_normal(u, v[0], v[1], v[2], v[3]);
        float nl = sqrtf(n.x * n.x + n.y * n.y);
        n.x /= nl; n.y /= nl;
        float rc = n.x * dx + n.y * dy;
        float rs = n.x * dy + n.y * dx;  // sic (:243)
        rdc_f2 m = rdc_spline_normal(u, tv[0], tv[1], tv[2], tv[3]);
        float ml = sqrtf(m.x * m.x + m.y * m.y);
        m.x /= ml; m.y /= ml;
        float ndx = m.x * rc - m.y * rs;
        float ndy = m.y * rc + m.x * rs;
        float fratio, fr, fg, fb;
        if (right) colour_stop(hw.cw.y, hw.wc.w, sc.color_right.u, sc.color_right.rgb, cu, fratio, fr, fg, fb);
        else {  // right list's range on the left arrays (:297)
          const uint4 wq = __ldg(wp + 3);
          colour_stop(hw.cw2.y, wq.y, sc.color_left.u, sc.color_left.rgb, cu, fratio, fr, fg, fb);
        }
        Fr *= fr; Fg *= fg; Fb *= fb;
        Bp *= blur_here;
        S += 1.0f / w_here;
        int klo, khi;
        const int Kt = (int)__ldg(sc.seg_chord_count + tseg);
        rdc_portal_skip(u, Kt, &klo, &khi);
        const uint32_t tbase = __ldg(sc.seg_chord_base + tseg);
        ox = o2.x; oy = o2.y; dx = ndx; dy = ndy;
        h = closest_chord<SMEM, PORTALS, STATS>(ac, a.brute != 0, ox, oy, dx, dy, false, tbase + (uint32_t)klo, tbase + (uint32_t)khi,
                                                __int_as_float(0x7f800000), cnt);
        continue;
      }
    }
    float ratio, r, g, b;
    terminal_colour(sc, hw, right, ratio, r, g, b);
    if (PORTALS && depth > 0) {
      out.r = Fr * r; out.g = Fg * g; out.b = Fb * b;
      out.blur = Bp * blur_here;
      out.w = 1.0f / (1.0f / w_here + S);
    } else {
      out.r = r; out.g = g; out.b = b;
      out.blur = blur_here;
      out.w = w_here;
    }
    return out;
  }
}

// k-th element of 0..n-1 ordered by distance from `mid`: mid, mid+1, mid-1, mid+2, ... and, once one side is used up, the rest
// of the other. A bijection of [0,n) for every mid in [0,n).
__device__ __forceinline__ uint32_t centre_out(uint32_t k, uint32_t mid, uint32_t n) {
  const uint32_t lo = mid, hi = n - 1 - mid, m = lo < hi ? lo : hi;
  if (k <= 2 * m) return (k & 1u) ? mid + (k + 1) / 2 : mid - k / 2;
  const uint32_t rest = k - 2 * m;
  return lo > hi ? mid - m - rest : mid + m + rest;
}

// Base direction of ray i: (1,0) rotated i times by the fp32 matrix of sincospi(2/N) — iterated, because
// the accumulated rounding is part of the ray set (DeviceCode.cu:99,110-112,167-171). Pixel-independent,
// so it is tabulated once per N.
__global__ void k_base_dirs(float2* out, int n_iter, float two_over_n) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  float rs, rc;
  rdc_sincospi(two_over_n, &rs, &rc);
  float x = 1.0f, y = 0.0f;
  for (int i = 0; i < n_iter; ++i) {
    out[i] = make_float2(x, y);
    float nx = x * rc - y * rs;
    float ny = x * rs + y * rc;
    x = nx; y = ny;
  }
}

// fewer than 8 rays per pixel: the jitter angle needs the range reduction (cold path, kept out of line)
__device__ __noinline__ void sincospi_general(float x, float* s, float* c) { rdc_sincospi(x, s, c); }

// atan2 to within 1e-4 rad (odd polynomial on [0,1], |error| < 2e-5, plus the approximate reciprocal): only
// used to bound an angular interval that is then widened by far more than that.
__device__ __forceinline__ float atan2_bound(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float hi = fmaxf(ax, ay), lo = fminf(ax, ay);
  float inv;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(fmaxf(hi, 1e-30f)));
  const float t = lo * inv, t2 = t * t;
  float r = fmaf(t2, -0.0134804700f, 0.0574773140f);
  r = fmaf(r, t2, -0.1212390710f);
  r = fmaf(r, t2, 0.1956359250f);
  r = fmaf(r, t2, -0.3329945970f);
  r = fmaf(r, t2, 0.9999956300f);
  r *= t;
  if (ay > ax) r = 1.5707963267948966f - r;
  if (x < 0.0f) r = 3.141592653589793f - r;
  return y < 0.0f ? -r : r;
}

// a rectangle of ray origins: [x0,x1] x [y0,y1]
struct Rect {
  float x0, x1, y0, y1;
};

// half the side of the square a pixel's ray origins are jittered in (DeviceCode.cu:135-136)
__device__ __forceinline__ float jitter(const RenderArgs& a) { return a.use_aa ? fabsf(a.zoom) : 0.0f; }

// Angular interval, in ray indices, under which `box` can be seen from ANY origin inside the rectangle
// `o`. Ray i leaves its origin in a direction whose angle lies in stratum (i, i+1]*2pi/N (base
// direction i plus a jitter of at most one stratum), so ray i can only hit the box if ((i - first) mod n) <= span.
// Returns false when nothing can be excluded (an origin may lie inside the box, or the interval covers all rays).
__device__ __forceinline__ bool angular_interval(float4 box, const Rect& o, int n, int& first, int& span) {
  // rounding of the subtractions below and of the origins themselves: a few ulp of the magnitudes involved
  const float mag = fabsf(o.x0) + fabsf(o.x1) + fabsf(o.y0) + fabsf(o.y1) + fabsf(box.x) + fabsf(box.y) + fabsf(box.z) + fabsf(box.w);
  const float m = 4e-6f * mag + 1e-6f;
  // the box relative to every possible origin (Minkowski difference)
  const float x0 = box.x - o.x1 - m, x1 = box.z - o.x0 + m;
  const float y0 = box.y - o.y1 - m, y1 = box.w - o.y0 + m;
  if (x0 <= 0.0f && x1 >= 0.0f && y0 <= 0.0f && y1 >= 0.0f) return false;
  const float cx = 0.5f * (x0 + x1), cy = 0.5f * (y0 + y1);
  float dmin = 0.0f, dmax = 0.0f;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float px = (c & 1) ? x1 : x0, py = (c & 2) ? y1 : y0;
    const float d = atan2_bound(cx * py - cy * px, cx * px + cy * py);  // signed angle from the centre direction
    dmin = fminf(dmin, d);
    dmax = fmaxf(dmax, d);
  }
  const float centre = atan2_bound(cy, cx);
  const float strata_per_rad = (float)n * 0.15915494309189535f;
  // safety: half a stratum, the drift of the iterated rotation (n steps of ~1e-7 rad, in strata) and the
  // error of atan2_bound (two of them meet in every interval end: 1e-3 rad covers it ten times over)
  const float safety = 0.5f + 4e-8f * (float)n * (float)n + 1e-3f * strata_per_rad;
  const float lo = (centre + dmin) * strata_per_rad - 1.0f - safety;  // ray i reaches up to stratum end i+1
  const float hi = (centre + dmax) * strata_per_rad + safety;
  const int ilo = (int)floorf(lo), ihi = (int)ceilf(hi);
  span = ihi - ilo;
  if (span >= n - 1) return false;
  first = ilo % n;
  if (first < 0) first += n;
  return true;
}

// bits [jlo, jhi] of a 32-bit word (empty when the range is)
__device__ __forceinline__ uint32_t bit_range(int jlo, int jhi) {
  jlo = max(jlo, 0);
  jhi = min(jhi, 31);
  if (jlo > jhi) return 0u;
  const int len = jhi - jlo + 1;
  return (len == 32 ? 0xFFFFFFFFu : (1u << len) - 1u) << jlo;
}

// For a run visible under ray indices {i : ((i - first) mod n) <= span}: which iterations j in [0, here) of
// the chunk starting at iteration cb (ray i = q + ((cb + j) << shift)) are among them.
__device__ __forceinline__ uint32_t iteration_mask(int first, int span, int q, int shift, int cb, int here, int n) {
  if (span < 0) return 0u;
  const uint32_t all = here == 32 ? 0xFFFFFFFFu : (1u << here) - 1u;
  if (span >= n - 1) return all;
  const int step = 1 << shift;
  auto rays = [&](int lo, int hi) {  // ray indices [lo, hi] -> iteration bits
    if (hi < q) return 0u;
    const int jlo = ((max(lo - q, 0) + step - 1) >> shift) - cb, jhi = ((hi - q) >> shift) - cb;
    return bit_range(jlo, jhi);
  };
  const int last = first + span;
  uint32_t m = rays(first, min(last, n - 1));
  if (last >= n) m |= rays(0, last - n);
  return m & all;
}

// Which rays of a pixel can reach the scene at all? (`o`: the pixel's jitter square)
__device__ __forceinline__ bool pixel_cull(const RenderArgs& a, const Rect& o, int& first, int& span) {
  const int n = a.n_iter;
  if (!a.cull || (float)n != a.n_rays || n < 8) return false;
  return angular_interval(a.sc.root_box, o, n, first, span);
}

// Origin and direction of primary ray i of a pixel (DeviceCode.cu:110-136): tabulated base direction,
// Philox draws in the reference's order (angle, x jitter, y jitter: :120,135,136).
__device__ __forceinline__ void gen_ray(const RenderArgs& a, uint32_t pixel, float base_x, float base_y, int i, bool small_angle,
                                        float& ox, float& oy, float& dx, float& dy) {
  const float2 base = __ldg(a.base_dirs + i);
  const rdc_u4 rnd = rdc_philox4x32_10(pixel, (uint32_t)i, 0u, 0u, a.seed, a.frame);
  ox = base_x; oy = base_y; dx = base.x; dy = base.y;
  if (a.use_aa) {
    float js, jc;
    const float ang = a.two_over_n * rdc_u01(rnd.x);
    if (small_angle) rdc_sincospi_kernel(ang, &js, &jc);
    else sincospi_general(ang, &js, &jc);
    dx = base.x * jc - base.y * js;
    dy = base.x * js + base.y * jc;
    ox = base_x + rdc_u01(rnd.y) * a.zoom;
    oy = base_y + rdc_u01(rnd.z) * a.zoom;
  }
}

// Largest axis gap between a box and the rectangle of origins `o`: a lower bound of the distance from any
// origin in the rectangle to any point of the box (0 when they overlap).
__device__ __forceinline__ float box_gap(float4 b, const Rect& o) {
  return fmaxf(fmaxf(fmaxf(b.x - o.x1, o.x0 - b.z), fmaxf(b.y - o.y1, o.y0 - b.w)), 0.0f);
}

// A distance bound `d` from the origins `o` (box gap, table radius), made smaller by the rounding of the gaps and of
// |D| = 1: a hit's t is its distance only up to those
__device__ __forceinline__ float shrunk(float d, const Rect& o) {
  return d * 0.9999f - (1e-5f * (fabsf(o.x0) + fabsf(o.x1) + fabsf(o.y0) + fabsf(o.y1)) + 1e-6f);
}

// Rank of each of the lane's K keys among keys[0, n): how many of them are smaller (keys are unique)
template <int K>
__device__ __forceinline__ void rank_keys(const uint32_t* keys, uint32_t n, const uint32_t (&key)[K], uint32_t (&rank)[K]) {
#pragma unroll
  for (int k = 0; k < K; ++k) rank[k] = 0u;
#pragma unroll 2
  for (uint32_t j = 0; j < n; ++j) {
    const uint32_t kj = keys[j];
#pragma unroll
    for (int k = 0; k < K; ++k) rank[k] += kj < key[k] ? 1u : 0u;
  }
}

struct LocalInfo {
  uint32_t n_slots;
  float radius;  // every run closer to the tile than this is in the table; +inf: the table holds the whole scene
};

// Local run table of a tile: the warp walks the tree breadth-first, 32 pending nodes per round, and collects
// the runs whose padded box comes closer than R to the tile's rectangle of origins (box_gap < R). The nearest
// kLocalSlots of them, sorted by that distance, become the table; its radius is R when all fit and the distance
// of the nearest run left out otherwise. A walk that overflows its buffers is repeated with a smaller R, one
// that finds less than half a table with a larger one. Everything here is a function of the tile and the scene
// only — no timing, no neighbours — so the table, and with it the order in which a pixel's rays are summed, is
// reproducible.
template <bool SMEM, bool STATS>
__device__ __forceinline__ LocalInfo gather_local(const Accel& ac, const Rect& o, float r0, WarpLocal* wlp, uint32_t lane,
                                                  Counters& cnt) {
  WarpLocal& wl = *wlp;
  const uint32_t below = (1u << lane) - 1u;
  const float inf = __int_as_float(0x7f800000);
  constexpr int kPer = kGatherCap / 32;  // candidates a lane looks after
  float R = r0;
  bool may_grow = true;
#pragma unroll 1
  for (int attempt = 0; attempt < kGatherAttempts; ++attempt) {
    uint32_t head = 0, tail = 1, found = 0;
    bool overflow = false;
    if (lane == 0) wl.ring[0] = 0u;
    __syncwarp();
#pragma unroll 1
    while (head < tail) {
      const uint32_t idx = head + lane;
      int left = 0, right = 0;
      float dl = inf, dr = inf;
      if (idx < tail) {
        const float4* np = reinterpret_cast<const float4*>(ac.nodes + wl.ring[idx % kGatherCap]);
        const float4 lb = load16<SMEM>(np), rb = load16<SMEM>(np + 1), ch = load16<SMEM>(np + 2);
        left = __float_as_int(ch.x);
        right = __float_as_int(ch.y);
        dl = box_gap(lb, o);
        dr = box_gap(rb, o);
        if (STATS) cnt.gathered++;
      }
      head = min(head + 32u, tail);
      const bool okl = dl < R, okr = dr < R;
      const uint32_t inner_l = __ballot_sync(0xFFFFFFFFu, okl && left >= 0), inner_r = __ballot_sync(0xFFFFFFFFu, okr && right >= 0);
      const uint32_t leaf_l = __ballot_sync(0xFFFFFFFFu, okl && left < 0), leaf_r = __ballot_sync(0xFFFFFFFFu, okr && right < 0);
      const uint32_t n_inner = __popc(inner_l) + __popc(inner_r), n_leaf = __popc(leaf_l) + __popc(leaf_r);
      if (tail - head + n_inner > (uint32_t)kGatherCap || found + n_leaf > (uint32_t)kGatherCap) {
        overflow = true;
        break;
      }
      __syncwarp();  // this round's nodes have been read: their ring entries may be overwritten
      if (okl) {
        if (left >= 0) wl.ring[(tail + __popc(inner_l & below)) % kGatherCap] = (uint32_t)left;
        else {
          const uint32_t at = found + __popc(leaf_l & below);
          wl.cand_run[at] = (uint32_t)~left;
          wl.cand_key[at] = (__float_as_uint(dl) & ~0xFFu) | at;  // gaps are >= 0: their bit patterns sort like the values
        }
      }
      if (okr) {
        if (right >= 0) wl.ring[(tail + __popc(inner_l) + __popc(inner_r & below)) % kGatherCap] = (uint32_t)right;
        else {
          const uint32_t at = found + __popc(leaf_l) + __popc(leaf_r & below);
          wl.cand_run[at] = (uint32_t)~right;
          wl.cand_key[at] = (__float_as_uint(dr) & ~0xFFu) | at;
        }
      }
      tail += n_inner;
      found += n_leaf;
      __syncwarp();
    }
    const bool last_try = attempt == kGatherAttempts - 1;
    if (overflow) {
      __syncwarp();
      R *= 0.6f;
      may_grow = false;
      continue;
    }
    if (found < (uint32_t)kLocalSlots / 2 && may_grow && found < ac.n_runs && !last_try) {
      R *= 2.0f;
      continue;
    }
    // rank every candidate by its key: the slot it gets
    uint32_t key[kPer], rank[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) key[k] = lane + 32u * k < found ? wl.cand_key[lane + 32u * k] : 0xFFFFFFFFu;
    rank_keys<kPer>(wl.cand_key, found, key, rank);
    float radius = R;
    if (found > (uint32_t)kLocalSlots) {  // the nearest run that is left out bounds the table
      uint32_t edge = 0u;
#pragma unroll
      for (int k = 0; k < kPer; ++k)
        if (rank[k] == (uint32_t)kLocalSlots && lane + 32u * k < found) edge = key[k] & ~0xFFu;
      radius = __uint_as_float(__reduce_max_sync(0xFFFFFFFFu, edge));
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k)
      if (lane + 32u * k < found && rank[k] < (uint32_t)kLocalSlots) {
        const uint32_t run = wl.cand_run[lane + 32u * k];
        wl.run[rank[k]] = run;
        wl.dist[rank[k]] = fmaxf(shrunk(__uint_as_float(key[k] & ~0xFFu), o), 0.0f);
        wl.box[rank[k]] = __ldg(ac.run_box + run);
      }
    __syncwarp();
    const uint32_t n_slots = min(found, (uint32_t)kLocalSlots);
    return LocalInfo{n_slots, n_slots == ac.n_runs ? inf : radius};
  }
  return LocalInfo{0u, 0.0f};  // too dense for a table at any radius tried: every ray goes to the tree
}

// pixel -> ray origin before the jitter (DeviceCode.cu:103-107: unsigned arithmetic, then a signed cast)
__device__ __forceinline__ float origin_x(const RenderArgs& a, uint32_t ix) {
  return (float)(int)(ix - (a.width / 2)) * a.zoom + a.off_x;
}
__device__ __forceinline__ float origin_y(const RenderArgs& a, uint32_t iy) {
  return a.orzan ? (float)(int)((a.height - iy) - (a.height / 2)) * a.zoom + a.off_y
                 : (float)(int)(iy - (a.height / 2)) * a.zoom + a.off_y;
}

// row of the full image for row `vy` of the output buffers (band- or strip-local, plus the skew): contiguous band, or
// strip (vy / kStripRows) of this rank's interleaved share
__device__ __forceinline__ uint32_t frame_row(const RenderArgs& a, uint32_t vy) {
  return (a.row_begin - a.row_skew) + ((vy / kStripRows) * a.strip_stride + a.strip_offset) * kStripRows + vy % kStripRows;
}

// the lane's pixel of a tile
struct Pixel {
  uint32_t pixel;         // global pixel index: split-independent random numbers
  size_t local;           // position in the output buffers
  float base_x, base_y;   // ray origin before the jitter
  bool valid;
};
__device__ __forceinline__ Pixel tile_pixel(const RenderArgs& a, uint32_t tile, uint32_t tiles_x, uint32_t lane) {
  const uint32_t ix = (tile % tiles_x) * kWarpTileW + lane % kWarpTileW;
  const uint32_t vy = (tile / tiles_x) * kWarpTileH + lane / kWarpTileW;
  const uint32_t iy = frame_row(a, vy);
  Pixel p;
  p.valid = ix < a.width && iy >= a.row_begin && iy < a.row_end;
  p.local = (size_t)(vy - a.row_skew) * a.width + ix;
  p.base_x = origin_x(a, ix);
  p.base_y = origin_y(a, iy);
  p.pixel = iy * a.width + ix;
  return p;
}

// the origins of every ray of a tile (all 32 pixels, jitter included)
__device__ __forceinline__ Rect tile_origins(const RenderArgs& a, uint32_t tile, uint32_t tiles_x) {
  const uint32_t tx0 = (tile % tiles_x) * kWarpTileW, gy0 = frame_row(a, (tile / tiles_x) * kWarpTileH);
  const float xa = origin_x(a, tx0), xb = origin_x(a, tx0 + (kWarpTileW - 1));
  const float ya = origin_y(a, gy0), yb = origin_y(a, gy0 + kWarpTileH - 1);
  const float jit = jitter(a);
  return Rect{fminf(xa, xb) - jit, fmaxf(xa, xb) + jit, fminf(ya, yb) - jit, fmaxf(ya, yb) + jit};
}

// a pixel's running sums (DeviceCode.cu:153-160)
struct PixelSums {
  float r = 0.0f, g = 0.0f, b = 0.0f, w = 0.0f, blur = 0.0f;
  __device__ __forceinline__ void add(const Sample& s) {
    w += s.w;
    r += s.r * s.w;
    g += s.g * s.w;
    b += s.b * s.w;
    blur += s.blur * s.w;
  }
};

// Group mode (table launches with more than one unit per tile): the G warps that take a tile's G units together. The
// tile's table (order, cut, slot intervals) is made once, by the group's first warp, in that warp's slot of the per-warp
// tables; everybody reads it from there.
struct Group {
  bool on;
  uint32_t G;         // warps per group = units per tile (2, 4 or 8); 1 when off
  uint32_t id;        // this warp's group inside the block
  uint32_t table_of;  // the group's first warp, which owns the tile's table
  GroupShared* gs;
  GroupTable* gt;
  // the group's warps meet at a barrier of their own (a named barrier; the whole block's when the group is the block)
  __device__ __forceinline__ void sync() const {
    if (G == (uint32_t)(kBlock / 32)) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(1u + id), "r"(32u * G) : "memory");
  }
};

// The per-warp tables of a launch in shared memory, behind the staged scene
struct WarpTables {
  WarpLocal* wl;  // local table: this warp's
  WarpCut* wc;    // cut table: the group's
  WarpOrder* wo;  // whole-scene and cut table: the group's
  Group grp;
};

// Stages nodes and runs (whole-scene table: and the runs' boxes) in shared memory, points `ac` at the scene and lays out
// the per-warp tables behind it.
template <bool SMEM, int MODE>
__device__ __forceinline__ WarpTables stage_scene(const RenderArgs& a, uint4* smem, Accel& ac) {
  constexpr bool CUT = MODE == kModeCut, TABLE = MODE == kModeTable || CUT, LOCAL = MODE == kModeLocal;
  ac.n_runs = a.sc.n_runs;
  uint32_t smem_words = 0;  // 16-byte words of dynamic shared memory handed out so far
  if (SMEM) {
    const uint32_t node_words = a.sc.n_nodes * (uint32_t)(sizeof(BvhNode) / 16);
    const uint32_t run_words = a.sc.n_runs * (uint32_t)kRunVec;
    const uint4* gn = reinterpret_cast<const uint4*>(a.sc.nodes);
    const uint4* gr = reinterpret_cast<const uint4*>(a.sc.runs);
    // once per persistent block: keep these loops rolled, the kernel has to fit the instruction cache
#pragma unroll 1
    for (uint32_t i = threadIdx.x; i < node_words; i += kBlock) smem[i] = __ldg(gn + i);
#pragma unroll 1
    for (uint32_t i = threadIdx.x; i < run_words; i += kBlock) smem[node_words + i] = __ldg(gr + i);
    ac.nodes = reinterpret_cast<const BvhNode*>(smem);
    ac.runs = reinterpret_cast<const float4*>(smem + node_words);
    ac.run_box = a.sc.run_box;
    smem_words = node_words + run_words;
    if (TABLE && !CUT) {
      const uint4* gb = reinterpret_cast<const uint4*>(a.sc.run_box);
#pragma unroll 1
      for (uint32_t i = threadIdx.x; i < a.sc.n_runs; i += kBlock) smem[smem_words + i] = __ldg(gb + i);
      ac.run_box = reinterpret_cast<const float4*>(smem + smem_words);
      smem_words += a.sc.n_runs;
    }
  } else {
    ac.nodes = a.sc.nodes;
    ac.runs = reinterpret_cast<const float4*>(a.sc.runs);
    ac.run_box = a.sc.run_box;
  }
  ac.slot_box = ac.run_box;  // whole-scene table: entry = run
  ac.slot_node = nullptr;
  if (SMEM) __syncthreads();
  const uint32_t warp = threadIdx.x >> 5;
  WarpTables t;
  Group& g = t.grp;
  g.on = TABLE && a.group != 0;
  g.G = g.on ? (uint32_t)a.group : 1u;
  g.id = g.on ? warp / g.G : 0u;
  g.table_of = g.on ? g.id * g.G : warp;
  t.wl = LOCAL ? reinterpret_cast<WarpLocal*>(smem + smem_words) + warp : nullptr;
  t.wc = CUT ? reinterpret_cast<WarpCut*>(smem + smem_words) + g.table_of : nullptr;
  t.wo = CUT ? &t.wc->order : TABLE ? reinterpret_cast<WarpOrder*>(smem + smem_words) + g.table_of : nullptr;
  g.gs = g.on ? reinterpret_cast<GroupShared*>(smem + smem_words + (kBlock / 32) * (CUT ? sizeof(WarpCut) : sizeof(WarpOrder)) / 16)
              : nullptr;
  g.gt = g.on ? &g.gs->table[g.id] : nullptr;
  if (CUT) {  // cut mode: table entries are the warp's own
    ac.slot_box = t.wc->box;
    ac.slot_node = t.wc->node;
  }
  return t;
}

// The warp's next work unit: its tile and its unit q of the tile's `split`; false when the frame is done.
// Units are handed out centre-out from the tile nearest the scene's centre, dearest first: a tile that looks at the scene
// from close by traces several times the rays of one far away, and a launch ends when its last unit does — with the long
// units up front the tail is made of short ones (a rank of 8 has 3.4 units per warp at 1080p: 0.264 ms where 0.221 is
// the mean). Which warp renders a tile when has no bearing on its pixels.
__device__ __forceinline__ bool fetch_unit(const RenderArgs& a, const Group& g, uint32_t tiles_x, uint32_t n_tile_rows,
                                           uint32_t& tile, uint32_t& q) {
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t n_units = tiles_x * n_tile_rows * a.split;
  uint32_t unit = 0;
  if (g.on) {
    g.sync();  // the previous tile is finished with: its table and partial sums may be overwritten
    if (warp == g.table_of && lane == 0) g.gt->tile = atomicAdd(a.work, 1u);
    g.sync();
    unit = g.gt->tile;  // (a tile, not a unit: the unit is the warp's number inside its group)
    if (unit >= n_units / a.split) return false;
  } else {
    if (lane == 0) unit = atomicAdd(a.work, 1u);
    unit = __shfl_sync(0xFFFFFFFFu, unit, 0);
    if (unit >= n_units) return false;
  }
  const uint32_t ord = g.on ? unit : unit / a.split;
  q = g.on ? warp - g.table_of : unit % a.split;
  tile = centre_out(ord / tiles_x, a.mid_ty, n_tile_rows) * tiles_x + centre_out(ord % tiles_x, a.mid_tx, tiles_x);
  return true;
}

// Cut table: start from the scene's seed cut and open the subtree nearest the tile, again and again, until the table
// is full or only leaves are left. Near the tile the entries end up as single runs (tested directly, like the
// whole-scene table's), far away they stay whole subtrees: the table is complete at any scene size and as fine as it
// needs to be where most rays end. A function of the tile and the scene only, like everything in the set-up.
// Returns the number of entries.
template <bool SMEM, bool STATS>
__device__ __forceinline__ uint32_t refine_cut(const RenderArgs& a, const Accel& ac, WarpCut* wc, const Rect& o, uint32_t lane,
                                               Counters& cnt) {
  if (lane < a.sc.n_cut) {
    wc->box[lane] = __ldg(a.sc.cut_box + lane);
    wc->node[lane] = __ldg(a.sc.cut_node + lane);
  }
  if (lane + 32u < a.sc.n_cut) {
    wc->box[lane + 32] = __ldg(a.sc.cut_box + lane + 32);
    wc->node[lane + 32] = __ldg(a.sc.cut_node + lane + 32);
  }
  uint32_t n_slots = a.sc.n_cut;
  __syncwarp();
#pragma unroll 1
  while (n_slots < kTableRuns) {
    uint32_t best = 0xFFFFFFFFu;
#pragma unroll
    for (int k = 0; k < kTableWords; ++k) {
      const uint32_t e = lane + 32u * k;
      if (e < n_slots && wc->node[e] >= 0) best = min(best, (__float_as_uint(box_gap(wc->box[e], o)) & ~0x3Fu) | e);
    }
    best = __reduce_min_sync(0xFFFFFFFFu, best);
    if (best == 0xFFFFFFFFu) break;  // only leaves left
    const uint32_t e = best & 0x3Fu;
    const float4* np = reinterpret_cast<const float4*>(ac.nodes + wc->node[e]);
    const float4 lb = load16<SMEM>(np), rb = load16<SMEM>(np + 1), ch = load16<SMEM>(np + 2);
    if (STATS && lane == 0) cnt.gathered++;
    __syncwarp();  // every lane has read the entry that is about to be replaced
    if (lane == 0) {
      wc->box[e] = lb;
      wc->node[e] = __float_as_int(ch.x);
      wc->box[n_slots] = rb;
      wc->node[n_slots] = __float_as_int(ch.y);
    }
    n_slots++;
    __syncwarp();
  }
  return n_slots;
}

// Whole-scene and cut table: put the entries in order of their distance from the tile (all-pairs ranking of at most 64
// keys, once per unit). A ray's candidates then come nearest first and its scan stops at the first slot beyond its hit:
// 0.41 boxes tested per ray instead of 0.77 on the headline frame.
__device__ __forceinline__ void order_table(const Accel& ac, WarpOrder* wo, uint32_t n_slots, const Rect& o, uint32_t lane) {
  uint32_t key[kTableWords], rank[kTableWords];
#pragma unroll
  for (int k = 0; k < kTableWords; ++k) {
    const uint32_t r = lane + 32u * k;
    key[k] = 0xFFFFFFFFu;
    if (r < n_slots) {  // gaps are >= 0: their bit patterns sort like the values; the entry in the low bits makes keys unique
      key[k] = (__float_as_uint(box_gap(ac.slot_box[r], o)) & ~0x3Fu) | r;
      wo->key[r] = key[k];
    }
  }
  __syncwarp();
  rank_keys<kTableWords>(wo->key, n_slots, key, rank);
#pragma unroll
  for (int k = 0; k < kTableWords; ++k)
    if (lane + 32u * k < n_slots) {
      wo->run[rank[k]] = lane + 32u * k;
      wo->dist[rank[k]] = fmaxf(shrunk(__uint_as_float(key[k] & ~0x3Fu), o), 0.0f);
    }
  __syncwarp();
}

// What a unit's ray loop needs of its tile's table
template <int W>
struct UnitTable {
  Slots sl;
  int first[W], span[W];  // ray-index interval of the lane's slots L, L+32, ...: span -1 never, n-1 always (local table: in WarpLocal)
  float settle_below;     // local table: a hit closer than this is final
  bool complete;          // the table holds every run: a miss is final, too
};

// The table ray loop of a unit: q traces rays i = q + j*split of the lane's pixel.
template <bool SMEM, bool PORTALS, bool STATS, int MODE, int W>
__device__ __forceinline__ void table_rays(const RenderArgs& a, const Accel& ac, WarpLocal* wl, UnitTable<W>& t, const Pixel& px,
                                           uint32_t q, bool small_angle, Counters& cnt, PixelSums& sum) {
  constexpr bool CUT = MODE == kModeCut, LOCAL = MODE == kModeLocal;
  const uint32_t lane = threadIdx.x & 31;
  const int n = a.n_iter, split = (int)a.split, shift = 31 - __clz(split);
  int last_slot = -1;       // the slot this lane's previous ray hit
  uint32_t queued = 0;      // deferred rays waiting in wl->ring
  // Deferred samples are summed apart from the direct ones and added at the end of the unit: when a batch
  // leaves depends on the other pixels of the tile (a band may cut some off), the two sums do not.
  if (LOCAL) {
#pragma unroll
    for (int c = 0; c < 5; ++c) wl->deferred[c][lane] = 0.0f;  // only ever touched by this lane: no barrier
  }

  // Up to 32 deferred rays, one per lane: regenerate the ray (owner's pixel, ray index), closest chord by the
  // tree under the known bound, shade; then the owners add the samples in queue order.
  auto flush = [&]() {
    const uint32_t batch = min(queued, 32u);
    uint32_t entry = 0;
    float bound = 0.0f;
    if (lane < batch) {
      entry = wl->ring[2 * lane];
      bound = __uint_as_float(wl->ring[2 * lane + 1]);
    }
    uint32_t move0 = 0, move1 = 0;
    const bool moves = lane + 32 < queued;
    if (moves) {
      move0 = wl->ring[2 * (lane + 32)];
      move1 = wl->ring[2 * (lane + 32) + 1];
    }
    __syncwarp();
    if (moves) {
      wl->ring[2 * lane] = move0;
      wl->ring[2 * lane + 1] = move1;
    }
    __syncwarp();
    queued -= batch;
    const uint32_t owner = entry >> 16;
    const int i = (int)(entry & 0xFFFFu);
    const uint32_t o_pixel = __shfl_sync(0xFFFFFFFFu, px.pixel, owner);
    const float o_bx = __shfl_sync(0xFFFFFFFFu, px.base_x, owner), o_by = __shfl_sync(0xFFFFFFFFu, px.base_y, owner);
    const uint32_t o_local = __shfl_sync(0xFFFFFFFFu, (uint32_t)px.local, owner);
    float pr = 0.0f, pg = 0.0f, pb = 0.0f, pw = 0.0f, pblur = 0.0f;
    if (lane < batch) {
      if (STATS) cnt.deferred++;
      float ox, oy, dx, dy;
      gen_ray(a, o_pixel, o_bx, o_by, i, small_angle, ox, oy, dx, dy);
      const Hit h = closest_chord<SMEM, PORTALS, STATS>(ac, false, ox, oy, dx, dy, true, 1u, 0u, bound, cnt);
      if (a.hit_ids) a.hit_ids[(size_t)o_local * (size_t)n + i] = h.id;
      const Sample s = trace_from<SMEM, PORTALS, STATS>(a, ac, h, ox, oy, dx, dy, cnt);
      pw = s.w; pr = s.r * s.w; pg = s.g * s.w; pb = s.b * s.w; pblur = s.blur * s.w;
    }
    // the running sums of the lane's deferred samples live in shared memory between batches (registers are
    // scarce in the ray loop); inside a batch they are continued in registers, one entry after the other in
    // queue order — where a batch ends must not matter to the bits
    float dw = wl->deferred[0][lane], dr = wl->deferred[1][lane], dg = wl->deferred[2][lane];
    float db = wl->deferred[3][lane], dblur = wl->deferred[4][lane];
#pragma unroll 1
    for (uint32_t k = 0; k < batch; ++k) {
      const uint32_t o = __shfl_sync(0xFFFFFFFFu, owner, k);
      const float w = __shfl_sync(0xFFFFFFFFu, pw, k), r = __shfl_sync(0xFFFFFFFFu, pr, k);
      const float g = __shfl_sync(0xFFFFFFFFu, pg, k), b = __shfl_sync(0xFFFFFFFFu, pb, k);
      const float bl = __shfl_sync(0xFFFFFFFFu, pblur, k);
      if (lane == o) {
        dw += w;
        dr += r; dg += g; db += b;
        dblur += bl;
      }
    }
    wl->deferred[0][lane] = dw; wl->deferred[1][lane] = dr; wl->deferred[2][lane] = dg;
    wl->deferred[3][lane] = db; wl->deferred[4][lane] = dblur;
  };

  // Which of this unit's rays (i = q + j*split) fall into the interval of the runs in slots L / L+32: one
  // bit per iteration j, 32 iterations at a time. The OR over all lanes lists the iterations that have any
  // candidate (local table: or that can reach the scene beyond the table); only those are visited.
  const int n_it = (int)q < n ? (n - 1 - (int)q) / split + 1 : 0;
  int cb0 = 0;  // first iteration of the current chunk
  uint32_t it[W], any = 0u;
  // masks of the chunk of 32 iterations that starts at cb0
  auto open_chunk = [&]() {
    const int here = min(32, n_it - cb0);
    uint32_t mine = 0u;
#pragma unroll
    for (int k = 0; k < W; ++k) {
      it[k] = LOCAL ? iteration_mask(wl->first[k][lane], wl->span[k][lane], (int)q, shift, cb0, here, n)
                    : iteration_mask(t.first[k], t.span[k], (int)q, shift, cb0, here, n);
      mine |= it[k];
    }
    any = __reduce_or_sync(0xFFFFFFFFu, mine);
    if (LOCAL) any |= iteration_mask(wl->root_first, wl->root_span, (int)q, shift, cb0, here, n);
    if (a.hit_ids && px.valid) {  // parity runs record every ray: mark the ones no run can reach
      uint32_t none = ~any & (here == 32 ? 0xFFFFFFFFu : (1u << here) - 1u);
      while (none) {
        const int j = __ffs(none) - 1;
        none &= none - 1;
        a.hit_ids[px.local * (size_t)n + (q + ((cb0 + j) << shift))] = kMiss;
      }
    }
  };
  // the next listed iteration of the chunk: one ray per lane
  auto next_ray = [&]() {
    const int j = __ffs(any) - 1;
    any &= any - 1;
    uint32_t m[W], m_any = 0u;
#pragma unroll
    for (int k = 0; k < W; ++k) {
      m[k] = __ballot_sync(0xFFFFFFFFu, (it[k] >> j) & 1u);
      m_any |= m[k];
    }
    const int i = (int)q + ((cb0 + j) << shift);
    bool defer = false;
    float bound = __int_as_float(0x7f800000);
    if (px.valid) {
      float ox, oy, dx, dy;
      gen_ray(a, px.pixel, px.base_x, px.base_y, i, small_angle, ox, oy, dx, dy);
      const Hit h = !LOCAL || m_any != 0u ? table_closest<SMEM, PORTALS, STATS, LOCAL, CUT, W>(ac, t.sl, m, last_slot, ox, oy, dx, dy, cnt)
                                          : miss_hit(__int_as_float(0x7f800000));
      if (LOCAL && !(h.leaf >= 0 ? h.t < t.settle_below : t.complete)) {
        defer = true;
        bound = h.t;
      } else {
        if (a.hit_ids) a.hit_ids[px.local * (size_t)n + i] = h.id;
        sum.add(trace_from<SMEM, PORTALS, STATS>(a, ac, h, ox, oy, dx, dy, cnt));
      }
    }
    if (LOCAL) {
      const uint32_t votes = __ballot_sync(0xFFFFFFFFu, defer);
      if (defer) {
        const uint32_t at = queued + __popc(votes & ((1u << lane) - 1u));
        wl->ring[2 * at] = (lane << 16) | (uint32_t)i;  // at < kDeferCap: at most 31 wait when up to 32 arrive
        wl->ring[2 * at + 1] = __float_as_uint(bound);
      }
      queued += __popc(votes);
      __syncwarp();
    }
  };
  if constexpr (!LOCAL) {
#pragma unroll 1
    for (; cb0 < n_it; cb0 += 32) {
      open_chunk();
      while (any) next_ray();
    }
  } else {
    // one loop, so that the deferred rays have ONE site (the tree walk and the shading are inlined there):
    // a full batch, or whatever is left when the unit ends
    cb0 = -32;
#pragma unroll 1
    for (;;) {
      while (any == 0u && cb0 + 32 < n_it) {
        cb0 += 32;
        open_chunk();
      }
      const bool done = any == 0u;
      if (!done) next_ray();
      if (queued >= 32u || (done && queued > 0u)) flush();
      if (done) break;
    }
    sum.w += wl->deferred[0][lane];
    sum.r += wl->deferred[1][lane];
    sum.g += wl->deferred[2][lane];
    sum.b += wl->deferred[3][lane];
    sum.blur += wl->deferred[4][lane];
  }
}

// The tree's ray loop of a unit: the rays of the pixel that can reach the scene, [lo0,hi0] and (when the angular range
// wraps) [lo1,hi1], visited in ascending order like the reference's loop. Everything else is a miss and adds nothing.
template <bool SMEM, bool PORTALS, bool STATS>
__device__ __forceinline__ void tree_rays(const RenderArgs& a, const Accel& ac, const Pixel& px, uint32_t q, bool small_angle,
                                          Counters& cnt, PixelSums& sum) {
  int lo0 = 0, hi0 = a.n_iter - 1, lo1 = 1, hi1 = 0;
  int cull_first = 0, cull_span = 0;
  const float jit = jitter(a);
  if (pixel_cull(a, Rect{px.base_x - jit, px.base_x + jit, px.base_y - jit, px.base_y + jit}, cull_first, cull_span)) {
    if (a.hit_ids)  // parity runs record every ray: mark the culled ones
#pragma unroll 1
      for (int i = (int)q; i < a.n_iter; i += (int)a.split) {
        int rel = i - cull_first;
        if (rel < 0) rel += a.n_iter;
        if (rel > cull_span) a.hit_ids[px.local * (size_t)a.n_iter + i] = kMiss;
      }
    const int last = cull_first + cull_span;
    if (last < a.n_iter) {
      lo0 = cull_first; hi0 = last;
    } else {  // wraps past ray N-1
      lo0 = 0; hi0 = last - a.n_iter;
      lo1 = cull_first; hi1 = a.n_iter - 1;
    }
  }
#pragma unroll 1
  for (int part = 0; part < 2; ++part) {
    const int lo = part ? lo1 : lo0, hi = part ? hi1 : hi0;
    // first index >= lo that belongs to this unit
    int i = lo + (int)((q + a.split - (uint32_t)lo % a.split) % a.split);
    for (; i <= hi; i += (int)a.split) {
      float ox, oy, dx, dy;
      gen_ray(a, px.pixel, px.base_x, px.base_y, i, small_angle, ox, oy, dx, dy);
      const Hit h = closest_chord<SMEM, PORTALS, STATS>(ac, a.brute != 0, ox, oy, dx, dy, true, 1u, 0u, __int_as_float(0x7f800000), cnt);
      if (a.hit_ids) a.hit_ids[px.local * (size_t)a.n_iter + i] = h.id;
      sum.add(trace_from<SMEM, PORTALS, STATS>(a, ac, h, ox, oy, dx, dy, cnt));
    }
  }
}

// A pixel's sums from its units' partial sums, added in unit order 0..split-1 — the same order whether they meet in
// shared or in global memory, so a pixel's bits do not depend on which path ran. rgbw(k), blur(k): unit k's partial sums.
template <class RGBW, class Blur>
__device__ __forceinline__ void add_units(uint32_t split, RGBW rgbw, Blur blur, PixelSums& s) {
  const float4 p0 = rgbw(0u);
  s.r = p0.x; s.g = p0.y; s.b = p0.z; s.w = p0.w;
  s.blur = blur(0u);
#pragma unroll 1
  for (uint32_t k = 1; k < split; ++k) {
    const float4 pk = rgbw(k);
    s.r += pk.x; s.g += pk.y; s.b += pk.z; s.w += pk.w;
    s.blur += blur(k);
  }
}

// Brings a tile's units together. Returns true for the warp that finishes the tile's pixels, with their sums in `s`.
__device__ __forceinline__ bool combine_units(const RenderArgs& a, const Group& g, uint32_t tile, uint32_t tiles_x, uint32_t q,
                                              const Pixel& px, PixelSums& s) {
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (g.on) {
    // the tile's units end together: partial sums meet in shared memory and the group's first warp adds them up
    g.gs->part_rgbw[warp][lane] = make_float4(s.r, s.g, s.b, s.w);
    g.gs->part_blur[warp][lane] = s.blur;
    g.sync();
    if (warp != g.table_of) return false;
    const float4* gr = &g.gs->part_rgbw[g.table_of][lane];
    const float* gb = &g.gs->part_blur[g.table_of][lane];
    add_units(a.split, [=](uint32_t k) { return gr[32 * k]; }, [=](uint32_t k) { return gb[32 * k]; }, s);
    return true;
  }
  if (a.split == 1) return true;
  // each unit leaves its partial sums in global memory and the last one to arrive adds them up
  const size_t part_stride = (size_t)a.local_rows * a.width;
  if (px.valid) {
    a.part_rgbw[q * part_stride + px.local] = make_float4(s.r, s.g, s.b, s.w);
    a.part_blur[q * part_stride + px.local] = s.blur;
  }
  __threadfence();
  __syncwarp();  // every lane's partial sums are out before lane 0 announces the unit
  unsigned int arrived = 0;
  if (lane == 0) arrived = atomicAdd(a.tile_arrivals + tile, 1u);
  arrived = __shfl_sync(0xFFFFFFFFu, arrived, 0);
  if (arrived != a.split - 1) return false;
  __threadfence();
  if (lane == 0) a.tile_arrivals[tile] = 0u;  // rewound for the next frame
  if (px.valid) {
    const float4* pr = a.part_rgbw + px.local;
    const float* pb = a.part_blur + px.local;
    add_units(a.split, [=](uint32_t k) { return __ldcg(pr + k * part_stride); }, [=](uint32_t k) { return __ldcg(pb + k * part_stride); }, s);
  }
  // The partial sums are dead now, but their lines would still be written back to HBM when L2 evicts them —
  // 4x the frame's algorithmic bytes (profiles/r01c_k_render_arch_ncu_summary.txt: 155 MB written for a 41 MB
  // frame). A tile row's eight float4 are exactly one aligned 128-byte line when the row lies inside the image:
  // tell L2 to drop it. Measured (profiles/r01c_discard_partials.log): 155 -> 30 MB written, frame time unchanged.
  __syncwarp();  // every lane of the row has its partial sums
  const uint32_t row_x0 = (tile % tiles_x) * kWarpTileW;
  if ((lane & 7u) == 0u && px.valid && row_x0 + kWarpTileW <= a.width) {
#pragma unroll 1
    for (uint32_t k = 0; k < a.split; ++k) {
      const float4* line = a.part_rgbw + k * part_stride + px.local;
      if ((reinterpret_cast<uintptr_t>(line) & 127u) == 0u) asm volatile("discard.global.L2 [%0], 128;" ::"l"(line) : "memory");
    }
  }
  return true;
}

// all rays missed -> 0/0 = NaN, as in the reference (DeviceCode.cu:176-181); .w is set to 1
__device__ __forceinline__ void write_pixel(const RenderArgs& a, const Pixel& px, const PixelSums& s, float& sigma_max) {
  const float4 rgb1 = make_float4(s.r / s.w, s.g / s.w, s.b / s.w, 1.0f);
  const float sigma = s.blur / s.w;
  if (a.n_targets == 0) {
    a.image[px.local] = rgb1;
    a.blur_map[px.local] = sigma;
  } else {
    // multi-GPU: straight to the pixel's place in every target frame — stores over NVLink when the frame
    // lives on a peer (8 pixels x 16 B = one 128-byte line per tile row), no gather afterwards
#pragma unroll 1
    for (uint32_t t = 0; t < a.n_targets; ++t) {
      a.target_image[t][px.pixel] = rgb1;
      a.target_blur[t][px.pixel] = sigma;
    }
  }
  sigma_max = fmaxf(sigma_max, sigma);  // NaN and negative sigmas do not raise the flag (the blur yields NaN for them either way)
}

// the counting build: the warp's work counters, and when the first and the last warp ran out of work
__device__ __forceinline__ void flush_counters(const RenderArgs& a, const Counters& cnt, uint32_t lane) {
  unsigned int r = __reduce_add_sync(0xFFFFFFFFu, cnt.rays), n = __reduce_add_sync(0xFFFFFFFFu, cnt.nodes);
  unsigned int c = __reduce_add_sync(0xFFFFFFFFu, cnt.chords), h = __reduce_add_sync(0xFFFFFFFFu, cnt.shaded);
  unsigned int d = __reduce_add_sync(0xFFFFFFFFu, cnt.deferred), g = __reduce_add_sync(0xFFFFFFFFu, cnt.gathered);
  if (lane == 0) {
    atomicAdd(a.stats + 0, (unsigned long long)r);
    atomicAdd(a.stats + 1, (unsigned long long)n);
    atomicAdd(a.stats + 2, (unsigned long long)c);
    atomicAdd(a.stats + 3, (unsigned long long)h);
    atomicAdd(a.stats + 4, (unsigned long long)d);
    atomicAdd(a.stats + 5, (unsigned long long)g);
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    atomicMin(a.stats + 7, now);
    atomicMax(a.stats + 8, now);
  }
}

// Persistent warps: every warp of the (SM-filling) grid keeps fetching work units from one global
// counter until the image is done. A tile is 8x4 pixels, one lane per pixel, all lanes on the same ray
// index — the most coherent mapping. Tiles differ in cost by an order of magnitude (how many rays reach
// the scene, how deep they go), and a lane that runs all N rays of a pixel back to back holds its warp
// for ~0.4 ms at 1080p/128 — far too coarse a grain to balance a 2.5 ms frame, let alone an eighth of it.
// So a tile's rays are dealt to `split` units (unit q takes rays i = q mod split); the units' partial sums
// are added up in unit order 0..split-1 (combine_units), which makes the result independent of timing and of
// how the frame is divided among GPUs.
template <bool SMEM, bool PORTALS, bool STATS, int MODE>
__global__ void __launch_bounds__(kBlock, kMinBlocks) k_render(const RenderArgs a) {
  constexpr bool CUT = MODE == kModeCut, TABLE = MODE == kModeTable || CUT, LOCAL = MODE == kModeLocal;
  constexpr int W = LOCAL ? kLocalWords : kTableWords;  // lane L looks after table slots L, L+32, ...
  extern __shared__ uint4 smem[];
  Accel ac;
  const WarpTables wt = stage_scene<SMEM, MODE>(a, smem, ac);
  const Group& grp = wt.grp;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tiles_x = (a.width + kWarpTileW - 1) / kWarpTileW;
  // Tiles are cut on the full frame's grid (rows 0-3, 4-7, ...) whatever band this launch renders: a tile's run
  // table, and with it the order in which its pixels' rays are summed, must not depend on the band.
  const uint32_t n_tile_rows = (a.local_rows + a.row_skew + kWarpTileH - 1) / kWarpTileH;
  const bool small_angle = a.two_over_n <= 0.25f && a.two_over_n >= 0.0f;  // N >= 8: no range reduction (bit-identical)
  float sigma_max = 0.0f;
  Counters cnt;
  if (STATS && lane == 0) {  // launch timeline of the counting build: when did the launch start ...
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    atomicMin(a.stats + 6, now);
  }
  uint32_t tile, q;
  while (fetch_unit(a, grp, tiles_x, n_tile_rows, tile, q)) {
    const Pixel px = tile_pixel(a, tile, tiles_x, lane);
    PixelSums sum;
    if (TABLE || LOCAL) {
      // Run table: lane L works out, once per unit, under which ray indices the runs in slots L and L+32 can
      // be seen from anywhere in the tile (all 32 pixels, jitter included). A ballot then tells every lane
      // which slots ray i has to be tested against — usually one or two, and none at all for most rays of a
      // sparse scene, which are then never generated. No tree walk.
      //  * whole-scene table (at most 64 runs): slot = run, every ray is settled by the table;
      //  * cut table: slot = subtree or run of the tile's own cut through the tree, every ray is settled by the table;
      //  * local table (larger scenes): the slots hold the runs within `radius` of the tile (gather_local).
      //    A hit closer than the radius is final — no run outside the table has a point that close. Any other
      //    ray (farther hit, or none) is deferred: queued and, 32 at a time, sent through the tree with its
      //    hit distance as the bound, one deferred ray per lane.
      const Rect o = tile_origins(a, tile, tiles_x);
      const int n = a.n_iter;
      const bool makes_table = !grp.on || warp == grp.table_of;
      UnitTable<W> t;
      t.settle_below = __int_as_float(0x7f800000);
      t.complete = true;
      uint32_t n_slots = CUT ? a.sc.n_cut : ac.n_runs;
      if (LOCAL) {
        const LocalInfo li = gather_local<SMEM, STATS>(ac, o, a.local_r0, wt.wl, lane, cnt);
        n_slots = li.n_slots;
        t.complete = li.radius == __int_as_float(0x7f800000);
        t.settle_below = shrunk(li.radius, o);
        int first_root = 0, span_root = -1;  // the rays that can reach the scene at all
        if (!t.complete && !angular_interval(a.sc.root_box, o, n, first_root, span_root)) {
          first_root = 0; span_root = n - 1;
        }
        if (lane == 0) {
          wt.wl->root_first = first_root;
          wt.wl->root_span = span_root;
        }
      }
      if (CUT && makes_table) n_slots = refine_cut<SMEM, STATS>(a, ac, wt.wc, o, lane, cnt);
      if (TABLE && makes_table) order_table(ac, wt.wo, n_slots, o, lane);
      t.sl = Slots{LOCAL ? wt.wl->run : wt.wo->run, LOCAL ? wt.wl->dist : wt.wo->dist, LOCAL ? wt.wl->box : nullptr};
#pragma unroll
      for (int k = 0; k < W; ++k) {
        t.first[k] = 0; t.span[k] = -1;
        if (makes_table && lane + 32u * k < n_slots &&
            !angular_interval(LOCAL ? wt.wl->box[lane + 32 * k] : ac.slot_box[wt.wo->run[lane + 32 * k]], o, n, t.first[k], t.span[k])) {
          t.first[k] = 0; t.span[k] = n - 1;
        }
        if (LOCAL) {
          wt.wl->first[k][lane] = t.first[k];
          wt.wl->span[k][lane] = t.span[k];
        }
      }
      if (TABLE && grp.on) {  // the group's first warp made the table: hand the slots' intervals to the others
        if (makes_table) {
#pragma unroll
          for (int k = 0; k < W; ++k) {
            grp.gt->first[lane + 32 * k] = t.first[k];
            grp.gt->span[lane + 32 * k] = t.span[k];
          }
        }
        grp.sync();
#pragma unroll
        for (int k = 0; k < W; ++k) {
          t.first[k] = grp.gt->first[lane + 32 * k];
          t.span[k] = grp.gt->span[lane + 32 * k];
        }
      }
      table_rays<SMEM, PORTALS, STATS, MODE, W>(a, ac, wt.wl, t, px, q, small_angle, cnt, sum);
    } else if (px.valid) {
      tree_rays<SMEM, PORTALS, STATS>(a, ac, px, q, small_angle, cnt, sum);
    }
    if (combine_units(a, grp, tile, tiles_x, q, px, sum) && px.valid) write_pixel(a, px, sum, sigma_max);
  }
  __syncwarp();
  if (a.max_sigma) {
    unsigned int bits = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(sigma_max));
    if (lane == 0 && bits != 0u) atomicMax(reinterpret_cast<unsigned int*>(a.max_sigma), bits);
  }
  if (STATS) flush_counters(a, cnt, lane);
  // the last warp to leave rewinds the tile counter for the next launch on this handle
  if (lane == 0) {
    const unsigned int warps = gridDim.x * (kBlock / 32);
    if (atomicAdd(a.work + 1, 1u) == warps - 1) {
      a.work[0] = 0u;
      a.work[1] = 0u;
    }
  }
}

// The kernels that are built, indexed by variant_index: the table mode only with shared-memory staging, the counting
// build only on the portals kernel (which it always uses).
typedef void (*RenderKernel)(RenderArgs);
constexpr int kVariants = 4 * 2 * 2 * 2;
constexpr int variant_index(int mode, bool smem, bool portals, bool stats) {
  return ((mode * 2 + (smem ? 1 : 0)) * 2 + (portals ? 1 : 0)) * 2 + (stats ? 1 : 0);
}
template <int V>
constexpr RenderKernel variant_kernel() {
  constexpr int mode = V >> 3;
  constexpr bool smem = V & 4, portals = V & 2, stats = V & 1;
  if constexpr ((mode == kModeTable && !smem) || (stats && !portals)) return nullptr;
  else return k_render<smem, portals, stats, mode>;
}
template <int... V>
constexpr std::array<RenderKernel, kVariants> kernel_table(std::integer_sequence<int, V...>) {
  return {variant_kernel<V>()...};
}
const std::array<RenderKernel, kVariants> kKernels = kernel_table(std::make_integer_sequence<int, kVariants>{});
static_assert(sizeof(rdc_scene::grid_blocks) == kVariants * sizeof(uint32_t), "one grid size per variant");

// Everything about a launch that follows from the scene and the frame parameters alone.
struct LaunchPlan {
  int n_iter = 0;
  int mode = kModeTree;
  bool smem = false, portals = false;
  uint32_t group = 0;  // warps per group in group mode (= split), 0 = off
  float local_r0 = 0.0f;
  size_t dyn = 0;
  int variant = 0;  // variant_index of the kernel
  uint32_t split = 1, strip_stride = 1, strip_offset = 0, local_rows = 0, row_skew = 0, local_tiles = 0;
  size_t local_pixels = 0;
};

// Widening of every box for a launch (SlabRay): the largest coordinate any of its ray origins can have is
// M = max(|offset_x|, |offset_y|) + (max(width, height) / 2 + 2) |zoom| (pixel index, anti-aliasing jitter and rounding);
// portal continuation rays start on the scene, within its extent. The slab and chord tests move a box by up to
// ~6 x 2^-23 x max(M, extent); the padding alone exceeds 16 x 2^-23 x extent (4e-6 = 33.5 x 2^-23), so
// w = max(0, 16 x 2^-23 x M - pad) makes padding + w >= 16 x 2^-23 x max(M, extent).
float slab_widening(const rdc_scene* s, const rdc_frame_params& p) {
  const double m = std::fmax(std::fabs((double)p.offset_x), std::fabs((double)p.offset_y)) +
                   (0.5 * std::max(p.image_width, p.image_height) + 2.0) * std::fabs((double)p.zoom_factor);
  const double w = 16.0 * std::ldexp(1.0, -23) * m * (1.0 + 1e-6) - (double)s->info.pad;
  return std::isfinite(w) && w > 0.0 ? (float)w : 0.0f;
}

__device__ __forceinline__ float4 widen_box(float4 b, float w) { return make_float4(b.x - w, b.y - w, b.z + w, b.w + w); }

// every box the traversal and the tables read, widened by w: node child boxes, run boxes, seed-cut boxes
__global__ void k_widen_boxes(DevScene src, float w, BvhNode* nodes, float4* run_box, float4* cut_box) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < src.n_nodes) {
    BvhNode n = src.nodes[i];
    n.lbox = widen_box(n.lbox, w);
    n.rbox = widen_box(n.rbox, w);
    nodes[i] = n;
  }
  if (i < src.n_runs) run_box[i] = widen_box(src.run_box[i], w);
  if (i < src.n_cut) cut_box[i] = widen_box(src.cut_box[i], w);
}

// The scene as a launch with widening w reads it: the scene itself for w = 0, else the handle's widened copies of its
// boxes, (re)made on `stream` when w differs from the last launch's (the handle's launches are serialised).
int widened_boxes(rdc_scene* s, float w, cudaStream_t stream, DevScene* out) {
  *out = s->dev;
  if (w == 0.0f) return 0;
  if (!s->wide_nodes) {
    RDC_CUDA(cudaMalloc((void**)&s->wide_nodes, (size_t)s->dev.n_nodes * sizeof(BvhNode)));
    s->allocations.push_back(s->wide_nodes);
  }
  if (!s->wide_run_box) {
    RDC_CUDA(cudaMalloc((void**)&s->wide_run_box, (size_t)s->dev.n_runs * sizeof(float4)));
    s->allocations.push_back(s->wide_run_box);
  }
  if (s->dev.n_cut && !s->wide_cut_box) {
    RDC_CUDA(cudaMalloc((void**)&s->wide_cut_box, (size_t)s->dev.n_cut * sizeof(float4)));
    s->allocations.push_back(s->wide_cut_box);
  }
  if (s->wide_w != w) {
    const uint32_t n = std::max(std::max(s->dev.n_nodes, s->dev.n_runs), s->dev.n_cut);
    k_widen_boxes<<<(n + 255) / 256, 256, 0, stream>>>(s->dev, w, s->wide_nodes, s->wide_run_box, s->wide_cut_box);
    RDC_CUDA(cudaGetLastError());
    s->wide_w = w;
  }
  out->nodes = s->wide_nodes;
  out->run_box = s->wide_run_box;
  if (s->dev.n_cut) out->cut_box = s->wide_cut_box;
  return 0;
}

int check_params(const rdc_frame_params& p) {
  if (p.image_width == 0 || p.image_height == 0 || p.row_begin >= p.row_end || p.row_end > p.image_height) {
    set_error("render: bad image size or row band [%u,%u) of %u", p.row_begin, p.row_end, p.image_height);
    return RDC_E_INVALID;
  }
  if (!(p.number_of_rays_per_pixel >= 1.0f) || p.number_of_rays_per_pixel > 65536.0f) {
    set_error("render: rays per pixel must be in [1, 65536]");
    return RDC_E_INVALID;
  }
  if (p.strip_stride > 1 && p.strip_offset >= p.strip_stride) {
    set_error("render: strip_offset %u must be below strip_stride %u", p.strip_offset, p.strip_stride);
    return RDC_E_INVALID;
  }
  if (p.max_trace_depth < 0 || p.max_trace_depth > 31) {
    set_error("render: max_trace_depth must be in [0, 31]");
    return RDC_E_INVALID;
  }
  if ((uint64_t)p.image_width * p.image_height > 0xFFFFFFFFull) {
    set_error("render: more than 2^32 pixels");
    return RDC_E_LIMIT;
  }
  if (p.route < RDC_ROUTE_AUTO || p.route > RDC_ROUTE_CUT_TABLE) {
    set_error("render: unknown route %d", p.route);
    return RDC_E_INVALID;
  }
  if (p.units_per_tile != 0 && p.units_per_tile != 1 && p.units_per_tile != 2 && p.units_per_tile != 4 && p.units_per_tile != (uint32_t)kMaxSplit) {
    set_error("render: units_per_tile must be 0 (automatic), 1, 2, 4 or 8");
    return RDC_E_INVALID;
  }
  if (!(p.local_radius >= 0.0f)) {
    set_error("render: local_radius must be 0 (automatic) or positive");
    return RDC_E_INVALID;
  }
  return 0;
}

LaunchPlan plan_launch(const rdc_scene* s, const rdc_frame_params& p) {
  LaunchPlan L;
  L.n_iter = (int)ceilf(p.number_of_rays_per_pixel);
  L.strip_stride = p.strip_stride > 1 ? p.strip_stride : 1;
  L.strip_offset = p.strip_stride > 1 ? p.strip_offset : 0;
  const uint32_t rows = p.row_end - p.row_begin;
  const uint32_t strips = (rows + kStripRows - 1) / kStripRows;  // of the band; this call renders those with t % stride == offset
  const uint32_t my_strips = L.strip_offset < strips ? (strips - L.strip_offset + L.strip_stride - 1) / L.strip_stride : 0;
  L.local_rows = L.strip_stride > 1 ? my_strips * kStripRows : rows;
  L.row_skew = L.strip_stride > 1 ? 0u : p.row_begin % kWarpTileH;  // strips: give row_begin as a multiple of 4 for split-independent bits
  const size_t scene_bytes = (size_t)s->dev.n_nodes * sizeof(BvhNode) + (size_t)s->dev.n_runs * sizeof(RunRecord);
  // nodes + runs are staged in shared memory when four blocks per SM still fit next to the per-warp tables
  const bool cut_capable = s->dev.n_cut > 0 && s->dev.n_runs > kTableRuns;
  L.smem = scene_bytes + (cut_capable ? (size_t)(kBlock / 32) * sizeof(WarpCut) + sizeof(GroupShared) : 0) <= kSmemSceneLimit;
  L.portals = s->info.has_portals != 0;
  const bool brute = p.traversal == RDC_TRAVERSAL_BRUTE_FORCE;
  // Run tables instead of the tree for primary rays: whole number of rays >= 8, LBVH mode.
  const bool masks_ok = (float)L.n_iter == p.number_of_rays_per_pixel && L.n_iter >= 8 && !brute && p.route != RDC_ROUTE_TREE;
  //  * the whole scene in one table: at most 64 runs;
  if (masks_ok && L.smem && s->dev.n_runs <= kTableRuns && p.route != RDC_ROUTE_LOCAL_TABLE) L.mode = kModeTable;
  //  * a table per tile over a CUT through the tree — at most 64 subtrees and leaves that together hold every run, nearest
  //    first, each walked only when the ray's stratum and the slab test let it: every larger scene that has a surface-area
  //    tree (accel.cu: up to 65 536 runs). Measured at 3840x2160 @256 against the tree and the local run table
  //    (profiles/r02h/sweep_modes.jsonl): lady_bug.xml 39.6 ms (tree 51.3, local 70.2), face.xml 47.9 (62.0, 68.7),
  //    dolphin.xml 94.7 (113.4, 108.1), roses_spirales.xml 64.3 (81.8, 68.3); zephyr.xml ties with the local table.
  else if (masks_ok && s->dev.n_cut > 0 && (p.route == RDC_ROUTE_AUTO || p.route == RDC_ROUTE_CUT_TABLE)) L.mode = kModeCut;
  //  * a table per tile of the runs around it (local run table): scenes beyond that (Morton tree, no cut — the synthetic
  //    100 k-curve scene), unless the view is zoomed out so far that a tile's
  //    own footprint already meets more runs than the table holds. First radius: the one at which a scene of
  //    uniform density would find 1.25 tables' worth of runs — (a + 2R + w)(b + 2R + h) n / A = 1.25 slots for a tile of a x b with
  //    mean run box w x h; the kernel adapts it per tile.
  //    Measured on the bundled scenes: below 1024 runs the tree is as fast or faster (RDC_ROUTE_LOCAL_TABLE overrides).
  else if (masks_ok && s->dev.n_runs >= (p.route == RDC_ROUTE_LOCAL_TABLE ? 1u : 1024u)) {
    const float4 rb = s->dev.root_box;
    const double area = (double)(rb.z - rb.x) * (double)(rb.w - rb.y);
    const double z = std::fabs((double)p.zoom_factor), jit = p.use_aa ? z : 0.0;
    const double pa = (kWarpTileW - 1) * z + 2 * jit + s->mean_run_w, pb = (kWarpTileH - 1) * z + 2 * jit + s->mean_run_h;
    const double per_run = area / s->dev.n_runs;  // scene area per run
    if (area > 0.0 && pa * pb < 0.5 * kLocalSlots * per_run) {
      const double disc = (pa + pb) * (pa + pb) - 4.0 * (pa * pb - 1.25 * kLocalSlots * per_run);
      const float r0 = (float)((std::sqrt(disc) - (pa + pb)) * 0.25);
      if (r0 > 0.0f && std::isfinite(r0)) {
        L.mode = kModeLocal;
        L.local_r0 = p.local_radius > 0.0f ? p.local_radius : r0;
      }
    }
  }
  const bool table = L.mode == kModeTable;
  const size_t warp_table[] = {0, sizeof(WarpOrder), sizeof(WarpLocal), sizeof(WarpCut)};  // per warp, by mode
  L.dyn = (L.smem ? scene_bytes + (table ? (size_t)s->dev.n_runs * sizeof(float4) : 0) : 0) + (size_t)(kBlock / 32) * warp_table[L.mode];
  L.variant = variant_index(L.mode, L.smem, L.portals || p.stats, p.stats);
  // Units per tile: how many work units a tile's rays are dealt to (unit q traces rays i = q mod split; the units' partial
  // sums are added in unit order). More units balance a launch better, fewer cost less: every unit pays for its run table
  // and its partial sums, and the rays of a unit lie `split` strata apart, which makes the previous ray's hit a worse
  // guess for the next (2.72 chords tested per ray at 4 units against 2.44 at 1 on the headline frame). Measured on the
  // headline frame and on a rank's share of it at 2, 4 and 8 GPUs (profiles/r02c/timeline.log): the fastest choice is the
  // one that leaves a warp about 13 units — 1 unit per tile for the whole 1080p frame (1.606 ms against 1.747 at 4), 2 for
  // half of it, 4 for a quarter or less. So: the smallest count that gives this LAUNCH at least 12 units per resident warp
  // when the whole scene sits in the run table; at least 48 on the tree and the local run table, whose units trace most of
  // their rays and last several times longer (lady_bug.xml 1080p on the tree: 7.70 ms at 4 units per tile, 9.47 ms at 1);
  // and 6.5 on the cut table, whose tiles each refine the cut first (lady_bug.xml 1080p: 5.10 ms at 1 unit per tile, 5.51 at 4;
  // a rank of 4: 1.43 ms at 2, 1.56 at 1; a rank of 8: 0.76 ms at 4, 0.83 at 8 — profiles/r02o/group.log). With more than one
  // unit per tile a table launch runs in group mode (below), so the units of a tile share its table.
  // The count is part of a pixel's summation order: launches that must agree bit for bit (a frame rendered whole and in
  // parts) pin rdc_frame_params::units_per_tile; hit indices never depend on it.
  const uint32_t tiles_x = (p.image_width + kWarpTileW - 1) / kWarpTileW;
  L.local_pixels = (size_t)L.local_rows * p.image_width;
  L.local_tiles = tiles_x * ((L.local_rows + L.row_skew + kWarpTileH - 1) / kWarpTileH);
  const uint64_t warps = (uint64_t)(s->sm_count > 0 ? s->sm_count : 148) * kMinBlocks * (kBlock / 32);
  uint32_t split = 1;
  // (in half units per warp) whole-scene table 12, cut table 6.5, tree and local table 48
  const uint64_t half_units_per_warp = table ? 24ull : L.mode == kModeCut ? 13ull : 96ull;
  while (split < (uint32_t)kAutoSplit && 2ull * L.local_tiles * split < half_units_per_warp * warps) split <<= 1;
  if (p.units_per_tile) split = p.units_per_tile;
  // (a local table is built per unit: it wants at least 64 rays per lane to pay for itself)
  while (split > 1 && ((uint32_t)L.n_iter < (L.mode == kModeLocal ? 64u : 16u) * split || (uint64_t)split * L.local_pixels * 20ull > (2ull << 30))) split >>= 1;
  L.split = split;
  // several units per tile on a table launch: that many warps of a block take them together (one table per tile, sums in shared memory)
  L.group = ((table || L.mode == kModeCut) && split > 1) ? split : 0u;
  if (L.group) L.dyn += sizeof(GroupShared);
  return L;
}

// The kernel of a plan's variant; on first use per handle: dynamic shared memory limit and the SM-filling grid size
// (which also forces the kernel's module to load — rdc_scene_reserve calls this so that no later launch has to).
int prepare_variant(rdc_scene* s, const LaunchPlan& L, RenderKernel* out) {
  const int variant = L.variant;
  const size_t dyn = L.dyn;
  const RenderKernel kernel = kKernels[variant];
  if (!kernel) {
    set_error("render: no kernel variant %d", variant);
    return RDC_E_INVALID;
  }
  if (s->grid_blocks[variant] == 0 || s->grid_dyn[variant] != dyn) {  // SM-filling grid: resident blocks per SM x SMs, per handle, variant and shared-memory size
    if (dyn > 48 * 1024) RDC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    int per_sm = 0, sms = 0;
    RDC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, dyn));
    RDC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    if (per_sm < 1 || sms < 1) {
      set_error("render: the kernel does not fit an SM");
      return RDC_E_LIMIT;
    }
    s->grid_blocks[variant] = (uint32_t)(per_sm * sms);
    s->grid_dyn[variant] = dyn;
  }
  *out = kernel;
  return 0;
}

// Scratch a launch of this plan needs; grows only. Allocating means a device-wide synchronisation (cudaFree), which
// is why rdc_scene_reserve exists.
int ensure_capacity(rdc_scene* s, const LaunchPlan& L, cudaStream_t stream) {
  if ((uint32_t)L.n_iter > s->base_dirs_capacity) {
    float2* fresh = nullptr;
    RDC_CUDA(cudaMalloc(&fresh, (size_t)L.n_iter * sizeof(float2)));
    s->allocations.push_back(fresh);  // the old table may still be read by a launch in flight: freed with the handle
    s->base_dirs = fresh;
    s->base_dirs_capacity = (uint32_t)L.n_iter;
    s->base_dirs_n = -1.0f;
  }
  if (L.split > 1 && !L.group && (L.local_pixels * L.split > s->part_capacity || L.local_tiles > s->tile_capacity)) {
    if (s->launched) RDC_CUDA(cudaEventSynchronize(s->launched));
    cudaFree(s->part_rgbw);
    cudaFree(s->part_blur);
    cudaFree(s->tile_arrivals);
    s->part_rgbw = nullptr; s->part_blur = nullptr; s->tile_arrivals = nullptr;
    s->part_capacity = 0; s->tile_capacity = 0;
    const size_t want = L.local_pixels * L.split;
    RDC_CUDA(cudaMalloc((void**)&s->part_rgbw, want * sizeof(float4)));
    RDC_CUDA(cudaMalloc((void**)&s->part_blur, want * sizeof(float)));
    RDC_CUDA(cudaMalloc((void**)&s->tile_arrivals, L.local_tiles * sizeof(unsigned int)));
    RDC_CUDA(cudaMemsetAsync(s->tile_arrivals, 0, L.local_tiles * sizeof(unsigned int), stream));
    s->part_capacity = want;
    s->tile_capacity = L.local_tiles;
  }
  return 0;
}

// ---- rdc_render_color_adjoint / rdc_render_blur_adjoint: the transpose of the frame in the colour or the blur stops ----
// For fixed frame parameters a pixel is sum_i w_i c_i / sum_i w_i with c_i = col[ind] (1 - rho) + col[ind+1] rho: ind, rho
// and w_i follow from the geometry and the u, weight and exponent lists only, so the image is linear in the colour values,
// and its transpose sends a pixel's gradient g to g w_i / W (1 - rho) at ind and g w_i / W rho at ind + 1 of the family
// the ray shades. The blur map is the same kind of map in the blur values (sigma = sum_i w_i b_i / sum_i w_i, one channel,
// one list). The rays are the render's: its tile grid, Philox draws, pixel culling and closest hit (the tree, which
// finds the first hits every route finds, or the brute force), and the terminal shading walks of trace_from.
// ---- rdc_render_weight_adjoint: the derivative of the image and the blur map in the weight and exponent stops ----
// w_i = m_i t_i^-e_i with m_i and e_i lerped from the weight and weight_degree lists; the frame is smooth in those values
// where W > 0. With s_i = <G, c_i> + g_sigma b_i and K = sum_i w_i s_i / W, dL/dw_i = (s_i - K) / W, and the chain through
// m_i and e_i sends (1 - rho_w) f_i (s_i - K) / W to weight[iw] (rho_w ... to iw + 1) and -(1 - rho_e) w_i ln t_i (s_i - K) / W
// to weight_degree[ie] (rho_e ... to ie + 1), f_i = t_i^-e_i.
struct AdjointArgs {
  RenderArgs r;                // the view (the output and work-unit fields stay unset)
  const float4* grad;          // colour, weight (or null): [local rows * width] dL/dRGB of each pixel of the band; .w ignored
  double* left;                // colour: [3 * colour_stops] Aᵀ grad in color_left ...
  double* right;               // ... and in color_right
  uint32_t tiles_x, n_tiles;
  int portals;                 // the scene has portal curves: a hit on one contributes nothing (max_trace_depth 0)
  const float* sigma_grad;     // blur, weight (or null): [local rows * width] dL/dsigma of each pixel of the band
  double* blur;                // blur: [blur_stops] A_bᵀ sigma_grad
  double* weight;              // weight: [weight_stops] dL/dweight
  double* degree;              // weight: [degree_stops] dL/dweight_degree
};

enum StopFamily : int { kColourStops, kBlurStops, kWeightStops };

constexpr uint32_t kNoStop = 0xFFFFFFFFu;

// Primary ray i of a pixel, its closest hit and the hit's walk data. False for a miss and for a hit on a portal curve
// (max_trace_depth 0: contributes nothing).
struct AdjointHit {
  Hit h;
  float dx, dy;
  HitWalks w;
};

__device__ __forceinline__ bool adjoint_hit(const AdjointArgs& aa, const Accel& ac, const Pixel& px, int i, bool small_angle,
                                            AdjointHit& r) {
  const RenderArgs& a = aa.r;
  const DevScene& sc = a.sc;
  Counters cnt;
  float ox, oy;
  gen_ray(a, px.pixel, px.base_x, px.base_y, i, small_angle, ox, oy, r.dx, r.dy);
  r.h = closest_chord<false, false, false>(ac, a.brute != 0, ox, oy, r.dx, r.dy, true, 1u, 0u, __int_as_float(0x7f800000), cnt);
  if (r.h.leaf < 0) return false;
  r.w = hit_walks(sc, r.h);
  return !(aa.portals && __ldg(sc.curve_connect + r.w.wd.z) >= 0);
}

// One primary ray of the adjoint, shaded with trace_from's terminal walks (hit_walks, stop_walk, terminal_colour); all
// zero for a miss or a portal hit. w = w_i; with KEY, the stop of FAMILY the ray interpolates from and the ratio rho
// (colour: key = ind << 1 | right; blur: key = ind). For the weights also s = <G, c_i> + g_sigma b_i (g.w = g_sigma) and,
// with KEY, the weight and exponent stops (iw, ie), their ratios, f = t^-e and t.
struct AdjointRay {
  float w = 0.0f;
  uint32_t key = kNoStop;
  float ratio = 0.0f;
  float f = 0.0f, t = 0.0f, rw = 0.0f, re = 0.0f;
  double s = 0.0;
  uint32_t iw = kNoStop, ie = kNoStop;
};

template <int FAMILY, bool KEY>
__device__ __forceinline__ AdjointRay adjoint_ray(const AdjointArgs& aa, const Accel& ac, const Pixel& px, int i, bool small_angle,
                                                  float4 g) {
  const DevScene& sc = aa.r.sc;
  AdjointRay out;
  AdjointHit r;
  if (!adjoint_hit(aa, ac, px, i, small_angle, r)) return out;
  const HitWalks& hw = r.w;
  const ScalarStop wm = stop_walk(sc.weight, hw.cw.w, hw.ws.w, hw.cu);
  const ScalarStop e = stop_walk(sc.weight_degree, hw.cw2.x, hw.wd.y, hw.cu);
  const float f = rdc_weight_falloff(r.h.t, e.value);
  out.w = wm.value * f;
  if constexpr (FAMILY == kWeightStops || (KEY && FAMILY == kColourStops)) {
    rdc_f2 v[4];
    load_control_points(sc, hw.seg, v);
    const bool right = rdc_is_ray_right(hw.u, r.dx, r.dy, v[0], v[1], v[2], v[3], aa.r.orzan != 0);
    float ratio, cr, cg, cb;
    const int ind = terminal_colour(sc, hw, right, ratio, cr, cg, cb);
    if constexpr (FAMILY == kColourStops) {
      out.key = ((uint32_t)ind << 1) | (right ? 1u : 0u);
      out.ratio = ratio;
    } else {
      const float blur = scalar_stop(sc.blur, hw.cw.z, hw.ws.y, hw.cu);
      // a zero gradient component adds nothing, whatever the stop value
      out.s = (g.x != 0.0f ? (double)g.x * cr : 0.0) + (g.y != 0.0f ? (double)g.y * cg : 0.0) +
              (g.z != 0.0f ? (double)g.z * cb : 0.0) + (g.w != 0.0f ? (double)g.w * blur : 0.0);
      if (KEY) {
        out.f = f, out.t = r.h.t, out.rw = wm.ratio, out.re = e.ratio;
        out.iw = (uint32_t)wm.ind, out.ie = (uint32_t)e.ind;
      }
    }
  }
  if constexpr (KEY && FAMILY == kBlurStops) {
    const ScalarStop b = stop_walk(sc.blur, hw.cw.z, hw.ws.y, hw.cu);
    out.key = (uint32_t)b.ind;
    out.ratio = b.ratio;
  }
  return out;
}

// Lanes whose rays end on the same stop `key` (usually most of the tile) add their terms up first (__match_any_sync, then
// a butterfly in fp64 per group, all lanes taking part), and the group's first lane issues one atomicAdd(double) per term
// at dst(key). terms(v, mine) writes a lane's terms into v, zeros unless `mine`. kNoStop: the lane adds nothing.
template <int kTerms, typename Terms, typename Dst>
__device__ __forceinline__ void scatter_groups(uint32_t lane, uint32_t key, Terms terms, Dst dst) {
  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, key);
  const bool leader = key != kNoStop && lane == (uint32_t)(__ffs(peers) - 1);
  uint32_t leaders = __ballot_sync(0xFFFFFFFFu, leader);
  while (leaders) {  // one group (one stop of one family) at a time
    const uint32_t l = (uint32_t)(__ffs(leaders) - 1);
    leaders &= leaders - 1;
    const uint32_t group = __shfl_sync(0xFFFFFFFFu, peers, l);
    const bool mine = (group >> lane) & 1u;
    double v[kTerms];
    terms(v, mine);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
      for (int c = 0; c < kTerms; ++c) v[c] += __shfl_xor_sync(0xFFFFFFFFu, v[c], off);
    if (lane == l) {
      double* d = dst(key);
#pragma unroll
      for (int c = 0; c < kTerms; ++c) atomicAdd(d + c, v[c]);
    }
  }
}

// One warp per 8x4 tile of the render's grid, one lane per pixel, all lanes on the same ray index. Pass 1 sums a pixel's
// weights W in the render's ray order (and, for the weights, sum_i w_i s_i and W in fp64); pass 2 traces the rays again and
// scatters through scatter_groups: six terms per group for the colours, two for the blur, two per family in two rounds for
// the weights.
template <int FAMILY>
__global__ void __launch_bounds__(kBlock) k_stop_adjoint(const AdjointArgs aa) {
  constexpr bool kColour = FAMILY == kColourStops;
  constexpr bool kWeight = FAMILY == kWeightStops;
  constexpr int kTerms = kColour ? 6 : 2;
  const RenderArgs& a = aa.r;
  const uint32_t lane = threadIdx.x & 31, tile = blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
  if (tile >= aa.n_tiles) return;  // (whole warps)
  Accel ac;
  ac.nodes = a.sc.nodes;
  ac.runs = reinterpret_cast<const float4*>(a.sc.runs);
  ac.run_box = a.sc.run_box;
  ac.n_runs = a.sc.n_runs;
  ac.slot_box = nullptr;
  ac.slot_node = nullptr;
  const bool small_angle = a.two_over_n <= 0.25f && a.two_over_n >= 0.0f;
  const int n = a.n_iter;
  const Pixel px = tile_pixel(a, tile, aa.tiles_x, lane);
  float4 g = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  if (px.valid) {
    if constexpr (kColour) {
      g = __ldg(aa.grad + px.local);
    } else if constexpr (kWeight) {  // g.w = dL/dsigma; a null gradient is zero
      if (aa.grad) g = __ldg(aa.grad + px.local);
      g.w = aa.sigma_grad ? __ldg(aa.sigma_grad + px.local) : 0.0f;
    } else {
      g.x = __ldg(aa.sigma_grad + px.local);
    }
  }
  // a pixel whose gradient is zero contributes nothing: its rays are not traced
  bool live = px.valid && (g.x != 0.0f || g.y != 0.0f || g.z != 0.0f || (kWeight && g.w != 0.0f));
  int cull_first = 0, cull_span = n - 1;
  const float jit = jitter(a);
  if (!pixel_cull(a, Rect{px.base_x - jit, px.base_x + jit, px.base_y - jit, px.base_y + jit}, cull_first, cull_span)) {
    cull_first = 0;
    cull_span = n - 1;
  }
  auto reaches = [&](int i) {  // ray i can reach the scene (tree_rays' intervals, visited in the same ascending order)
    int rel = i - cull_first;
    if (rel < 0) rel += n;
    return rel <= cull_span;
  };
  // pass 1: W = sum of the weights, in fp32 and in ray order like PixelSums::add
  float W = 0.0f;
  double W64 = 0.0, WS = 0.0;  // weights: W and sum_i w_i s_i in fp64
  if (live) {
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
      if (!reaches(i)) continue;
      const AdjointRay r = adjoint_ray<FAMILY, false>(aa, ac, px, i, small_angle, g);
      W += r.w;
      if constexpr (kWeight) {
        W64 += (double)r.w;
        WS += (double)r.w * r.s;
      }
    }
  }
  live = live && W != 0.0f;  // W == 0: the render writes NaN, the pixel is outside the image's linear map
  // weights: K and 1/W from the fp64 sums: sum_i w_i (s_i - K) then vanishes to fp64 rounding, so the weights' gradient
  // keeps the frame's invariance to scaling every weight
  const double inv_w = live ? (kWeight ? 1.0 / W64 : 1.0 / (double)W) : 0.0, K = WS * inv_w;
  // pass 2
#pragma unroll 1
  for (int i = 0; i < n; ++i) {
    const bool on = live && reaches(i);
    if (!__any_sync(0xFFFFFFFFu, on)) continue;
    AdjointRay r;
    if (on) r = adjoint_ray<FAMILY, true>(aa, ac, px, i, small_angle, g);
    if constexpr (kWeight) {
      const double q = r.iw == kNoStop ? 0.0 : (r.s - K) * inv_w;
      const double fw = (double)r.f * q, de = r.iw == kNoStop ? 0.0 : -(double)r.w * log((double)r.t) * q;
      scatter_groups<2>(
          lane, r.iw,
          [&](double* v, bool mine) { v[0] = mine ? fw * (double)(1.0f - r.rw) : 0.0, v[1] = mine ? fw * (double)r.rw : 0.0; },
          [&](uint32_t k) { return aa.weight + k; });
      scatter_groups<2>(
          lane, r.ie,
          [&](double* v, bool mine) { v[0] = mine ? de * (double)(1.0f - r.re) : 0.0, v[1] = mine ? de * (double)r.re : 0.0; },
          [&](uint32_t k) { return aa.degree + k; });
    } else {
      const double f = (double)r.w * inv_w, f1 = f * (double)r.ratio, f0 = f * (double)(1.0f - r.ratio);
      const double gx = g.x, gy = g.y, gz = g.z;
      auto terms = [&](double* v, bool mine) {
        if constexpr (kColour) {
          v[0] = mine ? gx * f0 : 0.0, v[1] = mine ? gy * f0 : 0.0, v[2] = mine ? gz * f0 : 0.0;
          v[3] = mine ? gx * f1 : 0.0, v[4] = mine ? gy * f1 : 0.0, v[5] = mine ? gz * f1 : 0.0;
        } else {
          v[0] = mine ? gx * f0 : 0.0, v[1] = mine ? gx * f1 : 0.0;
        }
      };
      scatter_groups<kTerms>(lane, r.key, terms, [&](uint32_t k) {
        return kColour ? ((k & 1u) ? aa.right : aa.left) + 3 * (size_t)(k >> 1) : aa.blur + k;
      });
    }
  }
}

// The fields of RenderArgs that describe the view, which the render and the adjoints share: the table of base directions
// for the launch's rays per pixel (made after ensure_capacity and the wait for the previous launch), the scene with the
// launch's widened boxes, the frame's size and band, the rays, the camera and the traversal.
int view_args(rdc_scene* s, const rdc_frame_params& p, int n_iter, cudaStream_t stream, RenderArgs& a) {
  if (s->base_dirs_n != p.number_of_rays_per_pixel) {
    k_base_dirs<<<1, 32, 0, stream>>>(s->base_dirs, n_iter, 2 / p.number_of_rays_per_pixel);
    RDC_CUDA(cudaGetLastError());
    s->base_dirs_n = p.number_of_rays_per_pixel;
  }
  if (int rc = widened_boxes(s, slab_widening(s, p), stream, &a.sc)) return rc;
  a.base_dirs = s->base_dirs;
  a.width = p.image_width;
  a.height = p.image_height;
  a.row_begin = p.row_begin;
  a.row_end = p.row_end;
  a.n_iter = n_iter;
  a.n_rays = p.number_of_rays_per_pixel;
  a.two_over_n = 2 / p.number_of_rays_per_pixel;
  a.zoom = p.zoom_factor;
  a.off_x = p.offset_x;
  a.off_y = p.offset_y;
  a.frame = p.frame;
  a.seed = p.seed;
  a.orzan = p.use_diffusion_curve_save;
  a.use_aa = p.use_aa;
  a.max_depth = p.max_trace_depth;
  a.brute = p.traversal == RDC_TRAVERSAL_BRUTE_FORCE;
  a.cull = p.traversal == RDC_TRAVERSAL_LBVH;  // the brute-force kernel really tests every ray against every chord
  return 0;
}

}  // namespace

int reserve(rdc_scene* s, const rdc_frame_params& p, cudaStream_t stream) {
  if (!s) {
    set_error("reserve: null argument");
    return RDC_E_INVALID;
  }
  if (int rc = check_params(p)) return rc;
  // the frame itself and every share of it a rank of 2..RDC_MAX_FRAME_TARGETS GPUs may be asked for (rdc_peer_*): a smaller
  // launch may deal its tiles to more units and so need partial sums the whole frame does not
  LaunchPlan L = plan_launch(s, p);
  if (L.local_rows == 0) return 0;
  for (uint32_t stride = 2; stride <= RDC_MAX_FRAME_TARGETS; ++stride) {
    rdc_frame_params q = p;
    q.strip_stride = stride;
    q.strip_offset = 0;
    const LaunchPlan S = plan_launch(s, q);
    if (S.split > 1 && S.local_pixels * S.split > (L.split > 1 ? L.local_pixels * L.split : 0)) {
      L.local_pixels = S.local_pixels;
      L.split = S.split;
    }
    if (S.local_tiles > L.local_tiles) L.local_tiles = S.local_tiles;
  }
  RenderKernel kernel = nullptr;
  if (int rc = prepare_variant(s, L, &kernel)) return rc;
  cudaFuncAttributes fa;
  RDC_CUDA(cudaFuncGetAttributes(&fa, k_base_dirs));
  return ensure_capacity(s, L, stream);
}

int launch_plan(const rdc_scene* s, const rdc_frame_params& p, rdc_launch_plan* out) {
  if (!s || !out) {
    set_error("launch plan: null argument");
    return RDC_E_INVALID;
  }
  if (int rc = check_params(p)) return rc;
  const LaunchPlan L = plan_launch(s, p);
  out->mode = L.mode;
  out->smem = L.smem ? 1 : 0;
  out->portals = (L.variant >> 1) & 1;
  out->stats = L.variant & 1;
  out->variant = L.variant;
  out->built = kKernels[L.variant] != nullptr ? 1 : 0;
  out->units_per_tile = L.split;
  out->group = L.group;
  out->dynamic_smem = L.dyn;
  return 0;
}

int render(rdc_scene* s, const rdc_frame_params& p, float4* image, float* blur_map, cudaStream_t stream, uint32_t n_targets,
           float* const* target_images, float* const* target_blur_maps) {
  if (!s || (n_targets == 0 && (!image || !blur_map))) {
    set_error("render: null argument");
    return RDC_E_INVALID;
  }
  if (n_targets > RDC_MAX_FRAME_TARGETS || (n_targets > 0 && (!target_images || !target_blur_maps))) {
    set_error("render: at most %d target frames", RDC_MAX_FRAME_TARGETS);
    return RDC_E_INVALID;
  }
  for (uint32_t t = 0; t < n_targets; ++t)
    if (!target_images[t] || !target_blur_maps[t]) {
      set_error("render: target frame %u is null", t);
      return RDC_E_INVALID;
    }
  if (int rc = check_params(p)) return rc;
  const LaunchPlan L = plan_launch(s, p);
  if (L.local_rows == 0) return 0;
  if (int rc = ensure_capacity(s, L, stream)) return rc;
  // One launch at a time per handle (shared work counters, partial sums, base directions)
  if (int rc = wait_previous_launch(s, stream)) return rc;

  RenderArgs a{};
  if (int rc = view_args(s, p, L.n_iter, stream, a)) return rc;
  a.image = image;
  a.blur_map = blur_map;
  a.n_targets = n_targets;
  for (uint32_t t = 0; t < n_targets; ++t) {
    a.target_image[t] = reinterpret_cast<float4*>(target_images[t]);
    a.target_blur[t] = target_blur_maps[t];
  }
  a.base_dirs = s->base_dirs;
  a.hit_ids = p.hit_ids;
  a.max_sigma = p.max_sigma;
  a.stats = p.stats;
  a.strip_stride = L.strip_stride;
  a.strip_offset = L.strip_offset;
  a.local_rows = L.local_rows;
  a.row_skew = L.row_skew;
  a.local_r0 = L.local_r0;
  a.work = s->work_counters;
  RenderKernel kernel = nullptr;
  if (int rc = prepare_variant(s, L, &kernel)) return rc;
  a.split = L.split;
  a.group = (int)L.group;
  {
    // the scene's centre in pixels of the full frame (inverse of DeviceCode.cu:103-107), then in tiles of this launch
    const float4 rb = s->dev.root_box;
    const double z = p.zoom_factor != 0.0f ? (double)p.zoom_factor : 1.0;
    const double px = (0.5 * ((double)rb.x + rb.z) - p.offset_x) / z + p.image_width / 2;
    const double sy = (0.5 * ((double)rb.y + rb.w) - p.offset_y) / z;
    const double py = p.use_diffusion_curve_save ? (double)p.image_height - (double)(p.image_height / 2) - sy : sy + p.image_height / 2;
    const uint32_t tiles_x = (p.image_width + kWarpTileW - 1) / kWarpTileW;
    const uint32_t tile_rows = (L.local_rows + L.row_skew + kWarpTileH - 1) / kWarpTileH;
    const double cx = std::fmin(std::fmax(px, 0.0), (double)p.image_width - 1.0);
    const double cy = std::fmin(std::fmax(py, (double)p.row_begin), (double)p.row_end - 1.0) - (double)(p.row_begin - L.row_skew);
    // strips: local row = (strip / stride) * 8 + row inside the strip, for the strips this launch renders
    const double local_y = L.strip_stride > 1 ? std::floor(cy / kStripRows / L.strip_stride) * kStripRows + std::fmod(cy, (double)kStripRows) : cy;
    a.mid_tx = std::min((uint32_t)(cx / kWarpTileW), tiles_x - 1);
    a.mid_ty = std::min((uint32_t)(std::fmax(local_y, 0.0) / kWarpTileH), tile_rows - 1);
  }
  a.part_rgbw = s->part_rgbw;
  a.part_blur = s->part_blur;
  a.tile_arrivals = s->tile_arrivals;
  const uint32_t grid = std::min(s->grid_blocks[L.variant], (L.local_tiles * L.split + kBlock / 32 - 1) / (kBlock / 32));
  // the work counters rewind themselves when a launch ends; a launch that was cut short must not poison the next
  RDC_CUDA(cudaMemsetAsync(s->work_counters, 0, 2 * sizeof(unsigned int), stream));
  kernel<<<grid, kBlock, L.dyn, stream>>>(a);
  RDC_CUDA(cudaGetLastError());
  return record_launch(s, stream);
}

namespace {

// The common part of color_adjoint, blur_adjoint and weight_adjoint: the checks, the wait for the handle's previous launch, the zeroing of
// the outputs and the launch of k_stop_adjoint<FAMILY>. `aa` carries the family's gradient and outputs; `what` names the call
// in messages, `stops` the family.
template <int FAMILY>
int stop_adjoint(rdc_scene* s, const rdc_frame_params& p, AdjointArgs aa, const char* what, const char* stops,
                 cudaStream_t stream) {
  if (int rc = check_params(p)) return rc;
  if (p.strip_stride > 1) {
    set_error("%s: strips (strip_stride %u) are not supported; use a contiguous row band", what, p.strip_stride);
    return RDC_E_INVALID;
  }
  if (s->info.has_portals && p.max_trace_depth > 0) {
    if (FAMILY == kWeightStops)
      set_error("%s: the scene has portals and max_trace_depth is %d; through a portal a ray's weight 1/(1/w_T + S) mixes "
                "the %s stops of several curves and its colour is a product (use max_trace_depth 0)", what, p.max_trace_depth,
                stops);
    else
      set_error("%s: the scene has portals and max_trace_depth is %d; through a portal the %s is a product of "
                "%s stops, not linear in them (use max_trace_depth 0)", what, p.max_trace_depth,
                FAMILY == kColourStops ? "image" : "blur map", stops);
    return RDC_E_INVALID;
  }
  LaunchPlan L;  // one unit per tile: only the table of base directions is needed
  L.n_iter = (int)ceilf(p.number_of_rays_per_pixel);
  if (int rc = ensure_capacity(s, L, stream)) return rc;
  if (int rc = wait_previous_launch(s, stream)) return rc;
  if (FAMILY == kColourStops) {
    const size_t bytes = 3 * (size_t)s->colour_stops * sizeof(double);
    RDC_CUDA(cudaMemsetAsync(aa.left, 0, bytes, stream));
    RDC_CUDA(cudaMemsetAsync(aa.right, 0, bytes, stream));
  } else if (FAMILY == kBlurStops) {
    RDC_CUDA(cudaMemsetAsync(aa.blur, 0, (size_t)s->blur_stops * sizeof(double), stream));
  } else {
    RDC_CUDA(cudaMemsetAsync(aa.weight, 0, (size_t)s->weight_stops * sizeof(double), stream));
    RDC_CUDA(cudaMemsetAsync(aa.degree, 0, (size_t)s->degree_stops * sizeof(double), stream));
  }
  RenderArgs& a = aa.r;
  if (int rc = view_args(s, p, L.n_iter, stream, a)) return rc;
  a.strip_stride = 1;
  a.strip_offset = 0;
  a.local_rows = p.row_end - p.row_begin;
  a.row_skew = p.row_begin % kWarpTileH;  // tiles on the full frame's grid, as in the render
  a.split = 1;
  aa.tiles_x = (p.image_width + kWarpTileW - 1) / kWarpTileW;
  aa.n_tiles = aa.tiles_x * ((a.local_rows + a.row_skew + kWarpTileH - 1) / kWarpTileH);
  aa.portals = s->info.has_portals;
  const uint32_t warps_per_block = kBlock / 32;
  k_stop_adjoint<FAMILY><<<(aa.n_tiles + warps_per_block - 1) / warps_per_block, kBlock, 0, stream>>>(aa);
  RDC_CUDA(cudaGetLastError());
  return record_launch(s, stream);
}

}  // namespace

int color_adjoint(rdc_scene* s, const rdc_frame_params& p, const float4* image_grad, double* grad_left, double* grad_right,
                  cudaStream_t stream) {
  if (!s || !image_grad || !grad_left || !grad_right) {
    set_error("color adjoint: null %s", !s ? "scene" : !image_grad ? "image_grad" : "output array");
    return RDC_E_INVALID;
  }
  AdjointArgs aa{};
  aa.grad = image_grad;
  aa.left = grad_left;
  aa.right = grad_right;
  return stop_adjoint<kColourStops>(s, p, aa, "color adjoint", "colour", stream);
}

int blur_adjoint(rdc_scene* s, const rdc_frame_params& p, const float* sigma_grad, double* grad_blur, cudaStream_t stream) {
  if (!s || !sigma_grad || !grad_blur) {
    set_error("render blur adjoint: null %s", !s ? "scene" : !sigma_grad ? "sigma_grad" : "output array");
    return RDC_E_INVALID;
  }
  AdjointArgs aa{};
  aa.sigma_grad = sigma_grad;
  aa.blur = grad_blur;
  return stop_adjoint<kBlurStops>(s, p, aa, "render blur adjoint", "blur", stream);
}

int weight_adjoint(rdc_scene* s, const rdc_frame_params& p, const float4* image_grad, const float* sigma_grad, double* grad_weight,
                   double* grad_degree, cudaStream_t stream) {
  if (!s || !grad_weight || !grad_degree || (!image_grad && !sigma_grad)) {
    set_error("render weight adjoint: null %s", !s ? "scene" : (!grad_weight || !grad_degree) ? "output array"
                                                                                                : "image_grad and sigma_grad");
    return RDC_E_INVALID;
  }
  AdjointArgs aa{};
  aa.grad = image_grad;
  aa.sigma_grad = sigma_grad;
  aa.weight = grad_weight;
  aa.degree = grad_degree;
  return stop_adjoint<kWeightStops>(s, p, aa, "render weight adjoint", "weight and exponent", stream);
}

}  // namespace rdc
