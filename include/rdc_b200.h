/* rdc_b200.h — C ABI of the B200-native diffusion-curve ray tracer.
 *
 * Drop-in boundary for ONE path of MikaZeilstra/RaytracingDiffusionCurves: "XML curve set + rays/pixel ->
 * float4 image" (ingest -> acceleration structure -> per-frame render -> variable-sigma blur). The
 * reference has no plugin/FFI interface; its seams are the ones cited below (paths relative to the
 * reference's optixHello/ directory). Plain pointers and sizes only; every entry point that can fail
 * returns int (0 = ok, >0 = cudaError_t, <0 = RDC_E_*), never throws, and records a message readable
 * through rdc_last_error_string(). Entry points that take a stream only enqueue work on it (no hidden
 * synchronisation) unless their comment says otherwise. Nothing in the library reads the environment: every
 * switch is a field of one of the structs below.
 *
 * Threading (optixHello.cpp runs one host thread and one stream): a handle (rdc_scene, rdc_group) may be used from
 * one host thread at a time. Device work of one rdc_scene is serialised by the library — a launch on the handle
 * first waits (stream-ordered, no host wait) for the handle's previous launch, whatever stream that was given —
 * because every launch shares the handle's work counters and scratch. Use one handle per device and per
 * concurrently rendered frame.
 */
#ifndef RDC_B200_H
#define RDC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RDC_E_INVALID (-1)  /* bad argument                        */
#define RDC_E_PARSE (-2)    /* malformed XML / unexpected schema   */
#define RDC_E_IO (-3)       /* file could not be read / written    */
#define RDC_E_LIMIT (-4)    /* a structural limit was exceeded     */

typedef void* rdc_stream; /* CUstream / cudaStream_t, as in Params::stream (params.h:45) */

/* ---- ingest: replaces the XML loop of optixHello.cpp:108-117,212-515 and its helpers :1302-1386 ---- */

typedef struct rdc_ingest_options {
  int use_diffusion_curve_save; /* USE_DIFFUSION_CURVE_SAVE (params.h:24): Orzan-2008 orientation */
  float default_weight_degree;  /* optixHello.cpp:94  (0.5)  */
  float endcap_size;            /* optixHello.cpp:96  (8)    */
} rdc_ingest_options;

/* Read-only view of the structure-of-arrays scene, same arrays (and names) as struct Params
 * (params.h:60-92). Index arrays hold uint2 {start,count} pairs as two consecutive uint32; vertices and
 * colours are float3 triples. Every *_u array carries two trailing +INF sentinels beyond n_* so the
 * reference's over-reading stop walk (DeviceCode.cu:39-43) stays in bounds. */
typedef struct rdc_scene_arrays {
  int image_width, image_height; /* curve_set@image_width/@image_height (optixHello.cpp:116-117) */
  uint32_t n_vertices, n_segments, n_curves;
  const float* vertices;             /* float3[n_vertices], uniform cubic B-spline control points */
  const uint32_t* segment_indices;   /* [n_segments] first vertex of each spline segment          */
  const uint32_t* curve_map;         /* [n_segments] segment -> curve                             */
  const uint32_t* curve_index;       /* [n_segments] ordinal of the segment inside its curve      */
  const int32_t* curve_connect;      /* [n_curves]   portal target curve or -1                    */
  const uint32_t* curve_map_inverse; /* [n_curves]   first segment of each curve                  */
  uint32_t n_color_left, n_color_right, n_blur, n_weight, n_weight_degree;
  const uint32_t* color_left_index;  const float* color_left;  const float* color_left_u;
  const uint32_t* color_right_index; const float* color_right; const float* color_right_u;
  const uint32_t* blur_index;        const float* blur;        const float* blur_u;
  const uint32_t* weight_index;      const float* weight;      const float* weight_u;
  const uint32_t* weight_degree_index; const float* weight_degree; const float* weight_degree_u;
} rdc_scene_arrays;

typedef struct rdc_host_scene rdc_host_scene; /* opaque, host memory */

void rdc_default_ingest_options(rdc_ingest_options* opts);
int rdc_ingest_xml_file(const char* path, const rdc_ingest_options* opts, rdc_host_scene** out);
int rdc_ingest_xml_memory(const char* text, size_t len, const rdc_ingest_options* opts, rdc_host_scene** out);
int rdc_host_scene_arrays(const rdc_host_scene* scene, rdc_scene_arrays* out);
void rdc_host_scene_destroy(rdc_host_scene* scene);
/* Binary cache of an ingested scene (skips XML parsing on the next run; same arrays bit for bit). */
int rdc_host_scene_save(const rdc_host_scene* scene, const char* path);
int rdc_host_scene_load(const char* path, rdc_host_scene** out);
/* canonical text dump of the element tree the loader sees (parser tests) ; caller frees with rdc_free */
int rdc_xml_dump_file(const char* path, char** out_text);
void rdc_free(void* p);

/* ---- acceleration structure: replaces optixAccelComputeMemoryUsage/optixAccelBuild over
 *      OPTIX_PRIMITIVE_TYPE_ROUND_CUBIC_BSPLINE (optixHello.cpp:765-830) and the per-array
 *      cudaMallocAsync+cudaMemcpyAsync uploads (:524-762) ---- */

#define RDC_TREE_AUTO 0   /* surface-area heuristic up to 65 536 runs, Morton radix tree above                 */
#define RDC_TREE_MORTON 1 /* Morton-code radix tree (Karras 2012), built on the GPU                           */
#define RDC_TREE_SAH 2    /* binned surface-area heuristic, built on the host                                 */
typedef struct rdc_accel_options {
  float curve_width;         /* optixHello.cpp:95 (1e-3): pads chord boxes                          */
  float flatness_tolerance;  /* max |curve - chord| in XML pixels; chords per segment follow from it */
  int max_chords_per_segment;
  int run_length;            /* chords per tree leaf, 1..8; 0 = choose from the scene's density        */
  int shading_records;       /* per-chord 128-byte shading records: 0 = library default (built when the
                                table fits 32 MB), -1 = never (shading walks the stop lists)            */
  int tree;                  /* RDC_TREE_*: how the tree over the leaf runs is built; same results either way */
} rdc_accel_options;

typedef struct rdc_scene rdc_scene; /* opaque: device-resident SoA scene + chords + LBVH, one per device */

typedef struct rdc_scene_info {
  uint32_t n_segments, n_curves, n_chords, n_runs, n_nodes, bvh_depth; /* runs = tree leaves (<= 8 chords each) */
  int has_portals;
  uint64_t device_bytes;    /* everything the handle owns on the device            */
  uint64_t traversal_bytes; /* nodes + leaf runs: what a ray touches                */
  float pad;                /* box padding actually used                           */
} rdc_scene_info;

void rdc_default_accel_options(rdc_accel_options* opts);
/* Uploads the arrays and builds chords, leaf runs and the tree over them (rdc_accel_options::tree) on `stream`.
 * Synchronises the stream before returning (the build reads back counts; the surface-area tree is built on the
 * host), like the reference's set-up phase. */
int rdc_accel_build(const rdc_scene_arrays* arrays, const rdc_accel_options* opts, rdc_stream stream, rdc_scene** out);
int rdc_scene_get_info(const rdc_scene* scene, rdc_scene_info* out);
/* Test hook: copies the chord list (original order) to host arrays of n_chords entries each.
 * geom = 4 floats per chord (ax,ay,bx,by); ids = 3 uint32 per chord (segment, k, K). Synchronous. */
int rdc_scene_download_chords(const rdc_scene* scene, float* geom, uint32_t* ids);
/* Test hook: copies the tables shading derives from the stop lists to host memory: seg_walk = n_segments x 64 bytes (per
 * segment, where each stop walk starts and ends), chord_walk = n_chords x 32 bytes (per chord, where each walk stands at the
 * chord's smallest parameter), chord_records = n_chords x 128 bytes of shading records when the handle has them (else pass
 * NULL). Waits for the handle's last launch or update. Synchronous. */
int rdc_scene_download_stop_tables(const rdc_scene* scene, void* seg_walk, void* chord_walk, void* chord_records);
/* Recolours a built scene: replaces the handle's five stop families (the n_* counts, *_index, values and *_u of `arrays`,
 * with the sentinels and padding of rdc_scene_arrays) and the three tables shading derives from them. Chords, runs, tree,
 * cut and boxes are kept, so an edit of colours, blur, weight or weight degree costs a copy and one small kernel instead of
 * a rebuild; edits of control points or curves need rdc_accel_build.
 *   Equivalence: afterwards every launch on the handle (rdc_render, rdc_render_to_frames, the frame-to-host and peer calls,
 *     every route) gives the same image, blur map, hit ids and counters, bit for bit, as the same launch on a handle that
 *     rdc_accel_build built from `arrays` with the same options.
 *   Geometry: the geometry fields of `arrays` must be those the handle was built from. n_vertices, n_segments and n_curves
 *     are checked; no other geometry array is read.
 *   Validation: the stop lists get the checks of rdc_accel_build (no null array; each curve's {start,count} inside its
 *     list). A rejection returns RDC_E_INVALID with a message and leaves the handle unchanged.
 *   Stream order: like a launch, the call's device work waits (stream-ordered, no host wait) for the handle's previous
 *     launch or update, whatever stream that was on, and the handle's next launch waits for it.
 *   Memory: the handle keeps room for the largest stop lists it has held. An update that fits overwrites them in place
 *     and only enqueues. The handle's first update also allocates its pinned staging buffer, and an update that needs
 *     more room waits for the handle's last launch and reallocates: those synchronise once. rdc_scene_info::device_bytes
 *     follows.
 *   The caller's arrays: the call packs them into the handle's pinned staging buffer before it returns, so the caller may
 *     free or change them at once. The buffer is reused: an update first waits on the host until the previous update's
 *     copy out of it has run, and that copy runs once the launch enqueued before the previous update has finished. */
int rdc_scene_update_stops(rdc_scene* scene, const rdc_scene_arrays* arrays, rdc_stream stream);
void rdc_scene_destroy(rdc_scene* scene);

/* ---- per-frame render: replaces optixLaunch(pipeline, stream, d_param, sizeof(Params), &sbt, W, H, 1)
 *      (optixHello.cpp:1184) running DeviceCode.cu:85-342 ---- */

#define RDC_STRIP_ROWS 8
#define RDC_TRAVERSAL_LBVH 0
#define RDC_TRAVERSAL_BRUTE_FORCE 1 /* every ray against every chord; validates the LBVH at full size */
/* how primary rays find their closest chord (rdc_frame_params::route). Every route finds the same first hits. With
 * units_per_tile pinned, the tree, the whole-scene table and the cut table give the same pixel bits; the local run table
 * adds the samples of the rays it defers to the tree after the others, so its pixels may differ in the last bits. */
#define RDC_ROUTE_AUTO 0        /* whole-scene run table up to 64 runs; per-tile cut table for every larger scene that
                                   has a surface-area tree (up to 65 536 runs); per-tile local run table beyond,
                                   when the view is close enough; the tree otherwise                           */
#define RDC_ROUTE_TREE 1        /* always the tree                                                            */
#define RDC_ROUTE_LOCAL_TABLE 2 /* per-tile local run table whatever the size of the scene                     */
#define RDC_ROUTE_CUT_TABLE 3   /* per-tile table over a cut through the tree, refined around every tile (scenes of
                                   more than 64 runs that have a surface-area tree)                            */

typedef struct rdc_frame_params {
  uint32_t image_width, image_height;   /* output size (params.h:48-49)                               */
  float number_of_rays_per_pixel;       /* a float, as in params.h:55                                 */
  float zoom_factor, offset_x, offset_y; /* params.h:95-97                                            */
  uint32_t frame;                       /* params.h:100; part of the Philox key                       */
  uint32_t seed;                        /* Philox key word 0                                          */
  uint32_t row_begin, row_end;          /* rows [row_begin,row_end) of the full image to render; the
                                           image/blur_map pointers address row_begin (band-local)     */
  uint32_t strip_stride, strip_offset;  /* stride > 1: the band is dealt out in strips of RDC_STRIP_ROWS
                                           rows and this call renders strips t with t % stride == offset,
                                           packed one after the other in the output buffers (load-balanced
                                           multi-GPU split). stride 0 or 1: the whole band.              */
  int use_diffusion_curve_save;         /* params.h:24                                                */
  int use_aa;                           /* params.h:28                                                */
  int max_trace_depth;                  /* params.h:32, 0..31                                         */
  int traversal;                        /* RDC_TRAVERSAL_*                                            */
  uint32_t* hit_ids;                    /* optional device array [rows*W*rpp]: chord id of each primary
                                           ray's first hit, 0xFFFFFFFF for a miss (parity tests)       */
  float* max_sigma;                     /* optional device float: atomically raised to the largest
                                           blur_map value written (lets the blur skip all-zero maps)   */
  unsigned long long* stats;            /* optional device uint64[9]; [0..5] atomically increased by: rays traced
                                           (continuations included), boxes tested (tree nodes and table
                                           slots), chords tested, hits shaded, primary rays the local run
                                           table deferred to the tree, nodes visited by the table queries;
                                           [6..8] the launch's timeline in ns of %globaltimer: start (set [6]
                                           and [7] to ~0 beforehand: they take minima), first warp out of
                                           work, last warp out. Selects a slower counting build of the
                                           kernel; feeds the roofline's work-per-ray figure (SURVEY.md 8d) */
  int route;                            /* RDC_ROUTE_*; 0 = automatic                                    */
  uint32_t units_per_tile;              /* work units a tile's rays are dealt to: 0 = automatic (chosen per
                                           launch from its size), else 1, 2, 4 or 8. Part of a pixel's
                                           summation order: launches that must agree BIT FOR BIT (a frame
                                           rendered whole and in bands, on 1 and on N GPUs) pin it to one
                                           value; hit indices never depend on it and RGB moves by ~1e-7   */
  float local_radius;                   /* first radius (scene units) the local run table tries around a tile;
                                           0 = from the scene's density                                   */
} rdc_frame_params;

void rdc_default_frame_params(rdc_frame_params* p, uint32_t width, uint32_t height, float rays_per_pixel);
/* Grows the handle's scratch (partial sums of split work units, tile counters, the table of base directions, the
 * frame buffers of rdc_render_frame_to_host when `host_frames` != 0) to what a frame of `params` needs. May allocate
 * and synchronise the device. After it, rdc_render / rdc_render_to_frames / rdc_render_frame_to_host_async with
 * parameters of at most this size and the same rays per pixel only enqueue; without it the first call at a new
 * size does this work itself (and so synchronises once). */
int rdc_scene_reserve(rdc_scene* scene, const rdc_frame_params* params, int host_frames, rdc_stream stream);
/* Test hook: which render kernel rdc_render would launch for `params` on this handle, and how. Validates the parameters
 * like rdc_render; no device work. */
typedef struct rdc_launch_plan {
  int mode;                /* 0 tree, 1 whole-scene run table, 2 local run table, 3 cut table              */
  int smem;                /* nodes + runs staged in shared memory                                         */
  int portals;             /* portal-capable kernel (the counting build always is)                         */
  int stats;               /* counting build (rdc_frame_params::stats set)                                 */
  int variant;             /* index into the library's kernel table                                        */
  int built;               /* a kernel exists for that index                                               */
  uint32_t units_per_tile; /* work units per tile actually used, after the reductions for few rays per pixel */
  uint32_t group;          /* warps that take a tile's units together, 0 = units combine in global memory  */
  uint64_t dynamic_smem;   /* bytes of dynamic shared memory per block                                     */
} rdc_launch_plan;
int rdc_scene_launch_plan(const rdc_scene* scene, const rdc_frame_params* params, rdc_launch_plan* out);
/* image = float4[rows*W] (xyz written, w = 1), blur_map = float[rows*W]; both device pointers. */
int rdc_render(rdc_scene* scene, const rdc_frame_params* params, float* image, float* blur_map, rdc_stream stream);

/* Multi-GPU form (SURVEY.md 8e: row bands / strips per GPU, gather to rank 0): renders the rows the parameters
 * select like rdc_render, but stores every finished pixel at its place in the FULL frame — image
 * float4[image_height*image_width], blur_map float[image_height*image_width] — of each of n_targets target frames.
 * The pointers may address peer GPUs' memory (NVLink peer access, CUDA IPC, symmetric memory): the render kernel's
 * stores ARE the gather. hit_ids / stats / max_sigma work as in rdc_render. Enqueue-only; the caller orders the
 * consumers of the target frames after this call on every rank (a barrier over the ranks' streams). */
#define RDC_MAX_FRAME_TARGETS 8
int rdc_render_to_frames(rdc_scene* scene, const rdc_frame_params* params, uint32_t n_targets, float* const* images,
                         float* const* blur_maps, rdc_stream stream);

/* ---- colour stops from an image: the transpose of rdc_render in the colour stops ----
 *
 * For fixed frame parameters the image rdc_render writes is linear in the colour values: a pixel is
 * sum_i w_i c_i / sum_i w_i over its rays, with c_i = col[ind] (1 - rho) + col[ind + 1] rho, and ind, rho and the weights
 * w_i follow from the geometry and the *_u, weight and weight_degree lists alone. So image = A x, with x the color_left and
 * color_right values, and fitting colours to a target picture is linear least squares (INTEGRATION.md §4).
 *   Transpose: grad_color_left and grad_color_right receive A^T image_grad, where A is the map from the colour values to the
 *     image rdc_render writes for `params`, over the rows of `params`' band: sum over pixels of <image_grad, A x> equals
 *     <x, grad> up to the fp32 rounding of the render. The rays are the render's (tile grid, Philox draws, culling, closest
 *     hits, terminal shading walks). Pixels the render leaves NaN (no ray hit, or all weights zero) contribute nothing.
 *   Layout: image_grad is a device float4[rows * W], band-local like rdc_render's image, dL/dRGB per pixel (.w ignored).
 *     The outputs are device double arrays laid out like rdc_scene_arrays::color_left / color_right of the handle's current
 *     stops: 3 * (max(n_color_left, n_color_right) + 2) entries each, padding and sentinels included.
 *   Overwrite: the call zeroes both arrays first, on the stream, then accumulates with atomicAdd(double): the result is
 *     not bit-reproducible from call to call (the order of the additions varies), only to fp64 rounding.
 *   Parameters read: the fields rdc_render uses for its rays, traversal included; route, units_per_tile, local_radius,
 *     hit_ids, stats and max_sigma are ignored. strip_stride > 1 is rejected.
 *   Portals: a scene with portal curves is rejected unless max_trace_depth == 0 (through a portal the image is a product of
 *     colour stops, so not linear in them); at depth 0 a hit on a portal curve contributes nothing, as in the render.
 *   Blur: the transpose is of the unblurred image; the blur map and gaussianBlur are outside it.
 *   Non-finite gradients: a non-finite image_grad on a pixel the render does not leave NaN propagates into the outputs;
 *     the caller zeroes such entries. A pixel whose gradient is zero traces no rays.
 *   Stream order and memory: like rdc_render. The call waits (stream-ordered, no host wait) for the handle's previous
 *     launch or update, whatever stream that was on, and the handle's next launch waits for it, so an adjoint enqueued after
 *     rdc_scene_update_stops sees the new u lists on any stream. It allocates nothing after rdc_scene_reserve for the same
 *     rays per pixel; without it the first call at a new rays-per-pixel count may synchronise once.
 *   Validation: RDC_E_INVALID with a message for a null scene, params, image_grad or output array, for what rdc_render
 *     rejects in the parameters, for strips, and for the portal case above. */
int rdc_render_color_adjoint(rdc_scene* scene, const rdc_frame_params* params, const float* image_grad,
                             double* grad_color_left, double* grad_color_right, rdc_stream stream);

/* ---- picking: the curve under a point (an editor's click, or every pixel of a view for hover and selection) ----
 *
 * Nearest: the pick of a point p is the chord with the smallest (d2, chord id) among all chords with d2 <= max_distance^2
 *   (fp32 product), where d2 = |p - c|^2 and c is the point of the chord nearest to p, both computed in fp32 exactly as
 *   rdc_point_chord (csrc/rdc_math.h) computes them. max_distance = +INF takes the nearest chord whatever its distance.
 *   The fields are those of that chord; the tree is only a faster way to the brute force's answer, so both tree builders
 *   and every run length give the same bits.
 * Miss: nothing within range, or a point with a NaN or infinite coordinate: chord, segment and curve RDC_PICK_NONE,
 *   flags 0, distance +INF, u, x and y NaN, and the three stop vectors NaN.
 * Side: RDC_PICK_RIGHT is set when rdc_is_ray_right(local u, D = c - p, control points, use_diffusion_curve_save) holds,
 *   i.e. a ray from p toward c would shade the colour_right list. At distance 0 (D = 0) the normal's dot product is 0, so
 *   the pick is on the right side when use_diffusion_curve_save is 0 and on the left side when it is 1.
 * Stops: at the pick's u, with the walks terminal shading uses (the walk starts of seg_walk and chord_walk, or the chord's
 *   shading record when it replaces the walks; rdc_interp_from, rdc_lerp_stop, rdc_lerp_color). On a portal curve they are
 *   the curve's own left and right lists, not the portal filter (which walks the right list's range on the left arrays,
 *   DeviceCode.cu:297).
 * Stream order: like a launch, the pick waits (stream-ordered, no host wait) for the handle's previous launch or update,
 *   whatever stream that was on, and the handle's next launch waits for the pick. A pick enqueued after
 *   rdc_scene_update_stops sees the new stops on any stream.
 * No scratch: a pick allocates nothing and never synchronises; it only enqueues, from the first call on.
 * Validation: RDC_E_INVALID with a message for a null scene or out, null points with n > 0, max_distance NaN or <= 0,
 *   and (frame form) null params, zero width, an empty or out-of-range row band, or strip_stride > 1. n == 0 enqueues
 *   nothing. */
#define RDC_PICK_NONE 0xFFFFFFFFu
#define RDC_PICK_RIGHT 1u  /* the point lies on the side shaded with color_right (rdc_is_ray_right with D = c - p) */
#define RDC_PICK_PORTAL 2u /* the curve is a portal (curve_connect >= 0)                                       */
typedef struct rdc_pick {
  uint32_t chord;   /* id of the nearest chord (rdc_scene_download_chords order); RDC_PICK_NONE: nothing within range */
  uint32_t segment; /* its spline segment                                                                          */
  uint32_t curve;   /* its curve                                                                                   */
  uint32_t flags;   /* RDC_PICK_RIGHT | RDC_PICK_PORTAL                                                            */
  float u;          /* curve parameter as the *_u stop lists use it: ordinal + (k + s) / K, the float ops of shading */
  float distance;   /* sqrtf(d2), scene units                                                                      */
  float x, y;       /* c, the nearest point on the chord                                                           */
} rdc_pick;         /* 32 bytes */

/* points: device float2[n], scene (XML pixel) coordinates. out: device rdc_pick[n]. stops: NULL or device float4[3n]
 * (16-byte aligned): {left r, g, b, blur}, {right r, g, b, weight}, {weight_degree, 0, 0, 0} at the pick's u. */
int rdc_scene_pick(rdc_scene* scene, const float* points, uint32_t n, float max_distance, int use_diffusion_curve_save,
                   rdc_pick* out, float* stops, rdc_stream stream);
/* One pick per pixel centre (rdc_view_pixel_to_scene) of rows [row_begin,row_end) of the view `params` describes: out
 * and stops are band-local like rdc_render's image (row row_begin first). Reads image_width, image_height, zoom_factor,
 * offset_x, offset_y, use_diffusion_curve_save and the row band; ignores the ray fields. strip_stride > 1 is rejected. */
int rdc_scene_pick_frame(rdc_scene* scene, const rdc_frame_params* params, float max_distance, rdc_pick* out, float* stops,
                         rdc_stream stream);
/* Host: the scene point rdc_scene_pick_frame picks for pixel (ix, iy) of the full frame — the render's ray origin before
 * the anti-aliasing jitter plus half a pixel, the centre of the square the pixel's rays start from. For a cursor click. */
int rdc_view_pixel_to_scene(const rdc_frame_params* params, uint32_t ix, uint32_t iy, float* x, float* y);

/* ---- one frame over the GPUs of a box (SURVEY.md 8e), all in C: frames the ranks share, a barrier in peer memory,
 *      and the per-frame drivers. A "rank" is one GPU with its own rdc_scene (scene and tree are replicated); ranks may
 *      live in one process (one host thread enqueueing on every device: rdc_peer_frames_connect_local) or in one process
 *      each (rdc_peer_frames_export / _connect_ipc: CUDA IPC handles, carried by whatever the launcher offers). The
 *      frame loop these replace is optixHello.cpp:1163-1259. world <= RDC_MAX_FRAME_TARGETS. ---- */
typedef struct rdc_peer_frames rdc_peer_frames;
#define RDC_PEER_HANDLE_BYTES 320 /* five 64-byte cudaIpcMemHandle_t per rank */
/* allocates this rank's buffers on the current device (rendered frame + sigma, two finished frames, flags) */
int rdc_peer_frames_create(uint32_t width, uint32_t height, int rank, int world, rdc_peer_frames** out);
int rdc_peer_frames_export(const rdc_peer_frames* frames, void* handle_bytes /* RDC_PEER_HANDLE_BYTES */);
/* all_handles: world * RDC_PEER_HANDLE_BYTES, rank-major (the rank's own entry is ignored) */
int rdc_peer_frames_connect_ipc(rdc_peer_frames* frames, const void* all_handles);
/* same process: all[r] was created as rank r on its own device; enables peer access both ways */
int rdc_peer_frames_connect_local(rdc_peer_frames* const* all, int world);
void rdc_peer_frames_destroy(rdc_peer_frames* frames);
/* All ranks' streams meet: work enqueued before it on any rank is complete and visible to every rank's work after it.
 * Enqueue-only (one tiny kernel: flags in peer memory, release/acquire at system scope); every rank must call it the
 * same number of times. A rank that never arrives raises an error flag after ~4 s instead of wedging the GPU
 * (rdc_peer_status, synchronous, reports it). */
int rdc_peer_barrier(rdc_peer_frames* frames, rdc_stream stream);
int rdc_peer_status(rdc_peer_frames* frames);
/* Device consumer: every rank renders its strips and stores them straight into the consumers' frames over NVLink; the
 * finished frame (blurred when use_blur and halo_rows > 0; halo_rows >= ceil(3 * largest sigma)) ends in one of rank 0's
 * two frame buffers, used in turn: *frame_out (rank 0; NULL elsewhere). `wait_event` (cudaEvent_t or NULL) is waited for
 * on `stream` right before the frame's first barrier: rank 0 passes "the consumer of the frame returned two calls ago is
 * done", because the peers start writing that buffer after this barrier. Enqueue-only. */
int rdc_peer_render_frame(rdc_scene* scene, rdc_peer_frames* frames, const rdc_frame_params* params, int use_blur,
                          int halo_rows, void* wait_event, rdc_stream stream, float** frame_out);
/* Host consumer: nothing is gathered on a GPU — every rank copies its own rows of the finished frame over its own PCIe
 * link into `host_frame`, ONE full frame float4[H*W] in pinned host memory that every rank addresses (rdc_host_frame_open
 * when the ranks are processes). Enqueue-only; the copy runs on the handle's copy stream and overlaps the next frame's
 * rendering. rdc_peer_frames_wait blocks until this rank's copies have landed. Use two host frames in turn. */
int rdc_peer_frame_to_host(rdc_scene* scene, rdc_peer_frames* frames, const rdc_frame_params* params, int use_blur,
                           int halo_rows, float* host_frame, rdc_stream stream);
int rdc_peer_frames_wait(rdc_peer_frames* frames);
/* A host frame all ranks can address: POSIX shared memory `name` (create != 0 on one rank, then 0 on the others),
 * mapped and registered with CUDA as pinned memory. */
int rdc_host_frame_open(const char* name, size_t bytes, int create, float** out);
int rdc_host_frame_close(const char* name, float* frame, size_t bytes, int unlink_it);
/* ceil(3 * largest blur value a frame of this scene can hold) — the blur's reach in rows (helperKernels.cu:65,74);
 * each portal passed multiplies sigma by another stop (DeviceCode.cu:311). 0: the scene has no blur. */
int rdc_host_scene_halo_rows(const rdc_host_scene* scene, int max_trace_depth, int* halo_rows);

/* ---- helper kernels: same names and signatures as helperKernels.cu's extern "C" launchers
 *      (declared at optixHello.cpp:51-54) ---- */
#ifndef RDC_NO_REFERENCE_HELPER_NAMES
/* helperKernels.cu:137-148. In-place capable (dest == source). Scratch comes from the stream-ordered
 * allocator instead of a per-frame cudaMalloc/cudaFree. `image` elements are float4. */
void gaussianBlur(void* dest, void* source, float* sigma, int width, int height, rdc_stream stream);
/* helperKernels.cu:43-45 */
void setFloatDevice(float* dest, unsigned int n, float src, rdc_stream stream);
/* helperKernels.cu:158-160. The Philox generator is counter-based and keeps no per-pixel state, so this
 * only validates its arguments; `states` may be NULL. */
void setupCurand(void* states, int width, int height, rdc_stream stream);
#endif
/* Blur with caller-provided scratch (float4[rows_with_halo*W]) on a band of rows, int result. `source`,
 * `sigma`, `dest` address row 0 of a buffer holding `height` rows; rows [row_begin,row_end) are produced.
 * max_sigma (optional device float written by rdc_render) lets both passes degrade to a copy when 0. */
int rdc_gaussian_blur(void* dest, const void* source, const float* sigma, void* scratch, int width, int height,
                      int row_begin, int row_end, const float* max_sigma, rdc_stream stream);
/* Same, but the horizontal pass only covers the rows the band's vertical pass can reach:
 * [row_begin - halo_rows, row_end + halo_rows) clipped to the buffer (halo_rows >= ceil(3 * largest sigma)). */
int rdc_gaussian_blur_band(void* dest, const void* source, const float* sigma, void* scratch, int width, int height,
                           int row_begin, int row_end, int halo_rows, const float* max_sigma, rdc_stream stream);

/* ---- whole frame through host memory: the body of the reference's frame loop (optixHello.cpp:1176-1244)
 *      minus window system: render -> [blur] -> copy to host -> synchronise ---- */
int rdc_render_frame_to_host(rdc_scene* scene, const rdc_frame_params* params, int use_blur, float* host_image,
                             rdc_stream stream);
/* Pipelined form: only enqueues (render and blur on `stream`, the copy to `host_image` — pinned memory — on the
 * handle's own copy stream, two device images used in turn), so the copy of one frame overlaps the rendering of the
 * next. rdc_frame_wait blocks until every enqueued frame is in host memory. Give consecutive frames different
 * host buffers. rdc_render_frame_to_host = async + wait. */
int rdc_render_frame_to_host_async(rdc_scene* scene, const rdc_frame_params* params, int use_blur, float* host_image,
                                   rdc_stream stream);
int rdc_frame_wait(rdc_scene* scene);

/* ---- output conventions of the F11 screenshot (glfw_events.cpp:73-94) ---- */
/* float4 image -> RGBA8: min(v*255,255), NaN -> 0, rows flipped when flip != 0. Host memory. */
int rdc_image_to_rgba8(const float* image, int width, int height, int flip, uint8_t* out);
/* binary PPM (P6) and PNG (RGBA, uncompressed deflate) writers for headless runs */
int rdc_write_ppm(const char* path, const uint8_t* rgba, int width, int height);
int rdc_write_png(const char* path, const uint8_t* rgba, int width, int height);
/* baseline JPEG (JFIF, YCbCr 4:4:4), the format of the reference's screenshot: stbi_write_jpg(name, W, H, 4, rgba, W*4)
 * at glfw_events.cpp:94 — alpha ignored, and its out-of-range quality argument ends up as 100. quality 1..100. */
int rdc_write_jpg(const char* path, const uint8_t* rgba, int width, int height, int quality);

/* image-level comparison of two float4 host images, RGB only, NaN-aware (pixels that are NaN in both are skipped):
 * PSNR in dB on the [0,1] scale and the largest absolute difference — what BASELINE.json asks to be reported */
int rdc_psnr(const float* a, const float* b, size_t n_pixels, double* psnr, double* max_abs);

/* ---- the steps either side of the path in the frame loop (SURVEY.md 8f) ---- */
/* scroll_callback (glfw_events.cpp:105-112): zoom_factor *= 1.5^-yoffset */
void rdc_view_scroll(rdc_frame_params* params, double yoffset);
/* mouse_cursor_callback while dragging (glfw_events.cpp:115-130): offset -= cursor delta * zoom_factor */
void rdc_view_drag(rdc_frame_params* params, double dx, double dy);
/* Running mean over frames, in the role of the OptiX temporal denoiser the reference enables
 * (optixHello.cpp:1186-1235): accum <- accum + (image - accum)/(frames_so_far + 1). float4 device buffers. */
int rdc_accumulate(float* accum, const float* image, size_t n_pixels, uint32_t frames_so_far, rdc_stream stream);

/* ---- synthetic scenes (SURVEY.md §8d config 5): n_curves single-segment curves, SplitMix64(seed),
 *      emitted as XML text in the reference's schema so it passes through the same loader.
 *      Caller frees *out_text with rdc_free. ---- */
int rdc_synth_xml(uint32_t n_curves, uint32_t width, uint32_t height, uint64_t seed, char** out_text, size_t* out_len);

/* ---- measurement aid: dependent-FFMA microbenchmark used as the FP32 roofline denominator.
 *      Launches `launches` kernels of 148*8 blocks x 256 threads, each thread doing iters*64 FFMAs, on
 *      `stream`; returns the flop count of ONE launch in *flops_per_launch. Enqueue-only. ---- */
int rdc_microbench_fp32(int iters, int launches, float* sink, double* flops_per_launch, rdc_stream stream);
/* L2-read microbenchmark (the L2-side denominator for scenes whose runs and tree live in L2): each launch reads `bytes`
 * of `buffer` (device memory, small enough to stay in L2) `passes` times with 128-bit loads that bypass L1. */
int rdc_microbench_l2(const void* buffer, size_t bytes, int passes, int launches, float* sink, double* bytes_per_launch,
                      rdc_stream stream);

const char* rdc_last_error_string(void);
const char* rdc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RDC_B200_H */
