// rdc_math.h — the single source of truth for every piece of arithmetic that decides WHICH
// chord a ray hits, WHICH side it shades and WHERE along the curve it lands.
//
// It is compiled three ways and must give bit-identical results in all of them:
//   * nvcc for sm_100a with  -fmad=false            (the product kernels, csrc/*.cu)
//   * g++ with               -ffp-contract=off      (product host code)
//   * g++ with               -ffp-contract=off      (oracle/ — test infrastructure that INCLUDES this
//                                                    header; the product never includes oracle/)
// Contract: every C operator (* + - /) and sqrtf is one IEEE-754 round-to-nearest operation, in source
// order. A fused multiply-add happens only where rdc_fma() is written. No fast-math, no FTZ.
//
// What follows the reference and where (all paths relative to /root/reference/optixHello):
//   rdc_spline_point / rdc_spline_normal   DeviceCode.cu:64-75   (same rounding sequence, weights factored out)
//   rdc_is_ray_right                       DeviceCode.cu:78-83
//   rdc_interp                             DeviceCode.cu:36-44   (flat-array linear walk, strict '<')
//   rdc_u01                                curand_uniform's (0,1] mapping (CUDA curand_uniform.h)
// What is new (the reference delegates it to closed OptiX/cuRAND code, SURVEY.md §8c):
//   rdc_philox4x32_10, rdc_sincospi, rdc_ray_chord, rdc_chord_count, rdc_slab
#ifndef RDC_MATH_H
#define RDC_MATH_H

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define RDC_HD __host__ __device__ __forceinline__
#else
#define RDC_HD static inline
#endif

// The one fused operation. fmaf() is FFMA on the device irrespective of -fmad and a correctly rounded
// fused multiply-add on the host (hardware with -mfma, libm otherwise).
RDC_HD float rdc_fma(float a, float b, float c) { return fmaf(a, b, c); }

struct rdc_f2 {
  float x, y;
};

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011). counter = (pixel, ray, depth, 0), key = (seed, frame).
// Replaces the per-pixel XORWOW state of helperKernels.cu:151-155 / DeviceCode.cu:120,135-136.
// ------------------------------------------------------------------------------------------------
struct rdc_u4 {
  uint32_t x, y, z, w;
};

RDC_HD rdc_u4 rdc_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)M0 * c0;
    uint64_t p1 = (uint64_t)M1 * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  rdc_u4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
  return o;
}

// uint32 -> (0,1]:  x * 2^-32 + 2^-33  (one fused op; 0xFFFFFFFF maps to exactly 1.0f). x is rounded to float first,
// as in curand_uniform, so where that conversion rounds a tie down to even (x = 2^24 + 1, 0x80000080, ...) the result
// is one ulp below the correctly rounded value.
RDC_HD float rdc_u01(uint32_t x) { return rdc_fma((float)x, 2.3283064365386963e-10f, 1.1641532182693481e-10f); }

// ------------------------------------------------------------------------------------------------
// sincospi: sin(pi x), cos(pi x). Deterministic polynomial (glibc has no sincospif and CUDA's is not
// reproducible on the host). Accuracy ~2 ulp, which is all a unit ray direction needs. Domain |x| < 2^127 (2x must
// not overflow); the render passes |x| <= 2.
// ------------------------------------------------------------------------------------------------
RDC_HD void rdc_sincospi_kernel(float r, float* s, float* c) {
  // |r| <= 0.25. Taylor in (pi r): sin to r^9, cos to r^10.
  float r2 = r * r;
  float ps = 0.08214588661112823f;              //  pi^9/9!
  ps = rdc_fma(ps, r2, -0.5992645293207921f);   // -pi^7/7!
  ps = rdc_fma(ps, r2, 2.550164039877345f);     //  pi^5/5!
  ps = rdc_fma(ps, r2, -5.16771278004997f);     // -pi^3/3!
  float r3 = r2 * r;
  *s = rdc_fma(r3, ps, r * 3.14159265358979f);
  float pc = -0.02580689139001406f;             // -pi^10/10!
  pc = rdc_fma(pc, r2, 0.2353306303588935f);    //  pi^8/8!
  pc = rdc_fma(pc, r2, -1.3352627688545893f);   // -pi^6/6!
  pc = rdc_fma(pc, r2, 4.058712126416768f);     //  pi^4/4!
  pc = rdc_fma(pc, r2, -4.934802200544679f);    // -pi^2/2!
  *c = rdc_fma(pc, r2, 1.0f);
}

RDC_HD void rdc_sincospi(float x, float* s, float* c) {
  float q = rintf(x * 2.0f);
  float r = rdc_fma(q, -0.5f, x);  // exact
  float sr, cr;
  rdc_sincospi_kernel(r, &sr, &cr);
  // quadrant = q mod 4, reduced in float (exact for every finite q). (int)q itself differs between the builds once
  // |q| >= 2^31: the device saturates, x86 gives INT_MIN.
  const float qm = q - 4.0f * floorf(q * 0.25f);
  const int iq = qm >= 0.0f && qm < 4.0f ? (int)qm : 0;  // NaN, inf: r is NaN anyway
  if (iq & 1) { float t = sr; sr = cr; cr = -t; }  // rotate by 90 degrees
  if (iq & 2) { sr = -sr; cr = -cr; }              // rotate by 180 degrees
  *s = sr; *c = cr;
}

// ------------------------------------------------------------------------------------------------
// Uniform cubic B-spline, 2-D (z is always 0 in the reference: optixHello.cpp:1318-1328).
// v = 4 control points. Same rounding sequence as DeviceCode.cu:64-75 with the scalar basis
// polynomials evaluated once instead of once per coordinate (identical values).
// ------------------------------------------------------------------------------------------------
RDC_HD rdc_f2 rdc_spline_point(float t, const rdc_f2 v0, const rdc_f2 v1, const rdc_f2 v2, const rdc_f2 v3) {
  float t3 = t * t * t;
  float w0 = -1 * t * t * t + 3 * t * t - 3 * t + 1;
  float w1 = 3 * t * t * t - 6 * t * t + 4;
  float w2 = -3 * t * t * t + 3 * t * t + 3 * t + 1;
  const float sixth = 1 / 6.0f;
  rdc_f2 r;
  r.x = sixth * (t3 * v3.x + v0.x * w0 + v1.x * w1 + v2.x * w2);
  r.y = sixth * (t3 * v3.y + v0.y * w0 + v1.y * w1 + v2.y * w2);
  return r;
}

// Right-hand normal (T.y, -T.x) of the spline tangent T. Not normalised.
RDC_HD rdc_f2 rdc_spline_normal(float t, const rdc_f2 v0, const rdc_f2 v1, const rdc_f2 v2, const rdc_f2 v3) {
  float d3 = 3 * t * t;
  float d0 = -3 * t * t + 6 * t - 3;
  float d1 = 9 * t * t - 12 * t;
  float d2 = -9 * t * t + 6 * t + 3;
  const float sixth = 1 / 6.0f;
  rdc_f2 r;
  r.x = sixth * (d3 * v3.y + v0.y * d0 + v1.y * d1 + v2.y * d2);
  r.y = -sixth * (d3 * v3.x + v0.x * d0 + v1.x * d1 + v2.x * d2);
  return r;
}

// DeviceCode.cu:78-83. orzan = USE_DIFFUSION_CURVE_SAVE.
RDC_HD bool rdc_is_ray_right(float t, float dx, float dy, const rdc_f2 v0, const rdc_f2 v1, const rdc_f2 v2,
                             const rdc_f2 v3, bool orzan) {
  rdc_f2 n = rdc_spline_normal(t, v0, v1, v2, v3);
  return ((n.x * dx + n.y * dy) <= 0) != orzan;
}

// ------------------------------------------------------------------------------------------------
// Stop-list walk, DeviceCode.cu:36-44. `us` is the FLAT array of all curves' stops; the walk may run one
// or two entries past the curve's own (start,count) range exactly like the reference does (SURVEY.md
// Appendix A.4). Memory safety comes from the +INF sentinels the ingest appends, not from a clamp.
// ------------------------------------------------------------------------------------------------
// The interpolation ratio only blends stop values (colours, blur, weights): it never decides a hit or a
// side, so the device build may use the 2-ulp reciprocal-multiply division; host and oracle divide exactly.
// Measured on a B200 (tests/test_shared_math_gpu.py): at most 1.95 ulp for |den| in [2^-126, 2^126]; 0 for
// |den| > 2^126 (where num/den is below 2^-122 for the stops' num); for a denormal den the same infinity as
// num/den where that overflows; zero, infinite and NaN operands as IEEE division.
RDC_HD float rdc_ratio(float num, float den) {
#if defined(__CUDA_ARCH__)
  return __fdividef(num, den);
#else
  return num / den;
#endif
}

// walk from `first` (any index the walk from the list's start is known to reach) up to `end` = start+count
RDC_HD int rdc_interp_from(uint32_t first, uint32_t end, float u, const float* us, float* ratio) {
  // same walk as DeviceCode.cu:39-43, carrying us[ind] and us[ind+1] in registers: one load per step
  const float* p = us + first;
  const float* const stop = us + end;
  float lo = p[0], hi = p[1];
  while (p < stop && hi < u) {
    ++p;
    lo = hi;
    hi = p[1];
  }
  *ratio = rdc_ratio(u - lo, hi - lo);
  return (int)(p - us);
}

RDC_HD int rdc_interp(uint32_t start, uint32_t count, float u, const float* us, float* ratio) {
  return rdc_interp_from(start, start + count, u, us, ratio);
}

// Where the walk stands once it has consumed every stop below u_min. For any u >= u_min the walk from
// `start` passes through this index (each stop it skipped satisfies us[j+1] < u_min <= u), so starting
// there gives the same result — also for non-monotonic lists. A spline segment's hits all have
// u >= its ordinal, which makes this a per-segment constant (device_scene.h: SegWalk).
RDC_HD uint32_t rdc_walk_hint(uint32_t start, uint32_t count, float u_min, const float* us) {
  uint32_t j = start;
  while (j < start + count && us[j + 1] < u_min) j++;
  return j;
}

RDC_HD float rdc_lerp_stop(float a, float b, float ratio) { return (1 - ratio) * a + ratio * b; }
// colour stops use the other operand order (DeviceCode.cu:53-55)
RDC_HD float rdc_lerp_color(float a, float b, float ratio) { return a * (1 - ratio) + b * ratio; }

// ------------------------------------------------------------------------------------------------
// Chord subdivision. A spline segment becomes K parameter-uniform chords; K bounds
// |P(u) - chord(u)| <= max|P''| / (8 K^2) <= tol  (position AND parametrisation error).
// P''(u) = (1-u)(B0 - 2 B1 + B2) + u (B1 - 2 B2 + B3).
// ------------------------------------------------------------------------------------------------
RDC_HD int rdc_chord_count(const rdc_f2 v0, const rdc_f2 v1, const rdc_f2 v2, const rdc_f2 v3, float tol, int kmax) {
  float ax = v0.x - 2 * v1.x + v2.x, ay = v0.y - 2 * v1.y + v2.y;
  float bx = v1.x - 2 * v2.x + v3.x, by = v1.y - 2 * v2.y + v3.y;
  float m = fmaxf(ax * ax + ay * ay, bx * bx + by * by);
  float k = ceilf(sqrtf(sqrtf(m) / (8.0f * tol)));
  if (!(k >= 1.0f)) k = 1.0f;  // also catches NaN
  if (k > (float)kmax) k = (float)kmax;
  return (int)k;
}

// parameter of chord end point k of K, and of a hit at fraction s on chord k
RDC_HD float rdc_chord_u(int k, int K) { return (float)k / (float)K; }
RDC_HD float rdc_hit_u(int k, int K, float s) { return ((float)k + s) / (float)K; }

// ------------------------------------------------------------------------------------------------
// Ray vs chord. Replaces OptiX's built-in round-cubic-B-spline intersector (optixHello.cpp:768,868-879;
// results consumed at DeviceCode.cu:196-198). Edge-function form: the ray's supporting line separates A
// and B iff cross(D,A-O) and cross(D,B-O) differ in sign. The value at a vertex shared by two chords is
// computed from identical inputs, so a polyline is watertight. s is the fraction along the chord, t the
// ray parameter of the hit point (projection form: stays accurate for grazing rays, and the hit point
// always lies inside the chord's bounding box, which is what makes BVH culling exact).
// inv_dd = rdc_inv_dd(D, primary).
// ------------------------------------------------------------------------------------------------
// edge value of a chord end point P seen from the ray: cross(D, P-O), with w = P-O
RDC_HD float rdc_edge(float dx, float dy, float wx, float wy) { return rdc_fma(dx, wy, -(dy * wx)); }

// second half of the test, given both end points relative to the origin and their edge values
RDC_HD bool rdc_chord_hit(float dx, float dy, float inv_dd, float wax, float way, float wbx, float wby, float ea,
                          float eb, float* t, float* s) {
  if ((ea > 0.0f) == (eb > 0.0f)) return false;
  float sv = ea / (ea - eb);
  sv = fminf(fmaxf(sv, 0.0f), 1.0f);
  float rx = rdc_fma(sv, wbx - wax, wax);
  float ry = rdc_fma(sv, wby - way, way);
  float tt = rdc_fma(rx, dx, ry * dy) * inv_dd;
  if (!(tt > 0.0f)) return false;
  *t = tt; *s = sv;
  return true;
}

RDC_HD bool rdc_ray_chord(float ox, float oy, float dx, float dy, float inv_dd, float ax, float ay, float bx,
                          float by, float* t, float* s) {
  float wax = ax - ox, way = ay - oy;
  float wbx = bx - ox, wby = by - oy;
  return rdc_chord_hit(dx, dy, inv_dd, wax, way, wbx, wby, rdc_edge(dx, dy, wax, way), rdc_edge(dx, dy, wbx, wby), t, s);
}

// 1/(D.D) as used by the chord test. Primary rays are (1,0) rotated up to N-1 times, i.e. unit length up to 1e-7 N, and
// their t is reported in units of |D|^2 like the ray parameter OptiX reports is in units of |D|: the
// factor is exactly 1 for them (no division on the hot path). Portal continuation rays are not unit
// length (DeviceCode.cu:243,255-256) and get the true reciprocal.
RDC_HD float rdc_inv_dd(float dx, float dy, bool primary) { return primary ? 1.0f : 1.0f / (dx * dx + dy * dy); }

// chords per leaf of the product's tree: a leaf is a run of up to RDC_RUN consecutive chords of one
// segment (RDC_RUN+1 points), so shared end points are stored and evaluated once
#define RDC_RUN 8

// Portal continuation rays start ON the target segment (at the true spline point, DeviceCode.cu:229),
// which lies within the flatness tolerance of chord k0 = floor(u K) of that segment. Like a ray that
// starts inside OptiX's swept tube, they do not see the surface they leave: chords k0-1..k0+1 of the
// target segment are skipped. Returns the inclusive k range.
// u K is clamped in float before the conversion: (int) of NaN, inf or anything beyond 2^31 differs between the builds.
RDC_HD void rdc_portal_skip(float u, int K, int* klo, int* khi) {
  int k0 = (int)fminf(fmaxf(u * (float)K, 0.0f), (float)(K > 1 ? K - 1 : 0));
  *klo = k0 > 0 ? k0 - 1 : 0;
  *khi = k0 < K - 1 ? k0 + 1 : K - 1;
}

// closest-hit ordering: smaller t wins, equal t -> smaller chord id (order-independent, so brute force
// and any BVH visit order agree)
RDC_HD bool rdc_hit_closer(float t, uint32_t id, float best_t, uint32_t best_id) {
  return t < best_t || (t == best_t && id < best_id);
}

// ------------------------------------------------------------------------------------------------
// Ray vs padded 2-D box (slab test). Returns entry parameter; *exit gets the exit parameter.
// idx/idy = 1/D with |D| clamped away from 0 (rdc_safe_inv) so that 0*inf never appears.
// ------------------------------------------------------------------------------------------------
RDC_HD float rdc_safe_inv(float d) {
  float a = fabsf(d) < 1e-30f ? copysignf(1e-30f, d) : d;
  return 1.0f / a;
}

RDC_HD float rdc_slab(float ox, float oy, float idx, float idy, float xmin, float ymin, float xmax, float ymax,
                      float* exit) {
  float tx1 = (xmin - ox) * idx, tx2 = (xmax - ox) * idx;
  float ty1 = (ymin - oy) * idy, ty2 = (ymax - oy) * idy;
  // fminf/fmaxf of +0 and -0 may return either zero (glibc and the device differ): + 0.0f makes a zero +0 in both
  float tn = fmaxf(fmaxf(fminf(tx1, tx2), fminf(ty1, ty2)), 0.0f) + 0.0f;
  *exit = fminf(fmaxf(tx1, tx2), fmaxf(ty1, ty2)) + 0.0f;
  return tn;
}

// relative slack applied to the best-so-far t when culling a box: covers the few ulp of rounding in
// rdc_slab so that a chord that would win is never culled.
#define RDC_CULL_SLACK 1.000002f

// ------------------------------------------------------------------------------------------------
// Point vs chord (rdc_scene_pick). s = the fraction along the chord of the point nearest to p, c = a + s e that
// point, d2 = |p - c|^2. No rdc_fma: one rounding per C operator, so a float32 numpy restatement gives the same bits.
// ------------------------------------------------------------------------------------------------
RDC_HD void rdc_point_chord(float px, float py, float ax, float ay, float bx, float by, float* s, float* cx, float* cy,
                            float* d2) {
  const float ex = bx - ax, ey = by - ay;
  const float wx = px - ax, wy = py - ay;
  const float ee = ex * ex + ey * ey;
  float sv = ee > 0.0f ? (wx * ex + wy * ey) / ee : 0.0f;
  sv = fminf(fmaxf(sv, 0.0f), 1.0f);
  const float x = ax + sv * ex, y = ay + sv * ey;
  const float dx = px - x, dy = py - y;
  *s = sv; *cx = x; *cy = y;
  *d2 = dx * dx + dy * dy;
}

// Squared distance from p to a box, in the same operations as d2 above: for any point c inside the box, |b.x - px| <=
// |cx - px| per axis, and rounding is monotone, so this never exceeds rdc_point_chord's d2 of c (pick.cu).
RDC_HD float rdc_point_box_d2(float px, float py, float xmin, float ymin, float xmax, float ymax) {
  const float dx = fmaxf(fmaxf(xmin - px, px - xmax), 0.0f);
  const float dy = fmaxf(fmaxf(ymin - py, py - ymax), 0.0f);
  return dx * dx + dy * dy;
}

// nearest-chord ordering: smaller d2 wins, equal d2 -> smaller chord id (the role rdc_hit_closer plays for rays: any
// visit order gives the brute force's answer)
RDC_HD bool rdc_pick_closer(float d2, uint32_t id, float best_d2, uint32_t best_id) {
  return d2 < best_d2 || (d2 == best_d2 && id < best_id);
}

// Centre of pixel (ix, iy) in scene coordinates: the render kernel's ray origin before the jitter (render.cu origin_x /
// origin_y, DeviceCode.cu:103-107: unsigned arithmetic, then a signed cast) plus half a pixel. Anti-aliasing jitters
// that origin by (0,1] x zoom per axis, so this is the centre of the square the pixel's rays start from, for negative
// zoom too.
RDC_HD float rdc_pixel_centre_x(uint32_t width, float zoom, float off_x, uint32_t ix) {
  return ((float)(int)(ix - (width / 2)) * zoom + off_x) + 0.5f * zoom;
}
RDC_HD float rdc_pixel_centre_y(uint32_t height, float zoom, float off_y, bool orzan, uint32_t iy) {
  const float base = orzan ? (float)(int)((height - iy) - (height / 2)) * zoom + off_y : (float)(int)(iy - (height / 2)) * zoom + off_y;
  return base + 0.5f * zoom;
}

// w = wm * t^-e  (DeviceCode.cu:330). Host and oracle use libm powf; the device build uses CUDA powf or a
// reciprocal square root when e == 0.5 (the default exponent, optixHello.cpp:94). Weights only scale
// colours, never decide a hit, so this is inside the 1e-4 RGB tolerance and outside the bit-exact set. Measured on a
// B200 over t in [1e-6, 1e6]: relative error 1.2e-7 for e = 0.5, 7.8e-7 for e = 1, 5.7e-6 for e = 3.7.
RDC_HD float rdc_weight_falloff(float t, float e) {
#if defined(__CUDA_ARCH__)
  if (e == 0.5f) return rsqrtf(t);
  return exp2f(-e * log2f(t));
#else
  return powf(t, -e);
#endif
}

#endif  // RDC_MATH_H
