// Test probe for csrc/rdc_math.h: one C entry point per function family, mapping rows of input words to rows of
// output words. The same file builds twice (tests/math_probe.py): with nvcc and the Makefile's NVFLAGS, where every
// entry point launches a kernel with one thread per row, and with g++ -x c++ and the Makefile's CXXFLAGS, where it
// loops over the rows on the host. Comparing the two builds word for word checks the header's claim that both give
// bit-identical results.
//
// Every entry point has the signature
//     int rdcp_<name>(int n, const uint32_t* in, uint32_t* out, const float* aux)
// `in` holds n rows of the function's input words and `out` n rows of its output words, row-major; a float travels as
// its bit pattern. `aux` is a table only the stop-list walks read. Device builds take device pointers and launch on
// the legacy default stream; they return the launch's cudaError_t, the host build returns 0.
#include <stdint.h>
#include <string.h>

#include "../../raytracingdiffusioncurves_b200/csrc/rdc_math.h"

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define PHD __host__ __device__
#else
#define PHD
#endif

namespace {

PHD inline float F(uint32_t w) {
  float f;
  memcpy(&f, &w, 4);
  return f;
}
PHD inline uint32_t W(float f) {
  uint32_t w;
  memcpy(&w, &f, 4);
  return w;
}
PHD inline rdc_f2 P(const uint32_t* r) {
  rdc_f2 p;
  p.x = F(r[0]);
  p.y = F(r[1]);
  return p;
}

#if defined(__CUDACC__)
template <class Op>
__global__ void k_rows(Op op, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) op(i);
}
template <class Op>
int run(const Op& op, int n) {
  if (n > 0) k_rows<<<(n + 255) / 256, 256>>>(op, n);
  return (int)cudaGetLastError();
}
#else
template <class Op>
int run(const Op& op, int n) {
  for (int i = 0; i < n; ++i) op(i);
  return 0;
}
#endif

// An operation sees row i of the inputs (NI words) and of the outputs (NO words).
#define RDCP_OP(name, NI, NO)                                                             \
  struct name##_op {                                                                      \
    const uint32_t* in;                                                                   \
    uint32_t* out;                                                                        \
    const float* aux;                                                                     \
    PHD void operator()(int i) const { body(in + (size_t)i * NI, out + (size_t)i * NO); } \
    PHD void body(const uint32_t* a, uint32_t* o) const;                                  \
  };                                                                                      \
  }                                                                                       \
  extern "C" int rdcp_##name(int n, const uint32_t* in, uint32_t* out, const float* aux) { \
    return run(name##_op{in, out, aux}, n);                                              \
  }                                                                                       \
  namespace {                                                                             \
  PHD void name##_op::body(const uint32_t* a, uint32_t* o) const

// ctr c0..c3, key k0 k1 -> 4 words
RDCP_OP(philox, 6, 4) {
  const rdc_u4 r = rdc_philox4x32_10(a[0], a[1], a[2], a[3], a[4], a[5]);
  o[0] = r.x; o[1] = r.y; o[2] = r.z; o[3] = r.w;
}

// x -> u01(x)
RDCP_OP(u01, 1, 1) { o[0] = W(rdc_u01(a[0])); }

// x -> sin(pi x), cos(pi x)
RDCP_OP(sincospi, 1, 2) {
  float s, c;
  rdc_sincospi(F(a[0]), &s, &c);
  o[0] = W(s); o[1] = W(c);
}

RDCP_OP(sincospi_kernel, 1, 2) {
  float s, c;
  rdc_sincospi_kernel(F(a[0]), &s, &c);
  o[0] = W(s); o[1] = W(c);
}

// t, v0..v3 -> point, normal
RDCP_OP(spline, 9, 4) {
  const rdc_f2 p = rdc_spline_point(F(a[0]), P(a + 1), P(a + 3), P(a + 5), P(a + 7));
  const rdc_f2 q = rdc_spline_normal(F(a[0]), P(a + 1), P(a + 3), P(a + 5), P(a + 7));
  o[0] = W(p.x); o[1] = W(p.y); o[2] = W(q.x); o[3] = W(q.y);
}

// t, dx, dy, v0..v3, orzan -> right?
RDCP_OP(is_ray_right, 12, 1) {
  o[0] = rdc_is_ray_right(F(a[0]), F(a[1]), F(a[2]), P(a + 3), P(a + 5), P(a + 7), P(a + 9), a[11] != 0);
}

// first, end, u over the stop table aux -> index, ratio
RDCP_OP(interp_from, 3, 2) {
  float ratio;
  o[0] = (uint32_t)rdc_interp_from(a[0], a[1], F(a[2]), aux, &ratio);
  o[1] = W(ratio);
}

// start, count, u_min over the stop table aux -> index
RDCP_OP(walk_hint, 3, 1) { o[0] = rdc_walk_hint(a[0], a[1], F(a[2]), aux); }

// a, b, ratio -> lerp_stop, lerp_color
RDCP_OP(lerp, 3, 2) {
  o[0] = W(rdc_lerp_stop(F(a[0]), F(a[1]), F(a[2])));
  o[1] = W(rdc_lerp_color(F(a[0]), F(a[1]), F(a[2])));
}

// v0..v3, tol, kmax -> K
RDCP_OP(chord_count, 10, 1) {
  o[0] = (uint32_t)rdc_chord_count(P(a), P(a + 2), P(a + 4), P(a + 6), F(a[8]), (int)a[9]);
}

// ox, oy, dx, dy, inv_dd, ax, ay, bx, by -> hit, t, s (t and s keep their initial bits on a miss)
RDCP_OP(ray_chord, 9, 3) {
  float t = F(0x7fc00001u), s = F(0x7fc00002u);
  o[0] = rdc_ray_chord(F(a[0]), F(a[1]), F(a[2]), F(a[3]), F(a[4]), F(a[5]), F(a[6]), F(a[7]), F(a[8]), &t, &s);
  o[1] = W(t); o[2] = W(s);
}

// dx, dy, inv_dd, wax, way, wbx, wby, ea, eb -> hit, t, s
RDCP_OP(chord_hit, 9, 3) {
  float t = F(0x7fc00001u), s = F(0x7fc00002u);
  o[0] = rdc_chord_hit(F(a[0]), F(a[1]), F(a[2]), F(a[3]), F(a[4]), F(a[5]), F(a[6]), F(a[7]), F(a[8]), &t, &s);
  o[1] = W(t); o[2] = W(s);
}

// dx, dy, primary -> 1/(D.D) or 1
RDCP_OP(inv_dd, 3, 1) { o[0] = W(rdc_inv_dd(F(a[0]), F(a[1]), a[2] != 0)); }

// u, K -> klo, khi
RDCP_OP(portal_skip, 2, 2) {
  int klo, khi;
  rdc_portal_skip(F(a[0]), (int)a[1], &klo, &khi);
  o[0] = (uint32_t)klo; o[1] = (uint32_t)khi;
}

RDCP_OP(safe_inv, 1, 1) { o[0] = W(rdc_safe_inv(F(a[0]))); }

// ox, oy, idx, idy, xmin, ymin, xmax, ymax -> entry, exit
RDCP_OP(slab, 8, 2) {
  float ex;
  const float tn = rdc_slab(F(a[0]), F(a[1]), F(a[2]), F(a[3]), F(a[4]), F(a[5]), F(a[6]), F(a[7]), &ex);
  o[0] = W(tn); o[1] = W(ex);
}

// px, py, ax, ay, bx, by -> s, cx, cy, d2
RDCP_OP(point_chord, 6, 4) {
  float s, cx, cy, d2;
  rdc_point_chord(F(a[0]), F(a[1]), F(a[2]), F(a[3]), F(a[4]), F(a[5]), &s, &cx, &cy, &d2);
  o[0] = W(s); o[1] = W(cx); o[2] = W(cy); o[3] = W(d2);
}

// px, py, xmin, ymin, xmax, ymax -> d2
RDCP_OP(point_box_d2, 6, 1) { o[0] = W(rdc_point_box_d2(F(a[0]), F(a[1]), F(a[2]), F(a[3]), F(a[4]), F(a[5]))); }

// size (width = height), zoom, offset, orzan, index -> centre x, centre y
RDCP_OP(pixel_centre, 5, 2) {
  o[0] = W(rdc_pixel_centre_x(a[0], F(a[1]), F(a[2]), a[4]));
  o[1] = W(rdc_pixel_centre_y(a[0], F(a[1]), F(a[2]), a[3] != 0, a[4]));
}

// num, den -> num / den (the device build's __fdividef)
RDCP_OP(ratio, 2, 1) { o[0] = W(rdc_ratio(F(a[0]), F(a[1]))); }

// t, e -> t^-e
RDCP_OP(weight_falloff, 2, 1) { o[0] = W(rdc_weight_falloff(F(a[0]), F(a[1]))); }

// Ray directions, restated from csrc/render.cu: k_base_dirs (the base direction of ray i, (1,0) rotated i times by the
// fp32 matrix of sincospi(2/N)) and gen_ray's jitter (the base direction rotated by sincospi(two_over_n * u01), through
// rdc_sincospi_kernel when two_over_n <= 1/4). Same operations in the same order; keep the two in step.
//
// two_over_n, n_iter in row 0 -> n_iter rows of (x, y). Serial like k_base_dirs: call with n = 1.
RDCP_OP(base_dirs, 2, 0) {
  float rs, rc;
  rdc_sincospi(F(a[0]), &rs, &rc);
  float x = 1.0f, y = 0.0f;
  uint32_t* d = out;
  for (int i = 0; i < (int)a[1]; ++i) {
    d[2 * i] = W(x); d[2 * i + 1] = W(y);
    float nx = x * rc - y * rs;
    float ny = x * rs + y * rc;
    x = nx; y = ny;
  }
  (void)o;
}

// base x, base y, two_over_n, u01 -> jittered direction
RDCP_OP(jitter, 4, 2) {
  const float bx = F(a[0]), by = F(a[1]), two_over_n = F(a[2]);
  const bool small_angle = two_over_n <= 0.25f && two_over_n >= 0.0f;
  float js, jc;
  const float ang = two_over_n * F(a[3]);
  if (small_angle) rdc_sincospi_kernel(ang, &js, &jc);
  else rdc_sincospi(ang, &js, &jc);
  o[0] = W(bx * jc - by * js);
  o[1] = W(bx * js + by * jc);
}

}  // namespace
