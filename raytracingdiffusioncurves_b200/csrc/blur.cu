// blur.cu — separable gather blur with a per-destination-pixel sigma.
//
// Same result as helperKernels.cu:48-148 (gaussHorizontal, gaussVertical, gaussianBlur): taps
// k in [-ceil(3 sigma), +ceil(3 sigma)], weight expf(-(k*k)/(sigma+1e-6)^2) (no factor 2), clamp-to-edge,
// renormalised, all four channels, the vertical pass reads the SAME un-blurred sigma map.
// What differs is the execution: a grid sized to the GPU (148 SMs x 16 blocks) instead of a fixed 512x256
// launch, accumulation in registers instead of read-modify-write on dest[i], scratch supplied
// by the caller (or the stream-ordered allocator) instead of cudaMalloc/cudaFree per frame, and an
// optional device flag that turns both passes into (at most) one copy when every sigma is zero.
#include "device_scene.h"

namespace rdc {
namespace {

constexpr int kThreads = 256;
constexpr unsigned kMaxBlocks = 148 * 16;  // 148 SMs x 16 resident blocks of 256 threads at most
constexpr float kMinSigma = 1e-6f;   // helperKernels.cu:27
constexpr float kMaxTaps = 16384.0f; // |k| bound for non-finite or absurd sigmas (edge pixels repeat anyway)

struct Taps {
  int first, last;
  float sig_square;
};

__device__ __forceinline__ Taps taps_for(float sigma) {
  // k_size = 2*ceilf(3*sigma)+1; for (int k = -k_size/2; k <= k_size/2; k++)   (helperKernels.cu:65,74)
  float k_size = 2 * ceilf(3 * sigma) + 1;
  Taps t;
  float lo = -k_size / 2, hi = k_size / 2;
  if (!(k_size == k_size)) {  // NaN sigma: the reference's loop condition is false at once -> 0/0
    t.first = 0;
    t.last = -1;
  } else {
    lo = fmaxf(lo, -kMaxTaps);
    hi = fminf(hi, kMaxTaps);
    t.first = (int)lo;               // truncation toward zero, like the reference's int conversion
    t.last = (int)floorf(hi);        // largest int k with (float)k <= hi
  }
  t.sig_square = (sigma + kMinSigma) * (sigma + kMinSigma);
  return t;
}

// weight of tap k; the forward passes and the transpose share it, so the transpose's tap sums have the forward's bits
__device__ __forceinline__ float tap_weight(int k, const Taps& t) { return expf(-(k * k) / t.sig_square); }

__device__ __forceinline__ bool all_sigma_zero(const float* max_sigma) {
  return max_sigma != nullptr && __ldg(max_sigma) == 0.0f;
}

// rows [h_begin,h_end): scratch = horizontal blur of source. With an all-zero sigma map the pass is the
// identity, so it writes `dest` directly (nothing at all when dest == source).
__global__ void k_blur_horizontal(const float4* __restrict__ source, float4* scratch, float4* dest,
                                  const float* __restrict__ sigma, int width, int h_begin, int h_end, const float* max_sigma) {
  const size_t count = (size_t)width * (h_end - h_begin), first = (size_t)h_begin * width;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  const bool identity = all_sigma_zero(max_sigma);
  if (identity && dest == source) return;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const size_t i = first + j;
    if (identity) {
      dest[i] = source[i];
      continue;
    }
    const int x = (int)(i % width);
    const size_t row = i - x;
    const Taps t = taps_for(sigma[i]);
    float accum = 0.0f;
    float4 d = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    for (int k = t.first; k <= t.last; ++k) {
      const int sx = max(0, min(x + k, width - 1));
      const float g = tap_weight(k, t);
      const float4 s = source[row + sx];
      accum += g;
      d.x += s.x * g;
      d.y += s.y * g;
      d.z += s.z * g;
      d.w += s.w * g;
    }
    scratch[i] = make_float4(d.x / accum, d.y / accum, d.z / accum, d.w / accum);
  }
}

// rows [row_begin,row_end): dest = vertical blur of scratch, rows clamped to [0,height-1]
__global__ void k_blur_vertical(const float4* __restrict__ scratch, float4* __restrict__ dest,
                                const float* __restrict__ sigma, int width, int height, int row_begin, int row_end,
                                const float* max_sigma) {
  if (all_sigma_zero(max_sigma)) return;
  const size_t count = (size_t)width * (row_end - row_begin), first = (size_t)row_begin * width;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const size_t i = first + j;
    const int x = (int)(i % width);
    const int y = (int)(i / width);
    const Taps t = taps_for(sigma[i]);
    float accum = 0.0f;
    float4 d = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    for (int k = t.first; k <= t.last; ++k) {
      const int sy = max(0, min(y + k, height - 1));
      const float g = tap_weight(k, t);
      const float4 s = scratch[(size_t)sy * width + x];
      accum += g;
      d.x += s.x * g;
      d.y += s.y * g;
      d.z += s.z * g;
      d.w += s.w * g;
    }
    dest[i] = make_float4(d.x / accum, d.y / accum, d.z / accum, d.w / accum);
  }
}

// ---- the transpose of the two passes (gaussian_blur_adjoint) ----
//
// Forward, per pixel p with taps [f, l] and a = sum_k g(k) (tap order):
//   T(x,y) = sum_k g(k) S(clampx(x+k), y) / a,   D(x,y) = sum_k g(k) T(x, clampy(y+k)) / a,   g and a of the pixel written.
// Transpose, gradient G on the band:  G^ = G / a on the band;  vertical: G_T(x,y') = sum_y G^(x,y) sum_{k: clampy(y+k)=y'} g(k);
// G_T / a(x,y');  horizontal: G_S(x',y') = sum_x (G_T/a)(x,y') sum_{k: clampx(x+k)=x'} g(k). Each sum is a gather (one thread
// per output pixel, no atomics, so repeats give the same bits) over the sources within the reach R = max(-f, l) of any
// pixel. Clamp-to-edge: output row / column 0 collects the taps at or below it, the last one the taps at or above it (a
// buffer one pixel wide collects all of them). A pixel without taps (NaN sigma, sigma <= -1/3) has a NaN forward output:
// it contributes nothing here.

// sum of the weights of taps [lo, hi], in tap order (the forward's accum when [lo, hi] = [first, last])
__device__ __forceinline__ float tap_sum(const Taps& t, int lo, int hi) {
  float s = 0.0f;
  for (int k = lo; k <= hi; ++k) s += tap_weight(k, t);
  return s;
}

// weight with which a pass at source position `from` (taps t) reads position `to` of a line of n: the taps k with
// clamp(from + k, 0, n - 1) == to
__device__ __forceinline__ float clamped_weight(const Taps& t, int from, int to, int n) {
  const int lo = to == 0 ? t.first : max(t.first, to - from);
  const int hi = to == n - 1 ? t.last : min(t.last, to - from);
  return lo <= hi ? tap_sum(t, lo, hi) : 0.0f;
}

// *reach = max(-first, last) over the buffer's pixels that have taps (the caller zeroes it); taps_for caps it at kMaxTaps
__global__ void k_blur_reach(const float* __restrict__ sigma, size_t count, const float* max_sigma, int* reach) {
  if (all_sigma_zero(max_sigma)) return;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  int r = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const Taps t = taps_for(sigma[i]);
    if (t.first <= t.last) r = max(r, max(-t.first, t.last));
  }
  r = __reduce_max_sync(0xffffffffu, r);
  if ((threadIdx.x & 31) == 0 && r > 0) atomicMax(reach, r);
}

// band rows: grad_source = grad_dest / a, 0 where the pixel has no taps (in place when the two are the same buffer). With
// an all-zero sigma map the blur is the identity on the band: a copy.
__global__ void k_blur_adjoint_scale(const float4* grad_dest, float4* grad_source, const float* __restrict__ sigma, int width,
                                     int row_begin, int row_end, const float* max_sigma) {
  const size_t count = (size_t)width * (row_end - row_begin), first = (size_t)row_begin * width;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  const bool identity = all_sigma_zero(max_sigma);
  if (identity && grad_dest == grad_source) return;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const size_t i = first + j;
    const float4 g = grad_dest[i];
    if (identity) {
      grad_source[i] = g;
      continue;
    }
    const Taps t = taps_for(sigma[i]);
    if (t.first > t.last) {
      grad_source[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      continue;
    }
    const float accum = tap_sum(t, t.first, t.last);
    grad_source[i] = make_float4(g.x / accum, g.y / accum, g.z / accum, g.w / accum);
  }
}

// rows [row_begin - R, row_end + R) of the buffer: scratch = (vertical transpose of the scaled band) / a, 0 where the
// pixel has no taps (the horizontal pass there reads nothing)
__global__ void k_blur_adjoint_vertical(const float4* __restrict__ scaled, float4* __restrict__ scratch,
                                        const float* __restrict__ sigma, int width, int height, int row_begin, int row_end,
                                        const int* __restrict__ reach, const float* max_sigma) {
  if (all_sigma_zero(max_sigma)) return;
  const int r = *reach;
  const int lo_row = max(0, row_begin - r), hi_row = min(height, row_end + r);
  const size_t count = (size_t)width * (hi_row - lo_row), first = (size_t)lo_row * width;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const size_t i = first + j;
    const int x = (int)(i % width);
    const int y = (int)(i / width);
    float4 d = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    const int y_end = min(row_end - 1, y + r);
    for (int sy = max(row_begin, y - r); sy <= y_end; ++sy) {
      const size_t s_i = (size_t)sy * width + x;
      const float w = clamped_weight(taps_for(sigma[s_i]), sy, y, height);
      if (w == 0.0f) continue;
      const float4 s = scaled[s_i];
      d.x += s.x * w;
      d.y += s.y * w;
      d.z += s.z * w;
      d.w += s.w * w;
    }
    const Taps t = taps_for(sigma[i]);
    if (t.first > t.last) {
      scratch[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      continue;
    }
    const float accum = tap_sum(t, t.first, t.last);
    scratch[i] = make_float4(d.x / accum, d.y / accum, d.z / accum, d.w / accum);
  }
}

// every row: grad_source = horizontal transpose of scratch on rows [row_begin - R, row_end + R), 0 on the other rows.
// With an all-zero sigma map, 0 outside the band and the band rows as k_blur_adjoint_scale left them.
__global__ void k_blur_adjoint_horizontal(const float4* __restrict__ scratch, float4* __restrict__ grad_source,
                                          const float* __restrict__ sigma, int width, int height, int row_begin, int row_end,
                                          const int* __restrict__ reach, const float* max_sigma) {
  const bool identity = all_sigma_zero(max_sigma);
  const int r = identity ? 0 : *reach;
  const int lo_row = max(0, row_begin - r), hi_row = min(height, row_end + r);
  const size_t count = (size_t)width * height;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const int x = (int)(i % width);
    const int y = (int)(i / width);
    if (y < lo_row || y >= hi_row) {
      grad_source[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      continue;
    }
    if (identity) continue;
    const size_t row = i - x;
    float4 d = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    const int x_end = min(width - 1, x + r);
    for (int sx = max(0, x - r); sx <= x_end; ++sx) {
      const float w = clamped_weight(taps_for(sigma[row + sx]), sx, x, width);
      if (w == 0.0f) continue;
      const float4 s = scratch[row + sx];
      d.x += s.x * w;
      d.y += s.y * w;
      d.z += s.z * w;
      d.w += s.w * w;
    }
    grad_source[i] = d;
  }
}

// ---- the derivative in sigma (gaussian_blur_sigma_adjoint) ----
//
// With the taps [f, l] of a pixel held fixed, a pass Y(p) = sum_k g(k) X(clamp(p+k)) / a is smooth in the sigma of the pixel
// it writes: g(k) = exp(-k^2 / s^2), s = sigma + 1e-6, dg/dsigma = g'(k) = g(k) 2 k^2 / s^3, and
//   dY(p)/dsigma(p) = sum_k g'(k) (X(clamp(p+k)) - Y(p)) / a.
// dest = V(H(S)) and each pass reads the sigma of the pixel it writes, so for a gradient G on the band
//   grad_sigma(q) = <G(q) / a(q),   sum_k g'(k) (T(x, clampy(y+k)) - D(q))>   (vertical pass, band rows)
//                 + <G_T(q) / a(q), sum_k g'(k) (S(clampx(x+k), y) - T(q))>   (horizontal pass, rows band +- R)
// with G / a what k_blur_adjoint_scale writes and G_T / a what k_blur_adjoint_vertical writes. Y is recomputed at the pixel
// with the forward's operations, so it has the forward's bits, and the difference X - Y is formed before the sum.

// one pass's term at pixel i: <factor, sum_k g'(k) (X(clamp(pos+k)) - Y)>, the line of X given by base + clamp(pos+k) * step
// for positions [0, n). A channel whose factor is 0 adds nothing, not even a NaN of the image; a pixel without taps gives 0.
__device__ __forceinline__ float sigma_term(const float4* __restrict__ image, float4 f, float sigma, size_t base, size_t step,
                                            int pos, int n) {
  const Taps t = taps_for(sigma);
  if (t.first > t.last || (f.x == 0.0f && f.y == 0.0f && f.z == 0.0f && f.w == 0.0f)) return 0.0f;
  float accum = 0.0f;
  float4 y = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (int k = t.first; k <= t.last; ++k) {
    const float g = tap_weight(k, t);
    const float4 s = image[base + (size_t)max(0, min(pos + k, n - 1)) * step];
    accum += g;
    y.x += s.x * g;
    y.y += s.y * g;
    y.z += s.z * g;
    y.w += s.w * g;
  }
  y = make_float4(y.x / accum, y.y / accum, y.z / accum, y.w / accum);
  const float c = 2.0f / (t.sig_square * (sigma + kMinSigma));  // 2 / s^3
  float4 d = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (int k = t.first; k <= t.last; ++k) {
    if (k == 0) continue;  // g'(0) = 0
    const float gp = tap_weight(k, t) * (float)(k * k) * c;
    const float4 s = image[base + (size_t)max(0, min(pos + k, n - 1)) * step];
    d.x += gp * (s.x - y.x);
    d.y += gp * (s.y - y.y);
    d.z += gp * (s.z - y.z);
    d.w += gp * (s.w - y.w);
  }
  return (f.x != 0.0f ? f.x * d.x : 0.0f) + (f.y != 0.0f ? f.y * d.y : 0.0f) + (f.z != 0.0f ? f.z * d.z : 0.0f) +
         (f.w != 0.0f ? f.w * d.w : 0.0f);
}

// VERTICAL: every row of grad_sigma is written, the band rows with the vertical term (factor = G / a, image = T), the others
// with 0. Otherwise rows [row_begin - R, row_end + R) add the horizontal term (factor = G_T / a, image = S). With an all-zero
// sigma map, 0 everywhere.
template <bool VERTICAL>
__global__ void k_blur_sigma_adjoint(const float4* __restrict__ factor, const float4* __restrict__ image,
                                     float* __restrict__ grad_sigma, const float* __restrict__ sigma, int width, int height,
                                     int row_begin, int row_end, const int* __restrict__ reach, const float* max_sigma) {
  const bool zero = all_sigma_zero(max_sigma);
  if (!VERTICAL && zero) return;
  const int r = VERTICAL ? 0 : *reach;
  const int lo_row = VERTICAL ? 0 : max(0, row_begin - r), hi_row = VERTICAL ? height : min(height, row_end + r);
  const size_t count = (size_t)width * (hi_row - lo_row), first = (size_t)lo_row * width;
  const size_t stride = (size_t)blockDim.x * gridDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
    const size_t i = first + j;
    const int x = (int)(i % width);
    const int y = (int)(i / width);
    if (VERTICAL) {
      grad_sigma[i] = zero || y < row_begin || y >= row_end ? 0.0f : sigma_term(image, factor[i], sigma[i], x, width, y, height);
    } else {
      grad_sigma[i] += sigma_term(image, factor[i], sigma[i], i - x, 1, x, width);
    }
  }
}

inline unsigned grid_for(size_t n) {
  const size_t blocks = (n + kThreads - 1) / kThreads;
  return (unsigned)(blocks < kMaxBlocks ? blocks : kMaxBlocks);
}

}  // namespace

// forces the blur kernels' module to load now (a later first launch would otherwise do it, and loading may have to
// wait for the device to go idle — not something to meet between two barrier kernels)
int blur_preload() {
  cudaFuncAttributes fa;
  RDC_CUDA(cudaFuncGetAttributes(&fa, k_blur_horizontal));
  RDC_CUDA(cudaFuncGetAttributes(&fa, k_blur_vertical));
  return 0;
}

int gaussian_blur(float4* dest, const float4* src, const float* sigma, float4* scratch, int width, int height,
                  int row_begin, int row_end, const float* max_sigma, cudaStream_t stream, int halo_rows) {
  if (!dest || !src || !sigma || !scratch || width <= 0 || height <= 0 || row_begin < 0 || row_end > height ||
      row_begin >= row_end) {
    set_error("blur: bad argument");
    return RDC_E_INVALID;
  }
  // rows the vertical pass of the band can read
  const int h_begin = halo_rows < 0 ? 0 : (row_begin - halo_rows > 0 ? row_begin - halo_rows : 0);
  const int h_end = halo_rows < 0 ? height : (row_end + halo_rows < height ? row_end + halo_rows : height);
  const size_t n_all = (size_t)width * (h_end - h_begin);
  const size_t n_band = (size_t)width * (row_end - row_begin);
  k_blur_horizontal<<<grid_for(n_all), kThreads, 0, stream>>>(src, scratch, dest, sigma, width, h_begin, h_end, max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_vertical<<<grid_for(n_band), kThreads, 0, stream>>>(scratch, dest, sigma, width, height, row_begin, row_end, max_sigma);
  RDC_CUDA(cudaGetLastError());
  return 0;
}

int gaussian_blur_adjoint(float4* grad_source, const float4* grad_dest, const float* sigma, float4* scratch, int width,
                          int height, int row_begin, int row_end, const float* max_sigma, cudaStream_t stream) {
  if (!grad_source || !grad_dest || !sigma || !scratch || width <= 0 || height <= 0 || row_begin < 0 || row_end > height ||
      row_begin >= row_end) {
    set_error("blur adjoint: bad argument");
    return RDC_E_INVALID;
  }
  const size_t n_all = (size_t)width * height;
  const size_t n_band = (size_t)width * (row_end - row_begin);
  int* reach = reinterpret_cast<int*>(scratch + n_all);
  RDC_CUDA(cudaMemsetAsync(reach, 0, sizeof(int), stream));
  k_blur_reach<<<grid_for(n_all), kThreads, 0, stream>>>(sigma, n_all, max_sigma, reach);
  RDC_CUDA(cudaGetLastError());
  k_blur_adjoint_scale<<<grid_for(n_band), kThreads, 0, stream>>>(grad_dest, grad_source, sigma, width, row_begin, row_end,
                                                                   max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_adjoint_vertical<<<grid_for(n_all), kThreads, 0, stream>>>(grad_source, scratch, sigma, width, height, row_begin,
                                                                    row_end, reach, max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_adjoint_horizontal<<<grid_for(n_all), kThreads, 0, stream>>>(scratch, grad_source, sigma, width, height, row_begin,
                                                                      row_end, reach, max_sigma);
  RDC_CUDA(cudaGetLastError());
  return 0;
}

// Scratch: T, then (once the vertical term has read it) G_T / a, in the first W*H float4; G / a of the band in the second;
// the reach after them.
int gaussian_blur_sigma_adjoint(float* grad_sigma, const float4* grad_dest, const float4* source, const float* sigma,
                                float4* scratch, int width, int height, int row_begin, int row_end, const float* max_sigma,
                                cudaStream_t stream) {
  if (!grad_sigma || !grad_dest || !source || !sigma || !scratch || width <= 0 || height <= 0 || row_begin < 0 ||
      row_end > height || row_begin >= row_end) {
    set_error("blur sigma adjoint: bad argument");
    return RDC_E_INVALID;
  }
  const size_t n_all = (size_t)width * height;
  const size_t n_band = (size_t)width * (row_end - row_begin);
  float4* pass = scratch;
  float4* scaled = scratch + n_all;
  int* reach = reinterpret_cast<int*>(scratch + 2 * n_all);
  RDC_CUDA(cudaMemsetAsync(reach, 0, sizeof(int), stream));
  k_blur_reach<<<grid_for(n_all), kThreads, 0, stream>>>(sigma, n_all, max_sigma, reach);
  RDC_CUDA(cudaGetLastError());
  k_blur_horizontal<<<grid_for(n_all), kThreads, 0, stream>>>(source, pass, pass, sigma, width, 0, height, max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_adjoint_scale<<<grid_for(n_band), kThreads, 0, stream>>>(grad_dest, scaled, sigma, width, row_begin, row_end,
                                                                   max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_sigma_adjoint<true><<<grid_for(n_all), kThreads, 0, stream>>>(scaled, pass, grad_sigma, sigma, width, height, row_begin,
                                                                       row_end, reach, max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_adjoint_vertical<<<grid_for(n_all), kThreads, 0, stream>>>(scaled, pass, sigma, width, height, row_begin, row_end,
                                                                    reach, max_sigma);
  RDC_CUDA(cudaGetLastError());
  k_blur_sigma_adjoint<false><<<grid_for(n_all), kThreads, 0, stream>>>(pass, source, grad_sigma, sigma, width, height,
                                                                        row_begin, row_end, reach, max_sigma);
  RDC_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace rdc
