// Augmented training-image preparation (reference dataset.py `_get_single_item` without depth): the pixel arithmetic of
// PIL's bilinear resize, `convert("L")`, torchvision's ColorJitter(brightness, contrast) through PIL's ImageEnhance,
// ToTensor + Normalize, and scikit-image's order-1 `rotate` (mode 'reflect', clip=True), bit for bit. The decode and
// every random draw stay on the loader workers; the host passes the drawn parameters and the coefficient tables.
//
//   imageprep_hpass_kernel  : horizontal PIL pass, uint8 -> uint8 intermediate [h_in, w_out, C]
//   imageprep_vpass_kernel  : vertical PIL pass + L; per-image sum of the first jitter operand, min / max of L
//   imageprep_finish_kernel : jitter + normalise + rotate + clip, fp16 store into the encoder's batch slot
//   imageprep_mask_cells_kernel : the rotated all-ones mask, evaluated only at the cells NEAREST-resizing picks
//
// Exactness notes: every float / double operation is written with an explicit _rn intrinsic (no FMA contraction); the
// contrast mean is an integer sum (exact with atomics), so the result does not depend on the reduction order.
#include <math.h>

#include "common.cuh"

namespace acez {

constexpr int kPrepMaxBatch = 8;   // images per launch (descriptors travel as kernel parameters)
constexpr int kPrepThreads = 256;

__host__ __device__ inline float f_mul(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
__host__ __device__ inline float f_add(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
__host__ __device__ inline float f_sub(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
__host__ __device__ inline float f_div(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}
__host__ __device__ inline double d_mul(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
__host__ __device__ inline double d_add(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
__host__ __device__ inline double d_sub(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}

// PIL ImagingResample, 8 bpc: 22 fraction bits, accumulator starts at one half, clip8 of the shifted sum.
__host__ __device__ inline int resize_sample(const uint8_t* p, long long stride, const int32_t* k, int count) {
  int acc = 1 << 21;
  for (int i = 0; i < count; ++i) acc += (int)p[i * stride] * k[i];
  const int v = acc >> 22;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

// PIL convert("RGB" -> "L"), ITU-R 601-2 luma in 16-bit fixed point.
__host__ __device__ inline int luma(int r, int g, int b) { return (19595 * r + 38470 * g + 7471 * b + 0x8000) >> 16; }

// PIL Image.blend(degenerate, image, alpha) for one L sample: float arithmetic, truncation, clamp when extrapolating
// (inside [0, 1] the clamp never applies, so one formula serves both branches).
__host__ __device__ inline int blend(int d, int v, float f) {
  const float t = f_add((float)d, f_mul(f, (float)(v - d)));
  if (t <= 0.f) return 0;
  if (t >= 255.f) return 255;
  return (int)t;
}

// ColorJitter in randperm order; `mean` is ImageEnhance.Contrast's degenerate value of the image it is applied to.
__host__ __device__ inline int jitter(int v, int contrast_first, float fb, float fc, int mean) {
  if (contrast_first) return blend(0, blend(mean, v, fc), fb);
  return blend(mean, blend(0, v, fb), fc);
}

// ToTensor + Normalize(mean 0.4, std 0.25) in fp32.
__host__ __device__ inline float normalize(int v) { return f_div(f_sub(f_div((float)v, 255.f), 0.4f), 0.25f); }

// scikit-image coord_map, mode 'reflect' (mirror about the edge pixel, which is not repeated).
__host__ __device__ inline long long reflect_index(long long dim, long long coord) {
  const long long cmax = dim - 1;
  if (cmax == 0) return 0;
  if (coord < 0) return (((-coord) / cmax) % 2 != 0) ? cmax - ((-coord) % cmax) : (-coord) % cmax;
  if (coord > cmax) return ((coord / cmax) % 2 != 0) ? cmax - (coord % cmax) : coord % cmax;
  return coord;
}

// Affine inverse map of one output pixel (x = column, y = row) to input (c, r), as skimage's _transform_affine.
__host__ __device__ inline void affine_map(const double* M, double x, double y, double& c, double& r) {
  c = d_add(d_add(d_mul(M[0], x), d_mul(M[1], y)), M[2]);
  r = d_add(d_add(d_mul(M[3], x), d_mul(M[4], y)), M[5]);
}

// One output sample of skimage's order-1 warp in mode 'reflect' (before the clip). `pix(row, col)` returns the input.
template <class Pix>
__host__ __device__ inline double rotate_sample(const double* M, int rows, int cols, int orow, int ocol, const Pix& pix) {
  double c, r;
  affine_map(M, (double)ocol, (double)orow, c, r);
  const long long minr = (long long)floor(r), minc = (long long)floor(c);
  const long long maxr = (long long)ceil(r), maxc = (long long)ceil(c);
  const double dr = d_sub(r, (double)minr), dc = d_sub(c, (double)minc);
  const long long r0 = reflect_index(rows, minr), r1 = reflect_index(rows, maxr);
  const long long c0 = reflect_index(cols, minc), c1 = reflect_index(cols, maxc);
  const double top = d_add(d_mul(d_sub(1.0, dc), pix(r0, c0)), d_mul(dc, pix(r0, c1)));
  const double bottom = d_add(d_mul(d_sub(1.0, dc), pix(r1, c0)), d_mul(dc, pix(r1, c1)));
  return d_add(d_mul(d_sub(1.0, dr), top), d_mul(dr, bottom));
}

// torch's nearest source index (upsample_nearest: `nearest_idx` with the float scale input / output).
__host__ __device__ inline int nearest_src(int o, int in, int out) {
  if (out == in) return o;
  if (out == 2 * in) return o >> 1;
  const float scale = f_div((float)in, (float)out);
  const int s = (int)floorf(f_mul((float)o, scale));
  return s < in - 1 ? s : in - 1;
}

// The reference's mask: ones(rows, cols) rotated in mode 'constant' (cval 0), kept where > 0, NEAREST-resized to
// (h8, w8). A sample is non-zero iff a tap of positive weight ({floor, ceil} of r and of c) lies inside the image.
__host__ __device__ inline int mask_cell(const double* M, int rows, int cols, int h8, int w8, int i, int j) {
  double c, r;
  affine_map(M, (double)nearest_src(j, cols, w8), (double)nearest_src(i, rows, h8), c, r);
  return r > -1.0 && r < (double)rows && c > -1.0 && c < (double)cols;
}

struct PrepStats {
  unsigned long long sum;   // sum of the first jitter operation's input to the contrast mean (see vpass)
  unsigned int max_l;       // max of L
  unsigned int inv_min_l;   // 255 - min of L (so that a zeroed slot is the identity of atomicMax)
};

struct PrepBatch {
  acez_image_prep_desc d[kPrepMaxBatch];
  uint8_t* tmp[kPrepMaxBatch];   // horizontal-pass output [h_in, w_out, C] (unused when w_in == w_out)
  uint8_t* lum[kPrepMaxBatch];   // L image [h_out, w_out]
  PrepStats* stats;              // [n]
  __half* out;                   // [n, 1, h_out, w_out]
  int n, h_out, w_out;
};

__global__ void __launch_bounds__(kPrepThreads) imageprep_hpass_kernel(const __grid_constant__ PrepBatch b) {
  const acez_image_prep_desc& d = b.d[blockIdx.z];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
  if (d.coef_x == nullptr || x >= b.w_out || row >= d.h_in) return;
  const int C = d.channels;
  const int32_t* k = d.coef_x + (long long)x * (2 + d.kx);
  const uint8_t* src = d.src + ((long long)row * d.w_in + k[0]) * C;
  uint8_t* dst = b.tmp[blockIdx.z] + ((long long)row * b.w_out + x) * C;
  for (int ch = 0; ch < C; ++ch) dst[ch] = (uint8_t)resize_sample(src + ch, C, k + 2, k[1]);
}

__global__ void __launch_bounds__(kPrepThreads) imageprep_vpass_kernel(const __grid_constant__ PrepBatch b) {
  const int img = blockIdx.z;
  const acez_image_prep_desc& d = b.d[img];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  const int C = d.channels;
  unsigned int s = 0, mx = 0, inv_mn = 0;
  if (x < b.w_out) {
    const uint8_t* h = d.coef_x ? b.tmp[img] : d.src;
    const long long stride = (long long)b.w_out * C;
    int v[3];
    if (d.coef_y) {
      const int32_t* k = d.coef_y + (long long)y * (2 + d.ky);
      const uint8_t* p = h + (long long)k[0] * stride + (long long)x * C;
      for (int ch = 0; ch < C; ++ch) v[ch] = resize_sample(p + ch, stride, k + 2, k[1]);
    } else {
      const uint8_t* p = h + (long long)y * stride + (long long)x * C;
      for (int ch = 0; ch < C; ++ch) v[ch] = p[ch];
    }
    const int L = C == 3 ? luma(v[0], v[1], v[2]) : v[0];
    b.lum[img][(long long)y * b.w_out + x] = (uint8_t)L;
    // the contrast mean is taken over the image the contrast step sees: L, or L after brightness
    s = (unsigned int)(d.contrast_first ? L : blend(0, L, d.brightness));
    mx = (unsigned int)L;
    inv_mn = 255u - (unsigned int)L;
  }
  unsigned long long s64 = s;
  for (int o = 16; o > 0; o >>= 1) {
    s64 += __shfl_xor_sync(0xffffffffu, s64, o);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    inv_mn = max(inv_mn, __shfl_xor_sync(0xffffffffu, inv_mn, o));
  }
  if ((threadIdx.x & 31) == 0 && blockIdx.x * blockDim.x + threadIdx.x < (unsigned)b.w_out) {
    PrepStats* st = b.stats + img;
    atomicAdd(&st->sum, s64);
    atomicMax(&st->max_l, mx);
    atomicMax(&st->inv_min_l, inv_mn);
  }
}

__global__ void __launch_bounds__(kPrepThreads) imageprep_finish_kernel(const __grid_constant__ PrepBatch b) {
  const int img = blockIdx.z;
  const acez_image_prep_desc& d = b.d[img];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= b.w_out) return;
  const PrepStats st = b.stats[img];
  // ImageEnhance.Contrast: int(ImageStat mean + 0.5), the mean in double
  const int mean = (int)d_add(__ddiv_rn((double)st.sum, (double)b.h_out * (double)b.w_out), 0.5);
  const uint8_t* lum = b.lum[img];
  const int cf = d.contrast_first;
  const float fb = d.brightness, fc = d.contrast;
  __half* out = b.out + (long long)img * b.h_out * b.w_out;
  if (!d.rotate) {
    out[(long long)y * b.w_out + x] = __float2half_rn(normalize(jitter(lum[(long long)y * b.w_out + x], cf, fb, fc, mean)));
    return;
  }
  const int w = b.w_out;
  auto pix = [&](long long r, long long c) { return (double)normalize(jitter(lum[r * w + c], cf, fb, fc, mean)); };
  double v = rotate_sample(d.affine, b.h_out, b.w_out, y, x, pix);
  // clip=True: the input's [min, max]; jitter and normalisation are monotonic, so they are those of L
  const double lo = (double)normalize(jitter(255 - (int)st.inv_min_l, cf, fb, fc, mean));
  const double hi = (double)normalize(jitter((int)st.max_l, cf, fb, fc, mean));
  v = fmin(fmax(v, lo), hi);
  out[(long long)y * w + x] = __float2half_rn(__double2float_rn(v));
}

struct MaskArgs {
  double M[6];
  int rows, cols, h8, w8;
  float* cells;
};

__global__ void __launch_bounds__(kPrepThreads) imageprep_mask_cells_kernel(const __grid_constant__ MaskArgs a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.h8 * a.w8) return;
  a.cells[t] = mask_cell(a.M, a.rows, a.cols, a.h8, a.w8, t / a.w8, t % a.w8) ? 1.f : 0.f;
}

// workspace: [n PrepStats, 256-aligned] then per image [L h_out*w_out][horizontal intermediate h_in*w_out*C], each
// 256-aligned
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

size_t prep_workspace(const acez_image_prep_desc* d, int n, int h_out, int w_out, size_t* lum_off, size_t* tmp_off) {
  size_t off = align256((size_t)n * sizeof(PrepStats));
  for (int i = 0; i < n; ++i) {
    if (lum_off) lum_off[i] = off;
    off += align256((size_t)h_out * w_out);
    if (tmp_off) tmp_off[i] = off;
    if (d[i].coef_x) off += align256((size_t)d[i].h_in * w_out * d[i].channels);
  }
  return off;
}

}  // namespace acez

extern "C" size_t acez_image_prep_workspace_bytes(const acez_image_prep_desc* descs, int n, int h_out, int w_out) {
  if (!descs || n <= 0 || h_out <= 0 || w_out <= 0) return 0;
  return acez::prep_workspace(descs, n, h_out, w_out, nullptr, nullptr);
}

extern "C" int acez_image_prep(const acez_image_prep_desc* descs, int n, int h_out, int w_out, void* workspace,
                               size_t workspace_bytes, void* out_f16, acez_stream_t stream) {
  using namespace acez;
  ACEZ_REQUIRE(descs && workspace && out_f16 && n > 0 && h_out > 0 && w_out > 0, "image_prep: bad arguments");
  for (int i = 0; i < n; ++i) {
    const acez_image_prep_desc& d = descs[i];
    ACEZ_REQUIRE(d.src && d.h_in > 0 && d.w_in > 0 && (d.channels == 1 || d.channels == 3),
                 "image_prep: image %d: bad source", i);
    ACEZ_REQUIRE((d.coef_x == nullptr) == (d.w_in == w_out) && (d.coef_y == nullptr) == (d.h_in == h_out),
                 "image_prep: image %d: a coefficient table is required exactly when that dimension is resized", i);
    ACEZ_REQUIRE((!d.coef_x || d.kx > 0) && (!d.coef_y || d.ky > 0), "image_prep: image %d: bad table width", i);
  }
  size_t lum_off[4096 / sizeof(size_t)], tmp_off[4096 / sizeof(size_t)];
  ACEZ_REQUIRE(n <= (int)(sizeof(lum_off) / sizeof(lum_off[0])), "image_prep: too many images (%d)", n);
  const size_t need = prep_workspace(descs, n, h_out, w_out, lum_off, tmp_off);
  ACEZ_REQUIRE(workspace_bytes >= need, "image_prep: workspace %zu < %zu bytes", workspace_bytes, need);
  int rc = acez_device_check();
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  ACEZ_CUDA(cudaMemsetAsync(ws, 0, (size_t)n * sizeof(PrepStats), s));
  for (int i0 = 0; i0 < n; i0 += kPrepMaxBatch) {
    PrepBatch b{};
    b.n = n - i0 < kPrepMaxBatch ? n - i0 : kPrepMaxBatch;
    b.h_out = h_out; b.w_out = w_out;
    b.stats = reinterpret_cast<PrepStats*>(ws) + i0;
    b.out = reinterpret_cast<__half*>(out_f16) + (size_t)i0 * h_out * w_out;
    int max_h_in = 0;
    bool any_h = false;
    for (int k = 0; k < b.n; ++k) {
      b.d[k] = descs[i0 + k];
      b.lum[k] = ws + lum_off[i0 + k];
      b.tmp[k] = ws + tmp_off[i0 + k];
      if (b.d[k].coef_x) { any_h = true; max_h_in = b.d[k].h_in > max_h_in ? b.d[k].h_in : max_h_in; }
    }
    const dim3 block(kPrepThreads);
    if (any_h) {
      imageprep_hpass_kernel<<<dim3((w_out + kPrepThreads - 1) / kPrepThreads, max_h_in, b.n), block, 0, s>>>(b);
      ACEZ_CUDA(cudaGetLastError());
    }
    const dim3 grid((w_out + kPrepThreads - 1) / kPrepThreads, h_out, b.n);
    imageprep_vpass_kernel<<<grid, block, 0, s>>>(b);
    ACEZ_CUDA(cudaGetLastError());
    imageprep_finish_kernel<<<grid, block, 0, s>>>(b);
    ACEZ_CUDA(cudaGetLastError());
  }
  return ACEZ_OK;
}

extern "C" int acez_image_mask_cells(const double* affine6, int h, int w, int h8, int w8, float* cells,
                                     acez_stream_t stream) {
  using namespace acez;
  ACEZ_REQUIRE(affine6 && cells && h > 0 && w > 0 && h8 > 0 && w8 > 0 && h8 <= h && w8 <= w,
               "image_mask_cells: bad arguments");
  int rc = acez_device_check();
  if (rc) return rc;
  MaskArgs a{};
  for (int k = 0; k < 6; ++k) a.M[k] = affine6[k];
  a.rows = h; a.cols = w; a.h8 = h8; a.w8 = w8; a.cells = cells;
  const int cells_n = h8 * w8;
  imageprep_mask_cells_kernel<<<(cells_n + kPrepThreads - 1) / kPrepThreads, kPrepThreads, 0,
                                reinterpret_cast<cudaStream_t>(stream)>>>(a);
  ACEZ_CUDA(cudaGetLastError());
  return ACEZ_OK;
}

// ----------------------------------------------------------------------------------------------
// host-callable views of the per-pixel arithmetic (CPU unit tests pin it against PIL / torchvision / the oracle)
// ----------------------------------------------------------------------------------------------
extern "C" int acez_host_resize_sample(const uint8_t* p, long long stride, const int32_t* k, int count) {
  return acez::resize_sample(p, stride, k, count);
}
extern "C" int acez_host_luma(int r, int g, int b) { return acez::luma(r, g, b); }
extern "C" int acez_host_jitter(int v, int contrast_first, float brightness, float contrast, int mean) {
  return acez::jitter(v, contrast_first, brightness, contrast, mean);
}
extern "C" float acez_host_normalize(int v) { return acez::normalize(v); }
// unclipped order-1 'reflect' sample of a float image [rows, cols] at output pixel (orow, ocol)
extern "C" double acez_host_rotate_sample(const double* affine6, const float* img, int rows, int cols, int orow, int ocol) {
  auto pix = [&](long long r, long long c) { return (double)img[r * cols + c]; };
  return acez::rotate_sample(affine6, rows, cols, orow, ocol, pix);
}
extern "C" int acez_host_mask_cell(const double* affine6, int rows, int cols, int h8, int w8, int i, int j) {
  return acez::mask_cell(affine6, rows, cols, h8, w8, i, j);
}
