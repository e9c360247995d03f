// ingest.cuh -- frame ingest before the first layer (SURVEY section 8f rank 4): the image resizing the
// reference's readers run on the host, on the GPU, so a decoder's uint8 surface goes resize -> first-layer
// change detection (cb_change_detect_u8 normalises on the fly) without touching the host.
//
//   * resize_bicubic_u8: PIL.Image.resize(size, BICUBIC) on 8-bit images -- what
//     torchvision.transforms.Scale(boxsize, interpolation=3) does in PoseDetector.preprocess
//     (poseDetection/openPose/PoseDetector.py:67).  Pillow's Resample.c, restated: separable, horizontal
//     pass first; per output coordinate a window [xmin, xmin + n) and n fixed-point weights (22 fractional
//     bits, computed in double on the host exactly as precompute_coeffs / normalize_coeffs_8bpc do);
//     accumulator = 1 << 21 + sum(pixel * weight), arithmetic shift by 22, saturate to 0..255; the
//     horizontally resized image is stored as 8-bit before the vertical pass.  BIT-EXACT against Pillow
//     (tests/test_ingest.py, tests/golden/ingest_golden.npz).
//   * resize_bilinear: skimage.transform.resize(img, shape, mode='constant') (order 1, clip) of
//     sceneLabeling/videoSequenceReader.py:64-67 applied to the uint8 frame / divisor: source coordinate
//     scale * (i + 0.5) - 0.5, four neighbours with constant padding, float64 arithmetic, fp32 result
//     written planar (the NCHW tensor the reader builds with permute(2,0,1).unsqueeze(0).float()).
//
// Byte / integer work, bound by HBM bytes (in + 2 x intermediate + out); images are a few MB.
#pragma once
#include "cb_common.cuh"

namespace cb {

constexpr int kResizePrecision = 32 - 8 - 2;                 // Pillow: PRECISION_BITS

// workspace layout (int32 words): [0] ksize_x [1] ksize_y [2] sH [3] sW [4] dH [5] dW [6] C [7] pad,
// bounds_x[2*dW], kk_x[dW*ksize_x], bounds_y[2*dH], kk_y[dH*ksize_y], then the uint8 intermediate sH*dW*C
struct ResizePlan {
  int ksize_x, ksize_y;
  size_t off_bx, off_kx, off_by, off_ky, off_tmp, bytes;    // byte offsets
};

inline int resize_ksize(int in_size, int out_size) {
  double scale = (double)in_size / out_size;
  if (scale < 1.0) scale = 1.0;
  return (int)ceil(2.0 * scale) * 2 + 1;
}

inline ResizePlan resize_plan(int sH, int sW, int dH, int dW, int C) {
  ResizePlan p;
  p.ksize_x = resize_ksize(sW, dW);
  p.ksize_y = resize_ksize(sH, dH);
  size_t o = 8 * sizeof(int32_t);
  p.off_bx = o; o += (size_t)2 * dW * 4;
  p.off_kx = o; o += (size_t)dW * p.ksize_x * 4;
  p.off_by = o; o += (size_t)2 * dH * 4;
  p.off_ky = o; o += (size_t)dH * p.ksize_y * 4;
  o = (o + 15) / 16 * 16;
  p.off_tmp = o; o += (size_t)sH * dW * C;
  p.bytes = (o + 15) / 16 * 16;
  return p;
}

inline double bicubic_filter(double x) {                    // Resample.c: bicubic_filter, a = -0.5
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

// Resample.c: precompute_coeffs (full box) + normalize_coeffs_8bpc
inline void resize_coeffs(int in_size, int out_size, int ksize, int32_t* bounds, int32_t* kk) {
  const double scale = (double)in_size / out_size;
  const double filterscale = scale < 1.0 ? 1.0 : scale;
  const double support = 2.0 * filterscale, ss = 1.0 / filterscale;
  double* w = new double[ksize];
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    double ww = 0.0;
    for (int x = 0; x < xmax; ++x) {
      w[x] = bicubic_filter((x + xmin - center + 0.5) * ss);
      ww += w[x];
    }
    int32_t* k = kk + (size_t)xx * ksize;
    for (int x = 0; x < ksize; ++x) {
      double v = 0.0;
      if (x < xmax) v = ww != 0.0 ? w[x] / ww : w[x];
      k[x] = v < 0 ? (int32_t)(-0.5 + v * (1 << kResizePrecision)) : (int32_t)(0.5 + v * (1 << kResizePrecision));
    }
    bounds[2 * xx] = xmin;
    bounds[2 * xx + 1] = xmax;
  }
  delete[] w;
}

__device__ __forceinline__ uint8_t resize_clip8(int v) {
  v >>= kResizePrecision;                                    // arithmetic shift, as Pillow's clip8 lookup
  return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v);
}

// One 8bpc pass along `axis` (0 = rows/y, 1 = columns/x).  Source and destination are addressed with byte
// strides (s_y, s_x, s_c), so HWC, planar and pitched surfaces all work.  One thread per output pixel,
// all channels (C <= 4); threads run along x, so both passes read and write coalesced rows.
template <int AXIS>
__global__ void __launch_bounds__(256)
resize_pass_u8_kernel(const uint8_t* __restrict__ src, long long s_y, long long s_x, long long s_c,
                      uint8_t* __restrict__ dst, long long d_y, long long d_x, long long d_c, int oH, int oW,
                      int C, const int32_t* __restrict__ bounds, const int32_t* __restrict__ kk, int ksize) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= oW || y >= oH) return;
  const int o = AXIS == 1 ? x : y;
  const int lo = __ldg(bounds + 2 * o), n = __ldg(bounds + 2 * o + 1);
  const int32_t* k = kk + (size_t)o * ksize;
  int acc[4] = {1 << (kResizePrecision - 1), 1 << (kResizePrecision - 1), 1 << (kResizePrecision - 1),
                1 << (kResizePrecision - 1)};
  const uint8_t* p = AXIS == 1 ? src + y * s_y + (long long)lo * s_x : src + (long long)lo * s_y + x * s_x;
  const long long step = AXIS == 1 ? s_x : s_y;
  for (int i = 0; i < n; ++i, p += step) {
    const int w = __ldg(k + i);
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (c < C) acc[c] += (int)p[c * s_c] * w;
  }
  uint8_t* q = dst + y * d_y + x * d_x;
#pragma unroll
  for (int c = 0; c < 4; ++c)
    if (c < C) q[c * d_c] = resize_clip8(acc[c]);
}

// skimage bilinear resize of a uint8 frame / divisor (float64 arithmetic), fp32 output with element strides
__global__ void __launch_bounds__(256)
resize_bilinear_kernel(const uint8_t* __restrict__ src, long long s_y, long long s_x, long long s_c, int sH,
                       int sW, float* __restrict__ dst, long long d_y, long long d_x, long long d_c, int oH,
                       int oW, int C, double divisor, double cval, double clip_lo, double clip_hi) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= oW || y >= oH) return;
  const double r = ((double)sH / oH) * (y + 0.5) - 0.5, c = ((double)sW / oW) * (x + 0.5) - 0.5;
  const double fr = floor(r), fc = floor(c);
  const int minr = (int)fr, minc = (int)fc, maxr = (int)ceil(r), maxc = (int)ceil(c);
  const double dr = r - fr, dc = c - fc;
  for (int ch = 0; ch < C; ++ch) {
    auto get = [&](int rr, int cc) -> double {
      if (rr < 0 || rr >= sH || cc < 0 || cc >= sW) return cval;
      return (double)src[rr * s_y + cc * s_x + ch * s_c] / divisor;
    };
    const double top = (1 - dc) * get(minr, minc) + dc * get(minr, maxc);
    const double bottom = (1 - dc) * get(maxr, minc) + dc * get(maxr, maxc);
    double v = (1 - dr) * top + dr * bottom;
    v = v < clip_lo ? clip_lo : v > clip_hi ? clip_hi : v;
    dst[y * d_y + x * d_x + ch * d_c] = (float)v;
  }
}

}  // namespace cb
