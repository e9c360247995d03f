// pool.cuh -- change-based 2x2 / stride-2 max pooling.
//
// Replaces maxPool2d_kernel (reference cbconv2d_cg_backend.cu:199-227, half :207-237): for each
// changed *input* pixel recompute its window maximum over all channels (init -inf, window clipped
// to the input) into the persistent pooled map.  One warp per changed pixel, lanes over channels
// (contiguous for the pixel-major layout).  When the change bitmap is supplied each window is
// recomputed once (by its first changed pixel) instead of up to four times; windows whose output
// coordinate is outside [oH,oW) are skipped (the reference writes out of bounds there).
// Traffic per distinct window: 4*C*s read + C*s written.
#pragma once
#include "cb_common.cuh"
#include "detect.cuh"

namespace cb {

__device__ __forceinline__ bool bit_at(const uint32_t* bits, long long row, int Wd, int x) {
  return (__ldg(bits + row * Wd + (x >> 5)) >> (x & 31)) & 1u;
}

template <typename T> __device__ __forceinline__ T neg_inf();
template <> __device__ __forceinline__ float neg_inf<float>() { return -INFINITY; }
template <> __device__ __forceinline__ __half neg_inf<__half>() { return __ushort_as_half(0xFC00); }
template <> __device__ __forceinline__ __nv_bfloat16 neg_inf<__nv_bfloat16>() {
  return __ushort_as_bfloat16(0xFF80);
}
__device__ __forceinline__ float max_keep(float v, float u) { return fmaxf(v, u); }   // cg.cu:220
__device__ __forceinline__ __half max_keep(__half v, __half u) { return __hgt(u, v) ? u : v; }  // half.cu:229
__device__ __forceinline__ __nv_bfloat16 max_keep(__nv_bfloat16 v, __nv_bfloat16 u) {
  return __hgt(u, v) ? u : v;
}

// The first changed pixel of a 2x2 window (in row-major order) owns it: only the owner recomputes the
// window.  (b, y, xx) is a changed pixel of the dilated bitmap `bits`.
__device__ __forceinline__ bool window_owner(const uint32_t* bits, int b, int y, int xx, int H, int W, int Wd) {
  const long long r = (long long)b * H + y;
  bool owner = true;
  if (xx & 1) owner = !bit_at(bits, r, Wd, xx - 1);
  if (owner && (y & 1)) {
    const int xe = xx & ~1;
    owner = !bit_at(bits, r - 1, Wd, xe) && !(xe + 1 < W && bit_at(bits, r - 1, Wd, xe + 1));
  }
  return owner;
}

// Element-wise maximum of the four 16-byte chunks of a 2x2 window
template <typename T, int VEC>
__device__ __forceinline__ uint4 window_max16(const uint4& v00, const uint4& v01, const uint4& v10, const uint4& v11) {
  uint4 res;
  const T* e00 = reinterpret_cast<const T*>(&v00);
  const T* e01 = reinterpret_cast<const T*>(&v01);
  const T* e10 = reinterpret_cast<const T*>(&v10);
  const T* e11 = reinterpret_cast<const T*>(&v11);
  T* er = reinterpret_cast<T*>(&res);
#pragma unroll
  for (int e = 0; e < VEC; ++e) {
    T v = max_keep(neg_inf<T>(), e00[e]);
    v = max_keep(v, e01[e]);
    v = max_keep(v, e10[e]);
    v = max_keep(v, e11[e]);
    er[e] = v;
  }
  return res;
}

template <typename T>
__global__ void __launch_bounds__(256)
maxpool2x2_kernel(const T* __restrict__ x, long long x_sb, long long x_sc, long long x_sy,
                  long long x_sx, const int32_t* __restrict__ idx,
                  const int32_t* __restrict__ count, const uint32_t* __restrict__ bits,
                  T* __restrict__ out, long long o_sb, long long o_sc, long long o_sy,
                  long long o_sx, int C, int H, int W, int oH, int oW) {
  const int n = *count;
  const int lane = threadIdx.x & 31;
  const int P = H * W, Wd = (W + 31) >> 5;
  const int wstride = gridDim.x * (blockDim.x >> 5);
  for (int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < n; j += wstride) {
    const int pix = idx[j];
    const int b = pix / P, p = pix - b * P;
    const int y = p / W, xx = p - y * W;
    const int yo = y >> 1, xo = xx >> 1;
    if (yo >= oH || xo >= oW) continue;
    if (bits && !window_owner(bits, b, y, xx, H, W, Wd)) continue;
    const int y0 = yo * 2, x0 = xo * 2;
    const bool hy = y0 + 1 < H, hx = x0 + 1 < W;
    const T* base = x + b * x_sb + y0 * x_sy + x0 * x_sx;
    T* o = out + b * o_sb + yo * o_sy + xo * o_sx;
    for (int c = lane; c < C; c += 32) {
      const T* q = base + c * x_sc;
      T v = neg_inf<T>();
      v = max_keep(v, q[0]);
      if (hx) v = max_keep(v, q[x_sx]);
      if (hy) {
        v = max_keep(v, q[x_sy]);
        if (hx) v = max_keep(v, q[x_sy + x_sx]);
      }
      o[c * o_sc] = v;
    }
  }
}

// Pixel-major 2x2 pooling: a group of G lanes (G = 1 << glog, see group_log2) owns one changed pixel,
// so a warp works on 32/G list entries at once with 16-byte loads/stores; the four window pixels are 4
// independent vector loads per lane.
// DETECT: pool + downstream change detection in one pass: the lane group that recomputes a pooled
// pixel still holds its new channel values, so it thresholds them against the NEXT layer's
// previous-input state right away, ORs the change bit into that layer's (pre-cleared) raw bitmap and
// maintains its state / operand planes.  Replaces three launches of the candidate path (pool, pooled
// compaction, sparse detection) and is exact for the same reason candidate detection is: only
// re-pooled pixels can differ from what the next layer saw last frame.  Without DETECT the next-layer
// arguments and UPDATE are unused, and `bits` may be null (then every listed pixel recomputes its
// window).  THR (with DETECT): thr_b holds the next layer's per-stream thresholds, fp32 [B], one load
// per window.
template <typename T, int VEC, int UPDATE, bool DETECT = true, bool THR = false>
__global__ void __launch_bounds__(256)
maxpool2x2_detect_kernel(const T* __restrict__ x, long long x_sb, long long x_sy, int xp,
                         const int32_t* __restrict__ idx, const int32_t* __restrict__ count,
                         const uint32_t* __restrict__ bits, T* __restrict__ out, long long o_sb,
                         long long o_sy, int op, int cpp, int glog, int H, int W, int oH, int oW,
                         T* __restrict__ nst, long long n_sb, long long n_sy, int np, AuxPlanes aux,
                         uint32_t* __restrict__ nbits, T thr, const float* __restrict__ thr_b) {
  const int n = *count;
  const int lane = threadIdx.x & 31;
  const int G = 1 << glog, ppw = 32 >> glog;                // lanes per pixel, pixels per warp
  const int sub = lane >> glog, gl = lane & (G - 1);
  const unsigned gmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (sub * G);
  const int P = H * W, Wd = (W + 31) >> 5, oWd = (oW + 31) >> 5;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long j0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * ppw;
       j0 < n; j0 += nwarps * ppw) {
    const long long j = j0 + sub;
    bool work = j < n;
    int b = 0, yo = 0, xo = 0;
    if (work) {
      const int pix = __ldg(idx + j);
      b = pix / P;
      const int p = pix - b * P;
      const int y = p / W, xx = p - y * W;
      yo = y >> 1;
      xo = xx >> 1;
      work = yo < oH && xo < oW && (!(DETECT || bits) || window_owner(bits, b, y, xx, H, W, Wd));
    }
    if (!DETECT && !work) continue;            // (lanes with nothing to pool wait at no ballot)
    const int y0 = yo * 2, x0 = xo * 2;
    const bool hy = y0 + 1 < H, hx = x0 + 1 < W;
    const T* base = x + b * x_sb + y0 * x_sy + (long long)x0 * xp;
    T* o = out + b * o_sb + yo * o_sy + (long long)xo * op;
    T* ns = nst + b * n_sb + yo * n_sy + (long long)xo * np;
    const long long opix = ((long long)b * oH + yo) * oW + xo;
    bool f = false;
    if (work) {
      const T tb = stream_thr<DETECT && THR>(thr_b, b, thr);
      for (int cc = gl; cc < cpp; cc += G) {
        const T* q = base + cc * VEC;
        uint4 v00 = ldg16(q), v01 = v00, v10 = v00, v11 = v00;
        if (hx) v01 = ldg16(q + xp);
        if (hy) {
          v10 = ldg16(q + x_sy);
          v11 = hx ? ldg16(q + x_sy + xp) : v10;
        }
        const uint4 sv = DETECT ? ld16(ns + cc * VEC) : uint4{};   // in flight with the window loads
        const uint4 res = window_max16<T, VEC>(v00, v01, v10, v11);
        st16(o + cc * VEC, res);
        if (DETECT) {
          f |= Chunk<T>::changed(sv, res, tb);
          if (UPDATE == CB_UPDATE_ALL) store_state<T>(ns + cc * VEC, res, aux, opix, cc * VEC);
        }
      }
    }
    if (!DETECT) continue;
    const bool chg = (__ballot_sync(0xffffffffu, f) & gmask) != 0u;
    if (work && chg) {
      if (gl == 0) atomicOr(nbits + ((long long)b * oH + yo) * oWd + (xo >> 5), 1u << (xo & 31));
      if (UPDATE == CB_UPDATE_CHANGED)          // feedback: accept the new pooled pixel
        for (int cc = gl; cc < cpp; cc += G)
          store_state<T>(ns + cc * VEC, ld16(o + cc * VEC), aux, opix, cc * VEC);
    }
  }
}

}  // namespace cb
