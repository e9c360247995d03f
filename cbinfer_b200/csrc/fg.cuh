// fg.cuh -- fine-grained change-based convolution (fp32, planar layout as in the reference).
//
// Replaces changeDetectionFG_kernel (reference cbconv2d_fg_backend.cu:7-23), the per-value
// torch.nonzero (conv2d_fg.py:82) and updateOutputFG_kernel (cbconv2d_fg_backend.cu:37-66),
// fused into one pass: a warp scans 32 input values, ballots the changed ones, then the whole
// warp cooperates on each changed value -- lanes spread over (co, ky, kx) -- and pushes
// W[co,ci,ky,kx]*d into the output with fire-and-forget red.global.add.f32.  The per-value mask
// uses the CUDA reference's strict '>' with flush-to-zero.  prev <- x afterwards (conv2d.py:175).
#pragma once
#include "cb_common.cuh"
#include "detect.cuh"

namespace cb {

__global__ void __launch_bounds__(256)
fg_update_kernel(const float* __restrict__ x, float* __restrict__ prev,
                 const float* __restrict__ w, float* __restrict__ out, int32_t* __restrict__ count,
                 int B, int Cin, int Cout, int H, int W, int kH, int kW, float thr) {
  const int lane = threadIdx.x & 31;
  const long long total = (long long)B * Cin * H * W;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  const int taps = kH * kW, work = Cout * taps;
  const long long HW = (long long)H * W;
  for (long long base = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32;
       base < total; base += nwarps * 32) {
    const long long i = base + lane;
    float d = 0.f;
    bool m = false;
    if (i < total) {
      const float xv = x[i], pv = prev[i];
      asm("sub.ftz.f32 %0, %1, %2;" : "=f"(d) : "f"(xv), "f"(pv));
      m = value_changed(xv, pv, thr);
      prev[i] = xv;
    }
    unsigned bal = __ballot_sync(0xffffffffu, m);
    if (lane == 0 && bal) atomicAdd(count, __popc(bal));
    while (bal) {
      const int src = __ffs(bal) - 1;
      bal &= bal - 1;
      const float dd = __shfl_sync(0xffffffffu, d, src);
      const long long pos = base + src;
      const int xx = (int)(pos % W);
      const int y = (int)((pos / W) % H);
      const int ci = (int)((pos / HW) % Cin);
      const int b = (int)(pos / (HW * Cin));
      float* ob = out + (long long)b * Cout * HW;
      for (int t = lane; t < work; t += 32) {
        const int co = t / taps, tap = t - co * taps;
        const int ky = tap / kW, kx = tap - ky * kW;
        const int yt = y - ky + kH / 2, xt = xx - kx + kW / 2;
        if (yt >= 0 && yt < H && xt >= 0 && xt < W)
          atomicAdd(ob + ((long long)co * H + yt) * W + xt,
                    __ldg(w + (((long long)co * Cin + ci) * kH + ky) * kW + kx) * dd);
      }
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Fine-grained update on the tensor cores (cb_fg_detect + cb_conv_accumulate).
//
// sum over changed values of W[co,ci,ky,kx] * d  ==  conv(D, W) with D = the thresholded delta map
// (d where |d| > thr, 0 elsewhere): the per-value scatter of updateOutputFG_kernel
// (cbconv2d_fg_backend.cu:37-66) is a convolution of a sparse map, and only output pixels within the
// filter footprint of a changed value receive anything.  fg_detect_kernel writes D as bf16 hi/lo
// operand planes (pixel-major, the layout the contraction gathers from) together with the raw pixel
// bitmap; the ordinary dilation/compaction lists the touched output pixels and the tcgen05 contraction
// runs over them with an accumulating epilogue (out += D * W, no bias).  Replaces one atomic per
// (changed value, tap, output channel) by dense MMA work over the touched pixels: scene layer 16->64
// 7x7 at 5 % change 9.98 ms -> the cost of the coarse-grained update plus one pass over the map.
//   XPM = 1: x is pixel-major like the state (16-byte chunks);  0: planar rows (transposed through
//   shared memory as in detect_planar_kernel).
// ------------------------------------------------------------------------------------------------
template <int XPM>
__global__ void __launch_bounds__(256)
fg_detect_kernel(const float* __restrict__ x, long long x_sb, long long x_sc, long long x_sy,
                 long long x_sx, float* __restrict__ prev, long long p_sb, long long p_sy, int pp,
                 __nv_bfloat16* __restrict__ dhi, __nv_bfloat16* __restrict__ dlo, int pitch16,
                 uint32_t* __restrict__ bits, int32_t* __restrict__ count, int B, int H, int W, int C,
                 int Wd, float thr, unsigned cpv_magic, int cps, int nw) {
  extern __shared__ __align__(16) unsigned char fg_smem[];
  uint4* xs = reinterpret_cast<uint4*>(fg_smem);                 // [nw*32][cps]
  __shared__ unsigned s_word[kPlanarMaxWords];
  __shared__ PlanarWord wi[kPlanarMaxWords];
  const int lane = threadIdx.x & 31;
  const long long nwords = (long long)B * H * Wd;
  const int word0 = blockIdx.x * nw;
  planar_words_setup(wi, s_word, word0, nw, nwords, H, W, Wd, x_sb, x_sy, x_sx, p_sb, p_sy, pp);
  const int cpv = (C + 3) / 4, tail = C % 4;
  const int nq = nw * 32 * cpv;
  if (XPM) {
    for (int q = threadIdx.x; q < nq; q += 256) {
      const int t = cpv == 1 ? q : (int)__umulhi((unsigned)q, cpv_magic), cc = q - t * cpv;
      const int w = t >> 5, px = t & 31;
      if (px < wi[w].npx) xs[t * cps + cc] = ldg16(x + wi[w].xoff + (long long)px * x_sx + cc * 4);
    }
  } else {
    planar_load_tile<float, 4>(xs, wi, x, x_sc, x_sx, nw, cpv, cps, C, cpv_magic);
  }
  __syncthreads();
  int nchg = 0;
  for (int q0 = 0; q0 < nq; q0 += 256) {
    const int q = min(q0 + (int)threadIdx.x, nq - 1);
    const bool in = q0 + (int)threadIdx.x < nq;
    const int t = cpv == 1 ? q : (int)__umulhi((unsigned)q, cpv_magic), cc = q - t * cpv;
    const int w = t >> 5, px = t & 31;
    unsigned m = 0u;
    if (in && px < wi[w].npx) {
      uint4 xv = xs[t * cps + cc];
      float* pptr = prev + wi[w].soff + (long long)px * pp + cc * 4;
      const uint4 pv = ld16(pptr);
      if (tail && cc == cpv - 1) xv = merge_tail<float, 4>(xv, pv, tail);
      const float xe[4] = {__uint_as_float(xv.x), __uint_as_float(xv.y), __uint_as_float(xv.z),
                           __uint_as_float(xv.w)};
      const float pe[4] = {__uint_as_float(pv.x), __uint_as_float(pv.y), __uint_as_float(pv.z),
                           __uint_as_float(pv.w)};
      __nv_bfloat16 h[4], l[4];
      bool any = false;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float d;
        asm("sub.ftz.f32 %0, %1, %2;" : "=f"(d) : "f"(xe[e]), "f"(pe[e]));   // cbconv2d_fg_backend.cu:19
        const bool chg = value_changed(xe[e], pe[e], thr);                    // fabs(d) > thr, :20
        any |= chg;
        nchg += chg ? 1 : 0;
        bf16_split(chg ? d : 0.f, h[e], l[e]);
      }
      const long long o = (wi[w].pix + px) * pitch16 + cc * 4;
      *reinterpret_cast<uint2*>(dhi + o) = *reinterpret_cast<uint2*>(h);
      *reinterpret_cast<uint2*>(dlo + o) = *reinterpret_cast<uint2*>(l);
      st16(pptr, xv);                                                         // prevInput = input (conv2d.py:175)
      if (any) m = 1u << px;
    }
    planar_flag(s_word, w, m);
  }
  nchg = __reduce_add_sync(0xffffffffu, nchg);
  if (lane == 0 && nchg && count) atomicAdd(count, nchg);
  __syncthreads();
  if (threadIdx.x < (unsigned)nw && wi[threadIdx.x].npx > 0) bits[word0 + threadIdx.x] = s_word[threadIdx.x];
}

inline int launch_fg_detect(cudaStream_t s, const float* x, long long x_sb, long long x_sc, long long x_sy,
                            long long x_sx, float* prev, long long p_sb, long long p_sy, int pp,
                            void* dhi, void* dlo, uint32_t* bits, int32_t* count, int B, int C, int H,
                            int W, float thr) {
  const int Wd = (W + 31) / 32;
  const long long words = (long long)B * H * Wd;
  if (count) cudaMemsetAsync(count, 0, sizeof(int32_t), s);
  if (words == 0) return 0;
  CB_CHECK_ARG(words < (1ll << 31), "fg_detect: image too large");
  const int cpv = (C + 3) / 4, cps = cpv | 1;
  CB_CHECK_ARG(pp % 4 == 0 && pp >= C && (p_sy % 4) == 0 && (p_sb % 4) == 0 && ((uintptr_t)prev % 16) == 0,
               "fg_detect: the state must be pixel-major with 16-byte aligned pixels");
  CB_CHECK_ARG(((uintptr_t)dhi % 16) == 0 && ((uintptr_t)dlo % 16) == 0, "fg_detect: unaligned delta planes");
  const bool xpm = x_sc == 1 && (C % 4) == 0 && (x_sx % 4) == 0 && (x_sy % 4) == 0 && (x_sb % 4) == 0 &&
                   ((uintptr_t)x % 16) == 0 && x_sx >= C;
  const int nw = planar_words_per_block(cpv, cps);
  const size_t smem = (size_t)nw * 32 * cps * 16;
  CB_CHECK_ARG(smem <= 200 * 1024, "fg_detect: too many channels (%d)", C);
  const unsigned magic = cpv > 1 ? (unsigned)((0x100000000ull + cpv - 1) / cpv) : 0u;
  auto kern = xpm ? fg_detect_kernel<1> : fg_detect_kernel<0>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  launch(kern, dim3((unsigned)((words + nw - 1) / nw)), dim3(256), smem, s, x, x_sb, x_sc, x_sy, x_sx, prev,
             p_sb, p_sy, pp, (__nv_bfloat16*)dhi, (__nv_bfloat16*)dlo, pitch16_of(C), bits, count, B, H, W, C,
             Wd, thr, magic, cps, nw);
  CB_CHECK_LAUNCH("fg_detect");
  return 0;
}

}  // namespace cb
