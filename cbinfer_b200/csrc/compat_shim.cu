// compat_shim.cu -- the REFERENCE's own FFI symbols on top of the C ABI of libcbinfer_sm100.so.
//
// The reference dlopens three libraries and calls them through cffi with the prototypes declared in
// pycbinfer/conv2d_cg.py:6-38 (changeDetection, changePropagation, genXMatrix, updateOutput,
// maxPool2d; the *_half_* twin exports the same names for fp16 data) and pycbinfer/conv2d_fg.py:13-29
// (updateOutputFG, changeDetectionFG).  This file exports exactly those symbols with exactly those
// argument lists and forwards them to include/cbinfer_b200.h, so the UNMODIFIED reference python
// files can bind the sm_100a kernels by dropping the three libraries built from it --
//     cbconv2d_cg_backend_<machine>.so        (default build)
//     cbconv2d_cg_half_backend_<machine>.so   (-DCB_COMPAT_HALF)
//     cbconv2d_fg_backend_<machine>.so        (-DCB_COMPAT_FG)
// -- next to them (cbinfer_b200/build.py: build_compat()).  What the shim adds to the ABI:
//   * the launch geometry arguments (gridz .. blockx) are accepted and ignored;
//   * the reference's byte change maps and host-side change counts are bridged to the library's
//     bitmaps / device-side counts with scratch buffers the shim owns (grow-only, per process);
//   * everything runs on the legacy default stream, as the reference's <<<grid, block>>> launches do.
// Layouts are the reference's: planar CHW, batch 1.  tests/test_gpu_compat_shim.py runs the same call
// sequences against these libraries and, where oracle/_ref is built, against the unmodified reference
// libraries; it always checks them against their own recorded outputs (tests/golden/compat_ops_golden.npz).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cbinfer_b200.h"

namespace {

struct Scratch {
  void* p = nullptr;
  size_t bytes = 0;
  // grow-only device buffer, zero-filled when (re)allocated
  void* get(size_t need) {
    if (need > bytes) {
      if (p) cudaFree(p);
      bytes = need + need / 2 + 256;
      if (cudaMalloc(&p, bytes) != cudaSuccess) { p = nullptr; bytes = 0; return nullptr; }
      cudaMemset(p, 0, bytes);
    }
    return p;
  }
};

#ifndef CB_COMPAT_FG
Scratch g_raw, g_idx, g_cnt, g_ws, g_bits;

void report(const char* what, int rc) {
  if (rc) fprintf(stderr, "cbinfer compat shim: %s failed: %s\n", what, cb_last_error());
}
#endif

#ifdef CB_COMPAT_HALF
constexpr int kDtype = CB_F16;
#else
constexpr int kDtype = CB_F32;
#endif

#ifdef CB_COMPAT_FG
// changeDetectionFG_kernel (cbconv2d_fg_backend.cu:7-23): per value d = in - prev; map = |d| > thr;
// diffs written only where changed
__global__ void shim_fg_detect(const float* __restrict__ in, const float* __restrict__ prev,
                               float* __restrict__ diffs, char* __restrict__ map, int n, float thr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float d;
  unsigned p;
  asm("{\n\t.reg .f32 a;\n\t.reg .pred q;\n\t"
      "sub.ftz.f32 %0, %2, %3;\n\t"
      "abs.ftz.f32 a, %0;\n\t"
      "setp.gt.ftz.f32 q, a, %4;\n\t"
      "selp.u32 %1, 1, 0, q;\n\t}"
      : "=f"(d), "=r"(p) : "f"(in[i]), "f"(prev[i]), "f"(thr));
  map[i] = (char)p;
  if (p) diffs[i] = d;
}

// updateOutputFG_kernel (cbconv2d_fg_backend.cu:37-66): a warp per changed value, lanes over
// (output channel, tap), fire-and-forget red.global.add
__global__ void shim_fg_update(const float* __restrict__ diffs, const float* __restrict__ w,
                               float* __restrict__ out, const long long* __restrict__ coords, int numOut,
                               int numIn, int H, int W, int kH, int kW, int n) {
  const int lane = threadIdx.x & 31;
  const int taps = kH * kW, work = numOut * taps;
  for (long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < n;
       c += (long long)gridDim.x * (blockDim.x >> 5)) {
    const int pos = (int)coords[c];
    const int ci = pos / (H * W), y = (pos / W) % H, x = pos % W;
    const float d = diffs[pos];
    for (int t = lane; t < work; t += 32) {
      const int co = t / taps, tap = t - co * taps;
      const int ky = tap / kW, kx = tap - ky * kW;
      const int yt = y - ky + kH / 2, xt = x - kx + kW / 2;
      if (yt >= 0 && yt < H && xt >= 0 && xt < W)
        atomicAdd(out + ((long long)co * H + yt) * W + xt,
                  __ldg(w + (((long long)co * numIn + ci) * kH + ky) * kW + kx) * d);
    }
  }
}
#endif

}  // namespace

extern "C" {

#ifndef CB_COMPAT_FG

/* conv2d_cg.py:7-13 -> cb_change_detect + cb_dilate_compact (byte map out) */
void changeDetection(int, int, int, int, int, int, const float* input, float* oldinput, bool* changeMatrix,
                     const int width, const int height, const int nInputPlane, const int kHHalf,
                     const int kWHalf, const float diffThreshold, const bool updateInputState) {
  const int B = 1, H = height, W = width, C = nInputPlane;
  const long long hw = (long long)H * W;
  uint32_t* raw = (uint32_t*)g_raw.get(cb_bitmap_words(B, H, W) * 4 + 4);
  int32_t* idx = (int32_t*)g_idx.get((size_t)hw * 4 + 4);
  int32_t* cnt = (int32_t*)g_cnt.get(16);
  void* ws = g_ws.get(cb_compact_ws_bytes(B, H, W));
  if (!raw || !idx || !cnt || !ws) { fprintf(stderr, "cbinfer compat shim: out of device memory\n"); return; }
  report("changeDetection", cb_change_detect(nullptr, kDtype, input, C * hw, hw, W, 1, oldinput, C * hw, hw, W, 1,
                                            CB_AUX_NONE, nullptr, nullptr, raw, B, C, H, W, diffThreshold,
                                            updateInputState ? CB_UPDATE_CHANGED : CB_UPDATE_NONE));
  report("changeDetection(dilate)", cb_dilate_compact(nullptr, raw, nullptr, (int8_t*)changeMatrix, idx, cnt, ws, B, H,
                                                      W, kHHalf, kWHalf, 0));
}

/* conv2d_cg.py:15-19 -> cb_map_to_bits + cb_dilate_compact */
void changePropagation(int, int, int, int, int, int, const bool* changeMatrixIn, bool* changeMatrixOut,
                       const int width, const int height, const int kHHalf, const int kWHalf) {
  const int B = 1, H = height, W = width;
  uint32_t* bits = (uint32_t*)g_bits.get(cb_bitmap_words(B, H, W) * 4 + 4);
  int32_t* idx = (int32_t*)g_idx.get((size_t)H * W * 4 + 4);
  int32_t* cnt = (int32_t*)g_cnt.get(16);
  void* ws = g_ws.get(cb_compact_ws_bytes(B, H, W));
  if (!bits || !idx || !cnt || !ws) { fprintf(stderr, "cbinfer compat shim: out of device memory\n"); return; }
  report("changePropagation", cb_map_to_bits(nullptr, (const int8_t*)changeMatrixIn, bits, B, H, W));
  report("changePropagation(dilate)", cb_dilate_compact(nullptr, bits, nullptr, (int8_t*)changeMatrixOut, idx, cnt, ws,
                                                        B, H, W, kHHalf, kWHalf, 0));
}

/* conv2d_cg.py:21-27 -> cb_gen_xmatrix */
void genXMatrix(int, int, int, int, int, int, float* columns, const float* input, const int* changeList,
                const int kW, const int kH, const int nInputPlane, const int width, const int height,
                const int numChanges) {
  report("genXMatrix", cb_gen_xmatrix(nullptr, kDtype, columns, input, changeList, kW, kH, nInputPlane, width, height,
                                      numChanges));
}

/* conv2d_cg.py:29-31 -> cb_update_output */
void updateOutput(int, int, int, int, int, int, float* columnsOut, float* output, int* changeList,
                  int numOutputPixel, int numChanges, int nOutputPlane, bool relu) {
  report("updateOutput", cb_update_output(nullptr, kDtype, columnsOut, output, changeList, numOutputPixel, numChanges,
                                          nOutputPlane, relu ? 1 : 0));
}

/* conv2d_cg.py:33-37 -> cb_maxpool2x2 (the host-side change count is staged into a device word) */
void maxPool2d(int, int, float* input, float* output, int* changeIndexes, int numChanges, int numCh,
               int iheight, int iwidth, int oheight, int owidth, int stridey, int stridex) {
  if (numChanges <= 0) return;
  if (stridey != 2 || stridex != 2) { fprintf(stderr, "cbinfer compat shim: maxPool2d: stride 2x2 only\n"); return; }
  int32_t* cnt = (int32_t*)g_cnt.get(16);
  if (!cnt) return;
  cudaMemcpyAsync(cnt + 1, &numChanges, sizeof(int), cudaMemcpyHostToDevice, nullptr);
  const long long ihw = (long long)iheight * iwidth, ohw = (long long)oheight * owidth;
  report("maxPool2d", cb_maxpool2x2(nullptr, kDtype, input, numCh * ihw, ihw, iwidth, 1, changeIndexes, cnt + 1, nullptr,
                                    output, numCh * ohw, ohw, owidth, 1, 1, numCh, iheight, iwidth, oheight, owidth));
}

#else  /* CB_COMPAT_FG */

/* conv2d_fg.py:20-24 */
void changeDetectionFG(const float* input, const float* prevInput, float* diffs, char* changeMap,
                       const int numVals, const float threshold) {
  if (numVals <= 0) return;
  shim_fg_detect<<<(numVals + 255) / 256, 256>>>(input, prevInput, diffs, changeMap, numVals, threshold);
}

/* conv2d_fg.py:14-18 */
void updateOutputFG(int, int, int, int, int, int, const float* diffs, const float* weight, float* output,
                    const long* changeCoords, const int numOut, const int numIn, const int height,
                    const int width, const int kH, const int kW, const int numChanges) {
  if (numChanges <= 0) return;
  int blocks = (numChanges + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  shim_fg_update<<<blocks, 256>>>(diffs, weight, output, (const long long*)changeCoords, numOut, numIn, height, width,
                                  kH, kW, numChanges);
}

#endif

}  // extern "C"
