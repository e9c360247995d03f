// cb_common.cuh -- shared helpers for libcbinfer_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>

#include "../../include/cbinfer_b200.h"

namespace cb {

// ---- error plumbing ------------------------------------------------------------------------
extern thread_local char g_err[512];
int fail(int code, const char* fmt, ...);

#define CB_CHECK_ARG(cond, ...)                                   \
  do {                                                            \
    if (!(cond)) return cb::fail(2, __VA_ARGS__);                 \
  } while (0)

#define CB_CHECK_LAUNCH(what)                                                           \
  do {                                                                                  \
    cudaError_t e_ = cudaGetLastError();                                                \
    if (e_ != cudaSuccess) return cb::fail(3, "%s: %s", what, cudaGetErrorString(e_));  \
  } while (0)

int sm_count();

// log2 of the lanes that share one pixel in the candidate-detection / pooling kernels: one lane per
// two 16-byte chunks, at most 16 lanes.  One lane per chunk would be the obvious choice; two chunks per
// lane halves the number of warps (one wave instead of two at 8 streams) and doubles the loads in
// flight per lane: measured pool+detect 11.3 -> 8.3 us, sparse detect 7.7 -> 6.7 us.
inline int group_log2(int chunks) {
  int g = 0;
  while (g < 4 && (2 << g) < chunks) ++g;
  return g;
}

// Calls f(std::integral_constant<int, update>{}), so that the kernels f launches take the update mode
// as a template argument; an unknown mode fails with "<what>: bad update_mode".
template <typename F>
inline int dispatch_update(int update, const char* what, F&& f) {
  switch (update) {
    case CB_UPDATE_NONE: return f(std::integral_constant<int, CB_UPDATE_NONE>{});
    case CB_UPDATE_CHANGED: return f(std::integral_constant<int, CB_UPDATE_CHANGED>{});
    case CB_UPDATE_ALL: return f(std::integral_constant<int, CB_UPDATE_ALL>{});
    default: return fail(2, "%s: bad update_mode %d", what, update);
  }
}

// per-stream threshold table given?  A compile-time kernel variant (THR), so the kernels launched
// without one compile exactly as they would without the feature
template <typename F>
inline int dispatch_thr(const void* thr_b, F&& f) {
  return thr_b ? f(std::true_type{}) : f(std::false_type{});
}

// cooperative != 0: the grid is launched only when ALL its CTAs can be resident at once (kernels whose
// CTAs wait for each other, e.g. the stream-K finisher spinning on its contributors' flags, must not
// be half-resident next to another grid on a concurrent stream)
template <typename... KArgs, typename... Args>
inline void launch_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                           cudaStream_t s, unsigned cluster_x, int cooperative, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  unsigned na = 0;
  if (cooperative) {
    attr[na].id = cudaLaunchAttributeCooperative;
    attr[na].val.cooperative = 1;
    ++na;
  }
  if (cluster_x > 1) {                         // thread-block cluster (cluster_x, 1, 1)
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster_x;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

template <typename... KArgs, typename... Args>
inline void launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                   Args&&... args) {
  launch_cluster(kern, grid, block, smem, s, 1u, 0, static_cast<Args&&>(args)...);
}

// ---- dtype helpers -------------------------------------------------------------------------
__host__ __device__ inline int esize(int dtype) { return dtype == CB_F32 ? 4 : 2; }
// channel pitch of the bf16 operand planes of an fp32 layer: a multiple of 16 bytes (an RGB input
// layer gets 16-byte pixels: the smallest pixel the tiled contraction's shared-memory descriptors
// can address, conv_tile.cuh)
__host__ __device__ inline int pitch16_of(int C) { return (C + 7) / 8 * 8; }

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_float<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

// ---- the per-value change test (bit-exact contract) ----------------------------------------
// fp32: reference compiles `fabs(state - in) > thr` with --use_fast_math
//       (cbconv2d_cg_backend.cu:56, build.sh:5) => sub.ftz / abs.ftz / setp.gt.ftz.
__device__ __forceinline__ bool value_changed(float s, float x, float thr) {
  unsigned r;
  asm("{\n\t.reg .f32 d;\n\t.reg .pred p;\n\t"
      "sub.ftz.f32 d, %1, %2;\n\t"
      "abs.ftz.f32 d, d;\n\t"
      "setp.gt.ftz.f32 p, d, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(r) : "f"(s), "f"(x), "f"(thr));
  return r != 0;
}
// fp16: thr_h = __float2half(thr); diff = __hsub(state, in); diff > thr_h || diff < -thr_h
//       (cbconv2d_cg_half_backend.cu:58-63).  bf16: same recipe in bf16 (no reference kernel).
__device__ __forceinline__ bool value_changed(__half s, __half x, __half thr) {
  __half d = __hsub(s, x);
  return __hgt(d, thr) | __hlt(d, __hneg(thr));
}
__device__ __forceinline__ bool value_changed(__nv_bfloat16 s, __nv_bfloat16 x, __nv_bfloat16 thr) {
  __nv_bfloat16 d = __hsub(s, x);
  return __hgt(d, thr) | __hlt(d, __hneg(thr));
}

// 16-byte chunk: any element changed?
template <typename T> struct Chunk;
template <> struct Chunk<float> {
  static __device__ __forceinline__ bool changed(const uint4& s, const uint4& x, float thr) {
    return value_changed(__uint_as_float(s.x), __uint_as_float(x.x), thr) |
           value_changed(__uint_as_float(s.y), __uint_as_float(x.y), thr) |
           value_changed(__uint_as_float(s.z), __uint_as_float(x.z), thr) |
           value_changed(__uint_as_float(s.w), __uint_as_float(x.w), thr);
  }
};
template <> struct Chunk<__half> {
  static __device__ __forceinline__ bool pair(unsigned s, unsigned x, __half2 thr2, __half2 nthr2) {
    __half2 d = __hsub2(*reinterpret_cast<__half2*>(&s), *reinterpret_cast<__half2*>(&x));
    return (__hgt2_mask(d, thr2) != 0u) | (__hlt2_mask(d, nthr2) != 0u);  // any lane
  }
  static __device__ __forceinline__ bool changed(const uint4& s, const uint4& x, __half thr) {
    __half2 t2 = __half2half2(thr), n2 = __hneg2(t2);
    return pair(s.x, x.x, t2, n2) | pair(s.y, x.y, t2, n2) | pair(s.z, x.z, t2, n2) |
           pair(s.w, x.w, t2, n2);
  }
};
template <> struct Chunk<__nv_bfloat16> {
  static __device__ __forceinline__ bool pair(unsigned s, unsigned x, __nv_bfloat162 thr2,
                                              __nv_bfloat162 nthr2) {
    __nv_bfloat162 d = __hsub2(*reinterpret_cast<__nv_bfloat162*>(&s),
                               *reinterpret_cast<__nv_bfloat162*>(&x));
    return (__hgt2_mask(d, thr2) != 0u) | (__hlt2_mask(d, nthr2) != 0u);
  }
  static __device__ __forceinline__ bool changed(const uint4& s, const uint4& x,
                                                 __nv_bfloat16 thr) {
    __nv_bfloat162 t2 = __bfloat162bfloat162(thr), n2 = __hneg2(t2);
    return pair(s.x, x.x, t2, n2) | pair(s.y, x.y, t2, n2) | pair(s.z, x.z, t2, n2) |
           pair(s.w, x.w, t2, n2);
  }
};

// ---- memory helpers ------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg16(const void* p) {
  return __ldg(reinterpret_cast<const uint4*>(p));
}
__device__ __forceinline__ uint4 ld16(const void* p) {          // coherent (state is read+written)
  return *reinterpret_cast<const uint4*>(p);
}
__device__ __forceinline__ void st16(void* p, const uint4& v) {
  *reinterpret_cast<uint4*>(p) = v;
}

// ---- per-stream change counts (cb_*_streams entry points) ----------------------------------
// Adds `c` to acc[b] for every stream b held by a lane of the warp: one atomic per (warp, stream).
// Lanes may hold streams in any order; b < 0 marks a lane with nothing to add.  All 32 lanes call.
__device__ __forceinline__ void stream_add_warp(int b, unsigned c, int32_t* acc) {
  const unsigned same = __match_any_sync(0xffffffffu, b);
  const unsigned sum = __reduce_add_sync(same, c);
  if (b >= 0 && sum && (int)(threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(acc + b, (int)sum);
}
// Run by the block that publishes a kernel's total, after every block's additions to `acc`:
// counts[b] = acc[b], and acc is left zero for the next launch.
__device__ __forceinline__ void stream_publish(int32_t* acc, int32_t* counts, int B) {
  for (int b = threadIdx.x; b < B; b += blockDim.x) counts[b] = atomicExch(acc + b, 0);
}

}  // namespace cb
