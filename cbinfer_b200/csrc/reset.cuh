// reset.cuh -- per-stream state reset (cb_reset_streams): stream b's slice of every listed
// pixel-major buffer gets its real channels set to +inf (or 0) and its pad channels to 0, for every
// b whose mask byte is set.  One launch covers all segments; the mask is read on the device, so the
// call can be captured into a CUDA graph and steered by rewriting the mask between replays.
#pragma once
#include "cb_common.cuh"

namespace cb {

constexpr int kResetThreads = 256;
constexpr int kResetChunksPerThread = 16;                                 // 16-byte chunks
constexpr long long kResetChunksPerCta = (long long)kResetThreads * kResetChunksPerThread;  // 64 KB
// segments per launch: keeps the parameter block under the 4 KB every driver accepts
constexpr int kResetMaxSegs = 96;

struct ResetSeg {
  char* base;              // stream 0's slice
  long long slice;         // bytes per stream (pixels * pitch)
  unsigned fill;           // element bits of the real channels (+inf or 0)
  int pitch;               // bytes per pixel
  int chan;                // bytes of real channels per pixel
  int es;                  // element size, 2 or 4
};

struct ResetBatch {
  int n;
  unsigned cta0[kResetMaxSegs + 1];    // first CTA (blockIdx.x) of each segment; cta0[n] = grid.x
  ResetSeg seg[kResetMaxSegs];
};
static_assert(sizeof(ResetBatch) + sizeof(void*) <= 4096, "reset_streams_kernel parameters exceed 4 KB");

// element-wise stores of `nbytes` bytes at p, whose first byte lies `w` bytes into a pixel (the
// unaligned head and tail of a slice)
__device__ __forceinline__ void reset_store_elems(char* p, long long nbytes, int w, const ResetSeg& s) {
  for (long long i = 0; i < nbytes; i += s.es) {
    const unsigned v = w < s.chan ? s.fill : 0u;
    if (s.es == 4) *reinterpret_cast<unsigned*>(p + i) = v;
    else *reinterpret_cast<unsigned short*>(p + i) = (unsigned short)v;
    w += s.es;
    if (w >= s.pitch) w -= s.pitch;
  }
}

// one 16-byte chunk whose first byte lies `w` bytes into a pixel
__device__ __forceinline__ uint4 reset_chunk(int w, const ResetSeg& s, const uint4& full) {
  if (w + 16 <= s.chan) return full;                                     // real channels only
  if (w >= s.chan && w + 16 <= s.pitch) return make_uint4(0u, 0u, 0u, 0u);  // pad channels only
  unsigned wd[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    unsigned v;
    if (s.es == 4) {
      v = w < s.chan ? s.fill : 0u;
      w += 4;
      if (w >= s.pitch) w -= s.pitch;
    } else {
      const unsigned lo = w < s.chan ? s.fill : 0u;
      w += 2;
      if (w >= s.pitch) w -= s.pitch;
      const unsigned hi = w < s.chan ? s.fill : 0u;
      w += 2;
      if (w >= s.pitch) w -= s.pitch;
      v = lo | (hi << 16);
    }
    wd[k] = v;
  }
  return make_uint4(wd[0], wd[1], wd[2], wd[3]);
}

// grid (sum over segments of their CTAs, B): CTA (x, b) writes one 64 KB piece of stream b's slice
// of one segment; the first CTA of a slice also writes its unaligned head and tail
__global__ void __launch_bounds__(kResetThreads) reset_streams_kernel(const __grid_constant__ ResetBatch rb,
                                                                      const uint8_t* __restrict__ mask) {
  const int b = blockIdx.y;
  if (mask[b] == 0) return;
  const unsigned x = blockIdx.x;
  int si = 0;
  while (x >= rb.cta0[si + 1]) ++si;
  const ResetSeg& s = rb.seg[si];
  char* const lo = s.base + (long long)b * s.slice;                      // a whole number of pixels
  char* const hi = lo + s.slice;
  char* const a0 = reinterpret_cast<char*>(((uintptr_t)lo + 15) & ~(uintptr_t)15);
  char* const a1 = reinterpret_cast<char*>((uintptr_t)hi & ~(uintptr_t)15);
  const unsigned k = x - rb.cta0[si];
  if (a0 >= a1) {                                                        // no aligned chunk at all
    if (k == 0 && threadIdx.x == 0) reset_store_elems(lo, s.slice, 0, s);
    return;
  }
  if (k == 0 && threadIdx.x == 0) {
    reset_store_elems(lo, a0 - lo, 0, s);
    reset_store_elems(a1, hi - a1, (int)((a1 - lo) % s.pitch), s);
  }
  uint4 full;
  if (s.es == 4) full = make_uint4(s.fill, s.fill, s.fill, s.fill);
  else {
    const unsigned f2 = s.fill | (s.fill << 16);
    full = make_uint4(f2, f2, f2, f2);
  }
  const long long nchunks = (a1 - a0) >> 4;
  const long long c0 = (long long)k * kResetChunksPerCta + threadIdx.x;
  if (c0 >= nchunks) return;
  // byte offset into the pixel of this thread's first chunk, then the step between its chunks
  int w = (int)((a0 - lo + c0 * 16) % s.pitch);
  const int step = (kResetThreads * 16) % s.pitch;
  uint4* const dst = reinterpret_cast<uint4*>(a0);
#pragma unroll 4
  for (int i = 0; i < kResetChunksPerThread; ++i) {
    const long long c = c0 + (long long)i * kResetThreads;
    if (c >= nchunks) break;
    st16(dst + c, reset_chunk(w, s, full));
    w += step;
    if (w >= s.pitch) w -= s.pitch;
  }
}

}  // namespace cb
