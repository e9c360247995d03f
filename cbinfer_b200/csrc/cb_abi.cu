// cb_abi.cu -- extern "C" entry points of libcbinfer_sm100.so (see include/cbinfer_b200.h).
// sm_100a only: no other architecture, no CPU path, no dispatch to other backends.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "cb_common.cuh"
#include "compact.cuh"
#include "conv_simt.cuh"
#include "conv_umma.cuh"
#include "conv_tile.cuh"
#include "detect.cuh"
#include "ingest.cuh"
#include "fg.cuh"
#include "pool.cuh"
#include "reset.cuh"
#include "staged.cuh"
#include "tail.cuh"

namespace cb {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
    cached_dev = dev;
  }
  return cached > 0 ? cached : 148;
}

static inline unsigned grid_for(long long total, int threads, int per_sm = 8) {
  long long blocks = (total + threads - 1) / threads;
  long long cap = (long long)sm_count() * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

}  // namespace cb

using namespace cb;

#define CB_DISPATCH_DTYPE(dtype, ...)                                               \
  switch (dtype) {                                                                  \
    case CB_F32: { using T = float; constexpr int VEC = 4; (void)VEC; __VA_ARGS__; } break;           \
    case CB_F16: { using T = __half; constexpr int VEC = 8; (void)VEC; __VA_ARGS__; } break;          \
    case CB_BF16: { using T = __nv_bfloat16; constexpr int VEC = 8; (void)VEC; __VA_ARGS__; } break;  \
    default: return cb::fail(2, "bad dtype %d", dtype);                             \
  }

extern "C" {

int cb_version(void) { return 100; }

const char* cb_last_error(void) { return cb::g_err; }

int cb_device_info(int* sms, int* major, int* minor) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return cb::fail(3, "no CUDA device");
  cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(minor, cudaDevAttrComputeCapabilityMinor, dev);
  return 0;
}

int cb_bitmap_row_words(int W) { return (W + 31) / 32; }
size_t cb_bitmap_words(int B, int H, int W) { return (size_t)B * H * ((W + 31) / 32); }
size_t cb_compact_ws_bytes(int B, int H, int W) { return cb::compact_ws_bytes(cb_bitmap_words(B, H, W)); }
int cb_plane_pitch16(int C) { return cb::pitch16_of(C); }
int cb_channel_pitch(int dtype, int C) {
  const int v = 16 / cb::esize(dtype);
  return (C + v - 1) / v * v;
}

// per-stream thresholds (the *_thr entry points): fp32 [B] in device memory, or NULL = the scalar
#define CB_CHECK_THR(thr_b, what) \
  CB_CHECK_ARG(((uintptr_t)(thr_b) % sizeof(float)) == 0, what ": thr_b is not aligned to 4 bytes")

// watched-pixel zone (the *_zone entry points): uint32 [B, H, Wd] bitmap in device memory, or NULL
#define CB_CHECK_ZONE(zone, what) \
  CB_CHECK_ARG(((uintptr_t)(zone) % sizeof(uint32_t)) == 0, what ": zone is not aligned to 4 bytes")

int cb_change_detect_zone(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                          long long x_sy, long long x_sx, void* state, long long s_sb, long long s_sc,
                          long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                          uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                          int update_mode, const uint8_t* active, const float* thr_b, const uint32_t* zone) {
  CB_CHECK_ARG(x && state && raw_bits, "change_detect: null pointer");
  CB_CHECK_ARG(B >= 0 && C > 0 && H >= 0 && W >= 0, "change_detect: bad shape");
  CB_CHECK_THR(thr_b, "change_detect");
  CB_CHECK_ZONE(zone, "change_detect");
  CB_DISPATCH_DTYPE(dtype, return (launch_detect<T, VEC>((cudaStream_t)stream, x, x_sb, x_sc, x_sy,
                                                        x_sx, state, s_sb, s_sc, s_sy, s_sx, aux_mode,
                                                        aux_hi, aux_lo, raw_bits, B, C, H, W, threshold,
                                                        update_mode, active, thr_b, zone)));
  return 0;
}

int cb_change_detect_thr(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                         long long x_sy, long long x_sx, void* state, long long s_sb, long long s_sc,
                         long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                         uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                         int update_mode, const uint8_t* active, const float* thr_b) {
  return cb_change_detect_zone(stream, dtype, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, aux_mode,
                               aux_hi, aux_lo, raw_bits, B, C, H, W, threshold, update_mode, active, thr_b, nullptr);
}

int cb_change_detect_streams(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                             long long x_sy, long long x_sx, void* state, long long s_sb, long long s_sc,
                             long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                             uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                             int update_mode, const uint8_t* active) {
  return cb_change_detect_thr(stream, dtype, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, aux_mode,
                              aux_hi, aux_lo, raw_bits, B, C, H, W, threshold, update_mode, active, nullptr);
}

int cb_change_detect(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                     long long x_sy, long long x_sx, void* state, long long s_sb, long long s_sc,
                     long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                     uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                     int update_mode) {
  return cb_change_detect_streams(stream, dtype, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx,
                                  aux_mode, aux_hi, aux_lo, raw_bits, B, C, H, W, threshold, update_mode, nullptr);
}

int cb_change_detect_u8_zone(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                             long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                             long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                             uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                             float threshold, int update_mode, const uint8_t* active, const float* thr_b,
                             const uint32_t* zone) {
  CB_CHECK_ARG(x && state && raw_bits, "change_detect_u8: null pointer");
  CB_CHECK_ARG(B >= 0 && C > 0 && H >= 0 && W >= 0, "change_detect_u8: bad shape");
  CB_CHECK_THR(thr_b, "change_detect_u8");
  CB_CHECK_ZONE(zone, "change_detect_u8");
  return launch_detect_u8((cudaStream_t)stream, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy,
                          s_sx, aux_mode, aux_hi, aux_lo, raw_bits, B, C, H, W, divisor, bias,
                          threshold, update_mode, active, thr_b, zone);
}

int cb_change_detect_u8_thr(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                            long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                            long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                            uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                            float threshold, int update_mode, const uint8_t* active, const float* thr_b) {
  return cb_change_detect_u8_zone(stream, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, aux_mode,
                                  aux_hi, aux_lo, raw_bits, B, C, H, W, divisor, bias, threshold, update_mode,
                                  active, thr_b, nullptr);
}

int cb_change_detect_u8_streams(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                                long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                                long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                                uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                                float threshold, int update_mode, const uint8_t* active) {
  return cb_change_detect_u8_thr(stream, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, aux_mode,
                                 aux_hi, aux_lo, raw_bits, B, C, H, W, divisor, bias, threshold, update_mode,
                                 active, nullptr);
}

int cb_change_detect_u8(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                        long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                        long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                        uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                        float threshold, int update_mode) {
  return cb_change_detect_u8_streams(stream, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, aux_mode,
                                     aux_hi, aux_lo, raw_bits, B, C, H, W, divisor, bias, threshold, update_mode,
                                     nullptr);
}

size_t cb_tile_ws_bytes(int B, int H, int W) { return cb::tile_ws_words(B, H, W) * sizeof(int32_t); }

// per-stream counts (the *_streams entry points): an output row needs its own accumulator
#define CB_CHECK_STREAMS(counts, acc, what)                                                        \
  CB_CHECK_ARG(!(counts) || ((acc) && (void*)(acc) != (void*)(counts)),                          \
               what ": stream_counts needs a separate stream_acc")

// a launch that has nothing to scan still writes its row of per-stream counts (zeros)
static int zero_stream_counts(cudaStream_t s, int32_t* counts, int B, const char* what) {
  if (counts && B > 0 && cudaMemsetAsync(counts, 0, (size_t)B * sizeof(int32_t), s) != cudaSuccess)
    return cb::fail(3, "%s: memset of the stream counts failed", what);
  return 0;
}

static int dilate_compact_impl(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int8_t* dil_map,
                      int32_t* idx, int32_t* count, void* ws, void* tile_ws, int B, int H, int W, int kHHalf,
                      int kWHalf, int clear_raw, int no_list, int32_t* stream_counts, int32_t* stream_acc) {
  CB_CHECK_ARG(raw_bits && (idx || no_list) && count && ws, "dilate_compact: null pointer");
  CB_CHECK_STREAMS(stream_counts, stream_acc, "dilate_compact");
  CB_CHECK_ARG(raw_bits != dil_bits, "dilate_compact: dil_bits must not alias raw_bits");
  CB_CHECK_ARG(kHHalf >= 0 && kWHalf >= 0 && kWHalf <= 31, "dilate_compact: kWHalf must be <= 31");
  CB_CHECK_ARG((long long)B * H * W < (1ll << 31), "dilate_compact: more than 2^31 pixels");
  const long long nwords = (long long)cb_bitmap_words(B, H, W);
  cudaStream_t s = (cudaStream_t)stream;
  if (nwords == 0) {
    cudaMemsetAsync(count, 0, sizeof(int32_t), s);
    CB_CHECK_LAUNCH("dilate_compact(memset)");
    return zero_stream_counts(s, stream_counts, B, "dilate_compact");
  }
  CB_CHECK_ARG(nwords < (1ll << 31), "dilate_compact: bitmap too large");
  const int ntiles = (int)((nwords + kCompactTile - 1) / kCompactTile);
  uint32_t* clear = clear_raw ? const_cast<uint32_t*>(raw_bits) : nullptr;
  if (stream_counts)
    cb::launch(dilate_compact_kernel<true>, ntiles, kCompactThreads, 0, s, raw_bits, dil_bits, dil_map, idx, count,
               ws, B, H, W, (W + 31) / 32, kHHalf, kWHalf, (int)nwords, ntiles, 0, 0, clear, (int32_t*)tile_ws,
               cb::tile_grid_y(H), cb::tile_grid_xp(W), no_list, stream_counts, stream_acc);
  else
    cb::launch(dilate_compact_kernel<false>, ntiles, kCompactThreads, 0, s, raw_bits, dil_bits, dil_map, idx, count,
               ws, B, H, W, (W + 31) / 32, kHHalf, kWHalf, (int)nwords, ntiles, 0, 0, clear, (int32_t*)tile_ws,
               cb::tile_grid_y(H), cb::tile_grid_xp(W), no_list, nullptr, nullptr);
  CB_CHECK_LAUNCH("dilate_compact");
  return 0;
}

int cb_dilate_compact_streams(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int8_t* dil_map,
                              int32_t* idx, int32_t* count, void* ws, int B, int H, int W, int kHHalf,
                              int kWHalf, int clear_raw, int32_t* stream_counts, int32_t* stream_acc) {
  return dilate_compact_impl(stream, raw_bits, dil_bits, dil_map, idx, count, ws, nullptr, B, H, W,
                             kHHalf, kWHalf, clear_raw, 0, stream_counts, stream_acc);
}

int cb_dilate_compact(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int8_t* dil_map,
                      int32_t* idx, int32_t* count, void* ws, int B, int H, int W, int kHHalf,
                      int kWHalf, int clear_raw) {
  return cb_dilate_compact_streams(stream, raw_bits, dil_bits, dil_map, idx, count, ws, B, H, W, kHHalf, kWHalf,
                                   clear_raw, nullptr, nullptr);
}

int cb_dilate_compact_tiles_streams(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits,
                                    int8_t* dil_map, int32_t* idx, int32_t* count, void* ws, void* tile_ws,
                                    int B, int H, int W, int kHHalf, int kWHalf, int clear_raw,
                                    int32_t* stream_counts, int32_t* stream_acc) {
  CB_CHECK_ARG(tile_ws, "dilate_compact_tiles: null tile workspace");
  CB_CHECK_STREAMS(stream_counts, stream_acc, "dilate_compact_tiles");
  if ((long long)cb_bitmap_words(B, H, W) == 0) cudaMemsetAsync((int32_t*)tile_ws + 1, 0, sizeof(int32_t), (cudaStream_t)stream);
  return dilate_compact_impl(stream, raw_bits, dil_bits, dil_map, idx, count, ws, tile_ws, B, H, W,
                             kHHalf, kWHalf, clear_raw, 0, stream_counts, stream_acc);
}

int cb_dilate_compact_tiles(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits,
                            int8_t* dil_map, int32_t* idx, int32_t* count, void* ws, void* tile_ws,
                            int B, int H, int W, int kHHalf, int kWHalf, int clear_raw) {
  return cb_dilate_compact_tiles_streams(stream, raw_bits, dil_bits, dil_map, idx, count, ws, tile_ws, B, H, W,
                                         kHHalf, kWHalf, clear_raw, nullptr, nullptr);
}

int cb_dilate_tiles_streams(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int32_t* count, void* ws,
                            void* tile_ws, int B, int H, int W, int kHHalf, int kWHalf, int clear_raw,
                            int32_t* stream_counts, int32_t* stream_acc) {
  CB_CHECK_ARG(tile_ws && dil_bits, "dilate_tiles: null pointer");
  CB_CHECK_STREAMS(stream_counts, stream_acc, "dilate_tiles");
  if ((long long)cb_bitmap_words(B, H, W) == 0) cudaMemsetAsync((int32_t*)tile_ws + 1, 0, sizeof(int32_t), (cudaStream_t)stream);
  return dilate_compact_impl(stream, raw_bits, dil_bits, nullptr, nullptr, count, ws, tile_ws, B, H, W,
                             kHHalf, kWHalf, clear_raw, 1, stream_counts, stream_acc);
}

int cb_dilate_tiles(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int32_t* count, void* ws,
                    void* tile_ws, int B, int H, int W, int kHHalf, int kWHalf, int clear_raw) {
  return cb_dilate_tiles_streams(stream, raw_bits, dil_bits, count, ws, tile_ws, B, H, W, kHHalf, kWHalf,
                                 clear_raw, nullptr, nullptr);
}

int cb_stream_bucket(void* stream, const int32_t* idx, const int32_t* count, int B, int hw,
                     int32_t* stream_counts, int32_t* stream_acc) {
  CB_CHECK_ARG(idx && count && stream_counts, "stream_bucket: null pointer");
  CB_CHECK_STREAMS(stream_counts, stream_acc, "stream_bucket");
  CB_CHECK_ARG(B > 0 && hw >= 0 && (long long)B * hw < (1ll << 31), "stream_bucket: bad shape B = %d, H*W = %d",
               B, hw);
  cudaStream_t s = (cudaStream_t)stream;
  if (hw == 0) return zero_stream_counts(s, stream_counts, B, "stream_bucket");
  const long long cap = (long long)sm_count() * 4, need = ((long long)B * hw + 255) / 256;
  const unsigned grid = (unsigned)(need < cap ? need : cap);
  cb::launch(stream_bucket_kernel, grid, 256, 0, s, idx, count, hw, B, stream_counts, stream_acc);
  CB_CHECK_LAUNCH("stream_bucket");
  return 0;
}

int cb_pool_compact(void* stream, const uint32_t* in_bits, uint32_t* out_bits, int32_t* idx,
                    int32_t* count, void* ws, int B, int H, int W, int oH, int oW) {
  CB_CHECK_ARG(in_bits && idx && count && ws, "pool_compact: null pointer");
  CB_CHECK_ARG(in_bits != out_bits, "pool_compact: out_bits must not alias in_bits");
  const long long nwords = (long long)cb_bitmap_words(B, oH, oW);
  cudaStream_t s = (cudaStream_t)stream;
  if (nwords == 0 || H == 0) {
    cudaMemsetAsync(count, 0, sizeof(int32_t), s);
    CB_CHECK_LAUNCH("pool_compact(memset)");
    return 0;
  }
  CB_CHECK_ARG(nwords < (1ll << 31), "pool_compact: bitmap too large");
  const int ntiles = (int)((nwords + kCompactTile - 1) / kCompactTile);
  cb::launch(dilate_compact_kernel<false>, ntiles, kCompactThreads, 0, s, in_bits, out_bits, nullptr, idx, count, ws,
                                                          B, oH, oW, (oW + 31) / 32, 0, 0,
                                                          (int)nwords, ntiles, H, (W + 31) / 32, nullptr,
                                                          nullptr, 0, 0, 0, nullptr, nullptr);
  CB_CHECK_LAUNCH("pool_compact");
  return 0;
}

int cb_change_detect_sparse_thr(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                long long x_sy, long long x_sx, void* state, long long s_sb,
                                long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                void* aux_hi, void* aux_lo, const int32_t* candidates, const int32_t* n_candidates,
                                uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                                int update_mode, int bits_are_clear, const float* thr_b) {
  CB_CHECK_ARG(x && state && raw_bits && candidates && n_candidates, "change_detect_sparse: null pointer");
  CB_CHECK_ARG(B >= 0 && C > 0 && H >= 0 && W >= 0, "change_detect_sparse: bad shape");
  CB_CHECK_THR(thr_b, "change_detect_sparse");
  CB_DISPATCH_DTYPE(dtype, return (launch_detect_sparse<T, VEC>(
                               (cudaStream_t)stream, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc,
                               s_sy, s_sx, aux_mode, aux_hi, aux_lo, candidates, n_candidates, raw_bits,
                               B, C, H, W,
                               threshold, update_mode, bits_are_clear, nullptr, thr_b)));
  return 0;
}

int cb_change_detect_sparse(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                            long long x_sy, long long x_sx, void* state, long long s_sb,
                            long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                            void* aux_hi, void* aux_lo, const int32_t* candidates, const int32_t* n_candidates,
                            uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                            int update_mode, int bits_are_clear) {
  return cb_change_detect_sparse_thr(stream, dtype, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx,
                                     aux_mode, aux_hi, aux_lo, candidates, n_candidates, raw_bits, B, C, H, W,
                                     threshold, update_mode, bits_are_clear, nullptr);
}

int cb_compact_small_max_words(void) { return cb::kCompactWin; }

int cb_change_detect_sparse_compact_thr(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                        long long x_sy, long long x_sx, void* state, long long s_sb,
                                        long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                        void* aux_hi, void* aux_lo, const int32_t* candidates,
                                        const int32_t* n_candidates, uint32_t* raw_bits, int B, int C, int H,
                                        int W, float threshold, int update_mode, int bits_are_clear,
                                        uint32_t* dil_bits, int32_t* idx, int32_t* count, void* sync_ws,
                                        int kHHalf, int kWHalf, int clear_raw, int32_t* stream_counts,
                                        int32_t* stream_acc, const float* thr_b) {
  CB_CHECK_ARG(x && state && raw_bits && candidates && n_candidates && idx && count && sync_ws,
               "change_detect_sparse_compact: null pointer");
  CB_CHECK_STREAMS(stream_counts, stream_acc, "change_detect_sparse_compact");
  CB_CHECK_THR(thr_b, "change_detect_sparse_compact");
  CB_CHECK_ARG(B >= 0 && C > 0 && H >= 0 && W >= 0, "change_detect_sparse_compact: bad shape");
  CB_CHECK_ARG(kHHalf >= 0 && kWHalf >= 0 && kWHalf <= 31, "change_detect_sparse_compact: kWHalf must be <= 31");
  CB_CHECK_ARG(raw_bits != dil_bits, "change_detect_sparse_compact: dil_bits must not alias raw_bits");
  const long long nwords = (long long)cb_bitmap_words(B, H, W);
  if (nwords == 0) {
    cudaMemsetAsync(count, 0, sizeof(int32_t), (cudaStream_t)stream);
    return zero_stream_counts((cudaStream_t)stream, stream_counts, B, "change_detect_sparse_compact");
  }
  CB_CHECK_ARG(nwords <= cb::kCompactWin, "change_detect_sparse_compact: bitmap of %lld words > %d", nwords,
               cb::kCompactWin);
  cb::FusedCompact fc{dil_bits, idx, count, (unsigned*)sync_ws, kHHalf, kWHalf, (int)nwords, clear_raw,
                      stream_counts, stream_acc, B};
  CB_DISPATCH_DTYPE(dtype, return (launch_detect_sparse<T, VEC>(
                               (cudaStream_t)stream, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc,
                               s_sy, s_sx, aux_mode, aux_hi, aux_lo, candidates, n_candidates, raw_bits,
                               B, C, H, W, threshold, update_mode, bits_are_clear, &fc, thr_b)));
  return 0;
}

int cb_change_detect_sparse_compact_streams(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                            long long x_sy, long long x_sx, void* state, long long s_sb,
                                            long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                            void* aux_hi, void* aux_lo, const int32_t* candidates,
                                            const int32_t* n_candidates, uint32_t* raw_bits, int B, int C, int H,
                                            int W, float threshold, int update_mode, int bits_are_clear,
                                            uint32_t* dil_bits, int32_t* idx, int32_t* count, void* sync_ws,
                                            int kHHalf, int kWHalf, int clear_raw, int32_t* stream_counts,
                                            int32_t* stream_acc) {
  return cb_change_detect_sparse_compact_thr(stream, dtype, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy,
                                             s_sx, aux_mode, aux_hi, aux_lo, candidates, n_candidates, raw_bits,
                                             B, C, H, W, threshold, update_mode, bits_are_clear, dil_bits, idx,
                                             count, sync_ws, kHHalf, kWHalf, clear_raw, stream_counts, stream_acc,
                                             nullptr);
}

int cb_change_detect_sparse_compact(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                    long long x_sy, long long x_sx, void* state, long long s_sb,
                                    long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                    void* aux_hi, void* aux_lo, const int32_t* candidates,
                                    const int32_t* n_candidates, uint32_t* raw_bits, int B, int C, int H,
                                    int W, float threshold, int update_mode, int bits_are_clear,
                                    uint32_t* dil_bits, int32_t* idx, int32_t* count, void* sync_ws,
                                    int kHHalf, int kWHalf, int clear_raw) {
  return cb_change_detect_sparse_compact_streams(stream, dtype, x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy,
                                                 s_sx, aux_mode, aux_hi, aux_lo, candidates, n_candidates, raw_bits,
                                                 B, C, H, W, threshold, update_mode, bits_are_clear, dil_bits, idx,
                                                 count, sync_ws, kHHalf, kWHalf, clear_raw, nullptr, nullptr);
}

int cb_map_to_bits(void* stream, const int8_t* map, uint32_t* bits, int B, int H, int W) {
  CB_CHECK_ARG(map && bits, "map_to_bits: null pointer");
  const long long nwords = (long long)cb_bitmap_words(B, H, W);
  if (nwords == 0) return 0;
  const long long blocks = (nwords + 7) / 8;
  cb::launch(map_to_bits_kernel, (unsigned)blocks, 256, 0, (cudaStream_t)stream, map, bits, H, W,
                                                                        (W + 31) / 32, nwords);
  CB_CHECK_LAUNCH("map_to_bits");
  return 0;
}

size_t cb_packed_weight_bytes(int dtype, int gemm, int Cout, int Cin, int kH, int kW) {
  const int Cp = gemm == CB_GEMM_TC_BF16X3 ? cb::pitch16_of(Cin) : cb_channel_pitch(dtype, Cin);
  if (gemm == CB_GEMM_SIMT_F32) {
    const int CoutP = (Cout + 3) / 4 * 4;
    return (size_t)kH * kW * Cp * CoutP * sizeof(float);
  }
  return cb::umma_packed_bytes(dtype, gemm, Cout, Cp, kH, kW);
}

int cb_pack_weights(void* stream, int dtype, int gemm, const void* weight, void* packed, int Cout,
                    int Cin, int kH, int kW) {
  CB_CHECK_ARG(weight && packed, "pack_weights: null pointer");
  const int Cp = gemm == CB_GEMM_TC_BF16X3 ? cb::pitch16_of(Cin) : cb_channel_pitch(dtype, Cin);
  cudaStream_t s = (cudaStream_t)stream;
  if (gemm == CB_GEMM_SIMT_F32) {
    const int CoutP = (Cout + 3) / 4 * 4;
    const long long total = (long long)kH * kW * Cp * CoutP;
    CB_DISPATCH_DTYPE(dtype, (cb::launch(pack_weights_simt_kernel<T>, grid_for(total, 256), 256, 0, s, 
                                 (const T*)weight, (float*)packed, Cout, Cin, kH, kW, Cp, CoutP)));
    CB_CHECK_LAUNCH("pack_weights");
    return 0;
  }
  return cb::umma_pack_weights(s, dtype, gemm, weight, packed, Cout, Cin, Cp, kH, kW);
}

size_t cb_conv_ws_bytes(void) {
  // flags + one fp32 partial tile per resident CTA slot; 256 KB per SM covers every tiling
  return (size_t)cb::UM_SK_FLAG_BYTES + (size_t)sm_count() * 256 * 1024;
}

static int conv_update_impl(const cb::RowMask& mk, void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                   int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                   const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                   int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes) {
  CB_CHECK_ARG(state && idx && count && packed_w && bias && out, "conv_update: null pointer");
  const int want_pitch = gemm == CB_GEMM_TC_BF16X3 ? cb::pitch16_of(Cin) : cb_channel_pitch(dtype, Cin);
  CB_CHECK_ARG(pitch_in == want_pitch, "conv_update: pitch_in %d != channel pitch %d", pitch_in,
               want_pitch);
  CB_CHECK_ARG(pitch_out >= Cout, "conv_update: pitch_out < Cout");
  CB_CHECK_ARG((kH & 1) && (kW & 1), "conv_update: even kernel sizes unsupported (padding==k//2)");
  CB_CHECK_ARG((long long)B * H * W < (1ll << 31), "conv_update: more than 2^31 pixels");
  if (B == 0 || H == 0 || W == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  CB_CHECK_ARG(!(mk.bits && gemm == CB_GEMM_SIMT_F32), "conv_update_masked: tensor-core modes only");
  if (gemm == CB_GEMM_SIMT_F32) {
    const int CoutP = (Cout + 3) / 4 * 4;
    const unsigned grid = (unsigned)(sm_count() * 4);
    CB_DISPATCH_DTYPE(dtype, (cb::launch(conv_simt_kernel<T>, grid, SM_THREADS, 0, s, 
                                 (const T*)state, pitch_in, idx, count, (const float*)packed_w, bias,
                                 (T*)out, pitch_out, H, W, Cout, CoutP, kH, kW, relu)));
    CB_CHECK_LAUNCH("conv_update(simt)");
    return 0;
  }
  return cb::umma_conv_update(s, dtype, gemm, state, state_lo, pitch_in, idx, count, packed_w, bias, out,
                              pitch_out, B, H, W, Cin, Cout, kH, kW, relu, ws, ws_bytes, mk);
}

int cb_conv_update(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                   int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                   const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                   int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes) {
  return conv_update_impl(cb::RowMask{nullptr, nullptr, nullptr, nullptr, 0}, stream, dtype, gemm, state,
                          state_lo, pitch_in, idx, count, packed_w, bias, out, pitch_out, B, H, W, Cin,
                          Cout, kH, kW, relu ? 1 : 0, ws, ws_bytes);
}

int cb_conv_accumulate(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                       int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                       void* out, int pitch_out, int B, int H, int W, int Cin, int Cout, int kH, int kW,
                       void* ws, size_t ws_bytes) {
  CB_CHECK_ARG(gemm != CB_GEMM_SIMT_F32, "conv_accumulate: tensor-core modes only");
  // flag bit 1 of the epilogue: out += contraction, bias unused (any valid pointer satisfies the checks)
  return conv_update_impl(cb::RowMask{nullptr, nullptr, nullptr, nullptr, 0}, stream, dtype, gemm, state,
                          state_lo, pitch_in, idx, count, packed_w, (const float*)packed_w, out, pitch_out,
                          B, H, W, Cin, Cout, kH, kW, 2, ws, ws_bytes);
}

int cb_fg_detect(void* stream, const float* x, long long x_sb, long long x_sc, long long x_sy,
                 long long x_sx, float* prev, long long p_sb, long long p_sy, int p_pitch, void* delta_hi,
                 void* delta_lo, uint32_t* raw_bits, int32_t* count, int B, int C, int H, int W,
                 float threshold) {
  CB_CHECK_ARG(x && prev && delta_hi && delta_lo && raw_bits, "fg_detect: null pointer");
  CB_CHECK_ARG(B >= 0 && C > 0 && H >= 0 && W >= 0, "fg_detect: bad shape");
  return cb::launch_fg_detect((cudaStream_t)stream, x, x_sb, x_sc, x_sy, x_sx, prev, p_sb, p_sy, p_pitch,
                              delta_hi, delta_lo, raw_bits, count, B, C, H, W, threshold);
}

int cb_conv_tiled_supported(int dtype, int gemm, int B, int H, int W, int Cin, int Cout, int kH, int kW) {
  if (gemm == CB_GEMM_SIMT_F32) return 0;
  const int Cp = gemm == CB_GEMM_TC_BF16X3 ? cb::pitch16_of(Cin) : cb_channel_pitch(dtype, Cin);
  cb::TilePlan plan;
  cb::umma_tile_plan(plan, dtype, gemm, Cp, B, H, W, Cout, cb_channel_pitch(dtype, Cout), kH, kW, 0);
  if (!plan.ok) return 0;
  return (plan.mma_clk_per_tile <= cb::kTileClkLimit || plan.short_k) ? 1 : 2;
}

static int conv_update_tiled_impl(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                         int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                         const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                         int H, int W, int Cin, int Cout, int kH, int kW, int relu, const cb::PoolFuse& pf,
                         const float* thr_b) {
  CB_CHECK_ARG(state && tile_ws && dil_bits && packed_w && bias && out, "conv_update_tiled: null pointer");
  CB_CHECK_ARG(gemm != CB_GEMM_SIMT_F32, "conv_update_tiled: tensor-core modes only");
  const int want_pitch = gemm == CB_GEMM_TC_BF16X3 ? cb::pitch16_of(Cin) : cb_channel_pitch(dtype, Cin);
  CB_CHECK_ARG(pitch_in == want_pitch, "conv_update_tiled: pitch_in %d != channel pitch %d", pitch_in,
               want_pitch);
  CB_CHECK_ARG(pitch_out >= Cout, "conv_update_tiled: pitch_out < Cout");
  CB_CHECK_ARG(gemm != CB_GEMM_TC_BF16X3 || dtype == CB_F32, "conv_update_tiled: 3xBF16 is for fp32 data");
  if (B == 0 || H == 0 || W == 0) return 0;
  return cb::umma_conv_update_tiled((cudaStream_t)stream, dtype, gemm, state, state_lo, pitch_in,
                                    (const int32_t*)tile_ws, dil_bits, packed_w, bias, out, pitch_out,
                                    B, H, W, Cout, kH, kW, relu, pf, thr_b);
}

int cb_conv_update_tiled(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                         int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                         const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                         int H, int W, int Cin, int Cout, int kH, int kW, int relu) {
  cb::PoolFuse pf;
  memset(&pf, 0, sizeof(pf));
  return conv_update_tiled_impl(stream, dtype, gemm, state, state_lo, pitch_in, tile_ws, dil_bits, packed_w,
                                bias, out, pitch_out, B, H, W, Cin, Cout, kH, kW, relu, pf, nullptr);
}

#ifdef CB_TILE_TRACE
/* debugging aid of trace builds only (tools/tile_trace.py): copy the tile kernel's per-CTA timeline out and clear it */
int cb_debug_tile_trace(long long* dst, int n_ctas) {
  if (n_ctas > 2048) n_ctas = 2048;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(dst, cb::cb_tile_trace, (size_t)n_ctas * cb::TL_TRACE_EV * sizeof(long long));
  static long long zeros[2048 * cb::TL_TRACE_EV];
  cudaMemcpyToSymbol(cb::cb_tile_trace, zeros, sizeof(zeros));
  return cb::TL_TRACE_EV;
}
#endif

int cb_conv_tiled_pool_supported(int dtype, int gemm, int Cout) {
  (void)dtype;
  return gemm != CB_GEMM_SIMT_F32 && cb::tile_pool_ok(gemm, Cout) ? 1 : 0;
}

static int tiled_pool_impl(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                              int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                              const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                              int H, int W, int Cin, int Cout, int kH, int kW, int relu,
                              void* pool_out, long long o_sb, long long o_sy, int o_pitch, int oH, int oW,
                              void* next_state, long long n_sb, long long n_sy, int n_pitch, int aux_mode,
                              void* aux_hi, void* aux_lo, uint32_t* next_raw_bits, float threshold,
                              int update_mode, const float* thr_b) {
  CB_CHECK_ARG(pool_out && next_state && next_raw_bits, "conv_update_tiled_pool: null pointer");
  CB_CHECK_THR(thr_b, "conv_update_tiled_pool");
  CB_CHECK_ARG(update_mode == CB_UPDATE_NONE || update_mode == CB_UPDATE_CHANGED || update_mode == CB_UPDATE_ALL,
               "conv_update_tiled_pool: bad update_mode %d", update_mode);
  const size_t es = cb::esize(dtype);
  const int vec = (int)(16 / es);
  const bool ok = (o_pitch % vec) == 0 && o_pitch == n_pitch && o_pitch >= Cout && pitch_out == o_pitch &&
                  ((o_sy * es) % 16) == 0 && ((n_sy * es) % 16) == 0 && ((o_sb * es) % 16) == 0 &&
                  ((n_sb * es) % 16) == 0 && ((uintptr_t)pool_out % 16) == 0 && ((uintptr_t)next_state % 16) == 0 &&
                  ((uintptr_t)out % 16) == 0;
  CB_CHECK_ARG(ok, "conv_update_tiled_pool: needs pixel-major, 16-byte aligned maps of equal pitch");
  cb::PoolFuse pf;
  memset(&pf, 0, sizeof(pf));
  pf.out = pool_out; pf.o_sb = o_sb; pf.o_sy = o_sy; pf.op = o_pitch; pf.oH = oH; pf.oW = oW;
  pf.nst = next_state; pf.n_sb = n_sb; pf.n_sy = n_sy; pf.np = n_pitch;
  pf.nbits = next_raw_bits; pf.thr = threshold; pf.update = update_mode;
  int rc = 0;
  CB_DISPATCH_DTYPE(dtype, rc = cb::make_aux<T>(pf.aux, aux_mode, aux_hi, aux_lo, next_state, Cout));
  if (rc) return rc;
  return conv_update_tiled_impl(stream, dtype, gemm, state, state_lo, pitch_in, tile_ws, dil_bits, packed_w,
                                bias, out, pitch_out, B, H, W, Cin, Cout, kH, kW, relu, pf, thr_b);
}

int cb_conv_update_tiled_pool_thr(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                                  int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                                  const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                                  int H, int W, int Cin, int Cout, int kH, int kW, int relu,
                                  void* pool_out, long long o_sb, long long o_sy, int o_pitch, int oH, int oW,
                                  void* next_state, long long n_sb, long long n_sy, int n_pitch, int aux_mode,
                                  void* aux_hi, void* aux_lo, uint32_t* next_raw_bits, float threshold,
                                  int update_mode, const float* thr_b) {
  return tiled_pool_impl(stream, dtype, gemm, state, state_lo, pitch_in, tile_ws, dil_bits, packed_w, bias, out,
                         pitch_out, B, H, W, Cin, Cout, kH, kW, relu, pool_out, o_sb, o_sy, o_pitch, oH, oW,
                         next_state, n_sb, n_sy, n_pitch, aux_mode, aux_hi, aux_lo, next_raw_bits, threshold,
                         update_mode, thr_b);
}

int cb_conv_update_tiled_pool(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                              int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                              const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                              int H, int W, int Cin, int Cout, int kH, int kW, int relu,
                              void* pool_out, long long o_sb, long long o_sy, int o_pitch, int oH, int oW,
                              void* next_state, long long n_sb, long long n_sy, int n_pitch, int aux_mode,
                              void* aux_hi, void* aux_lo, uint32_t* next_raw_bits, float threshold,
                              int update_mode) {
  return tiled_pool_impl(stream, dtype, gemm, state, state_lo, pitch_in, tile_ws, dil_bits, packed_w, bias, out,
                         pitch_out, B, H, W, Cin, Cout, kH, kW, relu, pool_out, o_sb, o_sy, o_pitch, oH, oW,
                         next_state, n_sb, n_sy, n_pitch, aux_mode, aux_hi, aux_lo, next_raw_bits, threshold,
                         update_mode, nullptr);
}

int cb_conv_update_masked_streams(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                                  int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                                  const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                                  int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes,
                                  uint32_t* mask_bits, int clear_mask, int32_t* count_out, void* sync_ws,
                                  int32_t* stream_counts, int32_t* stream_acc) {
  CB_CHECK_ARG(mask_bits && sync_ws, "conv_update_masked: null pointer");
  CB_CHECK_STREAMS(stream_counts, stream_acc, "conv_update_masked");
  CB_CHECK_ARG(!stream_counts || gemm != CB_GEMM_SIMT_F32, "conv_update_masked: tensor-core modes only");
  cb::RowMask mk;
  mk.bits = mask_bits;
  mk.clear = clear_mask ? mask_bits : nullptr;
  mk.count_out = count_out;
  mk.sync = (unsigned*)sync_ws;
  mk.nwords = (int)cb_bitmap_words(B, H, W);
  mk.stream_counts = stream_counts;
  mk.stream_acc = stream_acc;
  mk.B = B;
  if (stream_counts && (H == 0 || W == 0))                // nothing is launched below
    if (int rc = zero_stream_counts((cudaStream_t)stream, stream_counts, B, "conv_update_masked")) return rc;
  return conv_update_impl(mk, stream, dtype, gemm, state, state_lo, pitch_in, idx, count, packed_w, bias,
                          out, pitch_out, B, H, W, Cin, Cout, kH, kW, relu ? 1 : 0, ws, ws_bytes);
}

int cb_conv_update_masked(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                          int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                          const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                          int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes,
                          uint32_t* mask_bits, int clear_mask, int32_t* count_out, void* sync_ws) {
  return cb_conv_update_masked_streams(stream, dtype, gemm, state, state_lo, pitch_in, idx, count, packed_w, bias,
                                       out, pitch_out, B, H, W, Cin, Cout, kH, kW, relu, ws, ws_bytes, mask_bits,
                                       clear_mask, count_out, sync_ws, nullptr, nullptr);
}

int cb_tail_supported(int dtype, int gemm, int C0, int C1, int C2) {
  return dtype == CB_F32 && gemm == CB_GEMM_TC_BF16X3 && cb::tail_supported(C0, C1, C2) ? 1 : 0;
}

int cb_tail_update_thr(void* stream, const float* x, float* state1, const void* packed_w1, const float* bias1,
                       float* out1, int relu1, float thr1, float* state2, const void* packed_w2,
                       const float* bias2, float* out2, int pitch_out2, int relu2, float thr2,
                       const int32_t* candidates, const int32_t* n_candidates, int C0, int C1, int C2,
                       int update_mode, int32_t* count1, int32_t* count2, void* sync_ws, int B, int hw,
                       int32_t* stream_counts1, int32_t* stream_acc1, int32_t* stream_counts2,
                       int32_t* stream_acc2, const float* thr1_b, const float* thr2_b) {
  CB_CHECK_ARG(x && state1 && packed_w1 && bias1 && out1 && state2 && packed_w2 && bias2 && out2 && candidates &&
                   n_candidates && count1 && count2 && sync_ws, "tail_update: null pointer");
  CB_CHECK_STREAMS(stream_counts1, stream_acc1, "tail_update");
  CB_CHECK_STREAMS(stream_counts2, stream_acc2, "tail_update");
  CB_CHECK_ARG(!stream_counts1 == !stream_counts2, "tail_update: per-stream counts for both layers or neither");
  CB_CHECK_ARG(!(stream_counts1 || thr1_b || thr2_b) || (B > 0 && hw > 0), "tail_update: bad shape B = %d, H*W = %d",
               B, hw);
  CB_CHECK_THR(thr1_b, "tail_update");
  CB_CHECK_THR(thr2_b, "tail_update");
  CB_CHECK_ARG(update_mode == CB_UPDATE_NONE || update_mode == CB_UPDATE_CHANGED || update_mode == CB_UPDATE_ALL,
               "tail_update: bad update_mode %d", update_mode);
  CB_CHECK_ARG(((uintptr_t)x % 16) == 0 && ((uintptr_t)state1 % 16) == 0 && ((uintptr_t)out1 % 16) == 0 &&
                   ((uintptr_t)state2 % 16) == 0 && ((uintptr_t)out2 % 16) == 0 &&
                   ((uintptr_t)packed_w1 % 128) == 0 && ((uintptr_t)packed_w2 % 128) == 0,
               "tail_update: maps must be 16-byte, packed weights 128-byte aligned");
  cb::TailArgs a;
  a.x = x; a.st1 = state1; a.out1 = out1; a.st2 = state2; a.out2 = out2;
  a.cand = candidates; a.ncand = n_candidates; a.bias1 = bias1; a.bias2 = bias2;
  a.count1 = count1; a.count2 = count2; a.sync = (unsigned*)sync_ws;
  a.xp = C0; a.p1 = C1; a.p2 = pitch_out2; a.C0 = C0; a.C1 = C1; a.C2 = C2;
  a.relu1 = relu1; a.relu2 = relu2; a.update = update_mode; a.thr1 = thr1; a.thr2 = thr2;
  a.sc1 = stream_counts1; a.sc2 = stream_counts2; a.acc1 = stream_acc1; a.acc2 = stream_acc2;
  a.hw = hw; a.B = B;
  return cb::tail_update((cudaStream_t)stream, a, packed_w1, packed_w2, thr1_b, thr2_b);
}

int cb_tail_update_streams(void* stream, const float* x, float* state1, const void* packed_w1, const float* bias1,
                           float* out1, int relu1, float thr1, float* state2, const void* packed_w2,
                           const float* bias2, float* out2, int pitch_out2, int relu2, float thr2,
                           const int32_t* candidates, const int32_t* n_candidates, int C0, int C1, int C2,
                           int update_mode, int32_t* count1, int32_t* count2, void* sync_ws, int B, int hw,
                           int32_t* stream_counts1, int32_t* stream_acc1, int32_t* stream_counts2,
                           int32_t* stream_acc2) {
  return cb_tail_update_thr(stream, x, state1, packed_w1, bias1, out1, relu1, thr1, state2, packed_w2, bias2, out2,
                            pitch_out2, relu2, thr2, candidates, n_candidates, C0, C1, C2, update_mode, count1,
                            count2, sync_ws, B, hw, stream_counts1, stream_acc1, stream_counts2, stream_acc2,
                            nullptr, nullptr);
}

int cb_tail_update(void* stream, const float* x, float* state1, const void* packed_w1, const float* bias1,
                   float* out1, int relu1, float thr1, float* state2, const void* packed_w2,
                   const float* bias2, float* out2, int pitch_out2, int relu2, float thr2,
                   const int32_t* candidates, const int32_t* n_candidates, int C0, int C1, int C2,
                   int update_mode, int32_t* count1, int32_t* count2, void* sync_ws) {
  return cb_tail_update_streams(stream, x, state1, packed_w1, bias1, out1, relu1, thr1, state2, packed_w2, bias2,
                                out2, pitch_out2, relu2, thr2, candidates, n_candidates, C0, C1, C2, update_mode,
                                count1, count2, sync_ws, 0, 0, nullptr, nullptr, nullptr, nullptr);
}

int cb_maxpool2x2(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                  long long x_sy, long long x_sx, const int32_t* idx, const int32_t* count,
                  const uint32_t* dil_bits, void* out, long long o_sb, long long o_sc,
                  long long o_sy, long long o_sx, int B, int C, int H, int W, int oH, int oW) {
  CB_CHECK_ARG(x && idx && count && out, "maxpool2x2: null pointer");
  if (B == 0 || H == 0 || W == 0 || C == 0) return 0;
  const unsigned grid = (unsigned)(sm_count() * 16);
  const size_t es = cb::esize(dtype);
  const int vec = (int)(16 / es);
  // pixel-major fast path: channel-contiguous, 16-byte aligned pixels on both sides.  Chunks that
  // cover pad channels (pitch > C) are processed too: pads are zero on both sides by construction.
  const bool vec_ok = x_sc == 1 && o_sc == 1 && (x_sx % vec) == 0 && (o_sx % vec) == 0 &&
                      x_sx == o_sx && x_sx >= C && x_sx < (1 << 20) && ((x_sy * es) % 16) == 0 &&
                      ((o_sy * es) % 16) == 0 && ((x_sb * es) % 16) == 0 && ((o_sb * es) % 16) == 0 &&
                      ((uintptr_t)x % 16) == 0 && ((uintptr_t)out % 16) == 0 &&
                      (x_sx == C || (C + vec - 1) / vec * vec == x_sx);
  if (vec_ok) {
    const int cpp = (int)(x_sx / vec);
    CB_DISPATCH_DTYPE(dtype, (cb::launch(maxpool2x2_detect_kernel<T, VEC, CB_UPDATE_NONE, false>, grid, 256, 0,
                                         (cudaStream_t)stream, (const T*)x, x_sb, x_sy, (int)x_sx, idx, count,
                                         dil_bits, (T*)out, o_sb, o_sy, (int)o_sx, cpp, cb::group_log2(cpp), H, W,
                                         oH, oW, nullptr, 0ll, 0ll, 0, AuxPlanes{}, nullptr, T{}, nullptr)));
  } else {
    CB_DISPATCH_DTYPE(dtype, (cb::launch(maxpool2x2_kernel<T>, grid, 256, 0, (cudaStream_t)stream, 
                                 (const T*)x, x_sb, x_sc, x_sy, x_sx, idx, count, dil_bits, (T*)out,
                                 o_sb, o_sc, o_sy, o_sx, C, H, W, oH, oW)));
  }
  CB_CHECK_LAUNCH("maxpool2x2");
  return 0;
}

int cb_maxpool2x2_detect_thr(void* stream, int dtype, const void* x, long long x_sb, long long x_sy,
                             int x_pitch, const int32_t* idx, const int32_t* count,
                             const uint32_t* dil_bits, void* out, long long o_sb, long long o_sy,
                             int o_pitch, int B, int C, int H, int W, int oH, int oW, void* next_state,
                             long long n_sb, long long n_sy, int n_pitch, int aux_mode, void* aux_hi,
                             void* aux_lo, uint32_t* next_raw_bits, float threshold, int update_mode,
                             const float* thr_b) {
  CB_CHECK_ARG(x && idx && count && dil_bits && out && next_state && next_raw_bits,
               "maxpool2x2_detect: null pointer");
  CB_CHECK_THR(thr_b, "maxpool2x2_detect");
  if (B == 0 || H == 0 || W == 0 || C == 0) return 0;
  const size_t es = cb::esize(dtype);
  const int vec = (int)(16 / es);
  const bool ok = (x_pitch % vec) == 0 && x_pitch == o_pitch && o_pitch == n_pitch && x_pitch >= C &&
                  (C + vec - 1) / vec * vec == x_pitch && ((x_sy * es) % 16) == 0 &&
                  ((o_sy * es) % 16) == 0 && ((n_sy * es) % 16) == 0 && ((x_sb * es) % 16) == 0 &&
                  ((o_sb * es) % 16) == 0 && ((n_sb * es) % 16) == 0 && ((uintptr_t)x % 16) == 0 &&
                  ((uintptr_t)out % 16) == 0 && ((uintptr_t)next_state % 16) == 0;
  CB_CHECK_ARG(ok, "maxpool2x2_detect: needs pixel-major, 16-byte aligned tensors of equal pitch");
  const int cpp = x_pitch / vec;
  const int glog = cb::group_log2(cpp);
  const unsigned grid = (unsigned)(sm_count() * 16);
  cudaStream_t s = (cudaStream_t)stream;
  return dispatch_thr(thr_b, [&](auto R) { return dispatch_update(update_mode, "maxpool2x2_detect", [&](auto U) {
    CB_DISPATCH_DTYPE(dtype, {
      AuxPlanes aux;
      if (int rc = make_aux<T>(aux, aux_mode, aux_hi, aux_lo, next_state, C)) return rc;
      cb::launch(maxpool2x2_detect_kernel<T, VEC, U, true, R>, grid, 256, 0, s, (const T*)x, x_sb, x_sy, x_pitch, idx,
                 count, dil_bits, (T*)out, o_sb, o_sy, o_pitch, cpp, glog, H, W, oH, oW, (T*)next_state, n_sb,
                 n_sy, n_pitch, aux, next_raw_bits, thr_cast<T>(threshold), thr_b);
    })
    CB_CHECK_LAUNCH("maxpool2x2_detect");
    return 0;
  }); });
}

int cb_maxpool2x2_detect(void* stream, int dtype, const void* x, long long x_sb, long long x_sy,
                         int x_pitch, const int32_t* idx, const int32_t* count,
                         const uint32_t* dil_bits, void* out, long long o_sb, long long o_sy,
                         int o_pitch, int B, int C, int H, int W, int oH, int oW, void* next_state,
                         long long n_sb, long long n_sy, int n_pitch, int aux_mode, void* aux_hi,
                         void* aux_lo, uint32_t* next_raw_bits, float threshold, int update_mode) {
  return cb_maxpool2x2_detect_thr(stream, dtype, x, x_sb, x_sy, x_pitch, idx, count, dil_bits, out, o_sb, o_sy,
                                  o_pitch, B, C, H, W, oH, oW, next_state, n_sb, n_sy, n_pitch, aux_mode, aux_hi,
                                  aux_lo, next_raw_bits, threshold, update_mode, nullptr);
}

int cb_reset_streams(void* stream, const uint8_t* mask, int B, const cb_reset_segment* segments,
                     int n_segments) {
  CB_CHECK_ARG(B > 0 && B <= 65535, "reset_streams: B = %d out of [1, 65535]", B);
  CB_CHECK_ARG(n_segments >= 0, "reset_streams: negative segment count %d", n_segments);
  CB_CHECK_ARG(mask && (n_segments == 0 || segments), "reset_streams: null pointer");
  for (int i = 0; i < n_segments; ++i) {
    const cb_reset_segment& g = segments[i];
    CB_CHECK_ARG(g.dtype == CB_F32 || g.dtype == CB_F16 || g.dtype == CB_BF16,
                 "reset_streams: segment %d: bad dtype %d", i, g.dtype);
    const int es = cb::esize(g.dtype);
    CB_CHECK_ARG(g.fill == CB_RESET_FILL_ZERO || g.fill == CB_RESET_FILL_INF,
                 "reset_streams: segment %d: bad fill %d", i, g.fill);
    CB_CHECK_ARG(g.pixels >= 0 && g.pitch_bytes > 0 && g.pitch_bytes % es == 0,
                 "reset_streams: segment %d: pixels %lld, pitch %d bytes", i, g.pixels, g.pitch_bytes);
    CB_CHECK_ARG(g.channel_bytes >= 0 && g.channel_bytes % es == 0 && g.channel_bytes <= g.pitch_bytes,
                 "reset_streams: segment %d: %d channel bytes in a %d-byte pitch", i, g.channel_bytes,
                 g.pitch_bytes);
    CB_CHECK_ARG(g.pixels <= (1ll << 62) / g.pitch_bytes / B, "reset_streams: segment %d too large", i);
    CB_CHECK_ARG(g.pixels == 0 || (g.base && (uintptr_t)g.base % es == 0),
                 "reset_streams: segment %d: base not aligned to its %d-byte elements", i, es);
  }
  static const unsigned kInf[3] = {0x7f800000u, 0x7c00u, 0x7f80u};      // fp32, fp16, bf16
  cb::ResetBatch rb;
  rb.n = 0;
  rb.cta0[0] = 0;
  for (int i = 0; i <= n_segments; ++i) {
    const bool more = i < n_segments;
    long long slice = 0, ctas = 0;
    if (more) {
      slice = segments[i].pixels * segments[i].pitch_bytes;
      ctas = (slice + cb::kResetChunksPerCta * 16 - 1) / (cb::kResetChunksPerCta * 16);
      if (ctas == 0) continue;                                            // empty segment
    }
    // launch what is collected when the batch is full, the grid would grow past 2^31 - 1, or at the end
    if (rb.n > 0 && (!more || rb.n == cb::kResetMaxSegs || rb.cta0[rb.n] + ctas > 0x7fffffffll)) {
      cb::launch(reset_streams_kernel, dim3(rb.cta0[rb.n], (unsigned)B), dim3(cb::kResetThreads), 0,
                 (cudaStream_t)stream, rb, mask);
      CB_CHECK_LAUNCH("reset_streams");
      rb.n = 0;
    }
    if (!more) break;
    CB_CHECK_ARG(ctas <= 0x7fffffffll, "reset_streams: segment %d too large for one grid", i);
    const cb_reset_segment& g = segments[i];
    cb::ResetSeg& s = rb.seg[rb.n];
    s.base = (char*)g.base;
    s.slice = slice;
    s.fill = g.fill == CB_RESET_FILL_INF ? kInf[g.dtype] : 0u;
    s.pitch = g.pitch_bytes;
    s.chan = g.channel_bytes;
    s.es = cb::esize(g.dtype);
    rb.cta0[rb.n + 1] = rb.cta0[rb.n] + (unsigned)ctas;
    ++rb.n;
  }
  return 0;
}

int cb_gen_xmatrix(void* stream, int dtype, void* columns, const void* input, const int32_t* idx,
                   int kW, int kH, int C, int W, int H, int n) {
  if (n <= 0) return 0;
  CB_CHECK_ARG(columns && input && idx, "gen_xmatrix: null pointer");
  const long long total = (long long)n * C * kH * kW;
  CB_DISPATCH_DTYPE(dtype, (cb::launch(gen_xmatrix_kernel<T>, grid_for(total, 256, 16), 256, 0, (cudaStream_t)stream, 
                               (T*)columns, (const T*)input, idx, kW, kH, C, W, H, n)));
  CB_CHECK_LAUNCH("gen_xmatrix");
  return 0;
}

int cb_matrix_mult(void* stream, int dtype, const void* X, const void* weight, const void* bias,
                   void* Y, int n, int K, int Cout) {
  if (n <= 0) return 0;
  CB_CHECK_ARG(X && weight && bias && Y, "matrix_mult: null pointer");
  dim3 grid((Cout + 31) / 32, (n + 31) / 32);
  CB_CHECK_ARG(grid.y < 65536, "matrix_mult: n too large for the staged op");
  CB_DISPATCH_DTYPE(dtype, (cb::launch(matrix_mult_kernel<T>, grid, 256, 0, (cudaStream_t)stream, 
                               (const T*)X, (const T*)weight, (const T*)bias, (T*)Y, n, K, Cout)));
  CB_CHECK_LAUNCH("matrix_mult");
  return 0;
}

int cb_update_output(void* stream, int dtype, const void* Yt, void* output, const int32_t* idx,
                     int numOutputPixel, int n, int Cout, int relu) {
  if (n <= 0) return 0;
  CB_CHECK_ARG(Yt && output && idx, "update_output: null pointer");
  const long long total = (long long)n * Cout;
  CB_DISPATCH_DTYPE(dtype, (cb::launch(update_output_kernel<T>, grid_for(total, 256, 16), 256, 0, (cudaStream_t)stream, 
                               (const T*)Yt, (T*)output, idx, numOutputPixel, n, Cout, relu)));
  CB_CHECK_LAUNCH("update_output");
  return 0;
}

int cb_fg_update(void* stream, const float* x, float* prev, const float* weight, float* out,
                 int32_t* count, int B, int Cin, int Cout, int H, int W, int kH, int kW,
                 float threshold) {
  CB_CHECK_ARG(x && prev && weight && out && count, "fg_update: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(count, 0, sizeof(int32_t), s);
  const long long total = (long long)B * Cin * H * W;
  if (total == 0) return 0;
  cb::launch(fg_update_kernel, grid_for((total + 31) / 32 * 32, 256, 8), 256, 0, s, x, prev, weight, out, count, B, Cin,
                                                             Cout, H, W, kH, kW, threshold);
  CB_CHECK_LAUNCH("fg_update");
  return 0;
}

/* ---- frame ingest: resizing on the device (ingest.cuh) -------------------------------------------- */
size_t cb_resize_ws_bytes(int sH, int sW, int dH, int dW, int C) {
  if (sH <= 0 || sW <= 0 || dH <= 0 || dW <= 0 || C <= 0) return 0;
  return cb::resize_plan(sH, sW, dH, dW, C).bytes;
}

int cb_resize_bicubic_u8_init(void* stream, void* ws, int sH, int sW, int dH, int dW, int C) {
  CB_CHECK_ARG(ws && sH > 0 && sW > 0 && dH > 0 && dW > 0 && C >= 1 && C <= 4,
               "resize_bicubic_u8_init: bad arguments (1..4 channels)");
  const cb::ResizePlan p = cb::resize_plan(sH, sW, dH, dW, C);
  CB_CHECK_ARG(p.off_tmp < (1ull << 31), "resize_bicubic_u8_init: image too large");
  // the weight tables are a function of the four sizes only: computed here in double exactly as Pillow's
  // precompute_coeffs / normalize_coeffs_8bpc do, copied once; cb_resize_bicubic_u8 is then launch-only
  std::vector<int32_t> host(p.off_tmp / 4, 0);
  host[0] = p.ksize_x; host[1] = p.ksize_y; host[2] = sH; host[3] = sW; host[4] = dH; host[5] = dW; host[6] = C;
  cb::resize_coeffs(sW, dW, p.ksize_x, host.data() + p.off_bx / 4, host.data() + p.off_kx / 4);
  cb::resize_coeffs(sH, dH, p.ksize_y, host.data() + p.off_by / 4, host.data() + p.off_ky / 4);
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemcpyAsync(ws, host.data(), p.off_tmp / 4 * 4, cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return cb::fail(3, "resize_bicubic_u8_init: copying the weight tables failed: %s",
                    cudaGetErrorString(cudaGetLastError()));
  return 0;
}

int cb_resize_bicubic_u8(void* stream, const uint8_t* src, long long s_y, long long s_x, long long s_c,
                         uint8_t* dst, long long d_y, long long d_x, long long d_c, void* ws, int sH, int sW,
                         int dH, int dW, int C) {
  CB_CHECK_ARG(src && dst && ws && sH > 0 && sW > 0 && dH > 0 && dW > 0 && C >= 1 && C <= 4,
               "resize_bicubic_u8: bad arguments (1..4 channels)");
  const cb::ResizePlan p = cb::resize_plan(sH, sW, dH, dW, C);
  char* w = (char*)ws;
  uint8_t* tmp = (uint8_t*)(w + p.off_tmp);                    // [sH, dW, C] interleaved
  cudaStream_t s = (cudaStream_t)stream;
  cb::launch(cb::resize_pass_u8_kernel<1>, dim3((unsigned)((dW + 255) / 256), (unsigned)sH), dim3(256), 0, s, src,
                 s_y, s_x, s_c, tmp, (long long)dW * C, (long long)C, 1ll, sH, dW, C,
                 (const int32_t*)(w + p.off_bx), (const int32_t*)(w + p.off_kx), p.ksize_x);
  CB_CHECK_LAUNCH("resize_bicubic_u8(horizontal)");
  cb::launch(cb::resize_pass_u8_kernel<0>, dim3((unsigned)((dW + 255) / 256), (unsigned)dH), dim3(256), 0, s,
                 (const uint8_t*)tmp, (long long)dW * C, (long long)C, 1ll, dst, d_y, d_x, d_c, dH, dW, C,
                 (const int32_t*)(w + p.off_by), (const int32_t*)(w + p.off_ky), p.ksize_y);
  CB_CHECK_LAUNCH("resize_bicubic_u8(vertical)");
  return 0;
}

int cb_resize_bilinear_u8(void* stream, const uint8_t* src, long long s_y, long long s_x, long long s_c, int sH,
                          int sW, float* dst, long long d_y, long long d_x, long long d_c, int dH, int dW, int C,
                          float divisor, float cval, float clip_lo, float clip_hi) {
  CB_CHECK_ARG(src && dst && sH > 0 && sW > 0 && dH > 0 && dW > 0 && C >= 1 && divisor != 0.f,
               "resize_bilinear_u8: bad arguments");
  cb::launch(cb::resize_bilinear_kernel, dim3((unsigned)((dW + 255) / 256), (unsigned)dH), dim3(256), 0,
                 (cudaStream_t)stream, src, s_y, s_x, s_c, sH, sW, dst, d_y, d_x, d_c, dH, dW, C, (double)divisor,
                 (double)cval, (double)clip_lo, (double)clip_hi);
  CB_CHECK_LAUNCH("resize_bilinear_u8");
  return 0;
}

}  // extern "C"
