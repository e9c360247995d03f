/*
 * cbinfer_b200.h -- C ABI of libcbinfer_sm100.so, the B200 (sm_100a) backend behind the
 * pycbinfer surface.  Plain pointers and sizes only; no torch types.  This is the boundary the
 * reference crosses with cffi in pycbinfer/conv2d_cg.py:6-50 and pycbinfer/conv2d_fg.py:12-32;
 * each entry point names the reference symbol(s) it replaces.
 *
 * Conventions
 *   - every function returns 0 on success and a non-zero code on failure; the message is
 *     available from cb_last_error() (the reference launchers are `void` and unchecked,
 *     cbconv2d_cg_backend.cu:83-99).
 *   - `stream` is a cudaStream_t passed as void* (the reference launches on the legacy default
 *     stream).  All work is asynchronous on that stream; nothing synchronises the host.
 *   - launch geometry is the library's business: the reference's gridz..blockx arguments
 *     (conv2d_cg.py:7,17,23,31,35) are gone.
 *   - all memory is caller-owned, including workspaces (same ownership rule as the reference,
 *     where python allocates changeMap / XMatrix / state, conv2d_cg.py:105,249).
 *   - dtype codes: CB_F32 = 0, CB_F16 = 1, CB_BF16 = 2 (the reference selects between twin
 *     libraries with identical symbols instead, conv2d_cg.py:73,109,252,302).
 *   - tensors are described by a base pointer plus element strides (sb, sc, sy, sx) for the
 *     batch, channel, row and column dimension, so both the reference's planar NCHW layout
 *     (sc = H*W, sy = W, sx = 1) and the backend's native pixel-major layout (sc = 1,
 *     sx = pitch, sy = W*pitch) are accepted.  "pixel-major" arguments (state of the fused
 *     path) take a single `pitch` (elements per pixel, a multiple of 16 bytes / element size).
 *   - batch: B independent images (video streams).  The reference is batch 1.
 *   - pixel indices are int32, ascending, b*H*W + y*W + x  (reference: y*W+x, conv2d_cg.py:202).
 *   - change bitmaps hold one bit per pixel, row-padded: word (b*H + y) * cb_bitmap_row_words(W)
 *     + x/32, bit x%32.
 */
#ifndef CBINFER_B200_H
#define CBINFER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CB_F32 0
#define CB_F16 1
#define CB_BF16 2

/* how cb_change_detect maintains the previous-input state */
#define CB_UPDATE_NONE 0     /* leave state untouched (updateInputState=false, no copy)        */
#define CB_UPDATE_CHANGED 1  /* feedback loop: state[:,p] = in[:,p] at own-changed pixels only  */
#define CB_UPDATE_ALL 2      /* state = in everywhere (the prevInput.copy_(input) of conv2d.py:236) */

/* arithmetic of the contraction in cb_conv_update */
#define CB_GEMM_SIMT_F32 0   /* fp32 FFMA on CUDA cores (exact-fp32 products)                   */
#define CB_GEMM_TC 1         /* tcgen05: 1xTF32 for fp32 data, f16/bf16 for 16-bit data          */
#define CB_GEMM_TC_3X 2      /* tcgen05: 3xTF32 split (fp32-accurate, ~2e-6) for fp32 data       */
#define CB_GEMM_TC_BF16X3 3  /* tcgen05: 3xBF16 split of fp32 data (hi/lo bf16 pairs, ~2e-5) at
                                twice the tensor rate and half the bytes of 3xTF32                */

/* auxiliary operand planes cb_change_detect keeps in step with an fp32 state */
#define CB_AUX_NONE 0
#define CB_AUX_TF32_LO 1     /* aux_lo: fp32 plane v - trunc_tf32(v), same strides as the state    */
#define CB_AUX_BF16_PAIR 2   /* aux_hi / aux_lo: bf16 planes bf16(v), bf16(v - hi); pixel-major,
                                pitch = cb_plane_pitch16(C): 4 for C <= 4, else C rounded up to 8  */

/* ---- library ---------------------------------------------------------------------------- */
int cb_version(void);
const char* cb_last_error(void);
/* number of SMs / compute capability of the current device */
int cb_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- sizes ------------------------------------------------------------------------------ */
int cb_bitmap_row_words(int W);                       /* ceil(W/32)                             */
size_t cb_bitmap_words(int B, int H, int W);          /* B*H*ceil(W/32)                         */
size_t cb_compact_ws_bytes(int B, int H, int W);      /* workspace of cb_dilate_compact         */
int cb_channel_pitch(int dtype, int C);               /* C rounded up to 16 bytes               */
int cb_plane_pitch16(int C);                          /* pitch of the CB_AUX_BF16_PAIR planes   */
size_t cb_packed_weight_bytes(int dtype, int gemm, int Cout, int Cin, int kH, int kW);

/* ---- change detection ---------------------------------------------------------------------
 * replaces: changeDetection (conv2d_cg.py:7-13 -> cbconv2d_cg_backend.cu:6-100, half: :10-108),
 *           detection half only; the dilation lives in cb_dilate_compact.
 * raw_bits[word] bit = OR_c ( |state - x| > thr )   strict '>', fp32 flush-to-zero, fp16/bf16:
 * rounded difference vs rounded threshold, two one-sided tests (half.cu:58-63).
 * The whole bitmap (incl. row padding bits = 0) is written; no pre-zeroing needed.
 * aux_mode / aux_hi / aux_lo (fp32 only): auxiliary operand planes written wherever the state is
 * written (CB_AUX_*), consumed by cb_conv_update, so the operand split of the 3x modes is paid
 * once per accepted pixel instead of once per gathered filter tap. */
int cb_change_detect(void* stream, int dtype,
                     const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                     void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                     int aux_mode, void* aux_hi, void* aux_lo, uint32_t* raw_bits, int B, int C,
                     int H, int W, float threshold, int update_mode);

/* ---- uint8 frame ingest --------------------------------------------------------------------
 * cb_change_detect for a uint8 frame (camera / decoder output; strides in bytes, HWC or planar)
 * against a pixel-major fp32 state of pitch 4 (C <= 4).  The frame value is
 *   v = (float)u8 / divisor + bias      (IEEE division and addition, no contraction)
 * which is the normalisation the reference's readers apply on the host before the first layer:
 * /255 (sceneLabeling/videoSequenceReader.py:65), /256 - 0.5 (openPose/PoseDetector.py:72).
 * Bit-identical to cb_change_detect on the host-normalised fp32 frame; a quarter of the bytes
 * cross PCIe.  No reference counterpart (SURVEY.md 8f rank 4: detection on uint8 frames). */
int cb_change_detect_u8(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                        long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                        long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                        uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                        float threshold, int update_mode);

/* ---- active-stream mask ----------------------------------------------------------------------
 * cb_change_detect / cb_change_detect_u8 with an active-stream mask: active is uint8[B] in device
 * memory, read on the device (capturable in a CUDA graph), or NULL = every stream (then exactly the
 * plain entry points, which forward here with NULL).  For a stream b with active[b] == 0 the call
 * writes b's bitmap words as 0 and neither reads b's slice of x nor reads or writes b's state and
 * operand planes: b is skipped for this frame, as if it had been fed its previous frame again.  The
 * other streams are computed exactly as without the mask.  No reference counterpart (the reference
 * is batch 1; DESIGN.md section 3.13). */
int cb_change_detect_streams(void* stream, int dtype,
                             const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                             void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                             int aux_mode, void* aux_hi, void* aux_lo, uint32_t* raw_bits, int B, int C,
                             int H, int W, float threshold, int update_mode,
                             const uint8_t* active /* [B], device; 0 = skip; NULL = all */);
int cb_change_detect_u8_streams(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                                long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                                long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                                uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                                float threshold, int update_mode,
                                const uint8_t* active /* [B], device; 0 = skip; NULL = all */);

/* ---- propagation + compaction -------------------------------------------------------------
 * replaces: the scatter-dilate inside changeDetection_kernel (cbconv2d_cg_backend.cu:62-72),
 *           changePropagation (conv2d_cg.py:15-19 -> cbconv2d_cg_backend.cu:101-136) and
 *           changeIndexesExtr / torch.nonzero(...).int() (conv2d_cg.py:200-213) incl. its host
 *           sync: the count stays on the device.
 * Dilates raw_bits by (2*kHHalf+1)x(2*kWHalf+1) inside each image, then writes
 *   dil_bits (optional, may be NULL; may NOT alias raw_bits), dil_map (optional int8 [B,H,W]),
 *   idx[0..n) ascending, *count = n.   `ws` is cb_compact_ws_bytes() of zero-initialised
 * (once, at allocation) device memory private to the calling stream; the kernel leaves it
 * clean for the next call.  clear_raw != 0: raw_bits is zeroed once every tile has consumed it, so
 * a following cb_change_detect_sparse(bits_are_clear = 1) needs no memset. */
int cb_dilate_compact(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int8_t* dil_map,
                      int32_t* idx, int32_t* count, void* ws, int B, int H, int W, int kHHalf,
                      int kWHalf, int clear_raw);

/* cb_dilate_compact that also lists the dirty 8 x 16 output tiles (x 8 wide, y 16 tall, aligned to
 * the image origin) for cb_conv_update_tiled: tile_ws = cb_tile_ws_bytes(B,H,W) of device memory,
 * zeroed once at allocation, private to the stream; after the call word [1] holds the number of
 * tiles that contain at least one set bit of the dilated map and the (unordered) tile list sits
 * behind the stamps.  No reference counterpart (the reference gathers per changed pixel,
 * cbconv2d_cg_backend.cu:138-161). */
size_t cb_tile_ws_bytes(int B, int H, int W);
int cb_dilate_compact_tiles(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits,
                            int8_t* dil_map, int32_t* idx, int32_t* count, void* ws, void* tile_ws,
                            int B, int H, int W, int kHHalf, int kWHalf, int clear_raw);

/* cb_dilate_compact_tiles without the ordered index list: dilated bitmap (dil_bits, required), dirty
 * tile list (tile_ws) and *count = number of dilated pixels.  For layers whose only consumers walk
 * tiles (cb_conv_update_tiled[_pool]): no scan across the bitmap, no index expansion.  An ordered
 * list can still be produced later from dil_bits with cb_dilate_compact(kHHalf = kWHalf = 0). */
int cb_dilate_tiles(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int32_t* count, void* ws,
                    void* tile_ws, int B, int H, int W, int kHHalf, int kWHalf, int clear_raw);

/* ---- candidate ("sparse") detection ---------------------------------------------------------
 * Same per-pixel test and state maintenance as cb_change_detect, evaluated only at the
 * `*n_candidates` pixels listed in `candidates` (indices b*H*W + y*W + x, any order); raw_bits is
 * cleared and the bits of the changed candidates are set.  No reference counterpart: the reference
 * re-scans every layer's whole input (conv2d.py:222-224).  Equal to the dense scan whenever x is
 * untouched outside the candidate set, the threshold was not lowered since the previous frame and
 * the state is not fresh -- conditions the calling module checks (see CBConv2d.candidateDetect). */
int cb_change_detect_sparse(void* stream, int dtype,
                            const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                            void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                            int aux_mode, void* aux_hi, void* aux_lo,
                            const int32_t* candidates, const int32_t* n_candidates,
                            uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                            int update_mode, int bits_are_clear);

/* Small maps (bitmap of at most cb_compact_small_max_words() words, e.g. one 368 x 368 map or eight
 * 46 x 46 maps): cb_change_detect_sparse and cb_dilate_compact in ONE launch -- the last block of the
 * detection kernel dilates and compacts the bitmap (dil_bits optional, idx / count as cb_dilate_compact,
 * sync_ws = 4 bytes of zeroed device memory, left zero).  Same results as the two calls; a layer on a
 * small map is bound by its dependent-launch chain (reference: ~10 launches + a host sync per layer,
 * conv2d.py:222-251), so this takes it from three launches per frame to two.  Pixel-major tensors. */
int cb_compact_small_max_words(void);
int cb_change_detect_sparse_compact(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                    long long x_sy, long long x_sx, void* state, long long s_sb,
                                    long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                    void* aux_hi, void* aux_lo, const int32_t* candidates,
                                    const int32_t* n_candidates, uint32_t* raw_bits, int B, int C, int H,
                                    int W, float threshold, int update_mode, int bits_are_clear,
                                    uint32_t* dil_bits, int32_t* idx, int32_t* count, void* sync_ws,
                                    int kHHalf, int kWHalf, int clear_raw);

/* 2x2/stride-2 pooled view of a change bitmap, compacted: out bit (yo,xo) = OR of the input bits
 * of window (yo,xo); writes out_bits (optional), idx[0..n) ascending at pooled resolution
 * [B,oH,oW] and *count.  Hands change candidates across a CBPoolMax2d (the reference forwards the
 * input-resolution indices unchanged, conv2d.py:75-76, which no consumer can use).
 * ws: cb_compact_ws_bytes(B,oH,oW), same rules as cb_dilate_compact. */
int cb_pool_compact(void* stream, const uint32_t* in_bits, uint32_t* out_bits, int32_t* idx,
                    int32_t* count, void* ws, int B, int H, int W, int oH, int oW);

/* int8/bool map [B,H,W] (non-zero = set) -> bitmap.  Lets callers that hold a reference-style
 * changeMap (conv2d_cg.py:105) use cb_dilate_compact as changePropagation / changeIndexesExtr. */
int cb_map_to_bits(void* stream, const int8_t* map, uint32_t* bits, int B, int H, int W);

/* ---- fused gather + contraction + bias/ReLU + scatter -------------------------------------
 * replaces: genXMatrix (conv2d_cg.py:21-27 -> cbconv2d_cg_backend.cu:138-173),
 *           matrixMult_python / cuBLAS (conv2d_cg.py:342-349), the transpose copy
 *           (conv2d.py:247, conv2d_cg.py:305) and updateOutput (conv2d_cg.py:29-31 ->
 *           cbconv2d_cg_backend.cu:175-197).  X and Y are never materialised.
 * For j < *count: out[idx[j], co] = act( bias[co] + sum_{ky,kx,ci} W[co,ci,ky,kx] *
 *                                        state[pixel idx[j] + (ky-kH/2, kx-kW/2), ci] )
 * with zero outside the image and act = ReLU iff relu (v <= 0 -> 0, cg.cu:187).
 * state / out are pixel-major with the given pitches; bias is fp32[Cout]; packed_w comes from
 * cb_pack_weights with the same dtype/gemm/shape.  *count is read on the device.
 * Operands per mode: CB_GEMM_SIMT_F32 / CB_GEMM_TC: `state` only.  CB_GEMM_TC_3X (fp32): `state`
 * plus `state_lo` = the CB_AUX_TF32_LO plane.  CB_GEMM_TC_BF16X3 (fp32 output): `state` and
 * `state_lo` are the CB_AUX_BF16_PAIR planes (hi, lo) and pitch_in is their pitch.
 * ws / ws_bytes: optional stream-K workspace (cb_conv_ws_bytes() of device memory, zeroed once at
 * allocation, private to the calling stream; the kernel leaves it clean).  With it the tensor-core
 * path cuts the (tile, K block) space into equal shares per CTA, so the run time follows the
 * change count instead of jumping at tile-wave boundaries; NULL keeps whole tiles per CTA. */
size_t cb_conv_ws_bytes(void);
int cb_pack_weights(void* stream, int dtype, int gemm, const void* weight /*[Cout,Cin,kH,kW]*/,
                    void* packed, int Cout, int Cin, int kH, int kW);
int cb_conv_update(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                   int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                   const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                   int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes);

/* cb_conv_update for spatially clustered change sets (same result, same operands): the work unit
 * is a dirty 8 x 16 output tile from cb_dilate_compact_tiles' tile_ws; the tile's receptive-field
 * halo of `state` is staged ONCE in shared memory by TMA (cp.async.bulk.tensor, zero fill outside
 * the image) and the tensor cores read the im2col rows straight out of it through their
 * shared-memory descriptors; only pixels whose bit is set in dil_bits (the dilated change bitmap
 * of the same cb_dilate_compact_tiles call) are written.  Replaces genXMatrix
 * (cbconv2d_cg_backend.cu:138-161) + GEMM + updateOutput (:175-189) like cb_conv_update.
 * cb_conv_tiled_supported: 1 if the layer shape can run on this path AND its per-tile tensor work
 * is small enough for whole-tile granularity to pay (else use cb_conv_update), 2 if it can run
 * but is not recommended, 0 if unsupported (1x1 filters, operand pixels that are not 16/32/64 or a
 * multiple of 128 bytes).  Tensor-core gemm modes only. */
int cb_conv_tiled_supported(int dtype, int gemm, int B, int H, int W, int Cin, int Cout, int kH, int kW);
int cb_conv_update_tiled(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                         int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                         const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                         int H, int W, int Cin, int Cout, int kH, int kW, int relu);

/* cb_conv_update_tiled + the change-based 2x2 / stride-2 max pooling of its output (reference
 * maxPool2d, conv2d_cg.py:58-82 -> cbconv2d_cg_backend.cu:199-227) + the NEXT layer's change detection
 * on the re-pooled pixels, i.e. cb_conv_update_tiled followed by cb_maxpool2x2_detect, in ONE launch:
 * the epilogue that scatters a tile's rows also takes the 2x2 maxima of its 4 x 8 windows (pixels
 * of a touched window that were not recomputed are read back from `out`), writes pool_out,
 * thresholds against next_state, ORs the change bits into next_raw_bits (kept clear by the caller)
 * and maintains next_state / its operand planes per update_mode.  Needs Cout <= 64, Cout % 16 == 0
 * (cb_conv_tiled_pool_supported) and pixel-major maps of equal pitch. */
int cb_conv_tiled_pool_supported(int dtype, int gemm, int Cout);
int cb_conv_update_tiled_pool(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                              int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                              const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                              int H, int W, int Cin, int Cout, int kH, int kW, int relu,
                              void* pool_out, long long o_sb, long long o_sy, int o_pitch, int oH, int oW,
                              void* next_state, long long n_sb, long long n_sy, int n_pitch, int aux_mode,
                              void* aux_hi, void* aux_lo, uint32_t* next_raw_bits, float threshold,
                              int update_mode);

/* cb_conv_update over a SUPERSET index list: a listed pixel is processed only if its bit is set in
 * `mask_bits` (a raw change bitmap, e.g. what cb_change_detect_sparse just wrote for a 1x1 layer
 * whose candidates were idx/count).  Layers that need no dilation can then skip the ordered
 * compaction between detection and contraction (no reference counterpart; the reference runs
 * torch.nonzero there, conv2d_cg.py:200-213).  *count_out = number of processed pixels;
 * clear_mask != 0: the bitmap is zeroed once every CTA has consumed it.  sync_ws: 8 bytes of
 * device memory zeroed once by the caller (left clean).  Tensor-core modes only. */
int cb_conv_update_masked(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                          int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                          const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                          int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes,
                          uint32_t* mask_bits, int clear_mask, int32_t* count_out, void* sync_ws);

/* ---- two chained 1x1 layers in one launch ---------------------------------------------------
 * The trailing pointwise layers of a network on the candidate path (e.g. 256 -> 64 (+ReLU) -> 8):
 * per candidate pixel (the pixels the upstream layer just rewrote, `candidates`/`n_candidates`)
 *   layer 1: threshold x against state1 (cb_change_detect_sparse semantics, strict >), accept
 *            changed pixels into state1 (update_mode CB_UPDATE_CHANGED = feedback, CB_UPDATE_ALL =
 *            copy), out1[p] = act(bias1 + W1 . x[p]) for the changed ones;
 *   layer 2: threshold out1[p] against state2 for those pixels, accept, out2[p] = act(bias2 + W2 . out1[p]).
 * Replaces, per layer, changeDetection + nonzero + genXMatrix + GEMM + updateOutput
 * (pycbinfer/conv2d.py:222-251) -- here: cb_change_detect_sparse + cb_conv_update_masked twice --
 * with bit-identical results (same K order and 3xBF16 split).  fp32 pixel-major maps whose pitch
 * equals the channel count (C0 % 64 == 0, C0 <= 256; C1 in {16,32,64}; C2 <= 16, pitch_out2 % 4 == 0);
 * packed weights from cb_pack_weights(CB_F32, CB_GEMM_TC_BF16X3, ...).  *count1 / *count2 = pixels
 * each layer updated.  sync_ws: 12 bytes zeroed once (left clean).  The layers' operand planes
 * (CB_AUX_BF16_PAIR) are NOT maintained: rebuild them before using cb_conv_update on these layers. */
int cb_tail_supported(int dtype, int gemm, int C0, int C1, int C2);
int cb_tail_update(void* stream, const float* x, float* state1, const void* packed_w1, const float* bias1,
                   float* out1, int relu1, float thr1, float* state2, const void* packed_w2,
                   const float* bias2, float* out2, int pitch_out2, int relu2, float thr2,
                   const int32_t* candidates, const int32_t* n_candidates, int C0, int C1, int C2,
                   int update_mode, int32_t* count1, int32_t* count2, void* sync_ws);

/* ---- per-stream change counts ---------------------------------------------------------------
 * The *_streams entry points are the calls above plus one row of per-stream counts: on every call
 * (also one with nothing to do) stream_counts[b], b < B, is set to the part of the call's count that
 * lies in stream b -- pixel p belongs to stream p / (H*W) -- so the row sums to *count:
 *   cb_dilate_compact / _tiles / cb_dilate_tiles and cb_change_detect_sparse_compact: dilated pixels;
 *   cb_conv_update_masked: processed pixels (*count_out; tensor-core modes); cb_tail_update: the pixels
 *   each layer updated (*count1 -> stream_counts1, *count2 -> stream_counts2, B streams of hw pixels).
 * The row is written, never added to, so a CUDA graph needs no memset node for it.  stream_acc is the
 * row's accumulator: int32 [B] of device memory, zeroed once at allocation, private to the row and
 * left zero by every call; a non-NULL stream_counts needs it.  NULL stream_counts = the plain call
 * (the entry points above forward here with NULL).
 * cb_stream_bucket counts an index list the caller did not build with one of these calls (any order,
 * *count read on the device): stream_counts[b] = #{ j < *count : idx[j] / hw == b }, indices outside
 * [0, B*hw) not counted; its stream_acc is int32 [B + 1] (the last word counts finished blocks). */
int cb_dilate_compact_streams(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int8_t* dil_map,
                              int32_t* idx, int32_t* count, void* ws, int B, int H, int W, int kHHalf,
                              int kWHalf, int clear_raw, int32_t* stream_counts, int32_t* stream_acc);
int cb_dilate_compact_tiles_streams(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits,
                                    int8_t* dil_map, int32_t* idx, int32_t* count, void* ws, void* tile_ws,
                                    int B, int H, int W, int kHHalf, int kWHalf, int clear_raw,
                                    int32_t* stream_counts, int32_t* stream_acc);
int cb_dilate_tiles_streams(void* stream, const uint32_t* raw_bits, uint32_t* dil_bits, int32_t* count, void* ws,
                            void* tile_ws, int B, int H, int W, int kHHalf, int kWHalf, int clear_raw,
                            int32_t* stream_counts, int32_t* stream_acc);
int cb_change_detect_sparse_compact_streams(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                            long long x_sy, long long x_sx, void* state, long long s_sb,
                                            long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                            void* aux_hi, void* aux_lo, const int32_t* candidates,
                                            const int32_t* n_candidates, uint32_t* raw_bits, int B, int C, int H,
                                            int W, float threshold, int update_mode, int bits_are_clear,
                                            uint32_t* dil_bits, int32_t* idx, int32_t* count, void* sync_ws,
                                            int kHHalf, int kWHalf, int clear_raw, int32_t* stream_counts,
                                            int32_t* stream_acc);
int cb_conv_update_masked_streams(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                                  int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                                  const float* bias, void* out, int pitch_out, int B, int H, int W, int Cin,
                                  int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes,
                                  uint32_t* mask_bits, int clear_mask, int32_t* count_out, void* sync_ws,
                                  int32_t* stream_counts, int32_t* stream_acc);
int cb_tail_update_streams(void* stream, const float* x, float* state1, const void* packed_w1, const float* bias1,
                           float* out1, int relu1, float thr1, float* state2, const void* packed_w2,
                           const float* bias2, float* out2, int pitch_out2, int relu2, float thr2,
                           const int32_t* candidates, const int32_t* n_candidates, int C0, int C1, int C2,
                           int update_mode, int32_t* count1, int32_t* count2, void* sync_ws, int B, int hw,
                           int32_t* stream_counts1, int32_t* stream_acc1, int32_t* stream_counts2,
                           int32_t* stream_acc2);
int cb_stream_bucket(void* stream, const int32_t* idx, const int32_t* count, int B, int hw,
                     int32_t* stream_counts, int32_t* stream_acc);

/* ---- change-based 2x2/stride-2 max pooling ------------------------------------------------
 * replaces: maxPool2d (conv2d_cg.py:33-37 -> cbconv2d_cg_backend.cu:199-240, half :207-250).
 * For every changed input pixel idx[j] (j < *count) recompute the max of its 2x2 window over
 * all channels (init -inf, window clipped to the input) into out[b, :, y/2, x/2].  Windows whose
 * output coordinate falls outside [oH,oW) are skipped (the reference writes out of bounds there).
 * dil_bits (optional) is the bitmap the indices were compacted from; when given, each window is
 * recomputed once instead of up to four times. */
int cb_maxpool2x2(void* stream, int dtype,
                  const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                  const int32_t* idx, const int32_t* count, const uint32_t* dil_bits,
                  void* out, long long o_sb, long long o_sc, long long o_sy, long long o_sx,
                  int B, int C, int H, int W, int oH, int oW);

/* cb_maxpool2x2 fused with the NEXT layer's change detection (pixel-major tensors of equal pitch
 * only): every re-pooled pixel is thresholded against next_state on the spot, its bit OR-ed into
 * next_raw_bits (which the caller keeps cleared, see cb_dilate_compact clear_raw) and next_state /
 * its auxiliary planes are maintained per update_mode -- i.e. cb_maxpool2x2 + cb_pool_compact +
 * cb_change_detect_sparse in one launch, with identical results.  dil_bits is required. */
int cb_maxpool2x2_detect(void* stream, int dtype, const void* x, long long x_sb, long long x_sy,
                         int x_pitch, const int32_t* idx, const int32_t* count,
                         const uint32_t* dil_bits, void* out, long long o_sb, long long o_sy,
                         int o_pitch, int B, int C, int H, int W, int oH, int oW, void* next_state,
                         long long n_sb, long long n_sy, int n_pitch, int aux_mode, void* aux_hi,
                         void* aux_lo, uint32_t* next_raw_bits, float threshold, int update_mode);

/* ---- per-stream thresholds --------------------------------------------------------------------
 * The *_thr entry points are the newest variant of each threshold-taking call above plus thr_b: fp32
 * [B] in device memory, read on the device (capturable in a CUDA graph; a replay reads the values the
 * buffer holds then), or NULL = the scalar threshold for every stream (then exactly the call without
 * it, which forwards here with NULL).  Pixel p of stream b (b = p / (H*W)) is tested against thr_b[b]
 * instead of the scalar, rounded to the data type exactly as the scalar is (fp16 / bf16: round to
 * nearest), so a stream b computes bit for bit what the call computes with threshold = thr_b[b].
 * For cb_maxpool2x2_detect_thr and cb_conv_update_tiled_pool_thr thr_b is the NEXT layer's (the one
 * whose detection runs in the kernel); cb_tail_update_thr takes one table per layer (thr1_b, thr2_b,
 * each may be NULL) and needs B and hw whenever one of them is given.  thr_b must be 4-byte aligned.
 * No reference counterpart (the reference is batch 1; DESIGN.md section 3.15). */
int cb_change_detect_thr(void* stream, int dtype,
                         const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                         void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                         int aux_mode, void* aux_hi, void* aux_lo, uint32_t* raw_bits, int B, int C,
                         int H, int W, float threshold, int update_mode, const uint8_t* active,
                         const float* thr_b);
int cb_change_detect_u8_thr(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                            long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                            long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                            uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                            float threshold, int update_mode, const uint8_t* active, const float* thr_b);
int cb_change_detect_sparse_thr(void* stream, int dtype,
                                const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                                void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                                int aux_mode, void* aux_hi, void* aux_lo,
                                const int32_t* candidates, const int32_t* n_candidates,
                                uint32_t* raw_bits, int B, int C, int H, int W, float threshold,
                                int update_mode, int bits_are_clear, const float* thr_b);
int cb_change_detect_sparse_compact_thr(void* stream, int dtype, const void* x, long long x_sb, long long x_sc,
                                        long long x_sy, long long x_sx, void* state, long long s_sb,
                                        long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                                        void* aux_hi, void* aux_lo, const int32_t* candidates,
                                        const int32_t* n_candidates, uint32_t* raw_bits, int B, int C, int H,
                                        int W, float threshold, int update_mode, int bits_are_clear,
                                        uint32_t* dil_bits, int32_t* idx, int32_t* count, void* sync_ws,
                                        int kHHalf, int kWHalf, int clear_raw, int32_t* stream_counts,
                                        int32_t* stream_acc, const float* thr_b);
int cb_maxpool2x2_detect_thr(void* stream, int dtype, const void* x, long long x_sb, long long x_sy,
                             int x_pitch, const int32_t* idx, const int32_t* count,
                             const uint32_t* dil_bits, void* out, long long o_sb, long long o_sy,
                             int o_pitch, int B, int C, int H, int W, int oH, int oW, void* next_state,
                             long long n_sb, long long n_sy, int n_pitch, int aux_mode, void* aux_hi,
                             void* aux_lo, uint32_t* next_raw_bits, float threshold, int update_mode,
                             const float* thr_b);
int cb_conv_update_tiled_pool_thr(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                                  int pitch_in, const void* tile_ws, const uint32_t* dil_bits,
                                  const void* packed_w, const float* bias, void* out, int pitch_out, int B,
                                  int H, int W, int Cin, int Cout, int kH, int kW, int relu,
                                  void* pool_out, long long o_sb, long long o_sy, int o_pitch, int oH, int oW,
                                  void* next_state, long long n_sb, long long n_sy, int n_pitch, int aux_mode,
                                  void* aux_hi, void* aux_lo, uint32_t* next_raw_bits, float threshold,
                                  int update_mode, const float* thr_b);
int cb_tail_update_thr(void* stream, const float* x, float* state1, const void* packed_w1, const float* bias1,
                       float* out1, int relu1, float thr1, float* state2, const void* packed_w2,
                       const float* bias2, float* out2, int pitch_out2, int relu2, float thr2,
                       const int32_t* candidates, const int32_t* n_candidates, int C0, int C1, int C2,
                       int update_mode, int32_t* count1, int32_t* count2, void* sync_ws, int B, int hw,
                       int32_t* stream_counts1, int32_t* stream_acc1, int32_t* stream_counts2,
                       int32_t* stream_acc2, const float* thr1_b, const float* thr2_b);

/* ---- watched-pixel zones ----------------------------------------------------------------------
 * cb_change_detect_zone / cb_change_detect_u8_zone are cb_change_detect_thr / cb_change_detect_u8_thr
 * plus zone: a uint32 bitmap [B, H, Wd] (Wd = cb_bitmap_row_words(W); bit x % 32 of word x / 32, bits at
 * or beyond W ignored) in device memory, read on the device (capturable; a replay reads what the buffer
 * holds then), or NULL = every pixel watched (then exactly the call without it, which forwards here with
 * NULL).  A pixel of stream b whose zone bit is 0 counts as unchanged: its x is not read, its bit is 0 and
 * its state and operand planes are not written, under every update_mode.  Exception: a pixel whose state
 * holds +inf in one of its C channels (never accepted: a fresh state, or a stream reset by
 * cb_reset_streams) is tested as usual, so an excluded area never hands +inf to the contraction.
 * Rule: with a threshold >= 0, the call computes bit for bit what the call without a zone computes on
 * the frame x' that equals x at watched pixels and at pixels with +inf in their state, and equals the
 * state elsewhere.  The active mask wins: a skipped stream's words are 0 and its zone is not read.
 * A zone needs the narrow kernel: C <= 16 / element size and a pixel-major state of exactly one
 * 16-byte chunk per pixel (any x strides); other layouts, and a zone not aligned to 4 bytes, get
 * status 2.  No reference counterpart (DESIGN.md section 3.16). */
int cb_change_detect_zone(void* stream, int dtype,
                          const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                          void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                          int aux_mode, void* aux_hi, void* aux_lo, uint32_t* raw_bits, int B, int C,
                          int H, int W, float threshold, int update_mode, const uint8_t* active,
                          const float* thr_b, const uint32_t* zone);
int cb_change_detect_u8_zone(void* stream, const uint8_t* x, long long x_sb, long long x_sc,
                             long long x_sy, long long x_sx, float* state, long long s_sb, long long s_sc,
                             long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                             uint32_t* raw_bits, int B, int C, int H, int W, float divisor, float bias,
                             float threshold, int update_mode, const uint8_t* active, const float* thr_b,
                             const uint32_t* zone);

/* ---- per-stream state reset -----------------------------------------------------------------
 * Starts a new sequence in some streams of a batch without touching the others: for every b with
 * mask[b] != 0 (mask: uint8[B] in device memory, read on the device), stream b's slice of every
 * segment is rewritten.  A segment is one pixel-major buffer [B, pixels, pitch_bytes]: stream b's
 * slice is the `pixels * pitch_bytes` bytes at base + b * pixels * pitch_bytes.  In each pixel the
 * first channel_bytes bytes (the real channels) are set to +inf of the segment's dtype
 * (CB_RESET_FILL_INF) or to 0 (CB_RESET_FILL_ZERO); the pad channels behind them are set to 0.
 * A model whose every layer's state (previous input, previous output, pooled map: +inf; operand
 * planes: 0) is reset this way computes the reset streams' next frame exactly like a freshly
 * cleared model (DESIGN.md section 3.12).  One launch for up to 96 segments (more are split over
 * several launches); no host synchronisation, capturable in a CUDA graph.  base must be aligned to
 * the element size, pitch_bytes and channel_bytes multiples of it, channel_bytes <= pitch_bytes.
 * No reference counterpart (the reference is batch 1 and frees all state, conv2d.py:147-148). */
#define CB_RESET_FILL_ZERO 0
#define CB_RESET_FILL_INF 1
typedef struct cb_reset_segment {
  void* base;              /* stream 0's slice                                              */
  long long pixels;        /* pixels per stream (H * W)                                     */
  int pitch_bytes;         /* bytes per pixel                                               */
  int channel_bytes;       /* bytes of real channels per pixel                              */
  int dtype;               /* CB_F32 / CB_F16 / CB_BF16: element size and the +inf written  */
  int fill;                /* CB_RESET_FILL_INF or CB_RESET_FILL_ZERO                       */
} cb_reset_segment;
int cb_reset_streams(void* stream, const uint8_t* mask, int B, const cb_reset_segment* segments,
                     int n_segments);

/* ---- staged (unfused) ops in the reference's planar layout --------------------------------
 * 1:1 replacements used by the op-level wrappers and parity tests. n is a host count here,
 * exactly as in the reference signatures. */
/* genXMatrix: conv2d_cg.py:21-27 -> cbconv2d_cg_backend.cu:138-173 */
int cb_gen_xmatrix(void* stream, int dtype, void* columns, const void* input, const int32_t* idx,
                   int kW, int kH, int C, int W, int H, int n);
/* matrixMult_python: conv2d_cg.py:342-349 (fp32 accumulate; bias dtype = data dtype) */
int cb_matrix_mult(void* stream, int dtype, const void* X, const void* weight, const void* bias,
                   void* Y, int n, int K, int Cout);
/* updateOutput: conv2d_cg.py:29-31 -> cbconv2d_cg_backend.cu:175-197 (Yt is [Cout,n]) */
int cb_update_output(void* stream, int dtype, const void* Yt, void* output, const int32_t* idx,
                     int numOutputPixel, int n, int Cout, int relu);

/* ---- fine-grained path (fp32) -------------------------------------------------------------
 * replaces: changeDetectionFG (conv2d_fg.py:20-24 -> cbconv2d_fg_backend.cu:7-35),
 *           torch.nonzero (conv2d_fg.py:82) and updateOutputFG (conv2d_fg.py:14-18 ->
 *           cbconv2d_fg_backend.cu:37-79), fused: per value d = x - prev, if |d| > thr then
 *           out[co, y-ky+kH/2, x-kx+kW/2] += W[co,ci,ky,kx]*d for all co,ky,kx (atomic adds);
 *           afterwards prev = x (conv2d.py:175).  *count receives the number of changed values.
 * Planar NCHW fp32 tensors, batch B. */
int cb_fg_update(void* stream, const float* x, float* prev, const float* weight, float* out,
                 int32_t* count, int B, int Cin, int Cout, int H, int W, int kH, int kW,
                 float threshold);


/* Fine-grained update on the tensor cores (B200 path of the same stage; the module uses it, the
 * planar op above stays as the reference-layout drop-in).  The sum over the changed values of
 * W[co,ci,ky,kx]*d (updateOutputFG_kernel, cbconv2d_fg_backend.cu:37-66) equals conv(D, W) with
 * D = the thresholded delta map, so:
 *   cb_fg_detect      replaces changeDetectionFG (cbconv2d_fg_backend.cu:7-23) + torch.nonzero
 *                     (conv2d_fg.py:82): per value d = x - prev, D = d if |d| > thr else 0, written as
 *                     bf16 hi/lo operand planes [B,H,W,cb_plane_pitch16(C)] (zero-initialised by the
 *                     caller once; pad channels are never written); raw_bits = pixels with any changed
 *                     value; *count (optional) = number of changed values; prev <- x (conv2d.py:175).
 *                     x: any strides (fast paths: planar rows, or pixel-major like the state);
 *                     prev: pixel-major fp32 [B,H,W,p_pitch].
 *   cb_dilate_compact lists the output pixels inside the filter footprint of a changed value;
 *   cb_conv_accumulate = cb_conv_update over that list with an accumulating epilogue:
 *                     out[pix, :] += sum_taps D[pix+tap, :] . W  (no bias, no ReLU).  state/state_lo
 *                     are the delta planes for CB_GEMM_TC_BF16X3. */
int cb_fg_detect(void* stream, const float* x, long long x_sb, long long x_sc, long long x_sy,
                 long long x_sx, float* prev, long long p_sb, long long p_sy, int p_pitch, void* delta_hi,
                 void* delta_lo, uint32_t* raw_bits, int32_t* count, int B, int C, int H, int W,
                 float threshold);
int cb_conv_accumulate(void* stream, int dtype, int gemm, const void* state, const void* state_lo,
                       int pitch_in, const int32_t* idx, const int32_t* count, const void* packed_w,
                       void* out, int pitch_out, int B, int H, int W, int Cin, int Cout, int kH, int kW,
                       void* ws, size_t ws_bytes);

/* ---- frame ingest: resizing on the device --------------------------------------------------------
 * The step before the path (SURVEY 8f rank 4): the reference's readers resize every frame on the host
 * with third-party code before the first layer sees it.
 *   cb_resize_bicubic_u8   replaces torchvision.transforms.Scale(boxsize, interpolation=3) =
 *                          PIL.Image.resize(size, BICUBIC) on 8-bit images in PoseDetector.preprocess
 *                          (poseDetection/openPose/PoseDetector.py:66-68).  Pillow's separable fixed-point
 *                          resampler (Resample.c: horizontal pass first, 22-bit weights, 8-bit intermediate),
 *                          BIT-EXACT.  src / dst: byte strides (row, pixel, channel): HWC, planar or pitched;
 *                          1..4 channels.  ws = cb_resize_ws_bytes() of device memory, filled once per
 *                          geometry by cb_resize_bicubic_u8_init (host-computed weight tables, synchronous);
 *                          the resize call itself is two launches and capturable.  Feed dst to
 *                          cb_change_detect_u8(divisor 256, bias -0.5): bit-identical to ToTensor() followed
 *                          by mul_(255/256).add_(-0.5) (:69-72; util.padBottomRight returns its input).
 *   cb_resize_bilinear_u8  replaces img.astype(float) / 255 + skimage.transform.resize(img, [776, 1040],
 *                          mode='constant') + permute(2,0,1).float() (sceneLabeling/videoSequenceReader.py:
 *                          64-67): order-1 interpolation at scale * (i + 0.5) - 0.5 with constant padding
 *                          (cval), float64 arithmetic, clipped to [clip_lo, clip_hi] (skimage clips to the
 *                          input's value range), fp32 output with ELEMENT strides (row, pixel, channel). */
size_t cb_resize_ws_bytes(int sH, int sW, int dH, int dW, int C);
int cb_resize_bicubic_u8_init(void* stream, void* ws, int sH, int sW, int dH, int dW, int C);
int cb_resize_bicubic_u8(void* stream, const uint8_t* src, long long s_y, long long s_x, long long s_c,
                         uint8_t* dst, long long d_y, long long d_x, long long d_c, void* ws, int sH, int sW,
                         int dH, int dW, int C);
int cb_resize_bilinear_u8(void* stream, const uint8_t* src, long long s_y, long long s_x, long long s_c, int sH,
                          int sW, float* dst, long long d_y, long long d_x, long long d_c, int dH, int dW, int C,
                          float divisor, float cval, float clip_lo, float clip_hi);

#ifdef __cplusplus
}
#endif
#endif /* CBINFER_B200_H */
