// detect.cuh -- change detection: thresholded |x_t - x_{t-1}| -> 1 bit per pixel.
//
// Replaces the detection half of changeDetection[_1x1]_kernel
// (reference pycbinfer/cbconv2d_cg_backend.cu:6-81, half: cbconv2d_cg_half_backend.cu:10-88).
//
// One bitmap word = 32 consecutive pixels of one image row.
//   * vector path (pixel-major x and state): WPW warps share one word; each streams its slice of
//     the 32 pixels' channels as 16-byte chunks, fully coalesced, with 2*U loads in flight per
//     lane; per-chunk flags are folded to per-pixel flags with __ballot_sync + bit-range masks and
//     OR-ed across the word's warps through shared memory.
//   * narrow path (any x strides, state pixel = one 16-byte chunk, e.g. the RGB input frame).
//   * generic path (any strides on both sides).
// HBM-bound: algorithmic bytes = 2*C*P*s read (+ P/8 bitmap, + feedback writes).
//
// Active-stream mask (`active`, uint8 [B] on the device, may be null = every stream): the dense
// kernels decide per bitmap word (a word never spans two images, rows are padded to whole words).
// A word of a stream with active[b] == 0 is written as 0 and nothing of that stream's x, state or
// operand planes is loaded or stored; every block barrier is still reached by all threads.
//
// Per-stream thresholds (`thr_b`, fp32 [B] on the device, may be null = the scalar `thr` for every
// stream): every kernel that tests a threshold reads stream b's value once per decision unit (a
// bitmap word, a candidate) and rounds it to T with thr_cast, as the host rounds the scalar.  The
// table is a compile-time variant (THR): without it the kernels are the ones compiled before it existed.
//
// Watched-pixel zone (`zone`, uint32 [B, H, Wd] on the device in the bitmap layout, may be null = every
// pixel watched): detect_narrow_kernel only, as a compile-time variant (ZONE).  A warp loads its word's
// zone word once; a lane whose bit is 0 and whose state is finite in every real channel is reported
// unchanged without reading x or writing its state / operand planes.  A state pixel holding +inf in a
// real channel (never accepted: fresh or reset stream) is tested as usual.  Exactly the result of the
// call without a zone on the frame whose excluded finite pixels hold the state's values (threshold >= 0).
#pragma once
#include "cb_common.cuh"
#include "compact.cuh"

namespace cb {

template <typename T> __host__ __device__ inline T thr_cast(float t);
template <> __host__ __device__ inline float thr_cast<float>(float t) { return t; }
template <> __host__ __device__ inline __half thr_cast<__half>(float t) { return __float2half_rn(t); }
template <> __host__ __device__ inline __nv_bfloat16 thr_cast<__nv_bfloat16>(float t) {
  return __float2bfloat16_rn(t);
}

// stream b's threshold: thr_b[b] rounded to T (THR), or the scalar
template <bool THR, typename T>
__device__ __forceinline__ T stream_thr(const float* __restrict__ thr_b, int b, T thr) {
  if constexpr (THR) return thr_cast<T>(__ldg(thr_b + b));
  else return thr;
}

template <typename T, int VEC>
__device__ __forceinline__ uint4 merge_tail(uint4 xv, const uint4& sv, int tail) {
  T* xe = reinterpret_cast<T*>(&xv);
  const T* se = reinterpret_cast<const T*>(&sv);
#pragma unroll
  for (int e = 0; e < VEC; ++e)
    if (e >= tail) xe[e] = se[e];
  return xv;
}

// Auxiliary operand planes kept in step with the state (written wherever the state is written), so
// the contraction's operand split is paid once per accepted pixel instead of once per gathered tap:
//   mode 1: fp32 plane  lo = v - trunc_tf32(v)            (3xTF32: the raw state is the "hi" operand,
//           the tensor core ignores the 13 low mantissa bits)
//   mode 2: two bf16 planes  hi = bf16(v), lo = bf16(v - hi)   (3xBF16: ~16 mantissa bits at twice
//           the tensor rate and half the bytes of 3xTF32), pixel-major with their own pitch.
struct AuxPlanes {
  int mode;
  int pitch16;               // mode 2: bf16 elements per pixel (pitch16_of(C))
  long long lo_off;          // mode 1: element offset state -> lo plane (same strides as the state)
  __nv_bfloat16* hi16;       // mode 2
  __nv_bfloat16* lo16;
};

__device__ __forceinline__ unsigned tf32_lo(unsigned v) {
  return __float_as_uint(__uint_as_float(v) - __uint_as_float(v & 0xFFFFE000u));
}
__device__ __forceinline__ void bf16_split(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
// pix = global pixel index, ch0 = first channel of this 16-byte chunk
template <typename T>
__device__ __forceinline__ void store_state(T* sptr, const uint4& v, const AuxPlanes& aux,
                                            long long pix, int ch0) {
  st16(sptr, v);
  if (sizeof(T) == 4 && aux.mode == 1) {
    st16(sptr + aux.lo_off, make_uint4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)));
  } else if (sizeof(T) == 4 && aux.mode == 2) {
    __nv_bfloat16 h[4], l[4];
    bf16_split(__uint_as_float(v.x), h[0], l[0]);
    bf16_split(__uint_as_float(v.y), h[1], l[1]);
    bf16_split(__uint_as_float(v.z), h[2], l[2]);
    bf16_split(__uint_as_float(v.w), h[3], l[3]);
    const long long o = pix * aux.pitch16 + ch0;
    *reinterpret_cast<uint2*>(aux.hi16 + o) = *reinterpret_cast<uint2*>(h);
    *reinterpret_cast<uint2*>(aux.lo16 + o) = *reinterpret_cast<uint2*>(l);
  }
}
__device__ __forceinline__ void store_state_scalar(float* sptr, float v, const AuxPlanes& aux,
                                                   long long pix, int ch) {
  *sptr = v;
  if (aux.mode == 1) {
    sptr[aux.lo_off] = __uint_as_float(tf32_lo(__float_as_uint(v)));
  } else if (aux.mode == 2) {
    __nv_bfloat16 h, l;
    bf16_split(v, h, l);
    aux.hi16[pix * aux.pitch16 + ch] = h;
    aux.lo16[pix * aux.pitch16 + ch] = l;
  }
}
template <typename T>
__device__ __forceinline__ void store_state_scalar(T* sptr, T v, const AuxPlanes&, long long, int) {
  *sptr = v;
}

// streaming (evict-first) loads for data a frame scan reads exactly once per step: the input frame and
// the first layer's state (70 MB per step at 8 streams) should not push the small control structures
// and the maps the following kernels reuse out of L2
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ __half ld_stream(const __half* p) {
  const unsigned short v = __ldcs(reinterpret_cast<const unsigned short*>(p));
  return __ushort_as_half(v);
}
__device__ __forceinline__ __nv_bfloat16 ld_stream(const __nv_bfloat16* p) {
  const unsigned short v = __ldcs(reinterpret_cast<const unsigned short*>(p));
  return __ushort_as_bfloat16(v);
}
__device__ __forceinline__ uint4 ld16_stream(const void* p) { return __ldcs(reinterpret_cast<const uint4*>(p)); }

constexpr int kDetWarps = 8;                   // warps per block

// The bitmap word of this warp in the kernels that give each warp one word (32 pixels of a row):
// image b, row y and this lane's pixel column xx; false beyond the map.  32-bit index math (the host
// checks words < 2^31): two 64-bit divisions per warp were most of these kernels' instructions (ncu:
// 173 warp instructions per 32 pixels, SM 54 % busy on an HBM-bound scan)
__device__ __forceinline__ bool warp_word(unsigned& warp, int& b, int& y, int& xx, int B, int H, int Wd) {
  warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (warp >= (unsigned)(B * H * Wd)) return false;
  const unsigned r = warp / (unsigned)Wd;
  const int j = (int)(warp - r * (unsigned)Wd);
  b = (int)(r / (unsigned)H);
  y = (int)(r - (unsigned)b * (unsigned)H);
  xx = j * 32 + (threadIdx.x & 31);
  return true;
}

// One pixel, any strides, one channel at a time: any channel changed?  The state follows UPDATE.
template <typename T, int UPDATE>
__device__ __forceinline__ bool pixel_changed_scalar(const T* xp, long long x_sc, T* sp, long long s_sc,
                                                     int C, T thr, const AuxPlanes& aux, long long gpix) {
  bool f = false;
  for (int c = 0; c < C; ++c) {
    const T xv = xp[c * x_sc];
    f |= value_changed(sp[c * s_sc], xv, thr);
    if (UPDATE == CB_UPDATE_ALL) store_state_scalar(sp + c * s_sc, xv, aux, gpix, c);
  }
  if (UPDATE == CB_UPDATE_CHANGED && f)
    for (int c = 0; c < C; ++c) store_state_scalar(sp + c * s_sc, xp[c * x_sc], aux, gpix, c);
  return f;
}

// x: pixel-major, pitch xp (elements); state: pixel-major, pitch sp.  Rows may be strided (sy).
// U chunk-iterations are batched: all 2*U 16-byte loads of a batch are issued before the first
// ballot, so every lane keeps 2*U loads in flight (the ballots would otherwise serialise them).
// wlog = log2(warps per word): a block of 8 warps covers 8 >> wlog words.
template <typename T, int VEC, int UPDATE, int U, bool THR = false>
__global__ void __launch_bounds__(kDetWarps * 32)
detect_vec_kernel(const T* __restrict__ x, long long x_sb, long long x_sy, int xp,
                  T* __restrict__ st, long long s_sb, long long s_sy, int sp, AuxPlanes aux,
                  uint32_t* __restrict__ bits, int B, int H, int W, int C, int Wd, T thr,
                  unsigned cpv_magic, int wlog, const uint8_t* __restrict__ active,
                  const float* __restrict__ thr_b) {
  __shared__ unsigned s_word[kDetWarps];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int wpw = 1 << wlog;
  const int part = wid & (wpw - 1), slot = wid >> wlog;
  const int word = blockIdx.x * (kDetWarps >> wlog) + slot;      // < 2^31 words (host-checked)
  const bool inmap = word < B * H * Wd;
  if (wlog > 0) {
    if (threadIdx.x < kDetWarps) s_word[threadIdx.x] = 0u;
    __syncthreads();
  } else if (!inmap) {
    return;
  }
  const int cpv = (C + VEC - 1) / VEC;       // 16-byte chunks per pixel that hold real channels
  const int tail = C % VEC;                  // valid elements of the last chunk (0 = all)
  // q / cpv without a divide: exact for q*cpv < 2^32 (q <= 32*cpv here)
  auto pixel_of = [&](int q) { return cpv == 1 ? q : (int)__umulhi((unsigned)q, cpv_magic); };
  const T* xb = nullptr;
  T* sb = nullptr;
  int nq = 0;
  long long pixbase = 0;
  unsigned wordbits = 0;
  if (inmap) {
    const int j = word % Wd;
    const int r = word / Wd;
    const int y = r % H;
    const int b = r / H;
    const int x0 = j * 32;
    const int npx = min(32, W - x0);
    xb = x + b * x_sb + y * x_sy + (long long)x0 * xp;
    sb = st + b * s_sb + y * s_sy + (long long)x0 * sp;
    nq = (active && !__ldg(active + b)) ? 0 : npx * cpv;   // skipped stream: no loads, word 0
    pixbase = ((long long)b * H + y) * W + x0;
    const T tb = stream_thr<THR>(thr_b, b, thr);

    bool mychg = false;                      // flag of pixel `lane` (this warp's slice only)
    const int plo = lane * cpv, phi = plo + cpv;
    for (int q0 = part * 32 * U; q0 < nq; q0 += wpw * 32 * U) {
      uint4 xv[U], sv[U];
      T* sptr[U];
      int pxs[U], ccs[U];
      bool valid[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int q = q0 + u * 32 + lane;
        valid[u] = q < nq;
        const int px = pixel_of(q), cc = q - px * cpv;
        pxs[u] = px;
        ccs[u] = cc;
        sptr[u] = sb + (long long)px * sp + cc * VEC;
        if (valid[u]) {
          xv[u] = ldg16(xb + (long long)px * xp + cc * VEC);
          sv[u] = ld16(sptr[u]);
          if (tail && cc == cpv - 1) xv[u] = merge_tail<T, VEC>(xv[u], sv[u], tail);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        bool f = false;
        if (valid[u]) {
          f = Chunk<T>::changed(sv[u], xv[u], tb);
          if (UPDATE == CB_UPDATE_ALL) store_state<T>(sptr[u], xv[u], aux, pixbase + pxs[u], ccs[u] * VEC);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        const int qb = q0 + u * 32;
        const int lo = max(plo, qb) - qb, hi = min(phi, qb + 32) - qb;
        if (hi > lo) {
          const unsigned m = (hi - lo >= 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
          mychg |= (bal & m) != 0u;
        }
      }
    }
    wordbits = __ballot_sync(0xffffffffu, mychg);
  }
  if (wlog > 0) {                              // OR the partial words of the warps sharing a word
    if (inmap && lane == 0 && wordbits) atomicOr(&s_word[slot], wordbits);
    __syncthreads();
    wordbits = s_word[slot];
    if (!inmap) return;
  }
  if (part == 0 && lane == 0) bits[word] = wordbits;

  if (UPDATE == CB_UPDATE_CHANGED && wordbits) {  // feedback: accept the new value at changed pixels
    for (int q = part * 32 + lane; q < nq; q += wpw * 32) {
      const int px = pixel_of(q), cc = q - px * cpv;
      if ((wordbits >> px) & 1u) {
        uint4 xv = ldg16(xb + (long long)px * xp + cc * VEC);
        T* sp2 = sb + (long long)px * sp + cc * VEC;
        if (tail && cc == cpv - 1) xv = merge_tail<T, VEC>(xv, ld16(sp2), tail);
        store_state<T>(sp2, xv, aux, pixbase + px, cc * VEC);
      }
    }
  }
}

// Generic x (any strides, e.g. the user's planar NCHW frame) against a pixel-major state whose
// pixel is exactly one 16-byte chunk (C <= 4 fp32 / C <= 8 half): lane = pixel, the state is one
// vector load/store per pixel and x is read plane by plane (coalesced across lanes).
// S = uint8_t: frame ingest (decoder / camera output, any strides: HWC interleaved or planar) into a
// fp32 state.  The normalisation of the reference's readers -- frame/255
// (sceneLabeling/videoSequenceReader.py:65), frame/256 - 0.5 (openPose/PoseDetector.py:72) -- is
// applied on the fly with IEEE division and addition, so the result is bit-identical to detecting on
// the host-normalised fp32 frame, at a quarter of the host->device bytes.  Otherwise divisor and bias
// are unused.
// +inf in one of the first C elements of a state chunk: a pixel that was never accepted
__device__ __forceinline__ bool is_pos_inf(float v) { return __float_as_uint(v) == 0x7f800000u; }
__device__ __forceinline__ bool is_pos_inf(__half v) { return __half_as_ushort(v) == 0x7c00u; }
__device__ __forceinline__ bool is_pos_inf(__nv_bfloat16 v) { return __bfloat16_as_ushort(v) == 0x7f80u; }
template <typename T, int VEC>
__device__ __forceinline__ bool chunk_unaccepted(const uint4& v, int C) {
  const T* e = reinterpret_cast<const T*>(&v);
  bool r = false;
#pragma unroll
  for (int c = 0; c < VEC; ++c)
    if (c < C) r |= is_pos_inf(e[c]);
  return r;
}

template <typename T, int VEC, int UPDATE, typename S = T, bool THR = false, bool ZONE = false>
__global__ void __launch_bounds__(256)
detect_narrow_kernel(const S* __restrict__ x, long long x_sb, long long x_sc, long long x_sy,
                     long long x_sx, T* __restrict__ st, long long s_sb, long long s_sy,
                     AuxPlanes aux, uint32_t* __restrict__ bits, int B, int H, int W, int C,
                     int Wd, T thr, float divisor, float bias, const uint8_t* __restrict__ active,
                     const float* __restrict__ thr_b, const uint32_t* __restrict__ zone) {
  constexpr bool kU8 = std::is_same<S, uint8_t>::value;
  const float* lut = nullptr;
  if constexpr (kU8) {
    // the 256 possible normalised values, computed once per block with the IEEE division and addition
    // the host would use (bit-identical by construction): a table lookup per channel instead of a
    // division.  Every thread takes part before any warp leaves.
    __shared__ float s_lut[256];
    s_lut[threadIdx.x] = __fadd_rn(__fdiv_rn((float)threadIdx.x, divisor), bias);
    __syncthreads();
    lut = s_lut;
  }
  unsigned warp;
  int b, y, xx;
  if (!warp_word(warp, b, y, xx, B, H, Wd)) return;
  bool f = false;
  if (xx < W && (!active || __ldg(active + b))) {
    const S* xp = x + b * x_sb + y * x_sy + xx * x_sx;
    T* sp = st + b * s_sb + y * s_sy + (long long)xx * VEC;
    const uint4 sv = ld16_stream(sp);
    uint4 nv = sv;                             // pad lanes keep the state's (zero) value
    T* ne = reinterpret_cast<T*>(&nv);
    auto load_x = [&]() {
#pragma unroll
      for (int c = 0; c < VEC; ++c) {
        if (c >= C) continue;
        if constexpr (kU8) ne[c] = lut[__ldcs(xp + c * x_sc)];
        else ne[c] = ld_stream(xp + c * x_sc);
      }
    };
    bool test = true;
    if constexpr (ZONE) {
      // watched pixels load x without waiting for the state; an excluded one only if it was never accepted
      test = (__ldg(zone + warp) >> (threadIdx.x & 31)) & 1u;
      if (test) {
        load_x();
      } else if (chunk_unaccepted<T, VEC>(sv, C)) {
        load_x();
        test = true;
      }
    } else {
      load_x();
    }
    if (test) {
      f = Chunk<T>::changed(sv, nv, stream_thr<THR>(thr_b, b, thr));
      if (UPDATE == CB_UPDATE_ALL || (UPDATE == CB_UPDATE_CHANGED && f))
        store_state<T>(sp, nv, aux, ((long long)b * H + y) * W + xx, 0);
    }
  }
  const unsigned word = __ballot_sync(0xffffffffu, f);
  if ((threadIdx.x & 31) == 0) bits[warp] = word;
}

// Planar x (NCHW: the pixels of a row are contiguous, any channel stride -- what a dense layer or the
// user hands in) against a pixel-major state of more than one 16-byte chunk per pixel.  The two
// layouts want opposite lane mappings (x coalesces across pixels, the state across channels), so a
// block of 8 warps transposes `nw` bitmap words (32 pixels each) through shared memory:
//   phase 1: lane = pixel, warp = (word, channel chunk): VEC coalesced row loads per chunk -> one
//            16-byte shared-memory store at [pixel][chunk] (odd chunk pitch: conflict-free);
//   phase 2: thread = (pixel, chunk) in state order: 16-byte state load (coalesced), compare, state
//            / operand-plane store, pixel flags OR-ed into the word.
// nw is chosen so that every warp has ~4 (word, chunk) pairs: 4*VEC row loads in flight per lane.
// Both sides stream at full sector efficiency; the generic kernel reads the state at a stride of one
// pixel per lane (measured 1 TB/s at C = 64).
constexpr int kPlanarMaxWords = 8;
struct PlanarWord {
  long long xoff, soff, pix;     // element offsets of the word's first pixel in x / the state, global pixel index
  int npx;                       // valid pixels (0: word beyond the map, -1: word of a skipped stream)
};

__device__ __forceinline__ void planar_words_setup(PlanarWord* wi, unsigned* s_word, int word0, int nw,
                                                   long long nwords, int H, int W, int Wd, long long x_sb,
                                                   long long x_sy, long long x_sx, long long s_sb,
                                                   long long s_sy, int sp, const uint8_t* active = nullptr,
                                                   const float* thr_b = nullptr, float* s_thr = nullptr) {
  if (threadIdx.x < (unsigned)nw) {
    const long long word = (long long)word0 + threadIdx.x;
    PlanarWord w = {0, 0, 0, 0};
    if (word < nwords) {
      const int j = (int)(word % Wd);
      const long long r = word / Wd;
      const int y = (int)(r % H);
      const long long b = r / H;
      const int x0 = j * 32;
      // npx = -1: a word of a skipped stream; nothing of it is loaded, tested or stored, but it is
      // written (as 0), unlike a word beyond the map (npx = 0)
      w.npx = (active && !__ldg(active + b)) ? -1 : min(32, W - x0);
      w.xoff = b * x_sb + y * x_sy + x0 * x_sx;
      w.soff = b * s_sb + y * s_sy + (long long)x0 * sp;
      w.pix = (b * H + y) * W + x0;
      if (thr_b) s_thr[threadIdx.x] = __ldg(thr_b + b);   // a block's words may lie in two streams
    }
    wi[threadIdx.x] = w;
    s_word[threadIdx.x] = 0u;
  }
  __syncthreads();
}

// phase 1: x -> xs[(w*32 + px) * cps + cc]; chunks beyond C are zero-filled
template <typename T, int VEC>
__device__ __forceinline__ void planar_load_tile(uint4* xs, const PlanarWord* wi, const T* __restrict__ x,
                                                 long long x_sc, long long x_sx, int nw, int cpv, int cps,
                                                 int C, unsigned cpv_magic) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll 2
  for (int p = wid; p < nw * cpv; p += 8) {
    const int w = cpv == 1 ? p : (int)__umulhi((unsigned)p, cpv_magic), cc = p - w * cpv;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    T* ve = reinterpret_cast<T*>(&v);
    if (lane < wi[w].npx) {
      const T* xp = x + wi[w].xoff + lane * x_sx;
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        const int c = cc * VEC + e;
        if (c < C) ve[e] = __ldg(xp + c * x_sc);
      }
    }
    xs[(w * 32 + lane) * cps + cc] = v;
  }
}

// OR the pixel flag of this thread into its word's accumulator (warp-reduced when the warp's 32
// chunks belong to one word, which is the common case)
__device__ __forceinline__ void planar_flag(unsigned* s_word, int w, unsigned m) {
  const int w0 = __shfl_sync(0xffffffffu, w, 0), w1 = __shfl_sync(0xffffffffu, w, 31);
  if (w0 == w1) {
    m = __reduce_or_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicOr(&s_word[w0], m);
  } else if (m) {
    atomicOr(&s_word[w], m);
  }
}

template <typename T, int VEC, int UPDATE, bool THR = false>
__global__ void __launch_bounds__(256)
detect_planar_kernel(const T* __restrict__ x, long long x_sb, long long x_sc, long long x_sy,
                     T* __restrict__ st, long long s_sb, long long s_sy, int sp, AuxPlanes aux,
                     uint32_t* __restrict__ bits, int B, int H, int W, int C, int Wd, T thr,
                     unsigned cpv_magic, int cps, int nw, const uint8_t* __restrict__ active,
                     const float* __restrict__ thr_b) {
  extern __shared__ __align__(16) unsigned char dp_smem[];
  uint4* xs = reinterpret_cast<uint4*>(dp_smem);                 // [nw*32][cps]
  __shared__ unsigned s_word[kPlanarMaxWords];
  __shared__ PlanarWord wi[kPlanarMaxWords];
  __shared__ float s_thr[kPlanarMaxWords];                       // thr_b: each word's stream threshold
  const long long nwords = (long long)B * H * Wd;
  const int word0 = blockIdx.x * nw;
  planar_words_setup(wi, s_word, word0, nw, nwords, H, W, Wd, x_sb, x_sy, 1, s_sb, s_sy, sp, active,
                     THR ? thr_b : nullptr, s_thr);
  const int cpv = (C + VEC - 1) / VEC, tail = C % VEC;
  planar_load_tile<T, VEC>(xs, wi, x, x_sc, 1, nw, cpv, cps, C, cpv_magic);
  __syncthreads();
  const int nq = nw * 32 * cpv;
  for (int q0 = 0; q0 < nq; q0 += 256) {
    const int q = min(q0 + (int)threadIdx.x, nq - 1);            // (clamped lanes take no part below)
    const bool in = q0 + (int)threadIdx.x < nq;
    const int t = cpv == 1 ? q : (int)__umulhi((unsigned)q, cpv_magic), cc = q - t * cpv;
    const int w = t >> 5, px = t & 31;
    unsigned m = 0u;
    if (in && px < wi[w].npx) {
      uint4 xv = xs[t * cps + cc];
      T* sptr = st + wi[w].soff + (long long)px * sp + cc * VEC;
      const uint4 sv = ld16(sptr);
      if (tail && cc == cpv - 1) xv = merge_tail<T, VEC>(xv, sv, tail);
      if (Chunk<T>::changed(sv, xv, THR ? thr_cast<T>(s_thr[w]) : thr)) m = 1u << px;
      if (UPDATE == CB_UPDATE_ALL) store_state<T>(sptr, xv, aux, wi[w].pix + px, cc * VEC);
    }
    planar_flag(s_word, w, m);
  }
  __syncthreads();
  if (threadIdx.x < (unsigned)nw && wi[threadIdx.x].npx != 0) bits[word0 + threadIdx.x] = s_word[threadIdx.x];
  if (UPDATE == CB_UPDATE_CHANGED) {              // feedback: accept the new value at changed pixels
    for (int q = threadIdx.x; q < nq; q += 256) {
      const int t = cpv == 1 ? q : (int)__umulhi((unsigned)q, cpv_magic), cc = q - t * cpv;
      const int w = t >> 5, px = t & 31;
      if ((s_word[w] >> px) & 1u) {
        uint4 xv = xs[t * cps + cc];
        T* sptr = st + wi[w].soff + (long long)px * sp + cc * VEC;
        if (tail && cc == cpv - 1) xv = merge_tail<T, VEC>(xv, ld16(sptr), tail);
        store_state<T>(sptr, xv, aux, wi[w].pix + px, cc * VEC);
      }
    }
  }
}

// words per block of the planar kernels: every warp gets >= 2 (word, chunk) pairs, within 64 KB
inline int planar_words_per_block(int cpv, int cps) {
  // measured (tools/planar_bench.py, L2 flushed): 4 (word, chunk) pairs per warp, at most 4 words --
  // C=64 fp32 153 -> 135 us at nw=2, bf16 100 -> 94 us at nw=4; 8 words lose again (fewer, fatter blocks)
  int nw = 1;
  while (nw < 4 && nw * cpv < 32 && (size_t)(2 * nw) * 32 * cps * 16 <= 64 * 1024) nw *= 2;
  return nw;
}

template <typename T, int UPDATE, bool THR = false>
__global__ void __launch_bounds__(256)
detect_generic_kernel(const T* __restrict__ x, long long x_sb, long long x_sc, long long x_sy,
                      long long x_sx, T* __restrict__ st, long long s_sb, long long s_sc,
                      long long s_sy, long long s_sx, AuxPlanes aux,
                      uint32_t* __restrict__ bits, int B, int H, int W, int C, int Wd, T thr,
                      const uint8_t* __restrict__ active, const float* __restrict__ thr_b) {
  unsigned warp;
  int b, y, xx;
  if (!warp_word(warp, b, y, xx, B, H, Wd)) return;
  const bool f = xx < W && (!active || __ldg(active + b)) && pixel_changed_scalar<T, UPDATE>(x + b * x_sb + y * x_sy + xx * x_sx, x_sc,
                                                            st + b * s_sb + y * s_sy + xx * s_sx, s_sc, C,
                                                            stream_thr<THR>(thr_b, b, thr), aux,
                                                            ((long long)b * H + y) * W + xx);
  const unsigned word = __ballot_sync(0xffffffffu, f);
  if ((threadIdx.x & 31) == 0) bits[warp] = word;
}



template <typename T>
inline int make_aux(AuxPlanes& aux, int aux_mode, void* aux_hi, void* aux_lo, const void* state,
                    int C) {
  aux = AuxPlanes{0, 0, 0, nullptr, nullptr};
  if (aux_mode == 0) return 0;
  CB_CHECK_ARG(sizeof(T) == 4, "change_detect: auxiliary operand planes exist for fp32 data only");
  if (aux_mode == 1) {
    CB_CHECK_ARG(aux_lo && ((uintptr_t)aux_lo % 16) == 0, "change_detect: bad tf32 remainder plane");
    aux.mode = 1;
    aux.lo_off = (long long)((const T*)aux_lo - (const T*)state);
    return 0;
  }
  CB_CHECK_ARG(aux_mode == 2, "change_detect: bad aux_mode %d", aux_mode);
  CB_CHECK_ARG(aux_hi && aux_lo && ((uintptr_t)aux_hi % 16) == 0 && ((uintptr_t)aux_lo % 16) == 0,
               "change_detect: bad bf16 operand planes");
  aux.mode = 2;
  aux.pitch16 = pitch16_of(C);
  aux.hi16 = (__nv_bfloat16*)aux_hi;
  aux.lo16 = (__nv_bfloat16*)aux_lo;
  return 0;
}

// x and the state pixel-major: channel-contiguous pixels of whole 16-byte chunks, 16-byte aligned
// (the vector kernels)
template <typename T, int VEC>
inline bool pixel_major_ok(const void* x, long long x_sb, long long x_sc, long long x_sy, long long x_sx,
                           const void* state, long long s_sb, long long s_sc, long long s_sy, long long s_sx,
                           int C) {
  const size_t es = sizeof(T);
  return x_sc == 1 && s_sc == 1 && (x_sx % VEC) == 0 && (s_sx % VEC) == 0 && x_sx >= C && s_sx >= C &&
         ((x_sy * es) % 16) == 0 && ((s_sy * es) % 16) == 0 && ((x_sb * es) % 16) == 0 &&
         ((s_sb * es) % 16) == 0 && ((uintptr_t)x % 16) == 0 && ((uintptr_t)state % 16) == 0 &&
         x_sx < (1ll << 30) && s_sx < (1ll << 30);
}

template <typename T, int VEC>
int launch_detect(cudaStream_t stream, const void* x, long long x_sb, long long x_sc,
                  long long x_sy, long long x_sx, void* state, long long s_sb, long long s_sc,
                  long long s_sy, long long s_sx, int aux_mode, void* aux_hi, void* aux_lo,
                  uint32_t* bits, int B, int C, int H, int W, float threshold, int update,
                  const uint8_t* active, const float* thr_b, const uint32_t* zone) {
  const int Wd = (W + 31) / 32;
  const long long words = (long long)B * H * Wd;
  if (words == 0) return 0;
  const T thr = thr_cast<T>(threshold);
  const size_t es = sizeof(T);
  AuxPlanes aux;
  if (int rc = make_aux<T>(aux, aux_mode, aux_hi, aux_lo, state, C)) return rc;
  // the narrow kernel: state pixel = one 16-byte chunk, any x strides
  const bool narrow_fits = s_sc == 1 && s_sx == VEC && C <= VEC && ((s_sy * es) % 16) == 0 &&
                           ((s_sb * es) % 16) == 0 && ((uintptr_t)state % 16) == 0;
  if (zone) {                                 // only the narrow kernel has the ZONE variant
    CB_CHECK_ARG(narrow_fits, "change_detect: a zone needs a state pixel of one 16-byte chunk (C <= %d, pixel-major "
                 "state of pitch %d, 16-byte aligned)", VEC, VEC);
    CB_CHECK_ARG((words + 7) / 8 < (1ll << 31) && words < (1ll << 31), "change_detect: image too large");
    return dispatch_thr(thr_b, [&](auto R) { return dispatch_update(update, "change_detect", [&](auto U) {
      cb::launch(detect_narrow_kernel<T, VEC, U, T, R, true>, dim3((unsigned)((words + 7) / 8)), dim3(256), 0,
                 stream, (const T*)x, x_sb, x_sc, x_sy, x_sx, (T*)state, s_sb, s_sy, aux, bits, B, H, W, C, Wd, thr,
                 0.f, 0.f, active, thr_b, zone);
      CB_CHECK_LAUNCH("change_detect");
      return 0;
    }); });
  }
  const bool vec_ok = pixel_major_ok<T, VEC>(x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, C);
  const bool narrow_ok = !vec_ok && narrow_fits;
  const int cpv = (C + VEC - 1) / VEC;
  const unsigned magic = cpv > 1 ? (unsigned)((0x100000000ull + cpv - 1) / cpv) : 0u;
  // planar x, pixel-major multi-chunk state: transposed through shared memory (detect_planar_kernel)
  const int cps = cpv | 1;
  const int planar_nw = planar_words_per_block(cpv, cps);
  const size_t planar_smem = (size_t)planar_nw * 32 * cps * 16;
  const bool planar_ok = !vec_ok && !narrow_ok && x_sx == 1 && s_sc == 1 && (s_sx % VEC) == 0 && s_sx >= C &&
                         ((s_sy * es) % 16) == 0 && ((s_sb * es) % 16) == 0 && ((uintptr_t)state % 16) == 0 &&
                         s_sx < (1ll << 30) && planar_smem <= 200 * 1024;
  // warps per word: keep >= 4 load batches (of U*32 chunks) per warp, at most one block per word
  int wlog = 0;
  while (wlog < 3 && (32 * cpv) / (1 << (wlog + 1)) >= 4 * 4 * 32) ++wlog;
  const long long vec_blocks = (words + (kDetWarps >> wlog) - 1) / (kDetWarps >> wlog);
  const long long blocks = vec_ok ? vec_blocks : (words + 7) / 8;
  CB_CHECK_ARG(blocks < (1ll << 31) && words < (1ll << 31), "change_detect: image too large");
  dim3 grid((unsigned)blocks), block(256);
  return dispatch_thr(thr_b, [&](auto R) { return dispatch_update(update, "change_detect", [&](auto U) {
    if (vec_ok) {
      if (cpv >= 4)
        cb::launch(detect_vec_kernel<T, VEC, U, 4, R>, grid, block, 0, stream, (const T*)x, x_sb, x_sy, (int)x_sx,
                   (T*)state, s_sb, s_sy, (int)s_sx, aux, bits, B, H, W, C, Wd, thr, magic, wlog, active, thr_b);
      else
        cb::launch(detect_vec_kernel<T, VEC, U, 2, R>, grid, block, 0, stream, (const T*)x, x_sb, x_sy, (int)x_sx,
                   (T*)state, s_sb, s_sy, (int)s_sx, aux, bits, B, H, W, C, Wd, thr, magic, wlog, active, thr_b);
    } else if (narrow_ok) {
      cb::launch(detect_narrow_kernel<T, VEC, U, T, R>, grid, block, 0, stream, (const T*)x, x_sb, x_sc, x_sy, x_sx,
                 (T*)state, s_sb, s_sy, aux, bits, B, H, W, C, Wd, thr, 0.f, 0.f, active, thr_b, nullptr);
    } else if (planar_ok) {
      if (planar_smem > 48 * 1024)
        cudaFuncSetAttribute(detect_planar_kernel<T, VEC, U, R>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)planar_smem);
      cb::launch(detect_planar_kernel<T, VEC, U, R>, dim3((unsigned)((words + planar_nw - 1) / planar_nw)), block,
                 planar_smem, stream, (const T*)x, x_sb, x_sc, x_sy, (T*)state, s_sb, s_sy, (int)s_sx, aux, bits,
                 B, H, W, C, Wd, thr, magic, cps, planar_nw, active, thr_b);
    } else {
      cb::launch(detect_generic_kernel<T, U, R>, grid, block, 0, stream, (const T*)x, x_sb, x_sc, x_sy, x_sx,
                 (T*)state, s_sb, s_sc, s_sy, s_sx, aux, bits, B, H, W, C, Wd, thr, active, thr_b);
    }
    CB_CHECK_LAUNCH("change_detect");
    return 0;
  }); });
}


inline int launch_detect_u8(cudaStream_t stream, const void* x, long long x_sb, long long x_sc,
                            long long x_sy, long long x_sx, void* state, long long s_sb,
                            long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                            void* aux_hi, void* aux_lo, uint32_t* bits, int B, int C, int H, int W,
                            float divisor, float bias, float threshold, int update,
                            const uint8_t* active, const float* thr_b, const uint32_t* zone) {
  const int Wd = (W + 31) / 32;
  const long long words = (long long)B * H * Wd;
  if (words == 0) return 0;
  CB_CHECK_ARG(C <= 4 && s_sc == 1 && s_sx == 4 && (s_sy % 4) == 0 && (s_sb % 4) == 0 &&
                   ((uintptr_t)state % 16) == 0,
               "change_detect_u8: needs <= 4 channels and a pixel-major fp32 state of pitch 4");
  CB_CHECK_ARG(divisor != 0.f, "change_detect_u8: divisor must be non-zero");
  AuxPlanes aux;
  if (int rc = make_aux<float>(aux, aux_mode, aux_hi, aux_lo, state, C)) return rc;
  const long long blocks = (words + 7) / 8;
  CB_CHECK_ARG(blocks < (1ll << 31), "change_detect_u8: image too large");
  return dispatch_thr(thr_b, [&](auto R) { return dispatch_update(update, "change_detect_u8", [&](auto U) {
    if (zone)
      cb::launch(detect_narrow_kernel<float, 4, U, uint8_t, R, true>, dim3((unsigned)blocks), dim3(256), 0, stream,
                 (const uint8_t*)x, x_sb, x_sc, x_sy, x_sx, (float*)state, s_sb, s_sy, aux, bits, B, H, W, C, Wd,
                 threshold, divisor, bias, active, thr_b, zone);
    else
      cb::launch(detect_narrow_kernel<float, 4, U, uint8_t, R>, dim3((unsigned)blocks), dim3(256), 0, stream,
                 (const uint8_t*)x, x_sb, x_sc, x_sy, x_sx, (float*)state, s_sb, s_sy, aux, bits, B, H, W, C, Wd,
                 threshold, divisor, bias, active, thr_b, nullptr);
    CB_CHECK_LAUNCH("change_detect_u8");
    return 0;
  }); });
}


// ------------------------------------------------------------------------------------------------
// Candidate ("sparse") detection: the same per-pixel test, evaluated only at the pixels an
// upstream change-based layer reports as rewritten.  Exact w.r.t. the dense scan as long as x is
// unchanged everywhere else, the threshold was not lowered and the state is not fresh (the module
// checks this): an untouched pixel was either accepted last frame (state == x, difference 0) or
// is as far below the threshold as it was.  Replaces the O(C*P) scan with O(C*n_candidates).
// A group of 1 << glog lanes owns one candidate (16-byte chunks, pixel-major); set bits are
// OR-ed into the pre-zeroed bitmap.
// ------------------------------------------------------------------------------------------------
// FUSE: the last block to finish also dilates and compacts the (small) bitmap, see block_dilate_compact
struct FusedCompact {
  uint32_t* dil_bits;
  int32_t* idx;
  int32_t* count;
  unsigned* sync;                // one word, zero at rest: blocks done
  int kh, kw, nwords, clear;
  int32_t* stream_counts;        // TRACK: the count split by stream (int32 [B]) and its accumulator
  int32_t* stream_acc;
  int B;
};

template <typename T, int VEC, int UPDATE, bool FUSE = false, bool TRACK = false, bool THR = false>
__global__ void __launch_bounds__(256)
detect_sparse_vec_kernel(const T* __restrict__ x, long long x_sb, long long x_sy, int xp,
                         T* __restrict__ st, long long s_sb, long long s_sy, int sp,
                         AuxPlanes aux, const int32_t* __restrict__ cand,
                         const int32_t* __restrict__ ncand, uint32_t* __restrict__ bits, int H,
                         int W, int C, int Wd, T thr, int glog, FusedCompact fc,
                         const float* __restrict__ thr_b) {
  const int n = *ncand;
  const int lane = threadIdx.x & 31;
  const int G = 1 << glog, ppw = 32 >> glog;
  const int sub = lane >> glog, gl = lane & (G - 1);
  const unsigned gmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (sub * G);
  const int P = H * W;
  const int cpv = (C + VEC - 1) / VEC, tail = C % VEC;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long j0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * ppw;
       j0 < n; j0 += nwarps * ppw) {
    const long long j = j0 + sub;
    const bool have = j < n;
    int b = 0, y = 0, xx = 0, gpix = 0;
    T tb = thr;
    if (have) {
      const int pix = __ldg(cand + j);
      gpix = pix;
      b = pix / P;
      const int p = pix - b * P;
      y = p / W;
      xx = p - y * W;
      tb = stream_thr<THR>(thr_b, b, thr);
    }
    const T* xb = x + b * x_sb + y * x_sy + (long long)xx * xp;
    T* sb = st + b * s_sb + y * s_sy + (long long)xx * sp;
    bool f = false;
    if (have) {
      for (int cc = gl; cc < cpv; cc += G) {
        uint4 xv = ldg16(xb + cc * VEC);
        const uint4 sv = ld16(sb + cc * VEC);
        if (tail && cc == cpv - 1) xv = merge_tail<T, VEC>(xv, sv, tail);
        f |= Chunk<T>::changed(sv, xv, tb);
        if (UPDATE == CB_UPDATE_ALL) store_state<T>(sb + cc * VEC, xv, aux, gpix, cc * VEC);
      }
    }
    const bool chg = (__ballot_sync(0xffffffffu, f) & gmask) != 0u;   // any lane of my group
    if (have && chg) {
      if (gl == 0) atomicOr(bits + ((long long)b * H + y) * Wd + (xx >> 5), 1u << (xx & 31));
      if (UPDATE == CB_UPDATE_CHANGED) {
        for (int cc = gl; cc < cpv; cc += G) {
          uint4 xv = ldg16(xb + cc * VEC);
          if (tail && cc == cpv - 1) xv = merge_tail<T, VEC>(xv, ld16(sb + cc * VEC), tail);
          store_state<T>(sb + cc * VEC, xv, aux, gpix, cc * VEC);
        }
      }
    }
  }
  if (FUSE) {
    __shared__ uint32_t s_win[kCompactWin];
    __shared__ int s_warp[8];
    __shared__ unsigned s_last;
    __threadfence();                                          // my bitmap bits precede my done-increment
    __syncthreads();
    if (threadIdx.x == 0) {
      s_last = atomicAdd(fc.sync, 1u) == gridDim.x - 1u;
      if (s_last) *fc.sync = 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    block_dilate_compact<TRACK>(bits, fc.dil_bits, fc.idx, fc.count, s_win, s_warp, H, W, Wd, fc.kh, fc.kw,
                                fc.nwords, fc.clear != 0, fc.stream_counts, fc.stream_acc, fc.B);
  }
}

template <typename T, int UPDATE, bool THR = false>
__global__ void __launch_bounds__(256)
detect_sparse_generic_kernel(const T* __restrict__ x, long long x_sb, long long x_sc,
                             long long x_sy, long long x_sx, T* __restrict__ st, long long s_sb,
                             long long s_sc, long long s_sy, long long s_sx, AuxPlanes aux,
                             const int32_t* __restrict__ cand, const int32_t* __restrict__ ncand,
                             uint32_t* __restrict__ bits, int H, int W, int C, int Wd, T thr,
                             const float* __restrict__ thr_b) {
  const int n = *ncand;
  const int P = H * W;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n;
       j += (long long)gridDim.x * blockDim.x) {
    const int pix = __ldg(cand + j);
    const int b = pix / P, p = pix - b * P;
    const int y = p / W, xx = p - y * W;
    const T* xp = x + b * x_sb + y * x_sy + xx * x_sx;
    T* sp = st + b * s_sb + y * s_sy + xx * s_sx;
    if (pixel_changed_scalar<T, UPDATE>(xp, x_sc, sp, s_sc, C, stream_thr<THR>(thr_b, b, thr), aux, (long long)pix))
      atomicOr(bits + ((long long)b * H + y) * Wd + (xx >> 5), 1u << (xx & 31));
  }
}

template <typename T, int VEC>
int launch_detect_sparse(cudaStream_t stream, const void* x, long long x_sb, long long x_sc,
                         long long x_sy, long long x_sx, void* state, long long s_sb,
                         long long s_sc, long long s_sy, long long s_sx, int aux_mode,
                         void* aux_hi, void* aux_lo, const int32_t* cand, const int32_t* ncand, uint32_t* bits, int B, int C,
                         int H, int W, float threshold, int update, int bits_are_clear,
                         const FusedCompact* fuse, const float* thr_b) {
  const int Wd = (W + 31) / 32;
  const long long words = (long long)B * H * Wd;
  if (words == 0) return 0;
  if (!bits_are_clear && cudaMemsetAsync(bits, 0, (size_t)words * 4, stream) != cudaSuccess)
    return fail(3, "change_detect_sparse: memset failed");
  const T thr = thr_cast<T>(threshold);
  AuxPlanes aux;
  if (int rc = make_aux<T>(aux, aux_mode, aux_hi, aux_lo, state, C)) return rc;
  const bool vec_ok = pixel_major_ok<T, VEC>(x, x_sb, x_sc, x_sy, x_sx, state, s_sb, s_sc, s_sy, s_sx, C);
  unsigned grid = (unsigned)(sm_count() * 16);
  const int glog = group_log2((C + VEC - 1) / VEC);
  {
    // small maps: no more blocks than there are pixels to look at (every block of the fused variant
    // passes through one atomic)
    const long long ppb = (long long)(32 >> glog) * 8;         // candidates per block and round
    const long long need = ((long long)B * H * W + ppb - 1) / ppb;
    if (need < (long long)grid) grid = (unsigned)(need < 1 ? 1 : need);
  }
  CB_CHECK_ARG(!fuse || (vec_ok && words <= kCompactWin), "change_detect_sparse_compact: needs pixel-major "
               "tensors and a bitmap of at most %d words", kCompactWin);
  FusedCompact fc = fuse ? *fuse : FusedCompact{nullptr, nullptr, nullptr, nullptr, 0, 0, 0, 0, nullptr, nullptr, 0};
  return dispatch_thr(thr_b, [&](auto R) { return dispatch_update(update, "change_detect_sparse", [&](auto U) {
    if (vec_ok && fuse && fc.stream_counts)
      cb::launch(detect_sparse_vec_kernel<T, VEC, U, true, true, R>, grid, 256, 0, stream, (const T*)x, x_sb, x_sy,
                 (int)x_sx, (T*)state, s_sb, s_sy, (int)s_sx, aux, cand, ncand, bits, H, W, C, Wd, thr, glog, fc, thr_b);
    else if (vec_ok && fuse)
      cb::launch(detect_sparse_vec_kernel<T, VEC, U, true, false, R>, grid, 256, 0, stream, (const T*)x, x_sb, x_sy,
                 (int)x_sx, (T*)state, s_sb, s_sy, (int)s_sx, aux, cand, ncand, bits, H, W, C, Wd, thr, glog, fc, thr_b);
    else if (vec_ok)
      cb::launch(detect_sparse_vec_kernel<T, VEC, U, false, false, R>, grid, 256, 0, stream, (const T*)x, x_sb, x_sy,
                 (int)x_sx, (T*)state, s_sb, s_sy, (int)s_sx, aux, cand, ncand, bits, H, W, C, Wd, thr, glog, fc, thr_b);
    else
      cb::launch(detect_sparse_generic_kernel<T, U, R>, grid, 256, 0, stream, (const T*)x, x_sb, x_sc, x_sy, x_sx,
                 (T*)state, s_sb, s_sc, s_sy, s_sx, aux, cand, ncand, bits, H, W, C, Wd, thr, thr_b);
    CB_CHECK_LAUNCH("change_detect_sparse");
    return 0;
  }); });
}

}  // namespace cb
