// compact.cuh -- change propagation (dilation) + ordered compaction, bitmap domain.
//
// Replaces the scatter-dilate of changeDetection_kernel (reference cbconv2d_cg_backend.cu:62-72),
// changePropagation_kernel (:101-124) and torch.nonzero(...).int() incl. its host sync
// (conv2d_cg.py:200-213).
//
// One thread owns one bitmap word (32 pixels): vertical OR of the raw rows in the window,
// horizontal dilation with funnel shifts across the neighbouring words, __popc for the count,
// a block scan plus a single-pass chained ("decoupled look-back") scan across tiles for the
// global offsets, then the set bits are expanded to ascending int32 pixel indices.
// Traffic: P/8 bitmap bytes (re-read (2kH+1)*3 times out of L1/L2) + 4n index bytes.
#pragma once
#include "cb_common.cuh"

namespace cb {

#ifndef CB_COMPACT_THREADS
#define CB_COMPACT_THREADS 512
#endif
#ifndef CB_COMPACT_WPT
#define CB_COMPACT_WPT 1
#endif
constexpr int kCompactThreads = CB_COMPACT_THREADS;
constexpr int kCompactWPT = CB_COMPACT_WPT;                  // words per thread
constexpr int kCompactTile = kCompactThreads * kCompactWPT;  // words per tile (16384 pixels; measured best of 256..2048)
constexpr int kCompactWin = 6144;                            // staged raw window (words, 24 KB)

constexpr int kCompactResidentTiles = 2 * 132;  // blocks that are co-resident on any B200 (>= 132 SMs, >= 2 per SM)
struct CompactHeader {                         // first 16 bytes of the workspace
  unsigned reserved, done, epoch, ticket;
};

__host__ __device__ inline size_t compact_ws_bytes(size_t nwords) {
  const size_t tiles = (nwords + kCompactTile - 1) / kCompactTile;
  return sizeof(CompactHeader) + 8 * (tiles + 1);
}

// tile_state word: [63:34] tag (epoch-derived, never 0) | [33:32] status | [31:0] value
__device__ __forceinline__ unsigned long long pack_state(unsigned tag, unsigned status, unsigned v) {
  return ((unsigned long long)tag << 34) | ((unsigned long long)status << 32) | v;
}

// One dilated bitmap word: vertical OR of the raw rows in the window, then horizontal dilation
// with funnel shifts across the neighbouring words.
// `win` holds raw words [win0, win0 + len) of the flat bitmap (staged in shared memory when the
// window fits, else the global bitmap itself with win0 = 0).
__device__ __forceinline__ unsigned dilated_word(const uint32_t* __restrict__ win, int win0, int r,
                                                 int y, int j, int H, int W, int Wd, int kh,
                                                 int kw) {
  unsigned vp = 0, vc = 0, vn = 0;
  const int y0 = max(0, y - kh), y1 = min(H - 1, y + kh);
  const uint32_t* row = win + ((r - y + y0) * Wd + j - win0);
  for (int yy = y0; yy <= y1; ++yy, row += Wd) {
    vc |= row[0];
    if (j > 0) vp |= row[-1];
    if (j + 1 < Wd) vn |= row[1];
  }
  unsigned d = vc;
  for (int dx = 1; dx <= kw; ++dx) {
    d |= (vc << dx) | (vp >> (32 - dx));       // source pixel dx to the left
    d |= (vc >> dx) | (vn << (32 - dx));       // source pixel dx to the right
  }
  if (j == Wd - 1 && (W & 31)) d &= (1u << (W & 31)) - 1u;
  return d;
}

// Word j of row (b, yo) of the 2x2/stride-2 pooled view of a bitmap with Hin x Win pixels:
// bit xo = OR of the four input bits of window (yo, xo).  Used to hand pooled-resolution change
// candidates from a CBPoolMax2d to the next layer.
__device__ __forceinline__ unsigned compress_pairs(unsigned v) {
  unsigned t = (v | (v >> 1)) & 0x55555555u;
  t = (t | (t >> 1)) & 0x33333333u;
  t = (t | (t >> 2)) & 0x0f0f0f0fu;
  t = (t | (t >> 4)) & 0x00ff00ffu;
  t = (t | (t >> 8)) & 0x0000ffffu;
  return t;
}
__device__ __forceinline__ unsigned pooled_word(const uint32_t* __restrict__ raw, int b, int yo,
                                                int j, int Hin, int Wdin, int oW) {
  unsigned v0 = 0, v1 = 0;
  for (int dy = 0; dy < 2; ++dy) {
    const int y = 2 * yo + dy;
    if (y < Hin) {
      const uint32_t* row = raw + ((long long)b * Hin + y) * Wdin;
      if (2 * j < Wdin) v0 |= __ldg(row + 2 * j);
      if (2 * j + 1 < Wdin) v1 |= __ldg(row + 2 * j + 1);
    }
  }
  unsigned d = compress_pairs(v0) | (compress_pairs(v1) << 16);
  const int rem = oW - j * 32;
  if (rem < 32) d &= (1u << rem) - 1u;
  return d;
}

// List mode: tiles are taken by ticket (atomicAdd on the header's `ticket`), not by blockIdx -- every
// predecessor of a running tile then holds an earlier ticket, i.e. is running or finished, whatever
// order the hardware dispatches blocks in, so the look-back cannot starve (as in CUB's single-pass
// scan).  Tile-only mode has no scan across tiles and keeps blockIdx, and so do grids small enough to
// be resident as a whole.
// TRACK: the count is also split by stream: every warp adds its words' popcounts to stream_acc[b]
// (int32 [B], zero at rest), and the last tile copies it to stream_counts[b] and zeroes it again.
template <bool TRACK>
__global__ void __launch_bounds__(kCompactThreads)
dilate_compact_kernel(const uint32_t* __restrict__ raw, uint32_t* __restrict__ dil_bits,
                      int8_t* __restrict__ dil_map, int32_t* __restrict__ idx,
                      int32_t* __restrict__ count, void* ws, int B, int H, int W, int Wd, int kh,
                      int kw, int nwords, int ntiles, int pool_hin, int pool_wdin,
                      uint32_t* __restrict__ clear_bits, int32_t* __restrict__ tile_ws, int tile_ty,
                      int tile_xp, int no_list, int32_t* __restrict__ stream_counts,
                      int32_t* __restrict__ stream_acc) {
  CompactHeader* hdr = reinterpret_cast<CompactHeader*>(ws);
  volatile unsigned long long* tstate =
      reinterpret_cast<volatile unsigned long long*>(reinterpret_cast<char*>(ws) + sizeof(CompactHeader));
  constexpr int NW = kCompactThreads / 32;
  __shared__ int s_warp[NW];
  __shared__ int s_base;
  __shared__ uint32_t s_win[kCompactWin];

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  int tile = blockIdx.x;
  // (up to 2 blocks per SM the whole grid is resident at once and no order can starve anybody: those
  //  launches skip the ticket -- one more dependent global round trip, 2 us inside a step)
  if (!no_list && ntiles > kCompactResidentTiles) {
    if (tid == 0) s_base = (int)atomicAdd(&hdr->ticket, 1u);
    __syncthreads();
    tile = s_base;
    __syncthreads();
  }
  const unsigned epoch = *reinterpret_cast<volatile unsigned*>(&hdr->epoch);
  const unsigned tag = epoch % 0x3ffffffeu + 1u;

  // ---- stage the raw words this tile can touch (tile +- kh rows +- 1 word): one round of
  //      independent coalesced loads instead of (2kh+1) dependent ones per word ----------------
  const uint32_t* win = raw;
  int win0 = 0;
  if (!pool_hin) {
    const int lo = max(0, tile * kCompactTile - kh * Wd - 1);
    const int hi = min(nwords, (tile + 1) * kCompactTile + kh * Wd + 1);
    if (hi - lo <= kCompactWin) {
      for (int i = tid; i < hi - lo; i += kCompactThreads) s_win[i] = __ldg(raw + lo + i);
      win = s_win;
      win0 = lo;
      __syncthreads();
    }
  }

  // ---- dilated words (consecutive words per thread keep the index order) ------------------
  unsigned d[kCompactWPT];
  unsigned twin[kCompactWPT];                                // tiles this thread stamped first
  int tt0[kCompactWPT];
  int cnt = 0;
  const int w0 = tile * kCompactTile + tid * kCompactWPT;    // 32-bit index math: nwords < 2^31
#pragma unroll
  for (int i = 0; i < kCompactWPT; ++i) {
    const int w = w0 + i;
    d[i] = 0;
    twin[i] = 0;
    tt0[i] = 0;
    if (w < nwords) {
      const int j = w % Wd;
      const int r = w / Wd;
      const int y = r % H;
      d[i] = pool_hin ? pooled_word(raw, r / H, y, j, pool_hin, pool_wdin, W)
                      : dilated_word(win, win0, r, y, j, H, W, Wd, kh, kw);
      if (dil_bits) dil_bits[w] = d[i];
    }
    if (tile_ws) {
      // dirty 8 x 16 output tiles for the tiled contraction (conv_tile.cuh): a word covers four
      // tiles of one tile row; the first word to stamp a tile with this launch's tag appends it
      // (unordered list, every tile once).  The four exchanges of a word are independent; their
      // results are only needed after the index expansion, where the append position is reserved
      // once per warp.
      uint32_t* stamp = reinterpret_cast<uint32_t*>(tile_ws) + 4;
      int t0 = 0;
      unsigned win = 0;
      if (w < nwords && d[i]) {
        const int j = w % Wd, r = w / Wd;
        t0 = ((r / H) * tile_ty + (r % H) / 16) * tile_xp + 4 * j;
        unsigned old[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          old[q] = ((d[i] >> (8 * q)) & 0xffu) ? atomicExch(stamp + t0 + q, tag) : tag;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (old[q] != tag) win |= 1u << q;
      }
      twin[i] = win;
      tt0[i] = t0;
    }
    cnt += __popc(d[i]);
    // (a word never spans two streams: rows are padded to whole words)
    if constexpr (TRACK) stream_add_warp(w < nwords ? w / Wd / H : -1, __popc(d[i]), stream_acc);
  }
  if constexpr (TRACK) __threadfence();       // my additions precede the block's done-increment

  if (no_list) {
    // tiles only (the consumer walks the tile list and masks rows with dil_bits): no ordered index
    // list, hence no scan across tiles -- the change count is a plain sum (hdr->reserved)
    int tot = cnt;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if (lane == 0 && tot) atomicAdd(&hdr->reserved, (unsigned)tot);
  } else {
  // ---- block scan of popcounts -----------------------------------------------------------
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int v = lane < NW ? s_warp[lane] : 0;
    int inc2 = v;
#pragma unroll
    for (int o = 1; o < NW; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, inc2, o);
      if (lane >= o) inc2 += n;
    }
    if (lane < NW) s_warp[lane] = inc2 - v;                  // exclusive warp offsets
    const int total = __shfl_sync(0xffffffffu, inc2, NW - 1);

    // ---- chained scan across tiles (decoupled look-back), warp 0 ----------------------------
    int exclusive = 0;
    if (tile > 0) {
      if (lane == 0) tstate[tile] = pack_state(tag, 1u, (unsigned)total);    // aggregate
      int look = tile - 1;
      while (true) {
        const int t = look - lane;
        unsigned long long st = 0;
        if (t >= 0) {
          do { st = tstate[t]; } while ((unsigned)(st >> 34) != tag);
        }
        const unsigned status = t >= 0 ? (unsigned)((st >> 32) & 3u) : 2u;   // before tile 0: prefix 0
        const int val = t >= 0 ? (int)(unsigned)(st & 0xffffffffu) : 0;
        const unsigned pm = __ballot_sync(0xffffffffu, status == 2u);
        const int first = pm ? __ffs(pm) - 1 : 32;           // nearest tile with a full prefix
        int part = lane <= first ? val : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        exclusive += part;
        if (pm) break;
        look -= 32;
      }
    }
    if (lane == 0) {
      tstate[tile] = pack_state(tag, 2u, (unsigned)(exclusive + total));     // inclusive prefix
      s_base = exclusive;
      if (tile == ntiles - 1) *count = exclusive + total;
    }
  }
  __syncthreads();

  // ---- expand set bits to ascending pixel indices ------------------------------------------
  int o = s_base + s_warp[wid] + (incl - cnt);
  if (kCompactWPT == 1 && !dil_map) {
    // warp-cooperative expansion: the warp walks its non-empty words; lane i writes bit i of the
    // current word at its rank -> the 32 stores of a dense word are one coalesced 128-byte line
    // (per-thread expansion writes 32 lines per instruction when a block of pixels changed)
    const int w = w0;
    const bool have = w < nwords && d[0] != 0u;
    const int jj = have ? w % Wd : 0, rr = have ? w / Wd : 0;
    const int mypix0 = rr * W + jj * 32;
    unsigned todo = __ballot_sync(0xffffffffu, have);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const unsigned dd = __shfl_sync(0xffffffffu, d[0], src);
      const int oo = __shfl_sync(0xffffffffu, o, src);
      const int pp = __shfl_sync(0xffffffffu, mypix0, src);
      if ((dd >> lane) & 1u) idx[oo + __popc(dd & ((1u << lane) - 1u))] = pp + lane;
    }
  } else {
#pragma unroll
  for (int i = 0; i < kCompactWPT; ++i) {
    const int w = w0 + i;
    if (w >= nwords) break;
    const int j = w % Wd;
    const int r = w / Wd;                                    // r = b*H + y
    const int pix0 = r * W + j * 32;
    unsigned dd = d[i];
    while (dd) {
      const int bit = __ffs(dd) - 1;
      idx[o++] = pix0 + bit;
      dd &= dd - 1;
    }
    if (dil_map) {
      const int n = min(32, W - j * 32);
      int8_t* m = dil_map + pix0;
      for (int q = 0; q < n; ++q) m[q] = (int8_t)((d[i] >> q) & 1u);
    }
  }
  }

  }   // !no_list

  // ---- append the tiles this warp stamped first ------------------------------------------------
  if (tile_ws) {
#pragma unroll
    for (int i = 0; i < kCompactWPT; ++i) {
      const unsigned win = twin[i];
      const int t0 = tt0[i];
      const int mine = __popc(win);
      int incl_t = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl_t, o);
        if (lane >= o) incl_t += v;
      }
      const int total_t = __shfl_sync(0xffffffffu, incl_t, 31);
      int base_t = 0;
      if (total_t) {
        if (lane == 31) base_t = atomicAdd(tile_ws, total_t);
        base_t = __shfl_sync(0xffffffffu, base_t, 31);
        int pos = 4 + B * tile_ty * tile_xp + base_t + incl_t - mine;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if ((win >> q) & 1u) tile_ws[pos++] = t0 + q;
      }
    }
    __syncthreads();                            // all appends of this block precede its done-increment
  }

  // ---- leave the workspace clean for the next launch ---------------------------------------
  __shared__ unsigned s_last;
  if (tid == 0) {
    __threadfence();
    const unsigned prev = atomicAdd(&hdr->done, 1u);
    s_last = prev == (unsigned)ntiles - 1u;
    if (s_last) {
      hdr->done = 0;
      hdr->ticket = 0;
      if (no_list) {                            // every block added its popcounts before its done-increment
        *count = (int32_t)*reinterpret_cast<volatile unsigned*>(&hdr->reserved);
        hdr->reserved = 0;
      }
      if (tile_ws) {                            // every block appended before its done-increment
        tile_ws[1] = *reinterpret_cast<volatile int32_t*>(tile_ws);
        tile_ws[0] = 0;
      }
      __threadfence();
      *reinterpret_cast<volatile unsigned*>(&hdr->epoch) = epoch + 1u;
    }
  }
  // The last tile to finish (every tile has read its raw window by then) may zero the raw
  // bitmap, so next frame's candidate detection can OR bits into it without a memset launch.
  if (clear_bits) {
    __syncthreads();
    if (s_last)
      for (int i = tid; i < nwords; i += kCompactThreads) clear_bits[i] = 0u;
  }
  if constexpr (TRACK) {
    __syncthreads();
    if (s_last) stream_publish(stream_acc, stream_counts, B);
  }
}

// ------------------------------------------------------------------------------------------------
// block_dilate_compact -- dilation + ordered compaction of a SMALL bitmap (<= kCompactWin words, e.g. one
// 368 x 368 map or eight 46 x 46 maps) by ONE thread block, called by the last block of the kernel that
// produced the raw bitmap (detect_sparse_vec_kernel<.., FUSE>): a layer on a small map then needs two
// launches per frame (detect + compact, contraction) instead of three -- such layers are bound by the
// dependent-launch chain, not by bytes (pose network: 92 layers of <= 4416 bitmap words at batch 1).
// Same results as dilate_compact_kernel: dilated bitmap, ascending index list, count; optional
// zeroing of the raw bitmap.  All threads of the block must call it; `s_win` holds kCompactWin words.
// TRACK: the count split by stream is written to stream_counts[0, B), through stream_acc as in
// dilate_compact_kernel.
// ------------------------------------------------------------------------------------------------
template <bool TRACK>
__device__ __forceinline__ void block_dilate_compact(uint32_t* __restrict__ raw, uint32_t* __restrict__ dil_bits,
                                                     int32_t* __restrict__ idx, int32_t* __restrict__ count,
                                                     uint32_t* s_win, int* s_warp, int H, int W, int Wd,
                                                     int kh, int kw, int nwords, bool clear,
                                                     int32_t* stream_counts, int32_t* stream_acc, int B) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, wid = tid >> 5, nwarp = nthr >> 5;
  for (int i = tid; i < nwords; i += nthr) s_win[i] = __ldcg(raw + i);     // (written by other blocks: L2)
  __syncthreads();
  const int wpt = (nwords + nthr - 1) / nthr;                              // consecutive words per thread
  const int w0 = tid * wpt, w1 = min(nwords, w0 + wpt);
  int cnt = 0;
  for (int w = w0; w < w1; ++w) {
    const int j = w % Wd, r = w / Wd;
    const unsigned d = dilated_word(s_win, 0, r, r % H, j, H, W, Wd, kh, kw);
    if (dil_bits) dil_bits[w] = d;
    cnt += __popc(d);
  }
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  int woff = 0, total = 0;
  for (int q = 0; q < nwarp; ++q) {
    const int v = s_warp[q];
    if (q < wid) woff += v;
    total += v;
  }
  int o = woff + incl - cnt;
  for (int w = w0; w < w1; ++w) {
    const int j = w % Wd, r = w / Wd;
    unsigned d = dilated_word(s_win, 0, r, r % H, j, H, W, Wd, kh, kw);
    const int pix0 = r * W + j * 32;
    while (d) {
      idx[o++] = pix0 + __ffs(d) - 1;
      d &= d - 1;
    }
  }
  if (tid == 0) *count = total;
  if constexpr (TRACK) {
    // word k of every thread in one warp-wide step (lanes hold ascending words of few streams)
    for (int k = 0; k < wpt; ++k) {
      const int w = w0 + k;
      const bool have = w < w1;
      const unsigned d = have ? dilated_word(s_win, 0, w / Wd, (w / Wd) % H, w % Wd, H, W, Wd, kh, kw) : 0u;
      stream_add_warp(have ? w / Wd / H : -1, __popc(d), stream_acc);
    }
    __threadfence();
    __syncthreads();
    stream_publish(stream_acc, stream_counts, B);
  }
  if (clear)
    for (int i = tid; i < nwords; i += nthr) raw[i] = 0u;
}

// ------------------------------------------------------------------------------------------------
// stream_bucket_kernel -- per-stream counts of an index list the layer did not build itself (handed on
// from upstream or by the user; any order): counts[b] = #{ j < *count : idx[j] / hw == b }.  `acc` is
// int32 [B + 1], zero at rest: the per-stream sums, then the finished-block counter; the last block
// copies the sums to `counts` and leaves `acc` zero.  Indices outside [0, B*hw) are not counted.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
stream_bucket_kernel(const int32_t* __restrict__ idx, const int32_t* __restrict__ count, int hw, int B,
                     int32_t* __restrict__ counts, int32_t* __restrict__ acc) {
  __shared__ unsigned s_last;
  const int n = *count;
  for (long long j0 = (long long)blockIdx.x * blockDim.x; j0 < n; j0 += (long long)gridDim.x * blockDim.x) {
    const long long j = j0 + threadIdx.x;
    int b = -1;
    if (j < n) {
      const int v = __ldg(idx + j);
      if (v >= 0 && v / hw < B) b = v / hw;
    }
    stream_add_warp(b, 1u, acc);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(reinterpret_cast<unsigned*>(acc + B), 1u) == gridDim.x - 1u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  stream_publish(acc, counts, B);
  if (threadIdx.x == 0) acc[B] = 0;
}

__global__ void map_to_bits_kernel(const int8_t* __restrict__ map, uint32_t* __restrict__ bits,
                                   int H, int W, int Wd, long long nwords) {
  const int lane = threadIdx.x & 31;
  const long long w = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= nwords) return;
  const int j = (int)(w % Wd);
  const long long r = w / Wd;
  const int x = j * 32 + lane;
  const bool f = x < W && map[r * W + x] != 0;
  const unsigned word = __ballot_sync(0xffffffffu, f);
  if (lane == 0) bits[w] = word;
}

}  // namespace cb
