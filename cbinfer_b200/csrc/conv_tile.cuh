// conv_tile.cuh -- spatially tiled contraction: TMA-staged halo tiles + implicit im2col through the
// UMMA shared-memory descriptors.
//
// Same job as conv_umma.cuh (reference genXMatrix_kernel cbconv2d_cg_backend.cu:138-161 + the cuBLAS
// GEMM conv2d_cg.py:342-349 + updateOutput_kernel cbconv2d_cg_backend.cu:175-189), for change sets
// that are spatially clustered (blocks, dense frames): instead of gathering every receptive-field
// tap of every changed pixel (kH*kW copies of each state pixel), the work unit is an 8 x 16 tile of
// output pixels that contains at least one changed pixel (tile list built by cb_dilate_compact_tiles):
//
//   * ONE cp.async.bulk.tensor.4d (TMA, tile mode, out-of-image = zero fill) per operand plane
//     stages the (8+kW-1) x (16+kH-1) halo of the pixel-major state in shared memory -- every state
//     pixel crosses L2 -> SM once per tile, not once per tap;
//   * the A operand of tcgen05.mma is never materialised: an 8-row core group of the canonical
//     K-major layout = 8 x-consecutive halo pixels (row pitch = pixel bytes = swizzle width:
//     16 B none / 32 B / 64 B / 128 B), group stride SBO = halo row pitch, and the descriptor's
//     start address is simply the tap's pixel -- the hardware swizzle is a function of the absolute
//     shared-memory address, so any 16/32/64/128-byte aligned start reads TMA-swizzled data
//     correctly (probed on the B200: tools/umma_tile_probe.cu).  16-byte pixels (<= 8 sixteen-bit
//     channels, the RGB input layer) take two taps per K=16 instruction with LBO = tap distance;
//     pixels wider than 128 B are staged as 128-byte channel blocks;
//   * weights stream through a TMA ring exactly as in conv_umma.cuh (or stay resident when the whole
//     filter bank fits the ring), accumulators are double-buffered in TMEM, the epilogue writes
//     only the rows whose bit is set in the dilated change bitmap (bias / ReLU / convert / one
//     contiguous channel run per pixel) -- untouched pixels keep their exact previous bits.
//
// Warp roles: 0 weight TMA, 1 halo TMA, 2 MMA issuer (+ TMEM alloc), 3 spare, 4.. epilogue.
#pragma once
#include "conv_umma.cuh"
#include "detect.cuh"
#include "pool.cuh"

namespace cb {

constexpr int TL_W = 8, TL_H = 16;             // output tile (pixels): 128 rows of the M dimension
constexpr int TL_NHALO = 2;                    // halo buffers (tile i+1 loads while tile i computes; 1 if smem is tight)
constexpr int TL_MAXB = 12;                    // weight ring slots
constexpr int TL_CTRL_BYTES = 512;

__host__ __device__ inline int tile_grid_y(int H) { return (H + TL_H - 1) / TL_H; }
__host__ __device__ inline int tile_grid_x(int W) { return (W + TL_W - 1) / TL_W; }
// tile row stride: a 32-pixel bitmap word covers 4 tiles, kept inside one group of four
__host__ __device__ inline int tile_grid_xp(int W) { return ((W + 31) / 32) * 4; }
// tile workspace (int32 words): [0] append counter, [1] number of dirty tiles of the last
// cb_dilate_compact_tiles, [2..3] pad, then NT epoch stamps, then the tile list (NT entries)
__host__ __device__ inline size_t tile_ws_words(int B, int H, int W) {
  return 4 + 2 * (size_t)B * tile_grid_y(H) * tile_grid_xp(W);
}

// -DCB_TILE_TRACE: per-CTA timeline of the tile kernel (clock64 relative to kernel entry) for
// tools/tile_trace.py; not compiled into the product library
#ifdef CB_TILE_TRACE
constexpr int TL_TRACE_EV = 32;
__device__ long long cb_tile_trace[2048 * TL_TRACE_EV];
#define TL_TRACE(ev)                                                                              \
  do {                                                                                            \
    if ((ev) < TL_TRACE_EV && blockIdx.x < 2048)                                                  \
      cb_tile_trace[blockIdx.x * TL_TRACE_EV + (ev)] = clock64() - trace_t0;                      \
  } while (0)
#else
#define TL_TRACE(ev) do { } while (0)
#endif

struct TileCtrl {
  uint64_t b_full[TL_MAXB], b_empty[TL_MAXB];
  uint64_t halo_full[TL_NHALO], halo_empty[TL_NHALO];
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base, pad;
};
static_assert(sizeof(TileCtrl) <= TL_CTRL_BYTES, "ctrl block too large");

struct TileGeom {
  int B, H, W, Wd, TY, TXp;      // images, bitmap row words, tile grid
  int kH, kW, HWX, HWY;          // filter, halo extent (pixels)
  int Cp, Kp, num_kb;            // operand channel pitch (elements), K = kH*kW*Cp, K blocks
  int pix_row;                   // bytes of one halo pixel in a plane: min(pixel bytes, 128)
  int nblk;                      // 128-byte channel blocks per pixel (1 when the pixel is <= 128 B)
  int plane_bytes;               // shared-memory bytes of one (operand, block) plane, 1024-aligned
  int nb;                        // weight ring slots; nb >= num_kb (one N tile): weights resident
  int nhalo;                     // halo buffers in use (<= TL_NHALO)
  int layout;                    // UMMA layout type of the A descriptors
  int Cout, CoutPad, Op, relu;
};

// Optional fused tail of the epilogue: change-based 2x2 / stride-2 max pooling of the tile's output
// (reference maxPool2d_kernel, cbconv2d_cg_backend.cu:199-227) + the NEXT layer's change detection on
// the re-pooled pixels (the job of cb_maxpool2x2_detect, pool.cuh), so conv -> pool -> detect is one
// launch.  An 8 x 16 tile holds 4 x 8 whole windows (tiles are aligned to even coordinates); the four
// pixels of a window are lanes l, l^1, l^8, l^9 of one epilogue warp.  Pixels of a touched window
// that were not recomputed are read back from the output map, so the pooled value is the maximum
// of exactly the stored values.  out == nullptr: no fusion.
struct PoolFuse {
  void* out;                     // pooled map (pixel-major, element type = the conv's output type)
  long long o_sb, o_sy;
  int op, oH, oW;
  void* nst;                     // next layer's previous-input state (same shape as the pooled map)
  long long n_sb, n_sy;
  int np;
  AuxPlanes aux;                 // its operand planes (fp32 layers)
  uint32_t* nbits;               // its raw change bitmap (kept clear by its compaction)
  float thr;
  int update;                    // CB_UPDATE_*
};

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1,
                                            int c2, int c3, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}

__host__ __device__ constexpr bool tile_merge(bool split3, int bn) { return split3 && 4 * bn <= 512; }
__host__ __device__ constexpr int tile_tmem_cols(bool split3, int bn) {
  const int c = 2 * (tile_merge(split3, bn) ? 2 * bn : bn);
  return c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512;
}

// A-operand descriptor of a halo plane: start address filled in per K step
__device__ __forceinline__ uint64_t tile_adesc_base(uint32_t sbo_bytes, int layout) {
  return ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}

template <typename T, typename TO, bool SPLIT3, int BN, bool THR = false>
__global__ void __launch_bounds__(128 + um_epi(BN), BN <= 16 ? 4 : BN <= 64 ? 2 : 1)
conv_tile_kernel(const __grid_constant__ CUtensorMap amap_hi, const __grid_constant__ CUtensorMap amap_lo,
                 const __grid_constant__ CUtensorMap wmap, int32_t* tile_ws,
                 const uint32_t* dil_bits, const float* __restrict__ bias,
                 TO* __restrict__ out, const TileGeom g, const PoolFuse pf, const float* __restrict__ thr_b) {
#ifdef CB_TILE_TRACE
  const long long trace_t0 = clock64();
  if (threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    if (blockIdx.x < 2048) cb_tile_trace[blockIdx.x * TL_TRACE_EV + 31] = (long long)gt;
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    if (blockIdx.x < 2048) cb_tile_trace[blockIdx.x * TL_TRACE_EV + 29] = (long long)smid + 1;
  }
#endif
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int ES = sizeof(T), BK = UM_ROW_BYTES / ES, UK = 32 / ES, KS = BK / UK;
  constexpr int NSPLIT = SPLIT3 ? 2 : 1;
  constexpr int B_BYTES = BN * UM_ROW_BYTES, B_STAGE = NSPLIT * B_BYTES;
  // 3x split with N <= 128: the two products that share the `hi` state operand run as ONE
  // instruction against the stacked [w_hi; w_lo] tile (N = 2*BN, columns BN.. hold a_hi*w_lo) and the
  // epilogue adds the halves -- two instructions per K step instead of three (small-N instructions
  // are issue-bound, not tensor-bound)
  constexpr bool MERGE = tile_merge(SPLIT3, BN);
  constexpr int ACC_COLS = MERGE ? 2 * BN : BN;                // TMEM columns of one accumulator
  constexpr int TMEM_COLS = tile_tmem_cols(SPLIT3, BN);
  constexpr int EPI = um_epi(BN);
  // dirty tiles (cb_dilate_compact_tiles: written by another grid, hence L2 loads); the shuffle makes
  // the value uniform for the compiler
  const int ntl = __shfl_sync(0xffffffffu, __ldcg(tile_ws + 1), 0);
  const int ntiles_n = g.CoutPad / BN;
  const long long total = (long long)ntl * ntiles_n;
  if ((long long)blockIdx.x >= total) return;                // CTA-uniform, before any barrier / alloc
  if (smem_u32(smem) & 1023u) __trap();
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);    // provably warp-uniform role index
  const int NT = g.B * g.TY * g.TXp;
  const int32_t* tiles = tile_ws + 4 + NT;
  auto tile_at = [&](long long w) { return __ldcg(tiles + (int)(w / ntiles_n)); };
  const int halo_stage = NSPLIT * g.nblk * g.plane_bytes;
  uint8_t* bring = smem + g.nhalo * halo_stage;
  TileCtrl* ctrl = reinterpret_cast<TileCtrl*>(bring + g.nb * B_STAGE);
  const bool resident = ntiles_n == 1 && g.num_kb <= g.nb;
  const int ph = (g.kH - 1) / 2, pw = (g.kW - 1) / 2;

  if (tid == 0) {
    for (int s = 0; s < TL_MAXB; ++s) {
      mbar_init(&ctrl->b_full[s], 1);
      mbar_init(&ctrl->b_empty[s], 1);
    }
    for (int b = 0; b < TL_NHALO; ++b) {
      mbar_init(&ctrl->halo_full[b], 1);
      mbar_init(&ctrl->halo_empty[b], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&ctrl->tmem_full[b], 1);
      mbar_init(&ctrl->tmem_empty[b], EPI);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&ctrl->tmem_base)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&wmap)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&amap_hi)) : "memory");
    if (SPLIT3) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&amap_lo)) : "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (tid == 0) TL_TRACE(0);                                 // prologue done
  const uint32_t tmem_base = ctrl->tmem_base;
  const int tiles_per_img = g.TY * g.TXp;

  if (warp == 0) {
    // =============================== weight tiles (TMA ring) ================================
    // (whole warp, uniform operands, one elected lane issues: see the MMA warp)
    const bool leader = elect_one();
    const int nb = g.nb, num_kb = g.num_kb, CoutPad = g.CoutPad;
    uint32_t stage = 0, phase = 0;
    int it = 0;
    for (long long w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      if (resident && it > 0) break;
      const int nt = (int)(w % ntiles_n);
      for (int kb = 0; kb < num_kb; ++kb) {
        if (!resident) mbar_wait(&ctrl->b_empty[stage], phase ^ 1u);
        if (leader) {
          const uint32_t b_hi = smem_u32(bring + stage * B_STAGE);
          mbar_arrive_expect_tx(&ctrl->b_full[stage], (uint32_t)B_STAGE);
          tma_load_2d(b_hi, &wmap, kb * BK, nt * BN, &ctrl->b_full[stage]);
          if (SPLIT3) tma_load_2d(b_hi + B_BYTES, &wmap, kb * BK, CoutPad + nt * BN, &ctrl->b_full[stage]);
        }
        __syncwarp();
        if (++stage == (uint32_t)nb) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =============================== halo tiles (TMA, tile mode, zero fill) =================
    const bool leader = elect_one();
    const int BE = g.pix_row / ES;                           // channels per 128-byte block
    const uint32_t box_bytes = (uint32_t)(g.HWX * g.HWY * g.pix_row);
    const int nhalo = g.nhalo, nblk = g.nblk, plane_bytes = g.plane_bytes, TXp = g.TXp;
    int it = 0;
    for (long long w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      const int tile = __shfl_sync(0xffffffffu, tile_at(w), 0);
      const int b = tile / tiles_per_img, r = tile - b * tiles_per_img;
      const int ty = r / TXp, tx = r - ty * TXp;
      const int hb = it % nhalo;
      mbar_wait(&ctrl->halo_empty[hb], (uint32_t)(((it / nhalo) & 1) ^ 1));
      if (leader) {
        TL_TRACE(1 + it * 6 + 0);                            // halo TMA issued
        mbar_arrive_expect_tx(&ctrl->halo_full[hb], (uint32_t)(NSPLIT * nblk) * box_bytes);
        const uint32_t dst = smem_u32(smem + hb * halo_stage);
        for (int blk = 0; blk < nblk; ++blk) {
          tma_load_4d(dst + blk * plane_bytes, &amap_hi, blk * BE, tx * TL_W - pw, ty * TL_H - ph, b,
                      &ctrl->halo_full[hb]);
          if (SPLIT3)
            tma_load_4d(dst + (nblk + blk) * plane_bytes, &amap_lo, blk * BE, tx * TL_W - pw,
                        ty * TL_H - ph, b, &ctrl->halo_full[hb]);
        }
      }
      __syncwarp();
    }
  } else if (warp == 2) {
    // =============================== MMA issuer ==============================================
    // The WHOLE warp runs this loop -- control flow, barrier waits and every descriptor are then
    // warp-uniform, so they live in uniform registers and a tcgen05.mma costs a handful of
    // uniform-ALU instructions; one elected lane issues.  (Under `if (lane == 0)` the compiler cannot
    // prove uniformity and wraps every UTCHMMA in an ELECT / 5x R2UR / branch "waterfall" loop:
    // ~150 cycles per instruction, measured -- more than the tensor time of an N <= 256 tile.)
    // Descriptor offsets follow the K order (ky, kx, ci) incrementally; no table, no divisions.
    constexpr int KIND = sizeof(T) == 4 ? 0 : 1;
    constexpr int FMT = sizeof(T) == 4 ? 2 : (std::is_same<T, __half>::value ? 0 : 1);
    const uint32_t idesc = umma_idesc(FMT, BN);
    const uint32_t idesc2 = umma_idesc(FMT, MERGE ? 2 * BN : BN);
    // descriptors as (hi word: SBO | version | layout, constant) + (lo word: start >> 4 | LBO >> 4 << 16,
    // running): one uniform add per operand and K step (the uniform datapath executes in order at
    // ~10 cycles per dependent instruction, so every instruction in this loop is on the issue path)
    const uint32_t a_hi32 = (uint32_t)(tile_adesc_base((uint32_t)(g.HWX * g.pix_row), g.layout) >> 32);
    const uint32_t b_hi32 = (uint32_t)(umma_desc(0) >> 32);
    const bool leader = elect_one();
    const int pixb = g.Cp * ES, kH = g.kH, kW = g.kW, nblk = g.nblk, nhalo = g.nhalo, nb = g.nb;
    const int ntaps = kH * kW;
    const uint32_t pix16 = (uint32_t)g.pix_row >> 4;          // one halo pixel, in 16-byte units
    const uint32_t row16 = (uint32_t)g.HWX * pix16;          // one halo row
    const uint32_t plane16 = (uint32_t)g.plane_bytes >> 4;   // one channel-block plane
    const uint32_t lo16 = (uint32_t)nblk * plane16;          // hi plane(s) -> lo plane(s)
    const int steps_in = g.pix_row >> 5;                     // K steps inside one 128-byte block of a pixel
    const uint32_t bring16 = (smem_u32(bring) & 0x3FFFFu) >> 4;
    uint32_t stage = 0, phase = 0;
    int it = 0;
    for (long long w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      const int hb = it % nhalo;
      const uint32_t ab = (uint32_t)it & 1u, aph = ((uint32_t)it >> 1) & 1u;
      mbar_wait(&ctrl->halo_full[hb], (uint32_t)((it / nhalo) & 1));
      if (leader) TL_TRACE(1 + it * 6 + 1);                  // halo landed
      mbar_wait(&ctrl->tmem_empty[ab], aph ^ 1u);
      tc_fence_after();
      const uint32_t a16 = (smem_u32(smem + hb * halo_stage) & 0x3FFFFu) >> 4;
      const uint32_t tmem_d = tmem_base + ab * (uint32_t)ACC_COLS;
      uint32_t acc = 0, b_run = 0;
      int ks = 0, kbi = 0;
      // one K step: 32 bytes of K from the halo (A lo word `alo`) against the running weight slice
      auto step = [&](uint32_t alo) {
        if (ks == 0) {                                       // next weight stage (KS K steps each)
          if (resident) {
            stage = (uint32_t)(kbi % nb);
            if (it == 0 && kbi < nb) mbar_wait(&ctrl->b_full[stage], 0u);
          } else {
            mbar_wait(&ctrl->b_full[stage], phase);
          }
          tc_fence_after();
          if (leader && kbi == 0) TL_TRACE(1 + it * 6 + 5);  // first weight stage landed
          b_run = (bring16 + stage * (uint32_t)(B_STAGE >> 4)) | (1u << 16);
        }
        if (leader) {
          const uint64_t ad_hi = ((uint64_t)a_hi32 << 32) | alo;
          const uint64_t bd_hi = ((uint64_t)b_hi32 << 32) | b_run;
          if (MERGE) {
            const uint64_t ad_lo = ((uint64_t)a_hi32 << 32) | (alo + lo16);
            umma<KIND>(tmem_d, ad_hi, bd_hi, idesc2, acc);   // a_hi * [w_hi | w_lo]  (w_lo tile follows w_hi)
            umma<KIND>(tmem_d, ad_lo, bd_hi, idesc, 1u);     // a_lo * w_hi
          } else if (SPLIT3) {
            const uint64_t ad_lo = ((uint64_t)a_hi32 << 32) | (alo + lo16);
            const uint64_t bd_lo = ((uint64_t)b_hi32 << 32) | (b_run + (uint32_t)(B_BYTES >> 4));
            umma<KIND>(tmem_d, ad_lo, bd_hi, idesc, acc);
            umma<KIND>(tmem_d, ad_hi, bd_lo, idesc, 1u);
            umma<KIND>(tmem_d, ad_hi, bd_hi, idesc, 1u);
          } else {
            umma<KIND>(tmem_d, ad_hi, bd_hi, idesc, acc);
          }
        }
        acc = 1u;
        b_run += 2;
        if (++ks == KS) {
          ks = 0;
          ++kbi;
          if (!resident) {
            if (leader) umma_commit(&ctrl->b_empty[stage]);  // frees the weight stage when done
            if (++stage == (uint32_t)nb) { stage = 0; phase ^= 1u; }
          }
        }
      };
      if (pixb == 16) {
        // 16-byte pixels: two taps per instruction, LBO = distance to the second tap (next pixel,
        // or the first pixel of the next filter row: HWX - kW + 1 = TL_W pixels on)
        uint32_t u = a16;
        int kx = 0;
        for (int tap = 0; tap < ntaps; tap += 2) {
          const uint32_t u1 = u + (kx + 1 == kW ? (uint32_t)TL_W : 1u);
          const int kx1 = kx + 1 == kW ? 0 : kx + 1;
          // (a second tap beyond the filter meets zero weights: it re-reads the first one, so no
          //  uninitialised shared memory enters the product)
          const uint32_t lbo = tap + 1 < ntaps ? u1 - u : 0u;
          step(u | (lbo << 16));
          u = u1 + (kx1 + 1 == kW ? (uint32_t)TL_W : 1u);
          kx = kx1 + 1 == kW ? 0 : kx1 + 1;
        }
      } else {
        uint32_t arow = a16 | (1u << 16);
        for (int ky = 0; ky < kH; ++ky, arow += row16) {
          uint32_t atap = arow;
          for (int kx = 0; kx < kW; ++kx, atap += pix16) {
            uint32_t ablk = atap;
            for (int blk = 0; blk < nblk; ++blk, ablk += plane16)
              for (int j = 0; j < steps_in; ++j) step(ablk + 2u * (uint32_t)j);
          }
        }
      }
      if (ks != 0 && !resident) {                            // partial last weight stage
        if (leader) umma_commit(&ctrl->b_empty[stage]);
        if (++stage == (uint32_t)nb) { stage = 0; phase ^= 1u; }
      }
      if (leader) {
        umma_commit(&ctrl->tmem_full[ab]);                   // accumulator complete
        umma_commit(&ctrl->halo_empty[hb]);                  // halo buffer consumed
        TL_TRACE(1 + it * 6 + 2);                            // all MMAs of the tile issued
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // =============================== epilogue: TMEM -> bias / ReLU -> changed rows only ======
    const int q = warp & 3;                                  // TMEM lane quarter of this warp
    const int row = q * 32 + lane;
    const int rty = row >> 3, rtx = row & 7;
    constexpr int OVEC = 16 / (int)sizeof(TO);
    constexpr int NGROUP = EPI / 128;
    constexpr int COLS = (BN / NGROUP) < 16 ? 16 : (BN / NGROUP);
    const int cbeg = ((warp - 4) >> 2) * COLS;
    const bool pooling = pf.out != nullptr;                  // (host: BN <= 64, one N tile, Cout % 16 == 0)
    const TO pthr = thr_cast<TO>(pf.thr);
    int it = 0;
    for (long long w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      const int tile = tile_at(w);
      const int nt = (int)(w % ntiles_n);
      const int b = tile / tiles_per_img, r = tile - b * tiles_per_img;
      const int ty = r / g.TXp, tx = r - ty * g.TXp;
      const int y = ty * TL_H + rty, x = tx * TL_W + rtx;
      const bool inimg = y < g.H && x < g.W;
      bool on = false;
      if (inimg)
        on = (__ldcg(dil_bits + ((long long)b * g.H + y) * g.Wd + (x >> 5)) >> (x & 31)) & 1u;
      const uint32_t ab = (uint32_t)it & 1u, aph = ((uint32_t)it >> 1) & 1u;
      TO* orow = out + (((long long)b * g.H + (inimg ? y : 0)) * g.W + (inimg ? x : 0)) * g.Op;
      const unsigned onmask = __ballot_sync(0xffffffffu, on);
      // fused pooling: window = lanes (l & ~9) + {0, 1, 8, 9}; its top-left lane owns the pooled pixel
      const unsigned wmask = 0x303u << (lane & 0x16);
      const bool win_on = pooling && (onmask & wmask) != 0u;
      const int yo = y >> 1, xo = x >> 1;
      const bool owner = win_on && (lane & 9) == 0 && yo < pf.oH && xo < pf.oW;
      TO* po = reinterpret_cast<TO*>(pf.out) + b * pf.o_sb + yo * pf.o_sy + (long long)xo * pf.op;
      TO* ns = reinterpret_cast<TO*>(pf.nst) + b * pf.n_sb + yo * pf.n_sy + (long long)xo * pf.np;
      const long long opix = ((long long)b * pf.oH + yo) * pf.oW + xo;
      const TO tthr = stream_thr<THR>(thr_b, b, pthr);        // (THR: pooling) a tile lies in one image
      // What the pooling tail reads from global memory -- the stored values of a touched window's
      // untouched pixels, the next layer's state row of the window's owner -- has not been seen for a
      // frame: with the loads inside the column loop a tile's epilogue was a chain of 8 dependent
      // DRAM round trips (trace, cold: 6-8 us per tile for 64 channels).  The first 16-column slice is
      // fetched BEFORE waiting for the accumulator (hidden behind the tile's MMAs), every further slice
      // one iteration ahead.
      // (one-slice layers, BN <= 16, keep their loads inside the loop: they run four CTAs per SM on 64
      //  registers per thread, and 8 more vector registers across the wait would halve that)
      constexpr bool EARLY = BN > 16;
      constexpr int NV = 16 / OVEC;
      uint4 orv[NV], nsv[NV];
      auto fetch = [&](int c0, uint4* o, uint4* n) {
        const int co0 = nt * BN + c0;
        const bool need_o = win_on && inimg && !on && co0 < g.Cout;
        const bool need_n = owner && co0 < g.Cout;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          o[i] = need_o ? ld16(orow + co0 + i * OVEC) : make_uint4(0u, 0u, 0u, 0u);
          n[i] = need_n ? ld16(ns + co0 + i * OVEC) : make_uint4(0u, 0u, 0u, 0u);
        }
      };
      if (EARLY && pooling && onmask) fetch(cbeg, orv, nsv);
      mbar_wait(&ctrl->tmem_full[ab], aph);
      tc_fence_after();
      if (warp == 4 && lane == 0) TL_TRACE(1 + it * 6 + 3);  // accumulator complete (epilogue starts)
      const uint32_t trow = tmem_base + ab * (uint32_t)ACC_COLS + ((uint32_t)(q * 32) << 16);
      bool pchg = false;
      if (onmask) {
#pragma unroll 1
        for (int c0 = cbeg; c0 < cbeg + COLS && c0 < BN; c0 += 16) {
          uint4 orn[NV], nsn[NV];
          const bool more = EARLY && pooling && c0 + 16 < cbeg + COLS && c0 + 16 < BN;
          if (more) fetch(c0 + 16, orn, nsn);
          uint32_t acc[16];
          tmem_ld16(trow + (uint32_t)c0, acc);
          if (MERGE) {
            uint32_t acc2[16];
            tmem_ld16(trow + (uint32_t)(BN + c0), acc2);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = __float_as_uint(__uint_as_float(acc[i]) + __uint_as_float(acc2[i]));
          } else {
            tmem_ld_wait();
          }
          const int co0 = nt * BN + c0;
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = -INFINITY;
          if (on && co0 < g.Cout) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int co = co0 + i;
              float t = __uint_as_float(acc[i]) + (co < g.Cout ? __ldg(bias + co) : 0.f);
              if ((g.relu & 1) && t <= 0.f) t = 0.f;
              f[i] = t;
            }
            if (co0 + 16 <= g.Cout && (g.Op % OVEC) == 0) {
              if (sizeof(TO) == 4) {
#pragma unroll
                for (int i = 0; i < 16; i += 4)
                  *reinterpret_cast<float4*>(reinterpret_cast<float*>(orow) + co0 + i) =
                      make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
              } else {
#pragma unroll
                for (int i = 0; i < 16; i += 8) {
                  TO h[8];
#pragma unroll
                  for (int e = 0; e < 8; ++e) {
                    h[e] = from_float<TO>(f[i + e]);
                    f[i + e] = to_float(h[e]);               // the stored (rounded) value is what gets pooled
                  }
                  *reinterpret_cast<uint4*>(orow + co0 + i) = *reinterpret_cast<uint4*>(h);
                }
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (co0 + i < g.Cout) orow[co0 + i] = from_float<TO>(f[i]);
            }
          } else if (win_on && inimg && co0 < g.Cout) {
            // an untouched pixel of a touched window: its stored value takes part in the maximum
#pragma unroll
            for (int i = 0; i < 16; i += OVEC) {
              const uint4 v = EARLY ? orv[i / OVEC] : ld16(orow + co0 + i);
              const TO* e = reinterpret_cast<const TO*>(&v);
#pragma unroll
              for (int k = 0; k < OVEC; ++k) f[i + k] = to_float(e[k]);
            }
          }
          if (pooling) {
            // 2x2 maximum across the window's lanes, then the owner re-pools, thresholds against the
            // next layer's state and maintains it (cb_maxpool2x2_detect semantics)
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              f[i] = fmaxf(f[i], __shfl_xor_sync(0xffffffffu, f[i], 1));
              f[i] = fmaxf(f[i], __shfl_xor_sync(0xffffffffu, f[i], 8));
            }
            if (owner && co0 < g.Cout) {
#pragma unroll
              for (int i = 0; i < 16; i += OVEC) {
                TO h[OVEC];
#pragma unroll
                for (int k = 0; k < OVEC; ++k) h[k] = from_float<TO>(f[i + k]);
                const uint4 res = *reinterpret_cast<uint4*>(h);
                st16(po + co0 + i, res);
                const uint4 sv = EARLY ? nsv[i / OVEC] : ld16(ns + co0 + i);
                pchg |= Chunk<TO>::changed(sv, res, tthr);
                if (pf.update == CB_UPDATE_ALL) store_state<TO>(ns + co0 + i, res, pf.aux, opix, co0 + i);
              }
            }
          }
          if (more) {
#pragma unroll
            for (int i = 0; i < NV; ++i) {
              orv[i] = orn[i];
              nsv[i] = nsn[i];
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&ctrl->tmem_empty[ab]);
      if (owner && pchg) {
        const int oWd = (pf.oW + 31) >> 5;
        atomicOr(pf.nbits + ((long long)b * pf.oH + yo) * oWd + (xo >> 5), 1u << (xo & 31));
        if (pf.update == CB_UPDATE_CHANGED)                  // feedback: accept the new pooled pixel
          for (int c = 0; c < g.Cout; c += OVEC)
            store_state<TO>(ns + c, ld16(po + c), pf.aux, opix, c);
      }
      if (warp == 4 && lane == 0) TL_TRACE(1 + it * 6 + 4);  // epilogue of the tile done
    }
  }

  tc_fence_before();
  __syncthreads();
  if (tid == 0) TL_TRACE(30);                                // all roles done
#ifdef CB_TILE_TRACE
  if (tid == 0 && blockIdx.x < 2048) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    cb_tile_trace[blockIdx.x * TL_TRACE_EV + 28] = (long long)gt;
  }
#endif
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

// ---- host side ---------------------------------------------------------------------------------
struct TilePlan {
  bool ok;
  TileGeom g;
  int smem_bytes, occ;
  long long mma_clk_per_tile;    // rough tensor-pipe time of one tile (policy: cheap tiles only)
  bool short_k;                  // policy: short single-pass K loop, one N tile
};

// Can (and should) this layer run on the tile path?  es = operand element bytes, Cp = operand channel
// pitch, bn = N tile.
inline TilePlan tile_plan(int es, bool split3, int bn, int Cp, int B, int H, int W, int Cout,
                          int CoutPad, int Op, int kH, int kW, int relu) {
  TilePlan p;
  p.ok = false;
  p.short_k = false;
  TileGeom& g = p.g;
  const int pixb = Cp * es;
  if (!(pixb == 16 || pixb == 32 || pixb == 64 || (pixb % 128) == 0)) return p;
  if (kH * kW == 1 || !(kH & 1) || !(kW & 1)) return p;      // 1x1: nothing to reuse
  const int nsplit = split3 ? 2 : 1;
  const int bk = UM_ROW_BYTES / es;
  g.B = B; g.H = H; g.W = W; g.Wd = (W + 31) / 32;
  g.TY = tile_grid_y(H); g.TXp = tile_grid_xp(W);
  g.kH = kH; g.kW = kW; g.HWX = TL_W + kW - 1; g.HWY = TL_H + kH - 1;
  if (g.HWX > 256 || g.HWY > 256) return p;
  g.Cp = Cp; g.Kp = kH * kW * Cp;
  g.num_kb = (g.Kp + bk - 1) / bk;
  g.pix_row = pixb < 128 ? pixb : 128;
  g.nblk = pixb > 128 ? pixb / 128 : 1;
  g.plane_bytes = (g.HWX * g.HWY * g.pix_row + 1023) / 1024 * 1024;
  g.layout = g.pix_row == 16 ? 0 : g.pix_row == 32 ? 6 : g.pix_row == 64 ? 4 : 2;
  g.Cout = Cout; g.CoutPad = CoutPad; g.Op = Op; g.relu = relu ? 1 : 0;
  if ((long long)g.HWX * g.pix_row >= (1 << 18)) return p;
  const int b_stage = nsplit * bn * UM_ROW_BYTES;
  const int tmem_cols = tile_tmem_cols(split3, bn);
  const int budget2 = 112 * 1024, budget1 = 224 * 1024;
  const bool one_ntile = CoutPad == bn;
  int nb = 0, occ = 1, fixed = 0;
  g.nhalo = 0;
  for (int nh = TL_NHALO; nh >= 1 && !g.nhalo; --nh) {       // fewer halo buffers when smem is tight
    fixed = nh * nsplit * g.nblk * g.plane_bytes + TL_CTRL_BYTES;
    if (nh == TL_NHALO && one_ntile && g.num_kb <= TL_MAXB && fixed + g.num_kb * b_stage <= budget2 &&
        2 * tmem_cols <= 512) {
      nb = g.num_kb; occ = 2; g.nhalo = nh;                  // resident weights, two CTAs per SM
    } else if (nh == TL_NHALO && budget2 > fixed && (budget2 - fixed) / b_stage >= 4 && 2 * tmem_cols <= 512) {
      nb = (budget2 - fixed) / b_stage; occ = 2; g.nhalo = nh;
    } else if (budget1 > fixed && (budget1 - fixed) / b_stage >= (nh == 1 ? 2 : 3)) {
      nb = (budget1 - fixed) / b_stage; occ = 1; g.nhalo = nh;
      if (one_ntile && g.num_kb <= TL_MAXB && nb >= g.num_kb) nb = g.num_kb;
    }
  }
  if (!g.nhalo) return p;
  if (nb > TL_MAXB) nb = TL_MAXB;
  if (occ == 2) {
    // small layers (e.g. the RGB input layer: 50 KB, 64 TMEM columns): up to four CTAs per SM -- their
    // instructions are issue-bound, more issuing warps keep the tensor pipe busier
    int o = (227 * 1024) / (fixed + nb * b_stage + 1024);
    if (o > 512 / tmem_cols) o = 512 / tmem_cols;
    if (o > 4) o = 4;
    if (bn > 16 && o > 2) o = 2;                             // register side: __launch_bounds__ of the kernel
    if (o > occ) occ = o;
  }
  g.nb = nb;
  p.occ = occ;
  p.smem_bytes = fixed + nb * b_stage;
  const int uk = 32 / es;
  const long long ksteps = (g.Kp + uk - 1) / uk;
  const long long per = bn / 2 < 32 ? 32 : bn / 2;           // cycles per instruction (N/2, smem floor ~32)
  p.mma_clk_per_tile = ksteps * (split3 ? 3 : 1) * per * (CoutPad / bn);
  // single-pass layers whose K loop is short (<= 224 K steps, e.g. 64 channels x 7x7 in 16-bit data) and
  // that need one N tile: a tile is then cheaper than the index-list kernel's split-K round trip at every
  // change rate (measured, tools/tile_bench.py --set policy: 64->256 7x7 bf16 28 vs 39 us at 1 %, 29 vs 37
  // at 5 %, 180 vs 239 at 100 %), while 128 channels x 7x7 (392 K steps) only wins when everything changed
  p.short_k = !split3 && ksteps <= 224 && CoutPad == bn;
  p.ok = true;
  return p;
}

template <typename T>
inline CUtensorMapDataType tmap_dtype() {
  return sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
         : std::is_same<T, __half>::value ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                          : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

template <typename T, typename TO, bool SPLIT3, int BN, bool THR = false>
int launch_conv_tile(cudaStream_t s, const void* state, const void* state_lo, const int32_t* tile_ws,
                     const uint32_t* dil_bits, const void* packed, const float* bias, void* out,
                     const TilePlan& plan, const PoolFuse& pf, const float* thr_b) {
  const TileGeom& g = plan.g;
  auto enc = tensor_map_encoder();
  if (!enc) return fail(3, "conv_update_tiled: cuTensorMapEncodeTiled unavailable");
  constexpr int ES = sizeof(T), BK = UM_ROW_BYTES / ES, NSPLIT = SPLIT3 ? 2 : 1;
  const int KpPad = g.num_kb * BK;
  alignas(64) CUtensorMap wmap, amap[2];
  {
    const cuuint64_t gdim[2] = {(cuuint64_t)KpPad, (cuuint64_t)(NSPLIT * g.CoutPad)};
    const cuuint64_t gstr[1] = {(cuuint64_t)KpPad * ES};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BN};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(&wmap, tmap_dtype<T>(), 2, const_cast<void*>(packed), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(3, "conv_update_tiled: weight tensor map failed (%d)", (int)r);
  }
  const CUtensorMapSwizzle sw = g.pix_row == 16 ? CU_TENSOR_MAP_SWIZZLE_NONE
                                : g.pix_row == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                : g.pix_row == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  for (int pl = 0; pl < NSPLIT; ++pl) {
    const void* base = pl ? state_lo : state;
    const cuuint64_t pixb = (cuuint64_t)g.Cp * ES;
    const cuuint64_t gdim[4] = {(cuuint64_t)g.Cp, (cuuint64_t)g.W, (cuuint64_t)g.H, (cuuint64_t)g.B};
    const cuuint64_t gstr[3] = {pixb, pixb * g.W, pixb * g.W * g.H};
    const cuuint32_t box[4] = {(cuuint32_t)(g.pix_row / ES), (cuuint32_t)g.HWX, (cuuint32_t)g.HWY, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = enc(&amap[pl], tmap_dtype<T>(), 4, const_cast<void*>(base), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(3, "conv_update_tiled: state tensor map failed (%d)", (int)r);
  }
  if (!SPLIT3) amap[1] = amap[0];
  auto kern = conv_tile_kernel<T, TO, SPLIT3, BN, THR>;
  static thread_local int attr_dev = -1;
  int dev = 0;
  cudaGetDevice(&dev);
  if (attr_dev != dev) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return fail(3, "conv_update_tiled: cannot reserve shared memory");
    attr_dev = dev;
  }
  const long long max_items = (long long)g.B * g.TY * tile_grid_x(g.W) * (g.CoutPad / BN);
  // (the plan counts shared memory and TMEM columns; the register side is pinned by the kernel's
  //  __launch_bounds__: 4 CTAs per SM for N <= 16, 2 for N <= 64)
  long long grid = (long long)sm_count() * plan.occ;
  if (grid > max_items) grid = max_items;
  if (grid < 1) grid = 1;
  cb::launch(kern, dim3((unsigned)grid), dim3(128 + um_epi(BN)), (size_t)plan.smem_bytes, s, amap[0], amap[1],
             wmap, const_cast<int32_t*>(tile_ws), dil_bits, bias, (TO*)out, g, pf, thr_b);
  CB_CHECK_LAUNCH("conv_update_tiled");
  return 0;
}

// policy threshold: tiles whose tensor work is at most this many cycles (denser layers keep the
// index-list kernel, whose M tiles hold changed pixels only)
constexpr long long kTileClkLimit = 12000;

// fused pooling: one epilogue warp per TMEM lane quarter owns all channels of its pixels
inline bool tile_pool_ok(int gemm, int Cout) { return Cout <= 64 && (Cout % 16) == 0 && umma_bn(gemm, Cout) == umma_cout_pad(gemm, Cout); }

inline int umma_tile_plan(TilePlan& plan, int dtype, int gemm, int Cp, int B, int H, int W, int Cout,
                          int Op, int kH, int kW, int relu) {
  if (!(gemm == CB_GEMM_TC || gemm == CB_GEMM_TC_3X || gemm == CB_GEMM_TC_BF16X3)) { plan.ok = false; return 0; }
  const int bn = umma_bn(gemm, Cout), CoutPad = umma_cout_pad(gemm, Cout);
  plan = tile_plan(umma_operand_es(dtype, gemm), umma_is_split(dtype, gemm), bn, Cp, B, H, W, Cout,
                   CoutPad, Op, kH, kW, relu);
  return 0;
}

inline int umma_conv_update_tiled(cudaStream_t s, int dtype, int gemm, const void* state,
                                  const void* state_lo, int Cp, const int32_t* tile_ws,
                                  const uint32_t* dil_bits, const void* packed, const float* bias,
                                  void* out, int Op, int B, int H, int W, int Cout, int kH, int kW,
                                  int relu, const PoolFuse& pf, const float* thr_b) {
  TilePlan plan;
  umma_tile_plan(plan, dtype, gemm, Cp, B, H, W, Cout, Op, kH, kW, relu);
  CB_CHECK_ARG(plan.ok, "conv_update_tiled: layer shape not supported by the tile path");
  const bool split3 = gemm == CB_GEMM_TC_3X && dtype == CB_F32;
  const bool bf16x3 = gemm == CB_GEMM_TC_BF16X3;
  CB_CHECK_ARG(!(split3 || bf16x3) || state_lo, "conv_update_tiled: the 3x modes need state_lo");
  CB_CHECK_ARG(((uintptr_t)state % 16) == 0 && ((uintptr_t)packed % 128) == 0,
               "conv_update_tiled: state must be 16-byte and packed weights 128-byte aligned");
  const int bn = umma_bn(gemm, Cout);
  CB_CHECK_ARG(!pf.out || tile_pool_ok(gemm, Cout), "conv_update_tiled: fused pooling needs Cout <= 64, a multiple of 16");
  // per-stream thresholds belong to the fused detection: only the pooling tiles (N <= 64) have the THR variant
  CB_CHECK_ARG(!thr_b || (pf.out && bn <= 64), "conv_update_tiled: per-stream thresholds need the fused pooling");
#define CB_TBN_THR(T_, TO_, S3_, N_)                                                               \
  return thr_b ? launch_conv_tile<T_, TO_, S3_, N_, true>(s, state, state_lo, tile_ws, dil_bits, packed, bias, out, plan, pf, thr_b) \
               : launch_conv_tile<T_, TO_, S3_, N_>(s, state, state_lo, tile_ws, dil_bits, packed, bias, out, plan, pf, nullptr);
#define CB_TBN(T_, TO_, S3_)                                                                       \
  switch (bn) {                                                                                    \
    case 16: CB_TBN_THR(T_, TO_, S3_, 16)                                                          \
    case 32: CB_TBN_THR(T_, TO_, S3_, 32)                                                          \
    case 64: CB_TBN_THR(T_, TO_, S3_, 64)                                                          \
    case 128: return launch_conv_tile<T_, TO_, S3_, 128>(s, state, state_lo, tile_ws, dil_bits, packed, bias, out, plan, pf, nullptr); \
    case 256: return launch_conv_tile<T_, TO_, S3_, 256>(s, state, state_lo, tile_ws, dil_bits, packed, bias, out, plan, pf, nullptr); \
    default: return fail(2, "conv_update_tiled: unsupported N tile %d", bn);                      \
  }
  if (bf16x3) { CB_TBN(__nv_bfloat16, float, true) }
  switch (dtype) {
    case CB_F32:
      if (split3) { CB_TBN(float, float, true) } else { CB_TBN(float, float, false) }
    case CB_F16: CB_TBN(__half, __half, false)
    case CB_BF16: CB_TBN(__nv_bfloat16, __nv_bfloat16, false)
    default: return fail(2, "conv_update_tiled: bad dtype %d", dtype);
  }
#undef CB_TBN
#undef CB_TBN_THR
}

}  // namespace cb
