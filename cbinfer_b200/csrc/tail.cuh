// tail.cuh -- two chained 1x1 change-based layers in ONE launch (fp32 data, 3xBF16 contraction).
//
// For the trailing pointwise layers of a network (scene net: 256 -> 64 (+ReLU) -> 8) the reference
// runs, per layer, changeDetection + nonzero + genXMatrix + GEMM + updateOutput
// (pycbinfer/conv2d.py:222-251).  On the candidate path this repo ran four launches (sparse detect,
// masked contraction, sparse detect, masked contraction); a 1x1 layer needs no neighbourhood, so the
// whole chain is a per-pixel pipeline and fits one kernel.  Per tile of 128 candidate pixels (the
// pixels the upstream layer just rewrote):
//   A  16 warps load the candidates' new input rows and layer 1's state rows (16-byte loads, all
//      rows of a warp in flight), threshold them (cb_change_detect_sparse semantics), accept the
//      changed rows into the state and write their bf16 (hi, lo) split straight into the 128B-swizzled
//      K-major UMMA tile -- layer 1's operand planes never touch HBM;
//   B  one elected lane issues layer 1's tcgen05.mma sequence (same K order and 3-term split as
//      conv_umma.cuh: the results are bit-identical to cb_conv_update_masked);
//   C  four warps drain the accumulator: bias / ReLU, store the changed rows of layer 1's output,
//      threshold them against layer 2's state, accept, and write layer 2's operand tile;
//   D  layer 2's MMAs;   E  bias, store the changed rows of layer 2's output.
// Weights of both layers stay resident in shared memory (TMA, loaded once per CTA).
#pragma once
#include "conv_umma.cuh"
#include "detect.cuh"

namespace cb {

constexpr int TAIL_THREADS = 512;
constexpr int TAIL_ROWS = 128;

struct TailArgs {
  const float* x;                // layer 1 input map (pixel-major, pitch xp), e.g. the upstream conv's output
  float* st1;                    // layer 1 previous-input state (pixel-major, pitch xp)
  float* out1;                   // layer 1 output map (pitch p1)
  float* st2;                    // layer 2 previous-input state (pitch p1)
  float* out2;                   // layer 2 output map (pitch p2)
  const int32_t* cand;           // candidate pixels (b*H*W + y*W + x), any order
  const int32_t* ncand;
  const float* bias1;
  const float* bias2;
  int32_t* count1;               // out: pixels layer 1 / layer 2 updated
  int32_t* count2;
  unsigned* sync;                // 3 words, zeroed once: finished CTAs, count accumulators
  int xp, p1, p2;                // channel pitches (elements)
  int C0, C1, C2;                // channels: in, mid, out
  int relu1, relu2, update;      // update: CB_UPDATE_CHANGED (feedback) or CB_UPDATE_ALL
  float thr1, thr2;
  // TRACK: count1 / count2 split by stream b = pixel / hw into sc1 / sc2 (int32 [B] each), through the
  // accumulators acc1 / acc2 (int32 [B] each, zero at rest), which the last CTA copies and zeroes
  int32_t *sc1, *sc2, *acc1, *acc2;
  int hw, B;
};

struct TailCtrl {
  uint64_t w_full, mma1, mma2;
  uint32_t tmem_base, pad;
  int cnt[2];
  int flag1[TAIL_ROWS];
};

// byte offset of element (row r, k) inside one K block [128 rows x 64 bf16] of the 128B-swizzled
// K-major UMMA layout (8-row groups of 1024 bytes, 16-byte chunks XOR-ed with the row)
__device__ __forceinline__ uint32_t tail_sw128(int r, int k) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((((k & 63) >> 3) ^ (r & 7)) << 4) + (k & 7) * 2);
}

template <int N1, bool TRACK, bool THR>
__global__ void __launch_bounds__(TAIL_THREADS)
tail_kernel(const __grid_constant__ CUtensorMap w1map, const __grid_constant__ CUtensorMap w2map,
            const TailArgs a, const float* __restrict__ thr1_b, const float* __restrict__ thr2_b) {
  // THR: per-stream thresholds of the two layers (fp32 [B] each, b = pixel / hw), each may be null = thr1 / thr2
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int A_KB = TAIL_ROWS * UM_ROW_BYTES;             // one K block of an A plane: 16 KB
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int n = __shfl_sync(0xffffffffu, *a.ncand, 0);
  // Rows per tile: 128 (the MMA's M) when the candidates fill the grid; with fewer, the candidates are spread
  // over ALL CTAs in tiles of ceil(n / CTAs) rows (a multiple of 8 = one warp's rows), rows beyond that stay
  // empty.  A CTA's time is its serial load -> MMA -> epilogue -> MMA -> store chain, whose load and store
  // phases shrink with the rows, while the MMAs are negligible: 14 275 candidates on 148 CTAs = 138 tiles of
  // 104 rows instead of 112 of 128 on 112 CTAs.  Per-row results do not depend on the tile's other rows.
  int rpt = TAIL_ROWS;
  if (n < (int)gridDim.x * TAIL_ROWS) {
    rpt = (((n + (int)gridDim.x - 1) / (int)gridDim.x) + 7) & ~7;
    rpt = rpt < 8 ? 8 : rpt > TAIL_ROWS ? TAIL_ROWS : rpt;
  }
  const int ntiles = (n + rpt - 1) / rpt;
  const int nkb1 = a.C0 / 64;                                // K blocks of layer 1
  // shared memory: A planes (hi: nkb1 blocks, lo: nkb1 blocks; layer 2's operand tile reuses the
  // first two blocks), W1 (hi, lo: nkb1 blocks of [N1 x 64] each), W2 (hi, lo: [16 x 64]), ctrl
  uint8_t* a_hi = smem;
  uint8_t* a_lo = smem + nkb1 * A_KB;
  uint8_t* w1s = smem + 2 * nkb1 * A_KB;
  constexpr int W1_KB = N1 * UM_ROW_BYTES;                   // one K block of one W1 plane
  uint8_t* w2s = w1s + 2 * nkb1 * W1_KB;
  constexpr int W2_B = 16 * UM_ROW_BYTES;
  TailCtrl* ctrl = reinterpret_cast<TailCtrl*>(w2s + 2 * W2_B);
  auto retire = [&](int c1, int c2) {                        // every CTA passes here exactly once
    if (tid == 0) {
      if constexpr (TRACK) ctrl->pad = 0u;                   // (all threads: "this CTA publishes")
      if (c1) atomicAdd(a.sync + 1, (unsigned)c1);
      if (c2) atomicAdd(a.sync + 2, (unsigned)c2);
      __threadfence();
      if (atomicAdd(a.sync, 1u) == gridDim.x - 1u) {
        __threadfence();
        *a.count1 = (int32_t)atomicExch(a.sync + 1, 0u);
        *a.count2 = (int32_t)atomicExch(a.sync + 2, 0u);
        a.sync[0] = 0u;
        if constexpr (TRACK) ctrl->pad = 1u;
      }
    }
    if constexpr (TRACK) {
      __syncthreads();
      if (*reinterpret_cast<volatile uint32_t*>(&ctrl->pad)) {
        stream_publish(a.acc1, a.sc1, a.B);
        stream_publish(a.acc2, a.sc2, a.B);
      }
    }
  };
  if ((int)blockIdx.x >= ntiles) {                           // CTA-uniform, before any barrier / alloc
    retire(0, 0);
    return;
  }
  if (smem_u32(smem) & 1023u) __trap();
  if (tid == 0) {
    mbar_init(&ctrl->w_full, 1);
    mbar_init(&ctrl->mma1, 1);
    mbar_init(&ctrl->mma2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&ctrl->tmem_base)), "r"(128u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = ctrl->tmem_base;
  const bool leader = elect_one();                           // (per warp; used by warp 4 only)
  if (warp == 4 && leader) {                                 // resident weights: one TMA burst
    const int CoutPad1 = N1;
    mbar_arrive_expect_tx(&ctrl->w_full, (uint32_t)(2 * nkb1 * W1_KB + 2 * W2_B));
    for (int kb = 0; kb < nkb1; ++kb) {
      tma_load_2d(smem_u32(w1s + kb * W1_KB), &w1map, kb * 64, 0, &ctrl->w_full);
      tma_load_2d(smem_u32(w1s + (nkb1 + kb) * W1_KB), &w1map, kb * 64, CoutPad1, &ctrl->w_full);
    }
    tma_load_2d(smem_u32(w2s), &w2map, 0, 0, &ctrl->w_full);
    tma_load_2d(smem_u32(w2s + W2_B), &w2map, 0, 16, &ctrl->w_full);
  }
  const uint32_t d_hi32 = (uint32_t)(umma_desc(0) >> 32);
  const uint32_t idesc1 = umma_idesc(1, N1), idesc2 = umma_idesc(1, 16);
  const int cpr = a.C0 / 4;                                  // 16-byte chunks per input row
  int tot1 = 0, tot2 = 0;                                    // (epilogue threads: rows updated)
  uint32_t par = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, par ^= 1u) {
    // ---- A: detect layer 1 on 8 candidate rows per warp, accept, split into the operand tile ----
    {
      constexpr int RPW = TAIL_ROWS / (TAIL_THREADS / 32);   // 8 rows per warp
      constexpr int RB = 4;                                  // rows in flight per batch
      // the warp's 8 candidate indices in one load (lane i holds row i's): the row loads of both
      // batches then depend on ONE index round trip instead of one per batch
      int mypix = -1;
      {
        const int rr = warp * RPW + lane;
        const int j = tile * rpt + rr;
        if (lane < RPW && rr < rpt && j < n) mypix = __ldg(a.cand + j);
      }
      // THR: row i's layer-1 threshold, fetched by lane i with its index, so the load is in flight with
      // the row loads below rather than after them
      float mythr1 = a.thr1;
      if constexpr (THR) {
        if (thr1_b && mypix >= 0) mythr1 = __ldg(thr1_b + mypix / a.hw);
      }
#pragma unroll 1
      for (int r0 = 0; r0 < RPW; r0 += RB) {
        uint4 xv[RB][2], sv[RB][2];
        int pix[RB];
#pragma unroll
        for (int i = 0; i < RB; ++i) {
          pix[i] = __shfl_sync(0xffffffffu, mypix, r0 + i);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int c = lane + 32 * h;
            if (pix[i] >= 0 && c < cpr) {
              xv[i][h] = ld16(a.x + (long long)pix[i] * a.xp + c * 4);
              sv[i][h] = ld16(a.st1 + (long long)pix[i] * a.xp + c * 4);
            } else {
              xv[i][h] = make_uint4(0, 0, 0, 0);
              sv[i][h] = xv[i][h];
            }
          }
        }
#pragma unroll
        for (int i = 0; i < RB; ++i) {
          const int r = warp * RPW + r0 + i;
          bool f = false;
          const float t1 = THR ? __shfl_sync(0xffffffffu, mythr1, r0 + i) : a.thr1;
#pragma unroll
          for (int h = 0; h < 2; ++h) f |= Chunk<float>::changed(sv[i][h], xv[i][h], THR ? t1 : a.thr1);
          const bool chg = __ballot_sync(0xffffffffu, f) != 0u && pix[i] >= 0;
          if (lane == 0) ctrl->flag1[r] = chg ? pix[i] : -1;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int c = lane + 32 * h;
            if (pix[i] < 0 || c >= cpr) continue;
            if ((chg && a.update == CB_UPDATE_CHANGED) || a.update == CB_UPDATE_ALL)
              st16(a.st1 + (long long)pix[i] * a.xp + c * 4, xv[i][h]);
            if (chg) {
              __nv_bfloat16 hb[4], lb[4];
              bf16_split(__uint_as_float(xv[i][h].x), hb[0], lb[0]);
              bf16_split(__uint_as_float(xv[i][h].y), hb[1], lb[1]);
              bf16_split(__uint_as_float(xv[i][h].z), hb[2], lb[2]);
              bf16_split(__uint_as_float(xv[i][h].w), hb[3], lb[3]);
              const int k = c * 4;
              const uint32_t off = (uint32_t)((k >> 6) * A_KB) + tail_sw128(r, k);
              *reinterpret_cast<uint2*>(a_hi + off) = *reinterpret_cast<uint2*>(hb);
              *reinterpret_cast<uint2*>(a_lo + off) = *reinterpret_cast<uint2*>(lb);
            }
          }
        }
      }
    }
    fence_proxy_async_smem();                                // st.shared -> async proxy (UMMA)
    __syncthreads();
    // ---- B: layer 1 contraction (K order and 3-term split of conv_umma.cuh) -----------------
    if (warp == 4) {
      if (tile == (int)blockIdx.x) mbar_wait(&ctrl->w_full, 0u);
      tc_fence_after();
      if (leader) {
        const uint32_t ah = ((smem_u32(a_hi) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t al = ((smem_u32(a_lo) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t wh = ((smem_u32(w1s) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t wl = wh + (uint32_t)((nkb1 * W1_KB) >> 4);
        for (int kb = 0; kb < nkb1; ++kb) {
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t ao = (uint32_t)((kb * A_KB) >> 4) + 2u * ks, wo = (uint32_t)((kb * W1_KB) >> 4) + 2u * ks;
            const uint64_t dAh = ((uint64_t)d_hi32 << 32) | (ah + ao), dAl = ((uint64_t)d_hi32 << 32) | (al + ao);
            const uint64_t dWh = ((uint64_t)d_hi32 << 32) | (wh + wo), dWl = ((uint64_t)d_hi32 << 32) | (wl + wo);
            umma<1>(tmem, dAl, dWh, idesc1, (kb | ks) ? 1u : 0u);
            umma<1>(tmem, dAh, dWl, idesc1, 1u);
            umma<1>(tmem, dAh, dWh, idesc1, 1u);
          }
        }
        umma_commit(&ctrl->mma1);
      }
      __syncwarp();
    }
    // ---- C: layer 1 epilogue + layer 2 detection + layer 2 operand tile ------------------------
    int pix1 = -1;
    bool f2 = false;
    if (warp < 4) {
      const int row = warp * 32 + lane;
      pix1 = ctrl->flag1[row];
      float* o1 = a.out1 + (long long)(pix1 < 0 ? 0 : pix1) * a.p1;
      float* s2 = a.st2 + (long long)(pix1 < 0 ? 0 : pix1) * a.p1;
      // layer 2's state row (<= 64 channels) is fetched while layer 1's MMAs run: one memory round trip
      // for the whole row instead of one per 16-column slice of the accumulator
      uint4 s2v[N1 / 4];
#pragma unroll
      for (int i = 0; i < N1 / 4; ++i)
        s2v[i] = (pix1 >= 0 && 4 * i < a.C1) ? ld16(s2 + 4 * i) : make_uint4(0, 0, 0, 0);
      // (THR: layer 2's threshold of the row, also fetched while the MMAs run)
      const float t2 = THR && thr2_b && pix1 >= 0 ? __ldg(thr2_b + pix1 / a.hw) : a.thr2;
      mbar_wait(&ctrl->mma1, par);
      tc_fence_after();
      const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll
      for (int c0 = 0; c0 < N1; c0 += 16) {
        uint32_t acc[16];
        tmem_ld16(trow + (uint32_t)c0, acc);
        tmem_ld_wait();
        if (pix1 >= 0 && c0 < a.C1) {
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float t = __uint_as_float(acc[i]) + __ldg(a.bias1 + c0 + i);
            if (a.relu1 && t <= 0.f) t = 0.f;
            f[i] = t;
          }
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const uint4 v = make_uint4(__float_as_uint(f[i]), __float_as_uint(f[i + 1]), __float_as_uint(f[i + 2]),
                                       __float_as_uint(f[i + 3]));
            st16(o1 + c0 + i, v);
            const uint4 sv = s2v[(c0 + i) >> 2];
            f2 |= Chunk<float>::changed(sv, v, THR ? t2 : a.thr2);   // (a.thr2 read here, as without THR)
            if (a.update == CB_UPDATE_ALL) st16(s2 + c0 + i, v);
          }
          // layer 2's operand tile (K = C1 <= 64: one K block), rows of unchanged pixels are ignored later
          __nv_bfloat16 hb[16], lb[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) bf16_split(f[i], hb[i], lb[i]);
#pragma unroll
          for (int i = 0; i < 16; i += 8) {
            const uint32_t off = tail_sw128(row, c0 + i);
            *reinterpret_cast<uint4*>(a_hi + off) = *reinterpret_cast<uint4*>(hb + i);
            *reinterpret_cast<uint4*>(a_hi + A_KB + off) = *reinterpret_cast<uint4*>(lb + i);
          }
        }
      }
      if (pix1 >= 0 && f2 && a.update == CB_UPDATE_CHANGED)   // feedback: accept the new row into layer 2's state
        for (int c = 0; c < a.C1; c += 4) st16(s2 + c, ld16(o1 + c));
      tot1 += pix1 >= 0;
      tot2 += (pix1 >= 0 && f2);
      if constexpr (TRACK) {
        stream_add_warp(pix1 >= 0 ? pix1 / a.hw : -1, 1u, a.acc1);
        stream_add_warp(pix1 >= 0 && f2 ? pix1 / a.hw : -1, 1u, a.acc2);
        __threadfence();                                     // before this CTA's retire
      }
      tc_fence_before();
      fence_proxy_async_smem();
    }
    __syncthreads();
    // ---- D: layer 2 contraction ------------------------------------------------------------------
    if (warp == 4) {
      tc_fence_after();
      if (leader) {
        const uint32_t ah = ((smem_u32(a_hi) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t al = ah + (uint32_t)(A_KB >> 4);
        const uint32_t wh = ((smem_u32(w2s) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t wl = wh + (uint32_t)(W2_B >> 4);
        const int nks = a.C1 / 16;
        for (int ks = 0; ks < nks; ++ks) {
          const uint64_t dAh = ((uint64_t)d_hi32 << 32) | (ah + 2u * ks), dAl = ((uint64_t)d_hi32 << 32) | (al + 2u * ks);
          const uint64_t dWh = ((uint64_t)d_hi32 << 32) | (wh + 2u * ks), dWl = ((uint64_t)d_hi32 << 32) | (wl + 2u * ks);
          umma<1>(tmem + 64u, dAl, dWh, idesc2, ks ? 1u : 0u);
          umma<1>(tmem + 64u, dAh, dWl, idesc2, 1u);
          umma<1>(tmem + 64u, dAh, dWh, idesc2, 1u);
        }
        umma_commit(&ctrl->mma2);
      }
      __syncwarp();
    }
    // ---- E: layer 2 epilogue -------------------------------------------------------------------
    if (warp < 4) {
      mbar_wait(&ctrl->mma2, par);
      tc_fence_after();
      uint32_t acc[16];
      tmem_ld16(tmem + 64u + ((uint32_t)(warp * 32) << 16), acc);
      tmem_ld_wait();
      if (pix1 >= 0 && f2) {
        float* o2 = a.out2 + (long long)pix1 * a.p2;
#pragma unroll
        for (int c = 0; c < 16; ++c) {                       // (constant indices: acc stays in registers)
          if (c < a.C2) {
            float t = __uint_as_float(acc[c]) + __ldg(a.bias2 + c);
            if (a.relu2 && t <= 0.f) t = 0.f;
            o2[c] = t;
          }
        }
      }
      tc_fence_before();
    }
    __syncthreads();                                         // operand tiles and accumulators are free again
  }
  // per-CTA update counts -> global accumulators
  int* s_cnt = ctrl->cnt;
  if (tid == 0) { s_cnt[0] = 0; s_cnt[1] = 0; }
  __syncthreads();
  if (warp < 4) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      tot1 += __shfl_xor_sync(0xffffffffu, tot1, o);
      tot2 += __shfl_xor_sync(0xffffffffu, tot2, o);
    }
    if (lane == 0) { atomicAdd(&s_cnt[0], tot1); atomicAdd(&s_cnt[1], tot2); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(128u) : "memory");
  }
  retire(s_cnt[0], s_cnt[1]);
}

// ---- host ------------------------------------------------------------------------------------------
inline bool tail_supported(int C0, int C1, int C2) {
  return C0 % 64 == 0 && C0 >= 64 && C0 <= 256 && (C1 == 16 || C1 == 32 || C1 == 64) && C2 >= 1 && C2 <= 16;
}

inline int tail_update(cudaStream_t s, const TailArgs& a, const void* packed1, const void* packed2,
                       const float* thr1_b, const float* thr2_b) {
  CB_CHECK_ARG(tail_supported(a.C0, a.C1, a.C2), "tail_update: unsupported channel counts %d -> %d -> %d", a.C0,
               a.C1, a.C2);
  CB_CHECK_ARG(a.xp == a.C0 && a.p1 == a.C1 && a.p2 >= a.C2 && (a.p2 % 4) == 0,
               "tail_update: channel pitches must equal the channel counts (pixel-major fp32 maps)");
  auto enc = tensor_map_encoder();
  if (!enc) return fail(3, "tail_update: cuTensorMapEncodeTiled unavailable");
  alignas(64) CUtensorMap m1, m2;
  const int N1 = a.C1;
  {
    const cuuint64_t gdim[2] = {(cuuint64_t)a.C0, (cuuint64_t)(2 * N1)};
    const cuuint64_t gstr[1] = {(cuuint64_t)a.C0 * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)N1};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&m1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(packed1), gdim, gstr, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail(3, "tail_update: weight tensor map 1 failed");
  }
  {
    const cuuint64_t gdim[2] = {64, 32};                       // layer 2: KpPad = 64 (K = C1 <= 64), 2 x CoutPad (16)
    const cuuint64_t gstr[1] = {64 * 2};
    const cuuint32_t box[2] = {64, 16};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&m2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(packed2), gdim, gstr, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail(3, "tail_update: weight tensor map 2 failed");
  }
  const int nkb1 = a.C0 / 64;
  const size_t smem = (size_t)2 * nkb1 * TAIL_ROWS * UM_ROW_BYTES + (size_t)2 * nkb1 * N1 * UM_ROW_BYTES +
                      2 * 16 * UM_ROW_BYTES + sizeof(TailCtrl) + 64;
  const unsigned grid = (unsigned)sm_count();
#define CB_TAIL(N_, TR_, TH_)                                                                          \
  {                                                                                                  \
    static thread_local int adev = -1;                                                               \
    int dev = 0;                                                                                     \
    cudaGetDevice(&dev);                                                                             \
    if (adev != dev) {                                                                               \
      if (cudaFuncSetAttribute(tail_kernel<N_, TR_, TH_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024) != cudaSuccess) \
        return fail(3, "tail_update: cannot reserve shared memory");                                \
      adev = dev;                                                                                    \
    }                                                                                                \
    cb::launch(tail_kernel<N_, TR_, TH_>, dim3(grid), dim3(TAIL_THREADS), smem, s, m1, m2, a, thr1_b, thr2_b);       \
  }
#define CB_TAIL_THR(N_, TR_) { if (thr) CB_TAIL(N_, TR_, true) else CB_TAIL(N_, TR_, false) }
  const bool track = a.sc1 != nullptr, thr = thr1_b || thr2_b;
  switch (N1) {
    case 16: if (track) CB_TAIL_THR(16, true) else CB_TAIL_THR(16, false) break;
    case 32: if (track) CB_TAIL_THR(32, true) else CB_TAIL_THR(32, false) break;
    case 64: if (track) CB_TAIL_THR(64, true) else CB_TAIL_THR(64, false) break;
    default: return fail(2, "tail_update: bad mid channel count %d", N1);
  }
#undef CB_TAIL_THR
#undef CB_TAIL
  CB_CHECK_LAUNCH("tail_update");
  return 0;
}

}  // namespace cb
