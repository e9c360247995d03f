// conv_umma.cuh -- fused gather + tcgen05 contraction + bias/ReLU + scatter (the hot kernel).
//
// Replaces genXMatrix_kernel (reference cbconv2d_cg_backend.cu:138-161), the cuBLAS GEMM behind
// matrixMult_python (conv2d_cg.py:342-349), the transpose copy (conv2d.py:247) and
// updateOutput_kernel (cbconv2d_cg_backend.cu:175-189).  X, Y and Y^T never exist in memory.
//
// Implicit GEMM, D[128 x BN] (+)= A[128 x K] * B[BN x K]^T per tile:
//   M : 128 changed pixels (rows of the index list; the count is read on the device)
//   N : BN output channels
//   K : kH*kW*Cp ordered (ky,kx,ci): every filter tap is a contiguous channel run of the
//       pixel-major state, so one 16-byte chunk never straddles a tap.
// Warp roles (320 threads):
//   warps 0-7  gather producers: im2col rows of ONLY the changed receptive fields, 16-byte
//              cp.async copies global -> 128B-swizzled K-major smem tile (the UMMA canonical
//              layout), zero-filled outside the image.  In 3xTF32 mode the tf32 "hi" operand is
//              the raw fp32 state (the tensor core ignores the low 13 mantissa bits) and the
//              "lo" operand is the remainder plane cb_change_detect maintains.
//              The same warps run the epilogue: tcgen05.ld accumulators from TMEM, + bias,
//              ReLU, convert, scatter one contiguous channel run per pixel.
//   warp 8     TMA producer for the (regular) weight tiles: cp.async.bulk.tensor.2d, SWIZZLE_128B.
//   warp 9     MMA issuer: one elected thread issues tcgen05.mma (kind::tf32 / kind::f16) with
//              the accumulator in TMEM; tcgen05.commit releases smem stages / signals the epilogue.
// Stages are handed over with mbarriers (full/empty ring + tmem full/empty).
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include "cb_common.cuh"

namespace cb {

constexpr int UM_BM = 128;                     // rows per tile (UMMA M, cta_group::1)
constexpr int UM_PRODUCERS = 256;              // gather threads (warps 0-7)
// epilogue threads: warps 10.. ; one warp per TMEM lane quarter for narrow N tiles (keeps the CTA
// small enough for 2 CTAs/SM), two per quarter (splitting the columns) for N tiles >= 128
__host__ __device__ constexpr int um_epi(int bn) { return bn >= 128 ? 256 : 128; }
__host__ __device__ constexpr int um_threads(int bn) { return UM_PRODUCERS + 64 + um_epi(bn); }  // + TMA warp + MMA warp
constexpr int UM_ROW_BYTES = 128;              // K bytes per stage row = one swizzle-128B span

// ---- PTX wrappers ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
// Bounded wait: a protocol bug traps (sticky error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t spins = 0;; ++spins) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
    if ((spins & 1023u) == 1023u) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ll) __trap();      // ~2 s at 2 GHz
    }
  }
}
// ---- thread-block cluster helpers (split-K reduction over distributed shared memory) ----------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t spins = 0;; ++spins) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
    if ((spins & 1023u) == 1023u) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ll) __trap();
    }
  }
}
__device__ __forceinline__ float4 ld_cluster_f4(uint32_t cluster_addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(cluster_addr));
  return v;
}

// 16-byte async copy global -> shared (LDGSTS); src_bytes = 0 zero-fills (out-of-image taps)
__device__ __forceinline__ void cp_async8(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(src_bytes)
               : "memory");
}
// (.cg: L2 only; caching the gather in L1 with .ca measured no gain, profiles/r01_experiments.md)
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes)
               : "memory");
}
// arrive on `bar` once all cp.async issued so far by this thread have landed (counts as one of
// the barrier's expected arrivals)
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; KIND 0: tf32, 1: f16/bf16
template <int KIND>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                     uint32_t idesc, uint32_t accumulate) {
  if (KIND == 0)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// one lane of a converged warp (the same one every time)
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(p));
  return p != 0;
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 UMMA):
// start>>4 [0,14) | LBO>>4 = 1 [16,30) | SBO>>4 = 64 (8 rows x 128 B) [32,46) | version 1 [46,48)
// | layout SWIZZLE_128B = 2 [61,64).
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) |
         (2ull << 61);
}
// instruction descriptor: D=f32, A/B format fmt (0 f16, 1 bf16, 2 tf32), K-major both, N, M=128
__host__ __device__ inline uint32_t umma_idesc(int fmt, int N) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(UM_BM >> 4) << 24);
}

// ---- configuration -----------------------------------------------------------------------------
constexpr int UM_CTRL_BYTES = 2304;            // barriers + TMEM base + row table
// DEEP: one CTA per SM with as many stages as fit (used when few tiles exist: latency, not
// occupancy, is then the limiter).
template <typename T, bool SPLIT3, int BN, bool DEEP = false>
struct UmmaCfg {
  static constexpr int ES = sizeof(T);
  static constexpr int VEC = 16 / ES;                        // elements per 16-byte chunk
  static constexpr int BK = UM_ROW_BYTES / ES;               // K elements per stage
  static constexpr int UK = 32 / ES;                         // K elements per tcgen05.mma
  static constexpr int NSPLIT = SPLIT3 ? 2 : 1;
  static constexpr int A_BYTES = UM_BM * UM_ROW_BYTES;       // 16 KB
  static constexpr int B_BYTES = BN * UM_ROW_BYTES;
  static constexpr int STAGE_BYTES = NSPLIT * (A_BYTES + B_BYTES);
  // two CTAs per SM (<= ~100 KB each) unless a stage is so large that only one CTA fits
  static constexpr int CTAS_PER_SM = (DEEP || STAGE_BYTES > 48 * 1024) ? 1 : 2;
  static constexpr int RED_BYTES = DEEP ? UM_BM * BN * 4 : 0;   // split-K partial tile (fp32)
  static constexpr int BUDGET = DEEP ? 200 * 1024 - RED_BYTES : (CTAS_PER_SM == 1 ? 200 * 1024 : 98 * 1024);
  static constexpr int STAGES = (BUDGET / STAGE_BYTES) < 2 ? 2
                                : (BUDGET / STAGE_BYTES) > 8 ? 8 : (BUDGET / STAGE_BYTES);
  // two accumulators: the epilogue warps drain one while the MMA warp fills the other
  static constexpr int TMEM_COLS = 2 * BN <= 32 ? 32 : 2 * BN <= 64 ? 64 : 2 * BN <= 128 ? 128
                                   : 2 * BN <= 256 ? 256 : 512;
  static constexpr int TABLE_MAX = 1024;        // chunk-offset table entries (8 KB)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + UM_CTRL_BYTES +
                                    TABLE_MAX * 8 + RED_BYTES;
};

struct UmmaCtrl {                              // lives after the stage buffers
  uint64_t full[8], empty[8];
  uint64_t tmem_full[2], tmem_empty[2];        // per accumulator: MMAs done / drained
  uint64_t tab_full[2];                        // per row table: written by the gather warps
  uint64_t red_full, red_free;                 // split-K: partials delivered / partial buffer free
  uint32_t tmem_base, pad;
  int pix[2][UM_BM];                           // row tables (pixel index or -1), double-buffered
  int yx[2][UM_BM];
};
static_assert(sizeof(UmmaCtrl) <= UM_CTRL_BYTES, "ctrl block too large");

// Incremental (ky,kx,ci) decode of this thread's K position: advances by one stage (BK elements)
// per call, in stage order, without integer divisions in the hot loop.
struct KCursor {
  int ci, kx, ky, k;
  __device__ __forceinline__ void init(int k0, int Cp, int kW) {
    k = k0;
    const int tap = k0 / Cp;
    ci = k0 - tap * Cp;
    ky = tap / kW;
    kx = tap - ky * kW;
  }
  __device__ __forceinline__ void advance(int bk, int Cp, int kW) {
    k += bk;
    ci += bk;
    while (ci >= Cp) {
      ci -= Cp;
      if (++kx == kW) { kx = 0; ++ky; }
    }
  }
};

// Work segments (tile, K blocks [kb0, kb1)) of one CTA, walked identically by every warp role.
//   static  : tiles tile0, tile0 + step, ... each over the CTA's fixed K range
//   stream-K: the (tile, kb) space is cut into gridDim.x equal contiguous ranges, so every CTA gets
//             the same amount of work whatever the change count; tiles cut by a range boundary
//             are finished by the CTA holding their first K blocks (it reaches them last), the
//             others park their partial accumulators in a global workspace.
struct TileSeg {
  int tile, kb0, kb1;
  int step, total, nkb;
  long long u, u1;
  bool sk;
  __device__ __forceinline__ void init_static(int tile0, int step_, int total_, int k0, int k1) {
    sk = false; tile = tile0 - step_; step = step_; total = total_; kb0 = k0; kb1 = k1;
    nkb = 0; u = u1 = 0;
  }
  __device__ __forceinline__ void init_sk(long long u0, long long u1_, int num_kb) {
    sk = true; u = u0; u1 = u1_; nkb = num_kb; tile = 0; kb0 = kb1 = 0; step = total = 0;
  }
  __device__ __forceinline__ bool next() {
    if (!sk) { tile += step; return tile < total; }
    if (u >= u1) return false;
    tile = (int)(u / nkb);
    kb0 = (int)(u - (long long)tile * nkb);
    const long long left = u1 - u;
    kb1 = (left < (long long)(nkb - kb0)) ? kb0 + (int)left : nkb;
    u += kb1 - kb0;
    return true;
  }
};
constexpr int UM_SK_FLAG_BYTES = 4096;       // stream-K workspace: per-CTA flags, then partial tiles

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Row mask: `idx` may be a SUPERSET of the pixels to update (e.g. the previous layer's change list
// handed to a 1x1 layer as detection candidates); a row is processed only if its pixel's bit is set
// in `bits` (the raw change bitmap the detection just produced).  That removes the ordered
// compaction between detection and contraction for layers that need no dilation.  The number of
// processed pixels is written to *count_out; with `clear` the last CTA to finish zeroes the bitmap
// (ready for the next frame's atomicOr-ing detection).  `sync` = {done counter, count accumulator},
// zeroed once by the caller, left clean by the kernel.  With `stream_counts` (the kernel's TRACK
// variant) the processed pixels are also counted per stream b = pix / (H*W): added to stream_acc
// (int32 [B], zero at rest), copied to stream_counts and zeroed by the same last CTA.
struct RowMask {
  const uint32_t* bits;
  uint32_t* clear;
  int32_t* count_out;
  unsigned* sync;
  int nwords;
  int32_t* stream_counts;
  int32_t* stream_acc;
  int B;
};
// (s_flag: one word of dynamic shared memory -- the kernel must not own static shared memory)
template <bool TRACK>
__device__ __forceinline__ void rowmask_finish(const RowMask& mk, volatile unsigned* s_flag) {
  // every CTA of the selected variant passes here exactly once, after its last read of the bitmap
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned prev = atomicAdd(mk.sync, 1u);
    *s_flag = prev == gridDim.x - 1u;
  }
  __syncthreads();
  if (!*s_flag) return;
  __threadfence();
  if (threadIdx.x == 0) {
    if (mk.count_out) *mk.count_out = (int32_t)atomicExch(mk.sync + 1, 0u);
    mk.sync[0] = 0u;
  }
  if constexpr (TRACK) stream_publish(mk.stream_acc, mk.stream_counts, mk.B);
  if (mk.clear)
    for (int i = threadIdx.x; i < mk.nwords; i += blockDim.x) mk.clear[i] = 0u;
}

// packed weights: [NSPLIT][CoutPad][KpPad] elements of T (K-major); tensor map dims {KpPad, NSPLIT*CoutPad}
// T = operand element type in the state planes / shared memory, TO = element type of `out`
// (TO != T only for 3xBF16: bf16 hi/lo operand planes of an fp32 layer).
template <typename T, typename TO, bool SPLIT3, int BN, bool DEEP, bool TRACK>
__global__ void __launch_bounds__(um_threads(BN))
conv_umma_kernel(const __grid_constant__ CUtensorMap wmap, const T* __restrict__ state,
                 const T* __restrict__ state_lo, int Cp, const int32_t* __restrict__ idx, const int32_t* __restrict__ count,
                 const float* __restrict__ bias, TO* __restrict__ out, int Op, int H, int W,
                 int Cout, int CoutPad, int kH, int kW, int Kp, int relu, int sel_lo, int sel_hi,
                 uint32_t* __restrict__ sk_ws, const RowMask mk) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  using C = UmmaCfg<T, SPLIT3, BN, DEEP>;
  constexpr int UM_EPI = um_epi(BN), UM_THREADS = um_threads(BN);
  constexpr int RPT = UM_BM * 8 / UM_PRODUCERS;            // 16-byte chunks per thread per stage
  constexpr int RSTEP = UM_PRODUCERS / 8;                  // row stride between a thread's chunks
  const int n = __shfl_sync(0xffffffffu, *count, 0);        // (the shuffle makes the value uniform for the compiler)
  const int mtiles = (n + UM_BM - 1) / UM_BM;
  const int ntiles = CoutPad / BN;
  const int total_tiles = mtiles * ntiles;
  // sel window: two tilings of the same layer may be launched back to back; the change count
  // (known only on the device) decides which one does the work
  if (mtiles < sel_lo || mtiles >= sel_hi) return;
  // split-K: groups of KS consecutive CTAs of a cluster work on the same tile, each on 1/KS of
  // the K range; the group's first CTA sums the partial accumulators through distributed shared
  // memory.  KS is chosen HERE from the change count: the widest split (a power of two dividing
  // the launched cluster size) for which all tiles still run in one wave, else no split.
  const uint32_t KSmax = DEEP ? cluster_nctarank() : 1u, crank = DEEP ? cluster_ctarank() : 0u;
  uint32_t KS = KSmax;
  while (KS > 1 && (long long)total_tiles * KS > (long long)gridDim.x) KS >>= 1;
  const uint32_t krank = crank & (KS - 1), leader = crank - krank;
  const int tile0 = (int)(blockIdx.x / KS), tile_step = (int)(gridDim.x / KS);
  const bool sk = !DEEP && sk_ws != nullptr;              // stream-K (never together with clusters)
  if (!sk && tile0 >= total_tiles) {                      // group-uniform: before any barrier / alloc
    if (KSmax > 1) { cluster_sync_all(); cluster_sync_all(); }   // busy peers still sync twice
    if (mk.bits) rowmask_finish<TRACK>(mk, reinterpret_cast<volatile unsigned*>(smem_raw));
    return;
  }

  uint8_t* smem = smem_raw;
  if (smem_u32(smem) & 1023u) __trap();                   // SWIZZLE_128B tiles need 1024-byte alignment
  UmmaCtrl* ctrl = reinterpret_cast<UmmaCtrl*>(smem + C::STAGES * C::STAGE_BYTES);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);    // provably warp-uniform role index
  const int num_kb = (Kp + C::BK - 1) / C::BK;
  TileSeg seg0;
  const long long sk_units = (long long)total_tiles * num_kb;
  // stream-K runs on the first sk_grid CTAs only: with fewer (tile, K block) units than CTAs the
  // extra ones would own an empty range, never raise their flag, and the tile owner would wait
  // for them forever
  const long long sk_grid = sk ? (sk_units < (long long)gridDim.x ? (sk_units > 0 ? sk_units : 1)
                                                                  : (long long)gridDim.x) : 1;
  if (sk && (long long)blockIdx.x >= sk_grid) {            // CTA-uniform: before any barrier / alloc
    if (mk.bits) rowmask_finish<TRACK>(mk, reinterpret_cast<volatile unsigned*>(smem_raw));
    return;
  }
  if (sk)
    seg0.init_sk(sk_units * blockIdx.x / sk_grid, sk_units * (blockIdx.x + 1) / sk_grid, num_kb);
  else
    seg0.init_static(tile0, tile_step, total_tiles, (int)((long long)num_kb * krank / KS),
                     (int)((long long)num_kb * (krank + 1) / KS));
  float4* const sk_part = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(sk_ws) + UM_SK_FLAG_BYTES);
  constexpr int SK_SLOT = UM_BM * BN / 4;                   // float4 per partial tile
  constexpr int TMA_WARP = UM_PRODUCERS / 32, MMA_WARP = TMA_WARP + 1, EPI_WARP0 = MMA_WARP + 1;
  const int ph = (kH - 1) / 2, pw = (kW - 1) / 2;
  // Per 16-byte K chunk q (k = q*VEC): element offset of its filter tap relative to the pixel and
  // the tap's (dy,dx); built once per CTA so the gather loop has no divisions.
  int2* ktab = reinterpret_cast<int2*>(reinterpret_cast<uint8_t*>(ctrl) + UM_CTRL_BYTES);
  // 8-byte taps (Cp == 4 sixteen-bit channels, e.g. an RGB input layer's bf16 planes): a 16-byte
  // chunk holds two taps, gathered as two 8-byte copies with their own bounds test
  const bool half_taps = sizeof(T) == 2 && Cp == 4;
  const int upc = half_taps ? 2 : 1;                        // table units per 16-byte chunk
  const bool use_table = num_kb * 8 * upc <= C::TABLE_MAX;
  const uint32_t ktab_s = smem_u32(ktab);
  if (use_table) {
    for (int q = tid; q < num_kb * 8 * upc; q += UM_THREADS) {
      const int k = q * (C::VEC / upc);
      int2 e = make_int2(0, (int)0x80008000u);             // k beyond K: dy = dx = -32768 (invalid)
      if (k < Kp) {
        const int tap = k / Cp, ci = k - tap * Cp;
        const int ky = tap / kW, kx = tap - ky * kW;
        e.x = ((ky - ph) * W + (kx - pw)) * Cp + ci;
        e.y = (int)(((unsigned)(ky - ph) << 16) | ((unsigned)(kx - pw) & 0xffffu));
      }
      ktab[q] = e;
    }
  }

  if (tid == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&ctrl->full[s], UM_PRODUCERS + 1);
      mbar_init(&ctrl->empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&ctrl->tmem_full[b], 1);
      mbar_init(&ctrl->tmem_empty[b], UM_EPI);
      mbar_init(&ctrl->tab_full[b], 1);
    }
    mbar_init(&ctrl->red_full, (KS > 1 ? KS - 1 : 1) * UM_EPI);
    mbar_init(&ctrl->red_free, UM_EPI);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MMA_WARP) {                                  // TMEM allocation (one warp)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&ctrl->tmem_base)),
                 "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == TMA_WARP && lane == 0)
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&wmap)) : "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (DEEP && KSmax > 1) cluster_sync_all();               // peers' barriers exist before remote arrives
  const uint32_t tmem_base = ctrl->tmem_base;
  const int P = H * W;

  if (warp < TMA_WARP) {
    // =============================== gather producers ========================================
    uint32_t stage = 0, phase = 0, sidx = 0;
    const int c = tid & 7;                                  // my 16-byte chunk column
    const int r0 = tid >> 3;                                // my rows: r0 + RSTEP*it
    uint32_t soff[RPT];                                     // swizzled smem offsets of my chunks
#pragma unroll
    for (int it = 0; it < RPT; ++it) {
      const int r = r0 + RSTEP * it;
      soff[it] = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
    }
    TileSeg sg = seg0;
    while (sg.next()) {
      const int tile = sg.tile, kb0 = sg.kb0, kb1 = sg.kb1;
      const int mt = tile / ntiles;
      const uint32_t buf = sidx & 1u, use = sidx >> 1;
      ++sidx;
      if (tid < UM_BM) {                                    // row table of this tile
        // the table (and accumulator) `buf` was last used two segments ago: drained yet?
        mbar_wait(&ctrl->tmem_empty[buf], (use & 1u) ^ 1u);
        const int j = mt * UM_BM + tid;
        int pix = -1, yx = 0;
        if (j < n) {
          pix = __ldg(idx + j);
          const int p = pix % P;
          const int yy = p / W;
          yx = (yy << 16) | (p - yy * W);
          if (mk.bits) {                                    // superset list: keep flagged pixels only
            const int xx = p - yy * W;
            const uint32_t wbits = mk.bits[((long long)(pix / P) * H + yy) * ((W + 31) >> 5) + (xx >> 5)];
            if (!((wbits >> (xx & 31)) & 1u)) pix = -1;
          }
        }
        ctrl->pix[buf][tid] = pix;
        ctrl->yx[buf][tid] = yx;
        if (mk.bits && kb0 == 0 && tile - mt * ntiles == 0 && krank == 0) {   // once per M tile
          const unsigned m = __ballot_sync(0xffffffffu, pix >= 0);
          if ((tid & 31) == 0 && m) atomicAdd(mk.sync + 1, (unsigned)__popc(m));
          if constexpr (TRACK) {
            stream_add_warp(pix >= 0 ? pix / P : -1, 1u, mk.stream_acc);
            __threadfence();                                // before this CTA's rowmask_finish
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(UM_PRODUCERS) : "memory");   // producers only
      if (tid == 0) mbar_arrive(&ctrl->tab_full[buf]);      // release: the epilogue may read the table
      const long long lo_delta = SPLIT3 ? (state_lo - state) : 0;
      if (half_taps) {
        // 8-byte taps: lane = (row pair, chunk, half) so that one warp instruction writes both
        // halves of 16 chunks of 2 rows -- all 32 banks of the 128B-swizzled tile (2 wavefronts
        // instead of ~6 with a fixed half per instruction) -- and reads 16 consecutive taps per row
        const int hh = tid & 1, c2 = (tid >> 1) & 7, q0 = tid >> 4;      // rows q0 + 16*it
        constexpr int HR = UM_BM / 16;
        int hpix[HR], hyx[HR];
#pragma unroll
        for (int it = 0; it < HR; ++it) {
          hpix[it] = ctrl->pix[buf][q0 + 16 * it];
          hyx[it] = ctrl->yx[buf][q0 + 16 * it];
        }
        const uint32_t hoff = (uint32_t)((q0 >> 3) * 1024 + (q0 & 7) * 128 + ((c2 ^ (q0 & 7)) << 4) + 8 * hh);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&ctrl->empty[stage], phase ^ 1u);
          const uint32_t a_hi = smem_u32(smem + stage * C::STAGE_BYTES) + hoff;
          int2 e;
          asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];"
                       : "=r"(e.x), "=r"(e.y)
                       : "r"(ktab_s + (uint32_t)(((kb * 8 + c2) * 2 + hh) * 8)));
          const int dy = e.y >> 16, dx = (int)(short)(e.y & 0xffff);
#pragma unroll
          for (int it = 0; it < HR; ++it) {
            const bool ok = hpix[it] >= 0 && (unsigned)((hyx[it] >> 16) + dy) < (unsigned)H &&
                            (unsigned)((hyx[it] & 0xffff) + dx) < (unsigned)W;
            const T* src = ok ? state + ((long long)hpix[it] * 4 + e.x) : state;
            cp_async8(a_hi + it * 2048, src, ok ? 8u : 0u);
            if (SPLIT3) cp_async8(a_hi + C::A_BYTES + it * 2048, src + lo_delta, ok ? 8u : 0u);
          }
          cp_async_arrive_noinc(&ctrl->full[stage]);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
        }
        continue;
      }
      // per-row source pointers (pixel base) and coordinates of my RPT rows
      const T* rbase[RPT];
      int ry[RPT], rx[RPT];
#pragma unroll
      for (int it = 0; it < RPT; ++it) {
        const int pix = ctrl->pix[buf][r0 + RSTEP * it], yx = ctrl->yx[buf][r0 + RSTEP * it];
        rbase[it] = state + (long long)(pix < 0 ? 0 : pix) * Cp;
        ry[it] = pix < 0 ? -0x40000000 : (yx >> 16);        // invalid rows fail every bounds test
        rx[it] = yx & 0xffff;
      }
      KCursor cur;
      cur.init(kb0 * C::BK + c * C::VEC, Cp, kW);
      // Gather = async 16-byte copies straight into the swizzled UMMA tile (zero-filled outside
      // the image / beyond K); no register staging, so up to STAGES stages of loads are in flight.
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&ctrl->empty[stage], phase ^ 1u);
        const uint32_t a_hi = smem_u32(smem + stage * C::STAGE_BYTES);
        int dy, dx;
        long long koff;
        bool kvalid;
        if (use_table) {
          int2 e;                                            // explicit ld.shared (not a generic LD)
          asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];"
                       : "=r"(e.x), "=r"(e.y)
                       : "r"(ktab_s + (uint32_t)((kb * 8 + c) * 8)));
          koff = e.x;
          dy = e.y >> 16;
          dx = (int)(short)(e.y & 0xffff);
          kvalid = true;                                     // invalid chunks fail the bounds test
        } else {
          dy = cur.ky - ph;
          dx = cur.kx - pw;
          kvalid = cur.k < Kp;
          koff = ((long long)dy * W + dx) * Cp + cur.ci;
          cur.advance(C::BK, Cp, kW);
        }
#pragma unroll
        for (int it = 0; it < RPT; ++it) {
          const bool ok = kvalid && (unsigned)(ry[it] + dy) < (unsigned)H &&
                          (unsigned)(rx[it] + dx) < (unsigned)W;
          const T* src = ok ? rbase[it] + koff : state;
          cp_async16(a_hi + soff[it], src, ok ? 16u : 0u);
          if (SPLIT3) cp_async16(a_hi + C::A_BYTES + soff[it], src + lo_delta, ok ? 16u : 0u);
        }
        cp_async_arrive_noinc(&ctrl->full[stage]);
        if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp >= EPI_WARP0) {
    // =============================== epilogue: TMEM -> bias / ReLU -> scatter ================
    // One or two warps per TMEM lane quarter (warp % 4; two split the columns) drain accumulator
    // `buf` while the MMA warp fills the other one and the gather warps fetch the next segment.
    const int etid = tid - EPI_WARP0 * 32;
    const int q = warp & 3;                                  // TMEM lane quarter of this warp
    const int row = q * 32 + lane;
    uint32_t sidx = 0, red_phase = 0;
    TileSeg sg = seg0;
    while (sg.next()) {
      const int tile = sg.tile, kb0 = sg.kb0, kb1 = sg.kb1;
      const int nt = tile % ntiles;
      const uint32_t buf = sidx & 1u, use = sidx >> 1;
      ++sidx;
      // ---- epilogue: TMEM -> registers -> bias / ReLU -> scatter -------------------------
      mbar_wait(&ctrl->tab_full[buf], use & 1u);             // row table written
      mbar_wait(&ctrl->tmem_full[buf], use & 1u);            // accumulator complete
      tc_fence_after();
      const int pix = ctrl->pix[buf][row];
      const uint32_t trow = tmem_base + buf * (uint32_t)BN + ((uint32_t)(q * 32) << 16);
      TO* orow = out + (long long)(pix < 0 ? 0 : pix) * Op;
      constexpr int OVEC = 16 / (int)sizeof(TO);
      constexpr int NGROUP = UM_EPI / 128;                   // warps sharing a lane quarter
      constexpr int COLS = (BN / NGROUP) < 16 ? 16 : (BN / NGROUP);
      const int cbeg = ((warp - EPI_WARP0) >> 2) * COLS;
      // split-K partial buffer: float4 slot ((it*4 + i4) * 128 + etid) -> conflict-free, and the
      // same thread owns the same (row, columns) on every rank
      float4* red = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(ktab) + C::TABLE_MAX * 8);
      if (DEEP && KS > 1 && krank != 0) {
        mbar_wait_cluster(&ctrl->red_free, red_phase ^ 1u);  // rank 0 has consumed my last partial
        int it = 0;
#pragma unroll 1
        for (int c0 = cbeg; c0 < cbeg + COLS && c0 < BN; c0 += 16, ++it) {
          uint32_t acc[16];
          tmem_ld16(trow + (uint32_t)c0, acc);
          tmem_ld_wait();
#pragma unroll
          for (int i4 = 0; i4 < 4; ++i4)
            red[(it * 4 + i4) * UM_EPI + etid] =
                make_float4(__uint_as_float(acc[4 * i4]), __uint_as_float(acc[4 * i4 + 1]),
                            __uint_as_float(acc[4 * i4 + 2]), __uint_as_float(acc[4 * i4 + 3]));
        }
        tc_fence_before();
        mbar_arrive(&ctrl->tmem_empty[buf]);
        mbar_arrive_remote(map_to_rank(smem_u32(&ctrl->red_full), leader));   // release: partial visible
        red_phase ^= 1u;
        continue;
      }
      if (DEEP && KS > 1) mbar_wait_cluster(&ctrl->red_full, red_phase);   // all partials delivered
      // ---- stream-K: a tile cut by a range boundary -----------------------------------------
      int sk_c0 = 0, sk_c1 = 0;                              // contributors [sk_c0, sk_c1) to wait for
      if (!DEEP && sk && kb0 > 0) {
        // not the tile's first K blocks: park the partial accumulator, raise my flag, move on
        float4* slot = sk_part + (long long)blockIdx.x * SK_SLOT;
        int it2 = 0;
#pragma unroll 1
        for (int c0 = cbeg; c0 < cbeg + COLS && c0 < BN; c0 += 16, ++it2) {
          uint32_t acc[16];
          tmem_ld16(trow + (uint32_t)c0, acc);
          tmem_ld_wait();
#pragma unroll
          for (int i4 = 0; i4 < 4; ++i4)
            __stcg(&slot[(it2 * 4 + i4) * UM_EPI + etid],
                   make_float4(__uint_as_float(acc[4 * i4]), __uint_as_float(acc[4 * i4 + 1]),
                               __uint_as_float(acc[4 * i4 + 2]), __uint_as_float(acc[4 * i4 + 3])));
        }
        __threadfence();
        tc_fence_before();
        mbar_arrive(&ctrl->tmem_empty[buf]);
        asm volatile("bar.sync 2, %0;" ::"n"(UM_EPI) : "memory");
        if (etid == 0) st_release_gpu(sk_ws + blockIdx.x, 1u);
        continue;
      }
      if (!DEEP && sk && kb1 < num_kb) {
        // the tile's first K blocks, reached at the END of my range: the CTAs after me hold the
        // rest and processed it at the START of theirs
        sk_c0 = (int)blockIdx.x + 1;
        sk_c1 = sk_c0;
        const long long tile_end = (long long)(tile + 1) * num_kb;
        while (sk_c1 < (int)sk_grid && sk_units * sk_c1 / sk_grid < tile_end) ++sk_c1;
        if (etid == 0) {
          for (int cta = sk_c0; cta < sk_c1; ++cta) {
            long long t0 = 0;
            for (uint32_t spins = 0; ld_acquire_gpu(sk_ws + cta) == 0u; ++spins) {
              if ((spins & 1023u) == 1023u) {
                const long long now = clock64();
                if (t0 == 0) t0 = now;
                else if (now - t0 > 4000000000ll) __trap();
              }
            }
          }
        }
        asm volatile("bar.sync 2, %0;" ::"n"(UM_EPI) : "memory");
      }
      int it = 0;
#pragma unroll 1
      for (int c0 = cbeg; c0 < cbeg + COLS && c0 < BN; c0 += 16, ++it) {
        uint32_t acc[16];
        tmem_ld16(trow + (uint32_t)c0, acc);
        tmem_ld_wait();
        for (int cta = sk_c0; cta < sk_c1; ++cta) {          // stream-K partials (fixed order)
          const float4* slot = sk_part + (long long)cta * SK_SLOT;
#pragma unroll
          for (int i4 = 0; i4 < 4; ++i4) {
            const float4 p = __ldcg(&slot[(it * 4 + i4) * UM_EPI + etid]);
            acc[4 * i4] = __float_as_uint(__uint_as_float(acc[4 * i4]) + p.x);
            acc[4 * i4 + 1] = __float_as_uint(__uint_as_float(acc[4 * i4 + 1]) + p.y);
            acc[4 * i4 + 2] = __float_as_uint(__uint_as_float(acc[4 * i4 + 2]) + p.z);
            acc[4 * i4 + 3] = __float_as_uint(__uint_as_float(acc[4 * i4 + 3]) + p.w);
          }
        }
        if (DEEP && KS > 1) {
          for (uint32_t r = 1; r < KS; ++r) {
#pragma unroll
            for (int i4 = 0; i4 < 4; ++i4) {
              const float4 p = ld_cluster_f4(
                  map_to_rank(smem_u32(&red[(it * 4 + i4) * UM_EPI + etid]), leader + r));
              acc[4 * i4] = __float_as_uint(__uint_as_float(acc[4 * i4]) + p.x);
              acc[4 * i4 + 1] = __float_as_uint(__uint_as_float(acc[4 * i4 + 1]) + p.y);
              acc[4 * i4 + 2] = __float_as_uint(__uint_as_float(acc[4 * i4 + 2]) + p.z);
              acc[4 * i4 + 3] = __float_as_uint(__uint_as_float(acc[4 * i4 + 3]) + p.w);
            }
          }
        }
        const int co0 = nt * BN + c0;
        if (pix >= 0 && co0 < Cout) {
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int co = co0 + i;
            // relu bit 1 (cb_conv_accumulate): out += contraction, no bias (fine-grained delta update)
            float t = __uint_as_float(acc[i]) +
                      (co < Cout ? ((relu & 2) ? to_float(orow[co]) : __ldg(bias + co)) : 0.f);
            if ((relu & 1) && t <= 0.f) t = 0.f;
            f[i] = t;
          }
          if (co0 + 16 <= Cout && (Op % OVEC) == 0) {        // full, 16-byte aligned run
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
                for (int e = 0; e < 8; ++e) h[e] = from_float<TO>(f[i + e]);
                *reinterpret_cast<uint4*>(orow + co0 + i) = *reinterpret_cast<uint4*>(h);
              }
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (co0 + i < Cout) orow[co0 + i] = from_float<TO>(f[i]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&ctrl->tmem_empty[buf]);
      if (DEEP && KS > 1) {                                  // the peers may reuse their partial buffers
        for (uint32_t r = 1; r < KS; ++r) mbar_arrive_remote(map_to_rank(smem_u32(&ctrl->red_free), leader + r));
        red_phase ^= 1u;
      }
      if (sk_c1 > sk_c0) {                                   // partials consumed: leave the flags clean
        asm volatile("bar.sync 2, %0;" ::"n"(UM_EPI) : "memory");
        if (etid == 0)
          for (int cta = sk_c0; cta < sk_c1; ++cta) sk_ws[cta] = 0u;
      }
    }
  } else if (warp == TMA_WARP) {
    // =============================== TMA producer: weight tiles ==============================
    // (whole warp, uniform operands, one elected lane issues: see the MMA warp)
    const bool leader = elect_one();
    uint32_t stage = 0, phase = 0;
    TileSeg sg = seg0;
    while (sg.next()) {
      const int nt = sg.tile % ntiles, kb0 = sg.kb0, kb1 = sg.kb1;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&ctrl->empty[stage], phase ^ 1u);
        if (leader) {
          const uint32_t b_hi = smem_u32(smem + stage * C::STAGE_BYTES + C::NSPLIT * C::A_BYTES);
          mbar_arrive_expect_tx(&ctrl->full[stage], (uint32_t)(C::NSPLIT * C::B_BYTES));
          tma_load_2d(b_hi, &wmap, kb * C::BK, nt * BN, &ctrl->full[stage]);
          if (SPLIT3) tma_load_2d(b_hi + C::B_BYTES, &wmap, kb * C::BK, CoutPad + nt * BN, &ctrl->full[stage]);
        }
        __syncwarp();
        if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == MMA_WARP) {
    // =============================== MMA issuer ==============================================
    // The whole warp walks the segments (uniform control flow, descriptors in uniform registers);
    // one elected lane issues.  Under `if (lane == 0)` the compiler cannot prove the descriptors
    // uniform and wraps every UTCHMMA in an ELECT / R2UR / branch loop (~150 cycles each, more than
    // the 128 cycles of tensor work of an N = 256 instruction).
    constexpr int KIND = sizeof(T) == 4 ? 0 : 1;
    const uint32_t idesc =
        umma_idesc(sizeof(T) == 4 ? 2 : (std::is_same<T, __half>::value ? 0 : 1), BN);
    const bool leader = elect_one();
    const uint32_t d_hi32 = (uint32_t)(umma_desc(0) >> 32);  // SBO | version | SWIZZLE_128B
    uint32_t stage = 0, phase = 0, sidx = 0;
    TileSeg sg = seg0;
    while (sg.next()) {
      const int kb0 = sg.kb0, kb1 = sg.kb1;
      const uint32_t buf = sidx & 1u, use = sidx >> 1;
      ++sidx;
      const uint32_t tmem_d = tmem_base + buf * (uint32_t)BN;
      mbar_wait(&ctrl->tmem_empty[buf], (use & 1u) ^ 1u);    // epilogue drained this accumulator
      tc_fence_after();
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&ctrl->full[stage], phase);
        fence_proxy_async_smem();                            // cp.async writes -> async proxy (UMMA)
        tc_fence_after();
        // running low words of the descriptors: start >> 4 | LBO (1) << 16
        const uint32_t a_hi = ((smem_u32(smem + stage * C::STAGE_BYTES) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t a_lo = a_hi + (uint32_t)(C::A_BYTES >> 4);
        const uint32_t b_hi = a_hi + (uint32_t)((C::NSPLIT * C::A_BYTES) >> 4);
        const uint32_t b_lo = b_hi + (uint32_t)(C::B_BYTES >> 4);
        if (leader) {
#pragma unroll
          for (int ks = 0; ks < C::BK / C::UK; ++ks) {
            const uint32_t adv = (uint32_t)(ks * 2);         // 32 bytes of K per instruction
            const uint32_t first = (kb != kb0 || ks) ? 1u : 0u;
            const uint64_t dA = ((uint64_t)d_hi32 << 32) | (a_hi + adv);
            const uint64_t dB = ((uint64_t)d_hi32 << 32) | (b_hi + adv);
            if (SPLIT3) {
              const uint64_t dAl = ((uint64_t)d_hi32 << 32) | (a_lo + adv);
              const uint64_t dBl = ((uint64_t)d_hi32 << 32) | (b_lo + adv);
              umma<KIND>(tmem_d, dAl, dB, idesc, first);
              umma<KIND>(tmem_d, dA, dBl, idesc, 1u);
              umma<KIND>(tmem_d, dA, dB, idesc, 1u);
            } else {
              umma<KIND>(tmem_d, dA, dB, idesc, first);
            }
          }
          umma_commit(&ctrl->empty[stage]);                  // frees the smem stage when done
        }
        __syncwarp();
        if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
      }
      if (leader) umma_commit(&ctrl->tmem_full[buf]);        // accumulator complete
      __syncwarp();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (DEEP && KSmax > 1) cluster_sync_all();               // nobody leaves while peers may touch its smem
  if (warp == MMA_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
  }
  if (mk.bits) rowmask_finish<TRACK>(mk, &ctrl->pad);
}

// ---- weight packing ----------------------------------------------------------------------------
// weight [Cout][Cin][kH][kW] (T) -> packed [NSPLIT][CoutPad][KpPad] (T), k = (ky*kW+kx)*Cp + ci.
// fp32 + SPLIT3: plane 0 = tf32-truncated hi, plane 1 = lo = w - hi (exact).
// split: 0 none, 1 = tf32 hi (truncated) + lo, 2 = bf16 hi (rounded) + lo
template <typename T, typename TP>
__global__ void pack_weights_umma_kernel(const T* __restrict__ w, TP* __restrict__ packed, int Cout,
                                         int Cin, int kH, int kW, int Cp, int CoutPad, int KpPad,
                                         int split3) {
  const long long plane = (long long)CoutPad * KpPad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < plane;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % KpPad);
    const int co = (int)(i / KpPad);
    const int tap = k / Cp, ci = k - tap * Cp;
    const int ky = tap / kW, kx = tap - ky * kW;
    float f = 0.f;
    if (co < Cout && ci < Cin && tap < kH * kW)
      f = to_float(w[(((long long)co * Cin + ci) * kH + ky) * kW + kx]);
    if (split3 == 1) {
      const float hi = __uint_as_float(__float_as_uint(f) & 0xFFFFE000u);
      packed[i] = from_float<TP>(hi);
      packed[plane + i] = from_float<TP>(f - hi);
    } else if (split3 == 2) {
      const TP hi = from_float<TP>(f);
      packed[i] = hi;
      packed[plane + i] = from_float<TP>(f - to_float(hi));
    } else {
      packed[i] = from_float<TP>(f);     // exact: TP == T
    }
  }
}

inline int umma_bn(int gemm, int Cout) {
  const int maxbn = 256;
  int bn = 16;
  while (bn < Cout && bn < maxbn) bn <<= 1;
  return bn;
}
inline int umma_cout_pad(int gemm, int Cout) {
  const int bn = umma_bn(gemm, Cout);
  return (Cout + bn - 1) / bn * bn;
}
inline int umma_kp_pad_es(int es, int Cp, int kH, int kW) {
  const int bk = UM_ROW_BYTES / es;
  return (kH * kW * Cp + bk - 1) / bk * bk;
}
// operand element size of a (dtype, gemm) pair: 3xBF16 feeds bf16 planes of fp32 data
inline int umma_operand_es(int dtype, int gemm) {
  return gemm == CB_GEMM_TC_BF16X3 ? 2 : esize(dtype);
}
inline int umma_kp_pad(int dtype, int Cp, int kH, int kW) {
  return umma_kp_pad_es(esize(dtype), Cp, kH, kW);
}

inline bool umma_is_split(int dtype, int gemm) {
  return dtype == CB_F32 && (gemm == CB_GEMM_TC_3X || gemm == CB_GEMM_TC_BF16X3);
}
inline size_t umma_packed_bytes(int dtype, int gemm, int Cout, int Cp, int kH, int kW) {
  const int nsplit = umma_is_split(dtype, gemm) ? 2 : 1;
  const int es = umma_operand_es(dtype, gemm);
  return (size_t)nsplit * umma_cout_pad(gemm, Cout) * umma_kp_pad_es(es, Cp, kH, kW) * es;
}

inline int umma_pack_weights(cudaStream_t s, int dtype, int gemm, const void* weight, void* packed,
                             int Cout, int Cin, int Cp, int kH, int kW) {
  CB_CHECK_ARG(gemm == CB_GEMM_TC || gemm == CB_GEMM_TC_3X || gemm == CB_GEMM_TC_BF16X3,
               "pack_weights: bad gemm mode %d", gemm);
  CB_CHECK_ARG(gemm != CB_GEMM_TC_BF16X3 || dtype == CB_F32, "pack_weights: 3xBF16 is for fp32 data");
  const int es = umma_operand_es(dtype, gemm);
  const int CoutPad = umma_cout_pad(gemm, Cout), KpPad = umma_kp_pad_es(es, Cp, kH, kW);
  const long long plane = (long long)CoutPad * KpPad;
  long long blocks = (plane + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  switch (dtype) {
    case CB_F32:
      if (gemm == CB_GEMM_TC_BF16X3)
        cb::launch(pack_weights_umma_kernel<float, __nv_bfloat16>, (unsigned)blocks, 256, 0, s, 
            (const float*)weight, (__nv_bfloat16*)packed, Cout, Cin, kH, kW, Cp, CoutPad, KpPad, 2);
      else
        cb::launch(pack_weights_umma_kernel<float, float>, (unsigned)blocks, 256, 0, s, 
            (const float*)weight, (float*)packed, Cout, Cin, kH, kW, Cp, CoutPad, KpPad,
            gemm == CB_GEMM_TC_3X ? 1 : 0);
      break;
    case CB_F16:
      cb::launch(pack_weights_umma_kernel<__half, __half>, (unsigned)blocks, 256, 0, s, 
          (const __half*)weight, (__half*)packed, Cout, Cin, kH, kW, Cp, CoutPad, KpPad, 0);
      break;
    case CB_BF16:
      cb::launch(pack_weights_umma_kernel<__nv_bfloat16, __nv_bfloat16>, (unsigned)blocks, 256, 0, s, 
          (const __nv_bfloat16*)weight, (__nv_bfloat16*)packed, Cout, Cin, kH, kW, Cp, CoutPad,
          KpPad, 0);
      break;
    default: return fail(2, "pack_weights: bad dtype %d", dtype);
  }
  CB_CHECK_LAUNCH("pack_weights(umma)");
  return 0;
}

// ---- host: tensor map + launch -----------------------------------------------------------------
inline PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

template <typename T, typename TO, bool SPLIT3, int BN, bool DEEP, bool TRACK>
int launch_conv_umma(cudaStream_t s, int dtype, const void* state, const void* state_lo, int Cp,
                     const int32_t* idx,
                     const int32_t* count, const void* packed, const float* bias, void* out,
                     int Op, int B, int H, int W, int Cout, int CoutPad, int kH, int kW, int relu,
                     int sel_lo, int sel_hi, int ksplit, void* ws, size_t ws_bytes,
                     const RowMask& mk) {
  using C = UmmaCfg<T, SPLIT3, BN, DEEP>;
  const int Kp = kH * kW * Cp;
  const int KpPad = umma_kp_pad_es((int)sizeof(T), Cp, kH, kW);
  (void)dtype;
  auto enc = tensor_map_encoder();
  if (!enc) return fail(3, "conv_update: cuTensorMapEncodeTiled unavailable");
  alignas(64) CUtensorMap map;
  const cuuint64_t gdim[2] = {(cuuint64_t)KpPad, (cuuint64_t)(C::NSPLIT * CoutPad)};
  const cuuint64_t gstr[1] = {(cuuint64_t)KpPad * sizeof(T)};
  const cuuint32_t box[2] = {(cuuint32_t)C::BK, (cuuint32_t)BN};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : std::is_same<T, __half>::value ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                                  : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const CUresult r = enc(&map, dt, 2, const_cast<void*>(packed), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(3, "conv_update: cuTensorMapEncodeTiled failed (%d)", (int)r);
  auto kern = conv_umma_kernel<T, TO, SPLIT3, BN, DEEP, TRACK>;
  static thread_local int attr_dev = -1;
  int dev = 0;
  cudaGetDevice(&dev);
  if (attr_dev != dev) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES) !=
        cudaSuccess)
      return fail(3, "conv_update: cannot reserve %d bytes of shared memory", C::SMEM_BYTES);
    attr_dev = dev;
  }
  // shared memory actually needed: stages + alignment slack + ctrl + the K-chunk table of THIS
  // layer (small layers then fit a third CTA per SM -> more gather stages in flight)
  const int num_kb = KpPad / C::BK;
  const int upc = (sizeof(T) == 2 && Cp == 4) ? 2 : 1;
  const int table_entries = num_kb * 8 * upc <= C::TABLE_MAX ? num_kb * 8 * upc : 0;
  // (the 1024-byte alignment slack is only needed if the dynamic smem window is not already
  //  1024-aligned; it is when the kernel has no static shared memory, which the kernel checks)
  const int smem_bytes = DEEP ? C::STAGES * C::STAGE_BYTES + UM_CTRL_BYTES + C::TABLE_MAX * 8 + C::RED_BYTES
                              : C::STAGES * C::STAGE_BYTES + UM_CTRL_BYTES + table_entries * 8;
  int occ = C::CTAS_PER_SM;
  int occ_real = 0;                                          // what the runtime says fits (cooperative launches need it exact)
  if (!DEEP) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_real, kern, um_threads(BN), smem_bytes) == cudaSuccess &&
        occ_real > occ)
      occ = occ_real > 4 ? 4 : occ_real;
  }
  if (occ > 512 / C::TMEM_COLS) occ = 512 / C::TMEM_COLS;     // two accumulators per CTA must fit TMEM
  const long long max_tiles = (((long long)B * H * W + UM_BM - 1) / UM_BM) * (CoutPad / BN);
  // split-K (deep variant only): clusters of `ks` CTAs share a tile; keep ks <= stages / 4
  int ks = DEEP ? ksplit : 1;
  while (ks > 1 && num_kb / ks < 4) ks >>= 1;
  long long grid = (long long)sm_count() * occ / ks;       // clusters
  if (ks > 1) {
    // co-resident clusters of this size (GPC boundaries strand a few SMs); fall back to smaller
    // clusters when the big ones would leave more than ~15 % of the SMs unused
    static thread_local int act[4] = {-1, -1, -1, -1}, act_dev = -1;
    if (act_dev != dev) { act[0] = act[1] = act[2] = act[3] = -1; act_dev = dev; }
    for (; ks > 1; ks >>= 1) {
      const int slot = ks == 8 ? 3 : ks == 4 ? 2 : 1;
      if (act[slot] < 0) {
        cudaLaunchConfig_t qc = {};
        qc.gridDim = dim3((unsigned)(sm_count() / ks * ks));
        qc.blockDim = dim3(um_threads(BN));
        qc.dynamicSmemBytes = (size_t)smem_bytes;
        cudaLaunchAttribute qa[1];
        qa[0].id = cudaLaunchAttributeClusterDimension;
        qa[0].val.clusterDim.x = (unsigned)ks;
        qa[0].val.clusterDim.y = qa[0].val.clusterDim.z = 1;
        qc.attrs = qa;
        qc.numAttrs = 1;
        int nclusters = 0;
        if (cudaOccupancyMaxActiveClusters(&nclusters, kern, &qc) != cudaSuccess) {
          cudaGetLastError();
          nclusters = 0;
        }
        act[slot] = nclusters;
      }
      if ((long long)act[slot] * ks * 100 >= (long long)sm_count() * 85) break;
    }
    grid = ks > 1 ? act[ks == 8 ? 3 : ks == 4 ? 2 : 1] : (long long)sm_count() * occ;
  }
  // stream-K (coarse variant, K long enough to be worth cutting): every resident CTA slot gets an
  // equal share of the (tile, K block) space; needs flags + one partial tile per CTA of workspace
  uint32_t* sk_ws = nullptr;
  if (!DEEP && ws && num_kb >= 8 && ws_bytes > (size_t)UM_SK_FLAG_BYTES) {
    const long long slots = (long long)((ws_bytes - UM_SK_FLAG_BYTES) / ((size_t)UM_BM * BN * sizeof(float)));
    if (slots >= sm_count() / 2) {                           // enough partial-tile slots to be useful
      if (grid > slots) grid = slots;
      if (grid * (long long)sizeof(uint32_t) > UM_SK_FLAG_BYTES) grid = UM_SK_FLAG_BYTES / sizeof(uint32_t);
      if (occ_real > 0 && grid > (long long)sm_count() * occ_real) grid = (long long)sm_count() * occ_real;
      sk_ws = (uint32_t*)ws;
    }
  }
  if (!sk_ws && grid > max_tiles) grid = max_tiles;
  if (grid < 1) grid = 1;
  grid *= ks;
  // stream-K CTAs wait for each other's partial tiles: cooperative launch = all of them resident, also
  // next to another stream-K grid on a concurrent stream (PoseModel.parallelBranches)
  cb::launch_cluster(kern, (unsigned)grid, um_threads(BN), (size_t)smem_bytes, s, (unsigned)ks,
                     sk_ws ? 1 : 0, map, (const T*)state, (const T*)state_lo, Cp,
                                                        idx, count, bias,
                                                        (TO*)out, Op, H, W, Cout, CoutPad, kH, kW,
                                                        Kp, relu, sel_lo, sel_hi, sk_ws, mk);
  CB_CHECK_LAUNCH("conv_update(umma)");
  return 0;
}

template <typename T, typename TO, bool SPLIT3, bool DEEP, bool TRACK>
int dispatch_bn(int bn, cudaStream_t s, int dtype, const void* state, const void* state_lo, int Cp,
                const int32_t* idx,
                const int32_t* count, const void* packed, const float* bias, void* out, int Op,
                int B, int H, int W, int Cout, int CoutPad, int kH, int kW, int relu, int sel_lo,
                int sel_hi, int ksplit, void* ws, size_t ws_bytes, const RowMask& mk) {
#define CB_BN(N)                                                                              \
  case N:                                                                                     \
    return launch_conv_umma<T, TO, SPLIT3, N, DEEP, TRACK>(s, dtype, state, state_lo, Cp, idx, count, packed, bias, out, \
                                          Op, B, H, W, Cout, CoutPad, kH, kW, relu, sel_lo,   \
                                          sel_hi, ksplit, ws, ws_bytes, mk);
  if constexpr (DEEP) {                        // the deep variant only exists for N tiles <= 64
    switch (bn) {
      CB_BN(16) CB_BN(32) CB_BN(64)
      default: return fail(2, "conv_update: unsupported deep N tile %d", bn);
    }
  } else {
    switch (bn) {
      CB_BN(16) CB_BN(32) CB_BN(64) CB_BN(128) CB_BN(256)
      default: return fail(2, "conv_update: unsupported N tile %d", bn);
    }
  }
#undef CB_BN
}

inline int umma_conv_update(cudaStream_t s, int dtype, int gemm, const void* state,
                            const void* state_lo, int Cp, const int32_t* idx, const int32_t* count, const void* packed,
                            const float* bias, void* out, int Op, int B, int H, int W, int Cin,
                            int Cout, int kH, int kW, int relu, void* ws, size_t ws_bytes,
                            const RowMask& mk = RowMask{nullptr, nullptr, nullptr, nullptr, 0}) {
  (void)Cin;
  CB_CHECK_ARG(gemm == CB_GEMM_TC || gemm == CB_GEMM_TC_3X || gemm == CB_GEMM_TC_BF16X3,
               "conv_update: bad gemm mode %d", gemm);
  CB_CHECK_ARG(gemm != CB_GEMM_TC_BF16X3 || dtype == CB_F32, "conv_update: 3xBF16 is for fp32 data");
  CB_CHECK_ARG(H < 32768 && W < 32768, "conv_update: H, W must be < 32768");
  CB_CHECK_ARG(((uintptr_t)state % 16) == 0 && ((uintptr_t)packed % 128) == 0,
               "conv_update: state must be 16-byte and packed weights 128-byte aligned");
  const int bn = umma_bn(gemm, Cout), CoutPad = umma_cout_pad(gemm, Cout);
  const bool split3 = gemm == CB_GEMM_TC_3X && dtype == CB_F32;
  const bool bf16x3 = gemm == CB_GEMM_TC_BF16X3;
  CB_CHECK_ARG(!(bf16x3 && Cp == 4) || kH * kW <= 256,
               "conv_update: 8-byte-tap layers support up to 256 filter taps");
  CB_CHECK_ARG(!(split3 || bf16x3) || (state_lo && ((uintptr_t)state_lo % 16) == 0),
               "conv_update: the 3x modes need their 16-byte aligned lo operand plane (state_lo)");
  // Tiling policy.  Large N tiles minimise the im2col re-gather (the kernel is L2-bound on big
  // layers) but give few CTAs when few pixels changed; the count is only known on the device, so
  // when a small change set is plausible (expected tiles at 10 % change < half the SMs) a second,
  // finer tiling is launched as well and each kernel checks the count to see whether it is its turn.
  auto run_tt = [&](auto deep_tag, auto track_tag, int tile_n, int lo, int hi, int ksplit) -> int {
    constexpr bool DP = decltype(deep_tag)::value, TR = decltype(track_tag)::value;
    if (bf16x3)
      return dispatch_bn<__nv_bfloat16, float, true, DP, TR>(tile_n, s, dtype, state, state_lo, Cp, idx,
                                                         count, packed, bias, out, Op, B, H, W,
                                                         Cout, CoutPad, kH, kW, relu, lo, hi, ksplit, ws, ws_bytes, mk);
    switch (dtype) {
      case CB_F32:
        return split3 ? dispatch_bn<float, float, true, DP, TR>(tile_n, s, dtype, state, state_lo, Cp, idx, count,
                                                 packed, bias, out, Op, B, H, W, Cout, CoutPad, kH,
                                                 kW, relu, lo, hi, ksplit, ws, ws_bytes, mk)
                      : dispatch_bn<float, float, false, DP, TR>(tile_n, s, dtype, state, state_lo, Cp, idx, count,
                                                  packed, bias, out, Op, B, H, W, Cout, CoutPad,
                                                  kH, kW, relu, lo, hi, ksplit, ws, ws_bytes, mk);
      case CB_F16:
        return dispatch_bn<__half, __half, false, DP, TR>(tile_n, s, dtype, state, state_lo, Cp, idx, count, packed,
                                          bias, out, Op, B, H, W, Cout, CoutPad, kH, kW, relu, lo, hi, ksplit, ws, ws_bytes, mk);
      case CB_BF16:
        return dispatch_bn<__nv_bfloat16, __nv_bfloat16, false, DP, TR>(tile_n, s, dtype, state, state_lo, Cp, idx, count,
                                                 packed, bias, out, Op, B, H, W, Cout, CoutPad, kH,
                                                 kW, relu, lo, hi, ksplit, ws, ws_bytes, mk);
      default: return fail(2, "conv_update: bad dtype %d", dtype);
    }
  };
  auto run_t = [&](auto deep_tag, int tile_n, int lo, int hi, int ksplit = 1) -> int {
    return mk.stream_counts ? run_tt(deep_tag, std::true_type{}, tile_n, lo, hi, ksplit)
                            : run_tt(deep_tag, std::false_type{}, tile_n, lo, hi, ksplit);
  };
  const long long P = (long long)B * H * W;
  const int sms = sm_count();
  const long long exp_tiles = (P / 10 / UM_BM + 1) * (CoutPad / bn);
  // (short K - 1x1 layers, the RGB layer - gains nothing from the fine variant: a tile is only a
  //  few stages long, and the second launch costs ~2 us; measured 8.5 -> 6.8 and 11.1 -> 9.1 us)
  const int num_kb_all = umma_kp_pad_es(umma_operand_es(dtype, gemm), Cp, kH, kW) /
                         (UM_ROW_BYTES / umma_operand_es(dtype, gemm));
  if (exp_tiles < sms / 2 && num_kb_all >= 8) {
    // small-change regime: fewer tiles than SMs, so run ONE CTA per SM with a deep stage ring
    // (latency-bound otherwise) and, for wide layers, a 4x finer N tiling to spread the work
    int bn_small = bn > 64 ? (bn / 4 < 64 ? 64 : bn / 4) : bn;
    if (bn_small > 64) bn_small = 64;
    // switch point: the coarse tiling takes over once it alone fills ~2/3 of the SMs
    int m_switch = (2 * sms / 3) / (CoutPad / bn);
    // ... or much earlier when stream-K can spread few coarse tiles over all SMs (a tile cut into
    // <= ~4 K ranges keeps the finisher's partial sums cheap): measured cross-over ~sms/4 tiles
    if (ws && ws_bytes > (size_t)UM_SK_FLAG_BYTES && CoutPad == bn && m_switch > sms / 4)
      m_switch = sms / 4;
    if (m_switch < 1) m_switch = 1;
    // split-K over thread-block clusters: few tiles x long K (small maps, big filters) would
    // otherwise leave most SMs idle and each busy SM limited by its own L2 ingest rate
    const int num_kb = umma_kp_pad_es(umma_operand_es(dtype, gemm), Cp, kH, kW) /
                       (UM_ROW_BYTES / umma_operand_es(dtype, gemm));
    static const int ks_max = [] {
      const char* e = getenv("CBINFER_KSPLIT");              // tuning knob: cap (1 disables)
      const int v = e ? atoi(e) : 8;
      return v < 1 ? 1 : v > 8 ? 8 : v;
    }();
    int ksplit = 1;
    while (ksplit < ks_max && num_kb / (ksplit * 2) >= 6) ksplit *= 2;   // the kernel narrows it
    const int rc = run_t(std::true_type{}, bn_small, 0, m_switch, ksplit);
    if (rc) return rc;
    return run_t(std::false_type{}, bn, m_switch, 0x7fffffff);
  }
  return run_t(std::false_type{}, bn, 0, 0x7fffffff);
}

}  // namespace cb
