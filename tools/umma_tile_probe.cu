// umma_tile_probe.cu -- hardware probe for the spatially tiled contraction (conv_tile.cuh).
//
// Question: can tcgen05.mma read the im2col rows of a 7x7 filter tap STRAIGHT out of a TMA-loaded
// pixel-major halo tile, i.e. with a shared-memory matrix descriptor whose start address is the
// tap's pixel (any multiple of the pixel size, not a swizzle-atom boundary)?  Row r of an 8-row
// core group = 8 x-consecutive pixels (row pitch = pixel bytes = swizzle width), SBO = halo row
// pitch.  Modes:
//   0  16-byte pixels (8 bf16 channels), SWIZZLE_NONE, two taps per K=16 MMA (LBO = tap distance)
//   1  32-byte pixels, SWIZZLE_32B        2  64-byte pixels, SWIZZLE_64B
//   3  128-byte pixels, SWIZZLE_128B
//   4  channel-blocked planes [Cp/8][y][x][8] (one TMA box per block), SWIZZLE_NONE, LBO = plane
// Variants (swizzled modes): descriptor base_offset = 0 | (start >> 7) & 7.
// Prints MATCH / MISMATCH per (mode, variant, tile origin) against a host im2col reference (small
// integer data: exact in fp32) and the TMA halo load latency in cycles.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -O2 -o tools/umma_tile_probe.bin tools/umma_tile_probe.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../cbinfer_b200/csrc/conv_umma.cuh"

namespace cb {
thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) { (void)fmt; return code; }
int sm_count() { return 148; }
}  // namespace cb

using namespace cb;

constexpr int KH = 7, KW = 7, TW = 8, TH = 16, HWX = TW + KW - 1, HWY = TH + KH - 1;   // halo 14 x 22
constexpr int NOUT = 16;

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            int c3, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout, uint32_t base_off) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)(base_off & 7u) << 49) |
         ((uint64_t)layout << 61);
}

struct ProbeCtrl {
  uint64_t bar_tma, bar_mma;
  uint32_t tmem_base, pad;
};

// w: [NOUT][Kpad] bf16 (K = (ky,kx,ci), Kpad multiple of 64); out: [128][NOUT] fp32
__global__ void __launch_bounds__(128)
probe_kernel(const __grid_constant__ CUtensorMap amap, const __nv_bfloat16* __restrict__ w,
             float* __restrict__ out, int Cp, int Kpad, int mode, int variant, int x0, int y0,
             unsigned long long* cycles) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int pixb = Cp * 2;
  const int halo_bytes = HWX * HWY * pixb;
  const int b_off = (halo_bytes + 1023) / 1024 * 1024;
  const int num_kb = Kpad / 64;
  uint8_t* btile = smem + b_off;
  ProbeCtrl* ctrl = reinterpret_cast<ProbeCtrl*>(btile + num_kb * NOUT * 128);
  // weights -> K-major SWIZZLE_128B tiles (the layout the shipped kernel's TMA produces)
  for (int i = tid; i < NOUT * Kpad; i += blockDim.x) {
    const int n = i / Kpad, k = i - n * Kpad;
    const int kb = k >> 6, kk = k & 63;
    uint8_t* p = btile + kb * (NOUT * 128) + n * 128 + ((((kk >> 3) ^ (n & 7))) << 4) + (kk & 7) * 2;
    *reinterpret_cast<__nv_bfloat16*>(p) = w[i];
  }
  if (tid == 0) {
    mbar_init(&ctrl->bar_tma, 1);
    mbar_init(&ctrl->bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&ctrl->tmem_base)), "r"(32u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = ctrl->tmem_base;
  long long t0 = 0;
  if (tid == 0) {
    t0 = clock64();
    mbar_arrive_expect_tx(&ctrl->bar_tma, (uint32_t)halo_bytes);
    if (mode == 4) {
      for (int cb8 = 0; cb8 < Cp / 8; ++cb8)
        tma_load_4d(smem_u32(smem) + cb8 * (HWX * HWY * 16), &amap, cb8 * 8, x0 - KW / 2, y0 - KH / 2, 0,
                    &ctrl->bar_tma);
    } else {
      tma_load_4d(smem_u32(smem), &amap, 0, x0 - KW / 2, y0 - KH / 2, 0, &ctrl->bar_tma);
    }
  }
  mbar_wait(&ctrl->bar_tma, 0);
  if (tid == 0) {
    cycles[0] = (unsigned long long)(clock64() - t0);
    tc_fence_after();
    const uint32_t idesc = umma_idesc(1, NOUT);
    const uint32_t halo = smem_u32(smem), bbase = smem_u32(btile);
    const int K = KH * KW * Cp;
    const uint32_t layout = mode == 1 ? 6u : mode == 2 ? 4u : mode == 3 ? 2u : 0u;
    int first = 1;
    for (int k0 = 0; k0 < K; k0 += 16) {
      const int tap = k0 / Cp, ci0 = k0 - tap * Cp;
      const int ky = tap / KW, kx = tap - ky * KW;
      uint32_t a_addr, lbo = 16, sbo;
      if (mode == 0) {               // Cp == 8: taps `tap` and `tap + 1`
        const int t1 = tap + 1, ky1 = t1 / KW, kx1 = t1 - ky1 * KW;
        a_addr = halo + (uint32_t)((ky * HWX + kx) * 16);
        lbo = (uint32_t)(((ky1 * HWX + kx1) - (ky * HWX + kx)) * 16);
        sbo = HWX * 16;
      } else if (mode == 4) {        // channel-blocked planes of 8 channels
        a_addr = halo + (uint32_t)((ci0 / 8) * (HWX * HWY * 16) + (ky * HWX + kx) * 16);
        lbo = HWX * HWY * 16;
        sbo = HWX * 16;
      } else {
        a_addr = halo + (uint32_t)((ky * HWX + kx) * pixb + ci0 * 2);
        sbo = (uint32_t)(HWX * pixb);
      }
      const uint32_t boff = variant ? ((a_addr >> 7) & 7u) : 0u;
      const uint64_t adesc = make_desc(a_addr, lbo, sbo, layout, boff);
      const uint64_t bdesc = umma_desc(bbase + (uint32_t)((k0 >> 6) * (NOUT * 128) + (k0 & 63) * 2));
      umma<1>(tmem, adesc, bdesc, idesc, first ? 0u : 1u);
      first = 0;
    }
    umma_commit(&ctrl->bar_mma);
  }
  mbar_wait(&ctrl->bar_mma, 0);
  tc_fence_after();
  uint32_t acc[16];
  tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16), acc);
  tmem_ld_wait();
  const int m = warp * 32 + lane;
  for (int i = 0; i < NOUT; ++i) out[m * NOUT + i] = __uint_as_float(acc[i]);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(32u) : "memory");
  }
}

#define CK(x)                                                                      \
  do {                                                                             \
    cudaError_t e_ = (x);                                                          \
    if (e_ != cudaSuccess) {                                                       \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      exit(1);                                                                     \
    }                                                                              \
  } while (0)

static float bf(int v) { return (float)v; }

int main(int argc, char** argv) {
  const int only = argc > 1 ? atoi(argv[1]) : -1;      // one pass per process: a fault cannot hide the others
  const int H = 40, W = 36;
  auto enc = tensor_map_encoder();
  if (!enc) { printf("no cuTensorMapEncodeTiled\n"); return 1; }
  CK(cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  int all_ok = 1;
  const int mode_cp[5] = {8, 16, 32, 64, 16};
  for (int pass = 0; pass < 6; ++pass) {
    if (only >= 0 && pass != only) continue;
    const int mode = pass < 5 ? pass : 4;
    const int Cp = pass == 5 ? 64 : mode_cp[mode];     // mode 4 also at Cp = 64
    const int K = KH * KW * Cp, Kpad = (K + 63) / 64 * 64;
    std::vector<__nv_bfloat16> hs((size_t)H * W * Cp), hw((size_t)NOUT * Kpad);
    std::vector<int> is((size_t)H * W * Cp), iw((size_t)NOUT * Kpad, 0);
    srand(1234 + pass);
    for (size_t i = 0; i < is.size(); ++i) { is[i] = rand() % 9 - 4; hs[i] = __float2bfloat16(bf(is[i])); }
    for (int n = 0; n < NOUT; ++n)
      for (int k = 0; k < Kpad; ++k) {
        const int v = k < K ? rand() % 5 - 2 : 0;
        iw[(size_t)n * Kpad + k] = v;
        hw[(size_t)n * Kpad + k] = __float2bfloat16(bf(v));
      }
    __nv_bfloat16 *ds, *dw;
    float* dout;
    unsigned long long* dcy;
    CK(cudaMalloc(&ds, hs.size() * 2));
    CK(cudaMalloc(&dw, hw.size() * 2));
    CK(cudaMalloc(&dout, 128 * NOUT * 4));
    CK(cudaMalloc(&dcy, 8));
    CK(cudaMemcpy(ds, hs.data(), hs.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dw, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice));
    alignas(64) CUtensorMap map;
    const int boxc = mode == 4 ? 8 : Cp;
    const cuuint64_t gdim[4] = {(cuuint64_t)Cp, (cuuint64_t)W, (cuuint64_t)H, 1};
    const cuuint64_t gstr[3] = {(cuuint64_t)Cp * 2, (cuuint64_t)W * Cp * 2, (cuuint64_t)H * W * Cp * 2};
    const cuuint32_t box[4] = {(cuuint32_t)boxc, HWX, HWY, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUtensorMapSwizzle sw = mode == 1 ? CU_TENSOR_MAP_SWIZZLE_32B : mode == 2 ? CU_TENSOR_MAP_SWIZZLE_64B
                                  : mode == 3 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE;
    const CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ds, gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { printf("mode %d Cp %d: tensor map encode failed (%d)\n", mode, Cp, (int)r); all_ok = 0; continue; }
    const int origins[4][2] = {{0, 0}, {W - TW, H - TH}, {8, 16}, {13, 5}};
    const int nvar = (mode >= 1 && mode <= 3) ? 2 : 1;
    for (int variant = 0; variant < nvar; ++variant)
      for (int o = 0; o < 4; ++o) {
        const int x0 = origins[o][0], y0 = origins[o][1];
        CK(cudaMemset(dout, 0xff, 128 * NOUT * 4));
        const int smem_bytes = (HWX * HWY * Cp * 2 + 1023) / 1024 * 1024 + (Kpad / 64) * NOUT * 128 + 64;
        probe_kernel<<<1, 128, smem_bytes>>>(map, dw, dout, Cp, Kpad, mode, variant, x0, y0, dcy);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { printf("mode %d Cp %d variant %d: kernel error %s\n", mode, Cp, variant, cudaGetErrorString(e)); return 2; }
        std::vector<float> ho(128 * NOUT);
        unsigned long long cy = 0;
        CK(cudaMemcpy(ho.data(), dout, ho.size() * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(&cy, dcy, 8, cudaMemcpyDeviceToHost));
        int bad = 0;
        double maxerr = 0;
        for (int m = 0; m < 128; ++m) {
          const int y = y0 + m / 8, x = x0 + m % 8;
          for (int n = 0; n < NOUT; ++n) {
            long long acc = 0;
            for (int ky = 0; ky < KH; ++ky)
              for (int kx = 0; kx < KW; ++kx) {
                const int yy = y + ky - KH / 2, xx = x + kx - KW / 2;
                if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
                for (int c = 0; c < Cp; ++c)
                  acc += (long long)is[((size_t)yy * W + xx) * Cp + c] * iw[(size_t)n * Kpad + (ky * KW + kx) * Cp + c];
              }
            const double err = fabs((double)ho[m * NOUT + n] - (double)acc);
            if (err > maxerr) maxerr = err;
            if (err > 0.5) ++bad;
          }
        }
        printf("mode %d Cp %2d (pixel %3d B) variant base_off=%s origin (%2d,%2d): %s  bad %4d/2048 maxerr %.1f  tma %llu cycles\n",
               mode, Cp, Cp * 2, variant ? "addr>>7" : "0", x0, y0, bad ? "MISMATCH" : "MATCH", bad, maxerr, cy);
        if (bad && !(nvar == 2)) all_ok = 0;
      }
    cudaFree(ds); cudaFree(dw); cudaFree(dout); cudaFree(dcy);
  }
  printf("PROBE %s\n", all_ok ? "DONE" : "DONE (some no-swizzle modes mismatched)");
  return 0;
}
