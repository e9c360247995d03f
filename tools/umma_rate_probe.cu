// umma_rate_probe.cu -- how fast does ONE CTA issue/execute tcgen05.mma (M=128, kind::f16) for
// small N and for the A-operand access patterns of the tiled contraction?  One warp issues
// (warp-uniform code, elected lane), everything already in shared memory, no epilogue:
// cycles per instruction = the hardware floor for that descriptor pattern.
//   A patterns: 0 canonical SWIZZLE_128B tile (aligned, 128-byte rows)     [control]
//               1 halo taps, 32-byte pixels, SWIZZLE_32B (start = any 32-byte multiple)
//               2 halo taps, 16-byte pixels, no swizzle, two taps per instruction (LBO = tap distance)
//               3 halo taps, 128-byte pixels, SWIZZLE_128B (start = any 128-byte multiple)
//   seq: 1 = one MMA per K step, 3 = the 3xBF16 triple (a_lo*b_hi, a_hi*b_lo, a_hi*b_hi)
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -O2 -o tools/umma_rate_probe.bin tools/umma_rate_probe.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../cbinfer_b200/csrc/conv_tile.cuh"

namespace cb {
thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) { (void)fmt; return code; }
int sm_count() { return 148; }
}  // namespace cb
using namespace cb;

template <int N>
__global__ void __launch_bounds__(128) rate_kernel(int pattern, int seq, int reps, int nacc, unsigned long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  for (int i = threadIdx.x; i < 200 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (warp == 0) {
    const bool leader = elect_one();
    const uint32_t idesc = umma_idesc(1, N);
    const uint32_t abuf = smem_u32(smem), bbuf = abuf + 96 * 1024;     // A region 96 KB, B region after
    const int HWX = 14;
    const uint32_t pix = pattern == 1 ? 32u : pattern == 2 ? 16u : 128u;
    const uint64_t abase = pattern == 0 ? 0ull : tile_adesc_base(HWX * pix, pattern == 1 ? 6 : pattern == 2 ? 0 : 2);
    const long long t0 = clock64();
    if (pattern >= 10) {
      // minimal issue loop: running low words of the descriptors, one add each per K step
      const uint32_t px = pattern >= 11 ? 32u : 128u;
      const uint64_t ab = pattern >= 11 ? tile_adesc_base(HWX * px, 6) : (umma_desc(0) & ~0x3FFFull);
      const uint32_t ahi32 = (uint32_t)(ab >> 32), bhi32 = (uint32_t)(umma_desc(0) >> 32);
      const uint32_t lbo = 1u << 16;
      for (int r = 0; r < reps; ++r) {
        uint32_t alo = ((abuf & 0x3FFFFu) >> 4) | lbo, blo = ((bbuf & 0x3FFFFu) >> 4) | lbo;
        const uint32_t astep = pattern >= 11 ? px >> 4 : 2u;
        if (pattern == 12 || pattern == 13) {
          // four K steps per elected region (pattern 13: no branch at all, predicated issue)
#pragma unroll 1
          for (int i = 0; i < 48; i += 4) {
            uint32_t al[4], bl[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { al[j] = alo + (uint32_t)j * 2u; bl[j] = blo + (uint32_t)j * 2u; }
            if (leader) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint64_t ad_hi = ((uint64_t)ahi32 << 32) | al[j];
                const uint64_t ad_lo = ((uint64_t)ahi32 << 32) | (al[j] + 2560u);
                const uint64_t bd_hi = ((uint64_t)bhi32 << 32) | bl[j];
                if (seq == 3) {
                  umma<1>(tmem, ad_hi, bd_hi, idesc, 1u);
                  umma<1>(tmem, ad_lo, bd_hi, idesc, 1u);
                } else {
                  umma<1>(tmem, ad_hi, bd_hi, idesc, 1u);
                }
              }
            }
            alo += 8;
          }
        } else
#pragma unroll 1
        for (int i = 0; i < 49; ++i) {
          const uint64_t ad_hi = ((uint64_t)ahi32 << 32) | alo;
          const uint64_t ad_lo = ((uint64_t)ahi32 << 32) | (alo + 2560u);
          const uint64_t bd_hi = ((uint64_t)bhi32 << 32) | blo;
          const uint64_t bd_lo = ((uint64_t)bhi32 << 32) | (blo + (uint32_t)(N * 8));
          if (leader) {
            if (seq == 3) {
              umma<1>(tmem, ad_lo, bd_hi, idesc, 1u);
              umma<1>(tmem, ad_hi, bd_lo, idesc, 1u);
              umma<1>(tmem, ad_hi, bd_hi, idesc, 1u);
            } else {
              umma<1>(tmem, ad_hi, bd_hi, idesc, 1u);
            }
          }
          alo += astep;
          blo = (i & 3) == 3 ? blo - 6u : blo + 2u;
        }
      }
    } else
    for (int r = 0; r < reps; ++r) {
      uint32_t acc = 1;
      for (int ky = 0; ky < 7; ++ky)
        for (int kx = 0; kx < 7; ++kx) {
          const int tap = ky * 7 + kx;
          const uint32_t tm = tmem + (uint32_t)((tap % nacc) * N);
          uint64_t ad_hi, ad_lo;
          if (pattern == 0) {
            ad_hi = umma_desc(abuf + (uint32_t)((tap & 3) * 32 + (tap >> 2) * 16384 % 65536));
            ad_lo = umma_desc(abuf + 16384 + (uint32_t)((tap & 3) * 32));
          } else {
            const uint32_t off = (uint32_t)(ky * HWX + kx) * pix;
            const uint64_t ad = abase | ((uint64_t)(pattern == 2 ? 1u : 1u) << 16);
            ad_hi = ad | (uint64_t)(((abuf + off) & 0x3FFFFu) >> 4);
            ad_lo = ad | (uint64_t)(((abuf + 40960 + off) & 0x3FFFFu) >> 4);
          }
          const uint32_t b_hi = bbuf + (uint32_t)((tap >> 2) % (N > 64 ? 1 : 3)) * (2 * N * 128) + (uint32_t)(tap & 3) * 32;
          const uint32_t b_lo = b_hi + N * 128;
          if (leader) {
            if (seq == 3) {
              umma<1>(tm, ad_lo, umma_desc(b_hi), idesc, acc);
              umma<1>(tm, ad_hi, umma_desc(b_lo), idesc, 1u);
              umma<1>(tm, ad_hi, umma_desc(b_hi), idesc, 1u);
            } else {
              umma<1>(tm, ad_hi, umma_desc(b_hi), idesc, acc);
            }
          }
          acc = 1;
        }
    }
    if (leader) umma_commit(&bar);
    __syncwarp();
    mbar_wait(&bar, 0);
    const long long t1 = clock64();
    if (leader) out[0] = (unsigned long long)(t1 - t0);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
}

template <int N>
void run(int pattern, int seq, int nacc, int ctas, unsigned long long* d) {
  const int reps = 64;
  cudaFuncSetAttribute(rate_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  rate_kernel<N><<<ctas, 128, 200 * 1024>>>(pattern, seq, reps, nacc, d);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); exit(1); }
  unsigned long long cy = 0;
  cudaMemcpy(&cy, d, 8, cudaMemcpyDeviceToHost);
  const double n = (pattern == 12 ? 48.0 * (seq == 3 ? 2 : 1) : 49.0 * seq) * reps;
  printf("N=%3d pattern %d seq %d accumulators %d ctas %3d: %7.1f cycles / MMA  (tensor floor %d)\n", N, pattern, seq, nacc,
         ctas, cy / n, N / 2);
}

int main() {
  unsigned long long* d;
  cudaMalloc(&d, 8);
  for (int pattern = 10; pattern <= 12; ++pattern)
    for (int seq = 1; seq <= 3; seq += 2) {
      run<16>(pattern, seq, 1, 1, d);
      run<64>(pattern, seq, 1, 1, d);
      run<256>(pattern, seq, 1, 1, d);
    }
  for (int pattern = 0; pattern < 2; ++pattern)
    for (int seq = 1; seq <= 3; seq += 2) {
      run<16>(pattern, seq, 1, 1, d);
      run<64>(pattern, seq, 1, 1, d);
      run<256>(pattern, seq, 1, 1, d);
    }
  run<64>(11, 3, 1, 148, d);
  run<16>(11, 3, 1, 148, d);
  return 0;
}
