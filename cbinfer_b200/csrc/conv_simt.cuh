// conv_simt.cuh -- fused gather + contraction + bias/ReLU + scatter on CUDA cores (fp32 FFMA).
//
// Replaces genXMatrix_kernel (reference cbconv2d_cg_backend.cu:138-161), the cuBLAS GEMM behind
// matrixMult_python (conv2d_cg.py:342-349), the transpose copy (conv2d.py:247) and
// updateOutput_kernel (cbconv2d_cg_backend.cu:175-189) without materialising X, Y or Y^T.
//
// This is the exact-fp32-product path (CB_GEMM_SIMT_F32): implicit GEMM with M = changed
// pixels (device-side count), N = Cout, K = kH*kW*Cp ordered (ky,kx,ci) so that every tap is a
// contiguous channel run of the pixel-major state.  The tensor-core path lives in conv_umma.cuh.
#pragma once
#include "cb_common.cuh"

namespace cb {

constexpr int SM_BM = 64, SM_BN = 64, SM_BK = 16, SM_THREADS = 256;
constexpr int SM_APAD = 4;

template <typename T> __device__ __forceinline__ float4 load4(const T* p);
template <> __device__ __forceinline__ float4 load4<float>(const float* p) {
  return *reinterpret_cast<const float4*>(p);
}
template <> __device__ __forceinline__ float4 load4<__half>(const __half* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
template <> __device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// Wp: fp32 [Kp][CoutP] with Kp = kH*kW*Cp, k = (ky*kW+kx)*Cp + ci; CoutP = round_up(Cout,4).
template <typename T>
__global__ void __launch_bounds__(SM_THREADS)
conv_simt_kernel(const T* __restrict__ state, int Cp, const int32_t* __restrict__ idx,
                 const int32_t* __restrict__ count, const float* __restrict__ Wp,
                 const float* __restrict__ bias, T* __restrict__ out, int Op, int H, int W,
                 int Cout, int CoutP, int kH, int kW, int relu) {
  __shared__ __align__(16) float As[SM_BM][SM_BK + SM_APAD];
  __shared__ __align__(16) float Bs[SM_BK][SM_BN];
  __shared__ int s_pix[SM_BM];               // pixel index or -1
  __shared__ int s_y[SM_BM], s_x[SM_BM];

  const int n = *count;
  const int Kp = kH * kW * Cp;
  const int mtiles = (n + SM_BM - 1) / SM_BM;
  const int ntiles = (Cout + SM_BN - 1) / SM_BN;
  const int tid = threadIdx.x;
  const int tn = tid & 15, tm = tid >> 4;     // 16x16 threads, 4x4 outputs each
  const int a_row = tid >> 2, a_kc = (tid & 3) * 4;
  const int b_row = tid >> 4, b_col = (tid & 15) * 4;
  const int ph = (kH - 1) / 2, pw = (kW - 1) / 2;
  const int P = H * W;

  for (int tile = blockIdx.x; tile < mtiles * ntiles; tile += gridDim.x) {
    const int mt = tile / ntiles, nt = tile - mt * ntiles;
    const int m0 = mt * SM_BM, n0 = nt * SM_BN;
    __syncthreads();
    if (tid < SM_BM) {
      const int j = m0 + tid;
      int pix = -1, yy = 0, xx = 0;
      if (j < n) {
        pix = idx[j];
        const int p = pix % P;
        yy = p / W;
        xx = p - yy * W;
      }
      s_pix[tid] = pix;
      s_y[tid] = yy;
      s_x[tid] = xx;
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int jn = 0; jn < 4; ++jn) acc[i][jn] = 0.f;

    const int a_pix = s_pix[a_row], a_y = s_y[a_row], a_x = s_x[a_row];
    for (int k0 = 0; k0 < Kp; k0 += SM_BK) {
      // ---- gather A: one 4-element group per thread ------------------------------------
      {
        const int k = k0 + a_kc;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a_pix >= 0 && k < Kp) {
          const int tap = k / Cp, ci = k - tap * Cp;
          const int ky = tap / kW, kx = tap - ky * kW;
          const int iy = a_y + ky - ph, ix = a_x + kx - pw;
          if (iy >= 0 && iy < H && ix >= 0 && ix < W)
            v = load4<T>(state + ((long long)a_pix + (long long)(ky - ph) * W + (kx - pw)) * Cp + ci);
        }
        *reinterpret_cast<float4*>(&As[a_row][a_kc]) = v;
      }
      // ---- weights B: one float4 per thread -----------------------------------------------
      {
        const int k = k0 + b_row, co = n0 + b_col;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < Kp && co < CoutP) v = __ldg(reinterpret_cast<const float4*>(Wp + (long long)k * CoutP + co));
        *reinterpret_cast<float4*>(&Bs[b_row][b_col]) = v;
      }
      __syncthreads();
#pragma unroll
      for (int k4 = 0; k4 < SM_BK; k4 += 4) {
        float4 a[4], bv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(&As[tm * 4 + i][k4]);
#pragma unroll
        for (int q = 0; q < 4; ++q) bv[q] = *reinterpret_cast<const float4*>(&Bs[k4 + q][tn * 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float av[4] = {a[i].x, a[i].y, a[i].z, a[i].w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            acc[i][0] = fmaf(av[q], bv[q].x, acc[i][0]);
            acc[i][1] = fmaf(av[q], bv[q].y, acc[i][1]);
            acc[i][2] = fmaf(av[q], bv[q].z, acc[i][2]);
            acc[i][3] = fmaf(av[q], bv[q].w, acc[i][3]);
          }
        }
      }
      __syncthreads();
    }
    // ---- epilogue: bias, ReLU, scatter one contiguous channel run per pixel ----------------
    const int co0 = n0 + tn * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int pix = s_pix[tm * 4 + i];
      if (pix < 0) continue;
      T* o = out + (long long)pix * Op + co0;
#pragma unroll
      for (int jn = 0; jn < 4; ++jn) {
        if (co0 + jn < Cout) {
          float v = acc[i][jn] + __ldg(bias + co0 + jn);
          if (relu && v <= 0.f) v = 0.f;
          o[jn] = from_float<T>(v);
        }
      }
    }
  }
}

// weight [Cout][Cin][kH][kW] (dtype T) -> fp32 Wp[Kp][CoutP]
template <typename T>
__global__ void pack_weights_simt_kernel(const T* __restrict__ w, float* __restrict__ Wp, int Cout,
                                         int Cin, int kH, int kW, int Cp, int CoutP) {
  const long long total = (long long)kH * kW * Cp * CoutP;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % CoutP);
    const long long k = i / CoutP;
    const int ci = (int)(k % Cp);
    const int tap = (int)(k / Cp);
    const int ky = tap / kW, kx = tap - ky * kW;
    float v = 0.f;
    if (co < Cout && ci < Cin) v = to_float(w[(((long long)co * Cin + ci) * kH + ky) * kW + kx]);
    Wp[i] = v;
  }
}

}  // namespace cb
