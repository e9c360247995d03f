// staged.cuh -- the reference's unfused ops in its own planar layout (op-level drop-ins used by
// cbinfer_b200/conv2d_cg.py and the parity tests): genXMatrix, matrixMult, updateOutput.
#pragma once
#include "cb_common.cuh"

namespace cb {

// genXMatrix_kernel (reference cbconv2d_cg_backend.cu:138-161):
// X[j,(ci*kH+ky)*kW+kx] = in[ci, y_j+ky-(kH-1)/2, x_j+kx-(kW-1)/2] or 0 outside.
// Thread per (j, ci, ky, kx) element: writes are fully coalesced along the X row.
template <typename T>
__global__ void gen_xmatrix_kernel(T* __restrict__ cols, const T* __restrict__ in,
                                   const int32_t* __restrict__ idx, int kW, int kH, int C, int W,
                                   int H, int n) {
  const long long K = (long long)C * kH * kW;
  const long long total = K * n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i / K);
    int k = (int)(i - (long long)j * K);
    const int kx = k % kW; k /= kW;
    const int ky = k % kH;
    const int ci = k / kH;
    const int pos = idx[j];
    const int ix = pos % W + kx - (kW - 1) / 2;
    const int iy = pos / W + ky - (kH - 1) / 2;
    T v = from_float<T>(0.f);
    if (ix >= 0 && ix < W && iy >= 0 && iy < H) v = in[((long long)ci * H + iy) * W + ix];
    cols[i] = v;
  }
}

// matrixMult_python (conv2d_cg.py:342-349): Y[n,Cout] = X[n,K] . W[Cout,K]^T + bias, fp32
// accumulation.  32x32 tiles, 256 threads, 2x2 outputs per thread... kept simple: this staged op
// exists for API parity; the hot path is the fused kernel.
template <typename T>
__global__ void __launch_bounds__(256)
matrix_mult_kernel(const T* __restrict__ X, const T* __restrict__ Wt, const T* __restrict__ bias,
                   T* __restrict__ Y, int n, int K, int Cout) {
  __shared__ float Xs[32][33], Ws[32][33];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  for (int k0 = 0; k0 < K; k0 += 32) {
    for (int e = threadIdx.x; e < 1024; e += 256) {
      const int r = e >> 5, c = e & 31;
      Xs[r][c] = (m0 + r < n && k0 + c < K) ? to_float(X[(long long)(m0 + r) * K + k0 + c]) : 0.f;
      Ws[r][c] = (n0 + r < Cout && k0 + c < K) ? to_float(Wt[(long long)(n0 + r) * K + k0 + c]) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < 32; ++kk) {
      const float a0 = Xs[ty * 2][kk], a1 = Xs[ty * 2 + 1][kk];
      const float b0 = Ws[tx * 2][kk], b1 = Ws[tx * 2 + 1][kk];
      acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
      acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int m = m0 + ty * 2 + i, c = n0 + tx * 2 + j;
      if (m < n && c < Cout) Y[(long long)m * Cout + c] = from_float<T>(acc[i][j] + to_float(bias[c]));
    }
}

// updateOutput_kernel (reference cbconv2d_cg_backend.cu:175-189), Yt is [Cout, n]:
// out[co*HW + idx[j]] = (relu && v <= 0) ? 0 : v
template <typename T>
__global__ void update_output_kernel(const T* __restrict__ Yt, T* __restrict__ out,
                                     const int32_t* __restrict__ idx, int HW, int n, int Cout,
                                     int relu) {
  const long long total = (long long)n * Cout;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i / n), j = (int)(i - (long long)co * n);
    T v = Yt[i];
    if (relu && to_float(v) <= 0.f) v = from_float<T>(0.f);
    out[(long long)co * HW + idx[j]] = v;
  }
}

}  // namespace cb
