// Fixed-order reduction of per-CTA parameter-gradient partials, shared by the aggregation kernels (spmm.cu,
// spmm_max.cuh) and the attention softmax (edge_softmax.cu).  Internal linkage: every translation unit that includes
// this header gets its own copy.
#pragma once
#include "common.cuh"

namespace stag {

// Reduce per-CTA parameter-gradient partials in CTA order (deterministic).
static __global__ void param_finalize_kernel(const float* __restrict__ partial, int ncta, int D8, int D, int scalar,
                                             float* __restrict__ dp0, float* __restrict__ dp1) {
  __shared__ float red[2][256];
  const int tid = threadIdx.x;
  if (!scalar) {
    const int c = blockIdx.x * blockDim.x + tid;
    if (c >= D) return;
    float a = 0.f, b = 0.f;
    for (int k = 0; k < ncta; ++k) {
      a += partial[(size_t)k * 2 * D8 + c];
      b += partial[(size_t)k * 2 * D8 + D8 + c];
    }
    dp0[c] = a;
    dp1[c] = b;
  } else {
    float a = 0.f, b = 0.f;
    for (int c = tid; c < D; c += blockDim.x) {
      for (int k = 0; k < ncta; ++k) {
        a += partial[(size_t)k * 2 * D8 + c];
        b += partial[(size_t)k * 2 * D8 + D8 + c];
      }
    }
    red[0][tid] = a;
    red[1][tid] = b;
    __syncthreads();
    for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
      if (tid < o) {
        red[0][tid] += red[0][tid + o];
        red[1][tid] += red[1][tid + o];
      }
      __syncthreads();
    }
    if (tid == 0) {
      dp0[0] = red[0][0];
      dp1[0] = red[1][0];
    }
  }
}

}  // namespace stag
