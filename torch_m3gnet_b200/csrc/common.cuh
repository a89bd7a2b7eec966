// Shared device/host helpers for the m3gnet_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "m3gnet_b200.h"

namespace m3g {

void set_error(const char* fmt, ...);

#define M3G_REQUIRE(cond, ...)              \
  do {                                      \
    if (!(cond)) {                          \
      m3g::set_error(__VA_ARGS__);          \
      return M3G_ERR_INVALID;               \
    }                                       \
  } while (0)

#define M3G_LAUNCH_CHECK(name)                                                   \
  do {                                                                           \
    cudaError_t err__ = cudaGetLastError();                                      \
    if (err__ != cudaSuccess) {                                                  \
      m3g::set_error("%s: launch failed: %s", name, cudaGetErrorString(err__));  \
      return M3G_ERR_CUDA;                                                       \
    }                                                                            \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

static inline unsigned blocks_for(int64_t n, int per_block) {
  int64_t b = (n + per_block - 1) / per_block;
  if (b < 1) b = 1;
  return (unsigned)b;
}

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float sigmoidf_(float z) { return 1.0f / (1.0f + __expf(-z)); }
// accurate variants (expf) are used where the value feeds energies directly
__device__ __forceinline__ float sigmoid_acc(float z) { return 1.0f / (1.0f + expf(-z)); }
__device__ __forceinline__ float silu_acc(float z) { return z / (1.0f + expf(-z)); }
// d/dz [z*s(z)] = s (1 + z (1 - s))
__device__ __forceinline__ float silu_grad(float z) {
  float s = sigmoid_acc(z);
  return s * (1.0f + z * (1.0f - s));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// Fixed-order float64 reductions of the one-block-per-structure kernels (relax.cu, md.cu): xor butterfly in each warp,
// then the kWarps warp results in warp order; every thread gets the result.  sh holds kWarps doubles.
template <int kWarps>
__device__ __forceinline__ double block_sum(double t, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(FULL, t, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = t;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int q = 0; q < kWarps; ++q) s += sh[q];
  __syncthreads();  // sh is reused by the next reduction
  return s;
}

template <int kWarps>
__device__ __forceinline__ double block_max(double t, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_xor_sync(FULL, t, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = t;
  __syncthreads();
  double s = sh[0];
#pragma unroll
  for (int q = 1; q < kWarps; ++q) s = fmax(s, sh[q]);
  __syncthreads();
  return s;
}

// cutoff polynomial of nn/interaction.py:389-400 and its derivative w.r.t. r
__device__ __forceinline__ float cutoff_poly(float r, float r3) {
  float x = r / r3;
  if (!(x <= 1.0f)) return 0.0f;
  float x2 = x * x, x3 = x2 * x;
  return 1.0f - 6.0f * x3 * x2 + 15.0f * x2 * x2 - 10.0f * x3;
}
__device__ __forceinline__ float cutoff_poly_grad(float r, float r3) {
  float x = r / r3;
  if (!(x <= 1.0f)) return 0.0f;
  float x2 = x * x;
  // d/dx = -30 x^4 + 60 x^3 - 30 x^2
  return (-30.0f * x2 * x2 + 60.0f * x2 * x - 30.0f * x2) / r3;
}

}  // namespace m3g
