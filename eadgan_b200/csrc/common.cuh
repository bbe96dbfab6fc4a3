// Shared device/host helpers for libeadgan.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "eadgan.h"

// ---- host-side error plumbing (thread-local message, negative status) ------
int eadgan_set_error(int code, const char* fmt, ...);

#define EG_REQUIRE(cond, code, ...)                        \
  do {                                                     \
    if (!(cond)) return eadgan_set_error((code), __VA_ARGS__); \
  } while (0)

#define EG_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return eadgan_set_error(EADGAN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,          \
                              cudaGetErrorString(_e), __FILE__, __LINE__);              \
  } while (0)

void eg_count_launch();

#define EG_LAUNCH_CHECK(name)                                                           \
  do {                                                                                  \
    eg_count_launch();                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess)                                                              \
      return eadgan_set_error(EADGAN_ERR_CUDA, "launch of %s failed: %s", name,         \
                              cudaGetErrorString(_e));                                  \
  } while (0)

int eg_sm_count();

// ---- device helpers ---------------------------------------------------------
__device__ __forceinline__ float eg_ld(const void* p, int64_t i, int dtype) {
  return dtype == EADGAN_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i])
                              : reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void eg_st(void* p, int64_t i, int dtype, float v) {
  if (dtype == EADGAN_BF16)
    reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
  else
    reinterpret_cast<float*>(p)[i] = v;
}

__device__ __forceinline__ float eg_act(float v, int act, float slope) {
  switch (act) {
    case EADGAN_ACT_RELU: return v > 0.f ? v : 0.f;
    case EADGAN_ACT_LRELU: return v > 0.f ? v : v * slope;
    case EADGAN_ACT_TANH: return tanhf(v);
    case EADGAN_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    default: return v;
  }
}
// derivative of the activation expressed through its OUTPUT y
__device__ __forceinline__ float eg_act_grad(float y, int act, float slope) {
  switch (act) {
    case EADGAN_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case EADGAN_ACT_LRELU: return y > 0.f ? 1.f : slope;
    case EADGAN_ACT_TANH: return 1.f - y * y;
    case EADGAN_ACT_SIGMOID: return y * (1.f - y);
    default: return 1.f;
  }
}

__device__ __forceinline__ float eg_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double eg_warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum (blockDim.x multiple of 32, <= 1024); result valid in all threads
__device__ __forceinline__ float eg_block_sum(float v, float* smem32) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = eg_warp_sum(v);
  __syncthreads();
  if (lane == 0) smem32[wid] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  float r = (lane < nw) ? smem32[lane] : 0.f;
  r = eg_warp_sum(r);
  return r;
}
