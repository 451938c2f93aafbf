// Shared helpers for libteco.so (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/teco.h"

void teco_set_error(const char* fmt, ...);

#define TECO_CHECK_ARG(cond, ...)                 \
  do {                                            \
    if (!(cond)) {                                \
      teco_set_error(__VA_ARGS__);                \
      return TECO_E_INVALID;                      \
    }                                             \
  } while (0)

#define TECO_CUDA_LAUNCH_CHECK(name)                                              \
  do {                                                                            \
    cudaError_t e__ = cudaGetLastError();                                         \
    if (e__ != cudaSuccess) {                                                     \
      teco_set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__)); \
      return TECO_E_CUDA;                                                         \
    }                                                                             \
  } while (0)

#define TECO_CUDA_CALL(expr)                                                       \
  do {                                                                             \
    cudaError_t e__ = (expr);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      teco_set_error("%s failed: %s", #expr, cudaGetErrorString(e__));             \
      return TECO_E_CUDA;                                                          \
    }                                                                              \
  } while (0)

static inline int teco_ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// TMA tensor map over bf16 data with SWIZZLE_128B, 128-byte L2 promotion and zero fill out of bounds (TF 'SAME' padding
// of the convolutions).  dims[0] is the contiguous dimension; strides[i] is the byte stride of dims[i + 1].  On failure
// sets the error message, prefixed with `who`, and returns TECO_E_CUDA.
int teco_tmap_bf16(CUtensorMap* map, const char* who, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                   const cuuint32_t* box);
// The common case: NHWC [N][H][W][C] bf16, box = box_c channels x box_w pixels x box_h rows of one image.
int teco_tmap_nhwc(CUtensorMap* map, const char* who, const void* base, int N, int H, int W, int C, int box_c, int box_w, int box_h);

__device__ __forceinline__ float teco_act(float v, int act) {
  switch (act) {
    case TECO_ACT_RELU: return fmaxf(v, 0.f);
    case TECO_ACT_LRELU02: return v >= 0.f ? v : 0.2f * v;
    case TECO_ACT_TANH24: return tanhf(v) * 24.0f;
    case TECO_ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
    default: return v;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum for blockDim.x <= 1024 (multiple of 32); result valid in thread 0.
__device__ __forceinline__ float block_sum(float v, float* smem32) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) smem32[wid] = v;
  __syncthreads();
  float r = 0.f;
  if (wid == 0) {
    int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? smem32[lane] : 0.f;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;
}

int teco_sm_count();
