// Shared helpers for the icrl_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define ICRL_VPAD 1024        // vocabulary padded to the tensor-core tile (V = 1004 in the reference's data)
#define ICRL_H 512            // hidden / embedding / feature width (models.py:41,160,250)

// error codes returned across the C ABI (include/icrl_b200.h)
#define ICRL_OK 0
#define ICRL_ERR_ARG 1
#define ICRL_ERR_CUDA 2
#define ICRL_ERR_WATCHDOG 3

void icrl_set_error(const char* fmt, ...);

#define ICRL_CUDA(call)                                                              \
  do {                                                                               \
    cudaError_t e__ = (call);                                                        \
    if (e__ != cudaSuccess) {                                                        \
      icrl_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return ICRL_ERR_CUDA;                                                          \
    }                                                                                \
  } while (0)

#define ICRL_LAUNCH_CHECK() ICRL_CUDA(cudaGetLastError())

#define ICRL_REQUIRE(cond, msg)                                   \
  do {                                                            \
    if (!(cond)) {                                                \
      icrl_set_error("%s:%d requirement failed: %s (%s)", __FILE__, __LINE__, #cond, msg); \
      return ICRL_ERR_ARG;                                        \
    }                                                             \
  } while (0)

static inline int icrl_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// Column order of the LSTM gate gradients that the chain backward stores as fp16 pairs (chain_tc.cu, pass (S)) and the
// weight-gradient contraction and gate-table scatter read: within each block of 32 hidden units the 128 columns are
// ordered [unit quad q][gate a][unit j of the quad] instead of [gate a][unit], so that the lane that owns units
// 4q .. 4q+3 of all four gates stores one contiguous 32-byte run per plane.  natural = a * 512 + u.
__host__ __device__ __forceinline__ int icrl_gate_pair_col(int natural) {
  const int a = natural / ICRL_H, u = natural % ICRL_H;
  return 128 * (u >> 5) + 16 * ((u >> 2) & 7) + 4 * a + (u & 3);
}
__host__ __device__ __forceinline__ int icrl_gate_pair_natural(int col) {
  return ICRL_H * ((col >> 2) & 3) + 32 * (col >> 7) + 4 * ((col >> 4) & 7) + (col & 3);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
// SFU forms (MUFU.EX2 + MUFU.RCP), abs error ~1e-7 on O(1) gate values; 466 -> 180 cycles per LSTM cell on the
// serial chains (scripts/xchg_bench.cu) and 5x fewer instructions in the decode kernel's gate epilogue.
__device__ __forceinline__ float sigmoidf_sfu(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanhf_sfu(float x) { return 1.0f - 2.0f * __fdividef(1.0f, 1.0f + __expf(2.0f * x)); }
