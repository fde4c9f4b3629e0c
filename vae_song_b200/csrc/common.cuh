// common.cuh -- shared helpers for libb200vae (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "b200vae.h"

namespace b200vae {

constexpr float kSlope = 0.2f;       // module.py:122 LeakyReLU(0.2)
constexpr float kClampMin = 1e-2f;   // module.py:114

extern int g_last_cuda_error;
extern long long g_launch_count;

inline int check_launch() {
  ++g_launch_count;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return B200VAE_ECUDA;
  }
  return B200VAE_OK;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

int sm_count();

// ---- device helpers -------------------------------------------------------------------------------
__device__ __forceinline__ float slope_of(float h) { return h > 0.f ? 1.f : kSlope; }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace b200vae
