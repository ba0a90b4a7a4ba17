// Shared helpers for libac_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "../../include/ac_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libac_b200 targets sm_100a (B200) only"
#endif

namespace ac {

extern thread_local int g_last_cuda_error;
extern unsigned long long g_kernel_launches;   // kernels launched by this library (bench.py reports it)

inline int cuda_fail(cudaError_t e) {
  g_last_cuda_error = (int)e;
  return AC_ERR_CUDA;
}

#define AC_CUDA(expr)                                   \
  do {                                                  \
    cudaError_t _e = (expr);                            \
    if (_e != cudaSuccess) return ::ac::cuda_fail(_e);  \
  } while (0)

#define AC_LAUNCH_CHECK()                                        \
  do {                                                           \
    __atomic_fetch_add(&::ac::g_kernel_launches, 1ull, __ATOMIC_RELAXED); \
    AC_CUDA(cudaGetLastError());                                 \
  } while (0)

// 0 when the current device is CC 10.x.
int check_device();

__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// adaptive_avg_pool1d window of output index d for Lin -> Lout (ATen start/end index formulas)
__host__ __device__ inline int pool_start(int d, int Lin, int Lout) {
  return (int)(((int64_t)d * Lin) / Lout);
}
__host__ __device__ inline int pool_end(int d, int Lin, int Lout) {
  return (int)((((int64_t)d + 1) * Lin + Lout - 1) / Lout);
}

// Ownership of the unordered pair {i, j} of N images in the symmetric distance form: the image that sees the other one
// within the next floor((N-1)/2) positions of the circular order (ties at N/2 go to the smaller index).
__host__ __device__ inline bool pair_owned(int i, int j, int N) {
  int d = j - i;
  if (d < 0) d += N;
  if (d == 0) return false;
  if (2 * d < N) return true;
  if (2 * d == N) return i < j;
  return false;
}

// Ownership when images [n_old, N) join images [0, n_old) whose pairs are already known (ac_min_dist_sym_grow): a new
// image owns every pair with an old one, two new images follow pair_owned among the new images, and a pair of two old
// images has no owner.  n_old = 0 is pair_owned.
__host__ __device__ inline bool pair_owned_grow(int n_old, int i, int j, int N) {
  if (i < n_old) return false;
  if (j < n_old) return true;
  return pair_owned(i - n_old, j - n_old, N - n_old);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace ac
