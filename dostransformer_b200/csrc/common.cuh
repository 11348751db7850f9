// Shared helpers for libdost_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include "../../include/dost.h"

namespace dost {

constexpr int kNumSMs = 148;  // B200 (grid-size heuristics; persistent kernels query sm_count())

// SM count of the current device (cached per device index).
inline int sm_count() {
  static int cached[64] = {};
  int d = 0;
  cudaGetDevice(&d);
  d &= 63;
  if (cached[d] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d) != cudaSuccess || n <= 0) n = kNumSMs;
    cached[d] = n;
  }
  return cached[d];
}

// cudaFuncSetAttribute is per device: one flag per (kernel instantiation, device).  Usage:
//   static PerDevice cfg; if (bool* f = cfg.pending()) { ...set attribute...; *f = true; }
struct PerDevice {
  bool done[64] = {};
  bool* pending() {
    int d = 0;
    cudaGetDevice(&d);
    d &= 63;
    return done[d] ? nullptr : &done[d];
  }
};

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
// Device-visible error words (mapped host memory; nullptr until dost_device_errors_init): word i <-> bit (1 << i) of
// dost_device_errors().  Kernels raise a flag with `if (errw) errw[kErrIndexRange] = 1u;`.
constexpr int kDevErrWords = 8;
constexpr int kErrIndexRange = 0, kErrNmaxTooSmall = 1;
unsigned int* device_error_words();

inline int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("%s: %s", what, cudaGetErrorString(e));
    return DOST_ERR_LAUNCH;
  }
  count_launch();
  return DOST_OK;
}

#define DOST_REQUIRE(cond, ...)        \
  do {                                 \
    if (!(cond)) {                     \
      dost::set_error(__VA_ARGS__);    \
      return DOST_ERR_ARG;             \
    }                                  \
  } while (0)

template <typename T> struct VecOf;
template <> struct VecOf<float> { using type = float4; static constexpr int N = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int N = 2; };

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

// Counter-based Bernoulli keep mask shared by the attention kernels (forward and backward regenerate the
// same bits from (seed, linear index)).  splitmix64 finaliser.
__device__ __forceinline__ bool keep_mask(unsigned long long seed, unsigned long long idx, unsigned int thresh) {
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (idx + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return static_cast<unsigned int>(z >> 32) >= thresh;  // P(keep) = 1 - thresh / 2^32
}
// The seed a kernel hands to keep_mask: the launch's seed plus the optional device word seed_offset (dost.h), read once
// per thread before any loop.  A replayed CUDA graph keeps its launch arguments, so the host rewrites that word instead.
__device__ __forceinline__ unsigned long long mask_seed(unsigned long long seed, const unsigned long long* seed_offset) {
  return seed_offset ? seed + *seed_offset : seed;
}
inline unsigned int drop_threshold(double p) {
  double t = p * 4294967296.0;
  if (t < 0) t = 0;
  if (t > 4294967295.0) t = 4294967295.0;
  return static_cast<unsigned int>(t);
}

__host__ __device__ inline long long min64(long long a, long long b) { return a < b ? a : b; }
__host__ __device__ inline long long max64(long long a, long long b) { return a > b ? a : b; }
inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

}  // namespace dost
