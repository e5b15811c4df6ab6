// aware_b200 -- shared declarations for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#define AW_NFFT 1024
#define AW_HOP 256
#define AW_HALF 512
#define AW_NMEL 128
#define AW_NBITS 20
#define AW_MAX_BINS 256          // band width limit (225 bins @16 kHz, 81 @44.1 kHz)
#define AW_LEAKY 0.2f
#define AW_IN_EPS 1e-5
#define AW_ROW_TILE 128          // GEMM M tile; per-clip pooled frames are padded to this

namespace aw {

extern thread_local char g_err[512];
int set_error(const char* fmt, ...);

#define AW_CUDA(call)                                                              \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess)                                                        \
      return aw::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,           \
                           cudaGetErrorString(e__));                               \
  } while (0)

#define AW_LAUNCH_CHECK()                                                          \
  do {                                                                             \
    cudaError_t e__ = cudaGetLastError();                                          \
    if (e__ != cudaSuccess)                                                        \
      return aw::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__,       \
                           cudaGetErrorString(e__));                               \
  } while (0)

// at API entry: an error left behind by an earlier, unchecked call must not be blamed on this one
#define AW_ENTRY(name)                                                             \
  do {                                                                             \
    cudaError_t e__ = cudaGetLastError();                                          \
    if (e__ != cudaSuccess)                                                        \
      return aw::set_error("%s: CUDA error pending from an earlier call -> %s", name, \
                           cudaGetErrorString(e__));                               \
  } while (0)

#define AW_REQUIRE(cond, ...)                                                      \
  do {                                                                             \
    if (!(cond)) return aw::set_error(__VA_ARGS__);                                \
  } while (0)

// ---------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------
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
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  return v;
}

// Block-wide sum of doubles; result valid in thread 0.  `scratch` >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  double r = 0.0;
  if (w == 0) {
    r = lane < nw ? scratch[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;
}

// |v| and its sample index packed so that u64-max == (largest |v|, lowest index).
__device__ __forceinline__ unsigned long long pack_peak(float absval, unsigned idx) {
  return ((unsigned long long)__float_as_uint(absval) << 32) | (unsigned long long)(0xffffffffu - idx);
}
__device__ __forceinline__ float peak_value(unsigned long long p) {
  return __uint_as_float((unsigned)(p >> 32));
}
__device__ __forceinline__ unsigned peak_index(unsigned long long p) {
  return 0xffffffffu - (unsigned)(p & 0xffffffffu);
}

__device__ __forceinline__ float leaky(float x) { return x > 0.f ? x : AW_LEAKY * x; }

// round-to-nearest TF32 (keeps the value in a float container)
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// torch reflect padding: index i in [-512, L+512) -> [0, L)
__device__ __forceinline__ int reflect_idx(int i, int L) {
  i = i < 0 ? -i : i;
  return i >= L ? 2 * (L - 1) - i : i;
}

}  // namespace aw
