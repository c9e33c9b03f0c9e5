// Shared host/device helpers for libgte_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "gte.h"

namespace gte {

// thread-local error text behind gte_last_error_string()
char* err_buf();
int fail(int code, const char* fmt, ...);

inline cudaStream_t as_stream(gte_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// SM count of the current device (cached per device; immutable after first query)
int sm_count();

// process-wide A/B switches behind gte_set_tuning() (defaults = the product path)
int tuning(int key);

// number of kernels launched by this library since load (diagnostic; gte_launch_count())
void note_launch();

// Opt a kernel into `bytes` of dynamic shared memory on the CURRENT device (cudaFuncAttributeMaxDynamicSharedMemorySize
// is a per-device attribute).  Remembers the largest size set per (device, kernel); thread safe.  Returns GTE_OK or the
// failure already recorded with fail().
int ensure_dynamic_smem(const void* func, size_t bytes, const char* name);

#define GTE_CHECK_ARG(cond, ...)                                  \
  do {                                                            \
    if (!(cond)) return ::gte::fail(GTE_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define GTE_CHECK_LAUNCH(name)                                                            \
  do {                                                                                    \
    ::gte::note_launch();                                                                 \
    cudaError_t e__ = cudaGetLastError();                                                 \
    if (e__ != cudaSuccess)                                                               \
      return ::gte::fail(GTE_ERR_CUDA, "%s: launch failed: %s", name, cudaGetErrorString(e__)); \
  } while (0)

#define GTE_CHECK_CUDA(call, name)                                                  \
  do {                                                                              \
    cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess)                                                         \
      return ::gte::fail(GTE_ERR_CUDA, "%s: %s", name, cudaGetErrorString(e__));    \
  } while (0)

// ---------------------------------------------------------------- device --
#ifdef __CUDACC__
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Fixed-order reduction of `nb` partial vectors: result(i) = sum_b partial[b*stride + i].
// Block = 32 outputs (threadIdx.x & 31) x RED_SLICES slices (threadIdx.x >> 5): slice s adds
// partials s, s+SLICES, ... in ascending order, then slice 0 adds the slice sums in ascending
// order.  The order depends only on nb, so results are reproducible; unlike one thread walking
// all nb partials, the loads of a block are independent and coalesced.  Valid in threads with
// (threadIdx.x >> 5) == 0.  `smem` holds RED_SLICES*32 floats.  All threads must call it.
constexpr int RED_SLICES = 32;
constexpr int RED_THREADS = RED_SLICES * 32;
__device__ __forceinline__ float reduce_partials_block(const float* __restrict__ partial, int nb, int64_t stride,
                                                       int64_t i, bool valid, float* smem) {
  const int ox = threadIdx.x & 31, sy = threadIdx.x >> 5;
  float s = 0.f;
  if (valid)
    for (int b = sy; b < nb; b += RED_SLICES) s += partial[(int64_t)b * stride + i];
  smem[sy * 32 + ox] = s;
  __syncthreads();
  float t = 0.f;
  if (sy == 0)
    for (int k = 0; k < RED_SLICES; ++k) t += smem[k * 32 + ox];
  return t;
}

// torch.argmax of one row of c >= 1 values: the first maximal index, a NaN counting as maximal (the first NaN wins)
__device__ __forceinline__ int row_argmax(const float* __restrict__ lr, int c) {
  float mx = lr[0];
  int arg = 0;
  bool nan = mx != mx;
  for (int j = 1; j < c && !nan; ++j) {
    const float v = lr[j];
    if (v != v) {
      arg = j;
      nan = true;
    } else if (v > mx) {
      mx = v;
      arg = j;
    }
  }
  return arg;
}
#endif

}  // namespace gte
