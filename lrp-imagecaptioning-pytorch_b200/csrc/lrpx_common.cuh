// Shared helpers for liblrpx (sm_100a).  No torch types anywhere in this library.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/lrpx.h"

namespace lrpx {

void set_error(const char* fmt, ...);

#define LRPX_CHECK_ARG(cond, msg)                                  \
  do {                                                             \
    if (!(cond)) {                                                 \
      lrpx::set_error("%s: %s", __func__, msg);                    \
      return LRPX_E_INVALID;                                       \
    }                                                              \
  } while (0)

#define LRPX_CHECK_LAUNCH()                                                        \
  do {                                                                             \
    cudaError_t e__ = cudaGetLastError();                                          \
    if (e__ != cudaSuccess) {                                                      \
      lrpx::set_error("%s: CUDA launch failed: %s", __func__, cudaGetErrorString(e__)); \
      return LRPX_E_CUDA;                                                          \
    }                                                                              \
  } while (0)

// returns the status of a call that reports one (LRPX_OK or an error code) when it is not LRPX_OK
#define RUN(expr)                      \
  do {                                 \
    int rc__ = (expr);                 \
    if (rc__ != LRPX_OK) return rc__;  \
  } while (0)

// LRPtools/utils.py:16-18
__device__ __forceinline__ float safe_div(float num, float den) {
  return num / (den + (den == 0.f ? LRPX_Z_EPSILON : 0.f));
}
// gridTDmodel.py:757-759 / lrp_modules.py:19-20 :  z + eps*sign(z), exact zero -> eps
__device__ __forceinline__ float stab(float z) {
  float s = (z > 0.f) ? LRPX_EPSILON : ((z < 0.f) ? -LRPX_EPSILON : 0.f);
  float o = s + z;
  return o == 0.f ? LRPX_EPSILON : o;
}

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Dynamic shared memory above 48 KB needs cudaFuncSetAttribute, which applies to the CURRENT device only: set it once
// per (kernel, device).  `done` is the caller's static bit set of the devices already set up for `kernel` (devices
// from 64 on are set up on every call).
template <class Kernel>
static int ensure_smem_attr(Kernel kernel, int bytes, std::atomic<uint64_t>& done) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  const uint64_t bit = (e == cudaSuccess && dev < 64) ? (uint64_t)1 << dev : 0;
  if (bit && (done.load(std::memory_order_acquire) & bit)) return LRPX_OK;
  if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(max dynamic shared memory %d) failed: %s", bytes, cudaGetErrorString(e));
    return LRPX_E_CUDA;
  }
  done.fetch_or(bit, std::memory_order_release);
  return LRPX_OK;
}

}  // namespace lrpx
