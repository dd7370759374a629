// Shared host/device helpers for the wekws_b200 C-ABI library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <initializer_list>
#include <string>

#include "../../include/wekws_b200.h"

namespace wekws {

// ---- error plumbing: thread-local message, negative status codes, no exceptions ----
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define WEKWS_CUDA_OK(expr)                                                          \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess) {                                                         \
      ::wekws::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                         __FILE__, __LINE__);                                        \
      return WEKWS_ERR_CUDA;                                                         \
    }                                                                                \
  } while (0)

#define WEKWS_REQUIRE(cond, ...)                                                     \
  do {                                                                               \
    if (!(cond)) {                                                                   \
      ::wekws::set_error(__VA_ARGS__);                                               \
      return WEKWS_ERR_INVALID;                                                      \
    }                                                                                \
  } while (0)

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
    return WEKWS_ERR_CUDA;
  }
  return WEKWS_OK;
}

int device_sm_count();

// Raises the dynamic shared-memory limit of `kernels` to `bytes` once per device.  `done` is the launcher's own
// static per-device flag array: the attribute stays set for the life of the process.
template <typename... Kernels>
int set_max_dynamic_smem_once(bool (&done)[64], int bytes, Kernels... kernels) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || done[dev]) return WEKWS_OK;
  for (const void* k : {(const void*)kernels...})
    WEKWS_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done[dev] = true;
  return WEKWS_OK;
}

// ---- device helpers ----
#ifdef __CUDACC__
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
// Wait until at most `pending` most-recently committed groups are still in flight.
__device__ __forceinline__ void cp_async_wait_pending(int pending) {
  switch (pending) {
    case 0: asm volatile("cp.async.wait_group 0;\n" ::); break;
    case 1: asm volatile("cp.async.wait_group 1;\n" ::); break;
    case 2: asm volatile("cp.async.wait_group 2;\n" ::); break;
    default: asm volatile("cp.async.wait_group 3;\n" ::); break;
  }
}
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
#endif

}  // namespace wekws
