// Shared helpers for libmmb_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "mmb_b200.h"

namespace mmb {

// Thread-local last-error text behind mmb_last_error().
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
int sm_count();

#define MMB_CUDA(call)                                           \
  do {                                                           \
    cudaError_t e__ = (call);                                    \
    if (e__ != cudaSuccess) return ::mmb::cuda_fail(e__, #call); \
  } while (0)

// Every kernel launch of the library passes through MMB_LAUNCH_CHECK (or calls count_launch()
// itself): the launch counter behind mmb_launch_count() is how bench.py COUNTS `gpu_launches`
// instead of asserting a constant.
void count_launch(const char* name);
void note_kernel(int tag, const char* name);

#define MMB_LAUNCH_CHECK(name)                                    \
  do {                                                            \
    cudaError_t e__ = cudaGetLastError();                         \
    if (e__ != cudaSuccess) return ::mmb::cuda_fail(e__, name);   \
    ::mmb::count_launch(name);                                    \
  } while (0)

#define MMB_REQUIRE(cond, msg)             \
  do {                                     \
    if (!(cond)) {                         \
      ::mmb::set_error("%s: %s", __func__, msg); \
      return MMB_E_INVALID;                \
    }                                      \
  } while (0)

static inline cudaStream_t as_stream(mmb_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

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

// Streaming (evict-first) global accesses for data touched exactly once.
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float4* p, float4 v) { __stcs(p, v); }

// ---- shared-memory barriers and bulk async copies (sm_90+ PTX) ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace mmb
