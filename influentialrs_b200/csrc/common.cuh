// Shared helpers for the libirs_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/irs_b200.h"

namespace irs {

extern long long g_launches;   // counted by IRS_LAUNCHED(), read through irs_launch_count()

#define IRS_LAUNCHED()                                   \
  do {                                                   \
    ++::irs::g_launches;                                 \
    cudaError_t e__ = cudaGetLastError();                \
    if (e__ != cudaSuccess) return (int)e__;             \
  } while (0)

#define IRS_CUDA(call)                                   \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return (int)e__;             \
  } while (0)

// Lets `kernel` use `bytes` of dynamic shared memory on the current device.  The attribute is held per device, so the
// table of what was granted is keyed on (kernel address, device); the driver is called only to raise the limit, and
// steady-state launches make no call.  Thread-safe.
cudaError_t opt_in_smem(const void* kernel, size_t bytes);
template <typename... Args>
inline cudaError_t opt_in_smem(void (*kernel)(Args...), size_t bytes) { return opt_in_smem((const void*)kernel, bytes); }

constexpr int kNumSMs = 148;   // B200: 2 dies x 74 SMs

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 128-bit streaming load that does not pollute L1 (each gathered row is read once).
__device__ __forceinline__ float4 ld_nc_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_na_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Total order on (score desc, column asc) packed in one 64-bit key: larger key = better candidate.
// Floats are mapped to unsigned so that integer order == float order (-inf lowest; NaN never wins
// because callers replace NaN by -inf).
__host__ __device__ __forceinline__ uint32_t f32_orderable(float f) {
  uint32_t u;
#ifdef __CUDA_ARCH__
  u = __float_as_uint(f);
#else
  union { float f; uint32_t u; } c; c.f = f; u = c.u;
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float f32_from_orderable(uint32_t u) {
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ unsigned long long pack_key(float score, uint32_t col) {
  return ((unsigned long long)f32_orderable(score) << 32) | (unsigned long long)(0xffffffffu - col);
}
__host__ __device__ __forceinline__ float key_score(unsigned long long k) { return f32_from_orderable((uint32_t)(k >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_col(unsigned long long k) { return 0xffffffffu - (uint32_t)(k & 0xffffffffu); }

}  // namespace irs
