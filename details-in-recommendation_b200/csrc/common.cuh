// Shared helpers for libdir_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "dir_b200.h"

namespace dir {

constexpr int kSMs = 148;  // B200: 2 dies x 74 SMs

extern thread_local char g_err[512];
extern std::atomic<uint64_t> g_launches;

inline int fail(int code, const char* fmt, const char* a = "") {
  snprintf(g_err, sizeof(g_err), fmt, a);
  return code;
}

// after a <<<>>> launch: count it and surface launch errors
inline int launched(const char* what, int n = 1) {
  g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return DIR_EIO;
  }
  return 0;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- device helpers ---------------------------------------------------------------------
// Streaming 16-B load that does not allocate in L1 (rows are touched once per kernel).
__device__ __forceinline__ float4 ldg_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
// Streaming 16-B store (write-once outputs).
__device__ __forceinline__ void stg_stream(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
// L2 eviction-priority policies (createpolicy) and 16-B loads / stores carrying one.
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float4 ldg_hint(const float* p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(pol));
  return r;
}
// coherent (not .nc) 16-B load with an L2 policy: for rows this kernel also writes
__device__ __forceinline__ float4 ld_hint(const float* p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(pol)
               : "memory");
  return r;
}
__device__ __forceinline__ float ldg_hint1(const float* p, uint64_t pol) {
  float r;
  asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void stg_hint(float* p, float4 v, uint64_t pol) {
  asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p),
               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol)
               : "memory");
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace dir
