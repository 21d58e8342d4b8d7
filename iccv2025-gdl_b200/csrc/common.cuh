// common.cuh — shared host/device helpers for the gdl_b200 C-ABI library.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/gdl_b200.h"

namespace gdl {

void set_last_error(const char* msg);
int cuda_fail(cudaError_t e, const char* where);

#define GDL_CHECK_LAUNCH(where)                         \
  do {                                                  \
    cudaError_t e__ = cudaGetLastError();               \
    if (e__ != cudaSuccess) return gdl::cuda_fail(e__, where); \
  } while (0)

#define GDL_REQUIRE(cond, msg)        \
  do {                                \
    if (!(cond)) {                    \
      gdl::set_last_error(msg);       \
      return GDL_EINVAL;              \
    }                                 \
  } while (0)

typedef __nv_bfloat16 bf16;

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

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

// 8 bf16 <-> 8 floats through one 16-byte vector.
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return u;
}
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// Same, but allocating in L1 (neighbouring threads re-read the line).  volatile: a batch of these stays a batch
// (the compiler does not sink each load to its first use), which is what puts several requests in flight.
__device__ __forceinline__ uint4 ld_keep16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ uint2 ld_keep8(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// 32-byte (256-bit) global accesses (sm_100: LDG/STG.256): one full sector per lane, half the memory
// instructions of 16-byte vectors for thread-per-row access patterns.  p must be 32-byte aligned.
struct U32B {
  uint4 lo, hi;
};
__device__ __forceinline__ U32B ld_stream32(const void* p) {
  U32B r;
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r.lo.x), "=r"(r.lo.y), "=r"(r.lo.z), "=r"(r.lo.w), "=r"(r.hi.x), "=r"(r.hi.y), "=r"(r.hi.z),
                 "=r"(r.hi.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_global32(void* p, const uint4& lo, const uint4& hi) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(lo.x), "r"(lo.y), "r"(lo.z),
               "r"(lo.w), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w)
               : "memory");
}

static const int kNumSMs = 148;

// gdl_set_sweep() hint (elementwise.cu): non-zero = walk pixel ranges in descending order
extern thread_local int g_sweep_rev;

}  // namespace gdl
