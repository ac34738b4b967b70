// Device helpers shared by the tensor-core ALS kernels (als_tc.cu / als_ws64.cu: rank 64, als_tc128.cu / als_ws128.cu:
// rank 128).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include "als_prep.cuh"
#include "common.cuh"

namespace hals {

// Explicit shared-state-space accesses on 32-bit addresses: keeps the solver on LDS/STS (pointer
// arithmetic through uintptr_t otherwise degrades to generic LD/ST) and halves address registers.
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];\n" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};\n" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, float a) {
  asm volatile("st.shared.f32 [%0], %1;\n" ::"r"(addr), "f"(a) : "memory");
}

// Packed fp32x2 arithmetic (sm_100 FFMA2): two row elements per 64-bit register, one instruction.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};\n" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float lo2(f32x2 v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float hi2(f32x2 v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) {   // a * b + c, both halves
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;\n" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ void lds128x2(uint32_t addr, f32x2& p0, f32x2& p1) {
  asm volatile("ld.shared.v2.b64 {%0,%1}, [%2];\n" : "=l"(p0), "=l"(p1) : "r"(addr));
}
__device__ __forceinline__ f32x2 lds64x2(uint32_t addr) {
  f32x2 p;
  asm volatile("ld.shared.b64 %0, [%1];\n" : "=l"(p) : "r"(addr));
  return p;
}
__device__ __forceinline__ void sts128x2(uint32_t addr, f32x2 p0, f32x2 p1) {
  asm volatile("st.shared.v2.b64 [%0], {%1,%2};\n" ::"r"(addr), "l"(p0), "l"(p1) : "memory");
}

// Predicated (branch-free) shared stores, pred = any non-zero word: the pivot owner publishes without diverging its
// warp, and a role bit tests with one instruction.
__device__ __forceinline__ void sts128x2_if(uint32_t pred, uint32_t addr, f32x2 p0, f32x2 p1) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %3, 0;\n\t@p st.shared.v2.b64 [%0], {%1,%2};\n\t}\n"
               ::"r"(addr), "l"(p0), "l"(p1), "r"(pred) : "memory");
}
__device__ __forceinline__ void sts32_if(uint32_t pred, uint32_t addr, float a) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p st.shared.f32 [%0], %1;\n\t}\n"
               ::"r"(addr), "f"(a), "r"(pred) : "memory");
}

// Named barriers: 1 = the two solver warps, 2 = the two producer warps (0 is __syncthreads).
__device__ __forceinline__ void bar_sync_64(int id) { asm volatile("bar.sync %0, 64;\n" ::"r"(id) : "memory"); }


__device__ __forceinline__ void bar_arrive_n(int id, int nthreads) {   // non-blocking participation
  asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void bar_sync_n(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}

// the rank-128 long-row reduce + solve (als_tc128.cu), also the tail of als_ws128.cu
int als_launch_reduce_solve128(const float* slots, float* dst, float reg, const hals_als_plan* plan, void* dst_hl,
                               const float* gram, cudaStream_t st);

}  // namespace hals
