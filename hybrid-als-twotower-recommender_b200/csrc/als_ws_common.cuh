// Front end shared by the warp-specialised ALS kernels (als_ws64.cu: rank 64, als_ws128.cu: rank 128): device
// helpers, the CTA's equal-cost share of the plan, the zeroed rating blocks and the implicit-mode scaler role.  A stage
// holds K / 32 blocks of [KC][64] bf16 (H | L) and the rating block R.  The gather roles stay per rank: a template
// on K did not reproduce the rank-64 gather's code (operand set-up and the order of its cp.async issue).
#pragma once
#include <cuda_bf16.h>

#include "als_common.cuh"
#include "als_tc_common.cuh"
#include "umma.cuh"

namespace hals {
namespace ws {

constexpr int KC = 32;                       // ratings per stage
constexpr int kRowBytes = 128;               // one 64-wide bf16 MN atom row
constexpr int kBlk = KC * kRowBytes;         // 4096: one [KC][64] block
__host__ __device__ constexpr int stage_bytes(int K) { return (K / 32 + 1) * kBlk; }   // H | L | R (rank 128: H0 | H1 | L0 | L1 | R)

#ifdef HALS_WS_PROFILE
#define WS_T0() const long long t0__ = clock64()
#define WS_ACC(v) (v) += clock64() - t0__
#else
#define WS_T0() do { } while (0)
#define WS_ACC(v) do { } while (0)
#endif

__device__ __forceinline__ void sts64_if(uint32_t pred, uint32_t addr, f32x2 p) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p st.shared.b64 [%0], %1;\n\t}\n"
               ::"r"(addr), "l"(p), "r"(pred) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* mbar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(umma::smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ bool elect_one() {   // true in exactly one lane of the (converged) warp
  uint32_t p;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ f32x2 fmul2(f32x2 a, f32x2 b) { return ffma2(a, b, 0ull); }
__device__ __forceinline__ float rcp_fast(float d) {   // pivots are >= lambda * n > 0 and never denormal
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;\n" : "=f"(r) : "f"(d));
  return r;
}
__host__ __device__ constexpr int tri(int q, int c) { return q * (q + 1) / 2 + c; }
__device__ __forceinline__ void cp_async16_raw(uint32_t smem_dst, uint64_t gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ uint32_t cvt_bf16x2(float hi, float lo) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;\n" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ f32x2 unpack_bf16x2(uint32_t w) {             // (element 0, element 1) as fp32
  return pack2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}

// This CTA's share of the plan: a contiguous range of work items (equal cost across CTAs) and of their chunks.
struct Range {
  int64_t item_lo, item_hi, chunk_lo, chunk_hi;
};

// Threads 0 and 1 of the CTA: items [lo, hi) with lo = first item whose cost prefix reaches (total * b / grid).
__device__ __forceinline__ void cta_range(Range* range, const int64_t* __restrict__ item_cost0,
                                          const int64_t* __restrict__ item_chunk0, int64_t n_items, int tid) {
  const int64_t total = item_cost0[n_items];
  const int64_t bq = (int64_t)blockIdx.x + tid;
  const int64_t target = (total * bq + gridDim.x - 1) / gridDim.x;
  int64_t lo = 0, hi = n_items;              // lower bound of `target` in item_cost0[0..n_items]
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(item_cost0 + mid) < target) lo = mid + 1; else hi = mid;
  }
  if (bq == gridDim.x) lo = n_items;
  const int64_t ck = __ldg(item_chunk0 + lo);
  if (tid == 0) { range->item_lo = lo; range->chunk_lo = ck; } else { range->item_hi = lo; range->chunk_hi = ck; }
}

// The R block (rating columns of the B operand, last block of a stage) is zero except for the 4 bytes per rating the
// gather copies in.
template <int K, int kStages, int kThreads>
__device__ __forceinline__ void zero_r_blocks(uint8_t* base, int tid) {
  for (int i = tid; i < kStages * (kBlk / 16); i += kThreads)
    *reinterpret_cast<uint4*>(base + (i / (kBlk / 16)) * stage_bytes(K) + (stage_bytes(K) - kBlk) + (i % (kBlk / 16)) * 16) =
        make_uint4(0u, 0u, 0u, 0u);
}

// The gather roles (per rank: see als_ws64.cu for the scheme) keep their column indices in a per-warp ring of
// 2 x kBurst chunks.
constexpr int kBurst = 8;
constexpr int kGatherScratch = 2 * kBurst * 32 * 4 + 2 * kBurst * 8 + 2 * kBurst * 4;   // idx ring | pos | cnt

// ---- implicit mode (Hu-Koren): rescale a landed stage in place, row t (= lane) by sqrt(c_t), c = alpha |r| ----------
// s = sqrt(c) (h + l) in fp32, re-split into bf16 hi/lo: the SAME MMAs then build sum c y y^T, and the rating column
// (which carries (1 + c) / sqrt(c) where r > 0) gives b = sum_{r>0} (1 + c) y.  The body of each kernel's
// __noinline__ scaler_role (the role functions keep their per-kernel names: ptxas lays out and schedules a kernel's
// functions differently when their names change).
template <int K, int kStages, class Bars>
__device__ __forceinline__ void scale_stages(uint32_t stages, Bars* bars, const Range* rg, int lane) {
  const int64_t k_lo = rg->chunk_lo, k_hi = rg->chunk_hi;
  const uint32_t rowo = (uint32_t)lane * kRowBytes, x = (uint32_t)(lane & 7);
  const f32x2 one2 = pack2(1.f, 1.f), mone2 = pack2(-1.f, -1.f);
  uint32_t s = 0, su = 0;
  for (int64_t k = k_lo; k < k_hi; ++k) {
    umma::mbar_wait(&bars->st_full[s], su & 1);
    const uint32_t st = stages + s * stage_bytes(K);
    const float sc = lds32(st + stage_bytes(K) - kBlk + rowo + ((7u ^ x) << 4));
    const f32x2 sc2 = pack2(sc, sc);
#pragma unroll 2
    for (int i = 0; i < K / 8; ++i) {                   // the 16-byte chunks of row t: h in blocks [0, K/64), l after
      const uint32_t off = st + (uint32_t)(i >> 3) * kBlk + rowo + ((((uint32_t)i & 7u) ^ x) << 4);
      const float4 hv = lds128(off), lv = lds128(off + (K / 64) * kBlk);
      const uint32_t hw[4] = {__float_as_uint(hv.x), __float_as_uint(hv.y), __float_as_uint(hv.z), __float_as_uint(hv.w)};
      const uint32_t lw[4] = {__float_as_uint(lv.x), __float_as_uint(lv.y), __float_as_uint(lv.z), __float_as_uint(lv.w)};
      uint32_t oh[4], ol[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const f32x2 y = ffma2(unpack_bf16x2(hw[j]), one2, unpack_bf16x2(lw[j]));
        const f32x2 v = fmul2(y, sc2);
        oh[j] = cvt_bf16x2(hi2(v), lo2(v));
        const f32x2 r = ffma2(unpack_bf16x2(oh[j]), mone2, v);
        ol[j] = cvt_bf16x2(hi2(r), lo2(r));
      }
      sts128(off, __uint_as_float(oh[0]), __uint_as_float(oh[1]), __uint_as_float(oh[2]), __uint_as_float(oh[3]));
      sts128(off + (K / 64) * kBlk, __uint_as_float(ol[0]), __uint_as_float(ol[1]), __uint_as_float(ol[2]), __uint_as_float(ol[3]));
    }
    umma::fence_proxy_async();                          // generic-proxy writes -> the tensor core's async-proxy reads
    __syncwarp();
    if (lane == 0) umma::mbar_arrive(&bars->st_scaled[s]);
    if (++s == (uint32_t)kStages) { s = 0; ++su; }
  }
}

}  // namespace ws
}  // namespace hals
