// Kernels and launchers of als_prep.cu, shared by the tensor-core ALS routes and called from the C ABI (api.cu).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include "common.cuh"

namespace hals {

// fp32 [n][k] -> bf16 [n][h(k) | l(k)], h = bf16(y), l = bf16(y - h)
__global__ void split_bf16_kernel(const float* __restrict__ src, int64_t n_rows, int k, __nv_bfloat16* __restrict__ out);
int als_launch_split_bf16(const float* src, int64_t n_src, int k, void* out, cudaStream_t st);
int als_pack_ratings(const float* vals, int64_t nnz, uint32_t* out, cudaStream_t st);
int als_pack_ratings_implicit(const float* vals, int64_t nnz, float alpha, uint32_t* out_hl, float* out_scale, cudaStream_t st);
int als_count_positive(const float* vals, const int64_t* item_begin, const int32_t* item_len, int64_t n_items, int32_t* out,
                       cudaStream_t st);

// Long rows: every slice parks its partial (A, b, n) in a workspace slot.  Rows of more than kSlotGroup slices are
// pre-summed in groups of kSlotGroup consecutive slots (fixed order, into the group's first slot), rows of more than
// kSlotGroup^2 slices once more over the level-1 group leaders (als_launch_slot_group_sum); a reduce kernel then adds
// the partial sums that are left, every slot_final_stride(ns)-th slot, in slot order.
constexpr int kSlotGroup = 16;
__host__ __device__ inline int slot_final_stride(int ns) {
  return ns > kSlotGroup * kSlotGroup ? kSlotGroup * kSlotGroup : ns > kSlotGroup ? kSlotGroup : 1;
}
int als_launch_slot_group_sum(float* slots, const hals_als_plan* plan, int slot_floats, cudaStream_t st);

}  // namespace hals
