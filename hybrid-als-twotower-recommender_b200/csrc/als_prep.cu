// Kernels and launchers shared by the tensor-core ALS routes (the warp-specialised kernels als_ws64.cu / als_ws128.cu
// and the round-1 kernels als_tc.cu / als_tc128.cu): the bf16 hi|lo split of the source factors, the packed rating
// columns, the positive-rating counts of implicit mode, and the first levels of the long-row slot reduction.
#include <cuda_bf16.h>

#include "als_prep.cuh"

namespace hals {

__global__ void split_bf16_kernel(const float* __restrict__ src, int64_t n_rows, int k,
                                  __nv_bfloat16* __restrict__ out) {
  // one thread per 8 consecutive factors: writes a 16-byte h chunk and a 16-byte l chunk
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_row = k >> 3;
  if (gid >= n_rows * per_row) return;
  const int64_t row = gid / per_row;
  const int c = (int)(gid - row * per_row);
  const float4 a = *reinterpret_cast<const float4*>(src + row * k + c * 8);
  const float4 b = *reinterpret_cast<const float4*>(src + row * k + c * 8 + 4);
  const float y[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  __align__(16) __nv_bfloat16 h[8], l[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    h[i] = __float2bfloat16_rn(y[i]);
    l[i] = __float2bfloat16_rn(y[i] - __bfloat162float(h[i]));
  }
  __nv_bfloat16* o = out + row * (2 * k);
  *reinterpret_cast<uint4*>(o + c * 8) = *reinterpret_cast<const uint4*>(h);
  *reinterpret_cast<uint4*>(o + k + c * 8) = *reinterpret_cast<const uint4*>(l);
}

int als_launch_split_bf16(const float* src, int64_t n_src, int k, void* out, cudaStream_t st) {
  const int64_t nthreads = n_src * (k / 8);
  split_bf16_kernel<<<(unsigned)((nthreads + 255) / 256), 256, 0, st>>>(src, n_src, k, reinterpret_cast<__nv_bfloat16*>(out));
  HALS_LAUNCH_CHECK();
  return 0;
}

__global__ void pack_ratings_kernel(const float* __restrict__ vals, int64_t nnz, uint32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const float r = vals[i];
  const __nv_bfloat16 rh = __float2bfloat16_rn(r);
  const __nv_bfloat16 rl = __float2bfloat16_rn(r - __bfloat162float(rh));
  out[i] = (uint32_t)__bfloat16_as_ushort(rh) | ((uint32_t)__bfloat16_as_ushort(rl) << 16);
}

int als_pack_ratings(const float* vals, int64_t nnz, uint32_t* out, cudaStream_t st) {
  pack_ratings_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(vals, nnz, out);
  HALS_LAUNCH_CHECK();
  return 0;
}

// Implicit feedback (Hu-Koren, c = alpha |r|): the tensor-core kernel rescales gathered rows by sqrt(c) and takes the
// right-hand side from a rating column that holds (1 + c) / sqrt(c) where r > 0 and 0 elsewhere:
//   sum (sqrt(c) y)(sqrt(c) y)^T = sum c y y^T,   sum (sqrt(c) y) (1 + c) / sqrt(c) = sum_{r>0} (1 + c) y.
__global__ void pack_ratings_implicit_kernel(const float* __restrict__ vals, int64_t nnz, float alpha,
                                             uint32_t* __restrict__ out_hl, float* __restrict__ out_scale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const float r = vals[i];
  const float c = alpha * fabsf(r);
  const float sc = sqrtf(c);
  const float rho = r > 0.f && c > 0.f ? (1.f + c) / sc : 0.f;
  const __nv_bfloat16 rh = __float2bfloat16_rn(rho);
  const __nv_bfloat16 rl = __float2bfloat16_rn(rho - __bfloat162float(rh));
  out_hl[i] = (uint32_t)__bfloat16_as_ushort(rh) | ((uint32_t)__bfloat16_as_ushort(rl) << 16);
  out_scale[i] = sc;
}

int als_pack_ratings_implicit(const float* vals, int64_t nnz, float alpha, uint32_t* out_hl, float* out_scale, cudaStream_t st) {
  pack_ratings_implicit_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(vals, nnz, alpha, out_hl, out_scale);
  HALS_LAUNCH_CHECK();
  return 0;
}

// ratings > 0 of every work item (one warp per item): the n of Spark's lambda * n in implicit mode
__global__ void count_positive_kernel(const float* __restrict__ vals, const int64_t* __restrict__ item_begin,
                                      const int32_t* __restrict__ item_len, int64_t n_items, int32_t* __restrict__ out) {
  const int64_t it = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (it >= n_items) return;
  const int64_t b = item_begin[it];
  const int len = item_len[it];
  int n = 0;
  for (int t = lane; t < len; t += 32) n += vals[b + t] > 0.f;
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if (lane == 0) out[it] = n;
}

int als_count_positive(const float* vals, const int64_t* item_begin, const int32_t* item_len, int64_t n_items, int32_t* out,
                       cudaStream_t st) {
  count_positive_kernel<<<(unsigned)((n_items * 32 + 255) / 256), 256, 0, st>>>(vals, item_begin, item_len, n_items, out);
  HALS_LAUNCH_CHECK();
  return 0;
}

// Long rows, level 1 of the deterministic slot reduction: groups of kSlotGroup consecutive slots of one row
// are summed (fixed order) into the group's first slot; a Zipf-head row with hundreds of slices would otherwise
// be summed by a single CTA.  grid = (n_long_rows, ceil(max_nseg / kSlotGroup)).
// `stride` = distance between the partial sums of this level (1: raw slots, 16: the level-1 group leaders).
__global__ void __launch_bounds__(256)
als_slot_group_sum_kernel(float* __restrict__ workspace, const int32_t* __restrict__ long_slot0,
                          const int32_t* __restrict__ long_nseg, int slot_floats, int stride) {
  const int ns = long_nseg[blockIdx.x];
  const int span = kSlotGroup * stride;                 // slots covered by one group of this level
  const int g0 = blockIdx.y * span;
  if (g0 >= ns || ns <= stride * kSlotGroup) return;    // this row does not need this level
  const int g1 = min(ns, g0 + span);
  float* base = workspace + (size_t)(long_slot0[blockIdx.x] + g0) * slot_floats;
  for (int e = threadIdx.x; e < slot_floats; e += 256) {
    float s = base[e];
    for (int q = stride; q < g1 - g0; q += stride) s += base[(size_t)q * slot_floats + e];
    base[e] = s;
  }
}

int als_launch_slot_group_sum(float* slots, const hals_als_plan* plan, int slot_floats, cudaStream_t st) {
  // level 1: groups of 16 slices; level 2 (rows with more than 256 slices): groups of 16 level-1 leaders
  for (int stride = 1; stride <= kSlotGroup; stride *= kSlotGroup) {
    if (plan->max_nseg <= stride * kSlotGroup) break;
    const int span = stride * kSlotGroup;
    // rows sorted by slice count (csr.py): only the first n_long_gt16 / n_long_gt256 need this level
    const int64_t hint = stride == 1 ? plan->n_long_gt16 : plan->n_long_gt256;
    const int64_t rows = hint > 0 && hint < plan->n_long_rows ? hint : plan->n_long_rows;
    dim3 g((unsigned)rows, (unsigned)((plan->max_nseg + span - 1) / span));
    als_slot_group_sum_kernel<<<g, 256, 0, st>>>(slots, plan->long_slot0, plan->long_nseg, slot_floats, stride);
    HALS_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace hals
