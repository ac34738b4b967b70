// Interfaces between the exact SIMT scoring path (score_simt.cu) and the tensor-core path / public
// dispatch (score_tc.cu).
#pragma once
#include "common.cuh"

namespace hals {

struct ScoreOperands {
  const float* Ua; int64_t ua_stride; const float* Ia; int64_t ia_stride; int ka;
  const float* Ut; int64_t ut_stride; const float* It; int64_t it_stride; int kt;
};

size_t score_simt_workspace_bytes(int64_t n_users, int64_t n_items, int topk);
size_t score_simt_list_workspace_bytes(int64_t n_users, int64_t n_items, int topk);
int score_extrema_simt(const ScoreOperands& O, int64_t n_users, int64_t n_items, float* extrema,
                       const int32_t* user_list, const int32_t* user_count, cudaStream_t st);
// excl_rowptr / excl_items: optional per-user exclusion CSR (global item ids, ascending per row), both NULL or both set
int score_blend_topk_simt(const ScoreOperands& O, int64_t n_users, int64_t n_items, const float* extrema,
                          float w_als, float w_tt, int topk, int32_t item_offset, int32_t* out_idx,
                          float* out_score, void* workspace, const int32_t* user_list, const int32_t* user_count,
                          const int64_t* excl_rowptr, const int32_t* excl_items, cudaStream_t st);

}  // namespace hals

int check_score_args(const float* Ua, const float* Ia, int ka, const float* Ut, const float* It, int kt,
                     int64_t n_users, int64_t n_items);
