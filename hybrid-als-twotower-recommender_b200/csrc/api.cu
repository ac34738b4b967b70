// C-ABI glue: error state, launch counter, host-side ALS planner, half-step dispatch.
#include <cmath>
#include <cstdlib>
#include <vector>

#include "als_prep.cuh"

namespace hals {
thread_local char g_last_error[512] = "";
std::atomic<int64_t> g_launch_count{0};

int als_half_step_simt(const int32_t* colidx, const float* vals, const float* src, float* dst, int k,
                       float reg, int implicit, float alpha, const float* gram,
                       const hals_als_plan* plan, float* ws, cudaStream_t st, bool nonneg, int32_t* n_capped);
int als_half_step_tc128(const int32_t* colidx, const float* vals, const float* src, int64_t n_src, float* dst,
                        float reg, const hals_als_plan* plan, float* slots, void* split_buf, cudaStream_t st);
int als_half_step_tc64(const int32_t* colidx, const float* vals, const float* src, int64_t n_src, float* dst,
                       float reg, const hals_als_plan* plan, float* slots, void* split_buf, cudaStream_t st);
int als_half_step_ws128(const int32_t* colidx, const uint32_t* vals_hl, const float* src, int64_t n_src, float* dst,
                        float reg, const hals_als_plan* plan, float* slots, void* split_buf, void* dst_hl,
                        const float* gram, float* gram_tiles, cudaStream_t st);
int als_half_step_ws64(const int32_t* colidx, const uint32_t* vals_hl, const float* src, int64_t n_src, float* dst,
                       float reg, const hals_als_plan* plan, float* slots, void* split_buf, void* dst_hl,
                       const float* gram, float* gram_tiles, cudaStream_t st);
}  // namespace hals

using namespace hals;

static int padded_rank(int k) { return k <= 16 ? 16 : k <= 32 ? 32 : k <= 64 ? 64 : 128; }

extern "C" int hals_abi_version(void) { return HALS_ABI_VERSION; }
extern "C" const char* hals_last_error(void) { return g_last_error; }
extern "C" int64_t hals_launch_count(void) { return g_launch_count.load(); }
extern "C" int hals_max_rank(void) { return 128; }

// rank 64: a slice is 256 chunks of the persistent kernel (~6 % of a CTA's share on the MovieLens-20M shape) and the
// hottest rows stay below 256 slices, i.e. one level of slot pre-sums
extern "C" int32_t hals_als_default_seg_len(int k) { return k <= 64 ? 8192 : 4096; }

static size_t slot_region_bytes(int64_t n_slots, int k) {
  const size_t KP = (size_t)padded_rank(k);
  return (size_t)(n_slots > 0 ? n_slots : 0) * (KP * KP + KP + 4) * sizeof(float);
}
// tensor-core path: ranks 64 and 128; implicit feedback when the plan carries the operands packed for this alpha (HALS_FORCE_SIMT=1 routes everything to the SIMT path)
static bool use_tc(int k, int implicit, float alpha, const hals_als_plan* plan) {
  static const bool force_simt = [] { const char* e = getenv("HALS_FORCE_SIMT"); return e && e[0] == '1'; }();
  if (force_simt) return false;
  if (!implicit) return (k == 64 || k == 128) && plan->packed_alpha == 0.f;
  return (k == 64 || k == 128) && plan->vals_hl && plan->vals_scale && plan->item_npos && plan->chunk_pos && plan->packed_alpha == alpha &&
         alpha > 0.f;
}
static size_t gram_tile_bytes(int k) {   // Y^T Y in the solver's lane-tile order (implicit feedback, ranks 64 / 128)
  return k == 128 ? 128 * 72 * sizeof(float) : k == 64 ? 32 * 72 * sizeof(float) : 0;
}

extern "C" size_t hals_als_workspace_bytes(int64_t n_slots, int k, int64_t n_src) {
  // [partial (A,b,n) slots][bf16 h|l split of the source factors, tensor-core path]
  // [partial (A,b,n) slots][bf16 h|l split of the source factors + one all-zero row][Gram tiles (implicit, rank 128)]
  return slot_region_bytes(n_slots, k) + (size_t)(n_src > 0 ? n_src : 0) * 4 * (size_t)k + 1024 + gram_tile_bytes(k);
}

// Work items: first every slice of every long row (big, uniform items first so that the
// tail of the grid is made of short rows), then the remaining non-empty rows in order.
extern "C" int hals_als_plan_count_host(const int64_t* rowptr_host, int64_t m, int32_t seg_len,
                                        int64_t* n_items, int64_t* n_long_rows, int64_t* n_slots) {
  HALS_REQUIRE(rowptr_host && n_items && n_long_rows && n_slots, "null pointer");
  HALS_REQUIRE(seg_len >= 32 && m >= 0, "seg_len must be >= 32");
  int64_t items = 0, longs = 0, slots = 0;
  for (int64_t j = 0; j < m; ++j) {
    const int64_t len = rowptr_host[j + 1] - rowptr_host[j];
    if (len < 0) return fail(HALS_ERR_INVALID, "%s: rowptr not monotone%s", __func__);
    if (len == 0) continue;
    if (len > seg_len) {
      const int64_t ns = (len + seg_len - 1) / seg_len;
      items += ns; slots += ns; ++longs;
    } else {
      ++items;
    }
  }
  *n_items = items; *n_long_rows = longs; *n_slots = slots;
  return 0;
}

extern "C" int hals_als_plan_fill_host(const int64_t* rowptr_host, int64_t m, int32_t seg_len,
                                       int32_t* item_row, int64_t* item_begin, int32_t* item_len,
                                       int32_t* item_slot, int32_t* long_row, int32_t* long_slot0,
                                       int32_t* long_nseg) {
  HALS_REQUIRE(rowptr_host && item_row && item_begin && item_len && item_slot, "null pointer");
  HALS_REQUIRE(seg_len >= 32, "seg_len must be >= 32");
  struct Item { int32_t row; int64_t begin; int32_t len; int32_t slot; };
  std::vector<Item> segs, rows;
  rows.reserve((size_t)m);
  segs.reserve((size_t)(rowptr_host[m] / seg_len + 16));
  int64_t lr = 0, slot = 0;
  for (int64_t j = 0; j < m; ++j) {
    const int64_t b = rowptr_host[j], len = rowptr_host[j + 1] - b;
    if (len == 0) continue;
    if (len <= seg_len) { rows.push_back({(int32_t)j, b, (int32_t)len, -1}); continue; }
    HALS_REQUIRE(long_row && long_slot0 && long_nseg, "null long-row arrays");
    const int64_t ns = (len + seg_len - 1) / seg_len;
    // equal slices (not seg_len + remainder) so that slice costs are uniform
    const int64_t per = (len + ns - 1) / ns;
    long_row[lr] = (int32_t)j; long_slot0[lr] = (int32_t)slot; long_nseg[lr] = (int32_t)ns; ++lr;
    for (int64_t s = 0; s < ns; ++s) {
      const int64_t o = s * per;
      const int64_t l = (o + per <= len) ? per : len - o;
      segs.push_back({(int32_t)j, b + o, (int32_t)l, (int32_t)slot});
      ++slot;
    }
  }
  // Emission order: slices (gather-heavy, nothing to solve) are spread evenly among the whole rows (solve-heavy), so
  // that any contiguous run of items -- the persistent kernels take contiguous or round-robin shares of this list --
  // mixes the two in the global proportion and the gather and solve pipes of an SM both stay busy.
  const int64_t S = (int64_t)segs.size(), R = (int64_t)rows.size();
  int64_t it = 0, si = 0, ri = 0;
  auto emit = [&](const Item& x) {
    item_row[it] = x.row; item_begin[it] = x.begin; item_len[it] = x.len; item_slot[it] = x.slot; ++it;
  };
  while (si < S || ri < R) {
    // progress fractions (si + 1/2) / S vs (ri + 1/2) / R, compared without division
    const bool take_slice = si < S && (ri >= R || (2 * si + 1) * R <= (2 * ri + 1) * S);
    if (take_slice) emit(segs[si++]); else emit(rows[ri++]);
  }
  return 0;
}

extern "C" int64_t hals_als_plan_chunk_count_host(const int32_t* item_len, int64_t n_items) {
  if (!item_len || n_items < 0) return -1;
  int64_t n = 0;
  for (int64_t i = 0; i < n_items; ++i) {
    if (item_len[i] <= 0) return -1;
    n += (item_len[i] + 31) / 32;
  }
  return n;
}

extern "C" int hals_als_plan_chunks_host(const int32_t* item_len, const int64_t* item_begin, const int32_t* item_slot,
                                         int64_t n_items, int k, int64_t* item_chunk0, int64_t* item_cost0,
                                         int64_t* chunk_pos, int32_t* chunk_cnt) {
  HALS_REQUIRE(item_len && item_begin && item_slot && item_chunk0 && item_cost0 && chunk_pos && chunk_cnt, "null pointer");
  // cost of an item in chunk units: its chunks + the solve of a whole row (rank 64: measured ~6 chunk times with the
  // solvers of an SM working in parallel; rank 128: ~8-10k cycles per system against ~300 per chunk) or the parking
  // of a slice's partial sums
  const int64_t kSolveCost = k > 64 ? 32 : 6, kParkCost = k > 64 ? 6 : 2;
  int64_t c = 0, cost = 0;
  for (int64_t i = 0; i < n_items; ++i) {
    item_chunk0[i] = c;
    item_cost0[i] = cost;
    const int32_t len = item_len[i];
    HALS_REQUIRE(len > 0, "empty work item");
    for (int32_t o = 0; o < len; o += 32) { chunk_pos[c] = item_begin[i] + o; chunk_cnt[c] = len - o; ++c; }
    cost += (len + 31) / 32 + (item_slot[i] < 0 ? kSolveCost : kParkCost);
  }
  item_chunk0[n_items] = c;
  item_cost0[n_items] = cost;
  return 0;
}

extern "C" int hals_als_split_factors(const float* src, int64_t n_rows, int k, void* out_hl, void* stream) {
  HALS_REQUIRE(k == 64 || k == 128, "split factors exist for ranks 64 and 128");
  HALS_REQUIRE(n_rows >= 0, "negative count");
  if (n_rows == 0) return 0;
  HALS_REQUIRE(src && out_hl, "null pointer");
  return als_launch_split_bf16(src, n_rows, k, out_hl, (cudaStream_t)stream);
}

// Spark's regParam validator is gtEq(0): a negative reg can make A indefinite (silent NaN or garbage factors), a NaN
// or infinite one poisons every row.  reg = 0 is accepted, as in Spark.
static const char kRegCheck[] = "reg must be finite and >= 0";

extern "C" int hals_als_half_step_split(const int32_t* colidx, int64_t m_dst, const void* src_hl, int64_t n_src,
                                        float* dst, void* dst_hl, int k, float reg, const hals_als_plan* plan,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  HALS_REQUIRE(reg >= 0.f && std::isfinite(reg), kRegCheck);
  HALS_REQUIRE(plan != nullptr, "null plan");
  HALS_REQUIRE(k == 64 || k == 128, "split-form half-steps exist for ranks 64 and 128");
  HALS_REQUIRE(m_dst >= 0 && n_src >= 0, "negative count");
  if (m_dst == 0 || plan->n_items == 0) return 0;
  HALS_REQUIRE(colidx && src_hl && dst && dst_hl, "null pointer");
  HALS_REQUIRE(plan->vals_hl && plan->chunk_pos && plan->chunk_cnt && plan->item_chunk0 && plan->item_cost0,
               "the plan must carry packed ratings and the chunk table");
  HALS_REQUIRE(workspace != nullptr, "null workspace");
  if (workspace_bytes < slot_region_bytes(plan->n_slots, k) + 16) return fail(HALS_ERR_WORKSPACE, "%s: workspace too small%s", __func__);
  // rows without ratings are never written: the caller keeps them zero (fp32 and split)
  HALS_REQUIRE(plan->packed_alpha == 0.f, "the plan's ratings are packed for implicit feedback");
  if (k == 128)
    return als_half_step_ws128(colidx, plan->vals_hl, nullptr, n_src, dst, reg, plan, (float*)workspace,
                               const_cast<void*>(src_hl), dst_hl, nullptr, nullptr, (cudaStream_t)stream);
  return als_half_step_ws64(colidx, plan->vals_hl, nullptr, n_src, dst, reg, plan, (float*)workspace,
                            const_cast<void*>(src_hl), dst_hl, nullptr, nullptr, (cudaStream_t)stream);
}

extern "C" int hals_als_pack_ratings(const float* vals, int64_t nnz, uint32_t* out, void* stream) {
  HALS_REQUIRE(nnz >= 0, "negative count");
  if (nnz == 0) return 0;
  HALS_REQUIRE(vals && out, "null pointer");
  return als_pack_ratings(vals, nnz, out, (cudaStream_t)stream);
}

extern "C" int hals_als_pack_ratings_implicit(const float* vals, int64_t nnz, float alpha, uint32_t* out_hl, float* out_scale,
                                              void* stream) {
  HALS_REQUIRE(nnz >= 0, "negative count");
  HALS_REQUIRE(alpha > 0.f, "alpha must be positive");
  if (nnz == 0) return 0;
  HALS_REQUIRE(vals && out_hl && out_scale, "null pointer");
  return als_pack_ratings_implicit(vals, nnz, alpha, out_hl, out_scale, (cudaStream_t)stream);
}

extern "C" int hals_als_plan_count_positive(const float* vals, const int64_t* item_begin, const int32_t* item_len,
                                            int64_t n_items, int32_t* item_npos, void* stream) {
  HALS_REQUIRE(n_items >= 0, "negative count");
  if (n_items == 0) return 0;
  HALS_REQUIRE(vals && item_begin && item_len && item_npos, "null pointer");
  return als_count_positive(vals, item_begin, item_len, n_items, item_npos, (cudaStream_t)stream);
}

// Body of hals_als_half_step and hals_als_half_step_nonnegative.
static int als_half_step_impl(const int32_t* colidx, const float* vals, int64_t m_dst, const float* src, int64_t n_src,
                              float* dst, int k, float reg, int implicit, float alpha, const float* gram,
                              const hals_als_plan* plan, void* workspace, size_t workspace_bytes, void* stream,
                              bool nonneg, int32_t* n_capped) {
  HALS_REQUIRE(reg >= 0.f && std::isfinite(reg), kRegCheck);
  HALS_REQUIRE(plan != nullptr, "null plan");
  HALS_REQUIRE(k >= 1 && k <= 128, "rank must be in [1,128]");
  HALS_REQUIRE(m_dst >= 0, "negative row count");
  HALS_REQUIRE(!implicit || gram != nullptr, "implicit mode needs the Gram matrix");
  cudaStream_t st = (cudaStream_t)stream;
  if (m_dst == 0) return 0;
  HALS_REQUIRE(dst != nullptr, "null dst");
  // rows without ratings are absent from the Spark model; they are kept as zero rows
  HALS_CUDA(cudaMemsetAsync(dst, 0, sizeof(float) * (size_t)m_dst * k, st));
  if (plan->n_items == 0) return 0;
  HALS_REQUIRE(colidx && vals && src, "null pointer");
  HALS_REQUIRE(plan->item_row && plan->item_begin && plan->item_len && plan->item_slot, "null plan arrays");
  HALS_REQUIRE(workspace != nullptr, "null workspace");
  if (workspace_bytes < hals_als_workspace_bytes(plan->n_slots, k, n_src))
    return fail(HALS_ERR_WORKSPACE, "%s: workspace too small%s", __func__);
  HALS_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "workspace must be 16-byte aligned");
  // the tensor-core solvers have no bound-constrained variant: nonnegative half-steps always run the CUDA-core kernels
  if (nonneg) return als_half_step_simt(colidx, vals, src, dst, k, reg, implicit, alpha, gram, plan, (float*)workspace, st,
                                        true, n_capped);
  if (use_tc(k, implicit, alpha, plan)) {
    void* split = reinterpret_cast<uint8_t*>(workspace) + slot_region_bytes(plan->n_slots, k);
    if (implicit) {
      float* tiles = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(split) + (size_t)n_src * 4 * (size_t)k + 1024);
      return k == 128 ? als_half_step_ws128(colidx, plan->vals_hl, src, n_src, dst, reg, plan, (float*)workspace, split,
                                            nullptr, gram, tiles, st)
                      : als_half_step_ws64(colidx, plan->vals_hl, src, n_src, dst, reg, plan, (float*)workspace, split,
                                           nullptr, gram, tiles, st);
    }
    if (k == 128) {
      // HALS_TC128_IMPL=groups selects the round-1 kernel (two solver groups, no chunk table)
      static const bool old128 = [] { const char* e = getenv("HALS_TC128_IMPL"); return e && e[0] == 'g'; }();
      if (old128 || plan->vals_hl == nullptr || plan->chunk_pos == nullptr)
        return als_half_step_tc128(colidx, vals, src, n_src, dst, reg, plan, (float*)workspace, split, st);
      return als_half_step_ws128(colidx, plan->vals_hl, src, n_src, dst, reg, plan, (float*)workspace, split, nullptr,
                                 nullptr, nullptr, st);
    }
    // HALS_TC64_IMPL=cta4 selects the round-1 kernel (four 4-warp CTAs per SM); default: warp-specialised kernel
    static const bool old64 = [] { const char* e = getenv("HALS_TC64_IMPL"); return e && e[0] == 'c'; }();
    if (old64 || plan->vals_hl == nullptr || plan->chunk_pos == nullptr)
      return als_half_step_tc64(colidx, vals, src, n_src, dst, reg, plan, (float*)workspace, split, st);
    return als_half_step_ws64(colidx, plan->vals_hl, src, n_src, dst, reg, plan, (float*)workspace, split, nullptr, nullptr,
                              nullptr, st);
  }
  return als_half_step_simt(colidx, vals, src, dst, k, reg, implicit, alpha, gram, plan, (float*)workspace, st, false,
                            nullptr);
}

extern "C" int hals_als_half_step(const int64_t* rowptr, const int32_t* colidx, const float* vals,
                                  int64_t m_dst, const float* src, int64_t n_src, float* dst, int k,
                                  float reg, int implicit, float alpha, const float* gram,
                                  const hals_als_plan* plan, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  (void)rowptr;
  return als_half_step_impl(colidx, vals, m_dst, src, n_src, dst, k, reg, implicit, alpha, gram, plan, workspace,
                            workspace_bytes, stream, false, nullptr);
}

extern "C" int hals_als_half_step_nonnegative(const int64_t* rowptr, const int32_t* colidx, const float* vals,
                                              int64_t m_dst, const float* src, int64_t n_src, float* dst, int k,
                                              float reg, int implicit, float alpha, const float* gram,
                                              const hals_als_plan* plan, void* workspace, size_t workspace_bytes,
                                              void* stream, int32_t* n_capped) {
  (void)rowptr;
  // A = (Gram +) sum y y^T + reg n I is positive definite only with reg > 0; the NNLS minimiser rests on it
  HALS_REQUIRE(reg > 0.f, "nonnegative half-steps need reg > 0");
  return als_half_step_impl(colidx, vals, m_dst, src, n_src, dst, k, reg, implicit, alpha, gram, plan, workspace,
                            workspace_bytes, stream, true, n_capped);
}
