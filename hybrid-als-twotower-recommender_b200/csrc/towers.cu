// Two-tower forward (tower precompute).  Replaces the Keras graph of
// src/two_tower_model.py:38-89 evaluated by Model.predict at src/two_tower_model.py:145.
// The reference recomputes the (user-independent) item tower for every user and gathers
// the same user row |items| times (two_tower_model.py:139); here each tower is evaluated
// once per id and the result feeds the scoring GEMM.
//   one warp per output row; Dense weights staged once per CTA in shared memory;
//   LayerNormalization with Keras defaults (biased variance, eps inside the sqrt).
#include "tower_common.cuh"

namespace hals {

__global__ void __launch_bounds__(kTowerThreads)
tower_user_kernel(hals_tower_weights w, const int32_t* __restrict__ ids, int64_t n, float* __restrict__ out,
                  int64_t out_stride) {
  const int lane = threadIdx.x & 31;
  const int E = w.embedding_size;
  const int64_t warps = (int64_t)gridDim.x * (kTowerThreads / 32);
  for (int64_t r = (int64_t)blockIdx.x * (kTowerThreads / 32) + (threadIdx.x >> 5); r < n; r += warps) {
    const int id = ids[r];
    const bool ok = in_table(id, w.num_users);            // out-of-range id: zero embedding, no out-of-bounds read
    const float* e = w.user_emb + (int64_t)(ok ? id : 0) * E;
    const float v0 = (ok && lane < E) ? e[lane] : 0.f;
    const float v1 = (ok && lane + 32 < E) ? e[lane + 32] : 0.f;
    warp_layer_norm_store(v0, v1, E, lane, w.user_ln_g, w.user_ln_b, w.ln_eps, out + r * out_stride);
  }
}

__global__ void __launch_bounds__(kTowerThreads)
tower_item_kernel(hals_tower_weights w, const int32_t* __restrict__ item_ids, const int32_t* __restrict__ manu_ids,
                  const int32_t* __restrict__ cat_ids, const float* __restrict__ numeric, int64_t n,
                  float* __restrict__ out, int64_t out_stride) {
  extern __shared__ float sm[];
  const int E = w.embedding_size, MD = w.manu_dim, CD = w.cat_dim, H = w.num_hidden;
  const int C = E + MD + CD + H;          // concat width (82 in the reference)
  float* Wo = sm;                         // [C][E]
  float* cc = Wo + C * E;                 // per-warp concat vectors [8][C]
  for (int e = threadIdx.x; e < C * E; e += kTowerThreads) Wo[e] = w.out_w[e];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* c = cc + warp * C;
  const int64_t warps = (int64_t)gridDim.x * (kTowerThreads / 32);
  for (int64_t r = (int64_t)blockIdx.x * (kTowerThreads / 32) + warp; r < n; r += warps) {
    const int ii = item_ids[r], mi = manu_ids[r], ci = cat_ids[r];
    const bool oki = in_table(ii, w.num_items), okm = in_table(mi, w.num_manufacturers), okc = in_table(ci, w.num_categories);
    const float* ei = w.item_emb + (int64_t)(oki ? ii : 0) * E;
    const float* em = w.manu_emb + (int64_t)(okm ? mi : 0) * MD;
    const float* ec = w.cat_emb + (int64_t)(okc ? ci : 0) * CD;
    // MinMaxScaler.transform on (price, average_review_rating): x*scale_ + min_
    const float x0 = fmaf(numeric[r * 2 + 0], w.num_scale[0], w.num_offset[0]);
    const float x1 = fmaf(numeric[r * 2 + 1], w.num_scale[1], w.num_offset[1]);
    for (int f = lane; f < C; f += 32) {
      float v;
      if (f < E) v = oki ? ei[f] : 0.f;
      else if (f < E + MD) v = okm ? em[f - E] : 0.f;
      else if (f < E + MD + CD) v = okc ? ec[f - E - MD] : 0.f;
      else {
        const int h = f - E - MD - CD;    // Dense(16, relu) on the two numerics
        v = fmaxf(fmaf(x1, w.num_w[H + h], fmaf(x0, w.num_w[h], w.num_b[h])), 0.f);
      }
      c[f] = v;
    }
    __syncwarp();
    float z0 = lane < E ? w.out_b[lane] : 0.f;
    float z1 = lane + 32 < E ? w.out_b[lane + 32] : 0.f;
    for (int f = 0; f < C; ++f) {
      const float cf = c[f];
      if (lane < E) z0 = fmaf(cf, Wo[f * E + lane], z0);
      if (lane + 32 < E) z1 = fmaf(cf, Wo[f * E + lane + 32], z1);
    }
    warp_layer_norm_store(z0, z1, E, lane, w.item_ln_g, w.item_ln_b, w.ln_eps, out + r * out_stride);
    __syncwarp();
  }
}

static int tower_blocks(int64_t n) {
  int64_t b = (n + 7) / 8;
  const int64_t cap = 8 * (int64_t)sm_count();
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace hals

using namespace hals;

static int check_tower(const hals_tower_weights* w) {
  HALS_REQUIRE(w != nullptr, "null weights");
  HALS_REQUIRE(w->embedding_size >= 1 && w->embedding_size <= kTowerMaxE, "embedding_size must be in [1,64]");
  return 0;
}

extern "C" int hals_tower_user(const hals_tower_weights* w, const int32_t* user_ids, int64_t n, float* out,
                               int64_t out_stride, void* stream) {
  if (int rc = check_tower(w)) return rc;
  HALS_REQUIRE(w->user_emb && w->user_ln_g && w->user_ln_b && user_ids && out, "null pointer");
  HALS_REQUIRE(out_stride >= w->embedding_size, "out_stride too small");
  if (n == 0) return 0;
  tower_user_kernel<<<tower_blocks(n), kTowerThreads, 0, (cudaStream_t)stream>>>(*w, user_ids, n, out, out_stride);
  HALS_LAUNCH_CHECK();
  return 0;
}

extern "C" int hals_tower_item(const hals_tower_weights* w, const int32_t* item_ids,
                               const int32_t* manufacturer_ids, const int32_t* category_ids,
                               const float* numeric, int64_t n, float* out, int64_t out_stride, void* stream) {
  if (int rc = check_tower(w)) return rc;
  HALS_REQUIRE(w->item_emb && w->manu_emb && w->cat_emb && w->num_w && w->num_b && w->out_w && w->out_b &&
                   w->item_ln_g && w->item_ln_b, "null weight pointer");
  HALS_REQUIRE(item_ids && manufacturer_ids && category_ids && numeric && out, "null pointer");
  HALS_REQUIRE(out_stride >= w->embedding_size, "out_stride too small");
  HALS_REQUIRE(w->manu_dim >= 0 && w->cat_dim >= 0 && w->num_hidden >= 0, "negative width");
  if (n == 0) return 0;
  const int C = w->embedding_size + w->manu_dim + w->cat_dim + w->num_hidden;
  const size_t smem = sizeof(float) * ((size_t)C * w->embedding_size + 8 * C);
  HALS_REQUIRE(smem <= 200 * 1024, "tower too wide for shared memory");
  HALS_CUDA(cudaFuncSetAttribute(tower_item_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  tower_item_kernel<<<tower_blocks(n), kTowerThreads, smem, (cudaStream_t)stream>>>(
      *w, item_ids, manufacturer_ids, category_ids, numeric, n, out, out_stride);
  HALS_LAUNCH_CHECK();
  return 0;
}
