// Two-tower training: one minibatch step (forward + backward, fused) and one Adam step over every parameter.
// Replaces model.fit at src/two_tower_model.py:91-121 (Adam, MSE) behind TwoTowerModel.train.
//
//   tower_train_step_kernel: one warp per batch row (kRows rows per CTA), out_w staged in shared memory as in the
//     forward kernel.  Each row's embedding-row gradients go to its own slot in the workspace; the dense-tensor
//     gradients are summed over the CTA's rows in row order into one partial per CTA.  The CTA holding sorted
//     position k of a table stamps the row the id names with (t, k) when k is the first position of that id.
//   tower_adam_kernel: one launch.  Blocks [0, dense_blocks) own the dense tensors (one thread per element, the CTA
//     partials summed in CTA order); the rest own the embedding rows (one warp per row).  A stamped row sums its
//     per-position gradients from its first sorted position on, i.e. in ascending batch position (the sort is
//     stable); an unstamped row takes g = 0 and still decays its moments.  No float atomics anywhere.
#include "tower_common.cuh"

namespace hals {

constexpr int kTrainRows = 16;           // batch rows per CTA of the step kernel (two per warp)
constexpr int kAdamRowBlocksPerSm = 16;

struct TrainDims {
  int E, MD, CD, H, C, RW, D, S;
  // dense layout: out_w [C,E] | out_b [E] | num_w [2,H] | num_b [H] | user_ln_g | user_ln_b | item_ln_g | item_ln_b [E]
  __host__ __device__ int o_outb() const { return C * E; }
  __host__ __device__ int o_numw() const { return C * E + E; }
  __host__ __device__ int o_numb() const { return C * E + E + 2 * H; }
  __host__ __device__ int o_ln() const { return C * E + E + 3 * H; }
};

__host__ __device__ inline TrainDims train_dims(int E, int MD, int CD, int H) {
  TrainDims d;
  d.E = E; d.MD = MD; d.CD = CD; d.H = H;
  d.C = E + MD + CD + H;
  d.RW = 2 * E + MD + CD;                // per-row gradient slot: user | item | manufacturer | category
  d.D = d.C * E + E + 3 * H + 4 * E;     // dense elements; partial slot D holds the CTA's sum of squared residuals
  d.S = d.C + 5 * E + d.H + 3;           // shared floats per row: c | dz | xu | du | xi | di | dh | x0 x1 res^2
  return d;
}

struct TrainLayout {
  size_t tags, counter, rows, part, total;
  int64_t parts;
};

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

inline TrainLayout train_layout(const hals_tower_params& w, int64_t n) {
  const TrainDims d = train_dims(w.embedding_size, w.manu_dim, w.cat_dim, w.num_hidden);
  TrainLayout L;
  L.parts = (n + kTrainRows - 1) / kTrainRows;
  const int64_t table_rows = (int64_t)w.num_users + w.num_items + w.num_manufacturers + w.num_categories;
  L.tags = 0;
  L.counter = align256(sizeof(int2) * (size_t)table_rows);
  L.rows = L.counter + 256;
  L.part = L.rows + align256(sizeof(float) * (size_t)n * d.RW);
  L.total = L.part + sizeof(float) * (size_t)L.parts * (d.D + 1);
  return L;
}

__device__ __forceinline__ const int32_t* batch_ids(const hals_tower_batch& b, int t) {
  return t == 0 ? b.user_ids : t == 1 ? b.item_ids : t == 2 ? b.manufacturer_ids : b.category_ids;
}
__device__ __forceinline__ const int32_t* batch_order(const hals_tower_batch& b, int t) {
  return t == 0 ? b.order_user : t == 1 ? b.order_item : t == 2 ? b.order_manufacturer : b.order_category;
}
__device__ __forceinline__ int table_rows(const hals_tower_params& w, int t) {
  return t == 0 ? w.num_users : t == 1 ? w.num_items : t == 2 ? w.num_manufacturers : w.num_categories;
}
__device__ __forceinline__ int64_t table_tag0(const hals_tower_params& w, int t) {
  return t == 0 ? 0 : t == 1 ? (int64_t)w.num_users : t == 2 ? (int64_t)w.num_users + w.num_items
                                                              : (int64_t)w.num_users + w.num_items + w.num_manufacturers;
}

__global__ void __launch_bounds__(kTowerThreads)
tower_train_step_kernel(hals_tower_params w, hals_tower_batch b, int stamp, int2* __restrict__ tags,
                        float* __restrict__ rows, float* __restrict__ part, unsigned* __restrict__ counter,
                        float* __restrict__ loss) {
  extern __shared__ float sm[];
  const TrainDims dm = train_dims(w.embedding_size, w.manu_dim, w.cat_dim, w.num_hidden);
  const int E = dm.E, C = dm.C, H = dm.H, S = dm.S, EMC = E + dm.MD + dm.CD;
  const int64_t n = b.n;
  float* Wo = sm;                          // [C][E]
  float* rs = sm + C * E;                  // [kTrainRows][S]
  for (int e = threadIdx.x; e < C * E; e += kTowerThreads) Wo[e] = w.out_w[e];
  if (threadIdx.x < 4 * kTrainRows) {      // stamp the first sorted position of every id this CTA's positions hold
    const int t = threadIdx.x / kTrainRows;
    const int64_t k = (int64_t)blockIdx.x * kTrainRows + threadIdx.x % kTrainRows;
    if (k < n) {
      const int32_t *ids = batch_ids(b, t), *ord = batch_order(b, t);
      const int id = ids[ord[k]];
      if ((k == 0 || ids[ord[k - 1]] != id) && in_table(id, table_rows(w, t)))
        tags[table_tag0(w, t) + id] = make_int2(stamp, (int)k);
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool h0 = lane < E, h1 = lane + 32 < E;
  for (int j = 0; j < kTrainRows / 8; ++j) {
    const int r = warp + 8 * j;
    const int64_t p = (int64_t)blockIdx.x * kTrainRows + r;
    float* c = rs + r * S;
    float *dz = c + C, *xu = dz + E, *du = xu + E, *xi = du + E, *di = xi + E, *dh = di + E, *xs = dh + H;
    if (p >= n) {                          // past the batch: contributes zeros to the CTA partials
      for (int f = lane; f < S; f += 32) c[f] = 0.f;
      continue;
    }
    const int uid = b.user_ids[p], ii = b.item_ids[p], mi = b.manufacturer_ids[p], ci = b.category_ids[p];
    const bool oku = in_table(uid, w.num_users), oki = in_table(ii, w.num_items);
    const bool okm = in_table(mi, w.num_manufacturers), okc = in_table(ci, w.num_categories);
    // ---- forward: user tower
    const float* eu = w.user_emb + (int64_t)(oku ? uid : 0) * E;
    float xu0, xu1, invu;
    warp_layer_norm((oku && h0) ? eu[lane] : 0.f, (oku && h1) ? eu[lane + 32] : 0.f, E, lane, w.ln_eps, xu0, xu1, invu);
    const float gu0 = h0 ? w.user_ln_g[lane] : 0.f, gu1 = h1 ? w.user_ln_g[lane + 32] : 0.f;
    const float uo0 = h0 ? fmaf(xu0, gu0, w.user_ln_b[lane]) : 0.f;
    const float uo1 = h1 ? fmaf(xu1, gu1, w.user_ln_b[lane + 32]) : 0.f;
    // ---- forward: item tower (concat vector kept in shared memory; dh holds the hidden pre-activation for now)
    const float x0 = b.numeric[p * 2 + 0], x1 = b.numeric[p * 2 + 1];
    const float* ei = w.item_emb + (int64_t)(oki ? ii : 0) * E;
    const float* em = w.manu_emb + (int64_t)(okm ? mi : 0) * dm.MD;
    const float* ec = w.cat_emb + (int64_t)(okc ? ci : 0) * dm.CD;
    for (int f = lane; f < C; f += 32) {
      float v;
      if (f < E) v = oki ? ei[f] : 0.f;
      else if (f < E + dm.MD) v = okm ? em[f - E] : 0.f;
      else if (f < EMC) v = okc ? ec[f - E - dm.MD] : 0.f;
      else {
        const int h = f - EMC;
        const float pre = fmaf(x1, w.num_w[H + h], fmaf(x0, w.num_w[h], w.num_b[h]));
        dh[h] = pre;
        v = fmaxf(pre, 0.f);
      }
      c[f] = v;
    }
    __syncwarp();
    float z0 = h0 ? w.out_b[lane] : 0.f, z1 = h1 ? w.out_b[lane + 32] : 0.f;
    for (int f = 0; f < C; ++f) {
      const float cf = c[f];
      if (h0) z0 = fmaf(cf, Wo[f * E + lane], z0);
      if (h1) z1 = fmaf(cf, Wo[f * E + lane + 32], z1);
    }
    float xi0, xi1, invi;
    warp_layer_norm(z0, z1, E, lane, w.ln_eps, xi0, xi1, invi);
    const float gi0 = h0 ? w.item_ln_g[lane] : 0.f, gi1 = h1 ? w.item_ln_g[lane + 32] : 0.f;
    const float io0 = h0 ? fmaf(xi0, gi0, w.item_ln_b[lane]) : 0.f;
    const float io1 = h1 ? fmaf(xi1, gi1, w.item_ln_b[lane + 32]) : 0.f;
    // ---- loss: d(mean (pred - y)^2) / d pred = 2 (pred - y) / n
    const float res = warp_sum(uo0 * io0 + uo1 * io1) - b.labels[p];
    const float gp = 2.f * res / (float)n;
    const float du0 = gp * io0, du1 = gp * io1, di0 = gp * uo0, di1 = gp * uo1;
    // ---- backward through the user LayerNorm: dx = inv (dxh - mean(dxh) - xh mean(dxh xh)), dxh = dy * gamma
    {
      const float a0 = du0 * gu0, a1 = du1 * gu1;
      const float m1 = warp_sum(a0 + a1) / (float)E, m2 = warp_sum(a0 * xu0 + a1 * xu1) / (float)E;
      float* gr = rows + p * dm.RW;
      if (h0) gr[lane] = oku ? invu * (a0 - m1 - xu0 * m2) : 0.f;
      if (h1) gr[lane + 32] = oku ? invu * (a1 - m1 - xu1 * m2) : 0.f;
    }
    // ---- backward through the item LayerNorm -> dz (gradient of W_o . c + b_o)
    {
      const float a0 = di0 * gi0, a1 = di1 * gi1;
      const float m1 = warp_sum(a0 + a1) / (float)E, m2 = warp_sum(a0 * xi0 + a1 * xi1) / (float)E;
      if (h0) dz[lane] = invi * (a0 - m1 - xi0 * m2);
      if (h1) dz[lane + 32] = invi * (a1 - m1 - xi1 * m2);
    }
    if (h0) { xu[lane] = xu0; du[lane] = du0; xi[lane] = xi0; di[lane] = di0; }
    if (h1) { xu[lane + 32] = xu1; du[lane + 32] = du1; xi[lane + 32] = xi1; di[lane + 32] = di1; }
    if (lane == 0) { xs[0] = x0; xs[1] = x1; xs[2] = res * res; }
    __syncwarp();
    // ---- dc = W_o dz: the three gathered rows' gradients and, through the ReLU, the hidden layer's
    float* gr = rows + p * dm.RW + E;      // item | manufacturer | category, contiguous like the concat
    for (int f = lane; f < C; f += 32) {
      float acc = 0.f;
      for (int e = 0; e < E; ++e) acc = fmaf(Wo[f * E + e], dz[e], acc);
      if (f < E) gr[f] = oki ? acc : 0.f;
      else if (f < E + dm.MD) gr[f] = okm ? acc : 0.f;
      else if (f < EMC) gr[f] = okc ? acc : 0.f;
      else dh[f - EMC] = dh[f - EMC] > 0.f ? acc : 0.f;   // same lane wrote the pre-activation above
    }
    __syncwarp();
  }
  __syncthreads();
  // ---- dense partials of this CTA: rows summed in row order
  float* out = part + (int64_t)blockIdx.x * (dm.D + 1);
  for (int d = threadIdx.x; d <= dm.D; d += kTowerThreads) {
    float acc = 0.f;
    if (d < dm.o_outb()) {
      const int f = d / E, e = d - f * E;
      for (int r = 0; r < kTrainRows; ++r) acc = fmaf(rs[r * S + f], rs[r * S + C + e], acc);
    } else if (d < dm.o_numw()) {
      const int e = d - dm.o_outb();
      for (int r = 0; r < kTrainRows; ++r) acc += rs[r * S + C + e];
    } else if (d < dm.o_numb()) {
      const int k = (d - dm.o_numw()) / H, h = d - dm.o_numw() - k * H;
      for (int r = 0; r < kTrainRows; ++r) acc = fmaf(rs[r * S + C + 5 * E + H + k], rs[r * S + C + 5 * E + h], acc);
    } else if (d < dm.o_ln()) {
      const int h = d - dm.o_numb();
      for (int r = 0; r < kTrainRows; ++r) acc += rs[r * S + C + 5 * E + h];
    } else if (d < dm.D) {
      const int q = (d - dm.o_ln()) / E, e = d - dm.o_ln() - q * E;   // q: user g, user b, item g, item b
      const int dy = C + (q < 2 ? 2 : 4) * E, xh = C + (q < 2 ? 1 : 3) * E;
      for (int r = 0; r < kTrainRows; ++r)
        acc = (q & 1) ? acc + rs[r * S + dy + e] : fmaf(rs[r * S + dy + e], rs[r * S + xh + e], acc);
    } else {
      for (int r = 0; r < kTrainRows; ++r) acc += rs[r * S + C + 5 * E + H + 2];
    }
    out[d] = acc;
  }
  // ---- the last CTA to finish sums the squared residuals of all CTAs in CTA order
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last && warp == 0) {
    __threadfence();
    float s = 0.f;
    for (unsigned q = lane; q < gridDim.x; q += 32) s += __ldcg(part + (int64_t)q * (dm.D + 1) + dm.D);
    s = warp_sum(s);
    if (lane == 0) {
      *loss = s / (float)n;
      *counter = 0u;                       // ready for the next step
    }
  }
}

struct AdamScalars {
  float step_size, bc2_sqrt, w1, b2, omb2, eps;
};

__device__ __forceinline__ void adam_update(float* p, float* m, float* v, int64_t i, float g, const AdamScalars& s) {
  float mi = m[i], vi = v[i];
  mi = s.w1 < 0.5f ? fmaf(s.w1, g - mi, mi) : g - (g - mi) * (1.f - s.w1);   // torch's lerp(m, g, 1 - beta1)
  vi = fmaf(s.omb2 * g, g, vi * s.b2);
  const float denom = sqrtf(vi) / s.bc2_sqrt + s.eps;
  p[i] = p[i] + (-s.step_size) * (mi / denom);
  m[i] = mi;
  v[i] = vi;
}

__global__ void __launch_bounds__(kTowerThreads)
tower_adam_kernel(hals_tower_params w, hals_tower_params m, hals_tower_params v, hals_tower_batch b, int stamp,
                  const int2* __restrict__ tags, const float* __restrict__ rows, const float* __restrict__ part,
                  int parts, int dense_blocks, AdamScalars s) {
  const TrainDims dm = train_dims(w.embedding_size, w.manu_dim, w.cat_dim, w.num_hidden);
  if ((int)blockIdx.x < dense_blocks) {
    const int d = blockIdx.x * kTowerThreads + threadIdx.x;
    if (d >= dm.D) return;
    float g = 0.f;
    for (int q = 0; q < parts; ++q) g += part[(int64_t)q * (dm.D + 1) + d];
    float *P, *M, *V;
    int i;
    const int E = dm.E;
    if (d < dm.o_outb()) { P = w.out_w; M = m.out_w; V = v.out_w; i = d; }
    else if (d < dm.o_numw()) { P = w.out_b; M = m.out_b; V = v.out_b; i = d - dm.o_outb(); }
    else if (d < dm.o_numb()) { P = w.num_w; M = m.num_w; V = v.num_w; i = d - dm.o_numw(); }
    else if (d < dm.o_ln()) { P = w.num_b; M = m.num_b; V = v.num_b; i = d - dm.o_numb(); }
    else {
      const int q = (d - dm.o_ln()) / E;
      i = d - dm.o_ln() - q * E;
      P = q == 0 ? w.user_ln_g : q == 1 ? w.user_ln_b : q == 2 ? w.item_ln_g : w.item_ln_b;
      M = q == 0 ? m.user_ln_g : q == 1 ? m.user_ln_b : q == 2 ? m.item_ln_g : m.item_ln_b;
      V = q == 0 ? v.user_ln_g : q == 1 ? v.user_ln_b : q == 2 ? v.item_ln_g : v.item_ln_b;
    }
    adam_update(P, M, V, i, g, s);
    return;
  }
  // embedding rows: one warp per row, the four tables back to back
  const int lane = threadIdx.x & 31;
  const int64_t r1 = w.num_users, r2 = r1 + w.num_items, r3 = r2 + w.num_manufacturers, r4 = r3 + w.num_categories;
  const int64_t warps = (int64_t)(gridDim.x - dense_blocks) * (kTowerThreads / 32);
  for (int64_t R = (int64_t)(blockIdx.x - dense_blocks) * (kTowerThreads / 32) + (threadIdx.x >> 5); R < r4;
       R += warps) {
    const int t = R < r1 ? 0 : R < r2 ? 1 : R < r3 ? 2 : 3;
    const int row = (int)(R - (t == 0 ? 0 : t == 1 ? r1 : t == 2 ? r2 : r3));
    const int W = t == 0 || t == 1 ? dm.E : t == 2 ? dm.MD : dm.CD;
    const int off = t == 0 ? 0 : t == 1 ? dm.E : t == 2 ? 2 * dm.E : 2 * dm.E + dm.MD;
    float* P = t == 0 ? w.user_emb : t == 1 ? w.item_emb : t == 2 ? w.manu_emb : w.cat_emb;
    float* M = t == 0 ? m.user_emb : t == 1 ? m.item_emb : t == 2 ? m.manu_emb : m.cat_emb;
    float* V = t == 0 ? v.user_emb : t == 1 ? v.item_emb : t == 2 ? v.manu_emb : v.cat_emb;
    const int2 tag = tags[R];
    for (int col = lane; col < W; col += 32) {
      float g = 0.f;
      if (tag.x == stamp) {
        const int32_t *ids = batch_ids(b, t), *ord = batch_order(b, t);
        for (int64_t k = tag.y; k < b.n; ++k) {
          const int pos = ord[k];
          if (ids[pos] != row) break;
          g += rows[(int64_t)pos * dm.RW + off + col];
        }
      }
      adam_update(P, M, V, (int64_t)row * W + col, g, s);
    }
  }
}

}  // namespace hals

using namespace hals;

static int check_params(const hals_tower_params* w) {
  HALS_REQUIRE(w != nullptr, "null params");
  HALS_REQUIRE(w->embedding_size >= 1 && w->embedding_size <= kTowerMaxE, "embedding_size must be in [1,64]");
  HALS_REQUIRE(w->manu_dim >= 0 && w->cat_dim >= 0 && w->num_hidden >= 0, "negative width");
  HALS_REQUIRE(w->num_users > 0 && w->num_items > 0 && w->num_manufacturers > 0 && w->num_categories > 0,
               "table sizes must be given (> 0)");
  HALS_REQUIRE(w->user_emb && w->item_emb && w->manu_emb && w->cat_emb && w->num_w && w->num_b && w->out_w &&
                   w->out_b && w->user_ln_g && w->user_ln_b && w->item_ln_g && w->item_ln_b, "null tensor pointer");
  const TrainDims d = train_dims(w->embedding_size, w->manu_dim, w->cat_dim, w->num_hidden);
  HALS_REQUIRE(sizeof(float) * ((size_t)d.C * d.E + (size_t)kTrainRows * d.S) <= 200 * 1024,
               "tower too wide for shared memory");
  return 0;
}

static bool same_shape(const hals_tower_params* a, const hals_tower_params* b) {
  return a->embedding_size == b->embedding_size && a->manu_dim == b->manu_dim && a->cat_dim == b->cat_dim &&
         a->num_hidden == b->num_hidden && a->num_users == b->num_users && a->num_items == b->num_items &&
         a->num_manufacturers == b->num_manufacturers && a->num_categories == b->num_categories;
}

static int check_batch(const hals_tower_batch* b, int64_t t) {
  HALS_REQUIRE(b != nullptr, "null batch");
  HALS_REQUIRE(b->n >= 1 && b->n <= INT32_MAX, "batch size must be in [1, INT32_MAX]");
  HALS_REQUIRE(t >= 1 && t <= INT32_MAX, "step t must be in [1, INT32_MAX]");
  HALS_REQUIRE(b->user_ids && b->item_ids && b->manufacturer_ids && b->category_ids && b->numeric && b->labels &&
                   b->order_user && b->order_item && b->order_manufacturer && b->order_category, "null batch pointer");
  return 0;
}

extern "C" size_t hals_tower_train_workspace_bytes(const hals_tower_params* params, int64_t max_batch) {
  if (!params || max_batch < 1 || params->embedding_size < 1 || params->manu_dim < 0 || params->cat_dim < 0 ||
      params->num_hidden < 0 || params->num_users < 0 || params->num_items < 0 || params->num_manufacturers < 0 ||
      params->num_categories < 0)
    return 0;
  return train_layout(*params, max_batch).total;
}

extern "C" int hals_tower_train_step(const hals_tower_params* params, const hals_tower_batch* batch, int64_t t,
                                     void* workspace, size_t workspace_bytes, float* loss, void* stream) {
  if (int rc = check_params(params)) return rc;
  if (int rc = check_batch(batch, t)) return rc;
  HALS_REQUIRE(workspace && loss, "null pointer");
  const TrainLayout L = train_layout(*params, batch->n);
  if (workspace_bytes < L.total) return fail(HALS_ERR_WORKSPACE, "%s: workspace too small%s", __func__);
  const TrainDims d = train_dims(params->embedding_size, params->manu_dim, params->cat_dim, params->num_hidden);
  const size_t smem = sizeof(float) * ((size_t)d.C * d.E + (size_t)kTrainRows * d.S);
  char* ws = (char*)workspace;
  HALS_CUDA(cudaFuncSetAttribute(tower_train_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  tower_train_step_kernel<<<(unsigned)L.parts, kTowerThreads, smem, (cudaStream_t)stream>>>(
      *params, *batch, (int)t, (int2*)(ws + L.tags), (float*)(ws + L.rows), (float*)(ws + L.part),
      (unsigned*)(ws + L.counter), loss);
  HALS_LAUNCH_CHECK();
  return 0;
}

extern "C" int hals_tower_adam_step(const hals_tower_params* params, const hals_tower_params* m,
                                    const hals_tower_params* v, const hals_tower_batch* batch, int64_t t,
                                    const void* workspace, size_t workspace_bytes, double lr, double beta1,
                                    double beta2, double eps, void* stream) {
  if (int rc = check_params(params)) return rc;
  if (int rc = check_params(m)) return rc;
  if (int rc = check_params(v)) return rc;
  HALS_REQUIRE(same_shape(params, m) && same_shape(params, v), "m and v must have the shapes of params");
  if (int rc = check_batch(batch, t)) return rc;
  HALS_REQUIRE(workspace != nullptr, "null workspace");
  HALS_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0, "betas must lie in [0, 1)");
  HALS_REQUIRE(lr >= 0.0 && eps >= 0.0, "lr and eps must be >= 0");
  const TrainLayout L = train_layout(*params, batch->n);
  if (workspace_bytes < L.total) return fail(HALS_ERR_WORKSPACE, "%s: workspace too small%s", __func__);
  const TrainDims d = train_dims(params->embedding_size, params->manu_dim, params->cat_dim, params->num_hidden);
  // torch.optim.Adam (single-tensor): bias corrections and the step size in double, each used as an fp32 scalar
  const double bc1 = 1.0 - pow(beta1, (double)t), bc2 = 1.0 - pow(beta2, (double)t);
  AdamScalars s;
  s.step_size = (float)(lr / bc1);
  s.bc2_sqrt = (float)sqrt(bc2);
  s.w1 = (float)(1.0 - beta1);
  s.b2 = (float)beta2;
  s.omb2 = (float)(1.0 - beta2);
  s.eps = (float)eps;
  const int dense_blocks = (d.D + kTowerThreads - 1) / kTowerThreads;
  const int64_t table_rows =
      (int64_t)params->num_users + params->num_items + params->num_manufacturers + params->num_categories;
  int64_t row_blocks = (table_rows + kTowerThreads / 32 - 1) / (kTowerThreads / 32);
  const int64_t cap = (int64_t)kAdamRowBlocksPerSm * sm_count();
  if (row_blocks > cap) row_blocks = cap;
  const char* ws = (const char*)workspace;
  tower_adam_kernel<<<(unsigned)(dense_blocks + row_blocks), kTowerThreads, 0, (cudaStream_t)stream>>>(
      *params, *m, *v, *batch, (int)t, (const int2*)(ws + L.tags), (const float*)(ws + L.rows),
      (const float*)(ws + L.part), (int)L.parts, dense_blocks, s);
  HALS_LAUNCH_CHECK();
  return 0;
}
