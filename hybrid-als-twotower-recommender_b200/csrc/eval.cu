// Batched evaluation helpers around the hot path (SURVEY.md 8(f) rows 3 and 4):
//   hals_f1_at_k        F1@k of per-user top-k lists against the users' rated items -- the weight selector of
//                       src/hybrid_system.py:42-55, compute_f1_score at src/als_model.py:171-177 (one user per call,
//                       Python sets, in the reference)
//   hals_similar_items  the content-similar fallback for cold ids of src/als_model.py:79-104: top-3 cosine neighbours
//                       with similarity > 0.5, mean of their ratings or the global mean (O(items) sklearn calls per
//                       cold item in the reference)
// Both are exact restatements (integer set arithmetic; fp64 cosine, ties to the lower item position = the stable
// sort over the dict order the reference uses).  Beside them:
//   hals_ranking_metrics  Spark's RankingMetrics per row (precision@k, recall@k, NDCG@k, AP@k, AP), behind
//                         ALSModel.evaluate_ranking
#include "common.cuh"

namespace hals {

// One warp per row.  The list is read in 32-entry chunks: lane j holds entry base + j, binary-searches it in the row's
// sorted labels, and a ballot gives each hit its rank among the hits so far (the running count carried across
// chunks is what AP needs).  Each lane sums its own positions in fp64; the butterfly reduction at the end runs in a
// fixed order, so the result is bitwise reproducible.  No atomics, no workspace.
__global__ void ranking_metrics_kernel(const int32_t* __restrict__ pred, int64_t pred_stride, int k, int64_t n_rows,
                                       const int64_t* __restrict__ rowptr, const int32_t* __restrict__ labels,
                                       double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;                                // warp-uniform
  const int64_t lo = rowptr[r], na = rowptr[r + 1] - lo;
  const int32_t* a = labels + lo;
  // |L|: distinct labels (sorted, so a label counts where it differs from its predecessor; Spark builds lab.toSet)
  int64_t distinct = 0;
  for (int64_t j = lane; j < na; j += 32) distinct += (j == 0 || a[j] != a[j - 1]) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) distinct += __shfl_xor_sync(0xffffffffu, distinct, o);
  double* o5 = out + r * 5;
  if (distinct == 0) {                                    // Spark returns 0 for every metric of an empty label set
    if (lane < 5) o5[lane] = 0.0;
    return;
  }
  const int32_t* p = pred + r * pred_stride;
  const unsigned below = (1u << lane) - 1u;
  int carried = 0;                                        // hits before the current chunk
  double dcg = 0.0, ap = 0.0, idcg = 0.0;
  for (int64_t base = 0; base < k; base += 32) {
    const int64_t e = base + lane;
    const int32_t item = e < k ? p[e] : -1;
    // the list ends at its first negative entry (the top-k kernels pad with -1) or at k
    const unsigned ended = __ballot_sync(0xffffffffu, item < 0);
    const bool valid = (ended & (below | (1u << lane))) == 0;
    bool hit = false;
    if (valid) {
      int64_t l = 0, h = na;                              // lower bound in the sorted labels
      while (l < h) {
        const int64_t m = (l + h) >> 1;
        if (a[m] < item) l = m + 1; else h = m;
      }
      hit = l < na && a[l] == item;
    }
    const unsigned hits = __ballot_sync(0xffffffffu, hit);
    if (hit) {
      const double g = 1.0 / log2((double)(e + 2));
      dcg += g;
      ap += (double)(carried + __popc(hits & below) + 1) / (double)(e + 1);
    }
    carried += __popc(hits);
    if (ended) break;                                     // warp-uniform
  }
  // ideal DCG: a hit at each of the first min(|L|, k) positions
  const int64_t n_ideal = distinct < (int64_t)k ? distinct : (int64_t)k;
  for (int64_t i = lane; i < n_ideal; i += 32) idcg += 1.0 / log2((double)(i + 2));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dcg += __shfl_xor_sync(0xffffffffu, dcg, o);
    ap += __shfl_xor_sync(0xffffffffu, ap, o);
    idcg += __shfl_xor_sync(0xffffffffu, idcg, o);
  }
  if (lane == 0) {
    const double nl = (double)distinct;
    o5[0] = (double)carried / (double)k;
    o5[1] = (double)carried / nl;
    o5[2] = dcg / idcg;
    o5[3] = ap / (double)n_ideal;
    o5[4] = ap / nl;
  }
}

// one warp per user: predicted[u][0..k) (first k valid entries of a score-sorted list) vs the sorted item list
// actual_items[rowptr[u] .. rowptr[u+1])
__global__ void f1_at_k_kernel(const int32_t* __restrict__ pred, int64_t pred_stride, int k,
                               const int64_t* __restrict__ rowptr, const int32_t* __restrict__ actual, int64_t n_users,
                               float* __restrict__ f1, int32_t* __restrict__ tp_out) {
  const int lane = threadIdx.x & 31;
  const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= n_users) return;
  const int64_t lo = rowptr[u], hi = rowptr[u + 1];
  const int32_t* a = actual + lo;
  const int64_t na = hi - lo;
  int tp = 0;
  for (int e = lane; e < k; e += 32) {
    const int32_t item = pred[u * pred_stride + e];
    if (item < 0) continue;                               // list shorter than k
    int64_t l = 0, r = na;                                // lower bound in the sorted actual list
    while (l < r) {
      const int64_t m = (l + r) >> 1;
      if (a[m] < item) l = m + 1; else r = m;
    }
    if (l < na && a[l] == item) {
      // a predicted list never repeats an item; the actual list may (duplicate ratings): a set counts it once
      ++tp;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tp += __shfl_xor_sync(0xffffffffu, tp, o);
  if (lane == 0) {
    // distinct rated items (the reference builds set(actual.keys()))
    int64_t distinct = 0;
    for (int64_t j = 0; j < na; ++j) distinct += (j == 0 || a[j] != a[j - 1]) ? 1 : 0;
    const double precision = (double)tp / (double)k;
    const double recall = distinct > 0 ? (double)tp / (double)distinct : 0.0;
    const double f = (precision + recall) > 0 ? 2.0 * (precision * recall) / (precision + recall) : 0.0;
    f1[u] = (float)f;
    if (tp_out) tp_out[u] = tp;
  }
}

// one warp per query item: cosine similarity (fp64, sklearn's normalise-then-dot) to every other item, best three by
// (similarity desc, position asc), those above 0.5 are averaged
__global__ void similar_items_kernel(const double* __restrict__ feats, int d, const double* __restrict__ ratings,
                                     int64_t n_items, const int32_t* __restrict__ queries, int64_t n_queries,
                                     double global_mean, double* __restrict__ out, int32_t* __restrict__ out_nbr) {
  const int lane = threadIdx.x & 31;
  const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= n_queries) return;
  const int32_t qi = queries[q];
  double best_s[3] = {-2.0, -2.0, -2.0};
  int32_t best_i[3] = {-1, -1, -1};
  if (qi >= 0 && qi < n_items) {
    double t[8], tn = 0.0;
    for (int f = 0; f < d; ++f) { t[f] = feats[(int64_t)qi * d + f]; tn += t[f] * t[f]; }
    tn = sqrt(tn);
    if (tn == 0.0) tn = 1.0;                              // sklearn.preprocessing.normalize leaves zero rows alone
    for (int f = 0; f < d; ++f) t[f] /= tn;
    for (int64_t j = lane; j < n_items; j += 32) {
      if (j == qi) continue;
      double y[8], yn = 0.0;
      for (int f = 0; f < d; ++f) { y[f] = feats[j * d + f]; yn += y[f] * y[f]; }
      yn = sqrt(yn);
      if (yn == 0.0) yn = 1.0;
      double s = 0.0;
      for (int f = 0; f < d; ++f) s += t[f] * (y[f] / yn);
      // insert into the lane's sorted triple (strict > keeps the lower position first on ties: j ascends per lane)
      if (s > best_s[2]) {
        best_s[2] = s; best_i[2] = (int32_t)j;
        if (best_s[2] > best_s[1]) { const double a = best_s[1]; best_s[1] = best_s[2]; best_s[2] = a; const int32_t b = best_i[1]; best_i[1] = best_i[2]; best_i[2] = b; }
        if (best_s[1] > best_s[0]) { const double a = best_s[0]; best_s[0] = best_s[1]; best_s[1] = a; const int32_t b = best_i[0]; best_i[0] = best_i[1]; best_i[1] = b; }
      }
    }
  }
  // warp merge: three rounds of "best remaining head" (similarity desc, position asc)
  double sum = 0.0;
  int cnt = 0;
  int head = 0;
  for (int r = 0; r < 3; ++r) {
    double s = head < 3 ? best_s[head] : -2.0;
    int32_t i = head < 3 ? best_i[head] : -1;
    double ws = s;
    int32_t wi = i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double os = __shfl_xor_sync(0xffffffffu, ws, o);
      const int32_t oi = __shfl_xor_sync(0xffffffffu, wi, o);
      const bool take = (oi >= 0) && (wi < 0 || os > ws || (os == ws && oi < wi));
      if (take) { ws = os; wi = oi; }
    }
    if (wi >= 0 && wi == i) ++head;                       // the winning lane advances its list
    if (out_nbr && lane == 0) out_nbr[q * 3 + r] = (wi >= 0 && ws > 0.5) ? wi : -1;
    if (wi >= 0 && ws > 0.5) { sum += ratings[wi]; ++cnt; }
  }
  if (lane == 0) out[q] = cnt > 0 ? sum / (double)cnt : global_mean;
}

}  // namespace hals

using namespace hals;

extern "C" int hals_f1_at_k(const int32_t* pred_idx, int64_t pred_stride, int k, const int64_t* actual_rowptr,
                            const int32_t* actual_items, int64_t n_users, float* f1, int32_t* true_positives,
                            void* stream) {
  HALS_REQUIRE(pred_idx && actual_rowptr && actual_items && f1, "null pointer");
  HALS_REQUIRE(k >= 1 && pred_stride >= k && n_users >= 0, "invalid sizes");
  if (n_users == 0) return 0;
  f1_at_k_kernel<<<(unsigned)((n_users + 7) / 8), 256, 0, (cudaStream_t)stream>>>(pred_idx, pred_stride, k, actual_rowptr,
                                                                                 actual_items, n_users, f1, true_positives);
  HALS_LAUNCH_CHECK();
  return 0;
}

extern "C" int hals_ranking_metrics(const int32_t* pred_idx, int64_t pred_stride, int k, int64_t n_rows,
                                    const int64_t* label_rowptr, const int32_t* label_items, double* out,
                                    void* stream) {
  HALS_REQUIRE(pred_idx, "pred_idx is null");
  HALS_REQUIRE(label_rowptr, "label_rowptr is null");
  HALS_REQUIRE(label_items, "label_items is null");
  HALS_REQUIRE(out, "out is null");
  HALS_REQUIRE(k >= 1, "k must be >= 1");
  HALS_REQUIRE(pred_stride >= k, "pred_stride must be >= k");
  HALS_REQUIRE(n_rows >= 0, "n_rows must be >= 0");
  if (n_rows == 0) return 0;
  ranking_metrics_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      pred_idx, pred_stride, k, n_rows, label_rowptr, label_items, out);
  HALS_LAUNCH_CHECK();
  return 0;
}

extern "C" int hals_similar_items(const double* features, int n_features, const double* ratings, int64_t n_items,
                                  const int32_t* queries, int64_t n_queries, double global_mean, double* out,
                                  int32_t* out_neighbours, void* stream) {
  HALS_REQUIRE(features && ratings && queries && out, "null pointer");
  HALS_REQUIRE(n_features >= 1 && n_features <= 8 && n_items >= 0 && n_queries >= 0, "invalid sizes");
  if (n_queries == 0) return 0;
  similar_items_kernel<<<(unsigned)((n_queries + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      features, n_features, ratings, n_items, queries, n_queries, global_mean, out, out_neighbours);
  HALS_LAUNCH_CHECK();
  return 0;
}
