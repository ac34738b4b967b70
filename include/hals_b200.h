/* hals_b200.h -- C ABI of the B200-native ALS half-step and hybrid top-k scoring path.
 *
 * Drop-in boundary for HSoumi/hybrid-als-twotower-recommender.  The reference has no
 * FFI of its own: its hot path is three Python methods that delegate to third-party
 * engines (pyspark.ml ALS over Py4J, Keras Model.predict, sklearn MinMaxScaler, Python
 * sorted()).  Each entry point below replaces one such delegation; the reference call
 * site it replaces is cited as file:line (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing
 *     synchronises the device, nothing allocates device memory (caller-owned buffers,
 *     sizes from the *_workspace_bytes queries);
 *   - return value 0 = ok, non-zero = hals_status; hals_last_error() gives the message
 *     of the last failure on the calling thread;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails
 *     with HALS_ERR_CUDA.
 */
#ifndef HALS_B200_H_
#define HALS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HALS_ABI_VERSION 1

typedef enum hals_status {
  HALS_OK = 0,
  HALS_ERR_INVALID = 1,   /* bad argument (null pointer, unsupported rank, ...)   */
  HALS_ERR_CUDA = 2,      /* CUDA runtime error (message in hals_last_error())   */
  HALS_ERR_WORKSPACE = 3, /* caller workspace too small                           */
  HALS_ERR_UNSUPPORTED = 4
} hals_status;

int hals_abi_version(void);
const char* hals_last_error(void);
/* Number of kernels this library has launched in the calling process (all threads).
 * bench.py reads it around the timed region to report "gpu_launches". */
int64_t hals_launch_count(void);
/* Maximum factor rank / embedding width the kernels are compiled for. */
int hals_max_rank(void);

/* ------------------------------------------------------------------------------------
 * ALS half-step.  Replaces pyspark ALS.fit's computeFactors (NormalEquation.add,
 * CholeskySolver.solve) reached from src/als_model.py:62, with the parameters the
 * reference sets at src/als_model.py:52-60 (rank, regParam) plus Spark's implicitPrefs /
 * alpha (defaults false / 1.0).
 *
 * For every row j of a CSR matrix (ratings of destination row j against source rows):
 *   explicit:  A = sum_i y_i y_i^T,                b = sum_i r_ji y_i,          n = nnz_j
 *   implicit:  A = gram + sum_i c1 y_i y_i^T,      b = sum_{r>0} (1+c1) y_i,    n = #{r>0},  c1 = alpha*|r|
 *   A[d,d] += reg * n ;  dst_j = A^{-1} b (Cholesky).  Rows without ratings get 0.
 * reg must be finite and >= 0 (Spark's regParam validator, gtEq(0)); anything else is HALS_ERR_INVALID before any
 * CUDA call, here and in hals_als_half_step_split.  reg = 0 is accepted (A is then singular for a row with fewer
 * ratings than k).
 *
 * Work decomposition is described by a plan built once per CSR matrix: rows longer than
 * `seg_len` ratings are cut into segments whose partial (A,b) go through `workspace` and
 * are reduced in a fixed order (deterministic, no float atomics).
 * ---------------------------------------------------------------------------------- */
typedef struct hals_als_plan {
  int64_t n_items;           /* work items (row segments)                                  */
  int64_t n_long_rows;       /* rows cut into >1 segment                                   */
  int64_t n_slots;           /* partial (A,b) slots needed in the workspace                */
  int32_t seg_len;           /* segment length the plan was built for                      */
  int32_t max_nseg;          /* largest entry of long_nseg (0 when there are no long rows)  */
  const int32_t* item_row;   /* [n_items] destination row                                  */
  const int64_t* item_begin; /* [n_items] first rating (index into colidx/vals)            */
  const int32_t* item_len;   /* [n_items] ratings in this item                             */
  const int32_t* item_slot;  /* [n_items] workspace slot, or -1 when the item is a whole row */
  const int32_t* long_row;   /* [n_long_rows] destination row                              */
  const int32_t* long_slot0; /* [n_long_rows] first slot                                   */
  const int32_t* long_nseg;  /* [n_long_rows] number of slots                              */
  /* Optional: when the long-row arrays are sorted by long_nseg DESCENDING, the number of rows with more than 16 and
   * more than 256 slices -- the slot pre-sum launches then cover only those rows.  0 = unknown (all long rows). */
  int64_t n_long_gt16, n_long_gt256;
  /* Chunk table (optional; hals_als_plan_chunks_host).  The ratings of work item i, cut into pieces of 32, are chunks
   * [item_chunk0[i], item_chunk0[i+1]); the persistent rank-64 / rank-128 kernels give every CTA a CONTIGUOUS range of
   * items of equal cost (item_cost0 = prefix sum of chunks + a per-item solve / park cost) and stream its chunks. */
  int64_t n_chunks;
  const int64_t* item_chunk0; /* [n_items+1] */
  const int64_t* item_cost0;  /* [n_items+1] */
  const int64_t* chunk_pos;   /* [n_chunks] index of the chunk's first rating (into colidx / vals)              */
  const int32_t* chunk_cnt;   /* [n_chunks] ratings left in its item at that point (<= 32: the item's last chunk) */
  const uint32_t* vals_hl;   /* optional [nnz], same order as vals: bf16(r) | bf16(r - bf16(r)) << 16, written by
                                hals_als_pack_ratings once per ratings matrix.  The tensor-core kernels
                                copy it straight into the MMA operand; NULL selects the slower kernel that
                                converts the fp32 ratings itself. */
  /* Implicit feedback on the tensor cores (ranks 64 and 128; optional -- without them implicit mode runs the CUDA-core
   * kernel).
   * hals_als_pack_ratings_implicit fills vals_hl with (1 + c) / sqrt(c) where r > 0 (0 elsewhere) and vals_scale with
   * sqrt(c), c = alpha |r|; hals_als_plan_count_positive fills item_npos.  packed_alpha records the alpha they were
   * built for: 0 = vals_hl holds the plain ratings (explicit feedback). */
  const float* vals_scale;   /* [nnz] sqrt(alpha |r|)                                      */
  const int32_t* item_npos;  /* [n_items] ratings > 0 in the work item                     */
  float packed_alpha;
} hals_als_plan;

/* Host-side planner (pure CPU, no CUDA): sizes first, then fill caller arrays.
 * rowptr_host: [m+1] int64 on the HOST. */
int hals_als_plan_count_host(const int64_t* rowptr_host, int64_t m, int32_t seg_len,
                             int64_t* n_items, int64_t* n_long_rows, int64_t* n_slots);
int hals_als_plan_fill_host(const int64_t* rowptr_host, int64_t m, int32_t seg_len,
                            int32_t* item_row, int64_t* item_begin, int32_t* item_len,
                            int32_t* item_slot, int32_t* long_row, int32_t* long_slot0,
                            int32_t* long_nseg);
/* Chunk table of a filled plan (host arrays in, host arrays out; pure CPU).  hals_als_plan_chunk_count_host returns
 * the number of chunks, or -1 on invalid input. */
int64_t hals_als_plan_chunk_count_host(const int32_t* item_len, int64_t n_items);
int hals_als_plan_chunks_host(const int32_t* item_len, const int64_t* item_begin, const int32_t* item_slot,
                              int64_t n_items, int k /* rank: sets the solve : gather cost ratio */,
                              int64_t* item_chunk0, int64_t* item_cost0, int64_t* chunk_pos, int32_t* chunk_cnt);
/* Bytes of device workspace hals_als_half_step needs for a plan with n_slots slots and a
 * source factor matrix of n_src rows (the tensor-core path keeps a bf16 split copy of it). */
size_t hals_als_workspace_bytes(int64_t n_slots, int k, int64_t n_src);
/* Default segment length for rank k (ratings per work item). */
int32_t hals_als_default_seg_len(int k);
/* out[i] = bf16(vals[i]) | bf16(vals[i] - bf16(vals[i])) << 16 (device arrays); see hals_als_plan.vals_hl. */
int hals_als_pack_ratings(const float* vals, int64_t nnz, uint32_t* out, void* stream);
/* Implicit-feedback operands of the tensor-core kernel (see hals_als_plan.vals_scale); device arrays. */
int hals_als_pack_ratings_implicit(const float* vals, int64_t nnz, float alpha, uint32_t* out_hl, float* out_scale,
                                   void* stream);
int hals_als_plan_count_positive(const float* vals, const int64_t* item_begin, const int32_t* item_len, int64_t n_items,
                                 int32_t* item_npos, void* stream);

int hals_als_half_step(const int64_t* rowptr, const int32_t* colidx, const float* vals,
                       int64_t m_dst, const float* src, int64_t n_src, float* dst, int k,
                       float reg, int implicit, float alpha, const float* gram,
                       const hals_als_plan* plan /* device arrays inside */, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Nonnegative factors (Spark's ALS nonnegative=True, NNLSSolver): the same A and b as hals_als_half_step, in both modes,
 * and dst_j = argmin_{x >= 0} 1/2 x^T A x - b^T x, the unique minimiser (A is positive definite because reg n > 0).
 * Solved by block principal pivoting (Kim & Park 2011, Judice-Pires backup rule); each iterate solves the free
 * subsystem A_FF x_F = b_F by Cholesky, so the accuracy is that of hals_als_half_step.  Deterministic.
 *   - always the CUDA-core kernels, at ranks 64 and 128 too, whatever the plan carries (vals_hl etc. are ignored);
 *   - reg <= 0: HALS_ERR_INVALID;
 *   - the pivoting loop is capped at 3k + 8 free-set factorisations per row; a row that reaches the cap keeps its
 *     last iterate with x >= 0 (finite, nonnegative) and, when n_capped (device int32) is not NULL, is added to
 *     *n_capped atomically.  The caller zeroes *n_capped;
 *   - workspace: hals_als_workspace_bytes, as for hals_als_half_step.  Rows without ratings get 0. */
int hals_als_half_step_nonnegative(const int64_t* rowptr, const int32_t* colidx, const float* vals,
                                   int64_t m_dst, const float* src, int64_t n_src, float* dst, int k,
                                   float reg, int implicit, float alpha, const float* gram,
                                   const hals_als_plan* plan, void* workspace, size_t workspace_bytes,
                                   void* stream, int32_t* n_capped);

/* Ranks 64 and 128, factors kept in split form across half-steps (what als_engine does; the stateless call above re-splits
 * the whole source matrix every time, which is a replicated pass on every rank of a sharded run).
 *   hals_als_split_factors: out_hl[r] = [bf16(x) (k) | bf16(x - bf16(x)) (k)] for n_rows rows (k = 64 or 128).
 *   hals_als_half_step_split: src_hl = split source factors, [n_src + 1] rows of 2k bf16, ROW n_src ALL ZERO (the
 *     ragged tail of a chunk gathers it); every solved row j is written twice: dst[j] (fp32, k) and dst_hl[j] (its
 *     split, 2k bf16) -- dst and dst_hl are indexed by the plan's destination rows.  Rows without ratings are not
 *     touched.  colidx indexes rows of src_hl (a sharded engine stores the factors padded by owner rank, so that the
 *     all-gather of the freshly solved rows is in place, and remaps colidx once).  Explicit feedback only. */
int hals_als_split_factors(const float* src, int64_t n_rows, int k, void* out_hl, void* stream);
int hals_als_half_step_split(const int32_t* colidx, int64_t m_dst, const void* src_hl, int64_t n_src, float* dst,
                             void* dst_hl, int k, float reg, const hals_als_plan* plan, void* workspace,
                             size_t workspace_bytes, void* stream);

/* Dense Gram Y^T Y ([n,k] -> [k,k], fp32 out).  Replaces Spark's computeYtY (implicit
 * mode) behind src/als_model.py:62.  workspace: hals_gram_workspace_bytes(k). */
size_t hals_gram_workspace_bytes(int k);
int hals_gram(const float* src, int64_t n, int k, float* out, void* workspace,
              size_t workspace_bytes, void* stream);

/* Pairwise prediction: out[p] = <X[users[p]], Y[items[p]]> (fp32), NaN when the user or
 * item row is absent (present masks may be NULL = all present).  Replaces
 * ALSModel.transform at src/als_model.py:75. */
int hals_als_predict(const float* X, const float* Y, int k, const int32_t* users,
                     const int32_t* items, int64_t n, const uint8_t* user_present,
                     const uint8_t* item_present, float* out, void* stream);

/* Sum of squared errors over n (user,item,rating) triples -> *sse (double, device) and
 * *count (int64, device; pairs with both sides present).  RMSE harness for parity. */
size_t hals_als_sse_workspace_bytes(void);
int hals_als_sse(const float* X, const float* Y, int k, const int32_t* users,
                 const int32_t* items, const float* ratings, int64_t n, double* sse,
                 int64_t* count, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Batched evaluation around the hot path (SURVEY.md 8(f) rows 3, 4).
 *
 * hals_f1_at_k: F1@k of score-sorted per-user lists against the users' rated items -- compute_f1_score
 * (src/als_model.py:171-177), the weight selector of src/hybrid_system.py:42-55, for all users at once.
 *   pred_idx [n_users, pred_stride] item ids (first k entries used; -1 = no entry), actual_items sorted ascending
 *   within each user's range [actual_rowptr[u], actual_rowptr[u+1]) (duplicates count once, like a Python set).
 *   f1[u] = 2pr/(p+r), p = tp/k, r = tp/|actual|; 0 when there is nothing to match.  true_positives may be NULL.
 *
 * hals_similar_items: the cold-id fallback of src/als_model.py:79-104 for a batch of query items: cosine similarity
 * (fp64, sklearn's normalise-then-dot) of item `queries[q]` to every other item's feature row, the best three by
 * (similarity desc, position asc), of which those above 0.5 are kept; out[q] = mean of their ratings, or global_mean
 * when none qualifies (or the query is out of range).  out_neighbours ([n_queries,3], -1 padded) may be NULL.
 * ---------------------------------------------------------------------------------- */
int hals_f1_at_k(const int32_t* pred_idx, int64_t pred_stride, int k, const int64_t* actual_rowptr,
                 const int32_t* actual_items, int64_t n_users, float* f1, int32_t* true_positives, void* stream);
int hals_similar_items(const double* features /* [n_items, n_features] */, int n_features /* <= 8 */,
                       const double* ratings /* [n_items] */, int64_t n_items, const int32_t* queries,
                       int64_t n_queries, double global_mean, double* out, int32_t* out_neighbours, void* stream);

/* ------------------------------------------------------------------------------------
 * Two-tower forward.  Replaces the Keras graph built at src/two_tower_model.py:38-89 as
 * evaluated by Model.predict at src/two_tower_model.py:145.
 *   user:  LN(E_user[id])                                                  (:71-74)
 *   item:  LN(W_o . concat(E_item[id], E_manu[m], E_cat[c], relu(W_n.num+b_n)) + b_o)  (:41-64)
 * LN = Keras LayerNormalization(axis=-1, epsilon=eps): gamma*(x-mu)/sqrt(var+eps)+beta.
 * numeric is the RAW [n,2] (price, average_review_rating); num_scale/num_offset are the
 * fitted MinMaxScaler's scale_/min_ (src/two_tower_model.py:143), applied in-kernel.
 * ---------------------------------------------------------------------------------- */
typedef struct hals_tower_weights {
  int32_t embedding_size; /* E (<= 64)            */
  int32_t manu_dim;       /* 8                    */
  int32_t cat_dim;        /* 8                    */
  int32_t num_hidden;     /* 16                   */
  const float* user_emb;  /* [num_users, E]       */
  const float* item_emb;  /* [num_items, E]       */
  const float* manu_emb;  /* [num_manu, manu_dim] */
  const float* cat_emb;   /* [num_cat, cat_dim]   */
  const float* num_w;     /* [2, num_hidden]      */
  const float* num_b;     /* [num_hidden]         */
  const float* out_w;     /* [E+manu_dim+cat_dim+num_hidden, E] */
  const float* out_b;     /* [E]                  */
  const float* user_ln_g; /* [E] */
  const float* user_ln_b; /* [E] */
  const float* item_ln_g; /* [E] */
  const float* item_ln_b; /* [E] */
  float ln_eps;           /* 1e-3 (Keras default) */
  float num_scale[2];
  float num_offset[2];
  /* Rows of the four embedding tables.  An id outside [0, rows) contributes a zero embedding vector (what Keras'
   * GPU Embedding op does; its CPU op raises) instead of reading out of bounds.  0 = unknown: no check. */
  int32_t num_users, num_items, num_manufacturers, num_categories;
} hals_tower_weights;

int hals_tower_user(const hals_tower_weights* w, const int32_t* user_ids, int64_t n, float* out,
                    int64_t out_stride, void* stream);
int hals_tower_item(const hals_tower_weights* w, const int32_t* item_ids,
                    const int32_t* manufacturer_ids, const int32_t* category_ids,
                    const float* numeric /* [n,2] raw */, int64_t n, float* out,
                    int64_t out_stride, void* stream);

/* ------------------------------------------------------------------------------------
 * Hybrid scoring.  Replaces, for a batch of users at once, the per-user loop
 *   ALSModel.predict_for_user      src/als_model.py:68-91   (model.transform at :75)
 *   TwoTowerModel.predict_for_user src/two_tower_model.py:136-146 (model.predict at :145)
 *   adaptive_fusion                src/hybrid_system.py:57-75 (MinMaxScaler :66-67, blend :69-72)
 *   sorted(...)[:top_k]            src/hybrid_system.py:108
 *
 * Operands: Ua [n_users, ka], Ia [n_items, ka] (ALS factors), Ut [n_users, kt],
 * It [n_items, kt] (tower outputs), all fp32 row-major with the given row strides.
 *   s_a[u,i] = <Ua[u], Ia[i]>,  s_t[u,i] = <Ut[u], It[i]>
 *   blend[u,i] = w_a*(s_a-min_a[u])/(max_a[u]-min_a[u]) + w_t*(s_t-min_t[u])/(max_t[u]-min_t[u])
 * with a zero range contributing 0 (sklearn semantics).  Two passes, because the row
 * extrema must be known before any blend value is:
 *   1. hals_score_extrema      -> extrema[u] = (min_a, max_a, min_t, max_t) over this item shard
 *      (item-sharded runs min/max-allreduce `extrema` across ranks between the passes)
 *   2. hals_score_blend_topk   -> per-user top-k (item index int32 + blend fp32), order:
 *      blend descending, item index ascending on ties.  item_offset is added to indices
 *      (global numbering of an item shard).  The score matrix is never written to memory.
 * hals_topk_merge merges P partial lists per user ([P, n_users, k] -> [n_users, k]).
 * ---------------------------------------------------------------------------------- */
int hals_score_extrema(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride,
                       int ka, const float* Ut, int64_t ut_stride, const float* It,
                       int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                       float* extrema /* [n_users,4] */, void* workspace, size_t workspace_bytes, void* stream);

/* workspace for either entry point (pass topk = 0 for hals_score_extrema alone) */
size_t hals_score_workspace_bytes(int64_t n_users, int64_t n_items, int ka, int kt, int topk);
/* Byte offset, inside the workspace, of an int32 holding how many users of the LAST call the tensor-core
 * path could not prove exact and re-ran on the exact CUDA-core kernel; -1 when the call shape takes the
 * CUDA-core path altogether.  Diagnostic only. */
int64_t hals_score_flag_counter_offset(int64_t n_users, int64_t n_items, int ka, int kt, int topk);
int hals_score_blend_topk(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride,
                          int ka, const float* Ut, int64_t ut_stride, const float* It,
                          int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                          const float* extrema /* [n_users,4], global */, float w_als, float w_tt,
                          int topk, int32_t item_offset, int32_t* out_idx /* [n_users,topk] */,
                          float* out_score /* [n_users,topk] */, void* workspace,
                          size_t workspace_bytes, void* stream);
/* hals_score_blend_topk with a per-user exclusion set X_u (e.g. the items the user already rated), as a CSR:
 * X_u = excl_items[excl_rowptr[u] .. excl_rowptr[u+1]), u = 0 .. n_users-1 the rows of this call.  excl_rowptr values
 * are absolute offsets into excl_items, so rows [u0, u1) of a larger CSR are passed as excl_rowptr + u0.  Ids use the
 * call's global numbering (local index + item_offset), ascending within a row; duplicates are allowed, and ids outside
 * [item_offset, item_offset + n_items) are ignored (every shard of an item-sharded run can receive the same lists).
 *   - the result is the first topk items i not in X_u in the usual order (blend descending, then lower index), padded
 *     with -1 / -inf when fewer remain: the reference's `combined` with X_u removed before sorted(...)[:top_k];
 *   - the blend still uses the extrema over ALL items (hals_score_extrema is unchanged), so a kept item's score is
 *     bit-identical to its score in the call without exclusions;
 *   - both pointers NULL: exactly hals_score_blend_topk; only one NULL: HALS_ERR_INVALID.
 * Workspace: hals_score_workspace_bytes, as for hals_score_blend_topk. */
int hals_score_blend_topk_excluding(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride,
                                    int ka, const float* Ut, int64_t ut_stride, const float* It,
                                    int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                                    const float* extrema, float w_als, float w_tt, int topk, int32_t item_offset,
                                    int32_t* out_idx, float* out_score, const int64_t* excl_rowptr /* [n_users+1] */,
                                    const int32_t* excl_items, void* workspace, size_t workspace_bytes, void* stream);

int hals_topk_merge(const int32_t* part_idx, const float* part_score, int n_parts,
                    int64_t n_users, int topk, int32_t* out_idx, float* out_score, void* stream);

/* One user against a list of candidates, every score returned (the reference's
 * predict_for_user contract: a score for each item of all_items, src/als_model.py:79-88,
 * src/two_tower_model.py:146).  out[i] = <u, V[ids[i]]>; ids may be NULL (= 0..n-1). */
int hals_score_one_user(const float* u, const float* V, int64_t v_stride, int k,
                        const int32_t* ids, int64_t n, float* out, void* stream);

/* adaptive_fusion on the two aligned score lists of ONE user (src/hybrid_system.py:66-72),
 * every blended score returned (the list the reference sorts at :108 and saves at :110-111):
 *   out[i] = w_als * minmax(als)[i] + w_tt * minmax(tt)[i]
 * scratch4: 4 floats of device scratch (the two (min,max) pairs). */
int hals_fuse_lists(const float* als, const float* tt, int64_t n, float w_als, float w_tt, float* out,
                    float* scratch4, void* stream);

/* Self-test of the tcgen05 (UMMA) operand layouts: copies a caller-built shared-memory image,
 * issues n_mma tcgen05.mma instructions (M=128) with the given descriptor fields and returns
 * the TMEM accumulator as out[128][ncols].  Used only by tests/test_gpu_umma.py to pin the
 * layouts the tensor-core kernels rely on. */
int hals_debug_umma_probe(const void* img, int img_bytes, uint32_t a_off, uint32_t b_off, uint32_t a_lbo,
                          uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo, uint32_t swizzle, uint32_t idesc,
                          int n_mma, uint32_t a_step, uint32_t b_step, int kind_tf32, int ncols, float* out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HALS_B200_H_ */
