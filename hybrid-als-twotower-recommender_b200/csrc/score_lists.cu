// Hybrid scoring over per-row candidate lists (hals_score_blend_topk_lists).
//
// The reference calls get_hybrid_recommendations(user, all_items, ...) once per user (src/hybrid_system.py:95-116), so
// every user has its own candidate list, and the min-max scaling of both models spans that list alone.  Row r of a
// call owns positions [rowptr[r], rowptr[r+1]) of `cand`; each position names a row of Ia / It.
//
// One warp per row.  The user's operand rows sit in shared memory; candidates go 32 at a time: the warp copies their
// operand rows into shared memory (cp.async, coalesced along the row) and lane j computes the two dot products of
// candidate j with a sequential fmaf from 0.f -- the summation order of hals_score_one_user, so every score is
// bit-identical to the per-user path.  Pass A parks (s_a, s_t) in the workspace and keeps the row's extrema; pass B
// re-reads them (each lane its own positions), blends with blend_coef / blend_value and streams the keys through the
// topk.cuh append / compact machinery in a per-warp shared-memory buffer.
//
// Rows longer than kLsLong are cut into segments of kLsSeg positions, one warp each, so that a single huge list does
// not run on one warp: pass A per segment -> partial extrema; pass B per segment combines its row's partial extrema
// (fminf / fmaxf: exact, order-independent) and writes a partial top-k; a merge kernel sorts each long row's partial
// lists together.  The long rows and their segment slots are found on the device (lists_classify_kernel): the
// integer atomics there only assign slots, and no result depends on which slot a segment gets.
#include "common.cuh"
#include "score_common.cuh"
#include "topk.cuh"

namespace hals {

constexpr int kLsWarps = 2;       // warps per CTA (independent: no CTA-wide barrier)
constexpr int kLsChunk = 32;      // candidates staged per step (one per lane)
constexpr int64_t kLsLong = 8192; // longer rows take the segmented route
constexpr int64_t kLsSeg = 8192;  // positions per segment of a long row

struct ListArgs {
  const float* Ua; int64_t ua_stride; const float* Ia; int64_t ia_stride; int ka;
  const float* Ut; int64_t ut_stride; const float* It; int64_t it_stride; int kt;
  int64_t n_rows;
  const int64_t* rowptr; const int32_t* cand;
  const uint8_t* user_known; const uint8_t* item_known; const float* als_fallback;
  const float* row_weights; float w_als, w_tt;
  int raw, topk;
  int ld;           // shared-memory row stride (floats): ALS part at 0, tower part at ka4; ld/4 odd (conflict-free LDS.128)
  int ka4;          // ka rounded up to 4
  int wa, wt;       // cp.async width (floats: 1, 2 or 4) of the Ia / It rows
  float2* scores;   // [n_cand_total] (s_a, s_t) between pass A and pass B
};

// the segmented route's device-built tables (workspace)
struct LongArgs {
  int32_t* n_long;       // long rows found
  int32_t* n_seg;        // segment slots handed out
  int32_t* long_row;     // [n_long_max] row of each long row
  int32_t* long_slot0;   // [n_long_max] its first slot
  int32_t* long_nseg;    // [n_long_max] its number of slots
  int32_t* seg_long;     // [n_seg_max] long-row index of each slot
  float4* seg_ex;        // [n_seg_max] partial extrema
  uint64_t* seg_keys;    // [n_seg_max, topk] partial lists (sorted keys, kTopkEmpty padded)
};

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem_src));
}

__device__ __forceinline__ void copy_row(float* dst, const float* __restrict__ src, int k, int w, int lane) {
  if (w == 4) {
    for (int f = lane * 4; f < k; f += 128) cp_async16(dst + f, src + f);
  } else if (w == 2) {
    for (int f = lane * 2; f < k; f += 64) cp_async8(dst + f, src + f);
  } else {
    for (int f = lane; f < k; f += 32) cp_async4(dst + f, src + f);
  }
}

// sum_f u[f] * v[f], one fmaf per f in ascending order from 0.f (hals_score_one_user's order); u, v 16-byte aligned
__device__ __forceinline__ float dot_seq(const float* u, const float* v, int k) {
  float s = 0.f;
  int f = 0;
  for (; f + 4 <= k; f += 4) {
    const float4 a = *reinterpret_cast<const float4*>(u + f), b = *reinterpret_cast<const float4*>(v + f);
    s = fmaf(a.x, b.x, s); s = fmaf(a.y, b.y, s); s = fmaf(a.z, b.z, s); s = fmaf(a.w, b.w, s);
  }
  for (; f < k; ++f) s = fmaf(u[f], v[f], s);
  return s;
}

template <int CAP>
__host__ __device__ constexpr size_t ls_warp_bytes(int ld) { return (size_t)CAP * 8 + (size_t)(kLsChunk + 1) * ld * 4; }

// per-warp shared memory: [CAP] keys, then the user row [ld], then the staged candidate rows [32][ld]
template <int CAP>
struct WarpSmem {
  uint64_t* buf; float* urow; float* stage;
  __device__ WarpSmem(unsigned char* base, int warp, int ld) {
    unsigned char* p = base + (size_t)warp * ls_warp_bytes<CAP>(ld);
    buf = reinterpret_cast<uint64_t*>(p);
    urow = reinterpret_cast<float*>(p + (size_t)CAP * 8);
    stage = urow + ld;
  }
};

// stages row r's user operands; returns whether the user is known to ALS
__device__ __forceinline__ bool load_user(const ListArgs& A, int64_t r, float* urow, int lane) {
  const bool uk = A.user_known == nullptr || A.user_known[r] != 0;
  if (uk)
    for (int f = lane; f < A.ka; f += 32) urow[f] = A.Ua[r * A.ua_stride + f];
  for (int f = lane; f < A.kt; f += 32) urow[A.ka4 + f] = A.Ut[r * A.ut_stride + f];
  __syncwarp();
  return uk;
}

// Pass A over positions [p0, p1) of one row: parks (s_a, s_t) and returns (min_a, max_a, min_t, max_t) over the range
// (+inf, -inf, +inf, -inf when it is empty).  A cold user or item takes s_a = als_fallback[c] (predict_for_user).
__device__ float4 score_range(const ListArgs& A, bool uk, int64_t p0, int64_t p1, const float* urow, float* stage,
                              int lane) {
  const float inf = __int_as_float(0x7f800000);
  float mna = inf, mxa = -inf, mnt = inf, mxt = -inf;
  for (int64_t q = p0; q < p1; q += kLsChunk) {
    const int n = (int)min((int64_t)kLsChunk, p1 - q);
    const int32_t my_c = lane < n ? A.cand[q + lane] : 0;
    for (int j = 0; j < n; ++j) {
      const int64_t c = __shfl_sync(0xffffffffu, my_c, j);
      float* dst = stage + j * A.ld;
      if (uk) copy_row(dst, A.Ia + c * A.ia_stride, A.ka, A.wa, lane);
      copy_row(dst + A.ka4, A.It + c * A.it_stride, A.kt, A.wt, lane);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();
    if (lane < n) {
      const float* v = stage + lane * A.ld;
      const bool ik = A.item_known == nullptr || A.item_known[my_c] != 0;
      const float sa = (uk && ik) ? dot_seq(urow, v, A.ka) : A.als_fallback[my_c];
      const float st = dot_seq(urow + A.ka4, v + A.ka4, A.kt);
      A.scores[q + lane] = make_float2(sa, st);
      mna = fminf(mna, sa); mxa = fmaxf(mxa, sa);
      mnt = fminf(mnt, st); mxt = fmaxf(mxt, st);
    }
    __syncwarp();                       // every lane is done with the staged rows before the next copy
  }
  return make_float4(warp_min(mna), warp_max(mxa), warp_min(mnt), warp_max(mxt));
}

// Pass B over [p0, p1): blend the parked scores with the row's coefficients and keep the best `topk` keys (index = the
// absolute position p, so ties go to the lower list position).  Returns the key count; buf[0, count) holds them sorted.
template <int CAP>
__device__ int select_range(const ListArgs& A, int64_t r, float4 ex, int64_t p0, int64_t p1, uint64_t* buf, int lane) {
  // raw mode: identity coefficients, as hals_score_topk's raw mode
  const BlendCoef cf = blend_coef(A.raw ? make_float4(0.f, 1.f, 0.f, 1.f) : ex);
  const float wa = A.row_weights ? A.row_weights[2 * r] : A.w_als;
  const float wt = A.row_weights ? A.row_weights[2 * r + 1] : A.w_tt;
  int cnt = 0;
  uint64_t thr = kTopkEmpty;
  for (int64_t q = p0; q < p1; q += kLsChunk) {
    if (cnt + kLsChunk > CAP) cnt = topk_compact<CAP>(buf, cnt, A.topk, lane, &thr);
    const int64_t p = q + lane;
    uint64_t key = kTopkEmpty;
    if (p < p1) {
      const float2 s = A.scores[p];       // written by this lane in pass A (same position -> lane mapping)
      key = topk_key(blend_value(cf, wa, wt, s.x, s.y), (int32_t)p);
    }
    const bool pass = key > thr;
    const unsigned m = __ballot_sync(0xffffffffu, pass);
    if (pass) buf[cnt + __popc(m & ((1u << lane) - 1u))] = key;
    cnt += __popc(m);
    __syncwarp();
  }
  uint64_t t;
  return topk_compact<CAP>(buf, cnt, A.topk, lane, &t);
}

__device__ __forceinline__ void write_keys(const uint64_t* keys, int count, int topk, int32_t* oi, float* os, int lane) {
  for (int e = lane; e < topk; e += 32) {
    const bool ok = e < count && keys[e] != kTopkEmpty;
    oi[e] = ok ? topk_key_index(keys[e]) : -1;
    os[e] = ok ? topk_key_score(keys[e]) : -__int_as_float(0x7f800000);
  }
}

// one warp per row of at most kLsLong positions (longer rows are left to the segmented route)
template <int CAP>
__global__ void __maxnreg__(128)
lists_rows_kernel(ListArgs A, int32_t* __restrict__ out_pos, float* __restrict__ out_score) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r = (int64_t)blockIdx.x * kLsWarps + warp;
  if (r >= A.n_rows) return;                                   // warp-uniform
  const int64_t p0 = A.rowptr[r], p1 = A.rowptr[r + 1];
  if (p1 - p0 > kLsLong) return;
  WarpSmem<CAP> S(smem_raw, warp, A.ld);
  const bool uk = load_user(A, r, S.urow, lane);
  const float4 ex = score_range(A, uk, p0, p1, S.urow, S.stage, lane);
  const int c = select_range<CAP>(A, r, ex, p0, p1, S.buf, lane);
  write_keys(S.buf, c, A.topk, out_pos + r * A.topk, out_score + r * A.topk, lane);
}

// Finds the long rows and hands each a contiguous range of segment slots.
__global__ void lists_classify_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows, LongArgs L) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t len = rowptr[r + 1] - rowptr[r];
    if (len <= kLsLong) continue;
    const int nseg = (int)((len + kLsSeg - 1) / kLsSeg);
    const int li = atomicAdd(L.n_long, 1);
    const int s0 = atomicAdd(L.n_seg, nseg);
    L.long_row[li] = (int32_t)r; L.long_slot0[li] = s0; L.long_nseg[li] = nseg;
    for (int j = 0; j < nseg; ++j) L.seg_long[s0 + j] = li;
  }
}

// Segmented route, one warp per segment slot (persistent over the device-side slot count).
//   SELECT = false: pass A of the segment -> seg_ex[slot]
//   SELECT = true:  the row's extrema from all its segments, then pass B of the segment -> seg_keys[slot]
template <int CAP, bool SELECT>
__global__ void __maxnreg__(128) lists_seg_kernel(ListArgs A, LongArgs L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpSmem<CAP> S(smem_raw, warp, SELECT ? 0 : A.ld);
  const int n_seg = *L.n_seg;
  for (int s = blockIdx.x * kLsWarps + warp; s < n_seg; s += gridDim.x * kLsWarps) {
    const int li = L.seg_long[s];
    const int64_t r = L.long_row[li];
    const int s0 = L.long_slot0[li];
    const int64_t p0 = A.rowptr[r] + (int64_t)(s - s0) * kLsSeg, p1 = min(A.rowptr[r + 1], p0 + kLsSeg);
    if (!SELECT) {
      const bool uk = load_user(A, r, S.urow, lane);
      const float4 ex = score_range(A, uk, p0, p1, S.urow, S.stage, lane);
      if (lane == 0) L.seg_ex[s] = ex;
      __syncwarp();
    } else {
      const float inf = __int_as_float(0x7f800000);
      float4 ex = make_float4(inf, -inf, inf, -inf);
      for (int j = s0; j < s0 + L.long_nseg[li]; ++j) {
        const float4 e = L.seg_ex[j];
        ex.x = fminf(ex.x, e.x); ex.y = fmaxf(ex.y, e.y); ex.z = fminf(ex.z, e.z); ex.w = fmaxf(ex.w, e.w);
      }
      const int c = select_range<CAP>(A, r, ex, p0, p1, S.buf, lane);
      uint64_t* out = L.seg_keys + (size_t)s * A.topk;
      for (int e = lane; e < A.topk; e += 32) out[e] = e < c ? S.buf[e] : kTopkEmpty;
      __syncwarp();
    }
  }
}

// One warp per long row: its partial lists go through the same register bitonic merge as topk_merge_kernel (slots
// [0, topk) hold the running best, [CAP/2, CAP/2 + topk) receive the next list).
template <int CAP>
__global__ void lists_merge_kernel(LongArgs L, int topk, int32_t* __restrict__ out_pos, float* __restrict__ out_score) {
  constexpr int R = CAP / 32;
  const int lane = threadIdx.x & 31;
  const int n_long = *L.n_long;
  for (int li = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); li < n_long; li += (int)((gridDim.x * blockDim.x) >> 5)) {
    uint64_t v[R];
#pragma unroll
    for (int q = 0; q < R; ++q) v[q] = kTopkEmpty;
    const int s0 = L.long_slot0[li], ns = L.long_nseg[li];
    for (int s = s0; s < s0 + ns; ++s) {
      const uint64_t* part = L.seg_keys + (size_t)s * topk;
#pragma unroll
      for (int q = 0; q < R; ++q) {
        const int e = q * 32 + lane;
        if (e >= CAP / 2) v[q] = (e - CAP / 2 < topk) ? part[e - CAP / 2] : kTopkEmpty;
        else if (e >= topk) v[q] = kTopkEmpty;
      }
      warp_bitonic_desc<R>(v, lane);
    }
    const int64_t r = L.long_row[li];
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const int e = q * 32 + lane;
      if (e < topk) {
        const bool ok = v[q] != kTopkEmpty;
        out_pos[r * topk + e] = ok ? topk_key_index(v[q]) : -1;
        out_score[r * topk + e] = ok ? topk_key_score(v[q]) : -__int_as_float(0x7f800000);
      }
    }
  }
}

// workspace layout (every block 256-byte aligned)
struct ListsLayout {
  size_t scores, counters, long_row, long_slot0, long_nseg, seg_long, seg_ex, seg_keys, total;
  int64_t n_long_max, n_seg_max;
  ListsLayout(int64_t n_cand_total, int topk) {
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const bool segmented = n_cand_total > kLsLong;
    n_long_max = segmented ? n_cand_total / (kLsLong + 1) : 0;
    n_seg_max = segmented ? n_cand_total / kLsSeg + n_long_max : 0;   // sum of ceil(len / kLsSeg) over the long rows
    size_t o = 0;
    scores = o;     o += up((size_t)n_cand_total * sizeof(float2));
    counters = o;   o += segmented ? 256 : 0;
    long_row = o;   o += up((size_t)n_long_max * 4);
    long_slot0 = o; o += up((size_t)n_long_max * 4);
    long_nseg = o;  o += up((size_t)n_long_max * 4);
    seg_long = o;   o += up((size_t)n_seg_max * 4);
    seg_ex = o;     o += up((size_t)n_seg_max * sizeof(float4));
    seg_keys = o;   o += up((size_t)n_seg_max * topk * sizeof(uint64_t));
    total = o + 256;
  }
};

static int copy_width(const float* p, int64_t stride, int k) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  if (a % 16 == 0 && stride % 4 == 0 && k % 4 == 0) return 4;
  if (a % 8 == 0 && stride % 2 == 0 && k % 2 == 0) return 2;
  return 1;
}

template <int CAP>
static int launch_lists(const ListArgs& A, const ListsLayout& Lo, unsigned char* ws, int32_t* out_pos, float* out_score,
                        cudaStream_t st) {
  const size_t smem = kLsWarps * ls_warp_bytes<CAP>(A.ld);
  HALS_CUDA(cudaFuncSetAttribute(lists_rows_kernel<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  lists_rows_kernel<CAP><<<(unsigned)((A.n_rows + kLsWarps - 1) / kLsWarps), kLsWarps * 32, smem, st>>>(A, out_pos, out_score);
  HALS_LAUNCH_CHECK();
  if (Lo.n_long_max == 0) return 0;                           // no row can be longer than kLsLong
  LongArgs L{reinterpret_cast<int32_t*>(ws + Lo.counters), reinterpret_cast<int32_t*>(ws + Lo.counters) + 1,
             reinterpret_cast<int32_t*>(ws + Lo.long_row), reinterpret_cast<int32_t*>(ws + Lo.long_slot0),
             reinterpret_cast<int32_t*>(ws + Lo.long_nseg), reinterpret_cast<int32_t*>(ws + Lo.seg_long),
             reinterpret_cast<float4*>(ws + Lo.seg_ex), reinterpret_cast<uint64_t*>(ws + Lo.seg_keys)};
  HALS_CUDA(cudaMemsetAsync(L.n_long, 0, 2 * sizeof(int32_t), st));
  int64_t cb = (A.n_rows + 255) / 256;
  if (cb > 4 * sm_count()) cb = 4 * sm_count();
  lists_classify_kernel<<<(unsigned)cb, 256, 0, st>>>(A.rowptr, A.n_rows, L);
  HALS_LAUNCH_CHECK();
  int64_t sb = (Lo.n_seg_max + kLsWarps - 1) / kLsWarps;
  if (sb > 8 * sm_count()) sb = 8 * sm_count();
  HALS_CUDA(cudaFuncSetAttribute(lists_seg_kernel<CAP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  lists_seg_kernel<CAP, false><<<(unsigned)sb, kLsWarps * 32, smem, st>>>(A, L);
  HALS_LAUNCH_CHECK();
  lists_seg_kernel<CAP, true><<<(unsigned)sb, kLsWarps * 32, kLsWarps * ls_warp_bytes<CAP>(0), st>>>(A, L);
  HALS_LAUNCH_CHECK();
  int64_t mb = (Lo.n_long_max + 3) / 4;
  if (mb > 4 * sm_count()) mb = 4 * sm_count();
  lists_merge_kernel<CAP><<<(unsigned)mb, 128, 0, st>>>(L, A.topk, out_pos, out_score);
  HALS_LAUNCH_CHECK();
  return 0;
}

}  // namespace hals

using namespace hals;

extern "C" size_t hals_score_lists_workspace_bytes(int64_t n_cand_total, int topk) {
  if (n_cand_total < 0 || topk < 1 || topk > 256) return 0;
  return ListsLayout(n_cand_total, topk).total;
}

extern "C" int hals_score_blend_topk_lists(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride, int ka,
                                           const float* Ut, int64_t ut_stride, const float* It, int64_t it_stride, int kt,
                                           int64_t n_rows, int64_t n_cand_total, const int64_t* cand_rowptr,
                                           const int32_t* cand, const uint8_t* user_known, const uint8_t* item_known,
                                           const float* als_fallback, const float* row_weights, float w_als, float w_tt,
                                           int raw, int topk, int32_t* out_pos, float* out_score, void* workspace,
                                           size_t workspace_bytes, void* stream) {
  // every check comes before the first CUDA call
  HALS_REQUIRE(topk >= 1 && topk <= 256, "topk must be in [1,256]");
  if (int rc = check_score_args(Ua, Ia, ka, Ut, It, kt, n_rows, n_cand_total)) return rc;
  HALS_REQUIRE(n_cand_total <= INT32_MAX, "n_cand_total must fit the int32 positions of out_pos");
  HALS_REQUIRE(cand_rowptr && out_pos && out_score && workspace, "null pointer");
  HALS_REQUIRE(cand || n_cand_total == 0, "null pointer");
  HALS_REQUIRE(als_fallback || (!user_known && !item_known), "user_known / item_known need als_fallback");
  const ListsLayout Lo(n_cand_total, topk);
  if (workspace_bytes < Lo.total) return fail(HALS_ERR_WORKSPACE, "%s: workspace too small", __func__);
  if (n_rows == 0) return 0;
  unsigned char* ws = reinterpret_cast<unsigned char*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  ListArgs A{Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt, n_rows, cand_rowptr, cand,
             user_known, item_known, als_fallback, row_weights, w_als, w_tt, raw != 0, topk, 0, 0, 1, 1,
             reinterpret_cast<float2*>(ws + Lo.scores)};
  A.ka4 = (ka + 3) & ~3;
  A.ld = A.ka4 + ((kt + 3) & ~3);
  if ((A.ld / 4) % 2 == 0) A.ld += 4;
  if (ka) A.wa = copy_width(Ia, ia_stride, ka);
  if (kt) A.wt = copy_width(It, it_stride, kt);
  cudaStream_t st = (cudaStream_t)stream;
  const int cap = topk_capacity(topk);
  if (cap == 128) return launch_lists<128>(A, Lo, ws, out_pos, out_score, st);
  if (cap == 256) return launch_lists<256>(A, Lo, ws, out_pos, out_score, st);
  return launch_lists<512>(A, Lo, ws, out_pos, out_score, st);
}
