// Hybrid scoring, exact-fp32 CUDA-core path (any ka <= 128, kt <= 64, topk <= 256).
//
// Batched replacement of the reference's per-user scoring loop:
//   ALS scores      src/als_model.py:75        s_a[u,i] = <Ua[u], Ia[i]>
//   tower scores    src/two_tower_model.py:145  s_t[u,i] = <Ut[u], It[i]>
//   MinMax + blend  src/hybrid_system.py:66-72
//   top-k           src/hybrid_system.py:108
// A CTA owns 64 users and walks a contiguous range of items in tiles of 64; both score
// tiles live in registers (4x4 per thread), are blended in registers and filtered against
// the per-row threshold; nothing but the per-row candidate buffers reaches memory.
// Pass 1 (EXTREMA) keeps per-row min/max of both models instead.
// The tensor-core path (score_tc.cu) uses this kernel's epilogue machinery and is checked
// against it; this path is also the exact fallback for shapes the TC path does not take.
#include "common.cuh"
#include "score_common.cuh"
#include "topk.cuh"

namespace hals {

constexpr int kScThreads = 256;
constexpr int kScUsers = 64;
constexpr int kScItems = 64;

struct ScoreArgs {
  const float* Ua; int64_t ua_stride;
  const float* Ia; int64_t ia_stride;
  const float* Ut; int64_t ut_stride;
  const float* It; int64_t it_stride;
  int ka, kt;
  int64_t n_users, n_items;
  int64_t items_per_split;
  // optional indirection (exact re-run of flagged users after the tensor-core path): the kernel then
  // walks user_list[0 .. *user_count) instead of 0 .. n_users, looping over tiles persistently
  const int32_t* user_list;
  const int32_t* user_count;
  // list mode: positions [list_begin, min(*user_count, list_end)) are handled by this launch; candidate /
  // partial-list rows are addressed by (split, position - list_begin) with `row_stride` rows per split
  int64_t list_begin, list_end, row_stride;
};

__device__ __forceinline__ void atomic_min_f32(float* addr, float v) {
  // order-independent => deterministic
  int* a = reinterpret_cast<int*>(addr);
  int old = *a;
  while (__int_as_float(old) > v) {
    const int assumed = old;
    old = atomicCAS(a, assumed, __float_as_int(v));
    if (old == assumed) break;
  }
}
__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
  int* a = reinterpret_cast<int*>(addr);
  int old = *a;
  while (__int_as_float(old) < v) {
    const int assumed = old;
    old = atomicCAS(a, assumed, __float_as_int(v));
    if (old == assumed) break;
  }
}

__global__ void extrema_init_kernel(float* extrema, int64_t n_users) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u < n_users) {
    const float inf = __int_as_float(0x7f800000);
    reinterpret_cast<float4*>(extrema)[u] = make_float4(inf, -inf, inf, -inf);
  }
}

// true when the ascending list items[lo, hi) holds v
__device__ __forceinline__ bool sorted_contains(const int32_t* __restrict__ items, int64_t lo, int64_t hi, int32_t v) {
  const int64_t end = hi;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (items[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo < end && items[lo] == v;
}

// EXCL: items listed for a user in the exclusion CSR (excl_rowptr indexed by the user -- uid(r), not the tile row --,
// global item ids) never pass the filter; the lookup runs only for items that already beat the row threshold.
template <bool EXTREMA, int CAP, bool EXCL = false>
__global__ void __launch_bounds__(kScThreads)
score_simt_kernel(ScoreArgs A, float* __restrict__ extrema_out, const float* __restrict__ extrema_in,
                  float w_als, float w_tt, int topk, int32_t item_offset,
                  uint64_t* __restrict__ cand /* [splits][n_users][CAP] */,
                  int32_t* __restrict__ out_idx, float* __restrict__ out_score /* [splits][n_users][topk] */,
                  const int64_t* __restrict__ excl_rowptr = nullptr, const int32_t* __restrict__ excl_items = nullptr) {
  static_assert(!EXCL || !EXTREMA, "exclusion lists apply to the top-k pass");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = A.ka + A.kt;
  const int LD = K + 1;
  float* Us = reinterpret_cast<float*>(smem_raw);            // [64][LD]
  float* Is = Us + kScUsers * LD;                            // [64][LD]
  float* St = Is + kScItems * LD;                            // [64][65] blended tile (top-k pass)
  float* rowstat = St + kScUsers * 65;                       // [64][4]: extrema or coefficients
  __shared__ int cnt[kScUsers];
  __shared__ unsigned long long thr[kScUsers];
  __shared__ int64_t xrow[EXCL ? kScUsers : 1][2];            // EXCL: [begin, end) of each row's exclusion list

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int lane = tid & 31, warp = tid >> 5;
  const int split = blockIdx.y;
  const int64_t n_rows = A.user_list ? min((int64_t)*A.user_count, A.list_end) : A.n_users;
  const int64_t row_base = A.user_list ? A.list_begin : 0;
  const int64_t row_stride = A.user_list ? A.row_stride : A.n_users;
  const bool by_pos = A.user_list != nullptr && gridDim.y > 1;   // partial lists addressed by list position
  for (int64_t u0 = row_base + (int64_t)blockIdx.x * kScUsers; u0 < n_rows; u0 += (int64_t)gridDim.x * kScUsers) {
  __syncthreads();
  // row r of this tile is user uid(r); rows beyond n_rows are padding
  auto uid = [&](int r) -> int64_t { return A.user_list ? (int64_t)A.user_list[min(u0 + r, n_rows - 1)] : u0 + r; };
  const int64_t i_begin = (int64_t)split * A.items_per_split;
  const int64_t i_end = min(A.n_items, i_begin + A.items_per_split);

  // stage the user tile (both models side by side), zero rows beyond n_users
  for (int e = tid; e < kScUsers * K; e += kScThreads) {
    const int r = e / K, f = e - r * K;
    const int64_t u = uid(r);
    float v = 0.f;
    if (u0 + r < n_rows) v = f < A.ka ? A.Ua[u * A.ua_stride + f] : A.Ut[u * A.ut_stride + (f - A.ka)];
    Us[r * LD + f] = v;
  }
  if (tid < kScUsers) {
    cnt[tid] = 0;
    thr[tid] = kTopkEmpty;
    const int64_t u = uid(tid);
    if (EXCL && u0 + tid < n_rows) { xrow[tid][0] = excl_rowptr[u]; xrow[tid][1] = excl_rowptr[u + 1]; }
    float4 ex;
    if (EXTREMA) {
      const float inf = __int_as_float(0x7f800000);
      ex = make_float4(inf, -inf, inf, -inf);
    } else {
      // padding rows, and every row in raw mode (extrema_in == NULL: hals_score_topk), take the identity coefficients
      ex = (u0 + tid < n_rows && extrema_in) ? reinterpret_cast<const float4*>(extrema_in)[u] : make_float4(0, 1, 0, 1);
      const BlendCoef c = blend_coef(ex);
      ex = make_float4(c.min_a, c.sc_a, c.min_t, c.sc_t);
    }
    reinterpret_cast<float4*>(rowstat)[tid] = ex;
  }
  uint64_t* mycand = EXTREMA ? nullptr : cand + ((size_t)split * row_stride + (u0 - row_base)) * CAP;

  for (int64_t it0 = i_begin; it0 < i_end; it0 += kScItems) {
    __syncthreads();
    for (int e = tid; e < kScItems * K; e += kScThreads) {
      const int r = e / K, f = e - r * K;
      const int64_t i = it0 + r;
      float v = 0.f;
      if (i < i_end) v = f < A.ka ? A.Ia[i * A.ia_stride + f] : A.It[i * A.it_stride + (f - A.ka)];
      Is[r * LD + f] = v;
    }
    __syncthreads();

    float sa[4][4], st[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { sa[i][j] = 0.f; st[i][j] = 0.f; }
    for (int f = 0; f < A.ka; ++f) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = Us[(ty + 16 * i) * LD + f]; b[i] = Is[(tx + 16 * i) * LD + f]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) sa[i][j] = fmaf(a[i], b[j], sa[i][j]);
    }
    for (int f = A.ka; f < K; ++f) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = Us[(ty + 16 * i) * LD + f]; b[i] = Is[(tx + 16 * i) * LD + f]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) st[i][j] = fmaf(a[i], b[j], st[i][j]);
    }

    if (EXTREMA) {
      const float inf = __int_as_float(0x7f800000);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float mna = inf, mxa = -inf, mnt = inf, mxt = -inf;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (it0 + tx + 16 * j < i_end) {
            mna = fminf(mna, sa[i][j]); mxa = fmaxf(mxa, sa[i][j]);
            mnt = fminf(mnt, st[i][j]); mxt = fmaxf(mxt, st[i][j]);
          }
        }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {  // across the 16 tx lanes of this user row
          mna = fminf(mna, __shfl_xor_sync(0xffffffffu, mna, o));
          mxa = fmaxf(mxa, __shfl_xor_sync(0xffffffffu, mxa, o));
          mnt = fminf(mnt, __shfl_xor_sync(0xffffffffu, mnt, o));
          mxt = fmaxf(mxt, __shfl_xor_sync(0xffffffffu, mxt, o));
        }
        if (tx == 0) {  // rows ty+16i are owned by exactly one thread with tx == 0
          float* rs = rowstat + (ty + 16 * i) * 4;
          rs[0] = fminf(rs[0], mna); rs[1] = fmaxf(rs[1], mxa);
          rs[2] = fminf(rs[2], mnt); rs[3] = fmaxf(rs[3], mxt);
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 cf = reinterpret_cast<const float4*>(rowstat)[ty + 16 * i];
        BlendCoef c; c.min_a = cf.x; c.sc_a = cf.y; c.min_t = cf.z; c.sc_t = cf.w;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          St[(ty + 16 * i) * 65 + tx + 16 * j] = blend_value(c, w_als, w_tt, sa[i][j], st[i][j]);
      }
      __syncthreads();
      // warp w filters rows w*8 .. w*8+7; it is the only writer of those rows' buffers
      for (int rr = 0; rr < 8; ++rr) {
        const int r = warp * 8 + rr;
        if (u0 + r >= n_rows) break;
        uint64_t* buf = mycand + (size_t)r * CAP;
        int c = cnt[r];
        uint64_t t = thr[r];
        if (c + kScItems > CAP) {
          c = topk_compact<CAP>(buf, c, topk, lane, &t);
        }
        const int64_t xlo = EXCL ? xrow[r][0] : 0, xhi = EXCL ? xrow[r][1] : 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int col = lane + 32 * h;
          const int64_t i = it0 + col;
          const float s = St[r * 65 + col];
          const uint64_t key = topk_key(s, (int32_t)(i + item_offset));
          const bool pass = (i < i_end) && (key > t) &&
                            !(EXCL && sorted_contains(excl_items, xlo, xhi, (int32_t)(i + item_offset)));
          const unsigned m = __ballot_sync(0xffffffffu, pass);
          if (pass) buf[c + __popc(m & ((1u << lane) - 1u))] = key;
          c += __popc(m);
        }
        __syncwarp();
        if (lane == 0) { cnt[r] = c; thr[r] = t; }
      }
    }
  }

  __syncthreads();
  if (EXTREMA) {
    if (tid < kScUsers && u0 + tid < n_rows && i_end > i_begin) {
      const float* rs = rowstat + tid * 4;
      float* ex = extrema_out + uid(tid) * 4;
      if (gridDim.y == 1) {
        reinterpret_cast<float4*>(ex)[0] = make_float4(rs[0], rs[1], rs[2], rs[3]);
      } else {
        atomic_min_f32(ex + 0, rs[0]); atomic_max_f32(ex + 1, rs[1]);
        atomic_min_f32(ex + 2, rs[2]); atomic_max_f32(ex + 3, rs[3]);
      }
    }
  } else {
    for (int rr = 0; rr < 8; ++rr) {
      const int r = warp * 8 + rr;
      if (u0 + r >= n_rows) break;
      const int64_t u = uid(r);
      uint64_t* buf = mycand + (size_t)r * CAP;
      uint64_t t;
      const int c = topk_compact<CAP>(buf, cnt[r], topk, lane, &t);
      const size_t orow = by_pos ? (size_t)split * row_stride + (size_t)(u0 - row_base + r) : (size_t)split * A.n_users + u;
      int32_t* oi = out_idx + orow * topk;
      float* os = out_score + orow * topk;
      for (int e = lane; e < topk; e += 32) {
        if (e < c) {
          const uint64_t key = buf[e];
          oi[e] = topk_key_index(key);
          os[e] = topk_key_score(key);
        } else {
          oi[e] = -1;
          os[e] = -__int_as_float(0x7f800000);
        }
      }
    }
  }
  }  // tile loop
}

// Merge P partial lists per user: one warp per user streams P*topk keys through the same
// append/compact machinery (registers only).
template <int CAP>
__global__ void topk_merge_kernel(const int32_t* __restrict__ part_idx, const float* __restrict__ part_score,
                                  int n_parts, int64_t n_users, int topk, int32_t* __restrict__ out_idx,
                                  float* __restrict__ out_score, const int32_t* __restrict__ user_list = nullptr,
                                  const int32_t* __restrict__ user_count = nullptr, int64_t list_begin = 0,
                                  int64_t list_end = 0) {
  constexpr int R = CAP / 32;
  const int lane = threadIdx.x & 31;
  // plain mode: row u of the [P][n_users] partial arrays -> out[u].  list mode: partial row = list position
  // (relative to list_begin, n_users rows per part), destination = user_list[position].
  int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int64_t dst_row = u;
  if (user_list != nullptr) {
    const int64_t n = min((int64_t)*user_count, list_end) - list_begin;
    if (u >= n) return;
    dst_row = user_list[list_begin + u];
  }
  if (u >= n_users) return;
  uint64_t v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) v[r] = kTopkEmpty;
  // slots [0, topk) hold the running best, slots [CAP/2, CAP/2 + topk) receive the next list
  for (int p = 0; p < n_parts; ++p) {
    const int32_t* pi = part_idx + ((size_t)p * n_users + u) * topk;
    const float* ps = part_score + ((size_t)p * n_users + u) * topk;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int e = r * 32 + lane;
      if (e >= CAP / 2) {
        const int q = e - CAP / 2;
        uint64_t key = kTopkEmpty;
        if (q < topk) {
          const int32_t idx = pi[q];
          if (idx >= 0) key = topk_key(ps[q], idx);
        }
        v[r] = key;
      } else if (e >= topk) {
        v[r] = kTopkEmpty;
      }
    }
    warp_bitonic_desc<R>(v, lane);
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int e = r * 32 + lane;
    if (e < topk) {
      const bool ok = v[r] != kTopkEmpty;
      out_idx[dst_row * topk + e] = ok ? topk_key_index(v[r]) : -1;
      out_score[dst_row * topk + e] = ok ? topk_key_score(v[r]) : -__int_as_float(0x7f800000);
    }
  }
}

__global__ void score_one_user_kernel(const float* __restrict__ u, const float* __restrict__ V,
                                      int64_t v_stride, int k, const int32_t* __restrict__ ids, int64_t n,
                                      float* __restrict__ out) {
  extern __shared__ float us[];
  for (int f = threadIdx.x; f < k; f += blockDim.x) us[f] = u[f];
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = ids ? (int64_t)ids[i] : i;
    const float* v = V + row * v_stride;
    float s = 0.f;
    for (int f = 0; f < k; ++f) s = fmaf(us[f], v[f], s);
    out[i] = s;
  }
}

__global__ void list_extrema_kernel(const float* __restrict__ a, const float* __restrict__ t, int64_t n,
                                    float* __restrict__ ex) {
  const float inf = __int_as_float(0x7f800000);
  float mna = inf, mxa = -inf, mnt = inf, mxt = -inf;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float x = a[i], y = t[i];
    mna = fminf(mna, x); mxa = fmaxf(mxa, x); mnt = fminf(mnt, y); mxt = fmaxf(mxt, y);
  }
  mna = warp_min(mna); mxa = warp_max(mxa); mnt = warp_min(mnt); mxt = warp_max(mxt);
  if ((threadIdx.x & 31) == 0) {
    atomic_min_f32(ex + 0, mna); atomic_max_f32(ex + 1, mxa);
    atomic_min_f32(ex + 2, mnt); atomic_max_f32(ex + 3, mxt);
  }
}
__global__ void list_blend_kernel(const float* __restrict__ a, const float* __restrict__ t, int64_t n,
                                  const float* __restrict__ ex, float wa, float wt, float* __restrict__ out) {
  const BlendCoef c = blend_coef(*reinterpret_cast<const float4*>(ex));
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = blend_value(c, wa, wt, a[i], t[i]);
}

static size_t score_smem_bytes(int K) {
  return sizeof(float) * ((size_t)(kScUsers + kScItems) * (K + 1) + kScUsers * 65 + kScUsers * 4);
}

// how many item splits to use so that few-user calls still fill the GPU
static int score_splits(int64_t n_users, int64_t n_items) {
  const int64_t user_tiles = (n_users + kScUsers - 1) / kScUsers;
  const int64_t item_tiles = (n_items + kScItems - 1) / kScItems;
  int64_t want = (2 * (int64_t)sm_count() + user_tiles - 1) / user_tiles;
  if (want > item_tiles) want = item_tiles;
  if (want > 1024) want = 1024;
  if (want < 1) want = 1;
  return (int)want;
}

}  // namespace hals

using namespace hals;

int check_score_args(const float* Ua, const float* Ia, int ka, const float* Ut, const float* It, int kt,
                            int64_t n_users, int64_t n_items) {
  HALS_REQUIRE(ka >= 0 && ka <= 128 && kt >= 0 && kt <= 64 && ka + kt > 0, "ka must be <= 128 and kt <= 64");
  HALS_REQUIRE((ka == 0 || (Ua && Ia)) && (kt == 0 || (Ut && It)), "null operand");
  HALS_REQUIRE(n_users >= 0 && n_items >= 0, "negative size");
  return 0;
}

namespace hals {

size_t score_simt_workspace_bytes(int64_t n_users, int64_t n_items, int topk) {
  const int splits = score_splits(n_users, n_items);
  const size_t cap = topk_capacity(topk);
  size_t b = (size_t)splits * n_users * cap * sizeof(uint64_t);             // candidate buffers
  b += (size_t)splits * n_users * topk * (sizeof(int32_t) + sizeof(float));  // partial lists
  return b + 256;
}

// rows / splits of the list-mode (exact re-run) launches
static int64_t list_rows(int64_t n_users) { return n_users < 2048 ? n_users : 2048; }
static int list_splits(int64_t n_items) {
  int64_t t = (n_items + kScItems - 1) / kScItems;
  if (t > 64) t = 64;
  return (int)(t < 1 ? 1 : t);
}

size_t score_simt_list_workspace_bytes(int64_t n_users, int64_t n_items, int topk) {
  const size_t rows = (size_t)list_rows(n_users) * list_splits(n_items);
  return rows * topk_capacity(topk) * sizeof(uint64_t) + rows * topk * 8 + 256;
}

static void fill_split(ScoreArgs& A, int64_t n_items, int splits) {
  const int64_t tiles = (n_items + kScItems - 1) / kScItems;
  A.items_per_split = ((tiles + splits - 1) / splits) * kScItems;
  if (A.items_per_split == 0) A.items_per_split = kScItems;
}

// Exact extrema.  With a user list (device list + device count) only the listed users are recomputed
// (item-split, combined with order-independent atomic min/max); their rows must have been reset to
// (+inf,-inf,+inf,-inf) beforehand (score_flag_list_kernel does it) and every other row is left alone.
int score_extrema_simt(const ScoreOperands& O, int64_t n_users, int64_t n_items, float* extrema,
                       const int32_t* user_list, const int32_t* user_count, cudaStream_t st) {
  ScoreArgs A{O.Ua, O.ua_stride, O.Ia, O.ia_stride, O.Ut, O.ut_stride, O.It, O.it_stride, O.ka, O.kt,
              n_users, n_items, 0, user_list, user_count, 0, n_users, n_users};
  const bool listed = user_list != nullptr;
  if (!listed) {
    extrema_init_kernel<<<(unsigned)((n_users + 255) / 256), 256, 0, st>>>(extrema, n_users);
    HALS_LAUNCH_CHECK();
    if (n_items == 0) return 0;
  }
  // list mode re-runs a handful of users (typically one or two 64-user tiles): the item range is cut finely enough
  // to occupy the whole GPU -- extrema combine through order-independent atomic min/max, so splits cost nothing
  int splits = score_splits(n_users, n_items);
  if (listed) {
    const int64_t tiles = (n_items + kScItems - 1) / kScItems;
    int64_t s = 4 * (int64_t)sm_count();
    if (s > tiles) s = tiles;
    splits = (int)(s < 2 ? 2 : s);
  }
  fill_split(A, n_items, splits);
  const size_t smem = score_smem_bytes(O.ka + O.kt);
  HALS_CUDA(cudaFuncSetAttribute(score_simt_kernel<true, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t gx = (n_users + kScUsers - 1) / kScUsers;
  if (listed && gx > 8) gx = 8;                   // persistent over the (device-side) list length
  dim3 grid((unsigned)gx, (unsigned)splits);
  score_simt_kernel<true, 128><<<grid, kScThreads, smem, st>>>(A, extrema, nullptr, 0.f, 0.f, 0, 0, nullptr,
                                                                 nullptr, nullptr);
  HALS_LAUNCH_CHECK();
  return 0;
}

template <int CAPV, bool EXCL>
static int launch_simt_topk(const ScoreArgs& A, dim3 grid, size_t smem, const float* extrema, float w_als, float w_tt,
                            int topk, int32_t item_offset, uint64_t* cand, int32_t* oi, float* os,
                            const int64_t* excl_rowptr, const int32_t* excl_items, cudaStream_t st) {
  HALS_CUDA(cudaFuncSetAttribute(score_simt_kernel<false, CAPV, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  score_simt_kernel<false, CAPV, EXCL><<<grid, kScThreads, smem, st>>>(A, nullptr, extrema, w_als, w_tt, topk, item_offset,
                                                                       cand, oi, os, excl_rowptr, excl_items);
  HALS_LAUNCH_CHECK();
  return 0;
}
template <int CAPV>
static int launch_simt_topk_excl(const ScoreArgs& A, dim3 grid, size_t smem, const float* extrema, float w_als, float w_tt,
                                 int topk, int32_t item_offset, uint64_t* cand, int32_t* oi, float* os,
                                 const int64_t* excl_rowptr, const int32_t* excl_items, cudaStream_t st) {
  if (excl_rowptr != nullptr)
    return launch_simt_topk<CAPV, true>(A, grid, smem, extrema, w_als, w_tt, topk, item_offset, cand, oi, os, excl_rowptr,
                                        excl_items, st);
  return launch_simt_topk<CAPV, false>(A, grid, smem, extrema, w_als, w_tt, topk, item_offset, cand, oi, os, nullptr, nullptr, st);
}
static int launch_simt_topk_cap(int cap, const ScoreArgs& A, dim3 grid, size_t smem, const float* extrema, float w_als,
                                float w_tt, int topk, int32_t item_offset, uint64_t* cand, int32_t* oi, float* os,
                                const int64_t* xr, const int32_t* xi, cudaStream_t st) {
  if (cap == 128) return launch_simt_topk_excl<128>(A, grid, smem, extrema, w_als, w_tt, topk, item_offset, cand, oi, os, xr, xi, st);
  if (cap == 256) return launch_simt_topk_excl<256>(A, grid, smem, extrema, w_als, w_tt, topk, item_offset, cand, oi, os, xr, xi, st);
  return launch_simt_topk_excl<512>(A, grid, smem, extrema, w_als, w_tt, topk, item_offset, cand, oi, os, xr, xi, st);
}

int score_blend_topk_simt(const ScoreOperands& O, int64_t n_users, int64_t n_items, const float* extrema,
                          float w_als, float w_tt, int topk, int32_t item_offset, int32_t* out_idx,
                          float* out_score, void* workspace, const int32_t* user_list, const int32_t* user_count,
                          const int64_t* excl_rowptr, const int32_t* excl_items, cudaStream_t st) {
  const int cap = topk_capacity(topk);
  const size_t smem = score_smem_bytes(O.ka + O.kt);
  ScoreArgs A{O.Ua, O.ua_stride, O.Ia, O.ia_stride, O.Ut, O.ut_stride, O.It, O.it_stride, O.ka, O.kt,
              n_users, n_items, 0, user_list, user_count, 0, n_users, n_users};
  if (user_list == nullptr) {
    const int splits = score_splits(n_users, n_items);
    fill_split(A, n_items, splits);
    uint64_t* cand = (uint64_t*)workspace;
    int32_t* pidx = (int32_t*)(cand + (size_t)splits * n_users * cap);
    float* pscore = (float*)(pidx + (size_t)splits * n_users * topk);
    dim3 grid((unsigned)((n_users + kScUsers - 1) / kScUsers), (unsigned)splits);
    if (int rc = launch_simt_topk_cap(cap, A, grid, smem, extrema, w_als, w_tt, topk, item_offset, cand,
                                      splits == 1 ? out_idx : pidx, splits == 1 ? out_score : pscore, excl_rowptr, excl_items, st)) return rc;
    if (splits > 1) return hals_topk_merge(pidx, pscore, splits, n_users, topk, out_idx, out_score, (void*)st);
    return 0;
  }
  // exact re-run of a device-side user list.  The first list_rows() positions are item-split (fast even for a
  // handful of users against millions of items) and merged per position; any further positions run unsplit.
  const int64_t rows = list_rows(n_users);
  const int splits = list_splits(n_items) > 1 ? list_splits(n_items) : 2;
  uint64_t* cand = (uint64_t*)workspace;
  int32_t* pidx = (int32_t*)(cand + (size_t)splits * rows * cap);
  float* pscore = (float*)(pidx + (size_t)splits * rows * topk);
  A.list_begin = 0; A.list_end = rows; A.row_stride = rows;
  fill_split(A, n_items, splits);
  int64_t gx = (rows + kScUsers - 1) / kScUsers;
  if (gx > 32) gx = 32;
  if (int rc = launch_simt_topk_cap(cap, A, dim3((unsigned)gx, (unsigned)splits), smem, extrema, w_als, w_tt, topk,
                                    item_offset, cand, pidx, pscore, excl_rowptr, excl_items, st)) return rc;
  {
    const unsigned blocks = (unsigned)((rows + 3) / 4);
    if (cap == 128) topk_merge_kernel<128><<<blocks, 128, 0, st>>>(pidx, pscore, splits, rows, topk, out_idx, out_score, user_list, user_count, 0, rows);
    else if (cap == 256) topk_merge_kernel<256><<<blocks, 128, 0, st>>>(pidx, pscore, splits, rows, topk, out_idx, out_score, user_list, user_count, 0, rows);
    else topk_merge_kernel<512><<<blocks, 128, 0, st>>>(pidx, pscore, splits, rows, topk, out_idx, out_score, user_list, user_count, 0, rows);
    HALS_LAUNCH_CHECK();
  }
  if (n_users > rows) {   // overflow of the split region (more than 2048 unproven users): unsplit, one tile per CTA
    A.list_begin = rows; A.list_end = n_users; A.row_stride = n_users - rows;
    fill_split(A, n_items, 1);
    int64_t g2 = (n_users - rows + kScUsers - 1) / kScUsers;
    if (g2 > 4 * sm_count()) g2 = 4 * sm_count();
    // candidate rows of the overflow live in the plain (unsplit) SIMT workspace that follows the list region
    uint64_t* cand2 = (uint64_t*)((uint8_t*)workspace + score_simt_list_workspace_bytes(n_users, n_items, topk));
    if (int rc = launch_simt_topk_cap(cap, A, dim3((unsigned)g2, 1), smem, extrema, w_als, w_tt, topk, item_offset,
                                      cand2, out_idx, out_score, excl_rowptr, excl_items, st)) return rc;
  }
  return 0;
}

}  // namespace hals

extern "C" int hals_topk_merge(const int32_t* part_idx, const float* part_score, int n_parts,
                               int64_t n_users, int topk, int32_t* out_idx, float* out_score, void* stream) {
  HALS_REQUIRE(part_idx && part_score && out_idx && out_score, "null pointer");
  HALS_REQUIRE(topk >= 1 && topk <= 256 && n_parts >= 1, "topk must be in [1,256]");
  if (n_users == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int cap = topk_capacity(topk);
  const unsigned blocks = (unsigned)((n_users + 3) / 4);
  if (cap == 128) topk_merge_kernel<128><<<blocks, 128, 0, st>>>(part_idx, part_score, n_parts, n_users, topk, out_idx, out_score);
  else if (cap == 256) topk_merge_kernel<256><<<blocks, 128, 0, st>>>(part_idx, part_score, n_parts, n_users, topk, out_idx, out_score);
  else topk_merge_kernel<512><<<blocks, 128, 0, st>>>(part_idx, part_score, n_parts, n_users, topk, out_idx, out_score);
  HALS_LAUNCH_CHECK();
  return 0;
}

extern "C" int hals_score_one_user(const float* u, const float* V, int64_t v_stride, int k,
                                   const int32_t* ids, int64_t n, float* out, void* stream) {
  HALS_REQUIRE(u && V && out, "null pointer");
  HALS_REQUIRE(k >= 1 && k <= 4096, "bad width");
  if (n == 0) return 0;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
  score_one_user_kernel<<<(unsigned)blocks, 256, k * sizeof(float), (cudaStream_t)stream>>>(u, V, v_stride, k, ids, n, out);
  HALS_LAUNCH_CHECK();
  return 0;
}

extern "C" int hals_fuse_lists(const float* als, const float* tt, int64_t n, float w_als, float w_tt, float* out,
                               float* scratch4, void* stream) {
  HALS_REQUIRE(als && tt && out && scratch4, "null pointer");
  HALS_REQUIRE((reinterpret_cast<uintptr_t>(scratch4) & 15) == 0, "scratch4 must be 16-byte aligned");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 2 * sm_count()) blocks = 2 * sm_count();
  extrema_init_kernel<<<1, 32, 0, st>>>(scratch4, 1);
  HALS_LAUNCH_CHECK();
  list_extrema_kernel<<<(unsigned)blocks, 256, 0, st>>>(als, tt, n, scratch4);
  HALS_LAUNCH_CHECK();
  list_blend_kernel<<<(unsigned)blocks, 256, 0, st>>>(als, tt, n, scratch4, w_als, w_tt, out);
  HALS_LAUNCH_CHECK();
  return 0;
}
