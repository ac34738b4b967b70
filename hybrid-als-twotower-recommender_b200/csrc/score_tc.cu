// Hybrid scoring, tensor-core path: U . I^T on tcgen05 (bf16 operands staged by TMA, fp32
// accumulators in TMEM) with the selection fused into the epilogue, so the score matrix never
// leaves the SM.  Replaces the reference's per-user loop (src/hybrid_system.py:95-116 calling
// src/als_model.py:75 and src/two_tower_model.py:145).
//
// bf16 operands cannot by themselves give the reference's ordering (the blended score of the
// k-th and (k+1)-th of a million items differ by ~1e-3 of a standard deviation), so the tensor
// cores only GENERATE CANDIDATES and every reported number is exact fp32:
//   pass 1  per user, the 4 largest and 4 smallest bf16 scores of each model (candidates for the
//           MinMaxScaler extrema)                      -> exact fp32 re-scoring -> extrema[U,4]
//   pass 2  user operand folded to [alpha_u*u_als | beta_u*u_tt] (alpha = w/range), ONE accumulator
//           = blend - gamma_u; per-row threshold filter keeps the best CAP/2..CAP candidates
//                                                      -> exact fp32 blend of the candidates,
//                                                         sort, top-k (same code as the SIMT path)
// hals_score_topk (ALS top-k by raw dot product) is pass 2 alone: no scaling, so no extrema are needed (blend_topk).
// Each user carries a rigorous bound eps_u on |bf16 score - fp32 score| (2^-8 |u| max|i|, Cauchy-
// Schwarz).  A result is accepted only if the exact k-th score clears (candidate threshold +
// eps_u), i.e. no rejected item could belong to the answer; otherwise the user is flagged and
// re-done by the exact SIMT kernel (score_simt.cu) -- on the GPU, never on the host.
//
// Kernel shape: CTA = 128 users (UMMA M) x a contiguous item range, 10 warps (pass 1) or 18 warps (pass 2):
//   warp 0    TMA producer: user tile once, item K-blocks ([256 x 64] bf16, 128B swizzle) through a 4-stage ring
//   warp 1    MMA issuer: 4 x tcgen05.mma (M=128, N=256, K=16) per K-block, accumulators double-buffered in TMEM
//             (2 x 256 columns; pass 1 scores the two models as two consecutive accumulator jobs per item tile)
//   warps 2.. epilogue, PARTS warps per TMEM lane quarter (each takes 1/PARTS of the tile's columns; pass 1: 2, pass 2: 4,
//             one candidate stream per part): tcgen05.ld 32 / 64
//             columns per step with the next load in flight, thread = user row, FMNMX3 chains per 8-column octet
//             against the row threshold held in a register; only octets with a survivor walk their columns.
#include <cuda_bf16.h>

#include "common.cuh"
#include "tma.cuh"
#include "topk.cuh"
#include "umma.cuh"

namespace hals {

constexpr int kStM = 128;
constexpr int kStRing = 4;
// Epilogue warps per TMEM lane quarter (PARTS): each takes 1/PARTS of a tile's columns and, in pass 2, feeds its own
// candidate stream.  With 2 warps per scheduler the epilogue is latency-bound (38 % of its samples are fixed-latency
// waits, ncu round 2).  Pass 2 runs 4 parts = 16 epilogue warps at 96 registers; what makes that pay is halving the
// kept set and the buffer of a stream with it (4 streams x keep 64 see the same threshold -- the global rank-256 score
// -- and the same number of survivors as 2 x 128; a first try with 4 x 128 was 19 % SLOWER: 1.8x the survivors).  Pass 1
// keeps 2 parts (4 measured slower there: 717 vs 632 ms on the 1 M x 1.25 M leg, its lists need the registers).
#ifndef HALS_SCORE_PARTS
#define HALS_SCORE_PARTS 4
#endif
constexpr int kStParts1 = 2;                   // pass 1
constexpr int kStParts2 = HALS_SCORE_PARTS;    // pass 2
static_assert(kStParts2 == 2 || kStParts2 == 4, "column parts per tile");
constexpr int kStPartsMax = kStParts1 > kStParts2 ? kStParts1 : kStParts2;
constexpr int kStExC = 4;            // extrema candidates per list
#ifndef HALS_SCORE_W
#define HALS_SCORE_W 64              // columns per filter step of pass 2 (a candidate buffer keeps W slots free; 32: 5 % slower)
#endif

struct ScoreTcArgs {
  int nkb_a, nkb_t;                  // 64-wide K blocks of the ALS / tower part
  int64_t n_users, n_items;
  int64_t items_per_split;           // multiple of BN
  int n_splits;
  int keep;                          // candidates kept by a compaction (>= topk)
  int32_t item_offset;
};

// ---- operand preparation: fp32 row-major (two models) -> bf16 [rows][64*(nkb_a+nkb_t)] --------------
// One warp per row.  scale: optional per-row (alpha, beta) pair from blend coefficients.
// norm_out[row] = (|a-part|_2, |t-part|_2) of the written (scaled) values; max_norm: running maxima
// (non-negative floats order like their bit patterns -> atomicMax on the bits).
__global__ void score_prep_kernel(const float* __restrict__ A, int64_t a_stride, int ka, const float* __restrict__ T,
                                  int64_t t_stride, int kt, int64_t n_rows, int nkb_a, int nkb_t,
                                  const float* __restrict__ extrema, float w_als, float w_tt,
                                  __nv_bfloat16* __restrict__ out, float2* __restrict__ norm_out,
                                  unsigned int* __restrict__ max_norm_bits) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int Kp = 64 * (nkb_a + nkb_t), Ka = 64 * nkb_a;
  float sa = 1.f, st = 1.f;
  if (extrema != nullptr) {   // user side of pass 2: fold alpha = w/range (zero range contributes nothing)
    const float4 ex = reinterpret_cast<const float4*>(extrema)[row];
    const float ra = ex.y - ex.x, rt = ex.w - ex.z;
    sa = (ra != 0.f) ? w_als / ra : 0.f;
    st = (rt != 0.f) ? w_tt / rt : 0.f;
  }
  float na = 0.f, nt = 0.f;
  // each lane converts 8 consecutive outputs and writes them with one 16-byte store (Kp / 8 <= 32 chunks per row)
  const int f0 = lane * 8;
  if (f0 < Kp) {
    const bool is_a = f0 < Ka;                          // a chunk never straddles the two parts (Ka is a multiple of 64)
    const float* src = is_a ? A + row * a_stride : T + row * t_stride;
    const int g0 = is_a ? f0 : f0 - Ka, kk = is_a ? ka : kt;
    const float sc = is_a ? sa : st;
    float v[8];
    if (g0 + 8 <= kk && ((reinterpret_cast<uintptr_t>(src + g0) & 15) == 0)) {
      const float4 p = *reinterpret_cast<const float4*>(src + g0), q = *reinterpret_cast<const float4*>(src + g0 + 4);
      v[0] = p.x; v[1] = p.y; v[2] = p.z; v[3] = p.w; v[4] = q.x; v[5] = q.y; v[6] = q.z; v[7] = q.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = (g0 + i < kk) ? src[g0 + i] : 0.f;
    }
    float s2 = 0.f;
    __align__(16) __nv_bfloat16 o8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[i] *= sc;
      s2 = fmaf(v[i], v[i], s2);
      o8[i] = __float2bfloat16_rn(v[i]);
    }
    if (is_a) na = s2; else nt = s2;
    *reinterpret_cast<uint4*>(out + row * Kp + f0) = *reinterpret_cast<const uint4*>(o8);
  }
  na = sqrtf(warp_sum(na));
  nt = sqrtf(warp_sum(nt));
  if (lane == 0) {
    if (norm_out) norm_out[row] = make_float2(na, nt);
    if (max_norm_bits) {
      // racy pre-check keeps 1.25M rows from serialising on two addresses; the atomic decides
      if (__float_as_uint(na) > *(volatile unsigned int*)(max_norm_bits + 0)) atomicMax(max_norm_bits + 0, __float_as_uint(na));
      if (__float_as_uint(nt) > *(volatile unsigned int*)(max_norm_bits + 1)) atomicMax(max_norm_bits + 1, __float_as_uint(nt));
    }
  }
}

// sorted-descending insertion into a 4-entry list
__device__ __forceinline__ void insert4(float (&v)[kStExC], int (&ix)[kStExC], float s, int i) {
#pragma unroll
  for (int p = kStExC - 1; p >= 0; --p) {
    const bool here = (p == 0) || !(s > v[p - 1]);
    if (s > v[p]) {
      if (here) { v[p] = s; ix[p] = i; }
      else { v[p] = v[p - 1]; ix[p] = ix[p - 1]; }
    }
  }
}

// Out of line on purpose: the hot epilogue loop must stay small enough for the instruction cache.
template <int CAP>
__device__ __noinline__ int compact_row(uint64_t* buf, int count, int keep, int lane, float* thr_out) {
  return topk_select_compact<CAP>(buf, count, keep, lane, thr_out);
}

// Pass 2 with an exclusion list (EXCL): each epilogue thread walks its user's ascending list with a forward-only cursor.
// A thread meets its columns in ascending item order (half * HB + g * W + 8 * o + c within a tile, tiles ascending), so
// the cursor never moves back; it is consulted only for items that passed the threshold, and excluded items never enter
// a candidate buffer -- the threshold and the compactions only ever see allowed items.  Exactness is unchanged: the
// verification bounds what a stream REJECTED, and an excluded item cannot belong to the answer.  A user left with fewer
// than k allowed items has kth = -inf; if one of its streams still raised its threshold (the final trim to `keep`, or a
// compaction at k > 224) the verification flags it and the exact SIMT re-run, which filters too, produces the list.
struct ExclCursor {
  const int32_t* p;        // next unread entry
  int left;                // entries from p to the end of the row
  int32_t next;            // the smallest excluded id not yet passed (INT32_MAX: none)
  __device__ __forceinline__ void init(const int64_t* rowptr, const int32_t* items, int64_t u, int32_t first) {
    int64_t lo = rowptr[u], hi = rowptr[u + 1];
    const int64_t end = hi;
    while (lo < hi) {                                  // lower bound of `first`
      const int64_t mid = (lo + hi) >> 1;
      if (items[mid] < first) lo = mid + 1; else hi = mid;
    }
    p = items + lo;
    left = (int)(end - lo);
    next = left > 0 ? *p : 0x7fffffff;
  }
  // true when item `gi` (global id, ascending across calls) is excluded
  __device__ __forceinline__ bool excluded(int32_t gi) {
    while (next < gi) {
      ++p;
      next = --left > 0 ? *p : 0x7fffffff;
    }
    return next == gi;
  }
};

template <int PASS, int BN, int CAP, int PARTS, bool EXCL>
__global__ void __launch_bounds__(64 + 128 * PARTS, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap map_u, const __grid_constant__ CUtensorMap map_i, ScoreTcArgs A,
                float* __restrict__ ex_val /* [splits][U][4][4] */, int32_t* __restrict__ ex_idx,
                uint64_t* __restrict__ cand /* [splits][U][CAP] */, int32_t* __restrict__ cand_cnt,
                float* __restrict__ cand_thr /* [splits][U] */,
                const int64_t* __restrict__ excl_rowptr /* EXCL: [U+1] */, const int32_t* __restrict__ excl_items) {
  static_assert(!EXCL || PASS == 2, "exclusion lists apply to the top-k pass");
  constexpr int JPT = (PASS == 1) ? 2 : 1;             // accumulator jobs per item tile: pass 1 scores the two models
                                                       // one after the other (N = 256 each: an N = 128 MMA pair is
                                                       // shared-memory-bandwidth bound at M = 128)
  constexpr int BUFCOLS = BN;                          // TMEM columns per buffer (256), two buffers
  constexpr uint32_t kABlk = kStM * 128;               // bytes of one [128 x 64] bf16 block
  constexpr uint32_t kBBlk = BN * 128;
  extern __shared__ uint8_t smem_dyn[];
  __shared__ uint64_t full[kStRing], empty[kStRing], a_full, tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_slot;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint8_t* smA = base;                                 // [nkb][128][64] bf16
  const int nkb = A.nkb_a + A.nkb_t;
  uint8_t* smB = base + nkb * kABlk;                   // ring of [BN][64] bf16

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t u0 = (int64_t)blockIdx.x * kStM;
  const int split = blockIdx.y;
  const int64_t i_begin = (int64_t)split * A.items_per_split;
  const int64_t i_end = min(A.n_items, i_begin + A.items_per_split);
  const int n_tiles = i_end > i_begin ? (int)((i_end - i_begin + BN - 1) / BN) : 0;

  if (tid == 0) {
    for (int s = 0; s < kStRing; ++s) { umma::mbar_init(&full[s], 1); umma::mbar_init(&empty[s], 1); }
    umma::mbar_init(&a_full, 1);
    for (int b = 0; b < 2; ++b) { umma::mbar_init(&tmem_full[b], 1); umma::mbar_init(&tmem_empty[b], 4 * PARTS); }
    umma::mbar_fence_init();
    tma::prefetch_map(&map_u);
    tma::prefetch_map(&map_i);
  }
  if (warp == 1) umma::tmem_alloc(&tmem_slot, 512);
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
#ifdef HALS_SC_PROFILE
  long long pf[4] = {0, 0, 0, 0};
  long long tp = clock64();
#define HALS_SPF(i) do { const long long n__ = clock64(); pf[i] += n__ - tp; tp = n__; } while (0)
#else
#define HALS_SPF(i) do { } while (0)
#endif

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      tma::expect_tx(&a_full, nkb * kABlk);
      for (int kb = 0; kb < nkb; ++kb) tma::load_2d(smA + kb * kABlk, &map_u, &a_full, kb * 64, (int32_t)u0);
      uint32_t g = 0;
      for (int t = 0; t < n_tiles; ++t) {
        const int32_t row0 = (int32_t)(i_begin + (int64_t)t * BN);
        for (int kb = 0; kb < nkb; ++kb, ++g) {
          const uint32_t s = g % kStRing, u = g / kStRing;
          HALS_SPF(0);
          if (u > 0) umma::mbar_wait(&empty[s], (u - 1) & 1);
          HALS_SPF(1);
          tma::expect_tx(&full[s], kBBlk);
          tma::load_2d(smB + s * kBBlk, &map_i, &full[s], kb * 64, row0);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = umma::make_instr_desc(umma::kFmtBF16, false, false, kStM, BN);
      const uint32_t sA = umma::smem_u32(smA), sB = umma::smem_u32(smB);
      umma::mbar_wait(&a_full, 0);
      uint32_t g = 0;
      for (int t = 0; t < n_tiles; ++t) {
#pragma unroll
        for (int m = 0; m < JPT; ++m) {
          const uint32_t job = (uint32_t)t * JPT + m, buf = job & 1, use = job >> 1;
          const int kb0 = (PASS == 1 && m == 1) ? A.nkb_a : 0;
          const int kb1 = (PASS == 1 && m == 0) ? A.nkb_a : nkb;
          HALS_SPF(0);
          if (use > 0) umma::mbar_wait(&tmem_empty[buf], (use - 1) & 1);
          HALS_SPF(1);
          umma::fence_after_sync();
          const uint32_t d = tmem + buf * BUFCOLS;
          for (int kb = kb0; kb < kb1; ++kb, ++g) {
            const uint32_t s = g % kStRing, u = g / kStRing;
            HALS_SPF(0);
            umma::mbar_wait(&full[s], u & 1);
            HALS_SPF(2);
            umma::fence_after_sync();
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t ad = umma::make_smem_desc(sA + kb * kABlk + ks * 32, 16, 1024, umma::kSwizzle128B);
              const uint64_t bd = umma::make_smem_desc(sB + s * kBBlk + ks * 32, 16, 1024, umma::kSwizzle128B);
              umma::mma_bf16(d, ad, bd, idesc, !(kb == kb0 && ks == 0));
            }
            umma::commit(&empty[s]);
          }
          umma::commit(&tmem_full[buf]);                // a model without K blocks (rank 0) completes at once
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue: thread = user row
    const int q = warp & 3;                             // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;                   // which part of the tile's columns
    const int vs = split * PARTS + half;                // candidate stream ("virtual split") of this thread
    constexpr int HB = BN / PARTS;
    const int r = q * 32 + lane;
    const int64_t u = u0 + r;
    const bool live = u < A.n_users;
    const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);
    const float ninf = -__int_as_float(0x7f800000);

    // pass 1 state: 4 candidates for each of max_a, min_a (as -s), max_t, min_t (as -s)
    float xv[4][kStExC];
    int xi[4][kStExC];
    // pass 2 state
    float thr = ninf;
    int cnt = 0;
    uint64_t* mybuf = nullptr;
    if (PASS == 1) {
#pragma unroll
      for (int l = 0; l < 4; ++l)
#pragma unroll
        for (int p = 0; p < kStExC; ++p) { xv[l][p] = ninf; xi[l][p] = -1; }
    } else {
      mybuf = cand + ((size_t)vs * A.n_users + (live ? u : 0)) * CAP;
      if (!live) thr = __int_as_float(0x7f800000);
    }
    ExclCursor xc;
    if (EXCL) {
      if (live) xc.init(excl_rowptr, excl_items, u, (int32_t)i_begin + A.item_offset);
      else { xc.left = 0; xc.next = 0x7fffffff; }     // a dead row never has a survivor
    }

    for (int t = 0; t < n_tiles; ++t) {
     const int64_t it0 = i_begin + (int64_t)t * BN;
     const bool ragged = it0 + BN > i_end;              // only the last tile of a range
#pragma unroll
     for (int m = 0; m < JPT; ++m) {
      const uint32_t job = (uint32_t)t * JPT + m, buf = job & 1, use = job >> 1;
      HALS_SPF(0);
      umma::mbar_wait(&tmem_full[buf], use & 1);
      HALS_SPF(1);
      umma::fence_after_sync();
      // software pipeline over the 32-column groups of this warp's half: the tcgen05.ld of group g+1 is in
      // flight while group g is filtered
      const uint32_t tbase = tq + buf * BUFCOLS;
      constexpr int G = HB / 32;
      if (PASS == 1) {
        // job m holds model m's scores (0 = ALS, 1 = tower): lists 2m (maxima) and 2m+1 (minima, as -s)
        const bool present = (m == 0) ? (A.nkb_a > 0) : (A.nkb_t > 0);
        if (present) {
          // The group loop is ROLLED (pairs of groups, for the register double buffer): fully unrolled, the epilogue was
          // 60 KB of straight-line code that eight warps walk once per tile, and 37 % of the warp samples were
          // instruction-fetch stalls (ncu, round 2).
          // (four warps per scheduler: no register double buffer -- the other warps cover the tcgen05.ld latency and the
          //  two candidate lists per model need the registers)
          constexpr bool kDouble = PARTS < 4;
          constexpr int NB = kDouble ? 2 : 1;
          float vv[NB][32];
          if (kDouble) umma::tmem_ld32_issue(tbase + half * HB, vv[0]);
          static_assert(G % NB == 0, "groups are processed in pairs");
#pragma unroll 1
          for (int gp = 0; gp < G; gp += NB) {
#pragma unroll
          for (int gb = 0; gb < NB; ++gb) {
            const int g = gp + gb;
            const int c0 = half * HB + g * 32;
            if (!kDouble) umma::tmem_ld32_issue(tbase + c0, vv[0]);
            umma::tmem_wait_ld_dep(vv[gb]);
            if (kDouble && g + 1 < G) umma::tmem_ld32_issue(tbase + c0 + 32, vv[(gb + 1) % NB]);
            const float (&v)[32] = vv[gb];
            // Extremes of each 8-column octet first (FMNMX3 chains).  A warp runs an octet's per-column code only
            // when some lane can change one of its two lists there, and that code walks 8 columns, not 32.
            const float t0 = xv[2 * m][kStExC - 1], t1 = xv[2 * m + 1][kStExC - 1];
            float mx[4], mn[4];                         // all eight chains first: they overlap, the branches come after
#pragma unroll
            for (int o = 0; o < 4; ++o) {
              mx[o] = v[8 * o]; mn[o] = v[8 * o];
#pragma unroll
              for (int c = 1; c < 8; ++c) { mx[o] = fmaxf(mx[o], v[8 * o + c]); mn[o] = fminf(mn[o], v[8 * o + c]); }
            }
            const float gmx = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])), gmn = fminf(fminf(mn[0], mn[1]), fminf(mn[2], mn[3]));
            if (live && (gmx > t0 || -gmn > t1))
#pragma unroll
            for (int o = 0; o < 4; ++o) {
              if (mx[o] > t0 || -mn[o] > t1) {
                unsigned mk = 0;                         // thresholds may be stale within the octet: insert4 re-checks
#pragma unroll
                for (int c = 0; c < 8; ++c) mk |= ((v[8 * o + c] > t0 || -v[8 * o + c] > t1) ? 1u : 0u) << c;
                while (mk) {
                  const int c = __ffs(mk) - 1;
                  mk &= mk - 1;
                  const int64_t i = it0 + c0 + 8 * o + c;
                  if (!ragged || i < i_end) {
                    float s = v[8 * o];
#pragma unroll
                    for (int cc = 1; cc < 8; ++cc) s = (cc == c) ? v[8 * o + cc] : s;
                    insert4(xv[2 * m], xi[2 * m], s, (int)i);
                    insert4(xv[2 * m + 1], xi[2 * m + 1], -s, (int)i);
                  }
                }
              }
            }
          }
          }
        }
      } else {
        // W columns per step (two tcgen05.ld x32 in flight per buffer when the candidate buffer leaves room for 64
        // new keys): more independent FMNMX3 chains per wait, half as many waits, branches and ballots
        constexpr int W = (CAP >= 256 && PARTS == 2) ? HALS_SCORE_W : 32;   // (4 parts, one 64-column step: measured slower)
        constexpr int G2 = HB / W;
        constexpr int NB = G2 >= 2 ? 2 : 1;
        static_assert(G2 % NB == 0, "groups are processed in pairs");
        float vv[NB][W];
        if (NB == 2) {
#pragma unroll
          for (int x = 0; x < W / 32; ++x) umma::tmem_ld32_issue(tbase + half * HB + 32 * x, vv[0] + 32 * x);
        }
#pragma unroll 1
        for (int gp = 0; gp < G2; gp += NB) {
#pragma unroll
        for (int gb = 0; gb < NB; ++gb) {
          const int g = gp + gb;
          const int c0 = half * HB + g * W;
          if (NB == 1) {
#pragma unroll
            for (int x = 0; x < W / 32; ++x) umma::tmem_ld32_issue(tbase + c0 + 32 * x, vv[0] + 32 * x);
          }
#pragma unroll
          for (int x = 0; x < W / 32; ++x) umma::tmem_wait_ld_dep(vv[gb] + 32 * x);
          if (NB == 2 && g + 1 < G2) {
#pragma unroll
            for (int x = 0; x < W / 32; ++x) umma::tmem_ld32_issue(tbase + c0 + W + 32 * x, vv[(gb + 1) % NB] + 32 * x);
          }
          const float (&v)[W] = vv[gb];
          // Octet maxima (FMNMX3 chains) against the row threshold.  Survivors are ~0.4% of the items: most lanes
          // have none in a group, but some lane of the warp nearly always has one, so what matters is how much
          // code that lane drags the warp through -- an 8-column bitmask, and for the usual single survivor the
          // octet maximum IS its score (no register selection).
          float gm4[W / 8];
#pragma unroll
          for (int o = 0; o < W / 8; ++o) {
            gm4[o] = v[8 * o];
#pragma unroll
            for (int c = 1; c < 8; ++c) gm4[o] = fmaxf(gm4[o], v[8 * o + c]);
          }
          float gall = gm4[0];
#pragma unroll
          for (int o = 1; o < W / 8; ++o) gall = fmaxf(gall, gm4[o]);
          if (gall > thr)
#pragma unroll
          for (int o = 0; o < W / 8; ++o) {
            const float gm = gm4[o];
            if (gm > thr) {
              unsigned m = 0;
#pragma unroll
              for (int c = 0; c < 8; ++c) m |= (v[8 * o + c] > thr ? 1u : 0u) << c;
              const int64_t ib = it0 + c0 + 8 * o;
              if ((m & (m - 1)) == 0) {
                const int64_t i = ib + (__ffs(m) - 1);
                if ((!ragged || i < i_end) && !(EXCL && xc.excluded((int32_t)i + A.item_offset)))
                  mybuf[cnt++] = topk_key(gm, (int32_t)i);
              } else {
                while (m) {
                  const int c = __ffs(m) - 1;
                  m &= m - 1;
                  float s = v[8 * o];
#pragma unroll
                  for (int cc = 1; cc < 8; ++cc) s = (cc == c) ? v[8 * o + cc] : s;
                  const int64_t i = ib + c;
                  if ((!ragged || i < i_end) && !(EXCL && xc.excluded((int32_t)i + A.item_offset)))
                    mybuf[cnt++] = topk_key(s, (int32_t)i);
                }
              }
            }
          }
          // compaction: a row may not enter the next W columns with fewer than W free slots
          unsigned need = __ballot_sync(0xffffffffu, cnt > CAP - W);
          while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            const int64_t urow = u0 + q * 32 + src;
            uint64_t* b = cand + ((size_t)vs * A.n_users + urow) * CAP;
            const int c_src = __shfl_sync(0xffffffffu, cnt, src);
            float t_new;
            __syncwarp();
            const int c_new = compact_row<CAP>(b, c_src, A.keep, lane, &t_new);
            if (lane == src) { cnt = c_new; thr = t_new; }
          }
        }
        }
      }
      umma::fence_before_sync();
      __syncwarp();
      if (lane == 0) tma::arrive(&tmem_empty[buf]);
     }
    }

    if (PASS == 2) {
      // trim every stream to its best `keep` before the exact re-scoring (fewer candidates to re-score; the
      // verification bound then uses the keep-th bf16 score of the stream)
      unsigned need = __ballot_sync(0xffffffffu, live && cnt > A.keep);
      while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        const int64_t urow = u0 + q * 32 + src;
        uint64_t* b = cand + ((size_t)vs * A.n_users + urow) * CAP;
        const int c_src = __shfl_sync(0xffffffffu, cnt, src);
        float t_new;
        __syncwarp();
        const int c_new = compact_row<CAP>(b, c_src, A.keep, lane, &t_new);
        if (lane == src) { cnt = c_new; thr = t_new; }
      }
    }
    if (live) {
      if (PASS == 1) {
        const size_t o = (((size_t)vs * A.n_users + u) * 4) * kStExC;
#pragma unroll
        for (int l = 0; l < 4; ++l)
#pragma unroll
          for (int p = 0; p < kStExC; ++p) { ex_val[o + l * kStExC + p] = xv[l][p]; ex_idx[o + l * kStExC + p] = xi[l][p]; }
      } else {
        cand_cnt[(size_t)vs * A.n_users + u] = cnt;
        cand_thr[(size_t)vs * A.n_users + u] = thr;
      }
    }
  }

#ifdef HALS_SC_PROFILE
  HALS_SPF(0);
  if (blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 && warp < 3)
    printf("score_tc pass %d warp %d tiles %d: work %lld wait_a %lld wait_b %lld\n", PASS, warp, n_tiles, pf[0], pf[1], pf[2]);
#endif
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 1) umma::tmem_dealloc(tmem, 512);
}

// ---- exact fp32 re-scoring -------------------------------------------------------------------------
__device__ __forceinline__ float dot_seq(const float* __restrict__ a, const float* __restrict__ b, int k) {
  float s = 0.f;
  for (int f = 0; f < k; ++f) s = fmaf(a[f], b[f], s);   // same order as the SIMT path: bitwise-equal scores
  return s;
}

struct ExactArgs {
  const float* Ua; int64_t ua_stride; const float* Ia; int64_t ia_stride; int ka;
  const float* Ut; int64_t ut_stride; const float* It; int64_t it_stride; int kt;
  int64_t n_users; int n_splits;
};

// Pass 1: one thread per (user, list).  extrema[u] = exact (min_a, max_a, min_t, max_t); flag[u] |= 1 when the
// candidates cannot be proven to contain the true extremum.
__global__ void score_exact_extrema_kernel(ExactArgs E, const float* __restrict__ ex_val, const int32_t* __restrict__ ex_idx,
                                           const float2* __restrict__ unorm, const unsigned int* __restrict__ inorm_bits,
                                           float* __restrict__ extrema, int32_t* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int64_t gid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // one warp per (user, list)
  const int64_t u = gid >> 2;
  const int l = (int)(gid & 3);                        // 0 max_a, 1 min_a, 2 max_t, 3 min_t
  if (u >= E.n_users) return;
  const bool is_t = l >= 2, is_min = l & 1;
  const float ninf = -__int_as_float(0x7f800000);
  const float* uv = is_t ? E.Ut + u * E.ut_stride : E.Ua + u * E.ua_stride;
  const int k = is_t ? E.kt : E.ka;
  const int64_t istride = is_t ? E.it_stride : E.ia_stride;
  const float* ibase = is_t ? E.It : E.Ia;
  float uq[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) uq[q] = (lane + 32 * q < k) ? uv[lane + 32 * q] : 0.f;
  float best = ninf, bound = ninf;
  bool any = false;
  for (int s = 0; s < E.n_splits; ++s) {
    const size_t o = ((((size_t)s * E.n_users + u) * 4) + l) * kStExC;
    for (int p = 0; p < kStExC; ++p) {
      const int i = ex_idx[o + p];
      if (i < 0) continue;
      const float* iv = ibase + (int64_t)i * istride;
      float sc = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) if (lane + 32 * q < k) sc = fmaf(uq[q], iv[lane + 32 * q], sc);
      sc = warp_sum(sc);
      best = fmaxf(best, is_min ? -sc : sc);
      any = true;
    }
    // everything this split rejected scored (in bf16) no better than its weakest kept candidate
    if (ex_idx[o + kStExC - 1] >= 0) bound = fmaxf(bound, ex_val[o + kStExC - 1]);
  }
  if (lane != 0) return;
  const float2 un = unorm[u];
  const float eps = 1.05f * 0.00390625f * (is_t ? un.y * __uint_as_float(inorm_bits[1]) : un.x * __uint_as_float(inorm_bits[0]));
  if (k == 0) { best = 0.f; any = true; bound = ninf; }
  if (!any) best = is_min ? -__int_as_float(0x7f800000) : ninf;   // no items: (+inf, -inf) like the SIMT path
  extrema[u * 4 + (is_t ? 2 : 0) + (is_min ? 0 : 1)] = is_min ? -best : best;
  if (any && !(best >= bound + eps) && bound > ninf) atomicOr(flag + u, 1);
}

// Pass 2: candidates (bf16 score keys) -> exact fp32 blend keys, in place.  One warp per candidate stream
// (stream, user): the user's two vectors stay in registers, every candidate's item rows are read with
// coalesced 128-byte warp loads and reduced with shuffles (fp32; the summation order differs from the
// CUDA-core path's sequential fmaf only in the last bits).  extrema == NULL: raw mode (hals_score_topk, kt = 0,
// w = (1, 0)) with the identity coefficients (0, 1, 0, 1), so the key is the ALS dot product itself.
__global__ void score_exact_blend_kernel(ExactArgs E, const float* __restrict__ extrema, float w_als, float w_tt,
                                         int32_t item_offset, uint64_t* __restrict__ cand, const int32_t* __restrict__ cand_cnt,
                                         int cap, int sortn) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // (stream, user)
  if (row >= (int64_t)E.n_splits * E.n_users) return;
  int n = cand_cnt[row];
  if (n > sortn) n = sortn;
  if (n <= 0) return;
  const int64_t u = row % E.n_users;
  float ua[4], ut[2];
#pragma unroll
  for (int q = 0; q < 4; ++q) ua[q] = (lane + 32 * q < E.ka) ? E.Ua[u * E.ua_stride + lane + 32 * q] : 0.f;
#pragma unroll
  for (int q = 0; q < 2; ++q) ut[q] = (lane + 32 * q < E.kt) ? E.Ut[u * E.ut_stride + lane + 32 * q] : 0.f;
  const float4 ex = extrema ? reinterpret_cast<const float4*>(extrema)[u] : make_float4(0.f, 1.f, 0.f, 1.f);
  const float ra = ex.y - ex.x, rt = ex.w - ex.z;
  const float sca = (ra != 0.f) ? 1.f / ra : 1.f, sct = (rt != 0.f) ? 1.f / rt : 1.f;
  uint64_t* buf = cand + (size_t)row * cap;
  for (int e0 = 0; e0 < n; e0 += 32) {
    const uint64_t mykey = (e0 + lane < n) ? buf[e0 + lane] : 0ull;
    const int cnt = min(32, n - e0);
    uint64_t outkey = 0ull;
    for (int e = 0; e < cnt; ++e) {
      const int i = topk_key_index(__shfl_sync(0xffffffffu, mykey, e));
      const float* ia = E.Ia + (int64_t)i * E.ia_stride;
      const float* it = E.It + (int64_t)i * E.it_stride;
      float sa = 0.f, st = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) if (lane + 32 * q < E.ka) sa = fmaf(ua[q], ia[lane + 32 * q], sa);
#pragma unroll
      for (int q = 0; q < 2; ++q) if (lane + 32 * q < E.kt) st = fmaf(ut[q], it[lane + 32 * q], st);
      sa = warp_sum(sa);
      st = warp_sum(st);
      const float b = fmaf(w_als, (sa - ex.x) * sca, w_tt * ((st - ex.z) * sct));   // == blend_value()
      if (lane == e) outkey = topk_key(b, i + item_offset);
    }
    if (e0 + lane < n) buf[e0 + lane] = outkey;
  }
}

// Pass 2 finish: one warp per (split,user): sort the exact keys, write the top-k list, verify.
template <int CAP /* keys sorted per stream (>= trimmed count) */>
__global__ void score_select_kernel(int stride /* key slots per stream */, uint64_t* __restrict__ cand, const int32_t* __restrict__ cand_cnt,
                                    const float* __restrict__ cand_thr, const float* __restrict__ extrema,
                                    const float2* __restrict__ unorm_scaled, const unsigned int* __restrict__ inorm_bits,
                                    float w_als, float w_tt, int64_t n_users, int n_splits, int topk,
                                    int32_t* __restrict__ out_idx, float* __restrict__ out_score, int32_t* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (int64_t)n_splits * n_users) return;
  uint64_t* buf = cand + (size_t)row * stride;
  uint64_t tkey;
  const int have = cand_cnt[row] < CAP ? cand_cnt[row] : CAP;   // surplus keys (score ties at the trim threshold) count as rejected
  const int c = topk_compact<CAP>(buf, have, topk, lane, &tkey);
  int32_t* oi = out_idx + (size_t)row * topk;
  float* os = out_score + (size_t)row * topk;
  for (int e = lane; e < topk; e += 32) {
    if (e < c) { const uint64_t k = buf[e]; oi[e] = topk_key_index(k); os[e] = topk_key_score(k); }
    else { oi[e] = -1; os[e] = -__int_as_float(0x7f800000); }
  }
}

// Pass 2 verification, after the cross-split merge: every item a split rejected had bf16 (blend - gamma) <= thr_s,
// hence exact blend <= thr_s + gamma + eps.  The final list is provably the exact top-k when its k-th score
// clears that bound for every split; otherwise the user is flagged for the exact re-run.  Raw mode (extrema == NULL):
// the identity coefficients give alpha = w_als = 1 and gamma = 0 -- the accumulator is the bf16 dot product itself.
__global__ void score_verify_kernel(const float* __restrict__ cand_thr, const float* __restrict__ extrema,
                                    const float2* __restrict__ unorm_scaled, const unsigned int* __restrict__ inorm_bits,
                                    float w_als, float w_tt, int64_t n_users, int n_splits, int topk,
                                    const float* __restrict__ out_score, int32_t* __restrict__ flag) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n_users) return;
  const float ninf = -__int_as_float(0x7f800000);
  float thr = ninf;
  for (int s = 0; s < n_splits; ++s) thr = fmaxf(thr, cand_thr[(size_t)s * n_users + u]);
  if (!(thr > ninf)) return;                            // nothing was ever rejected
  const float4 ex = extrema ? reinterpret_cast<const float4*>(extrema)[u] : make_float4(0.f, 1.f, 0.f, 1.f);
  const float ra = ex.y - ex.x, rt = ex.w - ex.z;
  const float al = (ra != 0.f) ? w_als / ra : 0.f, be = (rt != 0.f) ? w_tt / rt : 0.f;
  const float gamma = -(al * ex.x + be * ex.z);
  const float2 un = unorm_scaled[u];
  const float eps = 1.05f * 0.00390625f * (un.x * __uint_as_float(inorm_bits[0]) + un.y * __uint_as_float(inorm_bits[1]));
  const float kth = out_score[u * topk + topk - 1];     // -inf when fewer than k items exist
  if (!(kth > thr + gamma + eps)) atomicOr(flag + u, 2);
}

// compacts the flagged users into a list (order irrelevant: every listed user is recomputed exactly)
__global__ void score_flag_list_kernel(const int32_t* __restrict__ flag, int64_t n_users, int mask, int32_t* __restrict__ list,
                                       int32_t* __restrict__ count, float* __restrict__ reset_extrema) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u < n_users && (flag[u] & mask)) {
    list[atomicAdd(count, 1)] = (int32_t)u;
    if (reset_extrema) {   // the exact re-run accumulates with atomic min/max
      const float inf = __int_as_float(0x7f800000);
      reinterpret_cast<float4*>(reset_extrema)[u] = make_float4(inf, -inf, inf, -inf);
    }
  }
}

}  // namespace hals

// =====================================================================================================
// Host side: public entry points (dispatch tensor-core / SIMT) and workspace carving
// =====================================================================================================
#include <cstdlib>

#include "score_common.cuh"

using namespace hals;

namespace {

constexpr int kTcBN = 256;      // items per tile in pass 2 (pass 1 uses 128 + 128 columns per buffer)

struct TcPlan {
  bool use_tc;
  int nkb_a, nkb_t, Kp, splits, cap, keep;
  int64_t items_per_split;
  // workspace offsets (bytes)
  size_t off_ub, off_ib, off_unorm, off_misc, off_flag, off_list, off_exv, off_exi, off_cand, off_cnt, off_thr,
      off_pidx, off_pscore, off_simt, total;
};

size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

TcPlan make_plan(int64_t n_users, int64_t n_items, int ka, int kt, int topk) {
  TcPlan p{};
  static const bool force_simt = [] { const char* e = getenv("HALS_FORCE_SIMT"); return e && e[0] == '1'; }();
  p.nkb_a = (ka + 63) / 64; p.nkb_t = (kt + 63) / 64; p.Kp = 64 * (p.nkb_a + p.nkb_t);
  // candidate capacity: the kept set (cap/2) must reach well below the k-th score so that the rigorous
  // bf16 error bound rarely overlaps it (k=100 of 1.25M items: rank 256 sits 0.23 sigma below rank 100)
  p.cap = topk <= 24 ? 128 : topk <= 56 ? 256 : 512;
  {
    int want = ((topk + 28 + 31) / 32) * 32;         // kept set of a candidate stream: k plus a safety margin
    if (want < 64) want = 64;
    p.keep = want < p.cap / 2 ? want : p.cap / 2;
  }
  if (kStParts2 == 4) {
    // four streams per row instead of two: half the kept set and half the buffer per stream.  The union still reaches
    // the global rank ~4 keep (the verification margin is unchanged) and a stream holds its share of the top-k with
    // overwhelming probability (k = 100: 25 +- 4.3 expected per stream against 64 kept); an adversarial item order
    // that defeats this fails the verification and is re-run exactly, as always.
    if (p.cap > 128) p.cap /= 2;
    p.keep = p.keep / 2 < 32 ? 32 : p.keep / 2;
    if (p.keep > p.cap / 2) p.keep = p.cap / 2;
  }
  // the tensor-core path pays off once the tile grid can fill the GPU; tiny calls stay on the exact SIMT path
  p.use_tc = !force_simt && tma::encode_fn() != nullptr && n_items >= 2048 && n_users * n_items >= (int64_t)1 << 22;
  const int64_t user_tiles = (n_users + kStM - 1) / kStM;
  const int64_t item_tiles = (n_items + kTcBN - 1) / kTcBN;
  int64_t splits = user_tiles > 0 ? (sm_count() + user_tiles - 1) / user_tiles : 1;
  {
    // one CTA per SM: pick the smallest multiple of the minimum split count whose CTA count fills whole waves
    // (512 user tiles on 148 SMs: 1 split = 3.46 waves -> 4, 2 splits = 6.92 -> 7)
    // The top-k pass pays for every extra candidate stream (more survivors to append and re-score), so it
    // only splits further when a wave would otherwise be mostly empty; the extrema pass splits freely.
    const int64_t base = splits;
    const double good_enough = topk > 0 ? 0.80 : 0.95;
    double best_eff = 0.0;
    for (int64_t mult = 1; mult <= 4; ++mult) {
      const double waves = (double)(user_tiles * base * mult) / sm_count();
      const double eff = waves / (double)(int64_t)(waves + 0.999999);
      if (eff > best_eff + 0.03) { best_eff = eff; splits = base * mult; }
      if (best_eff >= good_enough) break;
    }
  }
  if (splits > item_tiles) splits = item_tiles;
  if (splits > 64) splits = 64;
  if (splits < 1) splits = 1;
  p.items_per_split = ((item_tiles + splits - 1) / splits) * kTcBN;
  if (p.items_per_split < kTcBN) p.items_per_split = kTcBN;
  p.splits = (int)((n_items + p.items_per_split - 1) / p.items_per_split);
  if (p.splits < 1) p.splits = 1;
  size_t o = 0;
  const size_t su = (size_t)kStPartsMax * (size_t)p.splits * (size_t)n_users;   // candidate streams (column parts) per split
  {
    const int tk = topk > 0 ? topk : 1;
    const size_t plain = score_simt_workspace_bytes(n_users, n_items, tk);
    // list mode: split region for the first 2048 positions + one unsplit candidate row per remaining user
    const size_t listed = score_simt_list_workspace_bytes(n_users, n_items, tk) +
                          (size_t)n_users * topk_capacity(tk) * sizeof(uint64_t) + 256;
    p.off_simt = o;   o += align256(plain > listed ? plain : listed);
  }
  if (p.use_tc) {
    p.off_ub = o;     o += align256((size_t)n_users * p.Kp * 2);
    p.off_ib = o;     o += align256((size_t)n_items * p.Kp * 2);
    p.off_unorm = o;  o += align256((size_t)n_users * sizeof(float2));
    p.off_misc = o;   o += 256;                                  // item max norms (2 x u32), flagged count (i32 at +16)
    p.off_flag = o;   o += align256((size_t)n_users * 4);
    p.off_list = o;   o += align256((size_t)n_users * 4);
    p.off_exv = o;    o += align256(su * 16 * 4);
    p.off_exi = o;    o += align256(su * 16 * 4);
    p.off_cand = o;   o += align256(su * p.cap * 8);
    p.off_cnt = o;    o += align256(su * 4);
    p.off_thr = o;    o += align256(su * 4);
    p.off_pidx = o;   o += align256(su * (size_t)(topk > 0 ? topk : 1) * 4);
    p.off_pscore = o; o += align256(su * (size_t)(topk > 0 ? topk : 1) * 4);
  }
  p.total = o + 256;
  return p;
}

template <int PASS, int BN, int CAP, int PARTS, bool EXCL = false>
int launch_tc(const CUtensorMap& mu, const CUtensorMap& mi, const ScoreTcArgs& A, int nkb, float* exv, int32_t* exi,
              uint64_t* cand, int32_t* cnt, float* thr, cudaStream_t st, const int64_t* excl_rowptr = nullptr,
              const int32_t* excl_items = nullptr) {
  const size_t smem = (size_t)nkb * kStM * 128 + (size_t)kStRing * BN * 128 + 1024;
  HALS_CUDA(cudaFuncSetAttribute(score_tc_kernel<PASS, BN, CAP, PARTS, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)((A.n_users + kStM - 1) / kStM), (unsigned)A.n_splits);
  score_tc_kernel<PASS, BN, CAP, PARTS, EXCL><<<grid, 64 + 128 * PARTS, smem, st>>>(mu, mi, A, exv, exi, cand, cnt, thr,
                                                                                    excl_rowptr, excl_items);
  HALS_LAUNCH_CHECK();
  return 0;
}

template <int CAP>
int launch_tc_topk(const CUtensorMap& mu, const CUtensorMap& mi, const ScoreTcArgs& A, int nkb, uint64_t* cand,
                   int32_t* cnt, float* thr, cudaStream_t st, const int64_t* excl_rowptr, const int32_t* excl_items) {
  if (excl_rowptr != nullptr)
    return launch_tc<2, kTcBN, CAP, kStParts2, true>(mu, mi, A, nkb, nullptr, nullptr, cand, cnt, thr, st, excl_rowptr, excl_items);
  return launch_tc<2, kTcBN, CAP, kStParts2>(mu, mi, A, nkb, nullptr, nullptr, cand, cnt, thr, st);
}

}  // namespace

extern "C" size_t hals_score_workspace_bytes(int64_t n_users, int64_t n_items, int ka, int kt, int topk) {
  return make_plan(n_users, n_items, ka, kt, topk).total;
}

extern "C" int64_t hals_score_flag_counter_offset(int64_t n_users, int64_t n_items, int ka, int kt, int topk) {
  const TcPlan p = make_plan(n_users, n_items, ka, kt, topk);
  return p.use_tc ? (int64_t)(p.off_misc + 16) : -1;
}

extern "C" int hals_score_extrema(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride,
                                  int ka, const float* Ut, int64_t ut_stride, const float* It,
                                  int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                                  float* extrema, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_score_args(Ua, Ia, ka, Ut, It, kt, n_users, n_items)) return rc;
  HALS_REQUIRE(extrema, "null extrema");
  if (n_users == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const ScoreOperands O{Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt};
  const TcPlan p = make_plan(n_users, n_items, ka, kt, 0);
  if (!p.use_tc || n_items == 0) return score_extrema_simt(O, n_users, n_items, extrema, nullptr, nullptr, st);
  HALS_REQUIRE(workspace != nullptr, "null workspace");
  if (workspace_bytes < p.total) return fail(HALS_ERR_WORKSPACE, "%s: workspace too small%s", __func__);
  uint8_t* W = (uint8_t*)workspace;
  __nv_bfloat16* ub = (__nv_bfloat16*)(W + p.off_ub);
  __nv_bfloat16* ib = (__nv_bfloat16*)(W + p.off_ib);
  float2* unorm = (float2*)(W + p.off_unorm);
  unsigned int* inorm = (unsigned int*)(W + p.off_misc);
  int32_t* fcount = (int32_t*)(W + p.off_misc + 16);
  int32_t* flag = (int32_t*)(W + p.off_flag);
  int32_t* list = (int32_t*)(W + p.off_list);
  HALS_CUDA(cudaMemsetAsync(W + p.off_misc, 0, 256, st));
  HALS_CUDA(cudaMemsetAsync(flag, 0, (size_t)n_users * 4, st));
  score_prep_kernel<<<(unsigned)((n_items + 7) / 8), 256, 0, st>>>(Ia, ia_stride, ka, It, it_stride, kt, n_items, p.nkb_a,
                                                                    p.nkb_t, nullptr, 0.f, 0.f, ib, nullptr, inorm);
  HALS_LAUNCH_CHECK();
  score_prep_kernel<<<(unsigned)((n_users + 7) / 8), 256, 0, st>>>(Ua, ua_stride, ka, Ut, ut_stride, kt, n_users, p.nkb_a,
                                                                    p.nkb_t, nullptr, 0.f, 0.f, ub, unorm, nullptr);
  HALS_LAUNCH_CHECK();
  CUtensorMap mu, mi;
  if (!tma::make_bf16_rowmajor_map(&mu, ub, (uint64_t)n_users, (uint64_t)p.Kp, kStM) ||
      !tma::make_bf16_rowmajor_map(&mi, ib, (uint64_t)n_items, (uint64_t)p.Kp, kTcBN))
    return fail(HALS_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed%s", __func__);
  ScoreTcArgs A{p.nkb_a, p.nkb_t, n_users, n_items, p.items_per_split, p.splits, p.keep, 0};
  if (int rc = launch_tc<1, kTcBN, 128, kStParts1>(mu, mi, A, p.nkb_a + p.nkb_t, (float*)(W + p.off_exv), (int32_t*)(W + p.off_exi),
                                      nullptr, nullptr, nullptr, st)) return rc;
  ExactArgs E{Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt, n_users, kStParts1 * p.splits};
  score_exact_extrema_kernel<<<(unsigned)((n_users * 4 + 7) / 8), 256, 0, st>>>(
      E, (const float*)(W + p.off_exv), (const int32_t*)(W + p.off_exi), unorm, inorm, extrema, flag);
  HALS_LAUNCH_CHECK();
  score_flag_list_kernel<<<(unsigned)((n_users + 255) / 256), 256, 0, st>>>(flag, n_users, 1, list, fcount, extrema);
  HALS_LAUNCH_CHECK();
  return score_extrema_simt(O, n_users, n_items, extrema, list, fcount, st);   // exact re-run of unproven users
}

// The body of hals_score_blend_topk, hals_score_blend_topk_excluding (excl_rowptr == NULL: no exclusion) and
// hals_score_topk (raw mode: extrema == NULL, kt = 0, w = (1, 0); the kernels that read extrema then use the identity
// coefficients (0, 1, 0, 1), so every score is the plain dot product and no extrema pass is needed).
static int blend_topk(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride, int ka, const float* Ut,
                      int64_t ut_stride, const float* It, int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                      const float* extrema, float w_als, float w_tt, int topk, int32_t item_offset, int32_t* out_idx,
                      float* out_score, const int64_t* excl_rowptr, const int32_t* excl_items, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (int rc = check_score_args(Ua, Ia, ka, Ut, It, kt, n_users, n_items)) return rc;
  HALS_REQUIRE(out_idx && out_score && workspace, "null pointer");
  HALS_REQUIRE(topk >= 1 && topk <= 256, "topk must be in [1,256]");
  const TcPlan p = make_plan(n_users, n_items, ka, kt, topk);
  if (workspace_bytes < p.total) return fail(HALS_ERR_WORKSPACE, "%s: workspace too small%s", __func__);
  if (n_users == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const ScoreOperands O{Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt};
  uint8_t* W = (uint8_t*)workspace;
  if (!p.use_tc)
    return score_blend_topk_simt(O, n_users, n_items, extrema, w_als, w_tt, topk, item_offset, out_idx, out_score,
                                 W + p.off_simt, nullptr, nullptr, excl_rowptr, excl_items, st);
  __nv_bfloat16* ub = (__nv_bfloat16*)(W + p.off_ub);
  __nv_bfloat16* ib = (__nv_bfloat16*)(W + p.off_ib);
  float2* unorm = (float2*)(W + p.off_unorm);
  unsigned int* inorm = (unsigned int*)(W + p.off_misc);
  int32_t* fcount = (int32_t*)(W + p.off_misc + 16);
  int32_t* flag = (int32_t*)(W + p.off_flag);
  int32_t* list = (int32_t*)(W + p.off_list);
  uint64_t* cand = (uint64_t*)(W + p.off_cand);
  int32_t* cnt = (int32_t*)(W + p.off_cnt);
  float* thr = (float*)(W + p.off_thr);
  HALS_CUDA(cudaMemsetAsync(W + p.off_misc, 0, 256, st));
  HALS_CUDA(cudaMemsetAsync(flag, 0, (size_t)n_users * 4, st));
  score_prep_kernel<<<(unsigned)((n_items + 7) / 8), 256, 0, st>>>(Ia, ia_stride, ka, It, it_stride, kt, n_items, p.nkb_a,
                                                                    p.nkb_t, nullptr, 0.f, 0.f, ib, nullptr, inorm);
  HALS_LAUNCH_CHECK();
  score_prep_kernel<<<(unsigned)((n_users + 7) / 8), 256, 0, st>>>(Ua, ua_stride, ka, Ut, ut_stride, kt, n_users, p.nkb_a,
                                                                    p.nkb_t, extrema, w_als, w_tt, ub, unorm, nullptr);
  HALS_LAUNCH_CHECK();
  CUtensorMap mu, mi;
  if (!tma::make_bf16_rowmajor_map(&mu, ub, (uint64_t)n_users, (uint64_t)p.Kp, kStM) ||
      !tma::make_bf16_rowmajor_map(&mi, ib, (uint64_t)n_items, (uint64_t)p.Kp, kTcBN))
    return fail(HALS_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed%s", __func__);
  ScoreTcArgs A{p.nkb_a, p.nkb_t, n_users, n_items, p.items_per_split, p.splits, p.keep, item_offset};
  const int nkb = p.nkb_a + p.nkb_t;
  int rc;
  if (p.cap == 128) rc = launch_tc_topk<128>(mu, mi, A, nkb, cand, cnt, thr, st, excl_rowptr, excl_items);
  else if (p.cap == 256) rc = launch_tc_topk<256>(mu, mi, A, nkb, cand, cnt, thr, st, excl_rowptr, excl_items);
  else rc = launch_tc_topk<512>(mu, mi, A, nkb, cand, cnt, thr, st, excl_rowptr, excl_items);
  if (rc) return rc;
  const int vsplits = kStParts2 * p.splits;
  ExactArgs E{Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt, n_users, vsplits};
  int sortn = 64;                                       // streams leave the tensor-core kernel trimmed to `keep` keys;
  while (sortn < p.keep || sortn < topk) sortn <<= 1;   // a stream reports up to topk of them
  if (sortn > p.cap) sortn = p.cap;
  const int64_t slots = (int64_t)vsplits * n_users * sortn;
  (void)slots;
  score_exact_blend_kernel<<<(unsigned)(((int64_t)vsplits * n_users + 7) / 8), 256, 0, st>>>(E, extrema, w_als, w_tt, item_offset, cand, cnt, p.cap, sortn);
  HALS_LAUNCH_CHECK();
  int32_t* oi = (int32_t*)(W + p.off_pidx);
  float* os = (float*)(W + p.off_pscore);
  const unsigned sel_blocks = (unsigned)(((int64_t)vsplits * n_users + 3) / 4);
  if (sortn == 64) score_select_kernel<64><<<sel_blocks, 128, 0, st>>>(p.cap, cand, cnt, thr, extrema, unorm, inorm, w_als, w_tt, n_users, vsplits, topk, oi, os, flag);
  else if (sortn == 128) score_select_kernel<128><<<sel_blocks, 128, 0, st>>>(p.cap, cand, cnt, thr, extrema, unorm, inorm, w_als, w_tt, n_users, vsplits, topk, oi, os, flag);
  else if (sortn == 256) score_select_kernel<256><<<sel_blocks, 128, 0, st>>>(p.cap, cand, cnt, thr, extrema, unorm, inorm, w_als, w_tt, n_users, vsplits, topk, oi, os, flag);
  else score_select_kernel<512><<<sel_blocks, 128, 0, st>>>(p.cap, cand, cnt, thr, extrema, unorm, inorm, w_als, w_tt, n_users, vsplits, topk, oi, os, flag);
  HALS_LAUNCH_CHECK();
  if (int rc2 = hals_topk_merge(oi, os, vsplits, n_users, topk, out_idx, out_score, stream)) return rc2;
  score_verify_kernel<<<(unsigned)((n_users + 255) / 256), 256, 0, st>>>(thr, extrema, unorm, inorm, w_als, w_tt, n_users,
                                                                          vsplits, topk, out_score, flag);
  HALS_LAUNCH_CHECK();
  score_flag_list_kernel<<<(unsigned)((n_users + 255) / 256), 256, 0, st>>>(flag, n_users, 2, list, fcount, nullptr);
  HALS_LAUNCH_CHECK();
  return score_blend_topk_simt(O, n_users, n_items, extrema, w_als, w_tt, topk, item_offset, out_idx, out_score,
                               W + p.off_simt, list, fcount, excl_rowptr, excl_items, st);    // exact re-run of unproven users
}

extern "C" int hals_score_blend_topk(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride,
                                     int ka, const float* Ut, int64_t ut_stride, const float* It,
                                     int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                                     const float* extrema, float w_als, float w_tt, int topk,
                                     int32_t item_offset, int32_t* out_idx, float* out_score,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  HALS_REQUIRE(extrema, "null pointer");
  return blend_topk(Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt, n_users, n_items, extrema, w_als,
                    w_tt, topk, item_offset, out_idx, out_score, nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int hals_score_blend_topk_excluding(const float* Ua, int64_t ua_stride, const float* Ia, int64_t ia_stride,
                                               int ka, const float* Ut, int64_t ut_stride, const float* It,
                                               int64_t it_stride, int kt, int64_t n_users, int64_t n_items,
                                               const float* extrema, float w_als, float w_tt, int topk,
                                               int32_t item_offset, int32_t* out_idx, float* out_score,
                                               const int64_t* excl_rowptr, const int32_t* excl_items,
                                               void* workspace, size_t workspace_bytes, void* stream) {
  HALS_REQUIRE((excl_rowptr == nullptr) == (excl_items == nullptr), "excl_rowptr and excl_items must both be set or both NULL");
  HALS_REQUIRE(extrema, "null pointer");
  return blend_topk(Ua, ua_stride, Ia, ia_stride, ka, Ut, ut_stride, It, it_stride, kt, n_users, n_items, extrema, w_als,
                    w_tt, topk, item_offset, out_idx, out_score, excl_rowptr, excl_items, workspace, workspace_bytes, stream);
}

extern "C" int hals_score_topk(const float* Q, int64_t q_stride, const float* C, int64_t c_stride, int k, int64_t n_q,
                               int64_t n_c, int topk, int32_t c_offset, const int64_t* excl_rowptr,
                               const int32_t* excl_items, int32_t* out_idx, float* out_score, void* workspace,
                               size_t workspace_bytes, void* stream) {
  // every argument check comes before make_plan, whose SM count query is the first CUDA call
  HALS_REQUIRE(k >= 1 && k <= 128, "k (the factor rank) must be in [1,128]");
  HALS_REQUIRE(topk >= 1 && topk <= 256, "topk must be in [1,256]");
  HALS_REQUIRE(n_q >= 0 && n_c >= 0, "negative size");
  HALS_REQUIRE(Q && C && out_idx && out_score && workspace, "null pointer");
  HALS_REQUIRE((excl_rowptr == nullptr) == (excl_items == nullptr), "excl_rowptr and excl_items must both be set or both NULL");
  return blend_topk(Q, q_stride, C, c_stride, k, nullptr, 0, nullptr, 0, 0, n_q, n_c, nullptr, 1.f, 0.f, topk, c_offset,
                    out_idx, out_score, excl_rowptr, excl_items, workspace, workspace_bytes, stream);
}
