// ALS half-step, tensor-core path (explicit feedback, rank 64): the normal-equation build
// runs on tcgen05.mma with TMEM accumulators; replaces Spark's per-rating dspr/daxpy
// (NormalEquation.add) and CholeskySolver.solve reached from src/als_model.py:62.
//
// Precision: Spark accumulates in fp64; an fp32 tolerance needs better than one bf16 pass.
// Every source factor y is split once per half-step into two bf16 parts, h = bf16(y) and
// l = bf16(y - h) (|y - h - l| <= 2^-18 |y|), stored side by side ([n][h(64) | l(64)]).
//   A-operand  (M = 128, MN-major): rows 0..63 = h, rows 64..127 = l      (K = ratings)
//   B-operand  (N = 80,  MN-major): cols 0..63 = h, col 64 = bf16(r), col 65 = bf16(r - bf16(r))
//   D[0:64 , 0:64] = sum h h^T      D[64:128, 0:64] = sum l h^T
//   D[0:64 , 64:66] = sum h r_hi, sum h r_lo        D[64:128, 64] = sum l r_hi
//   A = D_hh + D_lh + D_lh^T  (drops only l l^T ~ 2^-18 relative),  b = the three r-columns.
// So ONE M=128 x N=80 x K=16 instruction per 16 ratings yields both the fp32-accurate Gram
// update and the right-hand side: 2.5 tensor cycles per rating per SM.
//
// Data movement: the h|l rows (256 B, contiguous) are gathered global->shared with cp.async
// straight into the 128B-swizzled MN-major layout the UMMA descriptors expect (layout pinned by
// tests/test_gpu_umma.py); 3-stage ring, stages recycled through tcgen05.commit -> mbarrier.
// Persistent CTAs (4 per SM: 128 TMEM columns each), static round-robin over work items; inside a CTA two
// producer warps gather + issue the MMAs of the next work item while two solver warps factorise the current one
// (als64_solve_tile: 2-D cyclic register tiling of the 64 x 64 system, see below).  ldlt64_rows (thread = matrix
// row) is the earlier solver; the long-row reduce kernel still uses it.
#include <cuda_bf16.h>

#include <cstdlib>

#include "als_common.cuh"
#include "als_tc_common.cuh"
#include "umma.cuh"

namespace hals {

constexpr int kTcThreads = 128;
#ifndef HALS_TC_KC
#define HALS_TC_KC 32
#endif
constexpr int kTcKC = HALS_TC_KC;  // ratings per stage (16 or 32)
#ifndef HALS_TC_STAGES
#define HALS_TC_STAGES 3
#endif
#ifndef HALS_TC_AHEAD
#define HALS_TC_AHEAD 2
#endif
constexpr int kTcStages = HALS_TC_STAGES;
constexpr int kTcAhead = HALS_TC_AHEAD;   // chunks in flight; one spare stage keeps the refill off the MMA-completion wait
constexpr int kTcK = 64;
constexpr int kTcRowBytes = 128;   // one 64-wide bf16 MN atom row
constexpr int kTcBlk = kTcKC * kTcRowBytes;          // 4096: one [KC][64] block
constexpr int kTcStageBytes = 3 * kTcBlk;            // H | L | R
constexpr int kTcLDP = 68;                            // published pivot rows: 16-byte aligned rows (ldlt64_rows)
constexpr int kTcLDS = 68;                            // accumulator hand-over rows: conflict-free 16-byte stores
constexpr int kTcSolverBytes = 64 * 68 * 4 + 256 + 256 + 128;   // Pall (every published pivot column) + y, z, x rows
constexpr int kTcTmemCols = 128;
constexpr int kTcN = 80;

// Register-resident solve of one 64x64 SPD system by the two solver warps (thread m owns row m
// of the symmetric matrix, a[0..63], and its right-hand side element a[64]).
// Square-root-free Cholesky (A = L D L^T, the same elimination dppsv performs up to the scaling
// of the columns): at step j the owner of row j publishes its raw row and 1/d_j
// (P[j][c] = a_j[c] for c > j, P[j][j] = 1/a_j[j]); every later row m does
//   w = a_m[j] / d_j ;  a_m[c] -= w * a_j[c]   for c in (j, 64]
// over its full remaining width (both triangles + rhs), so row j is complete when its turn
// comes and one broadcast per step is all the communication.  Steps 0..31 involve both warps
// (bar.sync among 64 threads); steps 32..63 live in warp 1 alone (__syncwarp).
// After the elimination a_m[64] = (L^-1 b)_m and the owner's registers a_c[j], j > c, still hold
// its raw pivot row, so the back substitution  x_c = (y_c - sum_{j>c} a_c[j] x_j) / d_c  runs out
// of each thread's own registers; only x_j travels (shuffles inside a warp, one shared-memory
// hand-over from warp 1 to warp 0).  Returns x_m.
template <int LDP>
__device__ __forceinline__ float ldlt64_rows(f32x2 (&ap)[32], float rhs, uint32_t P /* shared address */, int m,
                                             long long* pfs = nullptr) {
  // ap[i] = (a[2i], a[2i+1]) of this thread's matrix row; rhs = its right-hand side element (a[64])
  const int lane = m & 31;
  float inv_d = 0.f;
  float inv_next = __fdividef(1.0f, lo2(ap[0]));
#ifdef HALS_TC_PROFILE
  long long ts = clock64();
#define HALS_PFS(i) do { const long long n__ = clock64(); pfs[i] += n__ - ts; ts = n__; } while (0)
#else
#define HALS_PFS(i) do { } while (0)
#endif
  // The 64 elimination steps are NOT unrolled end to end (that is ~70 KB of straight-line code per
  // row and the solver then starves on instruction fetch); instead the row lives in a rotating
  // register window: 8 pivots per loop iteration are handled at fixed register positions 0..7, then
  // the window is rotated by 8 columns.  Register r holds absolute column (r + 8b) mod 64 in
  // iteration b; after 8 iterations every row is back in absolute alignment.  The pivot owner
  // publishes its whole window, so readers and owner agree on the rotation by construction.
  // Finished rows (m <= j) use a zero multiplier: their frozen pivot rows are never modified.
#define HALS_LDLT_STEP(NPAIRS, SYNC)                                                                  \
  {                                                                                                   \
    const int j = 8 * b + jj;                                                                         \
    const uint32_t Pj = P + (j & 1) * LDP * 4;   /* pivot rows are dead after their step: 2 slots */   \
    const float aj = (jj & 1) ? hi2(ap[jj / 2]) : lo2(ap[jj / 2]);                                    \
    const bool own = (m == j);                                                                        \
    const float inv = inv_next;          /* 1/a[j], computed during the previous step's update */     \
    if (own) inv_d = inv;                                                                             \
    _Pragma("unroll") for (int c4 = (jj / 4) * 4; c4 < 2 * (NPAIRS); c4 += 4) {                       \
      f32x2 p0 = ap[c4 / 2], p1 = ap[c4 / 2 + 1];                                                     \
      if (jj >= c4 && jj < c4 + 4) {                                                                  \
        if (jj - c4 == 0) p0 = pack2(inv, hi2(p0));                                                   \
        if (jj - c4 == 1) p0 = pack2(lo2(p0), inv);                                                   \
        if (jj - c4 == 2) p1 = pack2(inv, hi2(p1));                                                   \
        if (jj - c4 == 3) p1 = pack2(lo2(p1), inv);                                                   \
      }                                                                                               \
      sts128x2_if(own, Pj + c4 * 4, p0, p1);                                                          \
    }                                                                                                 \
    sts32_if(own, Pj + 64 * 4, rhs);                                                                  \
    SYNC;                                                                                             \
    const float nw = (m > j) ? -aj * lds32(Pj + jj * 4) : 0.f;                                        \
    const f32x2 nw2 = pack2(nw, nw);                                                                  \
    /* the pair holding the NEXT pivot goes first, so its reciprocal overlaps the rest of the update */ \
    const int pn = (jj + 1) / 2;          /* jj = 7: window register 8 = next block's pivot 0 */        \
    ap[pn] = ffma2(nw2, lds64x2(Pj + pn * 8), ap[pn]);                                                \
    inv_next = __fdividef(1.0f, ((jj + 1) & 1) ? hi2(ap[pn]) : lo2(ap[pn]));                          \
    _Pragma("unroll") for (int i = ((jj + 1) / 4) * 2; i < (NPAIRS); i += 2) {                        \
      f32x2 q0, q1;                                                                                   \
      lds128x2(Pj + i * 8, q0, q1);                                                                   \
      if (i != pn) ap[i] = ffma2(nw2, q0, ap[i]);                                                     \
      if (i + 1 != pn) ap[i + 1] = ffma2(nw2, q1, ap[i + 1]);                                         \
    }                                                                                                 \
    rhs = fmaf(nw, lds32(Pj + 64 * 4), rhs);                                                          \
  }
#define HALS_LDLT_ROTATE()                                                                            \
  {                                                                                                   \
    const f32x2 t0 = ap[0], t1 = ap[1], t2 = ap[2], t3 = ap[3];                                       \
    _Pragma("unroll") for (int i = 0; i < 28; ++i) ap[i] = ap[i + 4];                                 \
    ap[28] = t0; ap[29] = t1; ap[30] = t2; ap[31] = t3;                                               \
  }
#pragma unroll 1
  for (int b = 0; b < 4; ++b) {                          // pivots 0..31: both warps, full window
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) HALS_LDLT_STEP(32, bar_sync_64(1))
    HALS_LDLT_ROTATE()
  }
  HALS_PFS(0);
  if (m >= 32) {
#pragma unroll 1
    for (int b = 4; b < 8; ++b) {                        // pivots 32..63: warp 1 alone; live columns fit 16 pairs
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) HALS_LDLT_STEP(16, if (b == 4 && jj == 0) bar_sync_64(3); else __syncwarp())
      HALS_LDLT_ROTATE()
    }
  } else {                                               // warp 0: finish the rotation (4 x 8 columns)
    // non-blocking arrival on the barrier of pivot 32: warp 0's reads of the 2-slot pivot buffer are over
    // (barrier 3: a warp must not arrive twice on one generation of barrier 1)
    asm volatile("bar.arrive 3, 64;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) { const f32x2 tmp = ap[i]; ap[i] = ap[i + 16]; ap[i + 16] = tmp; }
  }
  HALS_PFS(1);
  // ---- back substitution ------------------------------------------------------------------------
  float acc = rhs;
  float x = 0.f;
  const uint32_t X = P + 2 * LDP * 4;                    // x_32..x_63 handed from warp 1 to warp 0
  if (m >= 32) {
#pragma unroll
    for (int j = 63; j >= 32; --j) {
      const float xj = __shfl_sync(0xffffffffu, acc * inv_d, j - 32);   // lane j-32 owns x_j
      if (m == j) x = xj;
      const float aj = (j & 1) ? hi2(ap[j / 2]) : lo2(ap[j / 2]);
      if (m < j) acc = fmaf(-aj, xj, acc);
    }
    sts32(X + lane * 4, x);
  }
  HALS_PFS(2);
  bar_sync_64(1);
  HALS_PFS(3);
  if (m < 32) {
#pragma unroll
    for (int j4 = 60; j4 >= 32; j4 -= 4) {
      const float4 q = lds128(X + (j4 - 32) * 4);
      acc = fmaf(-hi2(ap[j4 / 2 + 1]), q.w, acc);
      acc = fmaf(-lo2(ap[j4 / 2 + 1]), q.z, acc);
      acc = fmaf(-hi2(ap[j4 / 2]), q.y, acc);
      acc = fmaf(-lo2(ap[j4 / 2]), q.x, acc);
    }
#pragma unroll
    for (int j = 31; j >= 0; --j) {
      const float xj = __shfl_sync(0xffffffffu, acc * inv_d, j);
      if (m == j) x = xj;
      const float aj = (j & 1) ? hi2(ap[j / 2]) : lo2(ap[j / 2]);
      if (m < j) acc = fmaf(-aj, xj, acc);
    }
  }
  HALS_PFS(4);
  return x;
}

// ---- 2-D cyclic register tiling (the main kernel's solver) --------------------------------------------
// With thread = matrix row every thread needs the WHOLE pivot row at every step (64 threads x 256 B per step)
// and executes ~75 instructions per step for it.  Here solver thread s = 8*ti + tj owns the 8 x 8 sub-matrix
// A[ti + 8r][tj + 8c] (r, c = 0..7), so a step needs only the pivot column's entries of its 8 rows and (by
// symmetry) of its 8 columns -- 64 B instead of 256 B -- and the cyclic ownership keeps all 64 threads busy while
// the live part of the matrix shrinks (block JR updates (8-JR)^2 of the 64 entries).
//   registers  A[rp][c] = (A[ti + 16rp][tj + 8c], A[ti + 16rp + 8][tj + 8c])   (row pairs: a column of the tile is
//              four packed registers, published with two 16-byte stores, no repacking)
//   step j = 8*JR + jm: the eight threads with tj == jm publish column j into row j of Pall ([ti*8 + r] = entry
//              of row ti + 8r), one barrier, then every thread does  A[m][n] -= (A[m][j]/d) * A[n][j]  on its live
//              entries: the row multipliers arrive packed (one FFMA2-multiply by -1/d per pair), the column
//              values are broadcast into both halves of a register.
//   right-hand side: element m lives in ONE thread, (ti, tj) = (m % 8, m / 8), updated with one extra load.
// The loop over jm is rolled (register indices depend on JR only): the eight blocks are a few KB of code.
// Pall keeps every published column: row m of Pall is column m of L*D, read by the back-substitution
// (thread = row again, as in ldlt64_rows).  The whole solve is one out-of-line function so that it gets the full
// register budget: the kernel's loop state is saved around the call once per row instead of spilling per step.
constexpr int kTcPallLd = 68;                         // floats per Pall row (16-byte aligned rows)

template <int JR>
__device__ __forceinline__ void ldlt64_tile_block(f32x2 (&A)[4][8], float& bb, uint32_t pTi, uint32_t pTj,
                                                  uint32_t pMine, uint32_t Pall, uint32_t Y, int ti, int tj) {
  constexpr int RP0 = JR / 2;                           // first live row pair
  // Software pipeline: the barrier that makes column j+1 visible is issued right after its owners publish it,
  // BEFORE the bulk of step j's update (BAR.SYNC blocks only at the next shared-memory access), so the barrier
  // latency and the store drain hide behind FFMA2 work instead of sitting on the 64-step dependency chain.
  {
    const uint32_t ro = (uint32_t)(8 * JR) * (kTcPallLd * 4);
    const bool own = (tj == 0);
    sts128x2_if(own, pTi + ro, A[0][JR], A[1][JR]);
    sts128x2_if(own, pTi + ro + 16, A[2][JR], A[3][JR]);
    sts32_if(ti == 0 && tj == JR, Y + (uint32_t)(8 * JR) * 4u, bb);
    bar_sync_64(1);
  }
#pragma unroll 1
  for (int jm = 0; jm < 8; ++jm) {
    const int j = 8 * JR + jm;
    const uint32_t ro = (uint32_t)j * (kTcPallLd * 4);
    f32x2 w[4], lcp[4];
    lds128x2(pTi + ro, w[0], w[1]);
    lds128x2(pTi + ro + 16, w[2], w[3]);
    lds128x2(pTj + ro, lcp[0], lcp[1]);
    lds128x2(pTj + ro + 16, lcp[2], lcp[3]);
    const float d = lds32(Pall + ro + (uint32_t)(jm * 8 + JR) * 4u);
    const float yj = lds32(Y + (uint32_t)j * 4u);
    const float lm = lds32(pMine + ro);
    const float ninv = -__fdividef(1.0f, d);
    const f32x2 ninv2 = pack2(ninv, ninv);
#pragma unroll
    for (int rp = RP0; rp < 4; ++rp) w[rp] = ffma2(w[rp], ninv2, 0ull);
    {   // rows <= j are finished: zero multiplier (local row JR is finished iff ti <= jm; JR-1, if in the pair, always)
      float lo = lo2(w[RP0]), hi = hi2(w[RP0]);
      if (JR & 1) { lo = 0.f; hi = (ti > jm) ? hi : 0.f; }
      else lo = (ti > jm) ? lo : 0.f;
      w[RP0] = pack2(lo, hi);
    }
    {   // the block's pivot column first (columns <= j are finished: zero for tj <= jm) ...
      float l = (JR & 1) ? hi2(lcp[JR / 2]) : lo2(lcp[JR / 2]);
      l = (tj > jm) ? l : 0.f;
      const f32x2 l2 = pack2(l, l);
#pragma unroll
      for (int rp = RP0; rp < 4; ++rp) A[rp][JR] = ffma2(w[rp], l2, A[rp][JR]);
    }
    const bool act = (tj > JR) || (tj == JR && ti > jm);   // my right-hand-side row ti + 8*tj is below the pivot
    bb = act ? fmaf(lm * ninv, yj, bb) : bb;
    if (jm < 7) {   // ... so that column j+1 goes out before the rest of the update
      const bool own = (tj == jm + 1);
      const uint32_t r1 = ro + kTcPallLd * 4;
      sts128x2_if(own, pTi + r1, A[0][JR], A[1][JR]);
      sts128x2_if(own, pTi + r1 + 16, A[2][JR], A[3][JR]);
      sts32_if(ti == jm + 1 && tj == JR, Y + (uint32_t)(j + 1) * 4u, bb);
      bar_sync_64(1);
    }
#pragma unroll
    for (int c = JR + 1; c < 8; ++c) {
      const float l = (c & 1) ? hi2(lcp[c / 2]) : lo2(lcp[c / 2]);
      const f32x2 l2 = pack2(l, l);
#pragma unroll
      for (int rp = RP0; rp < 4; ++rp) A[rp][c] = ffma2(w[rp], l2, A[rp][c]);
    }
  }
}

// Gathers A = D_hh + D_lh + D_lh^T + lam*I (hand-over rows S1, S2 of stride kTcLDS) into the thread's tile, releases
// the stage ring (__syncthreads: the producers wait there too), factors, substitutes back.  Returns x_s.
__device__ __noinline__ float als64_solve_tile(uint32_t sS1, uint32_t sS2, uint32_t sB1, uint32_t sB2, uint32_t Pall,
                                               float lam, int s) {
  constexpr int LDS = kTcLDS;
  const int ti = s >> 3, tj = s & 7, lane = s & 31;
  const uint32_t Y = Pall + 64 * kTcPallLd * 4, Z = Y + 256, X = Z + 256;
  f32x2 A[4][8];
#pragma unroll
  for (int rp = 0; rp < 4; ++rp) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int n = tj + 8 * c;
      float v[2];
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        const int m = ti + 16 * rp + 8 * x;
        const uint32_t mn = (uint32_t)(m * LDS + n) * 4u, nm = (uint32_t)(n * LDS + m) * 4u;
        v[x] = lds32(sS1 + mn) + lds32(sS2 + mn) + lds32(sS2 + nm) + (m == n ? lam : 0.f);
      }
      A[rp][c] = pack2(v[0], v[1]);
    }
  }
  float bb = lds32(sB1 + (uint32_t)(ti + 8 * tj) * 4u) + lds32(sB2 + (uint32_t)(ti + 8 * tj) * 4u);
  __syncthreads();    // the stage ring (S1, S2 alias it) is free again: the producers start the next item
  const uint32_t pTi = Pall + (uint32_t)ti * 32u, pTj = Pall + (uint32_t)tj * 32u, pMine = Pall + (uint32_t)(ti * 8 + tj) * 4u;
  ldlt64_tile_block<0>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<1>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<2>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<3>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<4>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<5>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<6>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  ldlt64_tile_block<7>(A, bb, pTi, pTj, pMine, Pall, Y, ti, tj);
  // z = L^-1 b: element ti + 8*tj sits in this thread; hand row m's entry to thread m
  sts32(Z + (uint32_t)(ti + 8 * tj) * 4u, bb);
  bar_sync_64(1);
  const int m = s;
  const uint32_t rowm = Pall + (uint32_t)m * (kTcPallLd * 4);
  // entry j of column m of L*D: published by thread (j%8, m%8) at position (j%8)*8 + j/8
  auto elem = [&](int j) -> float { return lds32(rowm + (uint32_t)((j & 7) * 8 + (j >> 3)) * 4u); };
  float acc = lds32(Z + (uint32_t)m * 4u);
  const float inv_d = __fdividef(1.0f, elem(m));
  float x = 0.f;
  if (m >= 32) {
#pragma unroll
    for (int j = 63; j >= 32; --j) {
      const float lj = elem(j);
      const float xj = __shfl_sync(0xffffffffu, acc * inv_d, j - 32);   // lane j-32 owns x_j
      if (m == j) x = xj;
      if (m < j) acc = fmaf(-lj, xj, acc);
    }
    sts32(X + (uint32_t)lane * 4u, x);
  }
  bar_sync_64(1);
  if (m < 32) {
#pragma unroll
    for (int j = 63; j >= 32; --j) acc = fmaf(-elem(j), lds32(X + (uint32_t)(j - 32) * 4u), acc);
#pragma unroll
    for (int j = 31; j >= 0; --j) {
      const float lj = elem(j);
      const float xj = __shfl_sync(0xffffffffu, acc * inv_d, j);
      if (m == j) x = xj;
      if (m < j) acc = fmaf(-lj, xj, acc);
    }
  }
  return x;
}

#ifndef HALS_TC_CTAS_PER_SM
#define HALS_TC_CTAS_PER_SM 4
#endif
__global__ void __launch_bounds__(kTcThreads, HALS_TC_CTAS_PER_SM)
als_tc64_kernel(const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                const __nv_bfloat16* __restrict__ src_hl, float* __restrict__ dst, float reg,
                const int32_t* __restrict__ item_row, const int64_t* __restrict__ item_begin,
                const int32_t* __restrict__ item_len, const int32_t* __restrict__ item_slot,
                int64_t n_items, float* __restrict__ workspace, int n_sm) {
  constexpr int K = kTcK, KC = kTcKC, LDS = kTcLDS;
  extern __shared__ uint8_t smem_dyn[];
  __shared__ uint64_t mbar_free[kTcStages];
  __shared__ uint64_t mbar_acc;
  __shared__ uint32_t tmem_slot;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  // solver scratch behind the stage ring: every published pivot column (16 KB) + y, z, x hand-over rows
  const uint32_t sPall = umma::smem_u32(base + kTcStages * kTcStageBytes);
  // hand-over of the accumulators to the solver tiles; aliases the stage ring (free between the item's last MMA
  // and the producers' next gather): S1 = h h^T rows, S2 = l h^T rows (row stride 68 floats), then the two
  // right-hand-side pieces
  const uint32_t sS1 = umma::smem_u32(base), sS2 = sS1 + 64 * kTcLDS * 4, sB1 = sS2 + 64 * kTcLDS * 4, sB2 = sB1 + 256;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // Roles alternate with the CTA parity so that the solver warps of the co-resident CTAs spread
  // over all four SM sub-partitions (warp w issues on sub-partition w % 4): even CTAs solve on
  // warps 0,1 and produce on warps 2,3; odd CTAs the other way round (with the h / l blocks of the
  // stage swapped, so the solver pair always drains the h h^T rows from its own TMEM lanes).
  const bool swap = ((blockIdx.x / n_sm) & 1) != 0;   // CTAs b and b + n_sm share an SM
  const bool producer = swap ? (tid < 64) : (tid >= 64);
  const int ptid = swap ? tid : tid - 64;            // producer thread index 0..63
  const int stid = swap ? tid - 64 : tid;            // solver thread index = matrix row
  const int off_h = swap ? kTcBlk : 0, off_l = swap ? 0 : kTcBlk;
  const int t_sub = ptid >> 4, piece = ptid & 15;    // gather role: rating row within 4, 16-byte piece of the 256 B row
  if (warp == 0) umma::tmem_alloc(&tmem_slot, kTcTmemCols);
  if (tid == 0) {
    for (int s = 0; s < kTcStages; ++s) umma::mbar_init(&mbar_free[s], 1);
    umma::mbar_init(&mbar_acc, 1);
    umma::mbar_fence_init();
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint32_t sbase = umma::smem_u32(base);
  constexpr uint32_t idesc = umma::make_instr_desc(umma::kFmtBF16, true, true, 128, kTcN);

#ifdef HALS_TC_PROFILE
  long long pf[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long pfs[5] = {0, 0, 0, 0, 0};
  long long tp = clock64();
#define HALS_PF(i) do { const long long n__ = clock64(); pf[i] += n__ - tp; tp = n__; } while (0)
#else
#define HALS_PF(i) do { } while (0)
#endif
  uint32_t g = 0;         // chunks produced so far by this CTA (stage = g % stages)
  uint32_t acc_phase = 0;

  for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int row = item_row[item];
    const int64_t begin = item_begin[item];
    const int len = item_len[item];
    const int slot = item_slot[item];
    const int nc = (len + KC - 1) / KC;

    if (producer) {
      // lane t of each producer warp holds (column index, rating) of rating t of a chunk, fetched one
      // chunk ahead of its use so the dependent gather never waits on the index load
      auto fetch_idx = [&](int c, int& ci, float& rv) {
        const int q = c * KC + lane;
        const bool ok = lane < KC && q < len;
        ci = ok ? __ldg(colidx + begin + q) : -1;
        rv = (ok && ptid < 32) ? __ldg(vals + begin + q) : 0.f;
      };
      int ci_cur, ci_nxt = -1;
      float rv_cur, rv_nxt = 0.f;
      fetch_idx(0, ci_cur, rv_cur);
      if (nc > 1) fetch_idx(1, ci_nxt, rv_nxt);
      auto produce = [&](int c) {
        const uint32_t gi = g + c, s = gi % kTcStages, u = gi / kTcStages;
        if (u > 0) umma::mbar_wait(&mbar_free[s], (u - 1) & 1);
        uint8_t* st = base + s * kTcStageBytes;
        // the 16 threads sharing t read one contiguous 256-byte h|l row
        const int blk_off = (piece < 8 ? off_h : off_l);
        const int chunk = piece & 7;
#pragma unroll
        for (int i = 0; i < KC / 4; ++i) {
          const int t = t_sub + 4 * i;
          const int ci = __shfl_sync(0xffffffffu, ci_cur, t);
          cp_async16(st + blk_off + t * kTcRowBytes + ((chunk ^ (t & 7)) << 4),
                     reinterpret_cast<const uint8_t*>(src_hl) + (size_t)(ci < 0 ? 0 : ci) * (4 * K) + piece * 16, ci >= 0);
        }
        if (ptid < KC) {    // rating columns of the B operand: element 0 = bf16(r), element 1 = bf16(r - bf16(r))
          const __nv_bfloat16 rh = __float2bfloat16_rn(rv_cur);
          const __nv_bfloat16 rl = __float2bfloat16_rn(rv_cur - __bfloat162float(rh));
          const uint32_t packed = (uint32_t)__bfloat16_as_ushort(rh) | ((uint32_t)__bfloat16_as_ushort(rl) << 16);
          // chunks 0 and 1 of the row (N columns 64..79), swizzled
          *reinterpret_cast<uint4*>(st + 2 * kTcBlk + lane * kTcRowBytes + ((0 ^ (lane & 7)) << 4)) = make_uint4(packed, 0u, 0u, 0u);
          *reinterpret_cast<uint4*>(st + 2 * kTcBlk + lane * kTcRowBytes + ((1 ^ (lane & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
        }
        cp_async_commit();
        ci_cur = ci_nxt; rv_cur = rv_nxt;
        if (c + 2 < nc) fetch_idx(c + 2, ci_nxt, rv_nxt);
      };
      for (int c = 0; c < kTcAhead; ++c) {
        if (c < nc) produce(c); else cp_async_commit();
      }
      for (int c = 0; c < nc; ++c) {
        if (c + kTcAhead < nc) produce(c + kTcAhead); else cp_async_commit();
        cp_async_wait<kTcAhead>();
        umma::fence_proxy_async();
        bar_sync_64(2);
        if (ptid == 0) {
          umma::fence_after_sync();
          const uint32_t s = (g + c) % kTcStages;
          const uint32_t sa = sbase + s * kTcStageBytes;
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks) {
            const uint64_t ad = umma::make_smem_desc(sa + ks * 2048, kTcBlk, 1024, umma::kSwizzle128B);
            const uint64_t bd = umma::make_smem_desc(sa + off_h + ks * 2048, 2 * kTcBlk - off_h, 1024, umma::kSwizzle128B);
            umma::mma_bf16(tmem, ad, bd, idesc, (c | ks) != 0);
          }
          umma::commit(&mbar_free[s]);
          if (c == nc - 1) umma::commit(&mbar_acc);
        }
      }
    }
    g += nc;
    HALS_PF(0);   // producer: gather+mma issue / solver: ~0

    // ---- drain: TMEM -> registers (all four warps: a warp reads only its own 32 TMEM lanes) -----------
    umma::mbar_wait(&mbar_acc, acc_phase);
    acc_phase ^= 1;
    HALS_PF(1);   // wait for the accumulator
    umma::fence_after_sync();
    const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16);
    float a[65], e[16];
    umma::tmem_ld32(ta, a);
    umma::tmem_ld32(ta + 32, a + 32);
    umma::tmem_ld16(ta + 64, e);
    umma::fence_before_sync();
    {   // both halves go through shared memory: h h^T rows from the solver pair, l h^T rows from the producers
      const uint32_t dstrow = (producer ? sS2 + (uint32_t)ptid * (LDS * 4) : sS1 + (uint32_t)stid * (LDS * 4));
#pragma unroll
      for (int n = 0; n < 64; n += 4) sts128(dstrow + n * 4, a[n], a[n + 1], a[n + 2], a[n + 3]);
      if (producer) sts32(sB2 + ptid * 4, e[0]);
      else sts32(sB1 + stid * 4, e[0] + e[1]);
    }
    HALS_PF(2);   // drain
    __syncthreads();
    HALS_PF(3);   // wait at sync 1
    if (producer) {
      HALS_PF(4);
      __syncthreads();  // the stage ring is free again once the solver pair has read the hand-over rows
      HALS_PF(5);
    } else if (slot >= 0) {
      // slice of a long row: thread = row m, park (A, b, n) in the slot (same layout as the SIMT path)
      const int m = stid;
      float* W = workspace + (size_t)slot * ((size_t)K * K + K + 4);
#pragma unroll
      for (int n = 0; n < 64; n += 4) {
        const float4 q = lds128(sS2 + (uint32_t)m * (LDS * 4) + n * 4);
        *reinterpret_cast<float4*>(W + m * K + n) =
            make_float4(a[n] + q.x + lds32(sS2 + (uint32_t)(n) * (LDS * 4) + m * 4),
                        a[n + 1] + q.y + lds32(sS2 + (uint32_t)(n + 1) * (LDS * 4) + m * 4),
                        a[n + 2] + q.z + lds32(sS2 + (uint32_t)(n + 2) * (LDS * 4) + m * 4),
                        a[n + 3] + q.w + lds32(sS2 + (uint32_t)(n + 3) * (LDS * 4) + m * 4));
      }
      W[K * K + m] = e[0] + e[1] + lds32(sB2 + m * 4);
      if (m == 0) W[K * K + K] = (float)len;
      HALS_PF(4);
      __syncthreads();
      HALS_PF(5);
    } else {
      const float x = als64_solve_tile(sS1, sS2, sB1, sB2, sPall, reg * (float)len, stid);   // contains the __syncthreads
      dst[(int64_t)row * K + stid] = x;
      bar_sync_64(1);   // the solver scratch is reused by the next item
    }
    HALS_PF(6);   // solve
  }

#ifdef HALS_TC_PROFILE
  if ((tid % 32 == 0) && blockIdx.x < 1) printf("   tid %d solver phases: elim0-31 %lld elim32-63 %lld back1 %lld bar %lld back0 %lld\n", tid, pfs[0], pfs[1], pfs[2], pfs[3], pfs[4]);
  if ((tid == 0 || tid == 64) && blockIdx.x < 2)
    printf("cta %d tid %d items %d: gather %lld accwait %lld drain %lld sync1 %lld combine %lld sync2 %lld solve %lld\n",
           blockIdx.x, tid, (int)((n_items - blockIdx.x + gridDim.x - 1) / gridDim.x), pf[0], pf[1], pf[2], pf[3], pf[4], pf[5], pf[6]);
#endif
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, kTcTmemCols);
}

// Long rows (rank 64): sums the per-slice partial (A, b, n) slots in slot order -- deterministic -- adds the
// ridge and solves with the same register-resident LDL^T as the main kernel.  One 64-thread CTA per long row.
__global__ void __launch_bounds__(64)
als_reduce_solve64_kernel(const float* __restrict__ workspace, float* __restrict__ dst, float reg,
                          const int32_t* __restrict__ long_row, const int32_t* __restrict__ long_slot0,
                          const int32_t* __restrict__ long_nseg, __nv_bfloat16* __restrict__ dst_hl) {
  constexpr int K = kTcK, LDP = kTcLDP;
  __shared__ __align__(16) float P[3 * kTcLDP];
  const int m = threadIdx.x;
  const int row = long_row[blockIdx.x];
  const int s0 = long_slot0[blockIdx.x], ns = long_nseg[blockIdx.x];
  const size_t sf = (size_t)K * K + K + 4;
  float a[65];
#pragma unroll
  for (int n = 0; n < 65; ++n) a[n] = 0.f;
  float cnt = 0.f;
  const int stride = slot_final_stride(ns);             // rows with many slices were pre-summed per group (two levels)
  for (int q = 0; q < ns; q += stride) {
    const float* W = workspace + (size_t)(s0 + q) * sf;
#pragma unroll
    for (int n = 0; n < 64; n += 4) {
      const float4 v = *reinterpret_cast<const float4*>(W + m * K + n);
      a[n] += v.x; a[n + 1] += v.y; a[n + 2] += v.z; a[n + 3] += v.w;
    }
    a[64] += W[K * K + m];
    cnt += W[K * K + K];
  }
  const float lam = reg * cnt;
  f32x2 ap[32];
#pragma unroll
  for (int i = 0; i < 32; ++i)
    ap[i] = pack2(a[2 * i] + (2 * i == m ? lam : 0.f), a[2 * i + 1] + (2 * i + 1 == m ? lam : 0.f));
  const float x = ldlt64_rows<LDP>(ap, a[64], umma::smem_u32(P), m);
  dst[(int64_t)row * K + m] = x;
  if (dst_hl) {   // the bf16 hi|lo split the next half-step gathers (same rounding as split_bf16_kernel)
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    dst_hl[(int64_t)row * (2 * K) + m] = h;
    dst_hl[(int64_t)row * (2 * K) + K + m] = __float2bfloat16_rn(x - __bfloat162float(h));
  }
}

int als_half_step_tc64(const int32_t* colidx, const float* vals, const float* src, int64_t n_src, float* dst,
                       float reg, const hals_als_plan* plan, float* slots, void* split_buf, cudaStream_t st) {
  __nv_bfloat16* hl = reinterpret_cast<__nv_bfloat16*>(split_buf);
  if (int rc = als_launch_split_bf16(src, n_src, kTcK, hl, st)) return rc;
  const size_t smem = (size_t)kTcStages * kTcStageBytes + kTcSolverBytes + 1024;
  static_assert(kTcStages * kTcStageBytes >= 2 * 64 * kTcLDS * 4 + 512, "accumulator hand-over must fit in the stage ring");
  HALS_CUDA(cudaFuncSetAttribute(als_tc64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  static const int grid_mult = [] { const char* e = getenv("HALS_TC_GRID_MULT"); return e ? atoi(e) : HALS_TC_CTAS_PER_SM; }();
  int64_t grid = grid_mult * (int64_t)sm_count();
  if (grid > plan->n_items) grid = plan->n_items;
  als_tc64_kernel<<<(unsigned)grid, kTcThreads, smem, st>>>(colidx, vals, hl, dst, reg, plan->item_row,
                                                             plan->item_begin, plan->item_len, plan->item_slot,
                                                             plan->n_items, slots, sm_count());
  HALS_LAUNCH_CHECK();
  if (plan->n_long_rows > 0) {
    if (int rc = als_launch_slot_group_sum(slots, plan, kTcK * kTcK + kTcK + 4, st)) return rc;
    als_reduce_solve64_kernel<<<(unsigned)plan->n_long_rows, 64, 0, st>>>(slots, dst, reg, plan->long_row,
                                                                          plan->long_slot0, plan->long_nseg, nullptr);
    HALS_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace hals
