// ALS half-step, tensor-core path for rank 128 (explicit feedback): Netflix-shape config.
// Same construction as als_tc.cu (bf16 h/l split, tcgen05.mma into TMEM, register-resident
// square-root-free Cholesky), re-dimensioned for a 128 x 128 system; replaces Spark's
// NormalEquation.add + CholeskySolver.solve reached from src/als_model.py:62.
//
//   per 16 ratings, three instructions on the same gathered [32 ratings][h(128) | l(128)] bf16 stage:
//     D[:,   0:256] += H^T . [H | L]      (M = 128, N = 256)   -> h h^T (cols 0..127) and h l^T (128..255)
//     D[:, 256:272] += H^T . R            (M = 128, N = 16)    -> sum h r_hi, sum h r_lo
//     D[:, 272:288] += L^T . R            (M = 128, N = 16)    -> sum l r_hi
//   A = D_hh + D_hl + D_hl^T ,  b = D[.,256] + D[.,257] + D[.,272]          (drops l l^T ~ 2^-18)
//
// One persistent CTA per SM (the accumulator needs 288 of the 512 TMEM columns), 10 warps:
//   warps 0,1   producers: cp.async gather into the swizzled MN-major stage ring, one thread issues the MMAs
//   warps 2-5   solver group A, warps 6-9 solver group B: the groups take alternate work items, so while one
//               group eliminates (128 dependent pivot steps) the other drains / eliminates the next row and the
//               producers gather the one after.  A group drains row m of C = D_hh/2 + D_hl per thread (thread =
//               TMEM lane), then solves with the 2-D cyclic register tiling (als128_solve_tile, 16 x 8 thread grid).
// ldlt128_rows (thread = matrix row, rotating register window, 2-slot pivot buffer, shrinking named barriers) is the
// earlier solver; the long-row reduce kernel still uses it.
#include <cuda_bf16.h>

#include <cstdlib>

#include "als_common.cuh"
#include "als_tc_common.cuh"
#include "umma.cuh"

namespace hals {

constexpr int k8K = 128;
constexpr int k8KC = 32;                    // ratings per stage
constexpr int k8Stages = 3;
constexpr int k8Ahead = 2;
constexpr int k8Blk = k8KC * 128;           // one [KC][64] bf16 block (4 KB)
constexpr int k8StageBytes = 5 * k8Blk;     // H0 | H1 | L0 | L1 | R
constexpr int k8Threads = 320;
constexpr int k8LDP = 132;                  // pivot slot: 128 window floats + rhs (+ pad to 16 B)
constexpr int k8LDC = 132;                  // row stride of the hand-over matrix C / of Pall (16-byte aligned rows)
constexpr int k8GroupBytes = 128 * k8LDC * 4 + 4 * 512;        // C (aliased by Pall) + b, y, z, x rows
constexpr size_t k8SlotFloats = (size_t)k8K * k8K + k8K + 4;

// 128 x 128 SPD solve by one solver group (4 warps, thread = row m, rb = m / 32).
// ap[i] = (a[2i], a[2i+1]) of the row, rhs = right-hand side element.  Returns x_m.
__device__ __forceinline__ float ldlt128_rows(f32x2 (&ap)[64], float rhs, uint32_t P, uint32_t X, int m, int bar_base) {
  const int rb = m >> 5, lane = m & 31;
  float inv_d = 0.f;
  float inv_next = __fdividef(1.0f, lo2(ap[0]));
  // one elimination step at window position jj (0..3) of the current 4-pivot block
#define HALS_L128_STEP(NPAIRS)                                                                          \
  {                                                                                                     \
    const int j = 4 * b4 + jj;                                                                          \
    const uint32_t Pj = P + (j & 1) * (k8LDP * 4);                                                      \
    const float aj = (jj & 1) ? hi2(ap[jj / 2]) : lo2(ap[jj / 2]);                                      \
    const bool own = (m == j);                                                                          \
    const float inv = inv_next;                                                                         \
    if (own) inv_d = inv;                                                                               \
    _Pragma("unroll") for (int c4 = 0; c4 < 2 * (NPAIRS); c4 += 4) {                                    \
      f32x2 p0 = ap[c4 / 2], p1 = ap[c4 / 2 + 1];                                                       \
      if (c4 == 0) {                                                                                    \
        if (jj == 0) p0 = pack2(inv, hi2(p0));                                                          \
        if (jj == 1) p0 = pack2(lo2(p0), inv);                                                          \
        if (jj == 2) p1 = pack2(inv, hi2(p1));                                                          \
        if (jj == 3) p1 = pack2(lo2(p1), inv);                                                          \
      }                                                                                                 \
      sts128x2_if(own, Pj + c4 * 4, p0, p1);                                                            \
    }                                                                                                   \
    sts32_if(own, Pj + 128 * 4, rhs);                                                                   \
    /* the first step of a phase also waits for the warp that just ran out of rows: its reads of the   */ \
    /* 2-slot pivot buffer must be over before the slot is published again                              */ \
    if (jj == 0 && (b4 & 7) == 0 && ph > 0) bar_sync_n(bar_base + 2 + ph, 160 - 32 * ph);               \
    else if (ph == 3) __syncwarp();                                                                     \
    else bar_sync_n(bar_base + ph, 128 - 32 * ph);                                                      \
    const float nw = (m > j) ? -aj * lds32(Pj + jj * 4) : 0.f;                                          \
    const f32x2 nw2 = pack2(nw, nw);                                                                    \
    const int pn = (jj + 1) / 2;          /* jj = 3: window register 4 = next block's pivot 0 */        \
    ap[pn] = ffma2(nw2, lds64x2(Pj + pn * 8), ap[pn]);                                                  \
    inv_next = __fdividef(1.0f, ((jj + 1) & 1) ? hi2(ap[pn]) : lo2(ap[pn]));                            \
    _Pragma("unroll") for (int i = (jj == 3 ? 2 : 0); i < (NPAIRS); i += 2) {                           \
      f32x2 q0, q1;                                                                                     \
      lds128x2(Pj + i * 8, q0, q1);                                                                     \
      if (i != pn) ap[i] = ffma2(nw2, q0, ap[i]);                                                       \
      if (i + 1 != pn) ap[i + 1] = ffma2(nw2, q1, ap[i + 1]);                                           \
    }                                                                                                   \
    rhs = fmaf(nw, lds32(Pj + 128 * 4), rhs);                                                           \
  }
#pragma unroll 1
  for (int b4 = 0; b4 < 32; ++b4) {
    const int ph = b4 >> 3;                               // pivots 32 ph .. 32 ph + 31 belong to warp ph
    if (rb < ph) {                                        // this warp has no rows left (warp-uniform)
      bar_arrive_n(bar_base + 2 + ph, 160 - 32 * ph);     // hand-shake barrier (own id: a warp must not arrive twice
                                                          // on one barrier generation), see the first-step barrier below
      break;
    }
    if (b4 < 16) {
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) HALS_L128_STEP(64)
    } else {                                              // fewer than 64 live columns: half window
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) HALS_L128_STEP(32)
    }
    const f32x2 t0 = ap[0], t1 = ap[1];                   // rotate the window by 4 columns
#pragma unroll
    for (int i = 0; i < 62; ++i) ap[i] = ap[i + 2];
    ap[62] = t0; ap[63] = t1;
  }
#undef HALS_L128_STEP
  // A warp leaves the loop after 32 (rb + 1) columns of rotation; 96 more columns bring its own pivot block to
  // window registers 0..31 and the later columns (the frozen upper part of its rows) to registers 32.. .
#pragma unroll
  for (int i = 0; i < 16; ++i) {                          // in-place rotation by 48 pairs: 16 cycles of length 4
    const f32x2 t = ap[i];
    ap[i] = ap[i + 48]; ap[i + 48] = ap[i + 32]; ap[i + 32] = ap[i + 16]; ap[i + 16] = t;
  }
  // ---- back substitution: x_c = (y_c - sum_{j>c} a_c[j] x_j) / d_c, last warp first ---------------------
  float acc = rhs, x = 0.f;
#pragma unroll 1
  for (int w = 3; w >= 0; --w) {
    if (rb == w) {
      // contributions of the already solved x_j, j >= 32 (rb + 1): window registers 32 .. 127 - 32 rb
#pragma unroll
      for (int r4 = 32; r4 < 128; r4 += 4) {
        if (r4 < 128 - 32 * rb) {
          const float4 q = lds128(X + (32 * rb + r4) * 4);
          acc = fmaf(-lo2(ap[r4 / 2]), q.x, acc);
          acc = fmaf(-hi2(ap[r4 / 2]), q.y, acc);
          acc = fmaf(-lo2(ap[r4 / 2 + 1]), q.z, acc);
          acc = fmaf(-hi2(ap[r4 / 2 + 1]), q.w, acc);
        }
      }
#pragma unroll
      for (int jl = 31; jl >= 0; --jl) {                  // own block: pivot 32 rb + jl lives in lane jl
        const float xj = __shfl_sync(0xffffffffu, acc * inv_d, jl);
        if (lane == jl) x = xj;
        const float aj = (jl & 1) ? hi2(ap[jl / 2]) : lo2(ap[jl / 2]);
        if (lane < jl) acc = fmaf(-aj, xj, acc);
      }
      sts32(X + m * 4, x);
    }
    if (w > 0) bar_sync_n(bar_base, 128);
  }
  return x;
}

// ---- 2-D cyclic register tiling (main kernel) -----------------------------------------------------------
// als_tc.cu's tile solver at rank 128: the 128 threads of a solver group form a 16 x 8 grid, thread (ti, tj) owns
// A[ti + 16r][tj + 8c] (r = 0..7, c = 0..15; 64 packed registers, as many as the row layout needed), so a step
// moves 96 B of pivot data per thread instead of 512 B and updates only the live part of the tile.
//   registers   A[rp][c] = (A[ti + 32rp][tj + 8c], A[ti + 32rp + 16][tj + 8c])
//   Pall row j  [ti*8 + r] = A[ti + 16r][j]  (published by the 16 threads with tj == j % 8): a thread reads its 8 row
//               entries at [ti*8 ..], the entries of its even local columns at [tj*8 ..] and of its odd ones at
//               [(tj+8)*8 ..]  (column n = tj + 8c is row n of the symmetric matrix: n % 16 = tj + 8(c&1), n / 16 = c/2)
//   rhs         element m lives in thread (m % 16, m / 16)
// Blocks of 8 pivots (JC = j / 8) fix every register index; the loop over the pivot inside a block is rolled.
template <int JC>
__device__ __forceinline__ void ldlt128_tile_block(f32x2 (&A)[4][16], float& bb, uint32_t pTi, uint32_t pTjE, uint32_t pTjO,
                                                   uint32_t pMine, uint32_t Pall, uint32_t Y, int ti, int tj, int bar) {
  constexpr int JR = JC / 2;                            // local row index of this block's pivot rows
  constexpr int RP0 = JR / 2;                           // first live row pair
  constexpr int TI0 = 8 * (JC & 1);                     // pivot j = 8 JC + jm is row-owned by ti == TI0 + jm
  // Software pipeline (as in als_tc.cu): column j+1 is published, and the barrier issued, before the bulk of step
  // j's update, so the barrier latency hides behind FFMA2 work.
  {
    const uint32_t ro = (uint32_t)(8 * JC) * (k8LDC * 4);
    const bool own = (tj == 0);
    sts128x2_if(own, pTi + ro, A[0][JC], A[1][JC]);
    sts128x2_if(own, pTi + ro + 16, A[2][JC], A[3][JC]);
    sts32_if(ti == TI0 && tj == JR, Y + (uint32_t)(8 * JC) * 4u, bb);
    bar_sync_n(bar, 128);
  }
#pragma unroll 1
  for (int jm = 0; jm < 8; ++jm) {
    const int j = 8 * JC + jm;
    const uint32_t ro = (uint32_t)j * (k8LDC * 4);
    f32x2 w[4], le[4], lo[4];
    lds128x2(pTi + ro, w[0], w[1]);
    lds128x2(pTi + ro + 16, w[2], w[3]);
    // le[q] = local columns 4q, 4q+2 ; lo[q] = local columns 4q+1, 4q+3 ; dead quads are not loaded
    if (2 >= JC) lds128x2(pTjE + ro, le[0], le[1]); else if (6 >= JC) le[1] = lds64x2(pTjE + ro + 8);
    if (10 >= JC) lds128x2(pTjE + ro + 16, le[2], le[3]); else if (14 >= JC) le[3] = lds64x2(pTjE + ro + 24);
    if (3 >= JC) lds128x2(pTjO + ro, lo[0], lo[1]); else if (7 >= JC) lo[1] = lds64x2(pTjO + ro + 8);
    if (11 >= JC) lds128x2(pTjO + ro + 16, lo[2], lo[3]); else lo[3] = lds64x2(pTjO + ro + 24);
    const float d = lds32(Pall + ro + (uint32_t)((TI0 + jm) * 8 + JR) * 4u);
    const float yj = lds32(Y + (uint32_t)j * 4u);
    const float lm = lds32(pMine + ro);
    const float ninv = -__fdividef(1.0f, d);
    const f32x2 ninv2 = pack2(ninv, ninv);
#pragma unroll
    for (int rp = RP0; rp < 4; ++rp) w[rp] = ffma2(w[rp], ninv2, 0ull);
    {   // rows <= j are finished: zero multiplier (local row JR iff ti <= TI0 + jm; JR-1, if in the pair, always)
      float l0 = lo2(w[RP0]), h0 = hi2(w[RP0]);
      if (JR & 1) { l0 = 0.f; h0 = (ti > TI0 + jm) ? h0 : 0.f; }
      else l0 = (ti > TI0 + jm) ? l0 : 0.f;
      w[RP0] = pack2(l0, h0);
    }
    auto colval = [&](int c) -> float {
      const f32x2 src = (c & 1) ? lo[c >> 2] : le[c >> 2];
      return (c & 2) ? hi2(src) : lo2(src);
    };
    {   // the block's pivot column first (columns <= j are finished: zero for tj <= jm) ...
      const float l = (tj > jm) ? colval(JC) : 0.f;
      const f32x2 l2 = pack2(l, l);
#pragma unroll
      for (int rp = RP0; rp < 4; ++rp) A[rp][JC] = ffma2(w[rp], l2, A[rp][JC]);
    }
    const bool act = (tj > JR) || (tj == JR && ti > TI0 + jm);   // my right-hand-side row ti + 16*tj is below the pivot
    bb = act ? fmaf(lm * ninv, yj, bb) : bb;
    if (jm < 7) {   // ... so that column j+1 goes out before the rest of the update
      const bool own = (tj == jm + 1);
      const uint32_t r1 = ro + k8LDC * 4;
      sts128x2_if(own, pTi + r1, A[0][JC], A[1][JC]);
      sts128x2_if(own, pTi + r1 + 16, A[2][JC], A[3][JC]);
      sts32_if(ti == TI0 + jm + 1 && tj == JR, Y + (uint32_t)(j + 1) * 4u, bb);
      bar_sync_n(bar, 128);
    }
#pragma unroll
    for (int c = JC + 1; c < 16; ++c) {
      const float l = colval(c);
      const f32x2 l2 = pack2(l, l);
#pragma unroll
      for (int rp = RP0; rp < 4; ++rp) A[rp][c] = ffma2(w[rp], l2, A[rp][c]);
    }
  }
}

// C (row stride k8LDC): rows m of 0.5*D_hh + D_hl, so that A = C + C^T; B: right-hand side.  Pall aliases C.
// s = thread index inside the solver group (0..127); bar = the group's named barrier.  Returns x_s.
__device__ __noinline__ float als128_solve_tile(uint32_t C, uint32_t B, float lam, int s, int bar) {
  const int ti = s >> 3, tj = s & 7, lane = s & 31, wq = s >> 5;
  const uint32_t Pall = C, Y = B + 512, Z = Y + 512, X = Z + 512;
  f32x2 A[4][16];
#pragma unroll
  for (int rp = 0; rp < 4; ++rp) {
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const int n = tj + 8 * c;
      float v[2];
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        const int m = ti + 32 * rp + 16 * x;
        v[x] = lds32(C + (uint32_t)(m * k8LDC + n) * 4u) + lds32(C + (uint32_t)(n * k8LDC + m) * 4u) + (m == n ? lam : 0.f);
      }
      A[rp][c] = pack2(v[0], v[1]);
    }
  }
  float bb = lds32(B + (uint32_t)(ti + 16 * tj) * 4u);
  bar_sync_n(bar, 128);                                  // every thread holds its tile: Pall may overwrite C
  const uint32_t pTi = Pall + (uint32_t)ti * 32u, pTjE = Pall + (uint32_t)tj * 32u, pTjO = Pall + (uint32_t)(tj + 8) * 32u;
  const uint32_t pMine = Pall + (uint32_t)(ti * 8 + tj) * 4u;
  ldlt128_tile_block<0>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<1>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<2>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<3>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<4>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<5>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<6>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<7>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<8>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<9>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<10>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<11>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<12>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<13>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<14>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  ldlt128_tile_block<15>(A, bb, pTi, pTjE, pTjO, pMine, Pall, Y, ti, tj, bar);
  // z = L^-1 b: element ti + 16*tj sits in this thread; hand row m's entry to thread m = s
  sts32(Z + (uint32_t)(ti + 16 * tj) * 4u, bb);
  bar_sync_n(bar, 128);
  const int m = s;
  const uint32_t rowm = Pall + (uint32_t)m * (k8LDC * 4);
  // entry j of column m of L*D sits at position (j % 16) * 8 + j / 16 of Pall row m
  auto elem = [&](int j) -> float { return lds32(rowm + (uint32_t)((j & 15) * 8 + (j >> 4)) * 4u); };
  float acc = lds32(Z + (uint32_t)m * 4u), x = 0.f;
  const float inv_d = __fdividef(1.0f, elem(m));
  // x_c = (z_c - sum_{j>c} (L D)[j][c] x_j) / d_c, last warp first
#pragma unroll 1
  for (int wv = 3; wv >= 0; --wv) {
    if (wq == wv) {
#pragma unroll 8
      for (int j = 127; j >= 32 * (wv + 1); --j) acc = fmaf(-elem(j), lds32(X + (uint32_t)j * 4u), acc);
#pragma unroll 8
      for (int jl = 31; jl >= 0; --jl) {                 // own block: pivot 32 wv + jl lives in lane jl
        const float lj = elem(32 * wv + jl);
        const float xj = __shfl_sync(0xffffffffu, acc * inv_d, jl);
        if (lane == jl) x = xj;
        if (lane < jl) acc = fmaf(-lj, xj, acc);
      }
      sts32(X + (uint32_t)m * 4u, x);
    }
    if (wv > 0) bar_sync_n(bar, 128);
  }
  return x;
}

// Producer warps (0 and 1) of both rank-128 kernels: gather the h|l rows of every work item into the stage ring
// and issue the three MMAs per 16 ratings; `mbar_acc[it & 1]` signals "accumulator of item it complete",
// `mbar_tmem_free` is awaited before the first MMA of the next item.
__device__ __forceinline__ void als128_producer(uint8_t* base, uint32_t sbase, uint32_t tmem, uint64_t* mbar_free,
                                                uint64_t* mbar_acc, uint64_t* mbar_tmem_free,
                                                const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                                const __nv_bfloat16* __restrict__ src_hl,
                                                const int64_t* __restrict__ item_begin, const int32_t* __restrict__ item_len,
                                                int64_t n_items) {
  constexpr int K = k8K, KC = k8KC;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // ================================================================ producers
    constexpr uint32_t idesc256 = umma::make_instr_desc(umma::kFmtBF16, true, true, 128, 256);
    constexpr uint32_t idesc16 = umma::make_instr_desc(umma::kFmtBF16, true, true, 128, 16);
    const int t_sub = tid >> 5, piece = tid & 31;        // 2 rating rows per pass, 32 x 16-byte pieces per 512 B row
    const int blk_off = (piece >> 3) * k8Blk, chunk = piece & 7;
    uint32_t g = 0, it = 0;
    for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int64_t begin = item_begin[item];
      const int len = item_len[item];
      const int nc = (len + KC - 1) / KC;
      auto fetch_idx = [&](int c, int& ci, float& rv) {
        const int q = c * KC + lane;
        const bool ok = q < len;
        ci = ok ? __ldg(colidx + begin + q) : -1;
        rv = (ok && warp == 0) ? __ldg(vals + begin + q) : 0.f;
      };
      int ci_cur, ci_nxt = -1;
      float rv_cur, rv_nxt = 0.f;
      fetch_idx(0, ci_cur, rv_cur);
      if (nc > 1) fetch_idx(1, ci_nxt, rv_nxt);
      auto produce = [&](int c) {
        const uint32_t gi = g + c, s = gi % k8Stages, u = gi / k8Stages;
        if (u > 0) umma::mbar_wait(&mbar_free[s], (u - 1) & 1);
        uint8_t* st = base + s * k8StageBytes;
#pragma unroll
        for (int i = 0; i < KC / 2; ++i) {
          const int t = t_sub + 2 * i;
          const int ci = __shfl_sync(0xffffffffu, ci_cur, t);
          cp_async16(st + blk_off + t * 128 + ((chunk ^ (t & 7)) << 4),
                     reinterpret_cast<const uint8_t*>(src_hl) + (size_t)(ci < 0 ? 0 : ci) * (4 * K) + piece * 16, ci >= 0);
        }
        if (warp == 0) {   // rating columns: element 0 = bf16(r), element 1 = bf16(r - bf16(r))
          const __nv_bfloat16 rh = __float2bfloat16_rn(rv_cur);
          const __nv_bfloat16 rl = __float2bfloat16_rn(rv_cur - __bfloat162float(rh));
          const uint32_t packed = (uint32_t)__bfloat16_as_ushort(rh) | ((uint32_t)__bfloat16_as_ushort(rl) << 16);
          *reinterpret_cast<uint4*>(st + 4 * k8Blk + lane * 128 + ((0 ^ (lane & 7)) << 4)) = make_uint4(packed, 0u, 0u, 0u);
          *reinterpret_cast<uint4*>(st + 4 * k8Blk + lane * 128 + ((1 ^ (lane & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
        }
        cp_async_commit();
        ci_cur = ci_nxt; rv_cur = rv_nxt;
        if (c + 2 < nc) fetch_idx(c + 2, ci_nxt, rv_nxt);
      };
      for (int c = 0; c < k8Ahead; ++c) {
        if (c < nc) produce(c); else cp_async_commit();
      }
      for (int c = 0; c < nc; ++c) {
        if (c + k8Ahead < nc) produce(c + k8Ahead); else cp_async_commit();
        cp_async_wait<k8Ahead>();
        umma::fence_proxy_async();
        bar_sync_n(1, 64);
        if (tid == 0) {
          if (c == 0 && it > 0) umma::mbar_wait(mbar_tmem_free, (it - 1) & 1);   // previous accumulator drained
          umma::fence_after_sync();
          const uint32_t s = (g + c) % k8Stages;
          const uint32_t sa = sbase + s * k8StageBytes;
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks) {
            const uint64_t dH = umma::make_smem_desc(sa + ks * 2048, k8Blk, 1024, umma::kSwizzle128B);
            const uint64_t dL = umma::make_smem_desc(sa + 2 * k8Blk + ks * 2048, k8Blk, 1024, umma::kSwizzle128B);
            const uint64_t dR = umma::make_smem_desc(sa + 4 * k8Blk + ks * 2048, k8Blk, 1024, umma::kSwizzle128B);
            const bool accum = (c | ks) != 0;
            umma::mma_bf16(tmem, dH, dH, idesc256, accum);          // H^T [H | L]: the B descriptor walks H0 H1 L0 L1
            umma::mma_bf16(tmem + 256, dH, dR, idesc16, accum);     // H^T R
            umma::mma_bf16(tmem + 272, dL, dR, idesc16, accum);     // L^T R
          }
          umma::commit(&mbar_free[s]);
          if (c == nc - 1) umma::commit(&mbar_acc[it & 1]);
        }
      }
      g += nc;
    }
}

__global__ void __launch_bounds__(k8Threads, 1)
als_tc128_kernel(const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                 const __nv_bfloat16* __restrict__ src_hl, float* __restrict__ dst, float reg,
                 const int32_t* __restrict__ item_row, const int64_t* __restrict__ item_begin,
                 const int32_t* __restrict__ item_len, const int32_t* __restrict__ item_slot,
                 int64_t n_items, float* __restrict__ workspace) {
  constexpr int K = k8K;
  extern __shared__ uint8_t smem_dyn[];
  __shared__ uint64_t mbar_free[k8Stages];
  __shared__ uint64_t mbar_acc[2];        // accumulator complete, one per solver group
  __shared__ uint64_t mbar_tmem_free;     // accumulator drained
  __shared__ uint32_t tmem_slot;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool producer = warp < 2;
  const int group = producer ? -1 : (warp - 2) >> 2;
  const int m = 32 * (warp & 3) + lane;                 // solver: matrix row == TMEM lane
  if (warp == 0) umma::tmem_alloc(&tmem_slot, 512);
  if (tid == 0) {
    for (int s = 0; s < k8Stages; ++s) umma::mbar_init(&mbar_free[s], 1);
    umma::mbar_init(&mbar_acc[0], 1);
    umma::mbar_init(&mbar_acc[1], 1);
    umma::mbar_init(&mbar_tmem_free, 1);
    umma::mbar_fence_init();
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint32_t sbase = umma::smem_u32(base);

  if (producer) {
    als128_producer(base, sbase, tmem, mbar_free, mbar_acc, &mbar_tmem_free, colidx, vals, src_hl, item_begin, item_len, n_items);
  } else {
    // ================================================================ solver groups
    const uint32_t sC = umma::smem_u32(base + k8Stages * k8StageBytes + group * k8GroupBytes);   // C, later Pall
    const uint32_t sB = sC + 128 * k8LDC * 4;             // b | y | z | x rows (128 floats each)
    const int bar = 2 + group;                            // named barrier of this group (1 = producers)
    const uint32_t ta = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
    uint32_t it = 0, mine = 0;
    for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      if ((int)(it & 1) != group) continue;
      const int row = item_row[item];
      const int len = item_len[item];
      const int slot = item_slot[item];
      umma::mbar_wait(&mbar_acc[group], mine & 1);
      ++mine;
      umma::fence_after_sync();
      // drain: row m of C = D_hh / 2 + D_hl goes to shared memory (A = C + C^T), then the accumulator is free
      {
        float v[32], u[32];
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          umma::tmem_ld32(ta + c0, v);
          umma::tmem_ld32(ta + 128 + c0, u);
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            sts128(sC + (uint32_t)(m * k8LDC + c0 + i) * 4u, fmaf(0.5f, v[i], u[i]), fmaf(0.5f, v[i + 1], u[i + 1]),
                   fmaf(0.5f, v[i + 2], u[i + 2]), fmaf(0.5f, v[i + 3], u[i + 3]));
        }
        float e1[16], e2[16];
        umma::tmem_ld16(ta + 256, e1);
        umma::tmem_ld16(ta + 272, e2);
        sts32(sB + (uint32_t)m * 4u, e1[0] + e1[1] + e2[0]);
      }
      umma::fence_before_sync();
      bar_sync_n(bar, 128);                               // C complete, every TMEM read of this item done
      if (m == 0) umma::mbar_arrive(&mbar_tmem_free);
      if (slot >= 0) {
        // slice of a long row: thread = row m parks (A, b, n) in the slot (same layout as the SIMT path)
        float* W = workspace + (size_t)slot * k8SlotFloats;
#pragma unroll 4
        for (int n = 0; n < 128; n += 4) {
          const float4 q = lds128(sC + (uint32_t)(m * k8LDC + n) * 4u);
          *reinterpret_cast<float4*>(W + m * K + n) =
              make_float4(q.x + lds32(sC + (uint32_t)((n) * k8LDC + m) * 4u), q.y + lds32(sC + (uint32_t)((n + 1) * k8LDC + m) * 4u),
                          q.z + lds32(sC + (uint32_t)((n + 2) * k8LDC + m) * 4u), q.w + lds32(sC + (uint32_t)((n + 3) * k8LDC + m) * 4u));
        }
        W[K * K + m] = lds32(sB + (uint32_t)m * 4u);
        if (m == 0) W[K * K + K] = (float)len;
      } else {
        const float x = als128_solve_tile(sC, sB, reg * (float)len, m, bar);
        dst[(int64_t)row * K + m] = x;
      }
      bar_sync_n(bar, 128);                               // C / Pall and the hand-over rows are reused by the next item
    }
  }

  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, 512);
}

// Long rows (rank 128): slot sums (pre-summed per group of 16 by als_slot_group_sum_kernel) + ridge + solve.
__global__ void __launch_bounds__(128)
als_reduce_solve128_kernel(const float* __restrict__ workspace, float* __restrict__ dst, float reg,
                           const int32_t* __restrict__ long_row, const int32_t* __restrict__ long_slot0,
                           const int32_t* __restrict__ long_nseg, __nv_bfloat16* __restrict__ dst_hl,
                           const float* __restrict__ gram) {
  constexpr int K = k8K;
  __shared__ __align__(16) float PS[2 * k8LDP + 128];
  const int m = threadIdx.x;
  const int row = long_row[blockIdx.x];
  const int s0 = long_slot0[blockIdx.x], ns = long_nseg[blockIdx.x];
  float a[128];
#pragma unroll
  for (int n = 0; n < 128; ++n) a[n] = 0.f;
  float bm = 0.f, cnt = 0.f;
  const int stride = slot_final_stride(ns);               // rows with many slices were pre-summed per group (two levels)
  for (int q = 0; q < ns; q += stride) {
    const float* W = workspace + (size_t)(s0 + q) * k8SlotFloats;
#pragma unroll
    for (int n = 0; n < 128; n += 4) {
      const float4 v = *reinterpret_cast<const float4*>(W + m * K + n);
      a[n] += v.x; a[n + 1] += v.y; a[n + 2] += v.z; a[n + 3] += v.w;
    }
    bm += W[K * K + m];
    cnt += W[K * K + K];
  }
  const float lam = reg * cnt;
  if (gram != nullptr) {                                   // implicit feedback: + Y^T Y (row m of the symmetric matrix)
#pragma unroll
    for (int n = 0; n < 128; n += 4) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gram + m * K + n));
      a[n] += g.x; a[n + 1] += g.y; a[n + 2] += g.z; a[n + 3] += g.w;
    }
  }
  f32x2 ap[64];
#pragma unroll
  for (int i = 0; i < 64; ++i)
    ap[i] = pack2(a[2 * i] + (2 * i == m ? lam : 0.f), a[2 * i + 1] + (2 * i + 1 == m ? lam : 0.f));
  const uint32_t P = umma::smem_u32(PS);
  const float x = ldlt128_rows(ap, bm, P, P + 2 * k8LDP * 4, m, 1);
  dst[(int64_t)row * K + m] = x;
  if (dst_hl) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    dst_hl[(int64_t)row * (2 * K) + m] = h;
    dst_hl[(int64_t)row * (2 * K) + K + m] = __float2bfloat16_rn(x - __bfloat162float(h));
  }
}

int als_half_step_tc128(const int32_t* colidx, const float* vals, const float* src, int64_t n_src, float* dst,
                        float reg, const hals_als_plan* plan, float* slots, void* split_buf, cudaStream_t st) {
  __nv_bfloat16* hl = reinterpret_cast<__nv_bfloat16*>(split_buf);
  if (int rc = als_launch_split_bf16(src, n_src, k8K, split_buf, st)) return rc;
  // (a two-threads-per-row variant of the solver was measured slower: 208 vs 129 ms / sweep on c3 -- the
  //  256-thread step barrier and the extra column exchange cost more than the shorter per-thread stream saves)
  int64_t grid = sm_count();
  if (grid > plan->n_items) grid = plan->n_items;
  const size_t smem = (size_t)k8Stages * k8StageBytes + 2 * (size_t)k8GroupBytes + 1024;
  HALS_CUDA(cudaFuncSetAttribute(als_tc128_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  als_tc128_kernel<<<(unsigned)grid, k8Threads, smem, st>>>(colidx, vals, hl, dst, reg, plan->item_row, plan->item_begin,
                                                             plan->item_len, plan->item_slot, plan->n_items, slots);
  HALS_LAUNCH_CHECK();
  if (plan->n_long_rows > 0) {
    if (int rc = als_launch_slot_group_sum(slots, plan, (int)k8SlotFloats, st)) return rc;
    als_reduce_solve128_kernel<<<(unsigned)plan->n_long_rows, 128, 0, st>>>(slots, dst, reg, plan->long_row,
                                                                            plan->long_slot0, plan->long_nseg, nullptr, nullptr);
    HALS_LAUNCH_CHECK();
  }
  return 0;
}

// the long-row tail of the warp-specialised kernel (als_ws128.cu); the slot groups are already pre-summed
int als_launch_reduce_solve128(const float* slots, float* dst, float reg, const hals_als_plan* plan, void* dst_hl,
                               const float* gram, cudaStream_t st) {
  als_reduce_solve128_kernel<<<(unsigned)plan->n_long_rows, 128, 0, st>>>(slots, dst, reg, plan->long_row, plan->long_slot0,
                                                                          plan->long_nseg, reinterpret_cast<__nv_bfloat16*>(dst_hl),
                                                                          gram);
  HALS_LAUNCH_CHECK();
  return 0;
}

}  // namespace hals
