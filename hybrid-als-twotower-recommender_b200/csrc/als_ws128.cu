// ALS half-step, rank 128, warp-specialised persistent kernel (the default rank-128 path; Netflix-shape config 3).
// Replaces Spark's NormalEquation.add (dspr/daxpy per rating) and CholeskySolver.solve (dppsv) reached from
// src/als_model.py:62.  Arithmetic of als_tc128.cu (bf16 hi/lo split operands, three tcgen05.mma per 16 ratings,
// fp32 accumulation in TMEM, A = D_hh + D_hl + D_hl^T, square-root-free Cholesky); pipeline of als_ws64.cu:
//
//   one CTA per SM with a contiguous, equal-cost share of the plan's work items; 16 warps, mbarrier-linked roles
//     G  warps 12-13 gather: alternate 32-rating chunks of the CTA's chunk table, cp.async of the 512-byte h|l rows
//                    (one warp instruction = one row) into the swizzled MN-major stage, completion through the
//                    stage's mbarrier; column indices prefetched two bursts of 8 chunks ahead
//     M  warp 14     one elected thread: per 16 ratings  H^T [H | L] (N = 256),  H^T R and L^T R (N = 16 each)
//                    into THE accumulator (288 of the 512 TMEM columns: one row in the tensor pipe at a time)
//     S  warps 0-11  three solver groups of four warps (a group covers the four TMEM lane quarters): drain row m of
//                    C = D_hh / 2 + D_hl per thread into the shared hand-over matrix, release the accumulator, load the
//                    group's register tile A = C + C^T, release the hand-over matrix, solve.  Groups take rows
//                    round-robin: drain + tile load are serialised through the single hand-over matrix
//                    (~3.5k cycles per row), the 128-pivot eliminations of three rows overlap.
//   Implicit feedback (Hu-Koren, Spark implicitPrefs): A = Y^T Y + sum c y y^T + lambda n+ I, b = sum_{r>0} (1 + c) y with
//   c = alpha |r|.  Warp 15 rescales every landed stage in place, row t by sqrt(c_t) (s = sqrt(c) (h + l) in fp32, re-split
//   into bf16 hi/lo), so the SAME three MMAs build sum c y y^T; the rating column carries (1 + c) / sqrt(c) (0 unless
//   r > 0), so H^T R is b; the Gram matrix, permuted once per half-step into the solver's lane-tile order, is added when a
//   group loads its tile; n+ (ratings > 0 per work item) comes with the plan.
//   Solver = the one-tile-per-lane L D L^T of als_ws64.cu on 128 lanes: lane (ti = 0..7, tj = 0..15) owns rows
//   {ti + 16q, ti + 8 + 16q} x columns {tj + 16c} of the lower triangle (36 packed fp32x2), pivot columns go through
//   a 512-byte buffer, ONE named barrier of the group per pivot.  (The round-1 kernel, als_tc128.cu: two groups, full
//   square tiles, every published column kept in shared memory: 560 cycles per pivot step, 84 ms per c3 sweep.)
#include <cuda_bf16.h>

#include <cstdlib>

#include "als_ws_common.cuh"

namespace hals {
namespace ws128 {
using namespace ws;

constexpr int K = 128;
constexpr int kStageBytes = stage_bytes(K);  // H0 | H1 | L0 | L1 | R
constexpr int kStages = 6;
constexpr int kLdc = 132;                    // hand-over row stride (floats)
constexpr int kCBytes = 128 * kLdc * 4 + 512;            // C | b
constexpr int kGroups = 3;
constexpr int kGroupScratch = 4096;          // P (2 x 512) | Y (512) | DI (512) | T (1024) | RH (64) | X (512)
constexpr int kThreads = 512;
constexpr int kWarpGather = 12, kWarpMma = 14;
// setmaxnreg (warpgroup-wide): the kernel is compiled for 128 registers per thread; the front-end warpgroup (warps
// 12-15) gives 56 per thread back, which lets the three solver warpgroups grow to 144 -- room for the loads of the
// next pivot next to the operands of the current trailing update (checked on the host before the launch).
constexpr int kRegsLaunch = 128, kRegsFront = 72, kRegsSolver = 144;
static_assert((kThreads / 32 - 4 * kGroups) * (kRegsLaunch - kRegsFront) >= 4 * kGroups * (kRegsSolver - kRegsLaunch), "register pool");
constexpr size_t kSlotFloats = (size_t)K * K + K + 4;
static_assert(kStages % 2 == 0, "the two gather warps own alternate stages");

struct Bars {
  uint64_t st_full[kStages], st_free[kStages];
  uint64_t st_scaled[kStages];     // implicit mode: stage rescaled by sqrt(c) (what the MMA warp then waits for)
  uint64_t acc_full[kGroups];      // accumulator of a row complete, per destination group (a waiter may lag one phase)
  uint64_t acc_free;               // accumulator drained (128 arrivals of the draining group)
  uint64_t c_turn[kGroups];        // hand-over matrix free for group g's next row (arrival by the group before it)
};

// ---- G: gather (see als_ws64.cu for the scheme; here one warp instruction copies one 512-byte row) -------------
__device__ __noinline__ void gather_role(uint32_t stages, Bars* bars, uint8_t* gscratch, const Range* rg,
                                         const int32_t* __restrict__ colidx, const uint32_t* __restrict__ vals_hl,
                                         const float* __restrict__ vals_sc, const uint8_t* __restrict__ src_hl, int zero_row,
                                         const int64_t* __restrict__ chunk_pos, const int32_t* __restrict__ chunk_cnt,
                                         int gw, int lane) {
  const uint32_t ring = umma::smem_u32(gscratch);                       // int  [2][kBurst][32]
  const uint32_t mpos = ring + 2 * kBurst * 128;                        // i64  [2][kBurst]
  const uint32_t mcnt = mpos + 2 * kBurst * 8;                          // int  [2][kBurst]
  const int64_t k_hi = rg->chunk_hi;
  int64_t kw = rg->chunk_lo + gw;
  auto load_window = [&](int64_t& p, int& c) {
    const int64_t k = kw + 2 * lane;
    p = 0; c = 0;
    if (k < k_hi) { p = __ldg(chunk_pos + k); c = __ldg(chunk_cnt + k); }
    kw += 64;
  };
  int64_t wpos, npos;
  int wcnt, ncnt;
  load_window(wpos, wcnt);
  load_window(npos, ncnt);
  int wb = 0;
  int ci[kBurst];
  auto fill = [&](int buf) {
    if (lane >= wb * kBurst && lane < (wb + 1) * kBurst) {
      const uint32_t e = (uint32_t)(buf * kBurst + lane - wb * kBurst);
      asm volatile("st.shared.b64 [%0], %1;\n" ::"r"(mpos + e * 8u), "l"(wpos) : "memory");
      asm volatile("st.shared.b32 [%0], %1;\n" ::"r"(mcnt + e * 4u), "r"(wcnt) : "memory");
    }
#pragma unroll
    for (int c = 0; c < kBurst; ++c) {
      const int64_t pos = __shfl_sync(0xffffffffu, wpos, wb * kBurst + c);
      const int cnt = __shfl_sync(0xffffffffu, wcnt, wb * kBurst + c);
      ci[c] = lane < cnt ? __ldg(colidx + pos + lane) : zero_row;
    }
    if (++wb == 32 / kBurst) {
      wb = 0;
      wpos = npos; wcnt = ncnt;
      load_window(npos, ncnt);
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int c = 0; c < kBurst; ++c) sts32(ring + (uint32_t)((buf * kBurst + c) * 32 + lane) * 4u, __int_as_float(ci[c]));
    __syncwarp();
  };
  // lane = 16-byte piece of the 512-byte row: atom lane / 8 (H0 H1 L0 L1), chunk (lane % 8) ^ (t % 8) of row t
  uint32_t dsto[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) dsto[i] = (uint32_t)(lane >> 3) * kBlk + (uint32_t)(((lane & 7) ^ i) << 4);
  const uint64_t srcb = reinterpret_cast<uint64_t>(src_hl) + (uint64_t)lane * 16u;
  const uint32_t rdst = 4 * kBlk + (uint32_t)lane * kRowBytes + (uint32_t)((lane & 7) << 4);
  const uint32_t sdst = 4 * kBlk + (uint32_t)lane * kRowBytes + (uint32_t)((7 ^ (lane & 7)) << 4);   // a chunk no MMA reads
  uint32_t s = (uint32_t)gw, u = 0;
  fill(0);
  stash(0);
  fill(1);
  for (int buf = 0;; buf ^= 1) {
    bool done = false;
#pragma unroll 1
    for (int c = 0; c < kBurst; ++c) {
      int cnt;
      asm volatile("ld.shared.b32 %0, [%1];\n" : "=r"(cnt) : "r"(mcnt + (uint32_t)(buf * kBurst + c) * 4u));
      if (cnt <= 0) { done = true; break; }
      int64_t pos;
      asm volatile("ld.shared.b64 %0, [%1];\n" : "=l"(pos) : "r"(mpos + (uint32_t)(buf * kBurst + c) * 8u));
      if (u > 0) umma::mbar_wait(&bars->st_free[s], (u - 1) & 1);
      const uint32_t st = stages + s * kStageBytes;
      const uint32_t ir = ring + (uint32_t)((buf * kBurst + c) * 32) * 4u;
#pragma unroll
      for (int h = 0; h < 2; ++h) {          // 16 ratings at a time (register budget of the index vectors)
        const float4 c0 = lds128(ir + h * 64), c1 = lds128(ir + h * 64 + 16), c2 = lds128(ir + h * 64 + 32),
                     c3 = lds128(ir + h * 64 + 48);
        const float colf[16] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w, c3.x, c3.y, c3.z, c3.w};
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int t = 16 * h + i;
          uint64_t src;
          asm("mad.wide.u32 %0, %1, 512, %2;\n" : "=l"(src) : "r"((uint32_t)__float_as_int(colf[i])), "l"(srcb));
          cp_async16_raw(st + dsto[t & 7] + (uint32_t)t * kRowBytes, src);
        }
      }
      {
        const bool ok = lane < cnt;
        const uint32_t* rp = vals_hl + pos + (ok ? lane : 0);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(st + rdst), "l"(rp), "r"(ok ? 4 : 0) : "memory");
        if (vals_sc != nullptr) {
          const float* sp = vals_sc + pos + (ok ? lane : 0);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(st + sdst), "l"(sp), "r"(ok ? 4 : 0) : "memory");
        }
      }
      cp_async_mbar_arrive_noinc(&bars->st_full[s]);
      s += 2;
      if (s >= (uint32_t)kStages) { s -= kStages; ++u; }
    }
    if (done) break;
    stash(buf ^ 1);
    fill(buf);
  }
}

__device__ __noinline__ void scaler_role(uint32_t stages, Bars* bars, const Range* rg, int lane) {
  scale_stages<K, kStages>(stages, bars, rg, lane);
}

// ---- M: MMA issue --------------------------------------------------------------------------------------------
__device__ __noinline__ void mma_role(uint32_t sbase, uint32_t tmem, Bars* bars, const Range* rg,
                                      const int32_t* __restrict__ chunk_cnt, bool scaled, int lane) {
  uint64_t* const ready = scaled ? bars->st_scaled : bars->st_full;
  constexpr uint32_t idesc256 = umma::make_instr_desc(umma::kFmtBF16, true, true, 128, 256);
  constexpr uint32_t idesc16 = umma::make_instr_desc(umma::kFmtBF16, true, true, 128, 16);
  const int64_t k_lo = rg->chunk_lo, k_hi = rg->chunk_hi;
  uint32_t s = 0, su = 0, row = 0;
  bool first = true;
  int wc = 0, nc = 0;
  if (k_lo + lane < k_hi) wc = __ldg(chunk_cnt + k_lo + lane);
  if (k_lo + 32 + lane < k_hi) nc = __ldg(chunk_cnt + k_lo + 32 + lane);
  const bool leader = elect_one();
  const uint64_t dH0 = umma::make_smem_desc(sbase, kBlk, 1024, umma::kSwizzle128B);                 // H0 H1 (L0 L1)
  const uint64_t dL0 = umma::make_smem_desc(sbase + 2 * kBlk, kBlk, 1024, umma::kSwizzle128B);      // L0 L1
  const uint64_t dR0 = umma::make_smem_desc(sbase + 4 * kBlk, kBlk, 1024, umma::kSwizzle128B);      // R
  for (int64_t kb = k_lo; kb < k_hi; kb += 32) {
    const int nk = (int)(k_hi - kb < 32 ? k_hi - kb : 32);
    for (int i = 0; i < nk; ++i) {
      const int cnt = __shfl_sync(0xffffffffu, wc, i);
      if (leader) {
        if (first) {
          if (row > 0) umma::mbar_wait(&bars->acc_free, (row - 1) & 1);     // the previous row has left TMEM
          umma::fence_after_sync();
        }
        umma::mbar_wait(&ready[s], su & 1);
        const uint64_t so = (uint64_t)((s * kStageBytes) >> 4);
#pragma unroll
        for (int ks = 0; ks < KC / 16; ++ks) {
          const uint64_t ko = so + (uint64_t)(ks * 2048 >> 4);
          const bool accum = !(first && ks == 0);
          umma::mma_bf16(tmem, dH0 + ko, dH0 + ko, idesc256, accum);          // H^T [H | L]
          umma::mma_bf16(tmem + 256, dH0 + ko, dR0 + ko, idesc16, accum);     // H^T R
          umma::mma_bf16(tmem + 272, dL0 + ko, dR0 + ko, idesc16, accum);     // L^T R
        }
        umma::commit(&bars->st_free[s]);
        if (cnt <= KC) umma::commit(&bars->acc_full[row % kGroups]);
      }
      __syncwarp();
      first = cnt <= KC;
      if (first) ++row;
      if (++s == (uint32_t)kStages) { s = 0; ++su; }
    }
    wc = nc;
    nc = 0;
    if (kb + 64 + lane < k_hi) nc = __ldg(chunk_cnt + kb + 64 + lane);
  }
}

// ---- S: a group of four warps solves one 128 x 128 system -------------------------------------------------------
__device__ __forceinline__ void group_sync(int bar) { asm volatile("bar.sync %0, 128;\n" ::"r"(bar) : "memory"); }

// Pivot j = 16*JR + jm.  Row m = ti + 8*half + 16*q of the tile, column n = tj + 16*c.  The eight lanes with tj == jm
// publish column j; everybody reads its row multipliers (packed pairs), its column values and the published -1/d.
// Shared-memory passes, not issue slots, bound this loop (twelve warps share one 128-byte-per-clock pipe), so the
// layout of the published column is P[q / 2][ti][q % 2][half]: a 16-byte read of the eight rows ti of a quarter warp
// covers the 32 banks exactly once, and so does the publishing quarter warp's 16-byte store.  (First version:
// P[ti][q][half], 4-way conflicts on both: 827 cycles per pivot step on c3.)  Right-hand side rows (ti + 16 tj,
// ti + 8 + 16 tj) live in the lanes with tj < 8.  Same reasoning as als_ws64.cu for everything else.
template <int JR>
struct PivotIn {                      // what a lane reads of one published pivot column
  f32x2 w[8];                         // multipliers of its rows (before scaling by -1/d), entries q >= JR
  float l[8];                         // column values of its columns, entries c >= JR
  float ninv, zj;
  f32x2 wb;                           // multipliers of its right-hand-side rows
};

template <int JR>
__device__ __forceinline__ void elim_block(f32x2 (&R)[36], f32x2& bb2, const uint32_t P, const uint32_t Y,
                                           const uint32_t DI, const int ti, const int tj, const int gl, const int bar) {
  const uint32_t oW = (uint32_t)ti * 16u;                                        // + (q / 2) * 128 + (q % 2) * 8
  const uint32_t oL = (uint32_t)(tj & 7) * 16u + (uint32_t)(tj >> 3) * 4u;       // + (c / 2) * 128 + (c % 2) * 8
  const uint32_t oB = oW + (uint32_t)((tj & 7) >> 1) * 128u + (uint32_t)(tj & 1) * 8u;
  auto publish = [&](uint32_t Pn, bool own) {
    if (JR & 1) sts64_if(own, Pn + oW + (JR >> 1) * 128 + 8, R[tri(JR, JR)]);
#pragma unroll
    for (int q = (JR + 1) & ~1; q < 8; q += 2) sts128x2_if(own, Pn + oW + (q >> 1) * 128, R[tri(q, JR)], R[tri(q + 1, JR)]);
  };
  const bool rhs_warp = tj < 8;
  auto load = [&](PivotIn<JR>& in, int jm) {
    const uint32_t Pj = P + ((uint32_t)(jm & 1) << 9);
    const uint32_t j4 = (uint32_t)(16 * JR + jm) * 4u;
    if (JR & 1) in.w[JR] = lds64x2(Pj + oW + (JR >> 1) * 128 + 8);
#pragma unroll
    for (int q = (JR + 1) & ~1; q < 8; q += 2) lds128x2(Pj + oW + (q >> 1) * 128, in.w[q], in.w[q + 1]);
    in.ninv = lds32(DI + j4);
#pragma unroll
    for (int c = JR; c < 8; ++c) in.l[c] = lds32(Pj + oL + (c >> 1) * 128 + (c & 1) * 8);
    if (rhs_warp) {                   // warp-uniform: the right-hand side lives in the lanes with tj < 8
      in.zj = lds32(Y + j4);
      in.wb = lds64x2(Pj + oB);
    }
  };
  const bool below = tj > JR;
  const bool on = tj == JR;
  // One pivot: finish column JR of the tile (it holds the next pivot column), publish that column, barrier, THEN
  // issue the loads of the next pivot and run the trailing update of this one under their latency.
  auto step = [&](PivotIn<JR>& in, PivotIn<JR>& nx, int jm) {
    const int j = 16 * JR + jm;
    const f32x2 ninv2 = pack2(in.ninv, in.ninv);
    const float lj = tj > jm ? in.l[JR] : 0.f;
    const f32x2 lj2 = pack2(lj, lj);
    in.w[JR] = fmul2(in.w[JR], ninv2);
    R[tri(JR, JR)] = ffma2(in.w[JR], lj2, R[tri(JR, JR)]);
    const int jn = jm + 1;
    const float ninv_n = -rcp_fast((jn & 8) ? hi2(R[tri(JR, JR)]) : lo2(R[tri(JR, JR)]));
#pragma unroll
    for (int q = JR + 1; q < 8; ++q) {
      in.w[q] = fmul2(in.w[q], ninv2);
      R[tri(q, JR)] = ffma2(in.w[q], lj2, R[tri(q, JR)]);
    }
    if (rhs_warp) {
      const bool act_lo = below || (on && ti > jm), act_hi = below || (on && ti + 8 > jm);
      const f32x2 mb = fmul2(in.wb, ninv2);
      bb2 = ffma2(pack2(act_lo ? lo2(mb) : 0.f, act_hi ? hi2(mb) : 0.f), pack2(in.zj, in.zj), bb2);
      sts32_if(on && ti == (jn & 7) && jn < 16, Y + (uint32_t)(j + 1) * 4u, (jn & 8) ? hi2(bb2) : lo2(bb2));
    }
    {
      const bool own = (tj == jn);
      publish(P + ((uint32_t)(jn & 1) << 9), own);
      sts32_if(own && ti == (jn & 7), DI + (uint32_t)(j + 1) * 4u, ninv_n);
      group_sync(bar);
    }
    load(nx, jn);                     // (after the block's last pivot: reads nobody uses)
#pragma unroll
    for (int c = JR + 1; c < 8; ++c) {
      const f32x2 l2 = pack2(in.l[c], in.l[c]);
#pragma unroll
      for (int q = c; q < 8; ++q) R[tri(q, c)] = ffma2(in.w[q], l2, R[tri(q, c)]);
    }
  };
  publish(P, tj == 0);
  sts32_if(ti == 0 && tj == JR, Y + (uint32_t)(16 * JR) * 4u, lo2(bb2));
  sts32_if(gl == 0, DI + (uint32_t)(16 * JR) * 4u, -rcp_fast(lo2(R[tri(JR, JR)])));
  group_sync(bar);
  PivotIn<JR> a, b;
  a.zj = b.zj = 0.f;
  a.wb = b.wb = 0ull;
  load(a, 0);
#pragma unroll 1
  for (int jm = 0; jm < 16; jm += 2) {
    step(a, b, jm);
    step(b, a, jm + 1);
  }
}

// Back substitution by blocks of 16 unknowns, last block first; the 16 x 16 triangle of the block goes through T and is
// solved by the first quarter of ONE warp of the group (redundantly per lane; the warp rotates with the block so that
// the four sub-partitions share the work), which files the block's solution in X for the others.
template <int JR>
__device__ __forceinline__ void back_block(const f32x2 (&R)[36], f32x2 (&x2)[8], const uint32_t Y, const uint32_t DI,
                                           const uint32_t T, const uint32_t RH, const uint32_t X, const int ti,
                                           const int tj, const int gl, const int bar) {
  f32x2 acc0 = 0ull, acc1 = 0ull;
#pragma unroll
  for (int q = JR + 1; q < 8; ++q) {
    if ((q - JR) & 1) acc0 = ffma2(R[tri(q, JR)], x2[q], acc0);
    else acc1 = ffma2(R[tri(q, JR)], x2[q], acc1);
  }
  float ext = (lo2(acc0) + hi2(acc0)) + (lo2(acc1) + hi2(acc1));
  ext += __shfl_xor_sync(0xffffffffu, ext, 1);          // over ti: the eight lanes of a column are neighbours
  ext += __shfl_xor_sync(0xffffffffu, ext, 2);
  ext += __shfl_xor_sync(0xffffffffu, ext, 4);
  const float rh = lds32(Y + (uint32_t)(16 * JR + tj) * 4u) - ext;
  sts32(T + (uint32_t)(ti * 16 + tj) * 4u, lo2(R[tri(JR, JR)]));
  sts32(T + (uint32_t)((ti + 8) * 16 + tj) * 4u, hi2(R[tri(JR, JR)]));
  sts32_if(ti == 0, RH + (uint32_t)tj * 4u, rh);
  group_sync(bar);
  if (((gl >> 5) & 3) == (JR & 3) && (gl & 31) < 8) {   // one quarter warp: its 16-byte loads are single passes
    float r[16];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const float4 a = lds128(RH + 16 * v);
      r[4 * v] = a.x; r[4 * v + 1] = a.y; r[4 * v + 2] = a.z; r[4 * v + 3] = a.w;
    }
#pragma unroll
    for (int e = 15; e >= 0; --e) {
      r[e] = -r[e] * lds32(DI + (uint32_t)(16 * JR + e) * 4u);     // x_e (DI holds -1/d); r[e] now IS x_e
#pragma unroll
      for (int v = 0; v < (e + 3) / 4; ++v) {
        const float4 t = lds128(T + (uint32_t)(e * 16 + 4 * v) * 4u);
        if (4 * v < e) r[4 * v] = fmaf(-t.x, r[e], r[4 * v]);
        if (4 * v + 1 < e) r[4 * v + 1] = fmaf(-t.y, r[e], r[4 * v + 1]);
        if (4 * v + 2 < e) r[4 * v + 2] = fmaf(-t.z, r[e], r[4 * v + 2]);
        if (4 * v + 3 < e) r[4 * v + 3] = fmaf(-t.w, r[e], r[4 * v + 3]);
      }
    }
    if ((gl & 31) == 0) {
#pragma unroll
      for (int v = 0; v < 4; ++v) sts128(X + (uint32_t)(16 * JR + 4 * v) * 4u, r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]);
    }
  }
  group_sync(bar);                         // X of the block visible; T / RH are rewritten by the next block
  x2[JR] = pack2(lds32(X + (uint32_t)(16 * JR + ti) * 4u), lds32(X + (uint32_t)(16 * JR + 8 + ti) * 4u));
}

__device__ __noinline__ void solver_role(uint32_t sC, uint32_t scratch, uint32_t tmem, Bars* bars,
                                         float* __restrict__ dst, __nv_bfloat16* __restrict__ dst_hl,
                                         float* __restrict__ workspace, float reg, const int32_t* __restrict__ item_row,
                                         const int32_t* __restrict__ item_len, const int32_t* __restrict__ item_slot,
                                         const float* __restrict__ gram_tiles, const Range* rg, int group, int gl) {
  const int ti = gl & 7, tj = gl >> 3;
  const int bar = 1 + group;
  const uint32_t sB = sC + 128 * kLdc * 4;
  const uint32_t P = scratch, Y = P + 1024, DI = Y + 512, T = DI + 512, RH = T + 1024, X = RH + 64;
  const uint32_t ta = tmem + ((uint32_t)(32 * ((gl >> 5) & 3)) << 16);
  const int64_t n_items = rg->item_hi;
  const int m = gl;                                        // TMEM lane = matrix row while draining
#ifdef HALS_WS_PROFILE
  long long w_acc = 0, w_c = 0, t_drain = 0, t_load = 0, t_elim = 0, t_back = 0;
  int n_solved = 0;
#endif
  uint32_t mine = 0;
  for (int64_t it = rg->item_lo + group; it < n_items; it += kGroups, ++mine) {
    const int row = __ldg(item_row + it), len = __ldg(item_len + it), wslot = __ldg(item_slot + it);
    { WS_T0(); umma::mbar_wait(&bars->acc_full[group], mine & 1); WS_ACC(w_acc); }
    umma::fence_after_sync();
    // the hand-over matrix: free once the group before us has loaded its tile (first row of the CTA: free)
    if (!(group == 0 && mine == 0)) { WS_T0(); umma::mbar_wait(&bars->c_turn[group], (group == 0 ? mine - 1 : mine) & 1); WS_ACC(w_c); }
    {
      WS_T0();
      float v[32], u[32];
#pragma unroll 1
      for (int c0 = 0; c0 < 128; c0 += 32) {
        umma::tmem_ld32(ta + c0, v);
        umma::tmem_ld32(ta + 128 + c0, u);
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          sts128(sC + (uint32_t)(m * kLdc + c0 + i) * 4u, fmaf(0.5f, v[i], u[i]), fmaf(0.5f, v[i + 1], u[i + 1]),
                 fmaf(0.5f, v[i + 2], u[i + 2]), fmaf(0.5f, v[i + 3], u[i + 3]));
      }
      float e1[16], e2[16];
      umma::tmem_ld16(ta + 256, e1);
      umma::tmem_ld16(ta + 272, e2);
      sts32(sB + (uint32_t)m * 4u, e1[0] + e1[1] + e2[0]);
      umma::fence_before_sync();
      umma::mbar_arrive(&bars->acc_free);
      group_sync(bar);                                     // C complete
      WS_ACC(t_drain);
    }
    if (wslot >= 0) {
      // slice of a long row: park (A, b, n) in its workspace slot (layout of the SIMT path / reduce kernel)
      float* W = workspace + (size_t)wslot * kSlotFloats;
#pragma unroll 4
      for (int n = 0; n < 128; n += 4) {
        const float4 q = lds128(sC + (uint32_t)(m * kLdc + n) * 4u);
        *reinterpret_cast<float4*>(W + m * K + n) =
            make_float4(q.x + lds32(sC + (uint32_t)((n) * kLdc + m) * 4u), q.y + lds32(sC + (uint32_t)((n + 1) * kLdc + m) * 4u),
                        q.z + lds32(sC + (uint32_t)((n + 2) * kLdc + m) * 4u), q.w + lds32(sC + (uint32_t)((n + 3) * kLdc + m) * 4u));
      }
      W[K * K + m] = lds32(sB + (uint32_t)m * 4u);
      if (m == 0) W[K * K + K] = (float)len;
      group_sync(bar);
      if (gl == 0) umma::mbar_arrive(&bars->c_turn[(group + 1) % kGroups]);
      continue;
    }
    f32x2 R[36];
    f32x2 bb2;
    {
      WS_T0();
      const float lam = reg * (float)len;
      const uint32_t pd = sC + (uint32_t)(ti * kLdc + tj) * 4u, pt = sC + (uint32_t)(tj * kLdc + ti) * 4u;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int c = 0; c <= q; ++c) {
          float a[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t mn = (uint32_t)((16 * q + 8 * h) * kLdc + 16 * c) * 4u, nm = (uint32_t)(16 * c * kLdc + 16 * q + 8 * h) * 4u;
            a[h] = lds32(pd + mn) + lds32(pt + nm);
            if (q == c) a[h] += (ti + 8 * h == tj) ? lam : 0.f;
          }
          R[tri(q, c)] = pack2(a[0], a[1]);
        }
      }
      if (gram_tiles != nullptr) {                           // implicit: + Y^T Y, already in this lane's tile order
        const float4* gp = reinterpret_cast<const float4*>(gram_tiles) + gl * 18;
#pragma unroll
        for (int i = 0; i < 18; ++i) {
          const float4 g = __ldg(gp + i);
          R[2 * i] = ffma2(pack2(g.x, g.y), pack2(1.f, 1.f), R[2 * i]);
          R[2 * i + 1] = ffma2(pack2(g.z, g.w), pack2(1.f, 1.f), R[2 * i + 1]);
        }
      }
      const uint32_t ob = (uint32_t)(ti + 16 * (tj & 7)) * 4u;
      bb2 = tj < 8 ? pack2(lds32(sB + ob), lds32(sB + ob + 32)) : 0ull;
      group_sync(bar);
      if (gl == 0) umma::mbar_arrive(&bars->c_turn[(group + 1) % kGroups]);
      WS_ACC(t_load);
    }
    {
      WS_T0();
      elim_block<0>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<1>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<2>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<3>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<4>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<5>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<6>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      elim_block<7>(R, bb2, P, Y, DI, ti, tj, gl, bar);
      WS_ACC(t_elim);
    }
    {
      WS_T0();
      f32x2 x2[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) x2[q] = 0ull;
      back_block<7>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<6>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<5>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<4>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<3>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<2>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<1>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      back_block<0>(R, x2, Y, DI, T, RH, X, ti, tj, gl, bar);
      const float x = lds32(X + (uint32_t)gl * 4u);
      dst[(int64_t)row * K + gl] = x;
      if (dst_hl) {
        const __nv_bfloat16 h = __float2bfloat16_rn(x);
        dst_hl[(int64_t)row * (2 * K) + gl] = h;
        dst_hl[(int64_t)row * (2 * K) + K + gl] = __float2bfloat16_rn(x - __bfloat162float(h));
      }
      group_sync(bar);                                     // X is rewritten by the next row
      WS_ACC(t_back);
    }
#ifdef HALS_WS_PROFILE
    ++n_solved;
#endif
  }
#ifdef HALS_WS_PROFILE
  if (gl == 0 && blockIdx.x == 1)
    printf("S%d: solved %d wait_acc %lld wait_c %lld drain %lld load %lld elim %lld back %lld\n", group, n_solved, w_acc, w_c,
           t_drain, t_load, t_elim, t_back);
#endif
}

__global__ void __launch_bounds__(kThreads, 1)
als_ws128_kernel(const int32_t* __restrict__ colidx, const uint32_t* __restrict__ vals_hl,
                 const float* __restrict__ vals_sc, const float* __restrict__ gram_tiles,
                 const __nv_bfloat16* __restrict__ src_hl, float* __restrict__ dst, float reg,
                 const int32_t* __restrict__ item_row, const int32_t* __restrict__ item_len,
                 const int32_t* __restrict__ item_slot, const int64_t* __restrict__ item_chunk0,
                 const int64_t* __restrict__ item_cost0, const int64_t* __restrict__ chunk_pos,
                 const int32_t* __restrict__ chunk_cnt, int64_t n_items, int zero_row, float* __restrict__ workspace,
                 __nv_bfloat16* __restrict__ dst_hl) {
  extern __shared__ uint8_t smem_dyn[];
  __shared__ Bars bars;
  __shared__ Range range;
  __shared__ uint32_t tmem_slot;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) umma::tmem_alloc(&tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < kStages; ++s) {
      umma::mbar_init(&bars.st_full[s], 32);
      umma::mbar_init(&bars.st_free[s], 1);
      umma::mbar_init(&bars.st_scaled[s], 1);
    }
    for (int g = 0; g < kGroups; ++g) { umma::mbar_init(&bars.acc_full[g], 1); umma::mbar_init(&bars.c_turn[g], 1); }
    umma::mbar_init(&bars.acc_free, 128);
    umma::mbar_fence_init();
  }
  if (tid < 2) cta_range(&range, item_cost0, item_chunk0, n_items, tid);
  zero_r_blocks<K, kStages, kThreads>(base, tid);
  umma::fence_proxy_async();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint32_t sbase = umma::smem_u32(base);
  const uint32_t sC = sbase + kStages * kStageBytes;
  const uint32_t scratch = sC + kCBytes;
  uint8_t* gscratch = base + kStages * kStageBytes + kCBytes + kGroups * kGroupScratch;

  if (warp < 4 * kGroups) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(kRegsSolver));
    solver_role(sC, scratch + (uint32_t)(warp >> 2) * kGroupScratch, tmem, &bars, dst, dst_hl, workspace, reg, item_row,
                item_len, item_slot, gram_tiles, &range, warp >> 2, tid & 127);
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(kRegsFront));
    if (warp < kWarpMma)
    gather_role(sbase, &bars, gscratch + (warp - kWarpGather) * kGatherScratch, &range, colidx, vals_hl, vals_sc,
                reinterpret_cast<const uint8_t*>(src_hl), zero_row, chunk_pos, chunk_cnt, warp - kWarpGather, lane);
    else if (warp == kWarpMma) mma_role(sbase, tmem, &bars, &range, chunk_cnt, vals_sc != nullptr, lane);
    else if (vals_sc != nullptr) scaler_role(sbase, &bars, &range, lane);
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, 512);
}

}  // namespace ws128

// Y^T Y ([128][128], symmetric) -> the solver's lane-tile order: tiles[gl][tri(q, c)] = (G[ti + 16q][tj + 16c],
// G[ti + 8 + 16q][tj + 16c]) with gl = ti + 8 tj -- a lane adds its share with 18 contiguous 16-byte loads.
__global__ void gram_to_tiles128_kernel(const float* __restrict__ G, float* __restrict__ tiles) {
  const int gl = threadIdx.x, ti = gl & 7, tj = gl >> 3;
  for (int q = 0; q < 8; ++q)
    for (int c = 0; c <= q; ++c)
      for (int h = 0; h < 2; ++h)
        tiles[gl * 72 + ws128::tri(q, c) * 2 + h] = G[(ti + 8 * h + 16 * q) * ws128::K + tj + 16 * c];
}

// src != nullptr: fp32 source factors, split into `split_buf` first.  src == nullptr: `split_buf` already holds the
// split source ([n_src + 1][256] bf16, row n_src all zero); see als_half_step_ws64.
// gram != nullptr selects implicit feedback: the plan must carry vals_scale / item_npos (packed for the caller's alpha),
// `gram_tiles` is 36,864 bytes of scratch.
int als_half_step_ws128(const int32_t* colidx, const uint32_t* vals_hl, const float* src, int64_t n_src, float* dst,
                        float reg, const hals_als_plan* plan, float* slots, void* split_buf, void* dst_hl,
                        const float* gram, float* gram_tiles, cudaStream_t st) {
  using namespace ws128;
  __nv_bfloat16* hl = reinterpret_cast<__nv_bfloat16*>(split_buf);
  HALS_REQUIRE(n_src < (int64_t)1 << 31, "at most 2^31 - 1 source rows");
  if (src != nullptr) {
    if (int rc = als_launch_split_bf16(src, n_src, K, hl, st)) return rc;
    HALS_CUDA(cudaMemsetAsync(hl + (size_t)n_src * 2 * K, 0, 4 * K, st));
  }
  const bool implicit = gram != nullptr;
  if (implicit) {
    HALS_REQUIRE(plan->vals_scale && plan->item_npos && gram_tiles, "implicit mode needs the plan's vals_scale / item_npos");
    gram_to_tiles128_kernel<<<1, 128, 0, st>>>(gram, gram_tiles);
    HALS_LAUNCH_CHECK();
  }
  const size_t smem = (size_t)kStages * kStageBytes + kCBytes + (size_t)kGroups * kGroupScratch + 2 * kGatherScratch + 1024;
  static_assert(kStages * kStageBytes + kCBytes + kGroups * kGroupScratch + 2 * kGatherScratch + 1024 <= 227 * 1024 - 1024,
                "shared memory budget");
  HALS_CUDA(cudaFuncSetAttribute(als_ws128_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  static const int regs = [] { cudaFuncAttributes a{}; return cudaFuncGetAttributes(&a, als_ws128_kernel) == cudaSuccess ? a.numRegs : -1; }();
  if (regs != kRegsLaunch)   // the setmaxnreg arithmetic assumes exactly this allocation (a short pool would hang)
    return fail(HALS_ERR_CUDA, "%s: als_ws128_kernel was compiled for an unexpected register count%s", __func__);
  int64_t grid = sm_count();
  if (grid > plan->n_items) grid = plan->n_items;
  als_ws128_kernel<<<(unsigned)grid, kThreads, smem, st>>>(colidx, vals_hl, implicit ? plan->vals_scale : nullptr,
                                                          implicit ? gram_tiles : nullptr, hl, dst, reg, plan->item_row,
                                                          implicit ? plan->item_npos : plan->item_len, plan->item_slot, plan->item_chunk0, plan->item_cost0,
                                                          plan->chunk_pos, plan->chunk_cnt, plan->n_items, (int)n_src, slots,
                                                          reinterpret_cast<__nv_bfloat16*>(dst_hl));
  HALS_LAUNCH_CHECK();
  if (plan->n_long_rows > 0) {
    if (int rc = als_launch_slot_group_sum(slots, plan, (int)kSlotFloats, st)) return rc;
    if (int rc = als_launch_reduce_solve128(slots, dst, reg, plan, dst_hl, gram, st)) return rc;
  }
  return 0;
}

}  // namespace hals
