// ALS half-step, rank 64, warp-specialised persistent kernel (the default rank-64 path).
// Replaces Spark's NormalEquation.add (dspr/daxpy per rating) and CholeskySolver.solve (dppsv) reached from
// src/als_model.py:62; arithmetic identical to als_tc.cu (bf16 hi/lo split operands, fp32 accumulation in TMEM,
// A = D_hh + D_lh + D_lh^T, square-root-free Cholesky), but the row pipeline is decoupled:
//
//   one CTA per SM with a contiguous, equal-cost share of the plan's work items (Range); 16 warps, four roles linked
//   by mbarriers (no CTA-wide barrier anywhere on the path)
//     G  warps 9-10 gather: cp.async 16-byte pieces of the h|l rows straight into the swizzled MN-major stage
//                   (layout pinned by tests/test_gpu_umma.py), a flat stream of 32-rating chunks across row
//                   boundaries, completion through the stage mbarrier (cp.async.mbarrier.arrive), column indices prefetched two bursts of 8 chunks ahead
//                   (the implicit-mode scaler_role is shared with als_ws128.cu: als_ws_common.cuh)
//     M  warp 11    one thread issues tcgen05.mma (M=128, N=80, K=16) per 16 ratings into one of four TMEM
//                   accumulators; tcgen05.commit recycles the stage and publishes the finished accumulator
//     D  warps 12-15 drain: TMEM lane = matrix row; rows of h h^T (warps 0,1) and l h^T (warps 2,3) go to one of
//                   three shared-memory hand-over slots, the accumulator is released at once
//     S  warps 0-8  nine independent solvers, ONE WARP PER 64x64 SYSTEM: lower triangle in registers
//                   (2-D cyclic over a 4 x 8 lane grid, 36 packed fp32x2), pivot columns published through a
//                   256-byte per-warp buffer, __syncwarp only.  The 64-step chain of one system is hidden
//                   behind the eight other systems in flight on the SM.
//
// Why: the round-1 kernel (als_tc.cu, four 4-warp CTAs per SM) had 4 rows in flight per SM and a CTA barrier
// on each of the 64 pivot steps (~280 cycles per step; ncu: issue slots 44 %, top stall `barrier`).
#include <cuda_bf16.h>

#include <cstdlib>

#include "als_ws_common.cuh"

namespace hals {
namespace ws64 {
using namespace ws;

constexpr int K = 64;
constexpr int kStageBytes = stage_bytes(K);  // H | L | R
#ifndef HALS_WS_STAGES
#define HALS_WS_STAGES 10
#endif
constexpr int kStages = HALS_WS_STAGES;
constexpr int kAcc = 4, kAccCols = 128;      // TMEM accumulators (N = 80 columns used of each 128)
constexpr int kSlots = 2;
constexpr int kLd = 68;                      // hand-over row stride in floats: conflict-free 16-byte row stores
constexpr int kSlotBytes = 2 * 64 * kLd * 4 + 512;   // S1 (h h^T rows) | S2 (l h^T rows) | b1 | b2
constexpr int kSolvers = 9;
constexpr int kScratchBytes = 1536;          // per solver: P (2 x 256) | Y (256) | DI (256) | T (256) | RH (32)
constexpr int kN = 80;
constexpr int kThreads = 512;
// Role map.  The warp scheduler prefers the highest warp id among the ready warps of a sub-partition, so the light,
// latency-critical front end (gather, MMA issue, drain) sits ABOVE the solvers: with the solvers on top the gather
// warps got an issue slot every ~5 cycles and needed 400-700 cycles per chunk (measured), starving the whole pipe.
constexpr int kWarpSolver = 0, kWarpGather = 9, kWarpMma = 11, kWarpDrain = 12;
static_assert(kStages % 2 == 0, "the two gather warps own alternate stages");
static_assert(kWarpSolver + kSolvers == kWarpGather && kWarpDrain + 4 == kThreads / 32 && kWarpDrain % 4 == 0, "role map");
static_assert(kStageBytes % 512 == 0 && kSlotBytes % 512 == 0 && kScratchBytes % 512 == 0,
              "a solver's scratch is 512-byte aligned: its elimination steps flip the column buffer by bit 8");

struct Bars {
  uint64_t st_full[kStages], st_free[kStages];
  uint64_t st_scaled[kStages];   // implicit mode: stage rescaled by sqrt(c) (what the MMA warp then waits for)
  uint64_t acc_full[kAcc], acc_free[kAcc];
  uint64_t sol_full[kSolvers];   // per SOLVER, not per slot: a waiter may lag its barrier by one phase at most, and a
                                 // solver's consecutive rows are kSolvers / kSlots uses of a slot apart
  uint64_t slot_free[kSlots];
};

__device__ __forceinline__ float sel4(float a, float b, float c, float d, int i) {
  return i == 0 ? a : i == 1 ? b : i == 2 ? c : d;
}

// ---- G: gather ---------------------------------------------------------------------------------------
// The two gather warps take ALTERNATE chunks of the CTA's chunk table (chunk = up to 32 ratings of one item; warp w:
// chunks lo + w, lo + w + 2, ... -> stages w, w + 2, ...), independently of row boundaries and of the other roles,
// each with its own lookahead (no cross-warp synchronisation, no duplicated work):
//   * chunk table: lane i holds (pos, cnt) of the warp's i-th chunk of the window; the next window of 32 is loaded a
//     window ahead
//   * column indices: loaded in bursts of kBurst chunks, one burst ahead (registers), then parked in a per-warp
//     shared-memory ring the chunk loop reads -- the loop body exists once (a first version rotated a register queue
//     by name through an 8x unrolled body: 32 KB of code, 60 % of the gather warps' stall samples were instruction fetch)
//   * a chunk is 16 cp.async of 16 bytes per lane (lane = 16-byte piece of the 256-byte h|l row, two ratings per
//     instruction: 4 cache lines, fully coalesced) + 4 bytes of packed rating per lane.  Ratings past the end of an
//     item read the all-zero row n_src the split buffer carries, so no copy needs a predicate or a clamp.
// Completion goes through the stage's mbarrier (cp.async.mbarrier.arrive.noinc: the arrival fires when this thread's
// copies have landed), so the warp never waits for data.  No fence.proxy.async anywhere on the path (measured ~380
// cycles each, once per chunk, serial in whichever warp executes it): every byte of a stage is written by cp.async,
// whose completion through the mbarrier is what the MMA thread waits for -- the pattern of the cp.async
// warp-specialised mainloops in CUTLASS.
__device__ __noinline__ void gather_role(uint32_t stages, Bars* bars, uint8_t* gscratch, const Range* rg,
                                         const int32_t* __restrict__ colidx, const uint32_t* __restrict__ vals_hl,
                                         const float* __restrict__ vals_sc, const uint8_t* __restrict__ src_hl, int zero_row,
                                         const int64_t* __restrict__ chunk_pos, const int32_t* __restrict__ chunk_cnt,
                                         int gw, int lane) {
  const int t_sub = lane >> 4, piece = lane & 15;
  const uint32_t ring = umma::smem_u32(gscratch);                       // int  [2][kBurst][32]
  const uint32_t mpos = ring + 2 * kBurst * 128;                        // i64  [2][kBurst] first rating of the chunk
  const uint32_t mcnt = mpos + 2 * kBurst * 8;                          // int  [2][kBurst] ratings left in its item
  const int64_t k_hi = rg->chunk_hi;
  int64_t kw = rg->chunk_lo + gw;                                       // first chunk of the NEXT window to load
  auto load_window = [&](int64_t& p, int& c) {
    const int64_t k = kw + 2 * lane;
    p = 0; c = 0;                                                       // cnt 0 = past the end of the stream
    if (k < k_hi) { p = __ldg(chunk_pos + k); c = __ldg(chunk_cnt + k); }
    kw += 64;
  };
  int64_t wpos, npos;
  int wcnt, ncnt;
  load_window(wpos, wcnt);
  load_window(npos, ncnt);
  int wb = 0;                                                           // burst inside the window (4 per window)
  int ci[kBurst];
  auto fill = [&](int buf) {      // index loads of the next burst (stay in flight); its chunk table goes to buffer `buf`
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
    for (int c = 0; c < kBurst; ++c)   // rating `lane` -> slot (lane % 2) * 16 + lane / 2: a lane's 16 ratings are contiguous
      sts32(ring + (uint32_t)((buf * kBurst + c) * 32 + (lane & 1) * 16 + (lane >> 1)) * 4u, __int_as_float(ci[c]));
    __syncwarp();
  };

  // destination of copy i (rating t = t_sub + 2i): H or L block, row t, 16-byte chunk (piece % 8) ^ (t % 8);
  // t % 8 = t_sub + 2 (i % 4), so the four swizzled offsets repeat every four copies
  const uint32_t blk_off = piece < 8 ? 0u : (uint32_t)kBlk;
  uint32_t dsto[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int t = t_sub + 2 * i;
    dsto[i] = blk_off + (uint32_t)t * kRowBytes + (uint32_t)(((piece & 7) ^ (t & 7)) << 4);
  }
  const uint64_t srcb = reinterpret_cast<uint64_t>(src_hl) + (uint64_t)piece * 16u;
  const uint32_t rdst = 2 * kBlk + (uint32_t)lane * kRowBytes + (uint32_t)((lane & 7) << 4);
  const uint32_t sdst = 2 * kBlk + (uint32_t)lane * kRowBytes + (uint32_t)((7 ^ (lane & 7)) << 4);   // a chunk no MMA reads
  uint32_t g = 0, s = (uint32_t)gw, u = 0;   // chunks issued, stage, ring wraps
#ifdef HALS_WS_PROFILE
  long long w_free = 0, t_iss = 0, t_fill = 0;
#endif
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
      // this lane's 16 ratings (t = t_sub + 2i) sit next to each other in the ring: four 16-byte loads, issued before
      // anything depends on them (the asm statements keep their order: one load per copy would serialise the round trips)
      const uint32_t ir = ring + (uint32_t)((buf * kBurst + c) * 32 + t_sub * 16) * 4u;
      const float4 c0 = lds128(ir), c1 = lds128(ir + 16), c2 = lds128(ir + 32), c3 = lds128(ir + 48);
      if (u > 0) { WS_T0(); umma::mbar_wait(&bars->st_free[s], (u - 1) & 1); WS_ACC(w_free); }
      WS_T0();
      const uint32_t st = stages + s * kStageBytes;
      const float colf[16] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w, c3.x, c3.y, c3.z, c3.w};
#pragma unroll
      for (int i = 0; i < KC / 2; ++i) {
        uint64_t src;
        asm("mad.wide.u32 %0, %1, 256, %2;\n" : "=l"(src) : "r"((uint32_t)__float_as_int(colf[i])), "l"(srcb));
        cp_async16_raw(st + dsto[i & 3] + (uint32_t)(i >> 2) * (8 * kRowBytes), src);
      }
      // rating columns of the B operand (element 0 = bf16(r), element 1 = bf16(r - bf16(r))): 4 bytes per rating from
      // the packed array; the other 28 bytes of the two 16-byte chunks were zeroed once at kernel start
      {
        const bool ok = lane < cnt;
        const uint32_t* rp = vals_hl + pos + (ok ? lane : 0);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(st + rdst), "l"(rp), "r"(ok ? 4 : 0) : "memory");
        if (vals_sc != nullptr) {          // implicit mode: sqrt(alpha |r|) of rating `lane`, read by the scaler warp
          const float* sp = vals_sc + pos + (ok ? lane : 0);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(st + sdst), "l"(sp), "r"(ok ? 4 : 0) : "memory");
        }
      }
      cp_async_mbar_arrive_noinc(&bars->st_full[s]);
      WS_ACC(t_iss);
      ++g;
      s += 2;
      if (s >= (uint32_t)kStages) { s -= kStages; ++u; }
    }
    if (done) break;
    WS_T0();
    stash(buf ^ 1);                      // the burst loaded while this one was being issued
    fill(buf);                           // two bursts ahead: in flight during the next burst
    WS_ACC(t_fill);
  }
#ifdef HALS_WS_PROFILE
  if (lane == 0 && blockIdx.x == 1) printf("G%d: chunks %u wait_free %lld issue %lld fill %lld\n", gw, g, w_free, t_iss, t_fill);
#endif
}

__device__ __noinline__ void scaler_role(uint32_t stages, Bars* bars, const Range* rg, int lane) {
  scale_stages<K, kStages>(stages, bars, rg, lane);
}

// ---- M: MMA issue (whole warp walks the chunk table, lane 0 issues) --------------------------------------
__device__ __noinline__ void mma_role(uint32_t sbase, uint32_t tmem, Bars* bars, const Range* rg,
                                      const int32_t* __restrict__ chunk_cnt, bool scaled, int lane) {
  constexpr uint32_t idesc = umma::make_instr_desc(umma::kFmtBF16, true, true, 128, kN);
  uint64_t* const ready = scaled ? bars->st_scaled : bars->st_full;
  const int64_t k_lo = rg->chunk_lo, k_hi = rg->chunk_hi;
  uint32_t s = 0, su = 0, b = 0, bu = 0;
  bool first = true;                       // the next chunk starts a new item (= a new accumulator)
#ifdef HALS_WS_PROFILE
  long long w_acc = 0, w_full = 0, t_issue = 0;
#endif
  int wc = 0, nc = 0;                      // lane i: cnt of chunk (window base + i); next window prefetched
  if (k_lo + lane < k_hi) wc = __ldg(chunk_cnt + k_lo + lane);
  if (k_lo + 32 + lane < k_hi) nc = __ldg(chunk_cnt + k_lo + 32 + lane);
  // elect.sync names ONE issuing lane in a way the compiler can see (an `if (lane == 0)` makes it wrap every
  // tcgen05 instruction in a loop over the active lanes: ~450 cycles of fixed stalls per chunk, measured)
  const bool leader = elect_one();
  const uint64_t ad0 = umma::make_smem_desc(sbase, kBlk, 1024, umma::kSwizzle128B);        // stage 0, K step 0
  const uint64_t bd0 = umma::make_smem_desc(sbase, 2 * kBlk, 1024, umma::kSwizzle128B);
  for (int64_t kb = k_lo; kb < k_hi; kb += 32) {
    const int nk = (int)(k_hi - kb < 32 ? k_hi - kb : 32);
    for (int i = 0; i < nk; ++i) {
      const int cnt = __shfl_sync(0xffffffffu, wc, i);
      if (leader) {
        if (first) {
          if (bu > 0) { WS_T0(); umma::mbar_wait(&bars->acc_free[b], (bu - 1) & 1); WS_ACC(w_acc); }
          umma::fence_after_sync();
        }
        { WS_T0(); umma::mbar_wait(&ready[s], su & 1); WS_ACC(w_full); }
        WS_T0();
        const uint32_t td = tmem + b * kAccCols;
        const uint64_t so = (uint64_t)((s * kStageBytes) >> 4);       // the descriptors' start-address field counts 16 bytes
#pragma unroll
        for (int ks = 0; ks < KC / 16; ++ks)
          umma::mma_bf16(td, ad0 + so + (uint64_t)(ks * 2048 >> 4), bd0 + so + (uint64_t)(ks * 2048 >> 4), idesc,
                         !(first && ks == 0));
        umma::commit(&bars->st_free[s]);
        if (cnt <= KC) umma::commit(&bars->acc_full[b]);
        WS_ACC(t_issue);
      }
      __syncwarp();
      first = cnt <= KC;
      if (first) { if (++b == (uint32_t)kAcc) { b = 0; ++bu; } }
      if (++s == (uint32_t)kStages) { s = 0; ++su; }
    }
    wc = nc;
    nc = 0;
    if (kb + 64 + lane < k_hi) nc = __ldg(chunk_cnt + kb + 64 + lane);
  }
#ifdef HALS_WS_PROFILE
  if (blockIdx.x == 1 && leader) printf("M: wait_acc_free %lld wait_stage_full %lld issue %lld\n", w_acc, w_full, t_issue);
#endif
}

// ---- D: drain TMEM -> hand-over slot -----------------------------------------------------------------
__device__ __noinline__ void drain_role(uint32_t slots, uint32_t tmem, Bars* bars, const Range* rg, int nsolv, int tid) {
  const int warp = tid >> 5;
  const int64_t n_rows = rg->item_hi - rg->item_lo;
  uint32_t b = 0, bu = 0, sl = 0, slu = 0, sv = 0;
#ifdef HALS_WS_PROFILE
  long long w_acc = 0, w_slot = 0, t_ld = 0;
#endif
  for (int64_t it = 0; it < n_rows; ++it) {
    { WS_T0(); umma::mbar_wait(&bars->acc_full[b], bu & 1); WS_ACC(w_acc); }
    umma::fence_after_sync();
    const uint32_t ta = tmem + b * kAccCols + ((uint32_t)(warp * 32) << 16);
    float a[64], e[16];
    {
      WS_T0();
      umma::tmem_ld32(ta, a);
      umma::tmem_ld32(ta + 32, a + 32);
      umma::tmem_ld16(ta + 64, e);
      WS_ACC(t_ld);
    }
    umma::fence_before_sync();
    umma::mbar_arrive(&bars->acc_free[b]);
    if (slu > 0) { WS_T0(); umma::mbar_wait(&bars->slot_free[sl], (slu - 1) & 1); WS_ACC(w_slot); }
    const uint32_t sb = slots + sl * kSlotBytes;
    const int m = tid & 63;
    const uint32_t rowp = sb + (tid < 64 ? 0u : (uint32_t)(64 * kLd * 4)) + (uint32_t)m * (kLd * 4);
#pragma unroll
    for (int n = 0; n < 64; n += 4) sts128(rowp + n * 4, a[n], a[n + 1], a[n + 2], a[n + 3]);
    const uint32_t bp = sb + 2 * 64 * kLd * 4;
    if (tid < 64) sts32(bp + m * 4, e[0] + e[1]);
    else sts32(bp + 256 + m * 4, e[0]);
    umma::mbar_arrive(&bars->sol_full[sv]);
    if (++b == (uint32_t)kAcc) { b = 0; ++bu; }
    if (++sl == (uint32_t)kSlots) { sl = 0; ++slu; }
    if (++sv == (uint32_t)nsolv) sv = 0;
  }
#ifdef HALS_WS_PROFILE
  if (tid == 0 && blockIdx.x == 1) printf("D: wait_acc_full %lld tmem_ld %lld wait_slot_free %lld\n", w_acc, t_ld, w_slot);
#endif
}

// ---- S: one warp solves one 64 x 64 system -----------------------------------------------------------
// lane = 8*ti + tj (ti 0..3, tj 0..7) owns rows {ti + 8q, ti + 4 + 8q} and columns {tj + 8c}:
//   R[tri(q,c)] = (A[ti + 8q][tj + 8c], A[ti + 4 + 8q][tj + 8c])   for 0 <= c <= q <= 7   (lower triangle by 8x8
//   blocks; the diagonal blocks carry both triangles).
// Elimination step j = 8*JR + jm (A = L D L^T, right-looking): the four lanes with tj == jm hold column j; they
// publish it as P[ti][q] (the same packing as R, so readers get their row multipliers as packed pairs); every
// lane then needs 8-JR packed row values, 8-JR column values and the pivot:  A[m][n] -= (A[m][j]/d) * A[n][j].
// Finished columns stay in the registers as columns of L*D and feed the back substitution.
// Right-hand side: b[ti + 8tj], b[ti + 4 + 8tj] live in lane (ti, tj) as one packed pair; z = L^-1 b is
// published element by element (Y[j]) as the pivots pass.  A row's pair half is dead once its z is out, so the update
// runs on both halves of every lane (no row mask): only rows below the pivot are published later.
//
// Published column: P[q / 2][ti][q % 2][half] (row ti + 4 half + 8 q).  The first layout, P[ti][q][half], put rows
// ti and ti + 2 on the same banks: every column-value load and every publish was a 2-way conflict, and the solver
// warps keep the SM's one shared-memory pipe 72 % busy (ncu, user half of c2) -- wavefronts are what this loop pays.
// Step jm reads buffer jm % 2 and publishes column j + 1 into the other one: P is 512-byte aligned, so the lane's three
// base addresses flip bit 8 after each step.
struct Lane {
  uint32_t pw, pl, pb;   // P + my rows (+ (q / 2) * 64 + (q % 2) * 8), + row n = tj + 8c of a column, + my rhs rows
  uint32_t dsel;         // low 16 bits: byte selector of my diagonal-block pivot candidate (high half if tj >= 4);
                         // bit kRoleOwn: set if I hold the pivot of the column I own (ti == tj % 4)
  uint32_t roles;        // the role bytes; kRoleZ as in block JR == tj (elim_block clears it in the other blocks)
};
// Role bytes (bit jm = this lane's part in step jm of a block).  Each step shifts the word by one, so every test is
// one AND with a constant bit.
constexpr int kRoleLive = 0;    // tj > jm: my column of the diagonal block is not finished yet
constexpr int kRoleZ = 8;       // ti == (jm + 1) % 4, jm < 7, in block JR == tj: I hold row j + 1 of the rhs
constexpr int kRoleOwn = 16;    // tj == jm + 1: I publish column j + 1 (and 1/d of its pivot if dsel says so)
constexpr int kRoleZhi = 24;    // jm >= 3: row j + 1 is the high half of its pair.  The same in every lane, and it
                                // empties after the block's eight steps: it is also the loop counter.

// Built once per system from %laneid, not from a lane index kept in a register: the compiler would hoist all of it out
// of the solver's row loop and hold it (spilled) across the tile load and the back substitution.
__device__ __forceinline__ Lane lane_setup(uint32_t P) {
  uint32_t lane;
  asm volatile("mov.u32 %0, %%laneid;\n" : "=r"(lane));
  const uint32_t ti = lane >> 3, tj = lane & 7;
  Lane L;
  L.pw = P + ti * 16u;
  L.pl = P + (tj & 3) * 16u + (tj >> 2) * 4u;
  L.pb = L.pw + (tj >> 1) * 64u + (tj & 1) * 8u;
  L.dsel = (tj & 4 ? 0x7654u : 0x3210u) | (ti == (tj & 3) ? 3u << kRoleOwn : 0u);
  const uint32_t z = ti == 0 ? 0x08u : 0x11u << (ti - 1);       // steps jm with (jm + 1) % 4 == ti, jm < 7
  L.roles = (((1u << tj) - 1u) << kRoleLive) | (z << kRoleZ) | (((1u << tj) >> 1) << kRoleOwn) | (0xf8u << kRoleZhi);
  return L;
}

// pred ? a : b for a predicate that is a non-zero word (a role bit): one LOP3 into a predicate and one select
__device__ __forceinline__ float sel_if(uint32_t pred, float a, float b) {
  float r;
  asm("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %1, 0;\n\tselp.f32 %0, %2, %3, p;\n\t}\n" : "=f"(r) : "r"(pred), "f"(a), "f"(b));
  return r;
}

template <int JR>
__device__ __forceinline__ void publish_column(const f32x2 (&R)[36], uint32_t pw, uint32_t own) {
  if (JR & 1) sts64_if(own, pw + (JR >> 1) * 64 + 8, R[tri(JR, JR)]);
#pragma unroll
  for (int q = (JR + 1) & ~1; q < 8; q += 2) sts128x2_if(own, pw + (q >> 1) * 64, R[tri(q, JR)], R[tri(q + 1, JR)]);
}

// Step j = 8 JR + jm; yj = Y + 4 j, DI = Y + 256 holds 1/d.  The multipliers are +A[m][j]/d and the column values
// enter negated (an operand modifier of FFMA2): x * (-y) rounds exactly like -(x * y), so every product and sum is
// the one of A[m][n] += (A[m][j] * (-1/d)) * A[n][j].
template <int JR>
__device__ __forceinline__ void elim_step(f32x2 (&R)[36], f32x2& bb2, const Lane& L, const uint32_t yj, const uint32_t roles) {
  f32x2 w[8];
  float l[8];
  if (JR & 1) w[JR] = lds64x2(L.pw + (JR >> 1) * 64 + 8);
#pragma unroll
  for (int q = (JR + 1) & ~1; q < 8; q += 2) lds128x2(L.pw + (q >> 1) * 64, w[q], w[q + 1]);
  const float dinv = lds32(yj + 256);
#pragma unroll
  for (int c = JR; c < 8; ++c) l[c] = lds32(L.pl + (c >> 1) * 64 + (c & 1) * 8);
  const float zj = lds32(yj);
  const f32x2 wb = lds64x2(L.pb);
  const f32x2 dinv2 = pack2(dinv, dinv);
  const float lj = sel_if(roles & (1u << kRoleLive), l[JR], 0.f);   // columns <= j are finished
  // the diagonal block first: it holds the next pivot, whose reciprocal then overlaps the rest of the column
  // Rows <= j of the diagonal block are finished, but their multipliers are NOT zeroed: a finished row only owns
  // entries of finished columns (l = 0 below: untouched) and of the upper triangle inside the diagonal block, which
  // nothing ever reads (the column publish of a later pivot carries them as row multipliers of finished rows again;
  // the back substitution reads the strict lower triangle only).  Each half of a packed pair is its own row, so a
  // runaway value cannot leak into a live one.
  w[JR] = fmul2(w[JR], dinv2);
  R[tri(JR, JR)] = ffma2(w[JR], pack2(-lj, -lj), R[tri(JR, JR)]);
  // only the owner of column j + 1 with ti == tj % 4 stores this: its pivot is half tj / 4 of the pair
  const float dinv_n = rcp_fast(__uint_as_float(
      __byte_perm(__float_as_uint(lo2(R[tri(JR, JR)])), __float_as_uint(hi2(R[tri(JR, JR)])), L.dsel)));
#pragma unroll
  for (int q = JR + 1; q < 8; ++q) {      // the block's own column, so that column j+1 can go out early
    w[q] = fmul2(w[q], dinv2);
    R[tri(q, JR)] = ffma2(w[q], pack2(-lj, -lj), R[tri(q, JR)]);
  }
  bb2 = ffma2(fmul2(wb, dinv2), pack2(-zj, -zj), bb2);
  {   // publish column j + 1 into the other buffer (jm == 7: nobody owns "column 8" of the block -- no store, no branch)
    const uint32_t own = roles & (1u << kRoleOwn);
    publish_column<JR>(R, L.pw ^ 256u, own);
    sts32_if(roles & (1u << kRoleZ), yj + 4, sel_if(roles & (1u << kRoleZhi), hi2(bb2), lo2(bb2)));
    sts32_if(own & L.dsel, yj + 256 + 4, dinv_n);
    __syncwarp();
  }
#pragma unroll
  for (int c = JR + 1; c < 8; ++c) {
#pragma unroll
    for (int q = c; q < 8; ++q) R[tri(q, c)] = ffma2(w[q], pack2(-l[c], -l[c]), R[tri(q, c)]);
  }
}

// yj: Y + 4 * 8 JR on entry, the next block's on return
template <int JR>
__device__ __forceinline__ void elim_block(f32x2 (&R)[36], f32x2& bb2, Lane& L, uint32_t& yj) {
  // tj == JR <=> kRoleLive bits JR-1 set, JR clear
  const bool zblk = (L.roles & (JR ? 3u << (JR - 1) : 1u)) == (JR ? 1u << (JR - 1) : 0u);
  uint32_t roles = zblk ? L.roles : L.roles & ~(0xffu << kRoleZ);
  {   // column 8*JR goes out first, into buffer 0: its owners are the lanes tj == 0 (no kRoleLive bit), lane 0 holds
      // its pivot and publishes 1/d, lane (0, JR) holds row 8*JR of the rhs (the only kRoleZ bit 3 of the block)
    const bool own0 = (L.roles & (1u << kRoleLive)) == 0;
    publish_column<JR>(R, L.pw, own0);
    sts32_if(roles & (1u << (kRoleZ + 3)), yj, lo2(bb2));
    sts32_if(own0 && (L.dsel & (1u << kRoleOwn)), yj + 256, rcp_fast(lo2(R[tri(JR, JR)])));
    __syncwarp();
  }
#pragma unroll 1
  do {
    elim_step<JR>(R, bb2, L, yj, roles);
    L.pw ^= 256u; L.pl ^= 256u; L.pb ^= 256u;
    yj += 4;
    roles >>= 1;
  } while (roles >= 1u << kRoleZhi);
}

// Back substitution L^T x = D^-1 z by blocks of 8 unknowns, last block first.  The part of the sums that reaches
// below the block is one FFMA2 chain per lane over its column + a 4-lane reduction; the 8 x 8 triangle inside the
// block is shared through T and solved redundantly by every lane (no per-unknown communication).
template <int JR>
__device__ __forceinline__ void back_block(const f32x2 (&R)[36], f32x2 (&x2)[8], const uint32_t Y, const uint32_t DI,
                                           const uint32_t T, const uint32_t RH, const int ti, const int tj,
                                           const int lane, float& out0, float& out1) {
  f32x2 acc0 = 0ull, acc1 = 0ull;
#pragma unroll
  for (int q = JR + 1; q < 8; ++q) {
    if ((q - JR) & 1) acc0 = ffma2(R[tri(q, JR)], x2[q], acc0);
    else acc1 = ffma2(R[tri(q, JR)], x2[q], acc1);
  }
  float ext = (lo2(acc0) + hi2(acc0)) + (lo2(acc1) + hi2(acc1));
  ext += __shfl_xor_sync(0xffffffffu, ext, 8);
  ext += __shfl_xor_sync(0xffffffffu, ext, 16);
  const float rh = lds32(Y + (uint32_t)(8 * JR + tj) * 4u) - ext;
  sts32(T + (uint32_t)(ti * 8 + tj) * 4u, lo2(R[tri(JR, JR)]));
  sts32(T + (uint32_t)((ti + 4) * 8 + tj) * 4u, hi2(R[tri(JR, JR)]));
  sts32_if(ti == 0, RH + (uint32_t)tj * 4u, rh);
  __syncwarp();
  float r[8], di[8], xb[8];
  {
    const float4 a = lds128(RH), b = lds128(RH + 16);
    r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
    const float4 c = lds128(DI + (uint32_t)(8 * JR) * 4u), d = lds128(DI + (uint32_t)(8 * JR) * 4u + 16);
    di[0] = c.x; di[1] = c.y; di[2] = c.z; di[3] = c.w; di[4] = d.x; di[5] = d.y; di[6] = d.z; di[7] = d.w;
  }
#pragma unroll
  for (int e = 7; e >= 0; --e) {
    xb[e] = r[e] * di[e];                  // DI holds 1/d
    if (e > 0) {
      float t[8];
      const float4 a = lds128(T + (uint32_t)(e * 8) * 4u);
      t[0] = a.x; t[1] = a.y; t[2] = a.z; t[3] = a.w;
      if (e > 4) {
        const float4 b = lds128(T + (uint32_t)(e * 8 + 4) * 4u);
        t[4] = b.x; t[5] = b.y; t[6] = b.z; t[7] = b.w;
      }
#pragma unroll
      for (int c = 0; c < e; ++c) r[c] = fmaf(-t[c], xb[e], r[c]);
    }
  }
  __syncwarp();                            // T / RH are rewritten by the next block
  x2[JR] = pack2(sel4(xb[0], xb[1], xb[2], xb[3], ti), sel4(xb[4], xb[5], xb[6], xb[7], ti));
  if ((lane >> 2) == JR) {                 // lane l stores x[2l], x[2l+1]
    const int e2 = lane & 3;
    out0 = sel4(xb[0], xb[2], xb[4], xb[6], e2);
    out1 = sel4(xb[1], xb[3], xb[5], xb[7], e2);
  }
}

// One system, after its tile is loaded: eliminate (z = L^-1 b published in Y, 1/d in DI), then substitute back and
// store the row as fp32 and as the bf16 hi|lo split the NEXT half-step gathers (no separate split pass).
// P | Y | DI | T | RH = the warp's kScratchBytes of shared memory (DI = Y + 256: one address serves both).
__device__ __forceinline__ void eliminate(f32x2 (&R)[36], f32x2& bb2, const uint32_t P, const uint32_t Y) {
  Lane L = lane_setup(P);
  uint32_t yj = Y;
  elim_block<0>(R, bb2, L, yj);
  elim_block<1>(R, bb2, L, yj);
  elim_block<2>(R, bb2, L, yj);
  elim_block<3>(R, bb2, L, yj);
  elim_block<4>(R, bb2, L, yj);
  elim_block<5>(R, bb2, L, yj);
  elim_block<6>(R, bb2, L, yj);
  elim_block<7>(R, bb2, L, yj);
  __syncwarp();                            // DI[63] / Y[63] visible to every lane
}
__device__ __forceinline__ void back_store(const f32x2 (&R)[36], const uint32_t Y, const uint32_t DI, const uint32_t T,
                                           const uint32_t RH, int ti, int tj, int lane, float* __restrict__ dst,
                                           __nv_bfloat16* __restrict__ dst_hl, int row) {
  f32x2 x2[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) x2[q] = 0ull;
  float out0 = 0.f, out1 = 0.f;
  back_block<7>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<6>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<5>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<4>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<3>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<2>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<1>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  back_block<0>(R, x2, Y, DI, T, RH, ti, tj, lane, out0, out1);
  *reinterpret_cast<float2*>(dst + (int64_t)row * K + 2 * lane) = make_float2(out0, out1);
  if (dst_hl) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(out0, out1);
    const __nv_bfloat162 l = __floats2bfloat162_rn(out0 - __low2float(h), out1 - __high2float(h));
    __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(dst_hl + (int64_t)row * (2 * K));
    o[lane] = h;
    o[K / 2 + lane] = l;
  }
}

// The solver's kernel arguments, in shared memory and loaded where they are used: held in registers across the
// elimination, whose peak takes all 128, they were spilled.
struct SolverArgs {
  float* dst;
  __nv_bfloat16* dst_hl;
  float* workspace;
  const float* gram_tiles;
  const int32_t* item_row;
  const int32_t* item_len;
  const int32_t* item_slot;
  float reg;
};
template <class T>
__device__ __forceinline__ T* ld_arg(T* const& v) {          // volatile: not hoisted out of the row loop
  uint64_t r;
  asm volatile("ld.shared.u64 %0, [%1];\n" : "=l"(r) : "r"(umma::smem_u32(&v)));
  return reinterpret_cast<T*>(r);
}
__device__ __forceinline__ float ld_arg(const float& v) { return lds32(umma::smem_u32(&v)); }

__device__ __noinline__ void solver_role(uint32_t slots, uint32_t scratch, Bars* bars, const SolverArgs* args,
                                         const Range* rg, int nsolv, int w, int lane) {
  const int ti = lane >> 3, tj = lane & 7;
  const uint32_t P = scratch, Y = P + 512, DI = Y + 256, T = DI + 256, RH = T + 256;
  // this CTA's items (a share of one plan, far below 2^32)
  const uint32_t n_items = (uint32_t)(rg->item_hi - rg->item_lo);
#ifdef HALS_WS_PROFILE
  long long w_slot = 0, t_load = 0, t_elim = 0, t_back = 0;
  int n_solved = 0;
#endif
  // rows i = w, w + kSolvers, ... of this CTA's item sequence; slot = i % kSlots.  A row's metadata is loaded where it
  // is needed, behind the wait for its slot or the back substitution (prefetched a row ahead, and held across the
  // elimination, it took registers the elimination needs).
  for (uint32_t mine = 0;; ++mine) {     // rows this solver has taken
    const uint32_t i = (uint32_t)w + mine * (uint32_t)nsolv;
    if (i >= n_items) break;
    const int64_t it = rg->item_lo + i;
    const int len = __ldg(ld_arg(args->item_len) + it), wslot = __ldg(ld_arg(args->item_slot) + it);
    const uint32_t sl = i % kSlots;
    { WS_T0(); umma::mbar_wait(&bars->sol_full[w], mine & 1); WS_ACC(w_slot); }
    const uint32_t S1 = slots + sl * kSlotBytes, S2 = S1 + 64 * kLd * 4, B1 = S2 + 64 * kLd * 4, B2 = B1 + 256;
    if (wslot >= 0) {
      // slice of a long row: park (A, b, n) in its workspace slot (layout of the SIMT path / reduce kernel)
      float* W = ld_arg(args->workspace) + (size_t)wslot * ((size_t)K * K + K + 4);
      for (int e = lane; e < K * K; e += 32) {
        const int m = e >> 6, n = e & 63;
        W[e] = lds32(S1 + (uint32_t)(m * kLd + n) * 4u) + lds32(S2 + (uint32_t)(m * kLd + n) * 4u) +
               lds32(S2 + (uint32_t)(n * kLd + m) * 4u);
      }
      W[K * K + lane] = lds32(B1 + lane * 4) + lds32(B2 + lane * 4);
      W[K * K + 32 + lane] = lds32(B1 + (32 + lane) * 4) + lds32(B2 + (32 + lane) * 4);
      if (lane == 0) W[K * K + K] = (float)len;
      __syncwarp();
      if (lane == 0) umma::mbar_arrive(&bars->slot_free[sl]);
      continue;
    }
    f32x2 R[36];
    f32x2 bb2;
    {
      WS_T0();
      const float lam = ld_arg(args->reg) * (float)len;
      const uint32_t p1 = S1 + (uint32_t)(ti * kLd + tj) * 4u, p2 = S2 + (uint32_t)(ti * kLd + tj) * 4u;
      const uint32_t pt = S2 + (uint32_t)(tj * kLd + ti) * 4u;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int c = 0; c <= q; ++c) {
          float v[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t mn = (uint32_t)((8 * q + 4 * h) * kLd + 8 * c) * 4u, nm = (uint32_t)(8 * c * kLd + 8 * q + 4 * h) * 4u;
            v[h] = lds32(p1 + mn) + lds32(p2 + mn) + lds32(pt + nm);
            if (q == c) v[h] += (ti + 4 * h == tj) ? lam : 0.f;
          }
          R[tri(q, c)] = pack2(v[0], v[1]);
        }
      }
      const float* gram_tiles = ld_arg(args->gram_tiles);
      if (gram_tiles != nullptr) {                           // implicit: + Y^T Y, already in this lane's tile order
        const float4* gp = reinterpret_cast<const float4*>(gram_tiles) + lane * 18;
#pragma unroll
        for (int i = 0; i < 18; ++i) {
          const float4 g = __ldg(gp + i);
          R[2 * i] = ffma2(pack2(g.x, g.y), pack2(1.f, 1.f), R[2 * i]);
          R[2 * i + 1] = ffma2(pack2(g.z, g.w), pack2(1.f, 1.f), R[2 * i + 1]);
        }
      }
      const uint32_t ob = (uint32_t)(ti + 8 * tj) * 4u;
      bb2 = pack2(lds32(B1 + ob) + lds32(B2 + ob), lds32(B1 + ob + 16) + lds32(B2 + ob + 16));
      __syncwarp();
      if (lane == 0) umma::mbar_arrive(&bars->slot_free[sl]);
      WS_ACC(t_load);
    }
    {
      WS_T0();
      eliminate(R, bb2, P, Y);
      WS_ACC(t_elim);
    }
    {
      WS_T0();
      const int row = __ldg(ld_arg(args->item_row) + it);   // in flight during the back substitution
      back_store(R, Y, DI, T, RH, ti, tj, lane, ld_arg(args->dst), ld_arg(args->dst_hl), row);
      WS_ACC(t_back);
    }
#ifdef HALS_WS_PROFILE
    ++n_solved;
#endif
  }
#ifdef HALS_WS_PROFILE
  if (lane == 0 && blockIdx.x == 1)
    printf("S%d: solved %d wait_slot %lld load %lld elim %lld back %lld\n", w, n_solved, w_slot, t_load, t_elim, t_back);
#endif
}

__global__ void __launch_bounds__(kThreads, 1)
als_ws64_kernel(const int32_t* __restrict__ colidx, const uint32_t* __restrict__ vals_hl,
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
  __shared__ SolverArgs sargs;
  __shared__ uint32_t tmem_slot;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == kWarpDrain) umma::tmem_alloc(&tmem_slot, kAcc * kAccCols);
  if (tid == 32) {
    for (int s = 0; s < kStages; ++s) {
      umma::mbar_init(&bars.st_full[s], 32);
      umma::mbar_init(&bars.st_free[s], 1);
      umma::mbar_init(&bars.st_scaled[s], 1);
    }
    for (int b = 0; b < kAcc; ++b) { umma::mbar_init(&bars.acc_full[b], 1); umma::mbar_init(&bars.acc_free[b], 128); }
    for (int s = 0; s < kSlots; ++s) umma::mbar_init(&bars.slot_free[s], 1);
    for (int s = 0; s < kSolvers; ++s) umma::mbar_init(&bars.sol_full[s], 128);
    umma::mbar_fence_init();
  }
  if (tid < 2) cta_range(&range, item_cost0, item_chunk0, n_items, tid);
  if (tid == 64) sargs = SolverArgs{dst, dst_hl, workspace, gram_tiles, item_row, item_len, item_slot, reg};
  zero_r_blocks<K, kStages, kThreads>(base, tid);
  umma::fence_proxy_async();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint32_t sbase = umma::smem_u32(base);
#ifdef HALS_WS_PROFILE
  const long long t_cta0 = clock64();
#endif
  const uint32_t slots = sbase + kStages * kStageBytes;
  const uint32_t scratch = slots + kSlots * kSlotBytes;
  uint8_t* gscratch = base + kStages * kStageBytes + kSlots * kSlotBytes + kSolvers * kScratchBytes;

  // implicit mode: the last solver warp becomes the scaler (eight solvers instead of nine)
  const bool implicit = vals_sc != nullptr;
  const int nsolv = implicit ? kSolvers - 1 : kSolvers;
  if (warp >= kWarpDrain) {
    drain_role(slots, tmem, &bars, &range, nsolv, tid - kWarpDrain * 32);
  } else if (warp >= kWarpGather && warp < kWarpMma) {
    gather_role(sbase, &bars, gscratch + (warp - kWarpGather) * kGatherScratch, &range, colidx, vals_hl, vals_sc,
                reinterpret_cast<const uint8_t*>(src_hl), zero_row, chunk_pos, chunk_cnt, warp - kWarpGather, lane);
  } else if (warp == kWarpMma) {
    mma_role(sbase, tmem, &bars, &range, chunk_cnt, implicit, lane);
  } else if (warp - kWarpSolver < nsolv) {
    solver_role(slots, scratch + (uint32_t)(warp - kWarpSolver) * kScratchBytes, &bars, &sargs, &range, nsolv,
                warp - kWarpSolver, lane);
  } else {
    scaler_role(sbase, &bars, &range, lane);
  }
#ifdef HALS_WS_PROFILE
  const long long t_role = clock64() - t_cta0;
#endif
  umma::fence_before_sync();
  __syncthreads();
#ifdef HALS_WS_PROFILE
  if (lane == 0 && (warp == kWarpDrain || warp == kWarpGather || warp == kWarpMma || warp == kWarpSolver))
    printf("C %d w%d role %lld cta %lld\n", (int)blockIdx.x, warp, t_role, clock64() - t_cta0);
#endif
  if (warp == kWarpDrain) umma::tmem_dealloc(tmem, kAcc * kAccCols);
}

// Long rows: the slices of a row cut at plan time parked their partial (A, b, n) in workspace slots (rows of more
// than 16 / 256 slices were pre-summed in groups by als_slot_group_sum_kernel).  One CTA per long row: 128 threads sum
// the remaining <= 16 partials in slot order (coalesced, deterministic), warp 0 solves with the same one-warp LDL^T as
// the main kernel.  Replaces the round-1 reduce kernel (thread = matrix row, a CTA barrier per pivot: 20-48 us).
__global__ void __launch_bounds__(128)
als_reduce_solve64_warp_kernel(const float* __restrict__ workspace, float* __restrict__ dst,
                               __nv_bfloat16* __restrict__ dst_hl, float reg, const int32_t* __restrict__ long_row,
                               const int32_t* __restrict__ long_slot0, const int32_t* __restrict__ long_nseg,
                               const float* __restrict__ gram) {
  constexpr int SF = K * K + K + 4;
  __shared__ __align__(16) float sA[SF];
  __shared__ __align__(512) uint8_t sScratch[kScratchBytes];   // P flips buffers by bit 8
  const int tid = threadIdx.x, lane = tid & 31;
  const int row = long_row[blockIdx.x];
  const int s0 = long_slot0[blockIdx.x], ns = long_nseg[blockIdx.x];
  const int stride = slot_final_stride(ns);
  for (int e = tid * 4; e < SF; e += 128 * 4) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q = 0; q < ns; q += stride) {
      const float4 v = *reinterpret_cast<const float4*>(workspace + (size_t)(s0 + q) * SF + e);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(sA + e) = acc;
  }
  __syncthreads();
  if (tid >= 32) return;
  const int ti = lane >> 3, tj = lane & 7;
  const float lam = reg * sA[K * K + K];
  f32x2 R[36];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
#pragma unroll
    for (int c = 0; c <= q; ++c) {
      float v[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int m = ti + 4 * h + 8 * q, n = tj + 8 * c;
        v[h] = sA[m * K + n] + (m == n ? lam : 0.f) + (gram != nullptr ? __ldg(gram + m * K + n) : 0.f);
      }
      R[tri(q, c)] = pack2(v[0], v[1]);
    }
  }
  f32x2 bb2 = pack2(sA[K * K + ti + 8 * tj], sA[K * K + ti + 4 + 8 * tj]);
  const uint32_t P = umma::smem_u32(sScratch), Y = P + 512, DI = Y + 256, T = DI + 256, RH = T + 256;
  eliminate(R, bb2, P, Y);
  back_store(R, Y, DI, T, RH, ti, tj, lane, dst, dst_hl, row);
}

}  // namespace ws64

// Y^T Y ([64][64]) -> the one-warp solver's lane-tile order: tiles[lane][tri(q, c)] = (G[ti + 8q][tj + 8c],
// G[ti + 4 + 8q][tj + 8c]), lane = 8 ti + tj.
__global__ void gram_to_tiles64_kernel(const float* __restrict__ G, float* __restrict__ tiles) {
  const int lane = threadIdx.x, ti = lane >> 3, tj = lane & 7;
  for (int q = 0; q < 8; ++q)
    for (int c = 0; c <= q; ++c)
      for (int h = 0; h < 2; ++h)
        tiles[lane * 72 + ws64::tri(q, c) * 2 + h] = G[(ti + 4 * h + 8 * q) * ws64::K + tj + 8 * c];
}

// src != nullptr: fp32 source factors, split into `split_buf` first (the stateless C-ABI call).
// src == nullptr: `split_buf` already holds the split source ([n_src + 1][128] bf16, row n_src all zero) -- the
// engine keeps the factors in this form across half-steps: every solved row is written as fp32 (dst) AND as its
// bf16 hi|lo split (dst_hl, same row indexing as dst), so no split pass is needed and a sharded run all-gathers the
// split rows in place.
// gram != nullptr selects implicit feedback (the plan must carry vals_scale / item_npos packed for the caller's alpha;
// gram_tiles = 9,216 bytes of scratch).
int als_half_step_ws64(const int32_t* colidx, const uint32_t* vals_hl, const float* src, int64_t n_src, float* dst,
                       float reg, const hals_als_plan* plan, float* slots, void* split_buf, void* dst_hl,
                       const float* gram, float* gram_tiles, cudaStream_t st) {
  using namespace ws64;
  __nv_bfloat16* hl = reinterpret_cast<__nv_bfloat16*>(split_buf);
  HALS_REQUIRE(n_src < (int64_t)1 << 31, "at most 2^31 - 1 source rows");
  if (src != nullptr) {
    if (int rc = als_launch_split_bf16(src, n_src, K, hl, st)) return rc;
    // row n_src of the split buffer (inside the workspace's slack): all zero, what the ragged tail of an item gathers
    HALS_CUDA(cudaMemsetAsync(hl + (size_t)n_src * 2 * K, 0, 4 * K, st));
  }
  const size_t smem = (size_t)kStages * kStageBytes + (size_t)kSlots * kSlotBytes + (size_t)kSolvers * kScratchBytes +
                      2 * kGatherScratch + 1024;
  static_assert(kStages * kStageBytes + kSlots * kSlotBytes + kSolvers * kScratchBytes + 2 * kGatherScratch + 1024 <= 227 * 1024 - 1024,
                "shared memory budget");
  HALS_CUDA(cudaFuncSetAttribute(als_ws64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const bool implicit = gram != nullptr;
  if (implicit) {
    HALS_REQUIRE(plan->vals_scale && plan->item_npos && gram_tiles, "implicit mode needs the plan's vals_scale / item_npos");
    gram_to_tiles64_kernel<<<1, 32, 0, st>>>(gram, gram_tiles);
    HALS_LAUNCH_CHECK();
  }
  int64_t grid = sm_count();
  if (grid > plan->n_items) grid = plan->n_items;
  als_ws64_kernel<<<(unsigned)grid, kThreads, smem, st>>>(colidx, vals_hl, implicit ? plan->vals_scale : nullptr,
                                                         implicit ? gram_tiles : nullptr, hl, dst, reg, plan->item_row,
                                                         implicit ? plan->item_npos : plan->item_len, plan->item_slot, plan->item_chunk0, plan->item_cost0,
                                                         plan->chunk_pos, plan->chunk_cnt, plan->n_items, (int)n_src, slots,
                                                         reinterpret_cast<__nv_bfloat16*>(dst_hl));
  HALS_LAUNCH_CHECK();
  if (plan->n_long_rows > 0) {
    if (int rc = als_launch_slot_group_sum(slots, plan, K * K + K + 4, st)) return rc;
    als_reduce_solve64_warp_kernel<<<(unsigned)plan->n_long_rows, 128, 0, st>>>(
        slots, dst, reinterpret_cast<__nv_bfloat16*>(dst_hl), reg, plan->long_row, plan->long_slot0, plan->long_nseg, gram);
    HALS_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace hals
