// Pieces shared by the SIMT and tensor-core ALS paths: tile geometry, workspace slot layout and
// the in-shared-memory Cholesky solve (Spark's CholeskySolver.solve -> LAPACK dppsv, behind
// src/als_model.py:62).
#pragma once
#include "common.cuh"

namespace hals {

constexpr int kAlsThreads = 256;
constexpr int kAlsChunk = 32;

template <int KP>
struct AlsTile {
  static constexpr int TM = KP / 16;            // tile edge per thread
  static constexpr int V = TM >= 4 ? 4 : TM;    // vector width of a shared read
  static constexpr int NG = TM / V;             // vector groups
  static constexpr int LD = KP + 1;             // padded leading dimension of A in smem
  // logical row/column owned by (group g, lane-in-vector v) of thread coordinate t
  __device__ static __forceinline__ int idx(int g, int v, int t) { return g * (16 * V) + t * V + v; }
};

template <int KP>
struct AlsSmem {
  float A[((KP + 1) * AlsTile<KP>::LD + 3) / 4 * 4];  // k x k normal matrix + rhs row (row KP), 16B multiple
  alignas(16) float G[2][kAlsChunk * KP];                   // gathered source rows, double buffered
  int idx[3][kAlsChunk];
  float wa[3][kAlsChunk];                       // weight of y y^T
  float wb[3][kAlsChunk];                       // weight of y in b
};

// Floats of the reduce kernel's (KP + 1) x LD system, rounded up to 16 bytes.
__host__ __device__ inline size_t als_reduce_system_floats(int KP) { return ((size_t)(KP + 1) * (KP + 1) + 3) / 4 * 4; }

// Slot layout in the workspace: KP*KP (A, full square) + KP (b) + 1 (n) floats, padded to 4.
__host__ __device__ inline size_t als_slot_floats(int KP) { return (size_t)KP * KP + KP + 4; }

__host__ __device__ inline int als_padded_rank(int k) {
  return k <= 16 ? 16 : k <= 32 ? 32 : k <= 64 ? 64 : 128;
}

// In-place Cholesky of the leading k x k block of S (lower triangle), rhs in row KP,
// followed by the back substitution; result x is left in S[KP*LD + 0..k).
template <int KP>
__device__ void cholesky_solve_smem(float* S, int k) {
  constexpr int LD = AlsTile<KP>::LD;
  const int tid = threadIdx.x;
  // Cholesky-Crout, one column per iteration, one row per thread (rows j..k-1 and rhs row).
  for (int j = 0; j < k; ++j) {
    const int r = j + tid;                        // candidate row (r == k: the rhs row)
    const int row = (r == k) ? KP : r;
    const bool active = r <= k;
    float s = 0.f, d = 1.f;
    if (active) {
      const float* Lr = S + row * LD;
      const float* Lj = S + j * LD;
      float s0 = Lr[j], s1 = 0.f, d0 = Lj[j], d1 = 0.f;
      int p = 0;
      for (; p + 1 < j; p += 2) {
        const float a0 = Lj[p], a1 = Lj[p + 1];
        s0 = fmaf(-Lr[p], a0, s0);
        s1 = fmaf(-Lr[p + 1], a1, s1);
        d0 = fmaf(-a0, a0, d0);
        d1 = fmaf(-a1, a1, d1);
      }
      if (p < j) {
        const float a0 = Lj[p];
        s0 = fmaf(-Lr[p], a0, s0);
        d0 = fmaf(-a0, a0, d0);
      }
      // every thread derives the pivot itself: no barrier between pivot and column scale
      d = sqrtf(d0 + d1);
      s = s0 + s1;
    }
    __syncthreads();                              // all reads of A[j][j] done before it is overwritten
    if (active) S[row * LD + j] = (r == j) ? d : s / d;
    __syncthreads();                              // column j of L visible
  }
  // Back substitution L^T x = z by warp 0 (z = rhs row after the factorisation).
  if (tid < 32) {
    float* z = S + KP * LD;
    for (int j = k - 1; j >= 0; --j) {
      const float xj = z[j] / S[j * LD + j];
      __syncwarp();
      if (tid == 0) z[j] = xj;
      const float* Lj = S + j * LD;
      for (int i = tid; i < j; i += 32) z[i] = fmaf(-Lj[i], xj, z[i]);
      __syncwarp();
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------------------
// Nonnegative solve (Spark's nonnegative=True, NNLSSolver): x = argmin 1/2 x^T A x - b^T x subject to x >= 0.
//
// Block principal pivoting (Kim & Park 2011) with the Judice-Pires backup rule.  x_G = 0 on the bound set G, the free set
// F solves A_FF x_F = b_F by cholesky_solve_smem, g = A x - b.  Every index violating x_F >= 0 or g_G >= 0 is exchanged
// while that lowers the number of violations (or, three times, when it does not); after that only the largest violating
// index is exchanged until the count drops again.  A violation of g_G >= 0 must exceed kNnlsTol * (|A_GF| |x_F| + |b_G|),
// the fp32 rounding level of g, so that rounding cannot make a degenerate index (x_i = g_i = 0) flip forever.
//
// Shared memory: A stays where the build left it.  cholesky_solve_smem writes only the lower triangle, the diagonal and
// the rhs row, so A_FF is copied compactly into the leading |F| x |F| lower triangle from the strict upper triangle
// (which nothing overwrites) and from a copy of the diagonal; b is copied too.  Deterministic: fixed summation orders,
// block-wide counts by __syncthreads_count.
constexpr float kNnlsTol = 1e-5f;
// cap on the pivoting loop (free-set factorisations per row); a row that reaches it keeps its last iterate with x >= 0
__host__ __device__ inline int als_nnls_max_iter(int k) { return 3 * k + 8; }

template <int KP>
struct NnlsScratch {
  float d[KP];        // diagonal of A
  float b[KP];        // right-hand side
  int fidx[KP];       // free set, ascending
  int wcnt[(KP + 31) / 32];
  int vmax;           // largest violating index (backup rule)
};

// A (k x k, leading dimension LD) and b (row KP) in S as cholesky_solve_smem expects them; every thread tid < k
// returns x[tid] in xout.  Returns true (in every thread) when the row reached the iteration cap.
template <int KP>
__device__ bool nnls_solve_smem(float* S, int k, NnlsScratch<KP>& W, float& xout) {
  constexpr int LD = AlsTile<KP>::LD;
  const int tid = threadIdx.x;
  const bool own = tid < k;
  float* z = S + KP * LD;
  const float bi = own ? z[tid] : 0.f;
  if (own) { W.d[tid] = S[tid * LD + tid]; W.b[tid] = bi; }
  bool inF = false;                    // start: F empty, x = 0, g = -b
  float x = 0.f, xf = 0.f, g = -bi, gs = fabsf(bi);
  int best = k + 1, left = 3;          // fewest violations so far, full exchanges left without improving on it
  const int cap = als_nnls_max_iter(k);
  bool capped = false;
  for (int it = 0;; ++it) {
    const bool bx = own && inF && x < 0.f;
    const bool bg = own && !inF && g < -kNnlsTol * gs;
    if (tid == 0) W.vmax = -1;
    if (__syncthreads_count(bx) == 0) xf = x;             // x >= 0: the last feasible iterate
    const int nv = __syncthreads_count(bx || bg);
    if (nv == 0) break;
    if (it == cap) { capped = true; break; }
    bool full = true;
    if (nv < best) { best = nv; left = 3; }
    else if (left > 0) --left;
    else full = false;
    if (!full) {
      if (bx || bg) atomicMax(&W.vmax, tid);
      __syncthreads();
    }
    if (full ? (bx || bg) : tid == W.vmax) inF = !inF;
    // compact free list: ballots per warp, prefix over warps
    const unsigned m = __ballot_sync(0xffffffffu, own && inF);
    if ((tid & 31) == 0 && tid < KP) W.wcnt[tid >> 5] = __popc(m);
    __syncthreads();
    int pos = __popc(m & ((1u << (tid & 31)) - 1u)), nf = 0;
#pragma unroll
    for (int w = 0; w < (KP + 31) / 32; ++w) {
      const int c = W.wcnt[w];
      if (w < (tid >> 5)) pos += c;
      nf += c;
    }
    if (own && inF) W.fidx[pos] = tid;
    __syncthreads();
    // A_FF into the compact lower triangle (from the strict upper one and the diagonal copy), b_F into the rhs row
    for (int e = tid; e < nf * nf; e += kAlsThreads) {
      const int r = e / nf, c = e - r * nf;
      if (c < r) S[r * LD + c] = S[W.fidx[c] * LD + W.fidx[r]];
      else if (c == r) S[r * LD + r] = W.d[W.fidx[r]];
    }
    if (tid < nf) z[tid] = W.b[W.fidx[tid]];
    __syncthreads();
    cholesky_solve_smem<KP>(S, nf);
    if (own) {
      if (inF) {
        x = z[pos];
        g = 0.f;
        gs = 0.f;
      } else {
        float acc = -bi, mag = fabsf(bi);
        for (int q = 0; q < nf; ++q) {
          const int j = W.fidx[q];
          const float a = tid < j ? S[tid * LD + j] : S[j * LD + tid], xq = z[q];
          acc = fmaf(a, xq, acc);
          mag = fmaf(fabsf(a), fabsf(xq), mag);
        }
        x = 0.f;
        g = acc;
        gs = mag;
      }
    }
  }
  xout = fmaxf(capped ? xf : x, 0.f);
  return capped;
}

// Long rows: sums the per-slice partials in slot order, adds Gram / ridge, solves (als_simt.cu).
int als_launch_reduce_solve(const float* workspace, float* dst, int k, float reg, const float* gram,
                            const hals_als_plan* plan, cudaStream_t st, bool nonneg, int32_t* n_capped);

}  // namespace hals
