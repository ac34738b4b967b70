// ALS half-step, CUDA-core (SIMT fp32) path: any rank k <= 128.
//
// Replaces Spark's computeFactors (NormalEquation.add + CholeskySolver.solve) reached
// from the reference at src/als_model.py:62.  One CTA per work item (a destination row,
// or one <= seg_len slice of a long row):
//   * the item's ratings are walked in chunks of T=32; warp 0 stages (colidx, weights),
//     all threads gather the 32 source factor rows with cp.async into a double-buffered
//     shared tile (coalesced: a factor row is one contiguous k*4-byte run);
//   * the k x k normal matrix lives in registers, (KP/16)^2 entries per thread, rows and
//     columns interleaved so that the shared-memory reads are 16-byte vectors without
//     bank conflicts; b = sum w*y is kept by the first KP threads;
//   * whole rows are factorised in place (Cholesky-Crout in shared memory, the right
//     hand side carried as an extra row so the forward substitution is free) and the
//     solution is written straight to the destination factor row;
//   * slices of long rows write their partial (A, b, n) to the workspace; a second
//     kernel sums the slots in slot order (deterministic) and solves;
//   * nonnegative factors (Spark's nonnegative=True): the *_nnls_kernel instantiations replace the
//     Cholesky solve by the block-principal-pivoting NNLS of als_common.cuh, same build and reduce.
// This path is the correctness baseline and the fallback for ranks the tensor-core path
// (als_tc.cu) does not cover.
#include "als_common.cuh"

namespace hals {

// Body of the build kernels.  tid = threadIdx.x is read in the kernel itself, where its range is known (the plain
// kernels compile to the same code as before the body was shared).  NONNEG: solve with nnls_solve_smem (x >= 0) instead
// of cholesky_solve_smem; rows that reach its iteration cap are counted in *n_capped (optional).
template <int KP, bool IMPLICIT, bool VEC, bool NONNEG>
__device__ __forceinline__ void
als_build_solve(const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                const float* __restrict__ src, float* __restrict__ dst, int k, float reg,
                float alpha, const float* __restrict__ gram,
                const int32_t* __restrict__ item_row, const int64_t* __restrict__ item_begin,
                const int32_t* __restrict__ item_len, const int32_t* __restrict__ item_slot,
                float* __restrict__ workspace, int32_t* __restrict__ n_capped, const int tid) {
  using TL = AlsTile<KP>;
  constexpr int TM = TL::TM, V = TL::V, NG = TL::NG, LD = TL::LD, T = kAlsChunk;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AlsSmem<KP>& sm = *reinterpret_cast<AlsSmem<KP>*>(smem_raw);

  const int tx = tid & 15, ty = tid >> 4;
  const int item = blockIdx.x;
  const int row = item_row[item];
  const int64_t begin = item_begin[item];
  const int len = item_len[item];
  const int slot = item_slot[item];
  const int nchunks = (len + T - 1) / T;

  // zero the padded columns of both gather buffers once (never written by the gather)
  if (k < KP) {
    for (int e = tid; e < 2 * T * KP; e += kAlsThreads) (&sm.G[0][0])[e] = 0.f;
  }

  float acc[TM][TM];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TM; ++j) acc[i][j] = 0.f;
  float bacc = 0.f;
  int npos = 0;  // warp 0 only: number of ratings counted in n

  auto load_idx = [&](int c) {
    if (tid < T) {
      const int t = c * T + tid;
      const bool ok = t < len;
      const int64_t p = begin + (ok ? t : 0);
      const int ci = colidx[p];
      const float r = vals[p];
      float wa, wb;
      bool counted;
      if (IMPLICIT) {
        const float c1 = alpha * fabsf(r);
        wa = c1;
        counted = r > 0.f;
        wb = counted ? 1.f + c1 : 0.f;
      } else {
        wa = 1.f;
        wb = r;
        counted = true;
      }
      const int st = c % 3;
      sm.idx[st][tid] = ok ? ci : -1;   // -1: the gather zero-fills this row
      sm.wa[st][tid] = ok ? wa : 0.f;
      sm.wb[st][tid] = ok ? wb : 0.f;
      npos += __popc(__ballot_sync(0xffffffffu, ok && counted));
    }
  };
  auto gather = [&](int c) {
    const int st = c % 3;
    float* G = sm.G[c & 1];
    if (VEC) {
      const int k4 = k >> 2;
      for (int q = tid; q < T * k4; q += kAlsThreads) {
        const int t = q / k4, c4 = q - t * k4;
        const int ci = sm.idx[st][t];
        cp_async16(G + t * KP + c4 * 4, src + (int64_t)(ci < 0 ? 0 : ci) * k + c4 * 4, ci >= 0);
      }
    } else {
      for (int q = tid; q < T * k; q += kAlsThreads) {
        const int t = q / k, f = q - t * k;
        const int ci = sm.idx[st][t];
        cp_async4(G + t * KP + f, src + (int64_t)(ci < 0 ? 0 : ci) * k + f, ci >= 0);
      }
    }
  };

  load_idx(0);
  if (nchunks > 1) load_idx(1);
  __syncthreads();
  gather(0);
  cp_async_commit();

  for (int c = 0; c < nchunks; ++c) {
    if (c + 1 < nchunks) gather(c + 1);
    cp_async_commit();
    if (c + 2 < nchunks) load_idx(c + 2);
    cp_async_wait<1>();
    __syncthreads();

    const float* G = sm.G[c & 1];
    const float* wa = sm.wa[c % 3];
    const float* wb = sm.wb[c % 3];
#pragma unroll 4
    for (int t = 0; t < T; ++t) {
      float a[TM], b[TM];
      const float* g = G + t * KP;
#pragma unroll
      for (int gi = 0; gi < NG; ++gi) {
        if (V == 4) {
          const float4 va = *reinterpret_cast<const float4*>(g + TL::idx(gi, 0, ty));
          const float4 vb = *reinterpret_cast<const float4*>(g + TL::idx(gi, 0, tx));
          a[gi * 4 + 0] = va.x; a[gi * 4 + 1] = va.y; a[gi * 4 + 2] = va.z; a[gi * 4 + 3] = va.w;
          b[gi * 4 + 0] = vb.x; b[gi * 4 + 1] = vb.y; b[gi * 4 + 2] = vb.z; b[gi * 4 + 3] = vb.w;
        } else {
#pragma unroll
          for (int v = 0; v < V; ++v) {
            a[gi * V + v] = g[TL::idx(gi, v, ty)];
            b[gi * V + v] = g[TL::idx(gi, v, tx)];
          }
        }
      }
      if (IMPLICIT) {
        const float w = wa[t];
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] *= w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TM; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (tid < KP) {
      float s = 0.f;
#pragma unroll 8
      for (int t = 0; t < T; ++t) s = fmaf(wb[t], G[t * KP + tid], s);
      bacc += s;
    }
    __syncthreads();
  }
  cp_async_wait<0>();

  const float nf = (float)__shfl_sync(0xffffffffu, npos, 0);  // meaningful in warp 0

  if (slot >= 0) {
    // slice of a long row: park the partial sums, the reduce kernel finishes the row
    float* W = workspace + (size_t)slot * als_slot_floats(KP);
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TM; ++j)
        W[TL::idx(i / V, i % V, ty) * KP + TL::idx(j / V, j % V, tx)] = acc[i][j];
    if (tid < KP) W[KP * KP + tid] = bacc;
    if (tid == 0) W[KP * KP + KP] = nf;
    return;
  }

  float* S = sm.A;
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TM; ++j)
      S[TL::idx(i / V, i % V, ty) * LD + TL::idx(j / V, j % V, tx)] = acc[i][j];
  if (tid < KP) S[KP * LD + tid] = bacc;
  if (tid == 0) S[KP * LD + KP] = nf;
  __syncthreads();
  const float lam = reg * S[KP * LD + KP];
  if (IMPLICIT) {
    for (int e = tid; e < k * k; e += kAlsThreads) {
      const int i = e / k, j = e - i * k;
      S[i * LD + j] += gram[e];
    }
    __syncthreads();
  }
  if (tid < k) S[tid * LD + tid] += lam;
  __syncthreads();
  if (NONNEG) {
    // the gather buffers are idle now: they hold the solver's scratch
    static_assert(sizeof(NnlsScratch<KP>) <= sizeof(sm.G), "NNLS scratch must fit the gather buffers");
    float x;
    const bool capped = nnls_solve_smem<KP>(S, k, *reinterpret_cast<NnlsScratch<KP>*>(&sm.G[0][0]), x);
    if (tid < k) dst[(int64_t)row * k + tid] = x;
    if (capped && tid == 0 && n_capped != nullptr) atomicAdd(n_capped, 1);
    return;
  }
  cholesky_solve_smem<KP>(S, k);
  if (tid < k) dst[(int64_t)row * k + tid] = S[KP * LD + tid];
}

template <int KP, bool IMPLICIT, bool VEC>
__global__ void __launch_bounds__(kAlsThreads)
als_build_solve_kernel(const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                       const float* __restrict__ src, float* __restrict__ dst, int k, float reg,
                       float alpha, const float* __restrict__ gram,
                       const int32_t* __restrict__ item_row, const int64_t* __restrict__ item_begin,
                       const int32_t* __restrict__ item_len, const int32_t* __restrict__ item_slot,
                       float* __restrict__ workspace) {
  als_build_solve<KP, IMPLICIT, VEC, false>(colidx, vals, src, dst, k, reg, alpha, gram, item_row, item_begin,
                                            item_len, item_slot, workspace, nullptr, threadIdx.x);
}

// The same kernel with the nonnegative solve (a kernel name of its own: profiles tell the two apart).
template <int KP, bool IMPLICIT, bool VEC>
__global__ void __launch_bounds__(kAlsThreads)
als_build_solve_nnls_kernel(const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                            const float* __restrict__ src, float* __restrict__ dst, int k, float reg,
                            float alpha, const float* __restrict__ gram,
                            const int32_t* __restrict__ item_row, const int64_t* __restrict__ item_begin,
                            const int32_t* __restrict__ item_len, const int32_t* __restrict__ item_slot,
                            float* __restrict__ workspace, int32_t* __restrict__ n_capped) {
  als_build_solve<KP, IMPLICIT, VEC, true>(colidx, vals, src, dst, k, reg, alpha, gram, item_row, item_begin,
                                           item_len, item_slot, workspace, n_capped, threadIdx.x);
}

// Long rows: sum the per-slice partials in slot order, add Gram / ridge, solve.  NONNEG: the NNLS scratch follows the
// (KP + 1) x LD system in shared memory.
template <int KP, bool NONNEG>
__device__ __forceinline__ void
als_reduce_solve(const float* __restrict__ workspace, float* __restrict__ dst, int k,
                 float reg, const float* __restrict__ gram,
                 const int32_t* __restrict__ long_row, const int32_t* __restrict__ long_slot0,
                 const int32_t* __restrict__ long_nseg, int32_t* __restrict__ n_capped) {
  constexpr int LD = AlsTile<KP>::LD;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* S = reinterpret_cast<float*>(smem_raw);
  const int tid = threadIdx.x;
  const int row = long_row[blockIdx.x];
  const int s0 = long_slot0[blockIdx.x], ns = long_nseg[blockIdx.x];
  const size_t sf = als_slot_floats(KP);
  const int total = KP * KP + KP + 1;
  for (int e = tid; e < total; e += kAlsThreads) {
    float s = 0.f;
    const float* W = workspace + (size_t)s0 * sf + e;
    for (int q = 0; q < ns; ++q) s += W[(size_t)q * sf];
    int i, j;
    if (e < KP * KP) { i = e / KP; j = e - i * KP; } else { i = KP; j = e - KP * KP; }
    if (gram != nullptr && i < k && j < k) s += gram[i * k + j];
    S[i * LD + j] = s;
  }
  __syncthreads();
  const float lam = reg * S[KP * LD + KP];
  __syncthreads();
  if (tid < k) S[tid * LD + tid] += lam;
  __syncthreads();
  if (NONNEG) {
    float x;
    const bool capped = nnls_solve_smem<KP>(S, k, *reinterpret_cast<NnlsScratch<KP>*>(S + als_reduce_system_floats(KP)), x);
    if (tid < k) dst[(int64_t)row * k + tid] = x;
    if (capped && tid == 0 && n_capped != nullptr) atomicAdd(n_capped, 1);
    return;
  }
  cholesky_solve_smem<KP>(S, k);
  if (tid < k) dst[(int64_t)row * k + tid] = S[KP * LD + tid];
}

template <int KP>
__global__ void __launch_bounds__(kAlsThreads)
als_reduce_solve_kernel(const float* __restrict__ workspace, float* __restrict__ dst, int k,
                        float reg, const float* __restrict__ gram,
                        const int32_t* __restrict__ long_row, const int32_t* __restrict__ long_slot0,
                        const int32_t* __restrict__ long_nseg) {
  als_reduce_solve<KP, false>(workspace, dst, k, reg, gram, long_row, long_slot0, long_nseg, nullptr);
}

template <int KP>
__global__ void __launch_bounds__(kAlsThreads)
als_reduce_solve_nnls_kernel(const float* __restrict__ workspace, float* __restrict__ dst, int k,
                             float reg, const float* __restrict__ gram,
                             const int32_t* __restrict__ long_row, const int32_t* __restrict__ long_slot0,
                             const int32_t* __restrict__ long_nseg, int32_t* __restrict__ n_capped) {
  als_reduce_solve<KP, true>(workspace, dst, k, reg, gram, long_row, long_slot0, long_nseg, n_capped);
}

template <int KP>
static int launch_simt(const int32_t* colidx, const float* vals, const float* src, float* dst, int k,
                       float reg, int implicit, float alpha, const float* gram,
                       const hals_als_plan* plan, float* ws, cudaStream_t st, bool nonneg, int32_t* n_capped) {
  const size_t smem = sizeof(AlsSmem<KP>);
  const bool vec = (k % 4 == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  auto run = [&](auto kern) -> int {
    HALS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)plan->n_items, kAlsThreads, smem, st>>>(
        colidx, vals, src, dst, k, reg, alpha, gram, plan->item_row, plan->item_begin,
        plan->item_len, plan->item_slot, ws);
    HALS_LAUNCH_CHECK();
    return 0;
  };
  auto run_nn = [&](auto kern) -> int {
    HALS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)plan->n_items, kAlsThreads, smem, st>>>(
        colidx, vals, src, dst, k, reg, alpha, gram, plan->item_row, plan->item_begin,
        plan->item_len, plan->item_slot, ws, n_capped);
    HALS_LAUNCH_CHECK();
    return 0;
  };
  int rc;
  if (nonneg) {
    if (implicit) rc = vec ? run_nn(als_build_solve_nnls_kernel<KP, true, true>) : run_nn(als_build_solve_nnls_kernel<KP, true, false>);
    else rc = vec ? run_nn(als_build_solve_nnls_kernel<KP, false, true>) : run_nn(als_build_solve_nnls_kernel<KP, false, false>);
  } else {
    if (implicit) rc = vec ? run(als_build_solve_kernel<KP, true, true>) : run(als_build_solve_kernel<KP, true, false>);
    else rc = vec ? run(als_build_solve_kernel<KP, false, true>) : run(als_build_solve_kernel<KP, false, false>);
  }
  if (rc) return rc;
  if (plan->n_long_rows > 0)
    return als_launch_reduce_solve(ws, dst, k, reg, implicit ? gram : nullptr, plan, st, nonneg, n_capped);
  return 0;
}

template <int KP>
static int launch_reduce(const float* ws, float* dst, int k, float reg, const float* gram,
                         const hals_als_plan* plan, cudaStream_t st, bool nonneg, int32_t* n_capped) {
  const size_t smem2 = sizeof(float) * (KP + 1) * AlsTile<KP>::LD;
  if (nonneg) {
    const size_t smem3 = sizeof(float) * als_reduce_system_floats(KP) + sizeof(NnlsScratch<KP>);
    HALS_CUDA(cudaFuncSetAttribute(als_reduce_solve_nnls_kernel<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
    als_reduce_solve_nnls_kernel<KP><<<(unsigned)plan->n_long_rows, kAlsThreads, smem3, st>>>(
        ws, dst, k, reg, gram, plan->long_row, plan->long_slot0, plan->long_nseg, n_capped);
    HALS_LAUNCH_CHECK();
    return 0;
  }
  HALS_CUDA(cudaFuncSetAttribute(als_reduce_solve_kernel<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
  als_reduce_solve_kernel<KP><<<(unsigned)plan->n_long_rows, kAlsThreads, smem2, st>>>(
      ws, dst, k, reg, gram, plan->long_row, plan->long_slot0, plan->long_nseg);
  HALS_LAUNCH_CHECK();
  return 0;
}

int als_launch_reduce_solve(const float* ws, float* dst, int k, float reg, const float* gram,
                            const hals_als_plan* plan, cudaStream_t st, bool nonneg, int32_t* n_capped) {
  if (plan->n_long_rows <= 0) return 0;
  switch (als_padded_rank(k)) {
    case 16: return launch_reduce<16>(ws, dst, k, reg, gram, plan, st, nonneg, n_capped);
    case 32: return launch_reduce<32>(ws, dst, k, reg, gram, plan, st, nonneg, n_capped);
    case 64: return launch_reduce<64>(ws, dst, k, reg, gram, plan, st, nonneg, n_capped);
    default: return launch_reduce<128>(ws, dst, k, reg, gram, plan, st, nonneg, n_capped);
  }
}

int als_half_step_simt(const int32_t* colidx, const float* vals, const float* src, float* dst, int k,
                       float reg, int implicit, float alpha, const float* gram,
                       const hals_als_plan* plan, float* ws, cudaStream_t st, bool nonneg, int32_t* n_capped) {
  switch (als_padded_rank(k)) {
    case 16: return launch_simt<16>(colidx, vals, src, dst, k, reg, implicit, alpha, gram, plan, ws, st, nonneg, n_capped);
    case 32: return launch_simt<32>(colidx, vals, src, dst, k, reg, implicit, alpha, gram, plan, ws, st, nonneg, n_capped);
    case 64: return launch_simt<64>(colidx, vals, src, dst, k, reg, implicit, alpha, gram, plan, ws, st, nonneg, n_capped);
    default: return launch_simt<128>(colidx, vals, src, dst, k, reg, implicit, alpha, gram, plan, ws, st, nonneg, n_capped);
  }
}

}  // namespace hals
