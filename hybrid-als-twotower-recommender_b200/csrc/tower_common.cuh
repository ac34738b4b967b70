// Helpers shared by the tower forward kernels (towers.cu) and the tower training step (tower_train.cu).
#pragma once
#include "common.cuh"

namespace hals {

constexpr int kTowerThreads = 256;
constexpr int kTowerMaxE = 64;

// rows == 0: table size unknown, no check (ids are then trusted, as in ABI version 1 before the field existed)
__device__ __forceinline__ bool in_table(int id, int rows) { return rows <= 0 ? id >= 0 : (id >= 0 && id < rows); }

// Keras LayerNormalization statistics over the E values a warp holds (v0 = element lane, v1 = element lane + 32):
// x0, x1 = (v - mean) / sqrt(var + eps) (0 on lanes past E), inv = 1 / sqrt(var + eps).
__device__ __forceinline__ void warp_layer_norm(float v0, float v1, int E, int lane, float eps, float& x0, float& x1,
                                                float& inv) {
  const bool h0 = lane < E, h1 = lane + 32 < E;
  const float mean = warp_sum((h0 ? v0 : 0.f) + (h1 ? v1 : 0.f)) / (float)E;
  const float d0 = h0 ? v0 - mean : 0.f, d1 = h1 ? v1 - mean : 0.f;
  const float var = warp_sum(d0 * d0 + d1 * d1) / (float)E;
  inv = 1.0f / sqrtf(var + eps);
  x0 = d0 * inv;
  x1 = d1 * inv;
}

__device__ __forceinline__ void warp_layer_norm_store(float v0, float v1, int E, int lane, const float* g,
                                                      const float* b, float eps, float* out) {
  float x0, x1, inv;
  warp_layer_norm(v0, v1, E, lane, eps, x0, x1, inv);
  if (lane < E) out[lane] = fmaf(x0, g[lane], b[lane]);
  if (lane + 32 < E) out[lane + 32] = fmaf(x1, g[lane + 32], b[lane + 32]);
}

}  // namespace hals
