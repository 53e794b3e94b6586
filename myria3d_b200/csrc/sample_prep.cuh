// Device pieces shared by the single-sample preparation (sample_prep.cu) and the batched one (batch_prep.cu).
#pragma once
#include "common.cuh"

namespace b200 {

// Philox4x32-10 (the stream of decimate.cu): word 0 of the block for counter (i_lo, i_hi, c_lo, c_hi), key (k0, k1)
__device__ __forceinline__ uint32_t sp_philox(uint32_t i_lo, uint32_t i_hi, uint32_t c_lo, uint32_t c_hi, uint32_t k0, uint32_t k1) {
  uint32_t x0 = i_lo, x1 = i_hi, x2 = c_lo, x3 = c_hi;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
    const uint32_t y0 = hi1 ^ x1 ^ k0, y1 = lo1, y2 = hi0 ^ x3 ^ k1, y3 = lo0;
    x0 = y0, x1 = y1, x2 = y2, x3 = y3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return x0;
}

// voxel id of one point (GridSampling): sum_d floor((p_d - start_d) / size) * prod_{d' < d} (floor((end_d' - start_d') / size) + 1)
__device__ __forceinline__ uint32_t voxel_id(const float* p, float size, const float* start_end) {
  uint32_t id = 0, mul = 1;
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const float s = start_end[d], e = start_end[3 + d];
    const uint32_t c = (uint32_t)floorf(__fdiv_rn(__fsub_rn(p[d], s), size));
    const uint32_t nv = (uint32_t)floorf(__fdiv_rn(__fsub_rn(e, s), size)) + 1u;
    id += c * mul;
    mul *= nv;
  }
  return id;
}

// One warp pools the voxel run [s, e) of the sorted point indices `val` (rows base + val[t] of pos / x / y) into row v of
// the outputs: mean of pos / x rows (fp64 accumulation, index order), majority label (ties: lowest class).
__device__ __forceinline__ void pool_voxel_run(const uint32_t* __restrict__ val, int64_t base, int64_t s, int64_t e,
                                               const float* __restrict__ pos, const float* __restrict__ x, int cx,
                                               const int64_t* __restrict__ y, int num_classes, int64_t v, int lane,
                                               float* __restrict__ pos_out, float* __restrict__ x_out, int64_t* __restrict__ y_out) {
  const int cols = 3 + cx;
  for (int c = lane; c < cols; c += 32) {
    double acc = 0.0;
    for (int64_t t = s; t < e; ++t) {
      const int64_t i = base + val[t];
      acc += (c < 3) ? (double)pos[3 * i + c] : (double)x[i * cx + (c - 3)];
    }
    const float m = (float)(acc / (double)(e - s));
    if (c < 3)
      pos_out[3 * v + c] = m;
    else
      x_out[v * cx + (c - 3)] = m;
  }
  if (y != nullptr) {
    int best = 0, best_cnt = -1;
    for (int cl = lane; cl < num_classes; cl += 32) {
      int cnt = 0;
      for (int64_t t = s; t < e; ++t) cnt += (y[base + val[t]] == cl);
      if (cnt > best_cnt) best_cnt = cnt, best = cl;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int oc = __shfl_xor_sync(0xffffffffu, best_cnt, o), ob = __shfl_xor_sync(0xffffffffu, best, o);
      if (oc > best_cnt || (oc == best_cnt && ob < best)) best_cnt = oc, best = ob;
    }
    if (lane == 0) y_out[v] = best;
  }
}

}  // namespace b200
