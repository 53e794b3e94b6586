// Train / eval / predict batch preparation on the GPU: myria3d's per-sample transform chain
// (configs/datamodule/transforms/{preparations/points_budget.yaml, normalizations/default.yaml, augmentations/*.yaml},
// composed by pctl/datamodule/hdf5.py:76-89 as preparations + normalizations [+ augmentations]) run on a whole raw batch:
//   TargetTransform, DropPointsByClass      pctl/transforms/transforms.py:168-248     -> compact
//   GridSampling(0.25)                      torch_geometric 2.4 (as b200_grid_sampling_*) -> compact, voxelize, pool
//   MinimumNumNodes / MaximumNumNodes       transforms.py:48-84                        -> budget_draw
//   Center, NullifyLowestZ, NormalizePos, StandardizeRGBAndIntensity, RandomFlip, RandomRotate, Copy*  -> finalize
// Samples are the segments [ptr[b], ptr[b+1]) of the raw batch.  Every buffer before the pool is laid out like the raw
// batch (sample b at ptr[b]): dropping and pooling only shrink a sample, so nothing needs the host until the pooled
// voxel counts are known.  Launch counts do not depend on the number of samples.
#include <math_constants.h>

#include "sample_prep.cuh"

namespace b200 {

constexpr int BP_THREADS = 1024;
constexpr uint32_t BP_SALT_BUDGET = 0x6275640Bu, BP_SALT_AUGMENT = 0x61756703u;
enum { BP_TRAIN = 0, BP_EVAL = 1, BP_PREDICT = 2 };

// exclusive block scan of 0/1 flags over the 1024 threads; `ws` = 33 ints of shared memory; returns this thread's rank
__device__ __forceinline__ int bp_scan_flags(bool f, int* ws, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t m = __ballot_sync(0xffffffffu, f);
  if (lane == 0) ws[warp] = __popc(m);
  __syncthreads();
  if (warp == 0) {
    const int t = ws[lane];
    int v = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    ws[lane] = v - t;
    if (lane == 31) ws[32] = v;
  }
  __syncthreads();
  const int r = ws[warp] + __popc(m & ((1u << lane) - 1u));
  total = ws[32];
  __syncthreads();  // ws is reused by the next call
  return r;
}

template <typename T, typename Op>
__device__ __forceinline__ T bp_block_reduce(T v, T* ws, Op op) {  // ws: 32 elements of shared memory; result in all threads
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  if (lane == 0) ws[warp] = v;
  __syncthreads();
  T r = ws[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = op(r, ws[w]);
  __syncthreads();
  return r;
}
struct FMin { __device__ float operator()(float a, float b) const { return fminf(a, b); } };
struct FMax { __device__ float operator()(float a, float b) const { return fmaxf(a, b); } };
struct DSum { __device__ double operator()(double a, double b) const { return a + b; } };

// ---- (a) + (b): label map, drop flag, stable compaction, per-sample bounding box, voxel ids.  One CTA per sample.
// stats: [0] error flags, [1..8] bitmask of unknown codes, [9 + b] kept rows m_b, [9 + B + b] voxels (voxelize).
__global__ void __launch_bounds__(BP_THREADS)
bp_compact_kernel(const float* __restrict__ pos, const float* __restrict__ x, int cx, const int64_t* __restrict__ y,
                  const int64_t* __restrict__ idx, const int64_t* __restrict__ ptr, int num_samples,
                  const int32_t* __restrict__ lut, float size, float* __restrict__ pos_c, float* __restrict__ x_c,
                  int64_t* __restrict__ y_c, int64_t* __restrict__ idx_c, uint32_t* __restrict__ key,
                  uint32_t* __restrict__ val, int32_t* __restrict__ stats) {
  __shared__ int ws[33];
  __shared__ float fws[32];
  __shared__ float box[6];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int64_t s0 = ptr[b];
  const int n = (int)(ptr[b + 1] - s0);
  float lo[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, hi[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  int run = 0;
  for (int base = 0; base < n; base += BP_THREADS) {
    const int i = base + tid;
    bool keep = false;
    int64_t lab = 0;
    if (i < n) {
      keep = true;
      if (y != nullptr) {
        const int64_t code = y[s0 + i];
        if (lut == nullptr) {
          lab = code;
          keep = code != 65;
        } else if (code < 0 || code > 255) {
          atomicOr(&stats[0], B200_BATCH_PREP_E_CODE_RANGE);
          lab = -1;
        } else {
          lab = lut[code];
          if (lab < 0) {
            atomicOr(&stats[0], B200_BATCH_PREP_E_UNKNOWN_CODE);
            atomicOr(&stats[1 + (int)(code >> 5)], (int)(1u << (code & 31)));
          }
          keep = lab != 65;
        }
      }
    }
    int total;
    const int r = bp_scan_flags(keep, ws, total);
    if (keep) {
      const int64_t src = s0 + i, dst = s0 + run + r;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const float v = pos[3 * src + d];
        pos_c[3 * dst + d] = v;
        lo[d] = fminf(lo[d], v), hi[d] = fmaxf(hi[d], v);
      }
      for (int c = 0; c < cx; ++c) x_c[dst * cx + c] = x[src * cx + c];
      if (y != nullptr) y_c[dst] = lab;
      if (idx != nullptr) idx_c[dst] = idx[src];
    }
    run += total;
  }
  for (int d = 0; d < 3; ++d) {
    const float l = bp_block_reduce(lo[d], fws, FMin()), h = bp_block_reduce(hi[d], fws, FMax());
    if (tid == 0) box[d] = l, box[3 + d] = h;
  }
  if (tid == 0) {
    stats[9 + b] = run;
    if (run > 0) {  // voxel ids must fit in uint32 below the padding key 0xFFFFFFFF
      double cells = 1.0;
      for (int d = 0; d < 3; ++d) cells *= (double)floorf(__fdiv_rn(__fsub_rn(box[3 + d], box[d]), size)) + 1.0;
      if (!(cells <= 4294967295.0)) atomicOr(&stats[0], B200_BATCH_PREP_E_VOXEL_OVERFLOW);
    }
  }
  __syncthreads();
  for (int i = tid; i < n; i += BP_THREADS) {  // dropped slots get the largest key: they sort behind the sample's points
    key[s0 + i] = i < run ? voxel_id(pos_c + 3 * (s0 + i), size, box) : 0xFFFFFFFFu;
    val[s0 + i] = (uint32_t)i;
  }
}

// ---- (c): first element of every voxel run of the sorted keys -> run_start (sample-local positions), voxel count
__global__ void __launch_bounds__(BP_THREADS)
bp_heads_kernel(const uint32_t* __restrict__ key, const int64_t* __restrict__ ptr, int num_samples,
                int32_t* __restrict__ run_start, int32_t* __restrict__ stats) {
  __shared__ int ws[33];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int64_t s0 = ptr[b];
  const int m = stats[9 + b];
  int run = 0;
  for (int base = 0; base < m; base += BP_THREADS) {
    const int i = base + tid;
    const bool head = i < m && (i == 0 || key[s0 + i] != key[s0 + i - 1]);
    int total;
    const int r = bp_scan_flags(head, ws, total);
    if (head) run_start[s0 + run + r] = i;
    run += total;
  }
  if (tid == 0) stats[9 + num_samples + b] = run;
}

__device__ __forceinline__ int bp_segment_of(const int64_t* __restrict__ off, int num, int64_t v) {  // off[s] <= v < off[s+1]
  int lo = 0, hi = num - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (off[mid] <= v) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// ---- (d): one warp per (possible) voxel row of the batch; pooled rows of sample b at ptr[b]
__global__ void __launch_bounds__(128)
bp_pool_kernel(const uint32_t* __restrict__ val, const int32_t* __restrict__ run_start, const int64_t* __restrict__ ptr,
               int num_samples, int64_t n, const int32_t* __restrict__ stats, const float* __restrict__ pos_c,
               const float* __restrict__ x_c, int cx, const int64_t* __restrict__ y_c, int num_classes,
               float* __restrict__ pos_p, float* __restrict__ x_p, int64_t* __restrict__ y_p) {
  const int64_t v = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  const int b = bp_segment_of(ptr, num_samples, v);
  const int64_t s0 = ptr[b], j = v - s0;
  const int m = stats[9 + b], nv = stats[9 + num_samples + b];
  if (j >= nv) return;
  const int64_t s = s0 + run_start[v], e = s0 + ((j + 1 < nv) ? run_start[v + 1] : m);
  pool_voxel_run(val, s0, s, e, pos_c, x_c, cx, y_c, num_classes, v, lane, pos_p, x_p, y_p);
}

// ---- (e): random keys for the budget permutations: segment g = (sample seg_ids[2g], repetition seg_ids[2g+1]) of length
// seg_off[g+1] - seg_off[g]
__global__ void __launch_bounds__(256)
bp_budget_keys_kernel(const int64_t* __restrict__ seg_off, const int32_t* __restrict__ seg_ids, int num_segments,
                      uint64_t seed, const int64_t* __restrict__ counter, uint32_t* __restrict__ key, uint32_t* __restrict__ perm) {
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= seg_off[num_segments]) return;
  const int g = bp_segment_of(seg_off, num_segments, e);
  const uint64_t ctr = (uint64_t)(counter ? *counter : 0);
  const uint32_t j = (uint32_t)(e - seg_off[g]);
  // counter (row, repetition, draw counter); the sample enters the key (an odd multiple: distinct samples, distinct keys)
  const uint32_t sample = (uint32_t)seg_ids[2 * g], rep = (uint32_t)seg_ids[2 * g + 1];
  key[e] = sp_philox(j, rep, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed + sample * 0x9E3779B9u,
                     (uint32_t)(seed >> 32) ^ BP_SALT_BUDGET);
  perm[e] = j;
}

// ---- (f): one CTA per sample: gather the budget rows, fp64 statistics, normalisations, augmentations, collated outputs
__global__ void __launch_bounds__(BP_THREADS)
bp_finalize_kernel(int mode, const float* __restrict__ pos_p, const float* __restrict__ x_p, int cx,
                   const int64_t* __restrict__ y_p, const int64_t* __restrict__ ptr, const uint32_t* __restrict__ perm,
                   const int64_t* __restrict__ choice_off, const int64_t* __restrict__ out_ptr, int col_i, int col_rgb,
                   float scale, float flip_p, float rotate_degrees, uint64_t seed, const int64_t* __restrict__ counter,
                   float* __restrict__ pos_out, float* __restrict__ x_out, int64_t* __restrict__ y_out,
                   int64_t* __restrict__ batch_out, float* __restrict__ pos_sampled_copy, const float* __restrict__ pos_c,
                   const int64_t* __restrict__ y_c, const int32_t* __restrict__ stats, int num_samples,
                   const int64_t* __restrict__ full_ptr, float* __restrict__ pos_copy, int64_t* __restrict__ y_copy,
                   double* __restrict__ draws) {
  __shared__ double dws[32];
  __shared__ float fws[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int64_t p0 = ptr[b], o0 = out_ptr[b], coff = choice_off[b];
  const int s = (int)(out_ptr[b + 1] - o0);
  auto src = [&](int r) -> int64_t { return p0 + (coff >= 0 ? (int64_t)perm[coff + r] : (int64_t)r); };
  auto chan_i = [&](int64_t row) { return logf(__fadd_rn(x_p[row * cx + col_i], 1.f)); };

  // augmentation draws (RandomFlip(0, p), RandomFlip(1, p), RandomRotate(d, axis=2)): train mode only
  const uint64_t ctr = (uint64_t)(counter ? *counter : 0);
  bool flip[2] = {false, false};
  double deg = 0.0;
  if (mode == BP_TRAIN) {
    for (int k = 0; k < 3; ++k) {
      const uint32_t w = sp_philox((uint32_t)b, (uint32_t)k, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed,
                                   (uint32_t)(seed >> 32) ^ BP_SALT_AUGMENT);
      const double u = (double)w * 0x1p-32;  // [0, 1)
      if (k < 2) flip[k] = flip_p > 0.f && u < (double)flip_p;
      else if (rotate_degrees > 0.f) deg = -(double)rotate_degrees + 2.0 * (double)rotate_degrees * u;
    }
  }
  const double rad = 3.141592653589793 * deg / 180.0;
  const float cs = (float)cos(rad), sn = (float)sin(rad);
  if (tid == 0 && draws != nullptr) {
    draws[3 * b] = flip[0], draws[3 * b + 1] = flip[1], draws[3 * b + 2] = deg;
  }

  // pass 1: sums of pos, min z, channel sums
  double a[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  float zmin = CUDART_INF_F;
  for (int r = tid; r < s; r += BP_THREADS) {
    const int64_t q = src(r);
    a[0] += pos_p[3 * q], a[1] += pos_p[3 * q + 1], a[2] += pos_p[3 * q + 2];
    zmin = fminf(zmin, pos_p[3 * q + 2]);
    a[3] += chan_i(q);
    a[4] += x_p[q * cx + col_rgb];
  }
  for (int k = 0; k < 5; ++k) a[k] = bp_block_reduce(a[k], dws, DSum());
  zmin = bp_block_reduce(zmin, fws, FMin());
  float mean[3];
  for (int d = 0; d < 3; ++d) mean[d] = (float)(a[d] / (double)s);
  // min over rows commutes with the (monotone) rounded subtraction: min(z - m) = min(z) - m
  const float zlow = __fsub_rn(zmin, mean[2]);
  const double cmean_d[2] = {a[3] / (double)s, a[4] / (double)s};
  const float cmean[2] = {(float)cmean_d[0], (float)cmean_d[1]};

  // pass 2: unbiased variance of the two channels
  double q2[2] = {0.0, 0.0};
  for (int r = tid; r < s; r += BP_THREADS) {
    const int64_t q = src(r);
    const double di = (double)chan_i(q) - cmean_d[0], dr = (double)x_p[q * cx + col_rgb] - cmean_d[1];
    q2[0] += di * di, q2[1] += dr * dr;
  }
  float cstd[2];
  for (int k = 0; k < 2; ++k) {
    q2[k] = bp_block_reduce(q2[k], dws, DSum());
    const float sd = __fadd_rn((float)sqrt(q2[k] / (double)(s - 1)), 1e-6f);  // n = 1: 0 / 0 = NaN -> 1
    cstd[k] = isnan(sd) ? 1.f : sd;
  }

  // pass 3: outputs
  for (int r = tid; r < s; r += BP_THREADS) {
    const int64_t q = src(r), o = o0 + r;
    float p[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      p[d] = pos_p[3 * q + d];
      if (pos_sampled_copy != nullptr) pos_sampled_copy[3 * o + d] = p[d];
      p[d] = __fsub_rn(p[d], mean[d]);
    }
    p[2] = __fsub_rn(p[2], zlow);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      p[d] = __fmul_rn(p[d], scale);
      if (d < 2 && flip[d]) p[d] = -p[d];
    }
    if (deg != 0.0) {  // pos @ M^T, M = [[cos, sin, 0], [-sin, cos, 0], [0, 0, 1]]
      const float px = p[0], py = p[1];
      p[0] = __fadd_rn(__fmul_rn(px, cs), __fmul_rn(py, sn));
      p[1] = __fadd_rn(__fmul_rn(px, -sn), __fmul_rn(py, cs));
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) pos_out[3 * o + d] = p[d];
    for (int c = 0; c < cx; ++c) {
      float v = x_p[q * cx + c];
      if (c == col_i || c == col_rgb) {
        const int k = c == col_i ? 0 : 1;
        if (k == 0) v = chan_i(q);
        const float lim = __fmul_rn(3.f, cstd[k]);
        v = fminf(fmaxf(__fdiv_rn(__fsub_rn(v, cmean[k]), cstd[k]), -lim), lim);
      }
      x_out[o * cx + c] = v;
    }
    if (y_out != nullptr) y_out[o] = y_p[q];
    batch_out[o] = b;
  }

  // eval / predict copies of the sample after DropPointsByClass (before GridSampling)
  if (pos_copy != nullptr) {
    const int m = stats[9 + b];
    const int64_t f0 = full_ptr[b];
    for (int i = tid; i < 3 * m; i += BP_THREADS) pos_copy[3 * f0 + i] = pos_c[3 * p0 + i];
    if (y_copy != nullptr)
      for (int i = tid; i < m; i += BP_THREADS) y_copy[f0 + i] = y_c[p0 + i];
  }
  (void)num_samples;
}

}  // namespace b200

using namespace b200;

extern "C" int64_t b200_batch_prep_stats_len(int32_t num_samples) { return 9 + 2 * (int64_t)num_samples; }

extern "C" int b200_batch_prep_compact(int32_t mode, const float* pos, const float* x, int32_t cx, const int64_t* y,
                                       const int64_t* idx, const int64_t* ptr, int32_t num_samples, int64_t n,
                                       const int32_t* lut, float grid_size, float* pos_c, float* x_c, int64_t* y_c,
                                       int64_t* idx_c, uint32_t* key, uint32_t* val, int32_t* stats, void* stream) {
  B200_REQUIRE(mode >= BP_TRAIN && mode <= BP_PREDICT, B200_E_INVALID, "b200_batch_prep_compact: unknown mode %d", mode);
  B200_REQUIRE(pos && ptr && pos_c && key && val && stats && (cx == 0 || (x && x_c)) && (!y || y_c) && (!idx || idx_c),
               B200_E_INVALID, "b200_batch_prep_compact: null pointer");
  B200_REQUIRE(mode == BP_PREDICT || (y && lut), B200_E_INVALID,
               "b200_batch_prep_compact: train / eval mode needs the labels y and the label table lut");
  B200_REQUIRE(num_samples >= 1 && num_samples < 65536 && n >= 0 && n < (int64_t(1) << 31) && cx >= 0 && grid_size > 0.f,
               B200_E_INVALID, "b200_batch_prep_compact: bad sizes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(stats, 0, sizeof(int32_t) * (size_t)b200_batch_prep_stats_len(num_samples), st);
  if (e != cudaSuccess) return cuda_fail(e, "batch_prep memset");
  bp_compact_kernel<<<(unsigned)num_samples, BP_THREADS, 0, st>>>(pos, x, cx, y, idx, ptr, num_samples,
                                                                 mode == BP_PREDICT ? nullptr : lut, grid_size, pos_c, x_c,
                                                                 y_c, idx_c, key, val, stats);
  B200_CHECK_LAUNCH("bp_compact_kernel");
  return B200_OK;
}

extern "C" int b200_batch_prep_voxelize(uint32_t* key, uint32_t* val, uint32_t* key_tmp, uint32_t* val_tmp, const int64_t* ptr,
                                        int32_t num_samples, int32_t* run_start, int32_t* stats, void* stream) {
  B200_REQUIRE(key && val && key_tmp && val_tmp && ptr && run_start && stats, B200_E_INVALID,
               "b200_batch_prep_voxelize: null pointer");
  B200_REQUIRE(num_samples >= 1 && num_samples < 65536, B200_E_INVALID, "b200_batch_prep_voxelize: bad sizes");
  const int rc = b200_segmented_sort_pairs(key, val, key_tmp, val_tmp, ptr, num_samples, 32, stream);
  if (rc != B200_OK) return rc;
  bp_heads_kernel<<<(unsigned)num_samples, BP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(key, ptr, num_samples,
                                                                                                 run_start, stats);
  B200_CHECK_LAUNCH("bp_heads_kernel");
  return B200_OK;
}

extern "C" int b200_batch_prep_pool(const uint32_t* val, const int32_t* run_start, const int64_t* ptr, int32_t num_samples,
                                    int64_t n, const int32_t* stats, const float* pos_c, const float* x_c, int32_t cx,
                                    const int64_t* y_c, int32_t num_classes, float* pos_p, float* x_p, int64_t* y_p,
                                    void* stream) {
  B200_REQUIRE(val && run_start && ptr && stats && pos_c && pos_p && (cx == 0 || (x_c && x_p)) && (!y_c || y_p),
               B200_E_INVALID, "b200_batch_prep_pool: null pointer");
  B200_REQUIRE(num_samples >= 1 && n >= 0 && cx >= 0 && num_classes >= 0 && num_classes <= 256, B200_E_INVALID,
               "b200_batch_prep_pool: bad sizes");
  if (n == 0) return B200_OK;
  bp_pool_kernel<<<(unsigned)ceil_div(n, 4), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      val, run_start, ptr, num_samples, n, stats, pos_c, x_c, cx, y_c, num_classes, pos_p, x_p, y_p);
  B200_CHECK_LAUNCH("bp_pool_kernel");
  return B200_OK;
}

extern "C" int b200_batch_prep_budget_draw(const int64_t* seg_off, const int32_t* seg_ids, int32_t num_segments, int64_t total,
                                           uint64_t seed, const int64_t* counter, uint32_t* key, uint32_t* perm,
                                           uint32_t* key_tmp, uint32_t* perm_tmp, void* stream) {
  B200_REQUIRE(seg_off && seg_ids && key && perm && key_tmp && perm_tmp, B200_E_INVALID,
               "b200_batch_prep_budget_draw: null pointer");
  B200_REQUIRE(num_segments >= 0 && total >= 0 && total < (int64_t(1) << 31), B200_E_INVALID,
               "b200_batch_prep_budget_draw: bad sizes");
  if (num_segments == 0 || total == 0) return B200_OK;
  bp_budget_keys_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      seg_off, seg_ids, num_segments, seed, counter, key, perm);
  B200_CHECK_LAUNCH("bp_budget_keys_kernel");
  return b200_segmented_sort_pairs(key, perm, key_tmp, perm_tmp, seg_off, num_segments, 32, stream);
}

extern "C" int b200_batch_prep_finalize(int32_t mode, const float* pos_p, const float* x_p, int32_t cx, const int64_t* y_p,
                                        const int64_t* ptr, int32_t num_samples, const uint32_t* perm,
                                        const int64_t* choice_off, const int64_t* out_ptr, int32_t col_intensity,
                                        int32_t col_rgb, float scale, float flip_p, float rotate_degrees, uint64_t seed,
                                        const int64_t* counter, float* pos_out, float* x_out, int64_t* y_out,
                                        int64_t* batch_out, float* pos_sampled_copy, const float* pos_c, const int64_t* y_c,
                                        const int32_t* stats, const int64_t* full_ptr, float* pos_copy, int64_t* y_copy,
                                        double* draws, void* stream) {
  B200_REQUIRE(mode >= BP_TRAIN && mode <= BP_PREDICT, B200_E_INVALID, "b200_batch_prep_finalize: unknown mode %d", mode);
  B200_REQUIRE(pos_p && x_p && ptr && choice_off && out_ptr && pos_out && x_out && batch_out && (!y_p || y_out),
               B200_E_INVALID, "b200_batch_prep_finalize: null pointer");
  B200_REQUIRE(mode == BP_TRAIN || (pos_sampled_copy && pos_c && stats && full_ptr && pos_copy), B200_E_INVALID,
               "b200_batch_prep_finalize: null pointer (eval / predict copies)");
  B200_REQUIRE(mode != BP_EVAL || (y_c && y_copy), B200_E_INVALID,
               "b200_batch_prep_finalize: null pointer (eval target copy)");
  B200_REQUIRE(num_samples >= 1 && num_samples < 65536 && cx >= 1 && col_intensity >= 0 && col_intensity < cx && col_rgb >= 0 &&
                   col_rgb < cx && col_rgb != col_intensity && scale > 0.f && flip_p <= 1.f && rotate_degrees >= 0.f,
               B200_E_INVALID, "b200_batch_prep_finalize: bad sizes");
  bp_finalize_kernel<<<(unsigned)num_samples, BP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      mode, pos_p, x_p, cx, y_p, ptr, perm, choice_off, out_ptr, col_intensity, col_rgb, scale, flip_p, rotate_degrees, seed,
      counter, pos_out, x_out, y_out, batch_out, mode == BP_TRAIN ? nullptr : pos_sampled_copy, pos_c, y_c, stats, num_samples,
      full_ptr, mode == BP_TRAIN ? nullptr : pos_copy, mode == BP_EVAL ? y_copy : nullptr, draws);
  B200_CHECK_LAUNCH("bp_finalize_kernel");
  return B200_OK;
}
