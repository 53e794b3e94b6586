// Predict-time sample preparation on the GPU (SURVEY.md 8f-4): what myria3d does on the CPU between reading a LAS tile
// and handing receptive fields to the network,
//   split_cloud_into_samples   myria3d/pctl/dataset/utils.py:126-158     Chebyshev ball query around a mosaic of centres
//   GridSampling(0.25)         configs/datamodule/transforms/preparations/points_budget.yaml:76-79 (torch_geometric 2.4:
//                              voxel_grid + consecutive_cluster + scatter mean / label vote)
//   MaximumNumNodes(40000)     myria3d/pctl/transforms/transforms.py:48-60  (randperm(n)[:num]; MinimumNumNodes(:63-84) is
//                              built from the same draw on the host side)
//   Center                     torch_geometric.transforms.Center (pos - pos.mean(0)), points_budget.yaml:96-97
// as kernels behind the C ABI.  Building block: a segmented LSB radix sort (one CTA per segment, 4-bit digits, keys +
// payloads ping-ponging between two global buffers; blocked thread-to-element mapping keeps every pass stable).
#include <math_constants.h>

#include "common.cuh"
#include "sample_prep.cuh"

namespace b200 {

constexpr int SS_THREADS = 1024;

// ------------------------------------------------------------------------------------------------------------
// segmented radix sort: pairs (key, val) of segment s occupy [off[s], off[s+1]) of key_a/val_a; sorted ascending by the
// low `key_bits` bits of key (stable); the result lands back in key_a/val_a (an even number of passes is run).
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SS_THREADS)
seg_sort_kernel(uint32_t* __restrict__ key_a, uint32_t* __restrict__ val_a, uint32_t* __restrict__ key_b,
                uint32_t* __restrict__ val_b, const int64_t* __restrict__ off, int key_bits) {
  __shared__ uint32_t warp_tot[16][SS_THREADS / 32];
  __shared__ uint32_t digit_total[16], digit_base[16];
  const int seg = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t s0 = off[seg];
  const int n = (int)(off[seg + 1] - s0);
  if (n <= 1) return;
  const int per = (n + SS_THREADS - 1) / SS_THREADS;  // contiguous elements per thread (stability)
  const int lo = min(n, tid * per), hi = min(n, lo + per);
  int passes = (key_bits + 3) / 4;
  passes += passes & 1;  // even: the result ends in the A buffers
  uint32_t *ki = key_a + s0, *vi = val_a + s0, *ko = key_b + s0, *vo = val_b + s0;
  for (int p = 0; p < passes; ++p) {
    const int shift = 4 * p;
    uint32_t cnt[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) cnt[d] = 0;
    for (int i = lo; i < hi; ++i) {
      const uint32_t dg = (shift < 32) ? ((ki[i] >> shift) & 15u) : 0u;
#pragma unroll
      for (int d = 0; d < 16; ++d) cnt[d] += (dg == (uint32_t)d);
    }
    // exclusive scan over (digit, thread) in digit-major order
    uint32_t excl[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) {
      uint32_t v = cnt[d];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
      }
      excl[d] = v - cnt[d];  // within the warp
      if (lane == 31) warp_tot[d][warp] = v;
    }
    __syncthreads();
    if (warp < 16) {  // warp d scans the 32 warp totals of digit d
      const uint32_t t = warp_tot[warp][lane];
      uint32_t v = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
      }
      warp_tot[warp][lane] = v - t;
      if (lane == 31) digit_total[warp] = v;
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t run = 0;
      for (int d = 0; d < 16; ++d) {
        digit_base[d] = run;
        run += digit_total[d];
      }
    }
    __syncthreads();
    uint32_t pos[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) pos[d] = digit_base[d] + warp_tot[d][warp] + excl[d];
    for (int i = lo; i < hi; ++i) {
      const uint32_t kk = ki[i], vv = vi[i];
      const uint32_t dg = (shift < 32) ? ((kk >> shift) & 15u) : 0u;
      uint32_t dst = 0;
#pragma unroll
      for (int d = 0; d < 16; ++d)
        if (dg == (uint32_t)d) dst = pos[d]++;
      ko[dst] = kk;
      vo[dst] = vv;
    }
    __syncthreads();
    uint32_t* t1 = ki; ki = ko; ko = t1;
    uint32_t* t2 = vi; vi = vo; vo = t2;
  }
}

// ------------------------------------------------------------------------------------------------------------
// receptive fields: field (ix, iy) has centre (w/2 + ix*stride, w/2 + iy*stride) in coordinates relative to the cloud's
// (min x, min y); a point belongs to it iff max(|dx|, |dy|) <= radius (closed Chebyshev ball, scipy
// query_ball_point(p = inf)).  Fields are numbered ix * fields_per_axis + iy (the order of get_mosaic_of_centers).
// ------------------------------------------------------------------------------------------------------------
struct FieldRange {
  int x0, x1, y0, y1;
};
__device__ __forceinline__ FieldRange covering_fields(float dx, float dy, float half, float stride, float radius, int g) {
  // centres c_i = half + i * stride; |d - c_i| <= radius  <=>  (d - half - radius) / stride <= i <= (d - half + radius) / stride.
  // Candidates from the real-valued bounds, then the exact float test the oracle performs on |d - c_i|.
  FieldRange r;
  r.x0 = max(0, (int)floorf((dx - half - radius) / stride) - 1);
  r.x1 = min(g - 1, (int)floorf((dx - half + radius) / stride) + 1);
  r.y0 = max(0, (int)floorf((dy - half - radius) / stride) - 1);
  r.y1 = min(g - 1, (int)floorf((dy - half + radius) / stride) + 1);
  return r;
}
__device__ __forceinline__ bool in_field(float d, int i, float half, float stride, float radius) {
  // the reference tests in float64 (scipy's cKDTree holds the float32 coordinates as doubles; the centres come from
  // np.arange = start + i * step in float64)
  const double c = (double)half + (double)i * (double)stride;
  return fabs((double)d - c) <= (double)radius;
}

template <bool FILL>
__global__ void __launch_bounds__(256)
receptive_fields_kernel(const float* __restrict__ pos, int64_t n, float min_x, float min_y, float half, float stride,
                        float radius, int g, int64_t* __restrict__ counts, const int64_t* __restrict__ offsets,
                        unsigned long long* __restrict__ cursors, uint32_t* __restrict__ out_idx) {
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const float dx = __fsub_rn(pos[3 * i], min_x), dy = __fsub_rn(pos[3 * i + 1], min_y);
    const FieldRange r = covering_fields(dx, dy, half, stride, radius, g);
    for (int ix = r.x0; ix <= r.x1; ++ix) {
      if (!in_field(dx, ix, half, stride, radius)) continue;
      for (int iy = r.y0; iy <= r.y1; ++iy) {
        if (!in_field(dy, iy, half, stride, radius)) continue;
        const int f = ix * g + iy;
        if (FILL) {
          const unsigned long long slot = atomicAdd(&cursors[f], 1ull);
          out_idx[offsets[f] + (int64_t)slot] = (uint32_t)i;
        } else {
          atomicAdd(reinterpret_cast<unsigned long long*>(counts) + f, 1ull);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// grid sampling of ONE sample (torch_geometric.transforms.GridSampling, one cloud): voxel id per point
//   id = sum_d floor((p_d - start_d) / size) * prod_{d' < d} (floor((end_d' - start_d') / size) + 1)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
voxel_ids_kernel(const float* __restrict__ pos, int n, float size, const float* __restrict__ start_end /* [6] */,
                 uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint32_t id = voxel_id(pos + 3 * (int64_t)i, size, start_end);
  key[i] = id;
  val[i] = (uint32_t)i;
}

// sorted (voxel id, point index): flag the first element of every run and count the runs
__global__ void __launch_bounds__(256)
voxel_heads_kernel(const uint32_t* __restrict__ key, int n, int32_t* __restrict__ head, int32_t* __restrict__ num_voxels) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const int h = (i == 0 || key[i] != key[i - 1]) ? 1 : 0;
  head[i] = h;
  if (h) atomicAdd(num_voxels, 1);
}

// one warp per voxel run: mean of pos / x rows (fp64 accumulation, index order), majority label (ties: lowest class)
__global__ void __launch_bounds__(128)
voxel_pool_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ val, const int32_t* __restrict__ run_start,
                  int num_voxels, int n, const float* __restrict__ pos, const float* __restrict__ x, int cx,
                  const int64_t* __restrict__ y, int num_classes, float* __restrict__ pos_out, float* __restrict__ x_out,
                  int64_t* __restrict__ y_out, int32_t* __restrict__ count_out) {
  const int v = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (v >= num_voxels) return;
  const int s = run_start[v], e = (v + 1 < num_voxels) ? run_start[v + 1] : n;
  pool_voxel_run(val, 0, s, e, pos, x, cx, y, num_classes, v, lane, pos_out, x_out, y_out);
  if (lane == 0 && count_out) count_out[v] = e - s;
  (void)key;
}

// random 32-bit key per element (Philox4x32-10, the stream of decimate.cu) + identity payload
__global__ void __launch_bounds__(256)
random_keys_kernel(int64_t n, uint64_t seed, const int64_t* __restrict__ counter, uint32_t salt, uint32_t* __restrict__ key,
                   uint32_t* __restrict__ val) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint64_t ctr = (uint64_t)(counter ? *counter : 0);
  key[i] = sp_philox((uint32_t)i, (uint32_t)((uint64_t)i >> 32), (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed,
                     (uint32_t)(seed >> 32) ^ salt);
  val[i] = (uint32_t)i;
}

// pos -= mean(pos) over the rows of ONE sample (torch_geometric.transforms.Center), fp64 accumulation
__global__ void __launch_bounds__(1024)
center_kernel(float* __restrict__ pos, int n) {
  __shared__ double red[32][3];
  __shared__ float mean[3];
  double a[3] = {0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < n; i += 1024) {
    a[0] += pos[3 * i], a[1] += pos[3 * i + 1], a[2] += pos[3 * i + 2];
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    a[d] = warp_sum(a[d]);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][d] = a[d];
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int w = 0; w < 32; ++w) t += red[w][threadIdx.x];
    mean[threadIdx.x] = (float)(t / (double)n);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * n; i += 1024) pos[i] = __fsub_rn(pos[i], mean[i % 3]);
}

}  // namespace b200

using namespace b200;

extern "C" int b200_segmented_sort_pairs(uint32_t* keys, uint32_t* vals, uint32_t* keys_tmp, uint32_t* vals_tmp,
                                         const int64_t* offsets, int32_t num_segments, int32_t key_bits, void* stream) {
  B200_REQUIRE(keys && vals && keys_tmp && vals_tmp && offsets, B200_E_INVALID, "b200_segmented_sort_pairs: null pointer");
  B200_REQUIRE(num_segments >= 0 && key_bits >= 1 && key_bits <= 32, B200_E_INVALID, "b200_segmented_sort_pairs: bad sizes");
  if (num_segments == 0) return B200_OK;
  seg_sort_kernel<<<(unsigned)num_segments, SS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(keys, vals, keys_tmp, vals_tmp,
                                                                                                 offsets, key_bits);
  B200_CHECK_LAUNCH("seg_sort_kernel");
  return B200_OK;
}

extern "C" int b200_receptive_fields_count(const float* pos, int64_t n, float min_x, float min_y, float tile_width,
                                           float subtile_width, float subtile_overlap, int64_t* counts, void* stream) {
  B200_REQUIRE(pos && counts, B200_E_INVALID, "b200_receptive_fields_count: null pointer");
  B200_REQUIRE(subtile_overlap >= 0.f && subtile_width > subtile_overlap, B200_E_INVALID,
               "b200_receptive_fields: subtile_overlap must be in [0, subtile_width)");
  const int g = b200_receptive_fields_per_axis(tile_width, subtile_width, subtile_overlap);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(int64_t) * (size_t)g * g, st);
  if (e != cudaSuccess) return cuda_fail(e, "receptive_fields memset");
  if (n == 0) return B200_OK;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
  receptive_fields_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(pos, n, min_x, min_y, subtile_width / 2.f,
                                                                   subtile_width - subtile_overlap, floorf(subtile_width / 2.f),
                                                                   g, counts, nullptr, nullptr, nullptr);
  B200_CHECK_LAUNCH("receptive_fields_kernel<count>");
  return B200_OK;
}

extern "C" int32_t b200_receptive_fields_per_axis(float tile_width, float subtile_width, float subtile_overlap) {
  // len(np.arange(w/2, tile + w/2 - overlap, step = w - overlap))   (pctl/dataset/utils.py:29-38)
  const double start = subtile_width / 2.0, stop = (double)tile_width + subtile_width / 2.0 - subtile_overlap;
  const double step = (double)subtile_width - subtile_overlap;
  if (step <= 0.0 || stop <= start) return 0;
  return (int32_t)ceil((stop - start) / step);
}

extern "C" int b200_receptive_fields_fill(const float* pos, int64_t n, float min_x, float min_y, float tile_width,
                                          float subtile_width, float subtile_overlap, const int64_t* offsets,
                                          uint64_t* cursors, uint32_t* idx, uint32_t* idx_tmp, uint32_t* pay, uint32_t* pay_tmp,
                                          void* stream) {
  B200_REQUIRE(pos && offsets && cursors && idx && idx_tmp && pay && pay_tmp, B200_E_INVALID,
               "b200_receptive_fields_fill: null pointer");
  B200_REQUIRE(n < (int64_t(1) << 32), B200_E_UNSUPPORTED, "b200_receptive_fields_fill: more than 2^32 points");
  const int g = b200_receptive_fields_per_axis(tile_width, subtile_width, subtile_overlap);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(cursors, 0, sizeof(uint64_t) * (size_t)g * g, st);
  if (e != cudaSuccess) return cuda_fail(e, "receptive_fields memset");
  if (n == 0 || g == 0) return B200_OK;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
  receptive_fields_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(pos, n, min_x, min_y, subtile_width / 2.f,
                                                                  subtile_width - subtile_overlap, floorf(subtile_width / 2.f), g,
                                                                  nullptr, offsets, reinterpret_cast<unsigned long long*>(cursors),
                                                                  idx);
  B200_CHECK_LAUNCH("receptive_fields_kernel<fill>");
  int bits = 1;
  while (bits < 32 && (int64_t(1) << bits) < n) ++bits;
  // ascending point index inside every field (the atomics above filled them in arbitrary order); the payload is unused
  return b200_segmented_sort_pairs(idx, pay, idx_tmp, pay_tmp, offsets, g * g, bits, stream);
}

extern "C" int b200_grid_sampling_sort(const float* pos, int32_t n, float size, const float* start_end, uint32_t* key,
                                       uint32_t* val, uint32_t* key_tmp, uint32_t* val_tmp, const int64_t* offsets01,
                                       int32_t* head, int32_t* num_voxels, void* stream) {
  B200_REQUIRE(pos && start_end && key && val && key_tmp && val_tmp && offsets01 && head && num_voxels, B200_E_INVALID,
               "b200_grid_sampling_sort: null pointer");
  B200_REQUIRE(size > 0.f && n >= 0, B200_E_INVALID, "b200_grid_sampling_sort: bad size");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(num_voxels, 0, sizeof(int32_t), st);
  if (e != cudaSuccess) return cuda_fail(e, "grid_sampling memset");
  if (n == 0) return B200_OK;
  voxel_ids_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(pos, n, size, start_end, key, val);
  B200_CHECK_LAUNCH("voxel_ids_kernel");
  const int rc = b200_segmented_sort_pairs(key, val, key_tmp, val_tmp, offsets01, 1, 32, stream);
  if (rc != B200_OK) return rc;
  voxel_heads_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(key, n, head, num_voxels);
  B200_CHECK_LAUNCH("voxel_heads_kernel");
  return B200_OK;
}

extern "C" int b200_grid_sampling_pool(const uint32_t* key, const uint32_t* val, const int32_t* run_start, int32_t num_voxels,
                                       int32_t n, const float* pos, const float* x, int32_t cx, const int64_t* y,
                                       int32_t num_classes, float* pos_out, float* x_out, int64_t* y_out, int32_t* count_out,
                                       void* stream) {
  B200_REQUIRE(key && val && run_start && pos && pos_out && (cx == 0 || (x && x_out)) && (!y || y_out), B200_E_INVALID,
               "b200_grid_sampling_pool: null pointer");
  if (num_voxels <= 0) return B200_OK;
  voxel_pool_kernel<<<(unsigned)ceil_div(num_voxels, 4), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      key, val, run_start, num_voxels, n, pos, x, cx, y, num_classes, pos_out, x_out, y_out, count_out);
  B200_CHECK_LAUNCH("voxel_pool_kernel");
  return B200_OK;
}

extern "C" int b200_random_permutation(int64_t n, uint64_t seed, const int64_t* counter, uint32_t salt, uint32_t* key,
                                       uint32_t* perm, uint32_t* key_tmp, uint32_t* perm_tmp, const int64_t* offsets01,
                                       void* stream) {
  B200_REQUIRE(key && perm && key_tmp && perm_tmp && offsets01, B200_E_INVALID, "b200_random_permutation: null pointer");
  B200_REQUIRE(n >= 0 && n < (int64_t(1) << 31), B200_E_INVALID, "b200_random_permutation: n out of range");
  if (n == 0) return B200_OK;
  random_keys_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, seed, counter, salt, key, perm);
  B200_CHECK_LAUNCH("random_keys_kernel");
  return b200_segmented_sort_pairs(key, perm, key_tmp, perm_tmp, offsets01, 1, 32, stream);
}

extern "C" int b200_center_pos(float* pos, int32_t n, void* stream) {
  B200_REQUIRE(pos, B200_E_INVALID, "b200_center_pos: null pointer");
  if (n <= 0) return B200_OK;
  center_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(pos, n);
  B200_CHECK_LAUNCH("center_kernel");
  return B200_OK;
}
