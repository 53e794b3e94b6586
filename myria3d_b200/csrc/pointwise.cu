// Per-point shared-MLP kernels for sm_100a: Linear (forward, input-gradient, weight-gradient) with a
// concatenated two-segment input and a BatchNorm-statistics epilogue, BatchNorm finalisation and
// the fused affine + LeakyReLU (+ residual branch) forward / backward passes.
//
// Replaces SharedMLP = PyG MLP (myria3d/models/modules/pyg_randla_net.py:97-109), fc0 / fc_classif
// (:42,:53), the torch.cat of FPModule (:251) and the block tail lrelu(mlp2(x) + shortcut(x)) (:186-187);
// in the reference each layer is cuBLAS SGEMM + 2 BatchNorm passes + an activation pass (SURVEY.md 2c K4-K6).
//
// The contractions here are fp32 FMA register-tiled (64x64 or 128x32 CTA tiles, 16-deep k slices).
// TODO(round 2): tcgen05 TF32x3 tiles for the cout >= 64 layers.
#include "common.cuh"

namespace b200 {

constexpr int GEMM_THREADS = 256;
constexpr int GEMM_BK = 16;

// one row of the (virtually concatenated) activation matrix [a1 | a2]
struct CatRows {
  const float* a1;
  int64_t ld1;
  int c1;
  const float* a2;
  int64_t ld2;
  int c2;
  bool vec;  // every row segment is float4-addressable
};

__device__ __forceinline__ float cat_load1(const CatRows& A, int64_t row, int k) {
  if (k < A.c1) return __ldg(A.a1 + row * A.ld1 + k);
  if (k < A.c1 + A.c2) return __ldg(A.a2 + row * A.ld2 + (k - A.c1));
  return 0.f;
}
__device__ __forceinline__ float4 cat_load4(const CatRows& A, int64_t row, int k) {
  if (A.vec) {
    if (k < A.c1) return __ldg(reinterpret_cast<const float4*>(A.a1 + row * A.ld1 + k));
    if (k < A.c1 + A.c2) return __ldg(reinterpret_cast<const float4*>(A.a2 + row * A.ld2 + (k - A.c1)));
    return make_float4(0.f, 0.f, 0.f, 0.f);
  }
  return make_float4(cat_load1(A, row, k), cat_load1(A, row, k + 1), cat_load1(A, row, k + 2), cat_load1(A, row, k + 3));
}

// dense row-major matrix [rows, cols] (ld = cols)
__device__ __forceinline__ float4 dense_load4(const float* __restrict__ p, int64_t rows, int cols, bool vec, int64_t r,
                                              int c) {
  if (r >= rows) return make_float4(0.f, 0.f, 0.f, 0.f);
  const float* q = p + r * cols + c;
  if (vec && c + 3 < cols) return __ldg(reinterpret_cast<const float4*>(q));
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c + 0 < cols) v.x = __ldg(q + 0);
  if (c + 1 < cols) v.y = __ldg(q + 1);
  if (c + 2 < cols) v.z = __ldg(q + 2);
  if (c + 3 < cols) v.w = __ldg(q + 3);
  return v;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static CatRows make_cat(const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2) {
  CatRows A{a1, ld1, c1, a2, ld2, c2, false};
  bool v = aligned16(a1) && (ld1 % 4 == 0) && (c1 % 4 == 0);
  if (c2 > 0) v = v && aligned16(a2) && (ld2 % 4 == 0) && (c2 % 4 == 0);
  A.vec = v;
  return A;
}

template <int BM, int BN>
struct GemmTile {
  static constexpr int TM = BM / 16, TN = BN / 16;
  static_assert(BM % 16 == 0 && BN % 32 == 0, "tile (column pairs per thread)");
  float acc[TM][TN];
  __device__ __forceinline__ void zero() {
#pragma unroll
    for (int r = 0; r < TM; ++r)
#pragma unroll
      for (int s = 0; s < TN; ++s) acc[r][s] = 0.f;
  }
  // As[kk][row], Bs[kk][col]
  __device__ __forceinline__ void mac(const float (*As)[BM + 4], const float (*Bs)[BN + 4], int ty, int tx) {
#pragma unroll
    for (int kk = 0; kk < GEMM_BK; ++kk) {
      float a[TM], b[TN];
#pragma unroll
      for (int r = 0; r < TM; ++r) a[r] = As[kk][ty * TM + r];
#pragma unroll
      for (int s = 0; s < TN; ++s) b[s] = Bs[kk][tx * TN + s];
#pragma unroll
      for (int r = 0; r < TM; ++r)
#pragma unroll
        for (int s = 0; s < TN; s += 2) ffma2_bc(a[r], b[s], b[s + 1], acc[r][s], acc[r][s + 1]);  // FFMA2, same order
    }
  }
};

// ------------------------------------------------------------------ y = [a1|a2] W^T + bias
template <int BM, int BN>
__global__ void __launch_bounds__(GEMM_THREADS)
linear_fwd_kernel(CatRows A, const float* __restrict__ w, bool wvec, const float* __restrict__ bias,
                  float* __restrict__ y, int64_t n, int cout, double* __restrict__ colstats /* [row tiles][2*cout] */) {
  __shared__ __align__(16) float As[GEMM_BK][BM + 4];
  __shared__ __align__(16) float Bs[GEMM_BK][BN + 4];
  __shared__ double cs[2][BN];
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int col0 = blockIdx.y * BN;
  const int ktot = A.c1 + A.c2;
  GemmTile<BM, BN> T;
  T.zero();
  if (colstats)
    for (int t = tid; t < 2 * BN; t += GEMM_THREADS) (&cs[0][0])[t] = 0.0;

  // register-staged double buffering: the global loads of slice k0+16 are in flight while slice k0 is multiplied
  constexpr int NA = (BM * 4 + GEMM_THREADS - 1) / GEMM_THREADS, NB = (BN * 4 + GEMM_THREADS - 1) / GEMM_THREADS;
  float4 ra[NA], rb[NB];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int q = 0; q < NA; ++q) {
      const int s = tid + q * GEMM_THREADS;
      const int r = s >> 2, kq = s & 3;
      const int64_t row = row0 + r;
      ra[q] = (s < BM * 4 && row < n) ? cat_load4(A, row, k0 + kq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const int s = tid + q * GEMM_THREADS;
      const int r = s >> 2, kq = s & 3;
      rb[q] = (s < BN * 4) ? dense_load4(w, cout, ktot, wvec, col0 + r, k0 + kq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto commit = [&]() {
#pragma unroll
    for (int q = 0; q < NA; ++q) {
      const int s = tid + q * GEMM_THREADS;
      if (s < BM * 4) {
        const int r = s >> 2, kq = s & 3;
        As[kq * 4 + 0][r] = ra[q].x, As[kq * 4 + 1][r] = ra[q].y, As[kq * 4 + 2][r] = ra[q].z, As[kq * 4 + 3][r] = ra[q].w;
      }
    }
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const int s = tid + q * GEMM_THREADS;
      if (s < BN * 4) {
        const int r = s >> 2, kq = s & 3;
        Bs[kq * 4 + 0][r] = rb[q].x, Bs[kq * 4 + 1][r] = rb[q].y, Bs[kq * 4 + 2][r] = rb[q].z, Bs[kq * 4 + 3][r] = rb[q].w;
      }
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < ktot; k0 += GEMM_BK) {
    commit();
    __syncthreads();
    if (k0 + GEMM_BK < ktot) fetch(k0 + GEMM_BK);
    T.mac(As, Bs, ty, tx);
    __syncthreads();
  }

  constexpr int TM = GemmTile<BM, BN>::TM, TN = GemmTile<BM, BN>::TN;
  // BatchNorm statistics in fp64: var = E[y^2] - E[y]^2 cancels catastrophically in fp32 when
  // |mean| >> std (e.g. the 2-row batches of tiny clouds), and fp32 x fp32 products are exact in fp64
  double psum[TN], psq[TN];
#pragma unroll
  for (int s = 0; s < TN; ++s) psum[s] = 0.0, psq[s] = 0.0;
#pragma unroll
  for (int r = 0; r < TM; ++r) {
    const int64_t row = row0 + ty * TM + r;
    if (row >= n) continue;
#pragma unroll
    for (int s = 0; s < TN; ++s) {
      const int col = col0 + tx * TN + s;
      if (col < cout) {
        const float v = T.acc[r][s] + (bias ? __ldg(bias + col) : 0.f);
        y[row * cout + col] = v;
        if (colstats) {
          psum[s] += (double)v;
          psq[s] = fma((double)v, (double)v, psq[s]);
        }
      }
    }
  }
  if (colstats) {
#pragma unroll
    for (int s = 0; s < TN; ++s) {
      atomicAdd(&cs[0][tx * TN + s], psum[s]);
      atomicAdd(&cs[1][tx * TN + s], psq[s]);
    }
    __syncthreads();
    // one partial row per row tile, written (not accumulated): no global atomics, no zero-fill needed
    double* part = colstats + (int64_t)blockIdx.x * 2 * cout;
    for (int t = tid; t < BN; t += GEMM_THREADS) {
      const int col = col0 + t;
      if (col < cout) {
        part[col] = cs[0][t];
        part[cout + col] = cs[1][t];
      }
    }
  }
}

// ------------------------------------------------------------------ [ga1|ga2] = gy W
template <int BM, int BN>
__global__ void __launch_bounds__(GEMM_THREADS)
linear_bwd_input_kernel(const float* __restrict__ gy, bool gvec, const float* __restrict__ w, bool wvec,
                        float* __restrict__ ga1, int64_t ldg1, int c1, float* __restrict__ ga2, int64_t ldg2, int c2,
                        int64_t n, int cout) {
  __shared__ __align__(16) float As[GEMM_BK][BM + 4];
  __shared__ __align__(16) float Bs[GEMM_BK][BN + 4];
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int col0 = blockIdx.y * BN;
  const int ktot = c1 + c2;
  GemmTile<BM, BN> T;
  T.zero();

  constexpr int NA = (BM * 4 + GEMM_THREADS - 1) / GEMM_THREADS;
  constexpr int NB = (GEMM_BK * (BN / 4) + GEMM_THREADS - 1) / GEMM_THREADS;
  float4 ra[NA], rb[NB];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int q = 0; q < NA; ++q) {
      const int s = tid + q * GEMM_THREADS;
      const int r = s >> 2, kq = s & 3;
      ra[q] = (s < BM * 4) ? dense_load4(gy, n, cout, gvec, row0 + r, k0 + kq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const int s = tid + q * GEMM_THREADS;
      const int kk = s / (BN / 4), cq = s % (BN / 4);
      rb[q] = (s < GEMM_BK * (BN / 4)) ? dense_load4(w, cout, ktot, wvec, k0 + kk, col0 + cq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto commit = [&]() {
#pragma unroll
    for (int q = 0; q < NA; ++q) {
      const int s = tid + q * GEMM_THREADS;
      if (s < BM * 4) {
        const int r = s >> 2, kq = s & 3;
        As[kq * 4 + 0][r] = ra[q].x, As[kq * 4 + 1][r] = ra[q].y, As[kq * 4 + 2][r] = ra[q].z, As[kq * 4 + 3][r] = ra[q].w;
      }
    }
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const int s = tid + q * GEMM_THREADS;
      if (s < GEMM_BK * (BN / 4)) *reinterpret_cast<float4*>(&Bs[s / (BN / 4)][(s % (BN / 4)) * 4]) = rb[q];
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < cout; k0 += GEMM_BK) {
    commit();
    __syncthreads();
    if (k0 + GEMM_BK < cout) fetch(k0 + GEMM_BK);
    T.mac(As, Bs, ty, tx);
    __syncthreads();
  }

  constexpr int TM = GemmTile<BM, BN>::TM, TN = GemmTile<BM, BN>::TN;
#pragma unroll
  for (int r = 0; r < TM; ++r) {
    const int64_t row = row0 + ty * TM + r;
    if (row >= n) continue;
#pragma unroll
    for (int s = 0; s < TN; ++s) {
      const int col = col0 + tx * TN + s;
      if (col < c1) {
        if (ga1) ga1[row * ldg1 + col] = T.acc[r][s];
      } else if (col < ktot) {
        if (ga2) ga2[row * ldg2 + (col - c1)] = T.acc[r][s];
      }
    }
  }
}

// ------------------------------------------------------------------ gw += gy^T [a1|a2], gb += colsum(gy)
// The bias gradient rides along as one extra "ones" column of the activation matrix.
template <int BM, int BN>
__global__ void __launch_bounds__(GEMM_THREADS)
linear_bwd_weight_kernel(const float* __restrict__ gy, bool gvec, CatRows A, float* __restrict__ gw,
                         float* __restrict__ gb, int64_t n, int cout, int64_t rows_per_split) {
  __shared__ __align__(16) float As[GEMM_BK][BM + 4];  // As[kk][m] = gy[i0+kk][m0+m]
  __shared__ __align__(16) float Bs[GEMM_BK][BN + 4];  // Bs[kk][c] = A[i0+kk][c0+c]
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  const int m0 = blockIdx.x * BM;
  const int c0 = blockIdx.y * BN;
  const int ktot = A.c1 + A.c2;
  const int ncols = ktot + (gb ? 1 : 0);
  const int64_t i_begin = (int64_t)blockIdx.z * rows_per_split;
  const int64_t i_end = (i_begin + rows_per_split < n) ? (i_begin + rows_per_split) : n;
  GemmTile<BM, BN> T;
  T.zero();

  for (int64_t i0 = i_begin; i0 < i_end; i0 += GEMM_BK) {
    for (int s = tid; s < GEMM_BK * (BM / 4); s += GEMM_THREADS) {
      const int kk = s / (BM / 4), mq = s % (BM / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i0 + kk < i_end) v = dense_load4(gy, n, cout, gvec, i0 + kk, m0 + mq * 4);
      *reinterpret_cast<float4*>(&As[kk][mq * 4]) = v;
    }
    for (int s = tid; s < GEMM_BK * (BN / 4); s += GEMM_THREADS) {
      const int kk = s / (BN / 4), cq = s % (BN / 4);
      const int c = c0 + cq * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i0 + kk < i_end) {
        if (c + 3 < ktot) {
          v = cat_load4(A, i0 + kk, c);
        } else {
          float e[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int cc = c + u;
            e[u] = (cc < ktot) ? cat_load1(A, i0 + kk, cc) : ((cc == ktot && gb) ? 1.f : 0.f);
          }
          v = make_float4(e[0], e[1], e[2], e[3]);
        }
      }
      *reinterpret_cast<float4*>(&Bs[kk][cq * 4]) = v;
    }
    __syncthreads();
    T.mac(As, Bs, ty, tx);
    __syncthreads();
  }

  constexpr int TM = GemmTile<BM, BN>::TM, TN = GemmTile<BM, BN>::TN;
#pragma unroll
  for (int r = 0; r < TM; ++r) {
    const int m = m0 + ty * TM + r;
    if (m >= cout) continue;
#pragma unroll
    for (int s = 0; s < TN; ++s) {
      const int c = c0 + tx * TN + s;
      if (c < ktot)
        atomicAdd(gw + (int64_t)m * ktot + c, T.acc[r][s]);
      else if (c < ncols)
        atomicAdd(gb + m, T.acc[r][s]);
    }
  }
}

// ------------------------------------------------------------------ tall-skinny gw += gy^T [a1|a2|1]
// Level-0/1 layers: hundreds of thousands of rows, <= 64 channels on both sides.  A tile GEMM spends its time
// on barriers there; instead each WARP streams 16-row chunks through its private shared-memory slab and every
// lane keeps the outer-product column(s) it owns in registers:
//   lane l owns activation columns l and l+32; acc[c] += gy[row][c] * a[row][l]  (gy row: LDS.128 broadcast).
// The next chunk is fetched into registers (float4, all loads in flight at once) while the current one is
// being multiplied; one shared-memory reduction and one set of global atomics per CTA at the end.
constexpr int SK_THREADS = 128;
constexpr int SK_ROWS = 16;

// AW = activation columns covered (32: lane l owns column l; 64: columns l and l+32).
// FAST: cout == CO, gy 16-byte aligned, activation segments float4-addressable (CatRows::vec).
template <int CO, int AW, bool FAST>
__global__ void __launch_bounds__(SK_THREADS)
tn_skinny_kernel(const float* __restrict__ gy, int cout, CatRows A, float* __restrict__ gw, float* __restrict__ gb,
                 int64_t n, int64_t rows_per_cta) {
  constexpr bool TWO = (AW == 64);
  extern __shared__ __align__(16) float sk_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int NW = SK_THREADS / 32;
  float* GY = sk_smem + warp * (SK_ROWS * CO + SK_ROWS * AW);  // [SK_ROWS][CO]
  float* AA = GY + SK_ROWS * CO;                                 // [SK_ROWS][AW]
  float* R = sk_smem + NW * (SK_ROWS * CO + SK_ROWS * AW);       // [CO][AW] + [CO] CTA reduction buffer
  const int ktot = A.c1 + A.c2;

  float acc0[CO], acc1[TWO ? CO : 1];
  float bs0 = 0.f, bs1 = 0.f;  // bias gradient: column sums of gy (lane l: channels l, l + 32)
#pragma unroll
  for (int c = 0; c < CO; ++c) acc0[c] = 0.f;
#pragma unroll
  for (int c = 0; c < (TWO ? CO : 1); ++c) acc1[c] = 0.f;
  for (int t = lane; t < SK_ROWS * CO; t += 32) GY[t] = 0.f;  // padded channels stay zero
  for (int t = lane; t < SK_ROWS * AW; t += 32) AA[t] = 0.f;  // padded columns stay zero
  for (int t = threadIdx.x; t < CO * AW + CO; t += SK_THREADS) R[t] = 0.f;
  __syncwarp();

  const int64_t cta_begin = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t cta_end = (cta_begin + rows_per_cta < n) ? (cta_begin + rows_per_cta) : n;

  constexpr int GV = SK_ROWS * CO / 4 / 32;  // float4 per lane of a gy chunk (FAST)
  constexpr int AV = SK_ROWS * AW / 4 / 32;  // float4 per lane of an activation chunk (FAST)
  constexpr int RV = AW / 4;                 // float4 per activation row
  float4 gbuf[FAST ? GV : 1], abuf[FAST ? AV : 1];
  (void)gbuf;
  (void)abuf;

  auto fetch = [&](int64_t r0) {  // FAST: issue every load of the chunk, keep the data in registers
    if constexpr (FAST) {
      const int rows = (int)((cta_end - r0 < SK_ROWS) ? (cta_end - r0) : SK_ROWS);
      const float4* g4 = reinterpret_cast<const float4*>(gy + r0 * CO);
#pragma unroll
      for (int j = 0; j < GV; ++j) {
        const int t = lane + 32 * j;
        gbuf[j] = (t / (CO / 4) < rows) ? __ldg(g4 + t) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int j = 0; j < AV; ++j) {
        const int t = lane + 32 * j;
        const int row = t / RV, col = (t % RV) * 4;
        abuf[j] = (row < rows && col < ktot) ? cat_load4(A, r0 + row, col) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  };
  auto commit = [&](int64_t r0) {  // registers -> the warp's shared-memory slab (generic path: global -> smem)
    if constexpr (FAST) {
#pragma unroll
      for (int j = 0; j < GV; ++j) reinterpret_cast<float4*>(GY)[lane + 32 * j] = gbuf[j];
#pragma unroll
      for (int j = 0; j < AV; ++j) reinterpret_cast<float4*>(AA)[lane + 32 * j] = abuf[j];
    } else {
      const int rows = (int)((cta_end - r0 < SK_ROWS) ? (cta_end - r0) : SK_ROWS);
#pragma unroll 4
      for (int t = lane; t < SK_ROWS * cout; t += 32) {
        const int row = t / cout, c = t - row * cout;
        GY[row * CO + c] = (row < rows) ? __ldg(gy + r0 * cout + t) : 0.f;
      }
#pragma unroll 4
      for (int t = lane; t < SK_ROWS * AW; t += 32) {
        const int row = t / AW, col = t % AW;
        if (col < ktot) AA[t] = (row < rows) ? cat_load1(A, r0 + row, col) : 0.f;
      }
    }
  };

  int64_t r0 = cta_begin + warp * SK_ROWS;
  if (r0 < cta_end) fetch(r0);
  for (; r0 < cta_end; r0 += NW * SK_ROWS) {
    commit(r0);
    __syncwarp();
    const int64_t rn = r0 + NW * SK_ROWS;
    if (rn < cta_end) fetch(rn);  // overlaps with the multiply below
#pragma unroll 4
    for (int row = 0; row < SK_ROWS; ++row) {
      const float a0 = AA[row * AW + lane];
      const float a1 = TWO ? AA[row * AW + 32 + lane] : 0.f;
      if (lane < CO) bs0 += GY[row * CO + lane];
      if (CO > 32) bs1 += GY[row * CO + 32 + lane];
#pragma unroll
      for (int c4 = 0; c4 < CO / 4; ++c4) {
        const float4 g = *reinterpret_cast<const float4*>(GY + row * CO + c4 * 4);
        if constexpr (CO * (TWO ? 2 : 1) <= 64) {  // FFMA2: the activation in the broadcast slot
          ffma2_bc(a0, g.x, g.y, acc0[c4 * 4 + 0], acc0[c4 * 4 + 1]);
          ffma2_bc(a0, g.z, g.w, acc0[c4 * 4 + 2], acc0[c4 * 4 + 3]);
          if (TWO) {
            ffma2_bc(a1, g.x, g.y, acc1[c4 * 4 + 0], acc1[c4 * 4 + 1]);
            ffma2_bc(a1, g.z, g.w, acc1[c4 * 4 + 2], acc1[c4 * 4 + 3]);
          }
        } else {  // 128 accumulators: the even-aligned register pairs of the packed form would spill
          acc0[c4 * 4 + 0] = fmaf(g.x, a0, acc0[c4 * 4 + 0]);
          acc0[c4 * 4 + 1] = fmaf(g.y, a0, acc0[c4 * 4 + 1]);
          acc0[c4 * 4 + 2] = fmaf(g.z, a0, acc0[c4 * 4 + 2]);
          acc0[c4 * 4 + 3] = fmaf(g.w, a0, acc0[c4 * 4 + 3]);
          if (TWO) {
            acc1[c4 * 4 + 0] = fmaf(g.x, a1, acc1[c4 * 4 + 0]);
            acc1[c4 * 4 + 1] = fmaf(g.y, a1, acc1[c4 * 4 + 1]);
            acc1[c4 * 4 + 2] = fmaf(g.z, a1, acc1[c4 * 4 + 2]);
            acc1[c4 * 4 + 3] = fmaf(g.w, a1, acc1[c4 * 4 + 3]);
          }
        }
      }
    }
    __syncwarp();
  }
  __syncthreads();
#pragma unroll
  for (int c = 0; c < CO; ++c) {
    atomicAdd(&R[c * AW + lane], acc0[c]);
    if (TWO) atomicAdd(&R[c * AW + 32 + lane], acc1[c]);
  }
  if (lane < CO) atomicAdd(&R[CO * AW + lane], bs0);
  if (CO > 32) atomicAdd(&R[CO * AW + 32 + lane], bs1);
  __syncthreads();
  for (int t = threadIdx.x; t < CO * AW; t += SK_THREADS) {
    const int c = t / AW, col = t % AW;
    if (c < cout && col < ktot) atomicAdd(gw + (int64_t)c * ktot + col, R[t]);
  }
  if (gb)
    for (int c = threadIdx.x; c < cout; c += SK_THREADS) atomicAdd(gb + c, R[CO * AW + c]);
}

template <int CO, int AW>
static int launch_tn_skinny(const float* gy, int cout, const CatRows& A, float* gw, float* gb, int64_t n, cudaStream_t st) {
  const size_t smem = sizeof(float) * ((SK_THREADS / 32) * (SK_ROWS * CO + SK_ROWS * AW) + CO * AW + CO);
  const bool fast = (cout == CO) && aligned16(gy) && A.vec;
  auto kern = fast ? tn_skinny_kernel<CO, AW, true> : tn_skinny_kernel<CO, AW, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "tn_skinny smem attribute");
  int64_t ctas = (int64_t)num_sms() * 4;
  const int64_t max_ctas = ceil_div(n, (SK_THREADS / 32) * SK_ROWS);
  if (ctas > max_ctas) ctas = max_ctas;
  int64_t rows_per_cta = ceil_div(n, ctas);
  rows_per_cta = ceil_div(rows_per_cta, (SK_THREADS / 32) * SK_ROWS) * (SK_THREADS / 32) * SK_ROWS;
  ctas = ceil_div(n, rows_per_cta);
  kern<<<(unsigned)ctas, SK_THREADS, smem, st>>>(gy, cout, A, gw, gb, n, rows_per_cta);
  B200_CHECK_LAUNCH("tn_skinny_kernel");
  return B200_OK;
}

// generic dispatcher of gw[cout, c1+c2] += gy^T [a1|a2], gb += colsum(gy)
static bool tn_uses_tensor_cores(const float* gy, int cout, const CatRows& A, const float* gw, int64_t n) {
  return cout >= 64 && A.c1 + A.c2 >= 64 && n >= 512 && cout % 4 == 0 && A.vec && aligned16(gy) && aligned16(gw) &&
         tc_path_enabled(4);
}

static int launch_tn(const float* gy, int cout, const CatRows& A, float* gw, float* gb, int64_t n, float* ws,
                     size_t ws_bytes, cudaStream_t st) {
  const int ktot = A.c1 + A.c2;
  const int ncols = ktot + (gb ? 1 : 0);
  // >= 64 x 64 outputs: 5th-generation tensor cores (3xTF32), see tc_gemm.cu
  if (tn_uses_tensor_cores(gy, cout, A, gw, n))
    return launch_tc_tn(gy, cout, A.a1, A.ld1, A.c1, A.a2, A.ld2, A.c2, gw, gb, n, ws, ws_bytes, st);
  {
    // Narrow layers of levels 0-1.  The warp-streaming FMA kernel below reaches 1.3-1.9 TB/s on its vectorised path
    // (cout in {16, 32, 64}, float4-addressable rows); odd shapes (mlp1's 32 -> 4, fc0's 9 -> 32) fall to its scalar
    // path at 0.4-0.8 TB/s: those go to the tensor cores (tc_skinny.cu, measured 33-39 us against 49-85 us).
    const bool fma_fast = (cout == 16 || cout == 32 || cout == 64) && aligned16(gy) && A.vec;
    if (!fma_fast && tc_skinny_tn_ok(cout, ktot, gb != nullptr, n))
      return launch_tc_skinny_tn(gy, cout, A.a1, A.ld1, A.c1, A.a2, A.ld2, A.c2, gw, gb, n, st);
  }
  if (cout <= 64 && ktot <= 64 && n >= 4096) {
    const bool wide = ktot > 32;
    if (cout <= 16) return wide ? launch_tn_skinny<16, 64>(gy, cout, A, gw, gb, n, st) : launch_tn_skinny<16, 32>(gy, cout, A, gw, gb, n, st);
    if (cout <= 32) return wide ? launch_tn_skinny<32, 64>(gy, cout, A, gw, gb, n, st) : launch_tn_skinny<32, 32>(gy, cout, A, gw, gb, n, st);
    return wide ? launch_tn_skinny<64, 64>(gy, cout, A, gw, gb, n, st) : launch_tn_skinny<64, 32>(gy, cout, A, gw, gb, n, st);
  }
  const bool gvec = (reinterpret_cast<uintptr_t>(gy) & 15) == 0 && (cout % 4 == 0);
  const bool big = cout >= 128 && ncols >= 128;
  const int bm = big ? 128 : 64;
  const int64_t tiles = ceil_div(cout, bm) * ceil_div(ncols, bm);
  int64_t splits = ceil_div((int64_t)num_sms() * 2, tiles);  // few CTAs: every CTA ends with cout*ncols global atomics
  const int64_t max_splits = ceil_div(n, 128);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if (splits > 65535) splits = 65535;
  int64_t rows_per_split = ceil_div(n, splits);
  rows_per_split = ceil_div(rows_per_split, GEMM_BK) * GEMM_BK;
  splits = ceil_div(n, rows_per_split);
  dim3 grid((unsigned)ceil_div(cout, bm), (unsigned)ceil_div(ncols, bm), (unsigned)splits);
  if (big)
    linear_bwd_weight_kernel<128, 128><<<grid, GEMM_THREADS, 0, st>>>(gy, gvec, A, gw, gb, n, cout, rows_per_split);
  else
    linear_bwd_weight_kernel<64, 64><<<grid, GEMM_THREADS, 0, st>>>(gy, gvec, A, gw, gb, n, cout, rows_per_split);
  B200_CHECK_LAUNCH("linear_bwd_weight_kernel");
  return B200_OK;
}

// ------------------------------------------------------------------ BatchNorm finalisation
__global__ void bn_finalize_kernel(const double* __restrict__ colstats, int num_partials, int64_t count,
                                   const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, int64_t* __restrict__ num_batches_tracked,
                                   float momentum, float eps, float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out,
                                   float* __restrict__ invstd_out, int c) {
  if (blockIdx.x == 0 && threadIdx.x == 0 && colstats && num_batches_tracked) *num_batches_tracked += 1;
  // one CTA per channel: 128 threads stride over the partial rows (up to 1600 of them at level 0), then reduce
  __shared__ double sh1[4], sh2[4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int ch = blockIdx.x; ch < c; ch += gridDim.x) {
    double mean, var;
    if (colstats) {
      double s1 = 0.0, s2 = 0.0;
      for (int p = threadIdx.x; p < num_partials; p += blockDim.x) {
        s1 += colstats[(int64_t)p * 2 * c + ch];
        s2 += colstats[(int64_t)p * 2 * c + c + ch];
      }
      s1 = warp_sum(s1);
      s2 = warp_sum(s2);
      __syncthreads();  // sh1/sh2 of the previous channel have been consumed
      if (lane == 0) sh1[warp] = s1, sh2[warp] = s2;
      __syncthreads();
      if (threadIdx.x != 0) continue;
      s1 = sh1[0] + sh1[1] + sh1[2] + sh1[3];
      s2 = sh2[0] + sh2[1] + sh2[2] + sh2[3];
      mean = s1 / (double)count;
      var = s2 / (double)count - mean * mean;
      if (var < 0.0) var = 0.0;
      if (running_mean) {
        const double unbiased = (count > 1) ? var * (double)count / (double)(count - 1) : var;
        running_mean[ch] = (float)((1.0 - (double)momentum) * (double)running_mean[ch] + (double)momentum * mean);
        running_var[ch] = (float)((1.0 - (double)momentum) * (double)running_var[ch] + (double)momentum * unbiased);
      }
    } else {
      if (threadIdx.x != 0) continue;
      mean = (double)running_mean[ch];
      var = (double)running_var[ch];
    }
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float sc = gamma[ch] * invstd;
    scale[ch] = sc;
    shift[ch] = beta[ch] - (float)mean * sc;
    if (mean_out) mean_out[ch] = (float)mean;
    if (invstd_out) invstd_out[ch] = invstd;
  }
}

// ------------------------------------------------------------------ out = act(y1*s1 + t1 [+ y2*s2 + t2])
template <int V>
__global__ void __launch_bounds__(256)
affine_act_fwd_kernel(const float* __restrict__ y1, const float* __restrict__ s1, const float* __restrict__ t1,
                      const float* __restrict__ y2, const float* __restrict__ s2, const float* __restrict__ t2,
                      float slope, float* __restrict__ out, int64_t total, int c) {
  // per-channel (scale, shift) of both branches staged once per CTA: the element loop then reads them with one LDS per
  // branch and float4 instead of 2-4 global loads per ELEMENT (the kernel was L1-instruction-bound for c >= 128)
  extern __shared__ __align__(16) float coef[];  // [s1 | t1 | s2 | t2][c]
  for (int ch = threadIdx.x; ch < c; ch += 256) {
    coef[ch] = __ldg(s1 + ch);
    coef[c + ch] = __ldg(t1 + ch);
    coef[2 * c + ch] = y2 ? __ldg(s2 + ch) : 0.f;
    coef[3 * c + ch] = y2 ? __ldg(t2 + ch) : 0.f;
  }
  __syncthreads();
  for (int64_t idx = ((int64_t)blockIdx.x * 256 + threadIdx.x) * V; idx < total; idx += (int64_t)gridDim.x * 256 * V) {
    const int ch = (int)(idx % c);
    float a[V], b[V], o[V], cs1[V], ct1[V], cs2[V], ct2[V];
    if constexpr (V == 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(y1 + idx));
      a[0] = v.x, a[1] = v.y, a[2] = v.z, a[3] = v.w;
      const float4 p = *reinterpret_cast<const float4*>(coef + ch), q = *reinterpret_cast<const float4*>(coef + c + ch);
      cs1[0] = p.x, cs1[1] = p.y, cs1[2] = p.z, cs1[3] = p.w;
      ct1[0] = q.x, ct1[1] = q.y, ct1[2] = q.z, ct1[3] = q.w;
      if (y2) {
        const float4 u = __ldg(reinterpret_cast<const float4*>(y2 + idx));
        b[0] = u.x, b[1] = u.y, b[2] = u.z, b[3] = u.w;
        const float4 p2 = *reinterpret_cast<const float4*>(coef + 2 * c + ch), q2 = *reinterpret_cast<const float4*>(coef + 3 * c + ch);
        cs2[0] = p2.x, cs2[1] = p2.y, cs2[2] = p2.z, cs2[3] = p2.w;
        ct2[0] = q2.x, ct2[1] = q2.y, ct2[2] = q2.z, ct2[3] = q2.w;
      }
    } else {
      a[0] = __ldg(y1 + idx);
      cs1[0] = coef[ch], ct1[0] = coef[c + ch];
      if (y2) b[0] = __ldg(y2 + idx), cs2[0] = coef[2 * c + ch], ct2[0] = coef[3 * c + ch];
    }
#pragma unroll
    for (int u = 0; u < V; ++u) {
      float v = fmaf(a[u], cs1[u], ct1[u]);
      if (y2) v += fmaf(b[u], cs2[u], ct2[u]);
      o[u] = lrelu(v, slope);
    }
    if constexpr (V == 4)
      *reinterpret_cast<float4*>(out + idx) = make_float4(o[0], o[1], o[2], o[3]);
    else
      out[idx] = o[0];
  }
}

// ------------------------------------------------------------------ backward reductions
// red[0:c] = sum_i g, red[c:2c] = sum_i g * xhat,  g = grad_out * act'(out)
constexpr int RED_THREADS = 256;
__global__ void __launch_bounds__(RED_THREADS)
affine_act_bwd_reduce_kernel(const float* __restrict__ go, const float* __restrict__ out, float slope,
                             const float* __restrict__ y1, const float* __restrict__ mean1,
                             const float* __restrict__ invstd1, double* __restrict__ red1,
                             const float* __restrict__ y2, const float* __restrict__ mean2,
                             const float* __restrict__ invstd2, double* __restrict__ red2, int64_t n, int c,
                             int lanes /* pow2 >= min(c, 256) */) {
  extern __shared__ double sred[];  // [4][lanes]
  const int tid = threadIdx.x;
  const int lane = tid % lanes, rsub = tid / lanes, rstep = RED_THREADS / lanes;
  for (int cbase = 0; cbase < c; cbase += lanes) {
    const int ch = cbase + lane;
    float sg = 0.f, sgx1 = 0.f, sgx2 = 0.f;
    if (ch < c) {
      const float m1 = __ldg(mean1 + ch), is1 = __ldg(invstd1 + ch);
      const float m2 = y2 ? __ldg(mean2 + ch) : 0.f, is2 = y2 ? __ldg(invstd2 + ch) : 0.f;
      for (int64_t i = (int64_t)blockIdx.x * rstep + rsub; i < n; i += (int64_t)gridDim.x * rstep) {
        const int64_t off = i * c + ch;
        float g = __ldg(go + off);
        if (slope != 1.f) g *= (__ldg(out + off) > 0.f) ? 1.f : slope;
        sg += g;
        sgx1 = fmaf(g, (__ldg(y1 + off) - m1) * is1, sgx1);
        if (y2) sgx2 = fmaf(g, (__ldg(y2 + off) - m2) * is2, sgx2);
      }
    }
    for (int t = tid; t < 4 * lanes; t += RED_THREADS) sred[t] = 0.0;
    __syncthreads();
    if (ch < c) {
      atomicAdd(&sred[0 * lanes + lane], (double)sg);
      atomicAdd(&sred[1 * lanes + lane], (double)sgx1);
      if (y2) atomicAdd(&sred[2 * lanes + lane], (double)sgx2);
    }
    __syncthreads();
    if (tid < lanes && cbase + tid < c) {
      atomicAdd(red1 + cbase + tid, sred[0 * lanes + tid]);
      atomicAdd(red1 + c + cbase + tid, sred[1 * lanes + tid]);
      if (y2) {
        atomicAdd(red2 + cbase + tid, sred[0 * lanes + tid]);
        atomicAdd(red2 + c + cbase + tid, sred[2 * lanes + tid]);
      }
    }
    __syncthreads();
  }
}

// float4 version (c % 4 == 0): a thread owns 4 channels of every (rows-per-pass)-th row -- 4x fewer load instructions
// and 4x more bytes in flight per thread than the scalar kernel; the CTA covers c/4 lanes x 256/(c/4) rows per pass.
__device__ __forceinline__ void
bwd_reduce_vec4_body(const float* __restrict__ go, const float* __restrict__ out, float slope,
                     const float* __restrict__ y1, const float* __restrict__ mean1,
                     const float* __restrict__ invstd1, double* __restrict__ red1,
                     const float* __restrict__ y2, const float* __restrict__ mean2,
                     const float* __restrict__ invstd2, double* __restrict__ red2, int64_t n, int c,
                     int lanes /* pow2 >= min(c/4, 256) */, int bid, int nblk, float (*part)[RED_THREADS]) {
  const int tid = threadIdx.x;
  const int lane = tid % lanes, rsub = tid / lanes, rstep = RED_THREADS / lanes;
  const int c4 = c >> 2;
  for (int cbase = 0; cbase < c4; cbase += lanes) {
    const int q = cbase + lane;  // float4 column
    float sg[4] = {0.f, 0.f, 0.f, 0.f}, sx1[4] = {0.f, 0.f, 0.f, 0.f}, sx2[4] = {0.f, 0.f, 0.f, 0.f};
    if (q < c4) {
      const float4 m1 = __ldg(reinterpret_cast<const float4*>(mean1) + q), is1 = __ldg(reinterpret_cast<const float4*>(invstd1) + q);
      float4 m2 = make_float4(0.f, 0.f, 0.f, 0.f), is2 = m2;
      if (y2) m2 = __ldg(reinterpret_cast<const float4*>(mean2) + q), is2 = __ldg(reinterpret_cast<const float4*>(invstd2) + q);
      const float m1a[4] = {m1.x, m1.y, m1.z, m1.w}, i1a[4] = {is1.x, is1.y, is1.z, is1.w};
      const float m2a[4] = {m2.x, m2.y, m2.z, m2.w}, i2a[4] = {is2.x, is2.y, is2.z, is2.w};
      for (int64_t i = (int64_t)bid * rstep + rsub; i < n; i += (int64_t)nblk * rstep) {
        const int64_t off = i * c4 + q;
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(go) + off);
        const float4 a4 = __ldg(reinterpret_cast<const float4*>(y1) + off);
        float g[4] = {g4.x, g4.y, g4.z, g4.w};
        const float a[4] = {a4.x, a4.y, a4.z, a4.w};
        if (slope != 1.f) {
          const float4 o4 = __ldg(reinterpret_cast<const float4*>(out) + off);
          const float o[4] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) g[u] *= (o[u] > 0.f) ? 1.f : slope;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          sg[u] += g[u];
          sx1[u] = fmaf(g[u], (a[u] - m1a[u]) * i1a[u], sx1[u]);
        }
        if (y2) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(y2) + off);
          const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) sx2[u] = fmaf(g[u], (bb[u] - m2a[u]) * i2a[u], sx2[u]);
        }
      }
    }
    // per-thread partials -> shared memory (no atomics: CAS-emulated fp64 shared atomics with 32 row groups per address
    // cost more than the loads), then one thread per output sums its row groups in fp64
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      part[0 + u][tid] = sg[u];
      part[4 + u][tid] = sx1[u];
      part[8 + u][tid] = sx2[u];
    }
    __syncthreads();
    for (int t = tid; t < 12 * lanes; t += RED_THREADS) {
      const int kind = t / (4 * lanes), rem = t % (4 * lanes), ln = rem >> 2, u = rem & 3;
      const int ch = 4 * (cbase + ln) + u;
      if (ch >= c || (kind == 2 && !y2)) continue;
      double acc = 0.0;
      for (int r = 0; r < rstep; ++r) acc += (double)part[kind * 4 + u][r * lanes + ln];
      if (kind == 0) {
        atomicAdd(red1 + ch, acc);
        if (y2) atomicAdd(red2 + ch, acc);
      } else if (kind == 1) {
        atomicAdd(red1 + c + ch, acc);
      } else {
        atomicAdd(red2 + c + ch, acc);
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(RED_THREADS)
affine_act_bwd_reduce_vec4_kernel(const float* __restrict__ go, const float* __restrict__ out, float slope,
                                  const float* __restrict__ y1, const float* __restrict__ mean1,
                                  const float* __restrict__ invstd1, double* __restrict__ red1,
                                  const float* __restrict__ y2, const float* __restrict__ mean2,
                                  const float* __restrict__ invstd2, double* __restrict__ red2, int64_t n, int c, int lanes) {
  __shared__ float part[12][RED_THREADS];
  bwd_reduce_vec4_body(go, out, slope, y1, mean1, invstd1, red1, y2, mean2, invstd2, red2, n, c, lanes, (int)blockIdx.x,
                       (int)gridDim.x, part);
}

struct BnBranch {
  const float* y;
  const float* gamma;
  const float* mean;
  const float* invstd;
  const double* red;   // nullptr => plain affine: grad_y = g * scale
  const float* scale;
  float* grad_y;
  float* grad_gamma;
  float* grad_beta;
};

template <int V>
__device__ __forceinline__ void
bwd_apply_body(const float* __restrict__ go, const float* __restrict__ out, float slope, const BnBranch& b1,
               const BnBranch& b2, int64_t n, int c, int bid, int nblk, float* __restrict__ coef) {
  const int64_t total = n * c;
  const double inv_n = 1.0 / (double)n;
  // parameter gradients (train-mode BatchNorm): accumulated once, by the first CTA, into the caller's buffers
  // (the parameters' .grad, or zero-filled temporaries)
  if (bid == 0) {
    for (int ch = threadIdx.x; ch < c; ch += 256) {
      if (b1.red && b1.grad_gamma) {
        b1.grad_gamma[ch] += (float)__ldcg(b1.red + c + ch);
        b1.grad_beta[ch] += (float)__ldcg(b1.red + ch);
      }
      if (b2.y && b2.red && b2.grad_gamma) {
        b2.grad_gamma[ch] += (float)__ldcg(b2.red + c + ch);
        b2.grad_beta[ch] += (float)__ldcg(b2.red + ch);
      }
    }
  }
  // grad_y = k1 * (g - mg) - k4 * (y - mean) per channel, with k1 = gamma * invstd, mg = red[0]/n, k4 = k1 * invstd *
  // red[1]/n (train) or k1 = scale, mg = k4 = 0 (eval / plain affine): the four coefficients of both branches are
  // staged once per CTA (the element loop used 3 global + 2 fp64 loads and 2 fp64 multiplies per ELEMENT)
  // coef (shared memory of the caller): [branch][k1 | mg | k4 | mean][c]
  for (int ch = threadIdx.x; ch < c; ch += 256) {
#pragma unroll
    for (int br = 0; br < 2; ++br) {
      const BnBranch& bb = br == 0 ? b1 : b2;
      float k1 = 0.f, mg = 0.f, k4 = 0.f, mean = 0.f;
      if (br == 0 || bb.y) {
        if (bb.red) {
          const float is = __ldg(bb.invstd + ch);
          k1 = __ldg(bb.gamma + ch) * is;
          mg = (float)(__ldcg(bb.red + ch) * inv_n);
          k4 = k1 * is * (float)(__ldcg(bb.red + c + ch) * inv_n);
          mean = __ldg(bb.mean + ch);
        } else {
          k1 = __ldg(bb.scale + ch);
        }
      }
      float* t = coef + br * 4 * c;
      t[ch] = k1, t[c + ch] = mg, t[2 * c + ch] = k4, t[3 * c + ch] = mean;
    }
  }
  __syncthreads();
  const bool need_y1 = b1.red != nullptr, need_y2 = b2.y && b2.red;
  for (int64_t idx = ((int64_t)bid * 256 + threadIdx.x) * V; idx < total; idx += (int64_t)nblk * 256 * V) {
    const int ch0 = (int)(idx % c);
    float g[V], o[V], y1v[V], y2v[V];
#pragma unroll
    for (int u = 0; u < V; ++u) y1v[u] = 0.f, y2v[u] = 0.f, o[u] = 1.f;
    if constexpr (V == 4) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(go + idx));
      g[0] = a.x, g[1] = a.y, g[2] = a.z, g[3] = a.w;
      if (slope != 1.f) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(out + idx));
        o[0] = b.x, o[1] = b.y, o[2] = b.z, o[3] = b.w;
      }
      if (need_y1) {
        const float4 d = __ldg(reinterpret_cast<const float4*>(b1.y + idx));
        y1v[0] = d.x, y1v[1] = d.y, y1v[2] = d.z, y1v[3] = d.w;
      }
      if (need_y2) {
        const float4 d = __ldg(reinterpret_cast<const float4*>(b2.y + idx));
        y2v[0] = d.x, y2v[1] = d.y, y2v[2] = d.z, y2v[3] = d.w;
      }
    } else {
      g[0] = __ldg(go + idx);
      if (slope != 1.f) o[0] = __ldg(out + idx);
      if (need_y1) y1v[0] = __ldg(b1.y + idx);
      if (need_y2) y2v[0] = __ldg(b2.y + idx);
    }
    float k[2][4][V];
#pragma unroll
    for (int br = 0; br < 2; ++br) {
      if (br == 1 && !b2.y) break;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float* t = coef + (br * 4 + j) * c + ch0;
        if constexpr (V == 4) {
          const float4 q = *reinterpret_cast<const float4*>(t);
          k[br][j][0] = q.x, k[br][j][1] = q.y, k[br][j][2] = q.z, k[br][j][3] = q.w;
        } else {
          k[br][j][0] = t[0];
        }
      }
    }
    float r1[V], r2[V];
#pragma unroll
    for (int u = 0; u < V; ++u) {
      float gg = g[u];
      if (slope != 1.f) gg *= (o[u] > 0.f) ? 1.f : slope;
      r1[u] = k[0][0][u] * (gg - k[0][1][u]) - k[0][2][u] * (y1v[u] - k[0][3][u]);
      if (b2.y) r2[u] = k[1][0][u] * (gg - k[1][1][u]) - k[1][2][u] * (y2v[u] - k[1][3][u]);
    }
    if constexpr (V == 4) {
      *reinterpret_cast<float4*>(b1.grad_y + idx) = make_float4(r1[0], r1[1], r1[2], r1[3]);
      if (b2.y) *reinterpret_cast<float4*>(b2.grad_y + idx) = make_float4(r2[0], r2[1], r2[2], r2[3]);
    } else {
      b1.grad_y[idx] = r1[0];
      if (b2.y) b2.grad_y[idx] = r2[0];
    }
  }
}

template <int V>
__global__ void __launch_bounds__(256)
affine_act_bwd_apply_kernel(const float* __restrict__ go, const float* __restrict__ out, float slope, BnBranch b1,
                            BnBranch b2, int64_t n, int c) {
  extern __shared__ __align__(16) float coef_smem[];
  bwd_apply_body<V>(go, out, slope, b1, b2, n, c, (int)blockIdx.x, (int)gridDim.x, coef_smem);
}

// Reduce + apply of a train-mode BatchNorm backward in ONE launch (small levels: two latency-bound kernels and the gap
// between them cost more than the bytes).  MEASURED SLOWER (round 2: 15 launches x 16.8 us against 15 x (8.0 + 5.5) us of
// the two kernels; the co-residency rule below caps the grid at #SMs / 2 CTAs, too few for either phase), so the option
// "bn_backward_fused" is off by default and the two-kernel path runs; kept as an A/B switch and as a tested example of a
// safe software grid barrier.  The grid is at most half the SMs, two CTAs of this kernel fit an SM, and no
// other kernel of the library spins on a condition: all CTAs become co-resident, so the software grid barrier between
// the two phases (a counter the caller zeroed; acquire spin, bounded: a violated assumption traps instead of hanging)
// is safe.  The sums travel through the same fp64 `red` buffers as in the two-kernel path.
__global__ void __launch_bounds__(256, 2)
affine_act_bwd_fused_kernel(const float* __restrict__ go, const float* __restrict__ out, float slope, BnBranch b1, BnBranch b2,
                            double* __restrict__ red1, double* __restrict__ red2, unsigned int* __restrict__ barrier,
                            int64_t n, int c, int lanes) {
  __shared__ float part[12][RED_THREADS];
  extern __shared__ __align__(16) float coef_smem[];
  bwd_reduce_vec4_body(go, out, slope, b1.y, b1.mean, b1.invstd, red1, b2.y, b2.mean, b2.invstd, red2, n, c, lanes,
                       (int)blockIdx.x, (int)gridDim.x, part);
  __threadfence();  // this CTA's atomics are performed before its arrival is visible
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(barrier, 1u);
    unsigned int seen = 0;
    for (unsigned int spin = 0; spin < (1u << 22); ++spin) {  // ~ seconds; the real wait is microseconds
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(barrier) : "memory");
      if (seen >= gridDim.x) break;
    }
    if (seen < gridDim.x) __trap();
  }
  __syncthreads();
  bwd_apply_body<4>(go, out, slope, b1, b2, n, c, (int)blockIdx.x, (int)gridDim.x, coef_smem);
}

static int elementwise_grid(int64_t work_items) {
  int64_t blocks = ceil_div(work_items, 256);
  const int64_t cap = (int64_t)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

// (over the E edge rows of an LFA level the split-K plan bounds the rows one TMEM accumulator sums: tc_gemm.cu)
int accumulate_at_b(const float* a, int ca, const float* b, int cb, float* out, int64_t n, float* ws, size_t ws_bytes,
                    cudaStream_t st) {
  const CatRows B = make_cat(b, cb, cb, nullptr, 0, 0);
  return launch_tn(a, ca, B, out, nullptr, n, ws, ws_bytes, st);
}
size_t accumulate_at_b_workspace_bytes(int ca, int cb, int64_t n) { return tc_tn_workspace_bytes(ca, cb, n); }

}  // namespace b200

using namespace b200;

extern "C" int b200_linear_fwd(const float* a1, int64_t ld1, int32_t c1, const float* a2, int64_t ld2, int32_t c2,
                               const float* w, const float* bias, float* y, int64_t n, int32_t cout,
                               double* colstats, void* stream) {
  B200_REQUIRE(a1 && w && y, B200_E_INVALID, "b200_linear_fwd: null pointer");
  B200_REQUIRE(c1 > 0 && c2 >= 0 && cout > 0 && (c2 == 0 || a2), B200_E_INVALID, "b200_linear_fwd: bad sizes");
  B200_REQUIRE(ld1 >= c1 && (c2 == 0 || ld2 >= c2), B200_E_INVALID, "b200_linear_fwd: row stride < width");
  if (n <= 0) return B200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // 16/32/64-channel layers of levels 0-1: TMA-fed persistent row streaming (tma_rows.cu)
  if (tma_rows_enabled(1) && tma_rows_nn_ok(n, a1, ld1, c1, a2, ld2, c2, cout, y, cout, cout, nullptr, 0))
    return launch_tma_rows_nn(a1, ld1, c1, a2, ld2, c2, w, c1 + c2, true, bias, y, cout, cout, nullptr, 0, cout, n, colstats,
                              colstats ? (int)b200_linear_fwd_num_stat_partials(n, c1, c2, cout) : 0, st);
  if (tc_nt_shape_ok(n, c1, c2, cout) && tc_path_enabled(1))  // tcgen05 (3xTF32): every layer with >= 64 input and output channels
    return launch_tc_nt(a1, ld1, c1, a2, ld2, c2, w, cout, bias, y, cout, cout, nullptr, 0, colstats, n, st);
  if (linear_rows_ok(n, c1 + c2, cout))  // narrow layers of levels 0-1: one thread per row (linear_rows.cu)
    return launch_linear_rows(a1, ld1, c1, a2, ld2, c2, w, c1 + c2, true, bias, y, cout, cout, nullptr, 0, 0, n, colstats, st);
  const CatRows A = make_cat(a1, ld1, c1, a2, ld2, c2);
  const bool wvec = aligned16(w) && ((c1 + c2) % 4 == 0);
  if (cout <= 32) {
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)ceil_div(cout, 32));
    linear_fwd_kernel<128, 32><<<grid, GEMM_THREADS, 0, st>>>(A, w, wvec, bias, y, n, cout, colstats);
  } else if (cout >= 128 && c1 + c2 >= 64 && ceil_div(n, 128) * ceil_div(cout, 128) >= num_sms()) {
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)ceil_div(cout, 128));
    linear_fwd_kernel<128, 128><<<grid, GEMM_THREADS, 0, st>>>(A, w, wvec, bias, y, n, cout, colstats);
  } else {
    dim3 grid((unsigned)ceil_div(n, 64), (unsigned)ceil_div(cout, 64));
    linear_fwd_kernel<64, 64><<<grid, GEMM_THREADS, 0, st>>>(A, w, wvec, bias, y, n, cout, colstats);
  }
  B200_CHECK_LAUNCH("linear_fwd_kernel");
  return B200_OK;
}

// Input gradients go to the tensor cores below level 1 only: on >= 51 200 rows the layers are HBM-bound and the FMA
// kernel (no transpose pass, no idle TMEM lanes for narrow outputs) is as fast or faster (profiles/, DESIGN.md section 7).
static bool bwd_input_uses_tc(int64_t n, int ktot, int cout) {
  return n >= 1024 && n <= 32768 && tc_nt_shape_ok(n, cout, 0, ktot) && tc_path_enabled(2);
}

extern "C" int64_t b200_linear_bwd_input_workspace_bytes(int64_t n, int32_t c1, int32_t c2, int32_t cout) {
  return bwd_input_uses_tc(n, c1 + c2, cout) ? (int64_t)(c1 + c2) * cout * (int64_t)sizeof(float) : 0;
}

extern "C" int b200_linear_bwd_input(const float* grad_y, const float* w, float* ga1, int64_t ldg1, int32_t c1,
                                     float* ga2, int64_t ldg2, int32_t c2, void* workspace, int64_t workspace_bytes,
                                     int64_t n, int32_t cout, void* stream) {
  B200_REQUIRE(grad_y && w, B200_E_INVALID, "b200_linear_bwd_input: null pointer");
  B200_REQUIRE(c1 > 0 && c2 >= 0 && cout > 0, B200_E_INVALID, "b200_linear_bwd_input: bad sizes");
  if (n <= 0 || (!ga1 && !ga2)) return B200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ktot = c1 + c2;
  if (tma_rows_enabled(2) &&
      tma_rows_nn_ok(n, grad_y, cout, cout, nullptr, 0, 0, ktot, ga1, ldg1, c1, ga2, ldg2))
    return launch_tma_rows_nn(grad_y, cout, cout, nullptr, 0, 0, w, ktot, false, nullptr, ga1, ldg1, c1, ga2, ldg2, ktot, n,
                              nullptr, 0, st);
  if (workspace && workspace_bytes >= (int64_t)ktot * cout * (int64_t)sizeof(float) && aligned16(workspace) &&
      bwd_input_uses_tc(n, ktot, cout)) {
    // tcgen05: grad_a[i][k] = sum_m grad_y[i][m] * W^T[k][m]; W^T goes to the workspace first (<= 1.5 MB)
    float* wt = static_cast<float*>(workspace);
    int rc = launch_transpose(w, wt, cout, ktot, st);
    if (rc != B200_OK) return rc;
    return launch_tc_nt(grad_y, cout, cout, nullptr, 0, 0, wt, ktot, nullptr, ga1, ldg1, c1, ga2, ldg2, nullptr, n, st);
  }
  if (linear_rows_ok(n, cout, ktot))  // narrow layers of levels 0-1: the row-streaming kernel with W read as [cout][ktot]
    return launch_linear_rows(grad_y, cout, cout, nullptr, 0, 0, w, ktot, false, nullptr, ga1, ldg1, c1, ga2, ldg2, c2, n,
                              nullptr, st);
  const bool gvec = aligned16(grad_y) && (cout % 4 == 0);
  const bool wvec = aligned16(w) && (ktot % 4 == 0);
  if (ktot <= 32) {
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)ceil_div(ktot, 32));
    linear_bwd_input_kernel<128, 32><<<grid, GEMM_THREADS, 0, st>>>(grad_y, gvec, w, wvec, ga1, ldg1, c1, ga2, ldg2, c2, n, cout);
  } else if (ktot >= 128 && cout >= 64 && ceil_div(n, 128) * ceil_div(ktot, 128) >= num_sms()) {
    dim3 grid((unsigned)ceil_div(n, 128), (unsigned)ceil_div(ktot, 128));
    linear_bwd_input_kernel<128, 128><<<grid, GEMM_THREADS, 0, st>>>(grad_y, gvec, w, wvec, ga1, ldg1, c1, ga2, ldg2, c2, n, cout);
  } else {
    dim3 grid((unsigned)ceil_div(n, 64), (unsigned)ceil_div(ktot, 64));
    linear_bwd_input_kernel<64, 64><<<grid, GEMM_THREADS, 0, st>>>(grad_y, gvec, w, wvec, ga1, ldg1, c1, ga2, ldg2, c2, n, cout);
  }
  B200_CHECK_LAUNCH("linear_bwd_input_kernel");
  return B200_OK;
}

extern "C" int64_t b200_linear_bwd_weight_workspace_bytes(int64_t n, int32_t c1, int32_t c2, int32_t cout, int32_t has_bias) {
  if (n <= 0 || cout < 64 || c1 + c2 < 64) return 0;
  return (int64_t)tc_tn_workspace_bytes(cout, c1 + c2 + (has_bias ? 1 : 0), n);
}

extern "C" int b200_linear_bwd_weight(const float* grad_y, const float* a1, int64_t ld1, int32_t c1, const float* a2,
                                      int64_t ld2, int32_t c2, float* grad_w, float* grad_bias, void* workspace,
                                      int64_t workspace_bytes, int64_t n, int32_t cout, void* stream) {
  B200_REQUIRE(grad_y && a1 && grad_w, B200_E_INVALID, "b200_linear_bwd_weight: null pointer");
  B200_REQUIRE(c1 > 0 && c2 >= 0 && cout > 0 && (c2 == 0 || a2), B200_E_INVALID, "b200_linear_bwd_weight: bad sizes");
  if (n <= 0) return B200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const CatRows A = make_cat(a1, ld1, c1, a2, ld2, c2);
  B200_REQUIRE(!workspace || (reinterpret_cast<uintptr_t>(workspace) & 15) == 0, B200_E_INVALID,
               "b200_linear_bwd_weight: workspace must be 16-byte aligned");
  if (tma_rows_enabled(4) && tma_rows_tn_ok(n, grad_y, cout, a1, ld1, c1, a2, ld2, c2))
    return launch_tma_rows_tn(grad_y, cout, a1, ld1, c1, a2, ld2, c2, grad_w, grad_bias, n, st);
  return launch_tn(grad_y, cout, A, grad_w, grad_bias, n, static_cast<float*>(workspace),
                   workspace ? (size_t)workspace_bytes : 0, st);
}

extern "C" int64_t b200_linear_fwd_num_stat_partials(int64_t n, int32_t c1, int32_t c2, int32_t cout) {
  if (n <= 0) return 0;
  if (tc_nt_shape_ok(n, c1, c2, cout) && tc_path_enabled(1)) return ceil_div(n, tc_nt_rows_per_tile(n, cout));
  if (linear_rows_ok(n, c1 + c2, cout)) return linear_rows_grid(n);
  if (cout <= 32) return ceil_div(n, 128);
  if (cout >= 128 && c1 + c2 >= 64 && ceil_div(n, 128) * ceil_div(cout, 128) >= num_sms()) return ceil_div(n, 128);
  return ceil_div(n, 64);
}

extern "C" int b200_bn_finalize(const double* colstats, int32_t num_partials, int64_t count, const float* gamma,
                                const float* beta,
                                float* running_mean, float* running_var, int64_t* num_batches_tracked, float momentum,
                                float eps, float* scale, float* shift, float* mean, float* invstd, int32_t c,
                                void* stream) {
  B200_REQUIRE(gamma && beta && scale && shift && c > 0, B200_E_INVALID, "b200_bn_finalize: null pointer / c <= 0");
  B200_REQUIRE(colstats || (running_mean && running_var), B200_E_INVALID,
               "b200_bn_finalize: eval mode needs running statistics");
  B200_REQUIRE(!colstats || count > 0, B200_E_INVALID, "b200_bn_finalize: count must be positive");
  B200_REQUIRE((running_mean == nullptr) == (running_var == nullptr), B200_E_INVALID,
               "b200_bn_finalize: running_mean / running_var must come together");
  B200_REQUIRE(!colstats || num_partials >= 1, B200_E_INVALID, "b200_bn_finalize: num_partials must be >= 1");
  bn_finalize_kernel<<<(unsigned)c, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      colstats, num_partials, count, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, scale, shift, mean,
      invstd, c);
  B200_CHECK_LAUNCH("bn_finalize_kernel");
  return B200_OK;
}

extern "C" int b200_affine_act_fwd(const float* y1, const float* scale1, const float* shift1, const float* y2,
                                   const float* scale2, const float* shift2, float slope, float* out, int64_t n,
                                   int32_t c, void* stream) {
  B200_REQUIRE(y1 && scale1 && shift1 && out && c > 0, B200_E_INVALID, "b200_affine_act_fwd: null pointer");
  B200_REQUIRE(!y2 || (scale2 && shift2), B200_E_INVALID, "b200_affine_act_fwd: second branch incomplete");
  B200_REQUIRE(c <= 2048, B200_E_UNSUPPORTED, "b200_affine_act_fwd: at most 2048 channels (per-CTA coefficient table)");
  if (n <= 0) return B200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t total = n * c;
  const bool vec = (c % 4 == 0) && aligned16(y1) && aligned16(out) && (!y2 || aligned16(y2));
  if (vec)
    affine_act_fwd_kernel<4><<<elementwise_grid(total / 4), 256, 4 * c * sizeof(float), st>>>(y1, scale1, shift1, y2, scale2, shift2, slope, out, total, c);
  else
    affine_act_fwd_kernel<1><<<elementwise_grid(total), 256, 4 * c * sizeof(float), st>>>(y1, scale1, shift1, y2, scale2, shift2, slope, out, total, c);
  B200_CHECK_LAUNCH("affine_act_fwd_kernel");
  return B200_OK;
}

extern "C" int b200_affine_act_bwd_reduce(const float* grad_out, const float* out, float slope, const float* y1,
                                          const float* mean1, const float* invstd1, double* red1, const float* y2,
                                          const float* mean2, const float* invstd2, double* red2, int64_t n,
                                          int32_t c, void* stream) {
  B200_REQUIRE(grad_out && y1 && mean1 && invstd1 && red1 && c > 0, B200_E_INVALID, "b200_affine_act_bwd_reduce: null pointer");
  B200_REQUIRE(slope == 1.f || out, B200_E_INVALID, "b200_affine_act_bwd_reduce: activation needs `out`");
  B200_REQUIRE(!y2 || (mean2 && invstd2 && red2), B200_E_INVALID, "b200_affine_act_bwd_reduce: second branch incomplete");
  if (n <= 0) return B200_OK;
  if (c % 4 == 0 && aligned16(grad_out) && aligned16(y1) && (slope == 1.f || aligned16(out)) && (!y2 || aligned16(y2)) &&
      aligned16(mean1) && aligned16(invstd1) && (!y2 || (aligned16(mean2) && aligned16(invstd2)))) {
    int lanes = 1;
    while (lanes < c / 4 && lanes < RED_THREADS) lanes <<= 1;
    const int rstep = RED_THREADS / lanes;
    int64_t blocks = ceil_div(n, (int64_t)rstep * 4);
    const int64_t cap = (int64_t)num_sms() * 4;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    affine_act_bwd_reduce_vec4_kernel<<<(unsigned)blocks, RED_THREADS, 0,
                                        static_cast<cudaStream_t>(stream)>>>(grad_out, out, slope, y1, mean1, invstd1, red1, y2,
                                                                             mean2, invstd2, red2, n, c, lanes);
    B200_CHECK_LAUNCH("affine_act_bwd_reduce_vec4_kernel");
    return B200_OK;
  }
  int lanes = 1;
  while (lanes < c && lanes < RED_THREADS) lanes <<= 1;
  const int rstep = RED_THREADS / lanes;
  int64_t blocks = ceil_div(n, (int64_t)rstep * 8);
  const int64_t cap = (int64_t)num_sms() * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  affine_act_bwd_reduce_kernel<<<(unsigned)blocks, RED_THREADS, 4 * lanes * sizeof(double), static_cast<cudaStream_t>(stream)>>>(
      grad_out, out, slope, y1, mean1, invstd1, red1, y2, mean2, invstd2, red2, n, c, lanes);
  B200_CHECK_LAUNCH("affine_act_bwd_reduce_kernel");
  return B200_OK;
}

extern "C" int b200_affine_act_bwd_apply(const float* grad_out, const float* out, float slope, const float* y1,
                                         const float* gamma1, const float* mean1, const float* invstd1,
                                         const double* red1, const float* scale1, float* grad_y1, float* grad_gamma1,
                                         float* grad_beta1, const float* y2, const float* gamma2, const float* mean2,
                                         const float* invstd2, const double* red2, const float* scale2,
                                         float* grad_y2, float* grad_gamma2, float* grad_beta2, int64_t n, int32_t c,
                                         void* stream) {
  B200_REQUIRE(grad_out && grad_y1 && c > 0, B200_E_INVALID, "b200_affine_act_bwd_apply: null pointer");
  B200_REQUIRE(slope == 1.f || out, B200_E_INVALID, "b200_affine_act_bwd_apply: activation needs `out`");
  B200_REQUIRE(red1 ? (y1 && gamma1 && mean1 && invstd1) : (scale1 != nullptr), B200_E_INVALID,
               "b200_affine_act_bwd_apply: branch 1 incomplete");
  B200_REQUIRE(!y2 || (grad_y2 && (red2 ? (gamma2 && mean2 && invstd2) : (scale2 != nullptr))), B200_E_INVALID,
               "b200_affine_act_bwd_apply: branch 2 incomplete");
  B200_REQUIRE((grad_gamma1 == nullptr) == (grad_beta1 == nullptr) && (grad_gamma2 == nullptr) == (grad_beta2 == nullptr),
               B200_E_INVALID, "b200_affine_act_bwd_apply: grad_gamma / grad_beta must come together");
  B200_REQUIRE(c <= 1024, B200_E_UNSUPPORTED, "b200_affine_act_bwd_apply: at most 1024 channels (per-CTA coefficient table)");
  if (n <= 0) return B200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BnBranch b1{y1, gamma1, mean1, invstd1, red1, scale1, grad_y1, grad_gamma1, grad_beta1};
  BnBranch b2{y2, gamma2, mean2, invstd2, red2, scale2, grad_y2, grad_gamma2, grad_beta2};
  const int64_t total = n * c;
  bool vec = (c % 4 == 0) && aligned16(grad_out) && aligned16(grad_y1) && (!out || aligned16(out)) &&
             (!y1 || aligned16(y1)) && (!y2 || (aligned16(y2) && aligned16(grad_y2)));
  if (vec)
    affine_act_bwd_apply_kernel<4><<<elementwise_grid(total / 4), 256, 8 * c * sizeof(float), st>>>(grad_out, out, slope, b1, b2, n, c);
  else
    affine_act_bwd_apply_kernel<1><<<elementwise_grid(total), 256, 8 * c * sizeof(float), st>>>(grad_out, out, slope, b1, b2, n, c);
  B200_CHECK_LAUNCH("affine_act_bwd_apply_kernel");
  return B200_OK;
}

extern "C" int b200_affine_act_bwd(const float* grad_out, const float* out, float slope, const float* y1, const float* gamma1,
                                   const float* mean1, const float* invstd1, double* red1, float* grad_y1, float* grad_gamma1,
                                   float* grad_beta1, const float* y2, const float* gamma2, const float* mean2,
                                   const float* invstd2, double* red2, float* grad_y2, float* grad_gamma2, float* grad_beta2,
                                   uint32_t* barrier, int64_t n, int32_t c, void* stream) {
  B200_REQUIRE(grad_out && y1 && gamma1 && mean1 && invstd1 && red1 && grad_y1 && c > 0, B200_E_INVALID,
               "b200_affine_act_bwd: null pointer (train-mode BatchNorm backward: statistics and `red` are required)");
  B200_REQUIRE(slope == 1.f || out, B200_E_INVALID, "b200_affine_act_bwd: activation needs `out`");
  B200_REQUIRE(!y2 || (gamma2 && mean2 && invstd2 && red2 && grad_y2), B200_E_INVALID, "b200_affine_act_bwd: second branch incomplete");
  if (n <= 0) return B200_OK;
  const bool vec = c % 4 == 0 && c <= 1024 && aligned16(grad_out) && aligned16(y1) && aligned16(grad_y1) &&
                   (slope == 1.f || aligned16(out)) && aligned16(mean1) && aligned16(invstd1) &&
                   (!y2 || (aligned16(y2) && aligned16(grad_y2) && aligned16(mean2) && aligned16(invstd2)));
  if (vec && barrier && bn_backward_fused_enabled() && n * (int64_t)c <= ((int64_t)1 << 21)) {
    int lanes = 1;
    while (lanes < c / 4 && lanes < RED_THREADS) lanes <<= 1;
    const int rstep = RED_THREADS / lanes;
    int64_t blocks = ceil_div(n, (int64_t)rstep * 4);
    const int64_t cap = num_sms() / 2 > 0 ? num_sms() / 2 : 1;  // two instances can always be co-resident
    if (blocks > cap) blocks = cap;
    BnBranch b1{y1, gamma1, mean1, invstd1, red1, nullptr, grad_y1, grad_gamma1, grad_beta1};
    BnBranch b2{y2, gamma2, mean2, invstd2, red2, nullptr, grad_y2, grad_gamma2, grad_beta2};
    affine_act_bwd_fused_kernel<<<(unsigned)blocks, RED_THREADS, 8 * c * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
        grad_out, out, slope, b1, b2, red1, red2, barrier, n, c, lanes);
    B200_CHECK_LAUNCH("affine_act_bwd_fused_kernel");
    return B200_OK;
  }
  const int rc = b200_affine_act_bwd_reduce(grad_out, out, slope, y1, mean1, invstd1, red1, y2, mean2, invstd2, red2, n, c, stream);
  if (rc != B200_OK) return rc;
  return b200_affine_act_bwd_apply(grad_out, out, slope, y1, gamma1, mean1, invstd1, red1, nullptr, grad_y1, grad_gamma1,
                                   grad_beta1, y2, gamma2, mean2, invstd2, red2, nullptr, grad_y2, grad_gamma2, grad_beta2, n, c,
                                   stream);
}
