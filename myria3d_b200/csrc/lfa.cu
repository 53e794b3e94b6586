// Fused Local Spatial Encoding + attentive pooling (forward, backward) and the edge-moment
// pre-pass, for sm_100a.
//
// Replaces LocalFeatureAggregation.propagate()/message() of
// myria3d/models/modules/pyg_randla_net.py:121-152 -- in the reference ~20 library kernels over
// ~18 materialised [E, .] tensors (SURVEY.md 2c K3..K8) -- by ONE kernel per direction that keeps
// every per-edge quantity on chip:
//
//   tile   = TC centres x KT neighbour slots, processed by TC * (C/CW) threads; a persistent grid
//            walks the tiles.
//   build  : neighbour ids, (p_j, |p_j-p_i|) and p_i go to shared memory; F[edge][0:H) = x_j
//            (vectorised gathers), F[edge][H:C) = lrelu(enc_w . (p_i, p_j, dist) + enc_b).  The
//            10-d relative position vector of the reference is linear in those 7 numbers and the
//            encoder BatchNorm is linear in it, so both are folded into enc_w/enc_b on the host
//            (SURVEY.md App. D-7, D-8).
//   GEMM1  : a[k][n] = sum_m F[k][m] W_att[n][m]; thread (centre g, column group q) owns all KT
//            rows of its centre for CW columns -> the neighbourhood softmax and the weighted sum
//            are thread-local register reductions (no atomics, no scatter).
//   backward additionally: da = s*go*(f-o) to shared memory, GEMM2 dF = da.W + s*go (register
//            accumulators initialised with the direct term), x-gradients by vector red.global,
//            encoder-gradient partials in shared memory, GEMM3 dW += da^T F as 4x4 register blocks.
//
// These FMA kernels serve c in {8, 16} (K = 8 / 16 contractions: 94 % of the edges, too narrow for a 128-lane
// tensor tile); c in {32, 64, 128, 256} run on tcgen05 (lfa_tc.cu, lfa_tc256.cu), which maps channels to TMEM lanes
// and edges to columns so that the same thread-local softmax applies.  The FMA kernels of the wider levels stay as
// the reference of the tensor-core path (b200_set_option("tensor_cores", 0)).
#include <math_constants.h>

#include "common.cuh"

namespace b200 {

// ------------------------------------------------------------------------------------------
// edge moments: count, sum q, sum q q^T (fp64) with q = (p_i, p_j, |p_j - p_i|)
// ------------------------------------------------------------------------------------------
constexpr int MOM_THREADS = 128;
constexpr int MOM_VALS = 1 + 7 + 28;  // count, sums, upper triangle

__global__ void __launch_bounds__(MOM_THREADS)
edge_moments_kernel(const float* __restrict__ pos, const int32_t* __restrict__ nbr, int64_t n, int kt,
                    double* __restrict__ out) {
  double acc[MOM_VALS];
#pragma unroll
  for (int i = 0; i < MOM_VALS; ++i) acc[i] = 0.0;

  for (int64_t i = (int64_t)blockIdx.x * MOM_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * MOM_THREADS) {
    const float pix = pos[3 * i], piy = pos[3 * i + 1], piz = pos[3 * i + 2];
    const int32_t* row = nbr + i * kt;
    for (int k = 0; k < kt; ++k) {
      const int j = row[k];
      if (j < 0) break;  // valid neighbours are a prefix
      const float pjx = pos[3 * (int64_t)j], pjy = pos[3 * (int64_t)j + 1], pjz = pos[3 * (int64_t)j + 2];
      const float dx = pjx - pix, dy = pjy - piy, dz = pjz - piz;
      const float dist = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
      const double q[7] = {pix, piy, piz, pjx, pjy, pjz, dist};
      acc[0] += 1.0;
      int t = 8;
#pragma unroll
      for (int a = 0; a < 7; ++a) {
        acc[1 + a] += q[a];
#pragma unroll
        for (int b = a; b < 7; ++b) acc[t++] += q[a] * q[b];
      }
    }
  }

  __shared__ double red[MOM_THREADS / 32][MOM_VALS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < MOM_VALS; ++i) {
    const double v = warp_sum(acc[i]);
    if (lane == 0) red[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < MOM_VALS) {
    double v = 0.0;
    for (int w = 0; w < MOM_THREADS / 32; ++w) v += red[w][threadIdx.x];
    const int i = threadIdx.x;
    if (i < 8) {
      atomicAdd(out + i, v);
    } else {
      // unpack the upper-triangle slot into both symmetric positions of the 7x7 matrix
      int t = 8, ra = 0, rb = 0;
      for (int a = 0; a < 7; ++a)
        for (int b = a; b < 7; ++b) {
          if (t == i) {
            ra = a;
            rb = b;
          }
          ++t;
        }
      atomicAdd(out + 8 + ra * 7 + rb, v);
      if (ra != rb) atomicAdd(out + 8 + rb * 7 + ra, v);
    }
  }
}

// ------------------------------------------------------------------------------------------
// tile configuration
// ------------------------------------------------------------------------------------------
template <int C_, int KT_, int CW_, int TC_, int MINB_ = 3>
struct LfaCfg {
  static constexpr int C = C_, KT = KT_, CW = CW_, TC = TC_;
  static constexpr int MINB = MINB_;  // CTAs per SM the register allocator must leave room for
  static constexpr int H = C / 2;
  static constexpr int TPC = C / CW;          // threads per centre
  static constexpr int THREADS = TC * TPC;
  static constexpr int EDGES = TC * KT;
  static constexpr int CSTRIDE = KT * C + 4;  // floats per centre block (+4: spreads centres over banks)
  static constexpr int TILE_FLOATS = TC * CSTRIDE;
  static_assert(H % 4 == 0, "H must be a multiple of 4");
  static_assert(H % CW == 0, "a thread's columns must not straddle the x | encoding boundary");
  static_assert(THREADS % H == 0 || H % THREADS == 0, "encoder build mapping");
  static_assert(THREADS % 32 == 0, "whole warps");
};

template <int CW>
__device__ __forceinline__ void load_vec(float (&v)[CW], const float* __restrict__ p) {
  if constexpr (CW == 8) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    const float4 b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
  } else if constexpr (CW == 4) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w;
  } else {
    static_assert(CW == 2, "CW in {2,4,8}");
    const float2 a = *reinterpret_cast<const float2*>(p);
    v[0] = a.x, v[1] = a.y;
  }
}
template <int CW>
__device__ __forceinline__ void ldg_vec(float (&v)[CW], const float* __restrict__ p) {
  if constexpr (CW == 8) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + 4));
    v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
  } else if constexpr (CW == 4) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w;
  } else {
    const float2 a = __ldg(reinterpret_cast<const float2*>(p));
    v[0] = a.x, v[1] = a.y;
  }
}
template <int CW>
__device__ __forceinline__ void store_vec(float* __restrict__ p, const float (&v)[CW]) {
  if constexpr (CW == 8) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  } else if constexpr (CW == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
  }
}
// vector reduction into global memory (red.global.add.v4.f32 / v2.f32 on sm_90+)
template <int CW>
__device__ __forceinline__ void red_vec(float* __restrict__ p, const float (&v)[CW]) {
  if constexpr (CW == 8) {
    atomicAdd(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
    atomicAdd(reinterpret_cast<float4*>(p + 4), make_float4(v[4], v[5], v[6], v[7]));
  } else if constexpr (CW == 4) {
    atomicAdd(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
  } else {
    atomicAdd(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
  }
}

// ------------------------------------------------------------------------------------------
// build one tile: NB (neighbour ids), Q (p_j, dist), P (p_i), F (features)
// ------------------------------------------------------------------------------------------
// Neighbour ids of a tile, one register per edge this thread builds: fetched one tile ahead (the loads travel during
// the previous tile's contraction), so that the build starts with the dependent gathers instead of with a load.
template <class Cfg>
struct LfaIds {
  static constexpr int EPT = (Cfg::EDGES + Cfg::THREADS - 1) / Cfg::THREADS;
  // (K = 32 tables: the backward kernels are at their register limit -- the ids are loaded inside the build there)
  static constexpr bool AHEAD = (Cfg::KT <= 16);
  int j[AHEAD ? EPT : 1];
};
template <class Cfg>
__device__ __forceinline__ void lfa_prefetch_ids(LfaIds<Cfg>& ids, int64_t tile_base, int64_t n, int64_t ntiles_end,
                                                 const int32_t* __restrict__ nbr) {
  constexpr int KT = Cfg::KT, THREADS = Cfg::THREADS, EDGES = Cfg::EDGES;
  if constexpr (LfaIds<Cfg>::AHEAD) {
#pragma unroll
    for (int it = 0; it < LfaIds<Cfg>::EPT; ++it) {
      const int e = threadIdx.x + it * THREADS;
      const int64_t i = tile_base + e / KT;
      ids.j[it] = (e < EDGES && tile_base < ntiles_end && i < n) ? __ldg(nbr + i * KT + (e % KT)) : -1;
    }
  }
}

template <class Cfg>
__device__ __forceinline__ void lfa_build_tile(int64_t tile_base, int64_t n, const float* __restrict__ x,
                                               const float* __restrict__ pos, const LfaIds<Cfg>& ids,
                                               const int32_t* __restrict__ nbr, const float* __restrict__ enc_w, const float* __restrict__ enc_b,
                                               float* __restrict__ F, float4* __restrict__ Q,
                                               float4* __restrict__ P, int* __restrict__ NB) {
  constexpr int C = Cfg::C, KT = Cfg::KT, H = Cfg::H, THREADS = Cfg::THREADS, EDGES = Cfg::EDGES;
  constexpr int CSTRIDE = Cfg::CSTRIDE;
  constexpr int H4 = H / 4;
  constexpr bool GATHER_X_HERE = (H4 <= 2);  // narrow features: the edge's thread also gathers x_j (one latency, not two)
  const int tid = threadIdx.x;
  const float4* x4 = reinterpret_cast<const float4*>(x);

#pragma unroll
  for (int it = 0; it < LfaIds<Cfg>::EPT; ++it) {
    const int e = tid + it * THREADS;
    if (e >= EDGES) break;
    const int g = e / KT, kk = e % KT;
    const int64_t i = tile_base + g;
    int j;  // -1 beyond n / padded slots
    if constexpr (LfaIds<Cfg>::AHEAD) {
      j = ids.j[it];
    } else {
      j = (i < n) ? __ldg(nbr + i * KT + kk) : -1;
    }
    float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 pv = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 xv[GATHER_X_HERE ? H4 : 1];
#pragma unroll
    for (int m4 = 0; m4 < (GATHER_X_HERE ? H4 : 1); ++m4) xv[m4] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n) {
      pv = make_float4(__ldg(pos + 3 * i), __ldg(pos + 3 * i + 1), __ldg(pos + 3 * i + 2), 0.f);
      if (j >= 0) {
        const float pjx = __ldg(pos + 3 * (int64_t)j), pjy = __ldg(pos + 3 * (int64_t)j + 1),
                    pjz = __ldg(pos + 3 * (int64_t)j + 2);
        if constexpr (GATHER_X_HERE) {
#pragma unroll
          for (int m4 = 0; m4 < H4; ++m4) xv[m4] = __ldg(x4 + (int64_t)j * H4 + m4);
        }
        const float dx = pjx - pv.x, dy = pjy - pv.y, dz = pjz - pv.z;
        const float dist = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
        qv = make_float4(pjx, pjy, pjz, dist);
      }
    }
    NB[e] = j;
    Q[e] = qv;
    if (kk == 0) P[g] = pv;
    if constexpr (GATHER_X_HERE) {
#pragma unroll
      for (int m4 = 0; m4 < H4; ++m4) *reinterpret_cast<float4*>(F + g * CSTRIDE + kk * C + m4 * 4) = xv[m4];
    }
  }
  __syncthreads();

  // x_j gather into F[:, 0:H)
  if constexpr (!GATHER_X_HERE) {
    for (int t = tid; t < EDGES * H4; t += THREADS) {
      const int e = t / H4, m4 = t % H4;
      const int j = NB[e];
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j >= 0) v = __ldg(x4 + (int64_t)j * H4 + m4);
      *reinterpret_cast<float4*>(F + (e / KT) * CSTRIDE + (e % KT) * C + m4 * 4) = v;
    }
  }

  // encoder into F[:, H:C)
  if constexpr (THREADS >= H) {
    constexpr int EPI = THREADS / H;  // edges handled per iteration
    const int m = tid % H, e0 = tid / H;
    float w[7];
#pragma unroll
    for (int t = 0; t < 7; ++t) w[t] = __ldg(enc_w + m * 7 + t);
    const float b = __ldg(enc_b + m);
    for (int e = e0; e < EDGES; e += EPI) {
      const int g = e / KT;
      float v = 0.f;
      if (NB[e] >= 0) {
        const float4 p = P[g], q = Q[e];
        float z = b;
        z = fmaf(w[0], p.x, z), z = fmaf(w[1], p.y, z), z = fmaf(w[2], p.z, z);
        z = fmaf(w[3], q.x, z), z = fmaf(w[4], q.y, z), z = fmaf(w[5], q.z, z);
        z = fmaf(w[6], q.w, z);
        v = lrelu(z, kLReluSlope);
      }
      F[g * CSTRIDE + (e % KT) * C + H + m] = v;
    }
  } else {
    for (int m = tid; m < H; m += THREADS) {
      float w[7];
#pragma unroll
      for (int t = 0; t < 7; ++t) w[t] = __ldg(enc_w + m * 7 + t);
      const float b = __ldg(enc_b + m);
      for (int e = 0; e < EDGES; ++e) {
        const int g = e / KT;
        float v = 0.f;
        if (NB[e] >= 0) {
          const float4 p = P[g], q = Q[e];
          float z = b;
          z = fmaf(w[0], p.x, z), z = fmaf(w[1], p.y, z), z = fmaf(w[2], p.z, z);
          z = fmaf(w[3], q.x, z), z = fmaf(w[4], q.y, z), z = fmaf(w[5], q.z, z);
          z = fmaf(w[6], q.w, z);
          v = lrelu(z, kLReluSlope);
        }
        F[g * CSTRIDE + (e % KT) * C + H + m] = v;
      }
    }
  }
  __syncthreads();
}

// acc[k][cw] += sum_r A[k][r] * B[r][col0 + cw],  A = this centre's KT x C block in shared memory,
// B = [C][C] row-major in global memory (L1/L2 resident), columns col0.. owned by this thread.
template <class Cfg>
__device__ __forceinline__ void centre_gemm(float (&acc)[Cfg::KT][Cfg::CW], const float* __restrict__ A,
                                            const float* __restrict__ B, int col0) {
  constexpr int C = Cfg::C, KT = Cfg::KT, CW = Cfg::CW;
  // register double buffer for the B rows: the loads of rows r0+4..r0+7 are in flight while rows r0..r0+3 are
  // multiplied (the FFMAs were stalling on these L1/L2 loads: long-scoreboard in the ncu source view)
  float b[2][4][CW];
#pragma unroll
  for (int u = 0; u < 4; ++u) ldg_vec<CW>(b[0][u], B + (int64_t)u * C + col0);
#pragma unroll 1
  for (int r0 = 0; r0 < C; r0 += 8) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int r = r0 + 4 * half;
      if (r + 4 < C) {
#pragma unroll
        for (int u = 0; u < 4; ++u) ldg_vec<CW>(b[half ^ 1][u], B + (int64_t)(r + 4 + u) * C + col0);
      }
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(A + k * C + r);
        // packed FMAs over column pairs (FFMA2): same products, same accumulation order per column as the scalar loop
        const float2 ax = make_float2(a.x, a.x), ay = make_float2(a.y, a.y), az = make_float2(a.z, a.z), aw = make_float2(a.w, a.w);
#pragma unroll
        for (int cw = 0; cw < CW; cw += 2) {
          float2 v = make_float2(acc[k][cw], acc[k][cw + 1]);
          v = ffma2(ax, make_float2(b[half][0][cw], b[half][0][cw + 1]), v);
          v = ffma2(ay, make_float2(b[half][1][cw], b[half][1][cw + 1]), v);
          v = ffma2(az, make_float2(b[half][2][cw], b[half][2][cw + 1]), v);
          v = ffma2(aw, make_float2(b[half][3][cw], b[half][3][cw + 1]), v);
          acc[k][cw] = v.x, acc[k][cw + 1] = v.y;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, (Cfg::THREADS <= 128 ? Cfg::MINB : 1))
lfa_fwd_kernel(const float* __restrict__ x, const float* __restrict__ pos, const int32_t* __restrict__ nbr,
               const float* __restrict__ enc_w, const float* __restrict__ enc_b,
               const float* __restrict__ att_wt, float* __restrict__ out, int64_t n, int64_t ntiles) {
  constexpr int C = Cfg::C, KT = Cfg::KT, CW = Cfg::CW, TC = Cfg::TC, TPC = Cfg::TPC;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* F = reinterpret_cast<float*>(smem_raw);
  float4* Q = reinterpret_cast<float4*>(F + Cfg::TILE_FLOATS);
  float4* P = Q + Cfg::EDGES;
  int* NB = reinterpret_cast<int*>(P + TC);

  const int tid = threadIdx.x;
  const int g = tid / TPC, col0 = (tid % TPC) * CW;

  LfaIds<Cfg> ids;
  lfa_prefetch_ids<Cfg>(ids, (int64_t)blockIdx.x * TC, n, ntiles * TC, nbr);
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t tile_base = tile * TC;
    lfa_build_tile<Cfg>(tile_base, n, x, pos, ids, nbr, enc_w, enc_b, F, Q, P, NB);
    lfa_prefetch_ids<Cfg>(ids, (tile + gridDim.x) * TC, n, ntiles * TC, nbr);  // next tile: in flight during the contraction

    float acc[KT][CW];
#pragma unroll
    for (int k = 0; k < KT; ++k)
#pragma unroll
      for (int cw = 0; cw < CW; ++cw) acc[k][cw] = 0.f;
    const float* Fg = F + g * Cfg::CSTRIDE;
    centre_gemm<Cfg>(acc, Fg, att_wt, col0);

    int deg = 0;
#pragma unroll
    for (int k = 0; k < KT; ++k) deg += (NB[g * KT + k] >= 0) ? 1 : 0;

    float mx[CW], sum[CW], o[CW];
#pragma unroll
    for (int cw = 0; cw < CW; ++cw) mx[cw] = -CUDART_INF_F, sum[cw] = 0.f, o[cw] = 0.f;
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < deg) {
#pragma unroll
        for (int cw = 0; cw < CW; ++cw) mx[cw] = fmaxf(mx[cw], acc[k][cw]);
      }
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < deg) {
        float f[CW];
        load_vec<CW>(f, Fg + k * C + col0);
#pragma unroll
        for (int cw = 0; cw < CW; ++cw) {
          const float p = __expf(acc[k][cw] - mx[cw]);
          sum[cw] += p;
          o[cw] = fmaf(p, f[cw], o[cw]);
        }
      }
    const int64_t i = tile_base + g;
    if (i < n) {
#pragma unroll
      for (int cw = 0; cw < CW; ++cw) o[cw] = o[cw] / (sum[cw] + 1e-16f);
      store_vec<CW>(out + i * C + col0, o);
    }
    __syncthreads();  // tile buffers are rebuilt next iteration
  }
}

// ------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------
// Two flavours of the attention-weight gradient dW[n][m] = sum_e DA[e][n] F[e][m]:
//   SPLIT_DW = false (C <= 32, millions of edges): 4x4 register blocks per thread, accumulated over all
//              the tiles a persistent CTA visits, reduced once at the end (no per-tile atomics);
//   SPLIT_DW = true  (C >= 64, deep levels, few edges): the tile's DA and F rows are streamed to a
//              caller-provided workspace ([E, C] each) and a split-K GEMM (pointwise.cu) reduces them; the
//              fused kernel then needs neither C*C accumulators nor C*C atomics per tile, so it can use
//              small tiles and several CTAs per SM.
template <class Cfg>
struct LfaBwdPlan {
  static constexpr int C = Cfg::C, THREADS = Cfg::THREADS;
  static constexpr int NB4 = C / 4;                  // 4x4 output blocks per dimension
  static constexpr int NBLOCKS = NB4 * NB4;
  static constexpr int SLICES = (NBLOCKS >= THREADS) ? 1 : (THREADS / NBLOCKS);  // edge slices per block
  static constexpr int PASSES = (NBLOCKS >= THREADS) ? (NBLOCKS / THREADS) : 1;
  static constexpr bool GE_IN_REGS = (C <= 32);      // encoder-gradient partials live in registers
  // C <= 32: dW[n][m] partials are owned by the thread that already holds da[k][n] in registers (n = its CW columns):
  // dW[n][:] += da[k][n] * F[k][:] needs only broadcast LDS.128 of the centre's F rows (16 FMA per load) instead of
  // the 4x4-block GEMM3 whose strided row reads were 4-way bank conflicted and shared-memory bound.
  static constexpr bool DW_BY_CENTRE = (C <= 32);
  // Encoder-gradient partials in shared memory (C >= 64): one private [H][8] slab per group of threads in which every
  // encoder column has exactly ONE writer after an intra-warp shuffle reduction over the centres of the warp --
  // plain read-modify-write instead of contended float atomics (sm_100a emulates shared float atomicAdd with a CAS
  // loop: 37 M excess shared wavefronts out of 85 M in the c = 64 kernel, profiles/ncu_lfa_bwd64b_r01.summary.txt).
  static constexpr int GE_GROUP = (Cfg::TPC > 32) ? Cfg::TPC : 32;     // threads sharing a slab
  static constexpr int GE_SLABS = GE_IN_REGS ? 1 : (THREADS / GE_GROUP);
  __host__ __device__ static constexpr unsigned enc_lane_mask() {  // lanes of a warp whose columns lie in the encoder half
    unsigned m = 0;
    for (int l = 0; l < 32; ++l)
      if (((l % Cfg::TPC) * Cfg::CW) >= Cfg::H || Cfg::TPC > 32) m |= 1u << l;
    return m;
  }
};

template <class Cfg, bool SPLIT_DW>
__global__ void __launch_bounds__(Cfg::THREADS, (Cfg::THREADS <= 128 ? Cfg::MINB : 1))
lfa_bwd_kernel(const float* __restrict__ x, const float* __restrict__ pos, const int32_t* __restrict__ nbr,
               const float* __restrict__ enc_w, const float* __restrict__ enc_b,
               const float* __restrict__ att_wt, const float* __restrict__ att_w,
               const float* __restrict__ grad_out, float* __restrict__ grad_x, float* __restrict__ grad_enc_w,
               float* __restrict__ grad_enc_b, float* __restrict__ grad_att_w, float* __restrict__ da_out,
               float* __restrict__ f_out, int64_t n, int64_t ntiles) {
  constexpr int C = Cfg::C, KT = Cfg::KT, CW = Cfg::CW, TC = Cfg::TC, TPC = Cfg::TPC, H = Cfg::H;
  constexpr int THREADS = Cfg::THREADS, EDGES = Cfg::EDGES, CSTRIDE = Cfg::CSTRIDE;
  using Plan = LfaBwdPlan<Cfg>;
  static_assert(SPLIT_DW || Plan::PASSES <= 2, "register dW accumulation needs <= 2 passes");
  static_assert(SPLIT_DW || (Plan::SLICES <= 32 && (Plan::SLICES & (Plan::SLICES - 1)) == 0), "slices: power of two <= 32");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* F = reinterpret_cast<float*>(smem_raw);
  float* DA = F + Cfg::TILE_FLOATS;
  float4* Q = reinterpret_cast<float4*>(DA + Cfg::TILE_FLOATS);
  float4* P = Q + EDGES;
  int* NB = reinterpret_cast<int*>(P + TC);
  float* GE = reinterpret_cast<float*>(NB + EDGES);  // [GE_SLABS][H][8]: 7 weight grads + bias grad

  const int tid = threadIdx.x;
  const int g = tid / TPC, col0 = (tid % TPC) * CW;

  for (int t = tid; t < Plan::GE_SLABS * H * 8; t += THREADS) GE[t] = 0.f;

  constexpr int DWP = SPLIT_DW ? 1 : Plan::PASSES;
  float dw[DWP][16];
#pragma unroll
  for (int p = 0; p < DWP; ++p)
#pragma unroll
    for (int t = 0; t < 16; ++t) dw[p][t] = 0.f;
  constexpr bool DWC = !SPLIT_DW && Plan::DW_BY_CENTRE;
  float dwc[DWC ? CW : 1][DWC ? C : 1];
#pragma unroll
  for (int cw = 0; cw < (DWC ? CW : 1); ++cw)
#pragma unroll
    for (int m = 0; m < (DWC ? C : 1); ++m) dwc[cw][m] = 0.f;
  constexpr int GEW = Plan::GE_IN_REGS ? CW : 1;
  float ge_reg[GEW][8];
#pragma unroll
  for (int cw = 0; cw < GEW; ++cw)
#pragma unroll
    for (int t = 0; t < 8; ++t) ge_reg[cw][t] = 0.f;

  LfaIds<Cfg> ids;
  lfa_prefetch_ids<Cfg>(ids, (int64_t)blockIdx.x * TC, n, ntiles * TC, nbr);
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t tile_base = tile * TC;
    lfa_build_tile<Cfg>(tile_base, n, x, pos, ids, nbr, enc_w, enc_b, F, Q, P, NB);
    lfa_prefetch_ids<Cfg>(ids, (tile + gridDim.x) * TC, n, ntiles * TC, nbr);  // next tile: in flight during the contraction

    float acc[KT][CW];
#pragma unroll
    for (int k = 0; k < KT; ++k)
#pragma unroll
      for (int cw = 0; cw < CW; ++cw) acc[k][cw] = 0.f;
    const float* Fg = F + g * CSTRIDE;
    float* DAg = DA + g * CSTRIDE;
    centre_gemm<Cfg>(acc, Fg, att_wt, col0);

    int deg = 0;
#pragma unroll
    for (int k = 0; k < KT; ++k) deg += (NB[g * KT + k] >= 0) ? 1 : 0;
    const int64_t i = tile_base + g;

    {  // softmax backward: acc <- s*go (direct term of dF), DA <- s*go*(f - o)
      float mx[CW], sum[CW], o[CW], go[CW];
#pragma unroll
      for (int cw = 0; cw < CW; ++cw) mx[cw] = -CUDART_INF_F, sum[cw] = 0.f, o[cw] = 0.f, go[cw] = 0.f;
      if (i < n) ldg_vec<CW>(go, grad_out + i * C + col0);
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (k < deg) {
#pragma unroll
          for (int cw = 0; cw < CW; ++cw) mx[cw] = fmaxf(mx[cw], acc[k][cw]);
        }
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (k < deg) {
          float f[CW];
          load_vec<CW>(f, Fg + k * C + col0);
#pragma unroll
          for (int cw = 0; cw < CW; ++cw) {
            const float p = __expf(acc[k][cw] - mx[cw]);
            acc[k][cw] = p;
            sum[cw] += p;
            o[cw] = fmaf(p, f[cw], o[cw]);
          }
        }
      float inv[CW];
#pragma unroll
      for (int cw = 0; cw < CW; ++cw) {
        inv[cw] = 1.f / (sum[cw] + 1e-16f);
        o[cw] *= inv[cw];
      }
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        float da[CW], f[CW];
        load_vec<CW>(f, Fg + k * C + col0);  // zeros for invalid edges
        if (k < deg) {
#pragma unroll
          for (int cw = 0; cw < CW; ++cw) {
            const float sg = acc[k][cw] * inv[cw] * go[cw];
            acc[k][cw] = sg;
            da[cw] = sg * (f[cw] - o[cw]);
          }
        } else {
#pragma unroll
          for (int cw = 0; cw < CW; ++cw) {
            acc[k][cw] = 0.f;
            da[cw] = 0.f;
          }
        }
        store_vec<CW>(DAg + k * C + col0, da);
        if constexpr (DWC) {
          if (k < deg) {
#pragma unroll
            for (int m4 = 0; m4 < C / 4; ++m4) {
              const float4 fr = *reinterpret_cast<const float4*>(Fg + k * C + m4 * 4);  // broadcast within the centre
#pragma unroll
              for (int cw = 0; cw < CW; ++cw) {
                ffma2_bc(da[cw], fr.x, fr.y, dwc[cw][m4 * 4 + 0], dwc[cw][m4 * 4 + 1]);
                ffma2_bc(da[cw], fr.z, fr.w, dwc[cw][m4 * 4 + 2], dwc[cw][m4 * 4 + 3]);
              }
            }
          }
        }
        if constexpr (SPLIT_DW) {
          if (i < n) {  // stream the edge rows out for the split-K dW GEMM
            const int64_t row = (i * KT + k) * C + col0;
            store_vec<CW>(da_out + row, da);
            store_vec<CW>(f_out + row, f);
          }
        }
      }
    }
    __syncthreads();

    // GEMM2: dF[k][m] = sg[k][m] + sum_n DA[k][n] W[n][m]   (acc already holds sg)
    centre_gemm<Cfg>(acc, DAg, att_w, col0);

    if (col0 < H) {
      // gradient w.r.t. the gathered neighbour features
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (k < deg) {
          const int j = NB[g * KT + k];
          red_vec<CW>(grad_x + (int64_t)j * H + col0, acc[k]);
        }
    } else {
      // gradient w.r.t. the (folded) encoder: dz = dF * lrelu'(z), sign(z) = sign(e)
      const float4 p = P[g];
#pragma unroll
      for (int cw = 0; cw < CW; ++cw) {
        float gw[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) gw[t] = 0.f;
#pragma unroll
        for (int k = 0; k < KT; ++k)
          if (k < deg) {
            const float e = Fg[k * C + col0 + cw];
            const float dz = acc[k][cw] * (e > 0.f ? 1.f : kLReluSlope);
            const float4 q = Q[g * KT + k];
            gw[3] = fmaf(dz, q.x, gw[3]);
            gw[4] = fmaf(dz, q.y, gw[4]);
            gw[5] = fmaf(dz, q.z, gw[5]);
            gw[6] = fmaf(dz, q.w, gw[6]);
            gw[7] += dz;
          }
        gw[0] = gw[7] * p.x, gw[1] = gw[7] * p.y, gw[2] = gw[7] * p.z;
        if constexpr (Plan::GE_IN_REGS) {
#pragma unroll
          for (int t = 0; t < 8; ++t) ge_reg[cw][t] += gw[t];
        } else {
          // sum over the centres that share this warp (lanes l, l ^ TPC, ... hold the same columns), then the first
          // of them adds into the slab of its thread group: one writer per address, no atomics
          if constexpr (TPC < 32) {
            constexpr unsigned kMask = Plan::enc_lane_mask();
#pragma unroll
            for (int off = TPC; off < 32; off <<= 1)
#pragma unroll
              for (int t = 0; t < 8; ++t) gw[t] += __shfl_xor_sync(kMask, gw[t], off);
          }
          if ((tid & 31) < TPC || TPC >= 32) {
            float* ge = GE + ((tid / Plan::GE_GROUP) * H + (col0 - H + cw)) * 8;
            float4 a = *reinterpret_cast<float4*>(ge), b = *reinterpret_cast<float4*>(ge + 4);
            a.x += gw[0], a.y += gw[1], a.z += gw[2], a.w += gw[3];
            b.x += gw[4], b.y += gw[5], b.z += gw[6], b.w += gw[7];
            *reinterpret_cast<float4*>(ge) = a;
            *reinterpret_cast<float4*>(ge + 4) = b;
          }
        }
      }
    }

    if constexpr (!SPLIT_DW && !DWC) {
      // GEMM3: dW[n][m] += sum_e DA[e][n] F[e][m], 4x4 register blocks carried across tiles
#pragma unroll
      for (int pass = 0; pass < Plan::PASSES; ++pass) {
        const int ob = (Plan::SLICES > 1) ? (tid / Plan::SLICES) : (pass * THREADS + tid);
        const int es = (Plan::SLICES > 1) ? (tid % Plan::SLICES) : 0;
        const int nb = ob / Plan::NB4, mb = ob % Plan::NB4;
#pragma unroll 4
        for (int e = es; e < EDGES; e += Plan::SLICES) {
          const int off = (e / KT) * CSTRIDE + (e % KT) * C;
          const float4 a = *reinterpret_cast<const float4*>(DA + off + nb * 4);
          const float4 b = *reinterpret_cast<const float4*>(F + off + mb * 4);
          const float av[4] = {a.x, a.y, a.z, a.w};
          const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            ffma2_bc(av[r], bv[0], bv[1], dw[pass][r * 4 + 0], dw[pass][r * 4 + 1]);
            ffma2_bc(av[r], bv[2], bv[3], dw[pass][r * 4 + 2], dw[pass][r * 4 + 3]);
          }
        }
      }
    }
    __syncthreads();  // tile buffers are rebuilt next iteration
  }

  // flush the per-CTA partial gradients
  if constexpr (DWC) {
    // reduce the per-thread dW rows over the centres of the CTA in shared memory (the F tile is free now)
    float* DWS = F;  // [C][C]
    __syncthreads();
    for (int t = tid; t < C * C; t += THREADS) DWS[t] = 0.f;
    __syncthreads();
#pragma unroll
    for (int cw = 0; cw < CW; ++cw)
#pragma unroll
      for (int m = 0; m < C; ++m) atomicAdd(&DWS[(col0 + cw) * C + m], dwc[cw][m]);
    __syncthreads();
    for (int t = tid; t < C * C; t += THREADS) atomicAdd(grad_att_w + t, DWS[t]);
  }
  if constexpr (!SPLIT_DW && !DWC) {
#pragma unroll
    for (int pass = 0; pass < Plan::PASSES; ++pass) {
      const int ob = (Plan::SLICES > 1) ? (tid / Plan::SLICES) : (pass * THREADS + tid);
      const int es = (Plan::SLICES > 1) ? (tid % Plan::SLICES) : 0;
      const int nb = ob / Plan::NB4, mb = ob % Plan::NB4;
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        float v = dw[pass][t];
#pragma unroll
        for (int o = Plan::SLICES / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        dw[pass][t] = v;
      }
      if (es == 0) {
#pragma unroll
        for (int r = 0; r < 4; ++r)
          atomicAdd(reinterpret_cast<float4*>(grad_att_w + (int64_t)(nb * 4 + r) * C + mb * 4),
                    make_float4(dw[pass][r * 4 + 0], dw[pass][r * 4 + 1], dw[pass][r * 4 + 2], dw[pass][r * 4 + 3]));
      }
    }
  }
  if constexpr (Plan::GE_IN_REGS) {
    if (col0 >= H) {
#pragma unroll
      for (int cw = 0; cw < CW; ++cw)
#pragma unroll
        for (int t = 0; t < 8; ++t) atomicAdd(GE + (col0 - H + cw) * 8 + t, ge_reg[cw][t]);
    }
  }
  __syncthreads();
  for (int t = tid; t < H * 8; t += THREADS) {
    float v = 0.f;
#pragma unroll
    for (int sl = 0; sl < Plan::GE_SLABS; ++sl) v += GE[sl * H * 8 + t];
    const int m = t >> 3, s = t & 7;
    if (s < 7)
      atomicAdd(grad_enc_w + m * 7 + s, v);
    else
      atomicAdd(grad_enc_b + m, v);
  }
}

// ------------------------------------------------------------------------------------------
// dispatch
// ------------------------------------------------------------------------------------------
template <class Cfg>
static size_t lfa_fwd_smem() {
  return sizeof(float) * Cfg::TILE_FLOATS + sizeof(float4) * (Cfg::EDGES + Cfg::TC) + sizeof(int) * Cfg::EDGES;
}
template <class Cfg>
static size_t lfa_bwd_smem() {
  return sizeof(float) * 2 * Cfg::TILE_FLOATS + sizeof(float4) * (Cfg::EDGES + Cfg::TC) + sizeof(int) * Cfg::EDGES +
         sizeof(float) * LfaBwdPlan<Cfg>::GE_SLABS * Cfg::H * 8;
}

int persistent_grid(const void* kernel, int threads, size_t smem, int64_t ntiles) {
  int per_sm = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    per_sm = 1;
  }
  int64_t g = (int64_t)num_sms() * per_sm;
  if (g > ntiles) g = ntiles;
  return (int)(g < 1 ? 1 : g);
}

template <class Cfg>
static int launch_lfa_fwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w,
                          const float* enc_b, const float* att_wt, float* out, int64_t n, cudaStream_t st) {
  const size_t smem = lfa_fwd_smem<Cfg>();
  auto kern = lfa_fwd_kernel<Cfg>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "lfa_fwd smem attribute");
  const int64_t ntiles = ceil_div(n, Cfg::TC);
  const int grid = persistent_grid(reinterpret_cast<const void*>(kern), Cfg::THREADS, smem, ntiles);
  kern<<<grid, Cfg::THREADS, smem, st>>>(x, pos, nbr, enc_w, enc_b, att_wt, out, n, ntiles);
  B200_CHECK_LAUNCH("lfa_fwd_kernel");
  return B200_OK;
}

template <class Cfg, bool SPLIT_DW>
static int launch_lfa_bwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w,
                          const float* enc_b, const float* att_wt, const float* att_w, const float* go, float* gx,
                          float* gew, float* geb, float* gaw, float* ws, int64_t n, cudaStream_t st) {
  const size_t smem = lfa_bwd_smem<Cfg>();
  auto kern = lfa_bwd_kernel<Cfg, SPLIT_DW>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "lfa_bwd smem attribute");
  const int64_t ntiles = ceil_div(n, Cfg::TC);
  const int grid = persistent_grid(reinterpret_cast<const void*>(kern), Cfg::THREADS, smem, ntiles);
  float* da_out = SPLIT_DW ? ws : nullptr;
  float* f_out = SPLIT_DW ? ws + n * Cfg::KT * Cfg::C : nullptr;
  kern<<<grid, Cfg::THREADS, smem, st>>>(x, pos, nbr, enc_w, enc_b, att_wt, att_w, go, gx, gew, geb, gaw, da_out,
                                         f_out, n, ntiles);
  B200_CHECK_LAUNCH("lfa_bwd_kernel");
  if (SPLIT_DW) {  // dW_att[n][m] += sum_e DA[e][n] F[e][m]: split-K GEMM over the streamed edge rows
    float* part = ws + 2 * n * Cfg::KT * Cfg::C;
    return accumulate_at_b(da_out, Cfg::C, f_out, Cfg::C, gaw, n * Cfg::KT, part,
                           accumulate_at_b_workspace_bytes(Cfg::C, Cfg::C, n * Cfg::KT), st);
  }
  return B200_OK;
}

}  // namespace b200

extern "C" int b200_edge_moments(const float* pos, const int32_t* nbr, int64_t n, int32_t kt, double* out,
                                 void* stream) {
  using namespace b200;
  B200_REQUIRE(pos && nbr && out, B200_E_INVALID, "b200_edge_moments: null pointer");
  B200_REQUIRE(kt >= 1, B200_E_INVALID, "b200_edge_moments: kt=%d", kt);
  if (n <= 0) return B200_OK;
  int64_t blocks = ceil_div(n, MOM_THREADS);
  const int64_t cap = (int64_t)num_sms() * 4;
  if (blocks > cap) blocks = cap;
  edge_moments_kernel<<<(unsigned)blocks, MOM_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(pos, nbr, n, kt, out);
  B200_CHECK_LAUNCH("edge_moments_kernel");
  return B200_OK;
}

// (C, KT) -> (CW, TC) tables; see the header comment for the reasoning.
// X(C, KT, CW, TC[, SPLIT_DW]): THREADS = TC * C / CW.  Small tiles + CW = 4 keep registers near 128 and shared
// memory near 33 KB (fwd) / 66 KB (bwd) so that 3-4 CTAs share an SM.
#define B200_LFA_FWD_CASES(X) \
  X(8, 16, 2, 32) X(16, 16, 4, 32) X(32, 16, 2, 8) X(64, 16, 4, 8) X(128, 16, 4, 4) X(256, 16, 4, 2) \
  X(8, 32, 2, 32) X(16, 32, 4, 32) X(32, 32, 4, 16) X(64, 32, 4, 8) X(128, 32, 4, 4) X(256, 32, 4, 2)
#define B200_LFA_BWD_CASES(X) \
  X(8, 16, 2, 32, false) X(16, 16, 2, 16, false, 3) X(32, 16, 2, 8, false, 3) \
  X(64, 16, 4, 8, true) X(128, 16, 4, 4, true) X(256, 16, 4, 2, true) \
  X(8, 32, 2, 32, false) X(16, 32, 2, 16, false, 3) X(32, 32, 2, 8, false, 3) \
  X(64, 32, 4, 4, true) X(128, 32, 4, 2, true) X(256, 32, 4, 2, true)

extern "C" int b200_lfa_fwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w,
                            const float* enc_b, const float* att_wt, float* out, int64_t n, int32_t c, int32_t kt,
                            void* stream) {
  using namespace b200;
  B200_REQUIRE(x && pos && nbr && enc_w && enc_b && att_wt && out, B200_E_INVALID, "b200_lfa_fwd: null pointer");
  B200_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)att_wt & 15) == 0 && ((uintptr_t)out & 15) == 0, B200_E_INVALID,
               "b200_lfa_fwd: x, att_wt and out must be 16-byte aligned");
  if (n <= 0) return B200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  {  // c in {32, 64, 128, 256}: the contraction on the tensor cores (lfa_tc.cu, lfa_tc256.cu)
    const int rc = lfa_tc_fwd_dispatch(x, pos, nbr, enc_w, enc_b, att_wt, out, n, c, kt, st);
    if (rc != B200_E_UNSUPPORTED) return rc;
  }
#define X(C_, KT_, CW_, TC_) \
  if (c == C_ && kt == KT_) return launch_lfa_fwd<LfaCfg<C_, KT_, CW_, TC_>>(x, pos, nbr, enc_w, enc_b, att_wt, out, n, st);
  B200_LFA_FWD_CASES(X)
#undef X
  set_error("b200_lfa_fwd: unsupported (c=%d, kt=%d); c in {8,16,32,64,128,256}, kt in {16,32}", c, kt);
  return B200_E_UNSUPPORTED;
}

extern "C" int64_t b200_lfa_bwd_workspace_bytes(int64_t n, int32_t c, int32_t kt) {
  if (n <= 0) return 0;
  if (b200::lfa_tc_supported(c, kt)) return b200::lfa_tc_bwd_workspace_bytes(n, c, kt);
  if (c < 64) return 0;
  return 2 * n * (int64_t)kt * c * (int64_t)sizeof(float) + (int64_t)b200::accumulate_at_b_workspace_bytes(c, c, n * kt);
}

extern "C" int b200_lfa_bwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w,
                            const float* enc_b, const float* att_wt, const float* att_w, const float* grad_out,
                            float* grad_x, float* grad_enc_w, float* grad_enc_b, float* grad_att_w, void* workspace,
                            int64_t workspace_bytes, int64_t n, int32_t c, int32_t kt, void* stream) {
  using namespace b200;
  B200_REQUIRE(x && pos && nbr && enc_w && enc_b && att_wt && att_w && grad_out && grad_x && grad_enc_w &&
                   grad_enc_b && grad_att_w,
               B200_E_INVALID, "b200_lfa_bwd: null pointer");
  B200_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)att_wt & 15) == 0 && ((uintptr_t)att_w & 15) == 0 &&
                   ((uintptr_t)grad_out & 15) == 0 && ((uintptr_t)grad_x & 15) == 0 && ((uintptr_t)grad_att_w & 15) == 0,
               B200_E_INVALID, "b200_lfa_bwd: tensors must be 16-byte aligned");
  if (n <= 0) return B200_OK;
  B200_REQUIRE(workspace_bytes >= b200_lfa_bwd_workspace_bytes(n, c, kt) && (workspace || workspace_bytes == 0) &&
                   ((uintptr_t)workspace & 15) == 0,
               B200_E_INVALID, "b200_lfa_bwd: workspace of %lld bytes needed (16-byte aligned)",
               (long long)b200_lfa_bwd_workspace_bytes(n, c, kt));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  {  // c in {32, 64, 128}: every contraction on the tensor cores (lfa_tc.cu); c = 256 (lfa_tc256.cu): scores and dF
     // there, dW_att on the split-K tensor-core GEMM
    const int rc = lfa_tc_bwd_dispatch(x, pos, nbr, enc_w, enc_b, att_w, att_wt, grad_out, grad_x, grad_enc_w, grad_enc_b,
                                       grad_att_w, workspace, n, c, kt, st);
    if (rc != B200_E_UNSUPPORTED) return rc;
  }
  float* ws = static_cast<float*>(workspace);
#define X(C_, KT_, CW_, TC_, SPLIT_, ...)                                                                  \
  if (c == C_ && kt == KT_)                                                                                \
    return launch_lfa_bwd<LfaCfg<C_, KT_, CW_, TC_, ##__VA_ARGS__>, SPLIT_>(x, pos, nbr, enc_w, enc_b, att_wt, att_w, grad_out, \
                                                             grad_x, grad_enc_w, grad_enc_b, grad_att_w, ws, n, st);
  B200_LFA_BWD_CASES(X)
#undef X
  set_error("b200_lfa_bwd: unsupported (c=%d, kt=%d); c in {8,16,32,64,128,256}, kt in {16,32}", c, kt);
  return B200_E_UNSUPPORTED;
}
