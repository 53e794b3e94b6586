// Split-K weight-gradient GEMM on the 5th-generation tensor cores (tcgen05.mma kind::tf32, 3xTF32):
//     gw[m][c] += sum_i gy[i][m] * act[i][c],   gb[m] += sum_i gy[i][m]
// i.e. torch.nn.Linear's weight/bias gradients (SharedMLP, myria3d/models/modules/pyg_randla_net.py:97-109)
// and the attention-weight gradient dW_att = DA^T F of the fused LFA backward (lfa.cu).
//
// CTA = 128 output rows (m: channels of gy, one TMEM lane each) x BN output columns, one split of the row
// range.  The reduction dimension (rows i) streams through two shared-memory stages of 32 rows; both operands
// are transposed on the way in (thread <-> output row/column, 4 consecutive i per STS.128) into the K-major
// no-swizzle canonical layout of tc.cuh, split into tf32 hi/lo parts.  One thread issues 3 x 4 MMAs per stage
// (hi*hi + lo*hi + hi*lo: fp32-grade accuracy, see DESIGN.md section 4) and commits to the stage's mbarrier;
// the other threads are already loading the next stage, so global loads overlap the tensor pipe.  The fp32
// accumulator lives in TMEM (BN columns) for the whole split; the epilogue reads it back with tcgen05.ld and
// reduces into global memory (red.global.add).
#include <stdlib.h>

#include "tc.cuh"

namespace b200 {

constexpr int TCG_THREADS = 256;  // 8 warps: 2 per scheduler hide the split/store latency; warps w and w+4 share a TMEM lane quarter
constexpr int TCG_KC = 32;        // reduction rows per stage

struct CatRowsTC {  // [a1 | a2] activation rows; every segment is float4-addressable (checked by the caller)
  const float* a1;
  int64_t ld1;
  int c1;
  const float* a2;
  int64_t ld2;
  int c2;
};

__device__ __forceinline__ float4 cat_quad(const CatRowsTC& A, int64_t row, int k) {  // k % 4 == 0, k < c1 + c2
  if (k < A.c1) return __ldg(reinterpret_cast<const float4*>(A.a1 + row * A.ld1 + k));
  return __ldg(reinterpret_cast<const float4*>(A.a2 + row * A.ld2 + (k - A.c1)));
}

// 4 reduction rows x 4 output rows/columns in registers -> 4 x (hi, lo) STS.128 into the K-major operand
// layout [k-group][row][4 k].  The order in which the 4 rows are stored is rotated with the quad index so that
// the 8 lanes of a store phase hit 8 different 16-byte bank groups.
__device__ __forceinline__ void store_block(float* __restrict__ hi_base, float* __restrict__ lo_base, int rows_p1, int g,
                                            int quad, const float (&v)[4][4]) {
  // rotate the 4 rows of the block by c = (quad >> 1) & 3 with SELs (a lane-dependent register index would
  // compile to divergent branches): w[u][jj] = v[u][(jj + c) & 3]
  const int c = (quad >> 1) & 3;
  const bool r1 = (c & 1) != 0, r2 = (c & 2) != 0;
  float w[4][4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float a0 = r1 ? v[u][1] : v[u][0], a1 = r1 ? v[u][2] : v[u][1], a2 = r1 ? v[u][3] : v[u][2], a3 = r1 ? v[u][0] : v[u][3];
    w[u][0] = r2 ? a2 : a0, w[u][1] = r2 ? a3 : a1, w[u][2] = r2 ? a0 : a2, w[u][3] = r2 ? a1 : a3;
  }
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const int j = (jj + c) & 3;  // row 4*quad + j holds (k = 4g + u) -> w[u][jj]
    float4 hi, lo;
    tc::split_tf32(w[0][jj], hi.x, lo.x), tc::split_tf32(w[1][jj], hi.y, lo.y);
    tc::split_tf32(w[2][jj], hi.z, lo.z), tc::split_tf32(w[3][jj], hi.w, lo.w);
    const int off = (g * rows_p1 + 4 * quad + j) * 4;
    *reinterpret_cast<float4*>(hi_base + off) = hi;
    *reinterpret_cast<float4*>(lo_base + off) = lo;
  }
}

template <int BN>
__global__ void __launch_bounds__(TCG_THREADS, 1)
tc_tn_kernel(const float* __restrict__ gy, int cout, CatRowsTC A, float* __restrict__ gw, float* __restrict__ gb,
             float* __restrict__ partial /* [splits][cout][ncols] or nullptr (then: atomics into gw / gb) */,
             int64_t n, int64_t rows_per_split, uint32_t tmem_cols, long long* __restrict__ dbg /* nullptr in production */) {
  extern __shared__ __align__(128) float tcg_smem[];
  const bool rec = dbg && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 32;
  int nrec = 0;
#define B200_TS() do { if (rec && nrec < 120) dbg[nrec++] = clock64(); } while (0)
  B200_TS();
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t tmem_slot;
  constexpr size_t A_FLOATS = tc::operand_floats(128, TCG_KC);
  constexpr size_t B_FLOATS = tc::operand_floats(BN, TCG_KC);
  constexpr size_t STAGE_FLOATS = 2 * A_FLOATS + 2 * B_FLOATS;
  constexpr int KG = TCG_KC / 4;                      // k-groups per stage
  constexpr int PB = (BN / 4) * KG / TCG_THREADS;     // 4x4 blocks of the B operand per thread (0 for BN = 64: see below)

  const int tid = threadIdx.x, warp = tid >> 5;
  const int m0 = blockIdx.x * 128, c0 = blockIdx.y * BN;
  const int ktot = A.c1 + A.c2;
  const int ncols = ktot + (gb ? 1 : 0);
  const int64_t i_begin = (int64_t)blockIdx.z * rows_per_split;
  const int64_t i_end = (i_begin + rows_per_split < n) ? (i_begin + rows_per_split) : n;
  if (i_begin >= i_end) return;  // uniform: nothing to reduce in this split (host sizes splits so that none is empty)
  const int nchunks = (int)((i_end - i_begin + TCG_KC - 1) / TCG_KC);

  if (warp == 0) tc::tmem_alloc(&tmem_slot, tmem_cols);
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_fence_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_d = tmem_slot;
  const uint32_t idesc = tc::idesc_tf32(128, BN);
  B200_TS();  // [1] after alloc + barrier init
  bool alive = true;  // false after a barrier time-out: skip the remaining work, never hang

  // A operand block of this thread: output rows m0 + 4*aq .. +3, k-group ag (32 quads x 8 groups = 256 threads)
  const int aq = tid & 31, ag = tid >> 5;
  static_assert(128 / 4 * KG == TCG_THREADS, "one A block per thread");

  // Register-level software pipeline: the global loads of chunk s+1 are issued right after chunk s has been
  // stored to shared memory, so their DRAM latency hides behind the fences, the barrier, the MMA issue and the
  // next stage-free wait (one DRAM round trip per 32 rows would otherwise bound the kernel).
  float va[4][4];
  float vb[PB > 0 ? PB : 1][4][4];
  auto load_a = [&](int64_t i0) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = i0 + 4 * ag + u;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < i_end && m0 + 4 * aq < cout) t = __ldg(reinterpret_cast<const float4*>(gy + i * cout + m0 + 4 * aq));
      va[u][0] = t.x, va[u][1] = t.y, va[u][2] = t.z, va[u][3] = t.w;
    }
  };
  auto load_b = [&](int64_t i0, int blk, float (&v)[4][4]) {
    const int cq = blk % (BN / 4), g = blk / (BN / 4);
    const int col = c0 + 4 * cq;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = i0 + 4 * g + u;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < i_end) {
        if (col < ktot)
          t = cat_quad(A, i, col);
        else if (col == ktot && gb)
          t.x = 1.f;  // the bias-gradient column (ktot % 4 == 0: it opens a quad)
      }
      v[u][0] = t.x, v[u][1] = t.y, v[u][2] = t.z, v[u][3] = t.w;
    }
  };
  auto load_chunk = [&](int64_t i0) {
    load_a(i0);
    if constexpr (PB > 0) {
#pragma unroll
      for (int q = 0; q < PB; ++q) load_b(i0, tid + q * TCG_THREADS, vb[q]);
    } else {
      if (tid < (BN / 4) * KG) load_b(i0, tid, vb[0]);
    }
  };

  load_chunk(i_begin);
  B200_TS();  // [2] first loads issued
  for (int s = 0; s < nchunks && alive; ++s) {
    const int stage = s & 1;
    float* Ah = tcg_smem + stage * STAGE_FLOATS;
    float* Al = Ah + A_FLOATS;
    float* Bh = Al + A_FLOATS;
    float* Bl = Bh + B_FLOATS;

    // the stage may be overwritten only after the MMAs of chunk s-2 (its previous user) have completed
    if (s >= 2) {
      alive = tc::mbar_wait_bounded(&bars[stage], (uint32_t)(((s - 2) >> 1) & 1));
      alive = __syncthreads_and(alive) != 0;  // uniform verdict: nobody is left behind at the barrier below
    }
    if (!alive) break;
    B200_TS();  // [3 + 4s] stage free

    // tf32 hi/lo split + transposing stores of the chunk held in registers
    store_block(Ah, Al, 129, ag, aq, va);
    if constexpr (PB > 0) {
#pragma unroll
      for (int q = 0; q < PB; ++q) {
        const int blk = tid + q * TCG_THREADS;
        store_block(Bh, Bl, BN + 1, blk / (BN / 4), blk % (BN / 4), vb[q]);
      }
    } else {
      if (tid < (BN / 4) * KG) store_block(Bh, Bl, BN + 1, tid / (BN / 4), tid % (BN / 4), vb[0]);
    }
    B200_TS();  // [4 + 4s] stored (waited for this chunk's loads)
    if (s + 1 < nchunks) load_chunk(i_begin + (int64_t)(s + 1) * TCG_KC);  // prefetch: consumed next iteration
    B200_TS();  // [5 + 4s] next loads issued

    tc::fence_smem_to_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    B200_TS();  // [6 + 4s] after barrier
    if (tid == 0) {
      const uint32_t lbo_a = tc::lbo_bytes(128), lbo_b = tc::lbo_bytes(BN);
#pragma unroll
      for (int pass = 0; pass < 3; ++pass) {
        const uint32_t a_base = smem_u32((pass == 1) ? Al : Ah);  // hi*hi, lo*hi, hi*lo
        const uint32_t b_base = smem_u32((pass == 2) ? Bl : Bh);
#pragma unroll
        for (int ks = 0; ks < TCG_KC / 8; ++ks) {
          const uint64_t ad = tc::smem_desc(a_base + (uint32_t)(2 * ks) * lbo_a, lbo_a, tc::kSboBytes);
          const uint64_t bd = tc::smem_desc(b_base + (uint32_t)(2 * ks) * lbo_b, lbo_b, tc::kSboBytes);
          tc::mma_tf32(tmem_d, ad, bd, idesc, (s | pass | ks) != 0);
        }
      }
      tc::mma_commit(&bars[stage]);
    }
  }

  if (alive) {
    const int last = nchunks - 1;
    alive = tc::mbar_wait_bounded(&bars[last & 1], (uint32_t)((last >> 1) & 1));
  }
  alive = __syncthreads_and(alive) != 0;
  tc::fence_after_sync();
  B200_TS();  // last MMA complete
  if (alive) {
    // warp w reads TMEM lanes 32*(w%4) .. +31 (= output rows) and the column half w/4
    const int lane_q = warp & 3, half = warp >> 2;
    const int m = m0 + lane_q * 32 + (tid & 31);
    float* gw_row = gw + (int64_t)m * ktot;
    // partial mode: this split's tile goes to its own slab (plain stores); a second kernel adds the slabs up.
    // Millions of atomics onto a few hundred KB of gw cost ~40 us per GEMM whatever the math takes.
    const int ncols_pad = (ncols + 3) & ~3;  // slab rows padded to 16 bytes: float4 stores below
    float* prow = partial ? partial + ((int64_t)blockIdx.z * cout + m) * ncols_pad : nullptr;
#pragma unroll 1
    for (int cc = half * (BN / 2); cc < (half + 1) * (BN / 2); cc += 16) {
      float v[16];
      tc::tmem_ld16(tmem_d + ((uint32_t)(lane_q * 32) << 16) + (uint32_t)cc, v);
      if (m < cout) {
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int col = c0 + cc + 4 * j4;
          if (col + 3 < ktot) {
            const float4 q = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
            if (prow) {
              *reinterpret_cast<float4*>(prow + col) = q;
            } else {
              atomicAdd(reinterpret_cast<float4*>(gw_row + col), q);
            }
          } else if (col == ktot && gb) {
            if (prow)
              prow[col] = v[4 * j4];
            else
              atomicAdd(gb + m, v[4 * j4]);
          }
        }
      }
    }
  }
  B200_TS();  // epilogue done
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_d, tmem_cols);
  B200_TS();
  if (rec) dbg[127] = nrec;
#undef B200_TS
}


// gw[m][c] += sum_s partial[s][m][c] (c < ktot), gb[m] += sum_s partial[s][m][ktot]
__global__ void __launch_bounds__(256)
tc_reduce_partials_kernel(const float* __restrict__ partial, int splits, int cout, int ktot, int ncols,
                          float* __restrict__ gw, float* __restrict__ gb) {
  const int ncols_pad = (ncols + 3) & ~3;
  const int64_t total = (int64_t)cout * ncols, slab = (int64_t)cout * ncols_pad;
  for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (int64_t)gridDim.x * 256) {
    const int m = (int)(t / ncols), c = (int)(t % ncols);
    // up to 148 splits: eight independent loads in flight per thread instead of one dependent chain of L2 round trips
    const float* src = partial + (int64_t)m * ncols_pad + c;
    float acc = 0.f;
    int s = 0;
    for (; s + 8 <= splits; s += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldg(src + (int64_t)(s + u) * slab);
      acc += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    }
    for (; s < splits; ++s) acc += __ldg(src + (int64_t)s * slab);
    if (c < ktot)
      gw[(int64_t)m * ktot + c] += acc;
    else
      gb[m] += acc;
  }
}

long long* tc_debug_buffer();  // runtime.cu: b200_set_option("tc_timeline", ptr); null in production

struct TcTnPlan {
  int bn;
  int64_t splits, rows_per_split;
};

// A split accumulates its rows in one TMEM accumulator, 12 chained MMAs per 32 rows.  The tensor core's fp32 adder
// truncates (~6e-8 of the running sum per MMA, always towards zero), so a long split drifts: at myria3d's full
// 32 x 40 000-point batch the SMs / tiles plan gives 2 000+ rows per split.  Splits longer than kTcTnMaxRowsPerSplit
// (192 chained MMAs, fp32-grade) are cut into equal parts, so the grid stays a multiple of the one-wave plan.
constexpr int64_t kTcTnMaxRowsPerSplit = 512;

static TcTnPlan plan_tc_tn(int cout, int ncols, int64_t n) {
  TcTnPlan p;
  p.bn = (ncols <= 64) ? 64 : ((ncols % 256 == 0) ? 256 : 128);  // 256-wide tiles only when they divide the width
  const int64_t tiles = ceil_div(cout, 128) * ceil_div(ncols, p.bn);
  int64_t splits = (int64_t)num_sms() / tiles;
  const int64_t max_splits = ceil_div(n, 4 * TCG_KC);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int64_t rows = ceil_div(n, splits);
  if (rows > kTcTnMaxRowsPerSplit) rows = ceil_div(rows, ceil_div(rows, kTcTnMaxRowsPerSplit));
  if (rows < ceil_div(n, 65535)) rows = ceil_div(n, 65535);  // grid.z
  rows = ceil_div(rows, TCG_KC) * TCG_KC;
  p.rows_per_split = rows;
  p.splits = ceil_div(n, rows);
  return p;
}

size_t tc_tn_workspace_bytes(int cout, int ncols, int64_t n) {
  if (n <= 0) return 0;
  const TcTnPlan p = plan_tc_tn(cout, ncols, n);
  return (size_t)p.splits * cout * ((ncols + 3) & ~3) * sizeof(float);
}

template <int BN>
static int launch_tc_tn_bn(const float* gy, int cout, const CatRowsTC& A, float* gw, float* gb, float* partial,
                           const TcTnPlan& p, int64_t n, cudaStream_t st) {
  const int ktot = A.c1 + A.c2;
  const int ncols = ktot + (gb ? 1 : 0);
  const size_t smem = sizeof(float) * 2 * (2 * tc::operand_floats(128, TCG_KC) + 2 * tc::operand_floats(BN, TCG_KC));
  auto kern = tc_tn_kernel<BN>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "tc_tn smem attribute");
  dim3 grid((unsigned)ceil_div(cout, 128), (unsigned)ceil_div(ncols, BN), (unsigned)p.splits);
  uint32_t cols = 32;
  while ((int)cols < BN) cols <<= 1;
  kern<<<grid, TCG_THREADS, smem, st>>>(gy, cout, A, gw, gb, partial, n, p.rows_per_split, cols, tc_debug_buffer());
  B200_CHECK_LAUNCH("tc_tn_kernel");
  if (partial) {
    int64_t blocks = ceil_div((int64_t)cout * ncols, 256);
    if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
    tc_reduce_partials_kernel<<<(unsigned)blocks, 256, 0, st>>>(partial, (int)p.splits, cout, ktot, ncols, gw, gb);
    B200_CHECK_LAUNCH("tc_reduce_partials_kernel");
  }
  return B200_OK;
}

int launch_tc_tn(const float* gy, int cout, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2,
                 float* gw, float* gb, int64_t n, float* ws, size_t ws_bytes, cudaStream_t st) {
  const CatRowsTC A{a1, ld1, c1, a2, ld2, c2};
  const int ncols = c1 + c2 + (gb ? 1 : 0);
  const TcTnPlan p = plan_tc_tn(cout, ncols, n);
  float* partial = (ws && ws_bytes >= (size_t)p.splits * cout * ((ncols + 3) & ~3) * sizeof(float)) ? ws : nullptr;
  if (p.bn == 64) return launch_tc_tn_bn<64>(gy, cout, A, gw, gb, partial, p, n, st);
  if (p.bn == 256) return launch_tc_tn_bn<256>(gy, cout, A, gw, gb, partial, p, n, st);
  return launch_tc_tn_bn<128>(gy, cout, A, gw, gb, partial, p, n, st);
}

}  // namespace b200
