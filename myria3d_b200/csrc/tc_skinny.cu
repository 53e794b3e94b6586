// Weight / bias gradient of the NARROW Linear layers (<= 64 channels on both sides, hundreds of thousands of rows:
// every SharedMLP / fc layer of levels 0-1, pyg_randla_net.py:42,53,97-109) on the 5th-generation tensor cores:
//     gw[m][c] += sum_rows gy[row][m] * [a1 | a2][row][c],    gb[m] += sum_rows gy[row][m]
// i.e. a TN GEMM whose K dimension is the ROW index.  Both operands are row-major in HBM, i.e. "MN-major" for this
// product; 16-bit operands can be read that way from the no-swizzle shared-memory layout (tc.cuh), so a chunk of 128
// rows is converted to bf16 x 3 planes (rows = K, 16-byte vectors = 8 consecutive channels: exactly the global layout,
// no transposition) and fed to tcgen05.mma kind::f16 with BOTH operands MN-major; the six cross products give
// fp32-grade results.  The bias gradient rides along as one extra column of ones in the activation operand.
//
// Persistent CTA per SM: its slab of rows streams through a 2-stage ring (all 256 threads convert chunk t+1 while the
// tensor core multiplies chunk t: completion through tcgen05.commit -> mbarrier), the [64 x N] accumulator lives in
// TMEM (M = 64 tile: rows (m % 16) + 32 * (m / 16) of the lane space) for TSK_FLUSH chunks at a time, is then added to
// fp32 registers, and the slab's sum goes to gw / gb with one set of atomics per CTA.  Replaces the warp-streaming FMA kernel tn_skinny_kernel (0.7-1.5 TB/s algorithmic) on
// the B200 production path; that kernel stays as the `tensor_cores = 0` fallback.
#include "tc.cuh"

namespace b200 {

constexpr int TSK_THREADS = 256;
constexpr int TSK_ROWS = 128;  // rows (K) per chunk
// The tensor core's fp32 adder truncates (~6e-8 of the accumulator per instruction, always towards zero), so a TMEM
// chain's bias grows with its length.  A slab is n / 148 rows (8 650 on myria3d's 32 x 40 000-point batch: 68 chunks,
// 544 chained MMAs): every TSK_FLUSH chunks (64 chained MMAs) the accumulator is added to fp32 registers and restarted.
constexpr int TSK_FLUSH = 8;

struct TskArgs {
  const float* gy;
  int cout;
  const float* a1;
  int64_t ld1;
  int c1;
  const float* a2;
  int64_t ld2;
  int c2;
  float* gw;
  float* gb;
  int64_t n;
  int64_t rows_per_cta;
};

// MCH = 16-byte channel chunks of gy (cout <= 8 * MCH), NCH = chunks of [a1 | a2 | 1] (ktot + bias <= 8 * NCH)
template <int MCH, int NCH>
__global__ void __launch_bounds__(TSK_THREADS, 1)
tc_skinny_tn_kernel(const TskArgs p) {
  constexpr size_t G_PLANE = (size_t)MCH * (TSK_ROWS + 1) * 16, A_PLANE = (size_t)NCH * (TSK_ROWS + 1) * 16;
  constexpr size_t STAGE = 3 * (G_PLANE + A_PLANE);
  constexpr int N = NCH * 8;
  // two accumulators: the t1*t1 products in one, the five small cross products (<= 2^-8 of it) in the other: 8 instead
  // of 48 long-chain instructions per chunk (see TSK_FLUSH for the bound on the chain's length).
  constexpr uint32_t TMEM_COLS = 2 * N <= 32 ? 32 : (2 * N <= 64 ? 64 : 128);
  extern __shared__ __align__(128) unsigned char tsk_smem[];  // 2 stages (+ slack for the M = 64 read of MCH < 8 chunks)
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int ktot = p.c1 + p.c2;
  const int64_t row_begin = (int64_t)blockIdx.x * p.rows_per_cta;
  const int64_t row_end = (row_begin + p.rows_per_cta < p.n) ? row_begin + p.rows_per_cta : p.n;

  if (warp == 0) tc::tmem_alloc(&tmem_slot, TMEM_COLS);
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_fence_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_d = tmem_slot;
  const bool g_vec = (p.cout % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.gy) & 15) == 0);
  const bool a_vec = (p.c1 % 8 == 0) && (p.c2 % 8 == 0) && (p.ld1 % 4 == 0) && (p.ld2 % 4 == 0) &&
                     ((reinterpret_cast<uintptr_t>(p.a1) & 15) == 0) && (p.c2 == 0 || (reinterpret_cast<uintptr_t>(p.a2) & 15) == 0);

  // item = (row, 8 consecutive channels) of gy or of [a1 | a2 | 1]: one 16-byte vector in each of the 3 planes.
  // Consecutive lanes take consecutive rows (conflict-free shared-memory stores; every lane reads a full 32-byte sector).
  // The raw fp32 values of the NEXT chunk are loaded into registers right after the current chunk's MMAs are issued:
  // their latency hides behind the tensor core.
  constexpr int TOTAL_ITEMS = TSK_ROWS * (MCH + NCH);
  constexpr int ITEMS = (TOTAL_ITEMS + TSK_THREADS - 1) / TSK_THREADS;
  float4 ra[ITEMS], rb[ITEMS];
  auto load_chunk = [&](int64_t r0) {
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int it = tid + i * TSK_THREADS;
      ra[i] = rb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (TOTAL_ITEMS % TSK_THREADS != 0 && it >= TOTAL_ITEMS) continue;
      const int row = it % TSK_ROWS, ch = it / TSK_ROWS;
      const int64_t r = r0 + row;
      if (r >= row_end) continue;
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (ch < MCH) {
        const float* src = p.gy + r * p.cout + 8 * ch;
        if (g_vec) {
          ra[i] = __ldg(reinterpret_cast<const float4*>(src));
          rb[i] = __ldg(reinterpret_cast<const float4*>(src) + 1);
          continue;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (8 * ch + u < p.cout) v[u] = __ldg(src + u);
      } else {
        const int c0 = 8 * (ch - MCH);
        if (a_vec && c0 + 8 <= ktot) {
          const float* src = (c0 < p.c1) ? p.a1 + r * p.ld1 + c0 : p.a2 + r * p.ld2 + (c0 - p.c1);
          ra[i] = __ldg(reinterpret_cast<const float4*>(src));
          rb[i] = __ldg(reinterpret_cast<const float4*>(src) + 1);
          continue;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int c = c0 + u;
          if (c < p.c1)
            v[u] = __ldg(p.a1 + r * p.ld1 + c);
          else if (c < ktot)
            v[u] = __ldg(p.a2 + r * p.ld2 + (c - p.c1));
          else if (c == ktot)
            v[u] = 1.f;  // the bias-gradient column: sum over rows of gy
        }
      }
      ra[i] = make_float4(v[0], v[1], v[2], v[3]);
      rb[i] = make_float4(v[4], v[5], v[6], v[7]);
    }
  };
  auto store_chunk = [&](unsigned char* Gp, unsigned char* Ap) {
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int it = tid + i * TSK_THREADS;
      if (TOTAL_ITEMS % TSK_THREADS != 0 && it >= TOTAL_ITEMS) continue;
      const int row = it % TSK_ROWS, ch = it / TSK_ROWS;
      unsigned char* dst = (ch < MCH) ? Gp + ((size_t)ch * (TSK_ROWS + 1) + row) * 16
                                      : Ap + ((size_t)(ch - MCH) * (TSK_ROWS + 1) + row) * 16;
      const size_t plane = (ch < MCH) ? G_PLANE : A_PLANE;
      const float v[8] = {ra[i].x, ra[i].y, ra[i].z, ra[i].w, rb[i].x, rb[i].y, rb[i].z, rb[i].w};
      uint32_t t1[8], t2[8], t3[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) tc::split_bf16x3(v[u], t1[u], t2[u], t3[u]);
      *reinterpret_cast<uint4*>(dst) = make_uint4(tc::pack_hi16(t1[0], t1[1]), tc::pack_hi16(t1[2], t1[3]),
                                                   tc::pack_hi16(t1[4], t1[5]), tc::pack_hi16(t1[6], t1[7]));
      *reinterpret_cast<uint4*>(dst + plane) = make_uint4(tc::pack_hi16(t2[0], t2[1]), tc::pack_hi16(t2[2], t2[3]),
                                                           tc::pack_hi16(t2[4], t2[5]), tc::pack_hi16(t2[6], t2[7]));
      *reinterpret_cast<uint4*>(dst + 2 * plane) = make_uint4(tc::pack_hi16(t3[0], t3[1]), tc::pack_hi16(t3[2], t3[3]),
                                                               tc::pack_hi16(t3[4], t3[5]), tc::pack_hi16(t3[6], t3[7]));
    }
  };

  // TMEM -> registers: warp w reads lane quadrant w % 4 (row m = (lane & 15) + 16 * (w % 4)) and columns
  // (w / 4) * 16 + 32 * j .. +15 of both accumulators
  constexpr int NJ = (N + 31) / 32;
  float racc[NJ][16];
#pragma unroll
  for (int j = 0; j < NJ; ++j)
#pragma unroll
    for (int u = 0; u < 16; ++u) racc[j][u] = 0.f;
  auto drain_tmem = [&]() {
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int c0 = (warp >> 2) * 16 + 32 * j;
      if (c0 < N) {
        float v[16], w[16];
        tc::tmem_ld16(tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)c0, v);
        tc::tmem_ld16(tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(N + c0), w);
#pragma unroll
        for (int u = 0; u < 16; ++u) racc[j][u] += v[u] + w[u];
      }
    }
  };

  uint32_t phase[2] = {0, 0};
  int chunk = 0;
  if (row_begin < row_end) load_chunk(row_begin);
  for (int64_t r0 = row_begin; r0 < row_end; r0 += TSK_ROWS, ++chunk) {
    const int s = chunk & 1;
    unsigned char* Gp = tsk_smem + (size_t)s * STAGE;
    unsigned char* Ap = Gp + 3 * G_PLANE;
    if (chunk >= 2) {  // the MMAs that read this stage two chunks ago are done
      if (!tc::mbar_wait_bounded(&bars[s], phase[s], 20000000u)) __trap();
      tc::fence_after_sync();
      phase[s] ^= 1u;
    }
    store_chunk(Gp, Ap);
    if (chunk > 0 && chunk % TSK_FLUSH == 0) {
      // wait for the previous chunk's MMAs (the phase is not advanced: the wait two chunks on returns at once), add
      // the accumulator to registers; this chunk's MMAs restart it after the barrier below
      const int sp = (chunk - 1) & 1;
      if (!tc::mbar_wait_bounded(&bars[sp], phase[sp], 20000000u)) __trap();
      tc::fence_after_sync();
      drain_tmem();
    }
    tc::fence_smem_to_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    // ---- D[m][c] += sum_rows G[row][m] A[row][c]: both operands MN-major, K = 128 rows = 8 instructions x 6 passes
    if (warp == 0) {
      if (tc::elect_one_sync()) {
        constexpr uint32_t idesc = tc::idesc_bf16(64, N, /*a_mn=*/true, /*b_mn=*/true);
        const uint64_t g0 = tc::plane_desc_mn_base(smem_u32(Gp), TSK_ROWS);
        const uint64_t a0 = tc::plane_desc_mn_base(smem_u32(Ap), TSK_ROWS);
#pragma unroll
        for (int pass = 0; pass < 6; ++pass) {
          const uint64_t gd = tc::desc_advance(g0, (uint32_t)(tc::bf16x3_term_a(pass) * G_PLANE));
          const uint64_t ad = tc::desc_advance(a0, (uint32_t)(tc::bf16x3_term_b(pass) * A_PLANE));
#pragma unroll
          for (int ks = 0; ks < TSK_ROWS / 16; ++ks)
            tc::mma_bf16(tmem_d + (pass == 0 ? 0u : (uint32_t)N), tc::desc_advance(gd, ks * tc::kPlaneMnStepBytes),
                         tc::desc_advance(ad, ks * tc::kPlaneMnStepBytes), idesc, chunk % TSK_FLUSH != 0 || (pass > 1) || ks != 0);
        }
        tc::mma_commit(&bars[s]);
      }
      __syncwarp();
    }
    if (r0 + TSK_ROWS < row_end) load_chunk(r0 + TSK_ROWS);  // in flight while the tensor core works
  }
  // ---- drain, then one set of atomics per CTA
  for (int s = 0; s < 2; ++s) {
    const int pending = (chunk > s) ? 1 : 0;  // a commit of this stage is outstanding iff the stage was used at all ...
    if (pending) {
      if (!tc::mbar_wait_bounded(&bars[s], phase[s], 20000000u)) __trap();
      phase[s] ^= 1u;
    }
  }
  tc::fence_after_sync();
  if (chunk > 0) {
    drain_tmem();
    // M = 64 accumulator: row m sits in TMEM lane (m % 16) + 32 * (m / 16); warps w and w + 4 share a lane quadrant
    const int lane = tid & 31;
    const int m = (lane & 15) + 16 * (warp & 3);
    if ((lane < 16) && (m < p.cout)) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const int c0 = (warp >> 2) * 16 + 32 * j;
        if (c0 >= N) continue;
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          const int c = c0 + u;
          if (c < ktot)
            atomicAdd(p.gw + (int64_t)m * ktot + c, racc[j][u]);
          else if (c == ktot && p.gb != nullptr)
            atomicAdd(p.gb + m, racc[j][u]);
        }
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_d, TMEM_COLS);
}

template <int MCH, int NCH>
static int launch_tsk(const TskArgs& base, cudaStream_t st) {
  constexpr size_t G_PLANE = (size_t)MCH * (TSK_ROWS + 1) * 16, A_PLANE = (size_t)NCH * (TSK_ROWS + 1) * 16;
  // the M = 64 MN-major read of a gy plane with MCH < 8 chunks runs (8 - MCH) chunk strides past it: slack at the end
  constexpr size_t SLACK = (size_t)(8 - MCH) * (TSK_ROWS + 1) * 16;
  const size_t smem = 2 * 3 * (G_PLANE + A_PLANE) + SLACK;
  auto kern = tc_skinny_tn_kernel<MCH, NCH>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "tc_skinny smem attribute");
  TskArgs a = base;
  int64_t ctas = num_sms();
  const int64_t chunks = ceil_div(a.n, TSK_ROWS);
  if (ctas > chunks) ctas = chunks;
  a.rows_per_cta = ceil_div(chunks, ctas) * TSK_ROWS;
  ctas = ceil_div(a.n, a.rows_per_cta);
  kern<<<(unsigned)ctas, TSK_THREADS, smem, st>>>(a);
  B200_CHECK_LAUNCH("tc_skinny_tn_kernel");
  return B200_OK;
}

bool tc_skinny_tn_ok(int cout, int ktot, bool has_bias, int64_t n) {
  return tc_path_enabled(8) && cout >= 1 && cout <= 64 && ktot >= 1 && ktot + (has_bias ? 1 : 0) <= 64 && n >= 4096 &&
         !(cout > 32 && ktot + (has_bias ? 1 : 0) > 32);  // (64 x 64 would need 200 KB of stages: tc_tn_kernel's job)
}

int launch_tc_skinny_tn(const float* gy, int cout, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2,
                        float* gw, float* gb, int64_t n, cudaStream_t st) {
  TskArgs a{gy, cout, a1, ld1, c1, a2, ld2, c2, gw, gb, n, 0};
  const int mch = (cout + 7) / 8, nch = (c1 + c2 + (gb ? 1 : 0) + 7) / 8;
  const int nch2 = (nch <= 2) ? 2 : ((nch <= 4) ? 4 : 8);  // N = 16 / 32 / 64
#define B200_TSK(M_, N_) \
  if (mch <= M_ && nch2 == N_) return launch_tsk<M_, N_>(a, st);
  B200_TSK(2, 2) B200_TSK(2, 4) B200_TSK(2, 8) B200_TSK(4, 2) B200_TSK(4, 4) B200_TSK(4, 8) B200_TSK(8, 2) B200_TSK(8, 4)
#undef B200_TSK
  set_error("tc_skinny_tn: unsupported shape cout=%d ktot=%d", cout, c1 + c2);
  return B200_E_UNSUPPORTED;
}

}  // namespace b200
