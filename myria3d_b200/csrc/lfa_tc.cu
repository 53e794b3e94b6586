// Fused LocSE + attentive pooling, FORWARD and BACKWARD, with every contraction on the 5th-generation tensor cores
// (tcgen05.mma kind::f16 on fp16 x 2 split operands = fp32-grade products, accumulators in TMEM) -- the
// c in {32, 64, 128} levels of LocalFeatureAggregation (myria3d/models/modules/pyg_randla_net.py:121-152).
// Production path of b200_lfa_fwd / b200_lfa_bwd for these widths; narrower levels (c = 8, 16: K = 8 / 16
// contractions) stay on the FMA kernels of lfa.cu; c = 256 runs on lfa_tc256.cu (W_att streamed from L2 per tile).
//
// Orientation: CHANNELS on the 128 TMEM lanes, the tile's EDGES on the TMEM columns.  An epilogue thread owns one
// channel and reads, per centre, KT consecutive columns = the neighbours of that centre: the neighbourhood softmax
// and the weighted sum are thread-local register reductions (no shuffles, no atomics), exactly like the FMA kernel.
// For c < 128 the rows of W_att are REPLICATED 128 / c times along the M dimension, so that all 128 lanes (and all
// four lane quadrants = all warps) carry useful scores; replica r serves its own subset of the tile's centres.
//
// One persistent CTA per SM = 2 independent SLOTS of 256 threads (8 warps: 2 per TMEM lane quadrant).  A slot owns a
// tile (NE edges = NE / KT centres) at a time, its operand buffers, its TMEM columns and its mbarriers, and is
// synchronised with named barriers only, so the tensor-core phases of one slot overlap the gather / epilogue phases
// of the other; W_att (the largest operand) is staged once and shared.
//
// Operands are fp16 x 2 (v = hi + lo, three cross products hi*hi + lo*hi + hi*lo per contraction: 2^-22 relative in
// fp16's normal range).  The data is kept in that range by construction: F = BatchNorm + LeakyReLU outputs and the
// encoding (O(1)); W_att is staged as 16 * W; the softmax gradient dA is multiplied by a power of two derived from
// max |grad_out| (one 4-byte reduction kernel in front of the backward), undone when the results leave the SM.
// (bf16 x 3 with six products was measured first: same accuracy, twice the tensor-core instructions and 1.5x the
// shared memory -- the backward was tensor-pipe bound at 49 + N/2 cycles per instruction.)
//     W_att  in TENSOR MEMORY as the A operand (lanes = replicated row, 2 planes of c/2 columns): "Wk" = W[n][m] for
//            MMA1 and, for c <= 64, "Wm" = W^T for MMA3 (c = 128: MMA3 reads a shared-memory copy MN-major).  Staged
//            once per CTA with tcgen05.st; only the B operand travels from shared memory per instruction
//            (measured: 22 + N/2 cycles per M128 x N x K16 instruction against 50 + N/2 with A in shared memory).
//     F      shared-memory planes (tc.cuh: 16-byte vectors of 8 elements along the "chunked" dimension, rows 16 bytes
//            apart), rows = edge e, chunked along m; per slot, rebuilt per tile (x_j gather | lrelu(enc_w . q + enc_b))
//     dA     planes with rows = channel n, chunked along e; per slot, backward only: softmax gradient, written by the
//            epilogue threads
// and F, dA are read BOTH ways by the tensor core -- K-major (rows = M/N index) and MN-major (rows = K index) -- so that
// no per-tile operand is ever transposed or copied (16-bit operands only: see tc.cuh):
//     MMA1  S [n][e]  = sum_m W[n][m]  F[e][m]      A = Wk (TMEM),     B = F  (K-major)      scores
//     MMA3  dF[m][e] += sum_n W[n][m] dA[e][n]      A = Wm (TMEM),     B = dA (MN-major)     accumulator pre-loaded
//                                                                                             with s*go by tcgen05.st
//     MMA4  dW[n][m] += sum_e dA[e][n] F[e][m]      A = dA (K-major),  B = F  (MN-major)     TMEM-resident across the
//                                                   tiles of the slot; M = 64 tile for c <= 64; issued behind MMA3 and
//                                                   completing under E3 / scatter / the next tile's prologue
// The attention-weight gradient therefore never leaves the SM per tile (round 1 streamed two [E, c] tensors through
// HBM for it: 370 MB at c = 64); it is flushed with vector reductions every LTC_FLUSH tiles, which also bounds the
// length of the fp32 accumulation chain inside the tensor core (its adder truncates: ~6e-8 relative bias per step).
//
// Per tile (backward): build F -> MMA1 -> E1: softmax, o, dA -> smem, s*go -> TMEM -> MMA3 + MMA4 -> E3: encoder
// gradients in registers (carried across tiles), x-gradients transposed through shared memory and scattered with
// 16-byte vector reductions.  The epilogue threads take the fp32 feature values they need (weighted sum, f - o) from
// where they are exact: x_j straight from global memory (32 lanes = 32 consecutive channels = one 128-byte line,
// L1-resident from the build) and the encoding recomputed from the 7 geometry numbers.
#include <math_constants.h>

#include <type_traits>

#include "lfa_tc.cuh"

namespace b200 {

constexpr int LTC_SLOTS = 2;
constexpr int LTC_SLOT_THREADS = 256;
constexpr int LTC_THREADS = LTC_SLOTS * LTC_SLOT_THREADS;
constexpr int LTC_WPQ = LTC_SLOT_THREADS / 128;  // warps per TMEM lane quadrant in a slot
constexpr int LTC_FLUSH = 8;                     // tiles between two flushes of the dW accumulator
long long* tc_debug_buffer();                    // runtime.cu

template <int C, int NE, int KT, bool BWD>
struct LtcPlan {
  static constexpr int H = C / 2, H8 = H / 8, TC = NE / KT;
  static constexpr int R = 128 / C;                // replicas of W_att along M
  static constexpr int WORKERS = R * LTC_WPQ;      // (replica, warp-of-quadrant) pairs sharing a tile's centres
  static constexpr int CPT = TC / WORKERS;         // centres per epilogue thread and tile
  // W_att lives in TENSOR MEMORY as the A operand of MMA1 (lanes = replicated n, K = m: "Wk") and, for c <= 64, of
  // MMA3 (lanes = replicated m, K = n: "Wm"): 2 planes of C/2 columns each (two fp16 per column).  Only for c = 128,
  // where both do not fit beside the accumulators, MMA3 reads Wm from shared memory (MN-major view of W_att[n][m]).
  static constexpr bool WM_IN_TMEM = (C <= 64);
  static constexpr int M4 = (C == 128) ? 128 : 64;  // M of the dW tile (MMA4)
  static constexpr uint32_t W_PLANE_COLS = C / 2;
  static constexpr uint32_t W_COLS = 2 * W_PLANE_COLS * ((BWD && WM_IN_TMEM) ? 2 : 1);
  static constexpr size_t WM_PLANE = (BWD && !WM_IN_TMEM) ? (size_t)(C / 8) * (C + 1) * 16 : 0;  // rows n, chunks m
  static constexpr size_t F_PLANE = (size_t)(C / 8) * (NE + 1) * 16;
  static constexpr size_t DA_PLANE = (size_t)(NE / 8) * (C + 1) * 16;
  static constexpr size_t T_BYTES = tc::operand_floats(NE, H) * 4;  // fp32 [H/4][NE+1][4]: x-gradient transposition
  // shared part
  static constexpr size_t OFF_WM = 0;
  static constexpr size_t OFF_EW = OFF_WM + 2 * WM_PLANE;
  static constexpr size_t SHARED_BYTES = OFF_EW + 16 * 17 * (size_t)(H / 8);  // [H/8][17] float4 (1 pad)
  // per-slot part: dA | F | T | Q P | NB DEG.  The M = 128 read of the dA planes (c < 128 rows) runs past the end of
  // the last chunk into the next plane / F (garbage in dW lanes >= c that nobody reads): F follows dA.
  static constexpr size_t S_DA = 0;
  static constexpr size_t S_F = S_DA + (BWD ? 2 * DA_PLANE : 0);
  static constexpr size_t S_T = S_F + 2 * F_PLANE;
  static constexpr size_t S_Q = S_T + (BWD ? T_BYTES : 0);
  static constexpr size_t S_P = S_Q + 16 * (size_t)NE;
  static constexpr size_t S_NB = S_P + 16 * (size_t)TC;
  static constexpr size_t S_DEG = S_NB + 4 * (size_t)NE;
  static constexpr size_t SLOT_BYTES = S_DEG + 16 * ((TC + 3) / 4);
  static constexpr size_t SMEM_BYTES = SHARED_BYTES + LTC_SLOTS * SLOT_BYTES;
  static constexpr uint32_t SLOT_COLS = NE + (BWD ? C : 0);  // scores / dF accumulator | dW accumulator
  static constexpr uint32_t TMEM_COLS_NEEDED = W_COLS + LTC_SLOTS * SLOT_COLS;
  static constexpr uint32_t TMEM_COLS = TMEM_COLS_NEEDED <= 32    ? 32
                                        : TMEM_COLS_NEEDED <= 64  ? 64
                                        : TMEM_COLS_NEEDED <= 128 ? 128
                                        : TMEM_COLS_NEEDED <= 256 ? 256
                                                                  : 512;
  static_assert(C == 32 || C == 64 || C == 128, "channels (replicated) fill the 128 TMEM lanes");
  static_assert(KT == 16 || KT == 32, "neighbour slots");
  static_assert(NE % 32 == 0 && NE <= 256 && TC % WORKERS == 0 && CPT >= 1, "tile shape");
  static_assert(TMEM_COLS_NEEDED <= 512, "TMEM columns");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
  static_assert(SHARED_BYTES % 16 == 0 && SLOT_BYTES % 16 == 0, "alignment");
};

__device__ __forceinline__ void slot_sync(int slot) {
  asm volatile("bar.sync %0, %1;" ::"r"(1 + slot), "r"(LTC_SLOT_THREADS) : "memory");
}

// 4-byte scratch word of the backward: bit pattern of max |grad_out| (non-negative floats order like unsigned ints)
__global__ void __launch_bounds__(256)
lfa_absmax_kernel(const float* __restrict__ g, int64_t count, uint32_t* __restrict__ out) {
  float m = 0.f;
  const int64_t n4 = count / 4;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += (int64_t)gridDim.x * 256) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * 256 + threadIdx.x; i < count; i += (int64_t)gridDim.x * 256) m = fmaxf(m, fabsf(g[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

template <int C, int NE, int KT, bool BWD>
__global__ void __launch_bounds__(LTC_THREADS, 1)
lfa_tc_kernel(const float* __restrict__ x, const float* __restrict__ pos, const int32_t* __restrict__ nbr,
              const float* __restrict__ enc_w, const float* __restrict__ enc_b,
              const float* __restrict__ att_w /* backward: W_att [n][m] (may be null in the forward) */,
              const float* __restrict__ att_wt /* att_wt [m][n] = W_att[n][m] */,
              float* __restrict__ out,                                                   // forward
              const float* __restrict__ grad_out, float* __restrict__ grad_x,            // backward
              float* __restrict__ grad_enc_w, float* __restrict__ grad_enc_b, float* __restrict__ grad_att_w,
              const uint32_t* __restrict__ absmax_bits /* backward: max |grad_out| as float bits */,
              int64_t n, int64_t ntiles, long long* __restrict__ dbg) {
  using Plan = LtcPlan<C, NE, KT, BWD>;
  // power-of-two scale of the softmax gradient (backward): gscale = 2^(128 - e) for max |grad_out| in [2^(e-127), 2^(e-126))
  float gscale = 1.f, inv_gscale = 1.f;
  if constexpr (BWD) {
    const uint32_t e = (*absmax_bits) >> 23;
    if (e >= 24u && e <= 250u) {
      gscale = __uint_as_float((255u - e) << 23);
      inv_gscale = __uint_as_float((e - 1u) << 23);
    }
  }
  const float inv_dscale = inv_gscale / (kWScale * kWScale);  // dF accumulator carries gscale * kWScale^2
  inv_gscale /= kWScale;                                     // dW accumulator carries gscale * kWScale
  (void)inv_dscale;
  constexpr int H = Plan::H, H8 = Plan::H8, TC = Plan::TC, R = Plan::R, CPT = Plan::CPT;
  constexpr int ST = LTC_SLOT_THREADS;
  extern __shared__ __align__(128) unsigned char ltc_smem[];
  __shared__ __align__(8) uint64_t bars[LTC_SLOTS][3];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, slot = tid / ST, stid = tid % ST;
  const int swarp = stid >> 5, lane = tid & 31;

  unsigned char* Wm = ltc_smem + Plan::OFF_WM;  // 2 planes (backward, c = 128 only)
  // encoder weights [H/8 channel groups][8 channels][2]: (w0..w3), (w4, w5, w6, bias); one float4 of padding per
  // group: the H/8 groups read together by a quarter-warp of the build land in different banks
  float4* EW = reinterpret_cast<float4*>(ltc_smem + Plan::OFF_EW);
  unsigned char* sbase = ltc_smem + Plan::SHARED_BYTES + (size_t)slot * Plan::SLOT_BYTES;
  unsigned char* dAp = sbase + Plan::S_DA;  // 2 planes of DA_PLANE bytes
  unsigned char* Fp = sbase + Plan::S_F;    // 2 planes of F_PLANE bytes
  float* T = reinterpret_cast<float*>(sbase + Plan::S_T);
  float4* Q = reinterpret_cast<float4*>(sbase + Plan::S_Q);  // (p_j, dist) per edge
  float4* P = reinterpret_cast<float4*>(sbase + Plan::S_P);  // p_i per centre
  int* NB = reinterpret_cast<int*>(sbase + Plan::S_NB);
  int* DEG = reinterpret_cast<int*>(sbase + Plan::S_DEG);

  int nts = 0;
#define LTC_TS()                                                                            \
  do {                                                                                      \
    if (dbg != nullptr && blockIdx.x == 0 && tid == 0 && nts < 120) dbg[nts++] = clock64(); \
  } while (0)
  LTC_TS();

  // ---- shared-memory copy of W_att[n][m] for the MN-major read of MMA3 (backward, c = 128)
  if constexpr (BWD && !Plan::WM_IN_TMEM) {
    for (int idx = tid; idx < C * (C / 8); idx += LTC_THREADS) {
      const int nn = idx % C, j = idx / C;  // consecutive lanes = consecutive rows: conflict-free 16-byte stores
      const float4 a = __ldg(reinterpret_cast<const float4*>(att_w + (int64_t)nn * C + 8 * j));
      const float4 b = __ldg(reinterpret_cast<const float4*>(att_w + (int64_t)nn * C + 8 * j + 4));
      const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      float vs[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) vs[u] = v[u] * kWScale;
      uint4 p[2];
      tc::split8_f16x2(vs, p[0], p[1]);
#pragma unroll
      for (int t = 0; t < 2; ++t)
        *reinterpret_cast<uint4*>(Wm + t * Plan::WM_PLANE + ((size_t)j * (C + 1) + nn) * 16) = p[t];
    }
  }
  for (int idx = tid; idx < H; idx += LTC_THREADS) {
    const float* w = enc_w + idx * 7;
    EW[17 * (idx >> 3) + 2 * (idx & 7)] = make_float4(__ldg(w), __ldg(w + 1), __ldg(w + 2), __ldg(w + 3));
    EW[17 * (idx >> 3) + 2 * (idx & 7) + 1] = make_float4(__ldg(w + 4), __ldg(w + 5), __ldg(w + 6), __ldg(enc_b + idx));
  }

  if (tid < 32) tc::tmem_alloc(&tmem_slot, Plan::TMEM_COLS);
  if (stid == 0) {
    mbar_init(&bars[slot][0], 1);
    mbar_init(&bars[slot][1], 1);
    mbar_init(&bars[slot][2], 1);
    mbar_fence_init();
  }
  tc::fence_smem_to_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_wk = tmem_slot;                                   // A of MMA1: 2 planes x C/2 columns
  const uint32_t tmem_wm = tmem_slot + 2 * Plan::W_PLANE_COLS;          // A of MMA3 (c <= 64, backward)
  const uint32_t tmem_s = tmem_slot + Plan::W_COLS + (uint32_t)slot * Plan::SLOT_COLS;  // scores S / dF accumulator
  const uint32_t tmem_dw = tmem_s + (uint32_t)NE;                        // dW accumulator: C columns (backward)
  uint64_t* bar1 = &bars[slot][0];
  uint64_t* bar3 = &bars[slot][1];
  uint64_t* bar4 = &bars[slot][2];  // MMA4 (dW) completes behind E3 / scatter / the next tile's B1
  uint32_t phase = 0, phase4 = 0;
  bool mma4_pending = false;
  auto wait_mma4 = [&]() {
    if (mma4_pending) {
      tc::mbar_wait_or_trap(bar4, phase4);
      tc::fence_after_sync();
      phase4 ^= 1u;
      mma4_pending = false;
    }
  };

  // epilogue role: TMEM lane (quadrant q = warp % 4), channel = lane % C, replica = lane / C; the WORKERS
  // (replica, warp-of-quadrant) pairs take the centres g = worker, worker + WORKERS, ...
  const int lq = swarp & 3, wq = swarp >> 2;
  const int tl = lq * 32 + lane;  // TMEM lane
  const int ch = tl % C;
  const int worker = (tl / C) * LTC_WPQ + wq;
  const uint32_t lane_base = (uint32_t)(lq * 32) << 16;
  // ---- W_att into tensor memory (slot 0: the first warp of each lane quadrant writes Wk, the second one Wm).
  // lane tl holds row (tl % C): Wk[n][k = m] = W_att[n][m], Wm[m][k = n] = W_att[n][m].
  if (slot == 0 && (wq == 0 || (BWD && Plan::WM_IN_TMEM))) {
    const bool is_wk = (wq == 0);
    // lane = row ch of the operand; consecutive lanes read consecutive addresses in both cases:
    //   Wk[n][k = m] = W_att[n][m] = att_wt[m * C + n],   Wm[m][k = n] = W_att[n][m] = att_w[n * C + m]
    const float* src = is_wk ? att_wt : att_w;
#pragma unroll 1
    for (int k0 = 0; k0 < C; k0 += 32) {
      float v[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = kWScale * __ldg(src + (int64_t)(k0 + i) * C + ch);
      tc::tmem_st_row32_f16x2((is_wk ? tmem_wk : tmem_wm) + lane_base + (uint32_t)k0 / 2, Plan::W_PLANE_COLS, v);
    }
    tc::tmem_st_wait();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  float4 mw0 = make_float4(0.f, 0.f, 0.f, 0.f), mw1 = mw0;  // encoder weights of this thread's channel (ch >= H)
  if (ch >= H) {
    mw0 = EW[17 * ((ch - H) >> 3) + 2 * ((ch - H) & 7)];
    mw1 = EW[17 * ((ch - H) >> 3) + 2 * ((ch - H) & 7) + 1];
  }

  float gw[8];  // encoder-gradient partials of channel ch (>= H), carried across tiles
#pragma unroll
  for (int t = 0; t < 8; ++t) gw[t] = 0.f;
  int tiles_since_flush = 0;
  const int64_t tile_stride = (int64_t)gridDim.x * LTC_SLOTS;
  // thread e < NE keeps the neighbour id and the centre position of edge e of the NEXT tile in registers
  int pf_j = -1;
  float4 pf_p = make_float4(0.f, 0.f, 0.f, 0.f);
  auto prefetch = [&](int64_t t) {
    pf_j = -1;
    pf_p = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t i = t * TC + stid / KT;
    if (t < ntiles && i < n) {
      pf_j = __ldg(nbr + i * KT + stid % KT);
      pf_p = make_float4(__ldg(pos + 3 * i), __ldg(pos + 3 * i + 1), __ldg(pos + 3 * i + 2), 0.f);
    }
  };
  if (stid < NE) prefetch((int64_t)blockIdx.x * LTC_SLOTS + slot);
  LTC_TS();

  for (int64_t tile = (int64_t)blockIdx.x * LTC_SLOTS + slot; tile < ntiles; tile += tile_stride) {
    const int64_t tile_base = tile * TC;
    // ---- B1: neighbour ids (prefetched during the previous tile), geometry, degrees
    if (stid < NE) {
      const int e = stid, g = e / KT, kk = e % KT;
      const int j = pf_j;
      const float4 pv = pf_p;
      float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j >= 0) {
        const float pjx = __ldg(pos + 3 * (int64_t)j), pjy = __ldg(pos + 3 * (int64_t)j + 1), pjz = __ldg(pos + 3 * (int64_t)j + 2);
        const float dx = pjx - pv.x, dy = pjy - pv.y, dz = pjz - pv.z;
        qv = make_float4(pjx, pjy, pjz, sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz))));
      }
      NB[e] = j;
      Q[e] = qv;
      const unsigned valid = __ballot_sync(0xffffffffu, j >= 0);  // NE % 32 == 0: whole warps take this branch
      if (kk == 0) {
        P[g] = pv;
        DEG[g] = (KT == 32) ? __popc(valid) : __popc((valid >> (lane & 16)) & 0xffffu);
      }
      prefetch(tile + tile_stride);  // in flight until the next tile's B1
    }
    if constexpr (BWD) wait_mma4();  // the previous tile's dW MMAs still read F and dA
    slot_sync(slot);
    LTC_TS();
    // ---- B2 / B3: F = [x_j ; lrelu(enc_w . q + enc_b)]
    ltc_build_f<NE, KT, H, ST>(stid, x, NB, P, Q, EW, Fp, Plan::F_PLANE);
    tc::fence_smem_to_async();
    tc::fence_before_sync();
    slot_sync(slot);
    tc::fence_after_sync();
    LTC_TS();

    // ---- MMA1: S[n][e] = sum_m W[n][m] F[e][m]   (three fp16 cross products)
    if (swarp == 0) {
      if (tc::elect_one_sync()) {
        constexpr uint32_t idesc = tc::idesc_f16(128, NE);
        const uint64_t bd0 = tc::plane_desc_k_base(smem_u32(Fp), NE);
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t a_tmem = tmem_wk + (uint32_t)tc::f16x2_term_a(pass) * Plan::W_PLANE_COLS;
          const uint64_t bd = tc::desc_advance(bd0, (uint32_t)(tc::f16x2_term_b(pass) * Plan::F_PLANE));
#pragma unroll
          for (int k0 = 0; k0 < C; k0 += 16)
            tc::mma_bf16_ts(tmem_s, a_tmem + (uint32_t)k0 / 2, tc::desc_advance(bd, (k0 / 16) * tc::plane_k_step_bytes(NE)), idesc,
                            (pass | k0) != 0);
        }
        tc::mma_commit(bar1);
      }
      __syncwarp();
    }
    tc::mbar_wait_or_trap(bar1, phase);
    tc::fence_after_sync();
    LTC_TS();

    // ---- E1: thread = (channel, replica); softmax over the neighbourhood, pooled output, (backward) softmax gradient
    // (a full neighbourhood -- the common case -- takes the copy of the body without the k < deg predicates)
    auto e1_centre = [&](const int g, const int deg, auto full_tag) {
      constexpr bool FULL = decltype(full_tag)::value;
      float a[KT], f[KT];
      float go_v = 0.f;  // (backward) issued first: its latency hides behind the softmax
      if constexpr (BWD) {
        if (tile_base + g < n) go_v = __ldg(grad_out + (tile_base + g) * C + ch);
      }
      (void)go_v;
#pragma unroll
      for (int k0 = 0; k0 < KT; k0 += 16) {
        float v[16];
        tc::tmem_ld16(tmem_s + lane_base + (uint32_t)(g * KT + k0), v);
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k0 + k] = v[k];
      }
      const int64_t i = tile_base + g;
      // the fp32 feature of (edge, this channel): gathered x_j or the recomputed encoding (same operation order as
      // the build: bit-identical to the value the tensor core saw, before the fp16 split)
      if (ch < H) {
#pragma unroll
        for (int k = 0; k < KT; ++k) {
          const int j = NB[g * KT + k];
          f[k] = (j >= 0) ? __ldg(x + (int64_t)j * H + ch) : 0.f;
        }
      } else {
        const float4 p = P[g];
        const float sp = fmaf(mw0.z, p.z, fmaf(mw0.y, p.y, fmaf(mw0.x, p.x, mw1.w)));
#pragma unroll
        for (int k = 0; k < KT; ++k) {
          const float4 q = Q[g * KT + k];
          float s = sp;
          s = fmaf(mw0.w, q.x, s), s = fmaf(mw1.x, q.y, s), s = fmaf(mw1.y, q.z, s);
          s = fmaf(mw1.z, q.w, s);
          f[k] = (FULL || k < deg) ? lrelu(s, kLReluSlope) : 0.f;
        }
      }
      float mx = -CUDART_INF_F;
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (FULL || k < deg) mx = fmaxf(mx, a[k]);
      const float neg_mx = -mx * kLog2eOverWScale;
      float sum = 0.f, o = 0.f;
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        // (scores carry kWScale: exp(a / 16 - mx / 16) as one FFMA + ex2)
        const float p = (FULL || k < deg) ? tc::ex2_approx(fmaf(a[k], kLog2eOverWScale, neg_mx)) : 0.f;
        a[k] = p;
        sum += p;
        o = fmaf(p, f[k], o);
      }
      const float inv = 1.f / (sum + 1e-16f);
      o *= inv;
      if constexpr (!BWD) {
        if (i < n) out[i * C + ch] = o;
      } else {
        // everything downstream of grad_out carries the power-of-two gscale (max |grad_out| * gscale in [2, 4), times kWScale below): the
        // softmax gradient then sits in fp16's normal range whatever the loss scale is; undone in E3 / the dW flush
        // dA is stored as kWScale * gscale * dA: the accumulators of MMA3 / MMA4 then carry kWScale^2 * gscale and
        // kWScale * gscale (3 instead of 4 operations per edge here)
        const float gi = inv * go_v * (gscale * kWScale);
#pragma unroll
        for (int k8 = 0; k8 < KT; k8 += 8) {
          float da[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float sg = a[k8 + u] * gi;  // kWScale * s * go (0 for invalid edges: p = 0)
            da[u] = sg * (f[k8 + u] - o);     // kWScale * gradient w.r.t. the score
            a[k8 + u] = sg * kWScale;         // direct term of dF at the accumulator's scale kWScale^2 * gscale
          }
          uint4 p1, p2;
          tc::split8_f16x2(da, p1, p2);
          const size_t off = ((size_t)((g * KT + k8) >> 3) * (C + 1) + ch) * 16;
          *reinterpret_cast<uint4*>(dAp + off) = p1;
          *reinterpret_cast<uint4*>(dAp + Plan::DA_PLANE + off) = p2;
        }
#pragma unroll
        for (int k0 = 0; k0 < KT; k0 += 16) {
          float v[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] = a[k0 + k];
          tc::tmem_st16(tmem_s + lane_base + (uint32_t)(g * KT + k0), v);  // dF accumulator <- s * go
        }
      }
    };
#pragma unroll 1
    for (int ci = 0; ci < CPT; ++ci) {
      const int g = worker + ci * Plan::WORKERS;
      const int deg = DEG[g];
      if (deg == KT)
        e1_centre(g, deg, std::true_type{});
      else
        e1_centre(g, deg, std::false_type{});
    }
    if constexpr (!BWD) {
      tc::fence_before_sync();
      slot_sync(slot);  // TMEM and the F tile are free for the next tile
      tc::fence_after_sync();
      LTC_TS();
    } else {
      tc::tmem_st_wait();
      tc::fence_smem_to_async();
      tc::fence_before_sync();
      slot_sync(slot);
      tc::fence_after_sync();
      LTC_TS();

      // ---- MMA3: dF[m][e] += sum_n W[n][m] dA[e][n];  MMA4: dW[n][m] += sum_e dA[e][n] F[e][m]
      if (swarp == 0) {
        if (tc::elect_one_sync()) {
          const uint64_t da_mn0 = tc::plane_desc_mn_base(smem_u32(dAp), C);
          if constexpr (Plan::WM_IN_TMEM) {
            constexpr uint32_t idesc = tc::idesc_f16(128, NE, /*a_mn=*/false, /*b_mn=*/true);
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
              const uint32_t a_tmem = tmem_wm + (uint32_t)tc::f16x2_term_a(pass) * Plan::W_PLANE_COLS;
              const uint64_t bd = tc::desc_advance(da_mn0, (uint32_t)(tc::f16x2_term_b(pass) * Plan::DA_PLANE));
#pragma unroll
              for (int k0 = 0; k0 < C; k0 += 16)
                tc::mma_bf16_ts(tmem_s, a_tmem + (uint32_t)k0 / 2, tc::desc_advance(bd, (k0 / 16) * tc::kPlaneMnStepBytes), idesc, true);
            }
          } else {
            constexpr uint32_t idesc = tc::idesc_f16(128, NE, /*a_mn=*/true, /*b_mn=*/true);
            const uint64_t wm0 = tc::plane_desc_mn_base(smem_u32(Wm), C);
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
              const uint64_t ad = tc::desc_advance(wm0, (uint32_t)(tc::f16x2_term_a(pass) * Plan::WM_PLANE));
              const uint64_t bd = tc::desc_advance(da_mn0, (uint32_t)(tc::f16x2_term_b(pass) * Plan::DA_PLANE));
#pragma unroll
              for (int k0 = 0; k0 < C; k0 += 16)
                tc::mma_bf16(tmem_s, tc::desc_advance(ad, (k0 / 16) * tc::kPlaneMnStepBytes),
                             tc::desc_advance(bd, (k0 / 16) * tc::kPlaneMnStepBytes), idesc, true);
            }
          }
          tc::mma_commit(bar3);
          {
            // c <= 64: an M = 64 tile (half the A-operand traffic; rows land in lanes (n % 16) + 32 * (n / 16))
            constexpr uint32_t idesc = tc::idesc_f16(Plan::M4, C, /*a_mn=*/false, /*b_mn=*/true);
            const uint64_t da_k0 = tc::plane_desc_k_base(smem_u32(dAp), C);
            const uint64_t f_mn0 = tc::plane_desc_mn_base(smem_u32(Fp), NE);
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
              const uint64_t ad = tc::desc_advance(da_k0, (uint32_t)(tc::f16x2_term_a(pass) * Plan::DA_PLANE));
              const uint64_t bd = tc::desc_advance(f_mn0, (uint32_t)(tc::f16x2_term_b(pass) * Plan::F_PLANE));
#pragma unroll
              for (int k0 = 0; k0 < NE; k0 += 16)
                tc::mma_bf16(tmem_dw, tc::desc_advance(ad, (k0 / 16) * tc::plane_k_step_bytes(C)),
                             tc::desc_advance(bd, (k0 / 16) * tc::kPlaneMnStepBytes), idesc, tiles_since_flush != 0 || (pass | k0) != 0);
            }
          }
          tc::mma_commit(bar4);
        }
        __syncwarp();
      }
      mma4_pending = true;
      tc::mbar_wait_or_trap(bar3, phase);
      tc::fence_after_sync();
      LTC_TS();

      // ---- E3: thread = (channel m, replica); encoder gradients stay in registers, x-gradients go through T
      auto e3_centre = [&](const int g, const int deg, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        float d[KT];
#pragma unroll
        for (int k0 = 0; k0 < KT; k0 += 16) {
          float v[16];
          tc::tmem_ld16(tmem_s + lane_base + (uint32_t)(g * KT + k0), v);
#pragma unroll
          for (int k = 0; k < 16; ++k) d[k0 + k] = v[k];
        }
        if (ch < H) {
          const int toff = ((ch >> 2) * (NE + 1) + g * KT) * 4 + (ch & 3);
#pragma unroll
          for (int k = 0; k < KT; ++k) T[toff + 4 * k] = d[k] * inv_dscale;
        } else {
          const float4 p = P[g];
          const float sp = fmaf(mw0.z, p.z, fmaf(mw0.y, p.y, fmaf(mw0.x, p.x, mw1.w)));
          float gsum = 0.f;
#pragma unroll
          for (int k = 0; k < KT; ++k)
            if (FULL || k < deg) {
              const float4 q = Q[g * KT + k];
              float s = sp;  // lrelu'(z) from the recomputed pre-activation
              s = fmaf(mw0.w, q.x, s), s = fmaf(mw1.x, q.y, s), s = fmaf(mw1.y, q.z, s);
              s = fmaf(mw1.z, q.w, s);
              const float dz = d[k] * (s > 0.f ? inv_dscale : inv_dscale * kLReluSlope);
              gw[3] = fmaf(dz, q.x, gw[3]);
              gw[4] = fmaf(dz, q.y, gw[4]);
              gw[5] = fmaf(dz, q.z, gw[5]);
              gw[6] = fmaf(dz, q.w, gw[6]);
              gsum += dz;
            }
          gw[0] = fmaf(gsum, p.x, gw[0]);
          gw[1] = fmaf(gsum, p.y, gw[1]);
          gw[2] = fmaf(gsum, p.z, gw[2]);
          gw[7] += gsum;
        }
      };
#pragma unroll 1
      for (int ci = 0; ci < CPT; ++ci) {
        const int g = worker + ci * Plan::WORKERS;
        const int deg = DEG[g];
        if (deg == KT)
          e3_centre(g, deg, std::true_type{});
        else
          e3_centre(g, deg, std::false_type{});
      }
      ++tiles_since_flush;
      const bool last_tile = tile + tile_stride >= ntiles;
      if (tiles_since_flush == LTC_FLUSH || last_tile) {
        wait_mma4();
        // dW[n][m] of this slot: M = 128: lane = row n; M = 64: row n sits in lane (n % 16) + 32 * (n / 16).
        // The warps of a lane quadrant split the columns.
        const int n_row = (Plan::M4 == 128) ? tl : (tl & 15) + 16 * (tl >> 5);
        const bool quad_has_rows = (Plan::M4 == 128) ? (lq * 32 < C) : (lq * 16 < C);  // warp-uniform
        if (quad_has_rows) {
          for (int c0 = wq * (C / LTC_WPQ); c0 < (wq + 1) * (C / LTC_WPQ); c0 += 16) {
            float v[16];
            tc::tmem_ld16(tmem_dw + lane_base + (uint32_t)c0, v);
            if ((Plan::M4 == 128 || (tl & 31) < 16) && n_row < C) {
              float4* dst = reinterpret_cast<float4*>(grad_att_w + (int64_t)n_row * C + c0);
#pragma unroll
              for (int u = 0; u < 4; ++u)
                atomicAdd(dst + u, make_float4(v[4 * u] * inv_gscale, v[4 * u + 1] * inv_gscale, v[4 * u + 2] * inv_gscale,
                                               v[4 * u + 3] * inv_gscale));
            }
          }
        }
        tiles_since_flush = 0;
      }
      tc::fence_before_sync();
      slot_sync(slot);
      tc::fence_after_sync();
      LTC_TS();
      // ---- scatter the x-gradients
      ltc_scatter_x<NE, H, ST>(stid, T, NB, grad_x);
      // the next tile's B1 only writes NB / Q / P / DEG, all of which the scatter above still reads
      slot_sync(slot);
      LTC_TS();
    }
    phase ^= 1u;
  }

  if constexpr (BWD) {
    if (ch >= H) {
#pragma unroll
      for (int t = 0; t < 7; ++t) atomicAdd(grad_enc_w + (ch - H) * 7 + t, gw[t]);  // zeros if this slot had no tile
      atomicAdd(grad_enc_b + (ch - H), gw[7]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (tid < 32) tc::tmem_dealloc(tmem_slot, Plan::TMEM_COLS);
  LTC_TS();
  if (dbg != nullptr && blockIdx.x == 0 && tid == 0) {
    dbg[127] = nts;
    dbg[126] = gridDim.x;
  }
#undef LTC_TS
}

template <int C, int NE, int KT, bool BWD>
static int launch_lfa_tc(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                         const float* att_w, const float* att_wt, float* out, const float* go, float* gx, float* gew, float* geb,
                         float* gaw, const uint32_t* absmax, int64_t n, cudaStream_t st) {
  using Plan = LtcPlan<C, NE, KT, BWD>;
  auto kern = lfa_tc_kernel<C, NE, KT, BWD>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Plan::SMEM_BYTES);
  if (e != cudaSuccess) return cuda_fail(e, "lfa_tc smem attribute");
  const int64_t ntiles = ceil_div(n, Plan::TC);
  int64_t grid = num_sms();  // one persistent CTA per SM (TMEM: every CTA allocates up to all 512 columns)
  if (grid > ceil_div(ntiles, LTC_SLOTS)) grid = ceil_div(ntiles, LTC_SLOTS);
  kern<<<(unsigned)grid, LTC_THREADS, Plan::SMEM_BYTES, st>>>(x, pos, nbr, enc_w, enc_b, att_w, att_wt, out, go, gx, gew, geb, gaw,
                                                             absmax, n, ntiles, tc_debug_buffer());
  B200_CHECK_LAUNCH("lfa_tc_kernel");
  return B200_OK;
}

// (C, KT, NE forward, NE backward).  Tile sizes: every epilogue thread gets >= 1 centre (NE / KT a multiple of
// 2 * 128 / C), shared memory <= 227 KB, W columns + 2 * (NE + C) TMEM columns <= 512.
// K = 32 neighbour tables (BASELINE configs[4]) would need twice the shared memory per centre: FMA kernels.
// (C, KT, edges per forward tile, edges per backward tile).  K = 32 tables (BASELINE configs[4]): c = 64 both ways;
// c = 128 forward only -- its backward tile (W_att in shared memory + dA, F, T planes for >= 2 centres of 32 edges) does
// not fit 227 KB, the FMA kernel stays; c = 32 would need 8 centres x 32 edges = 256 TMEM columns per slot.
#define B200_LFA_TC_CASES(X) X(32, 16, 128, 128) X(64, 16, 128, 128) X(128, 16, 128, 32) X(64, 32, 128, 128)
#define B200_LFA_TC_FWD_ONLY_CASES(X) X(128, 32, 64, 0)

// returns B200_E_UNSUPPORTED when this (c, kt) has no tensor-core kernel (the caller then uses the FMA kernel);
// c = 256 goes to lfa_tc256.cu
int lfa_tc_fwd_dispatch(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                        const float* att_wt, float* out, int64_t n, int c, int kt, cudaStream_t st) {
  if (!tc_path_enabled(16)) return B200_E_UNSUPPORTED;
  if (c == 256) return lfa_tc256_fwd(x, pos, nbr, enc_w, enc_b, att_wt, out, n, kt, st);
#define X(C_, KT_, NEF_, NEB_)                                                                                     \
  if (c == C_ && kt == KT_)                                                                                        \
    return launch_lfa_tc<C_, NEF_, KT_, false>(x, pos, nbr, enc_w, enc_b, nullptr, att_wt, out, nullptr, nullptr, nullptr, \
                                               nullptr, nullptr, nullptr, n, st);
  B200_LFA_TC_CASES(X)
  B200_LFA_TC_FWD_ONLY_CASES(X)
#undef X
  return B200_E_UNSUPPORTED;
}

// Backward workspace of the tensor-core path: one scratch word (the maximum |grad_out| of the call), 16-byte aligned;
// c = 256 adds the fp32 dA and F edge rows and the partials of the split-K dW GEMM behind it.
int64_t lfa_tc_bwd_workspace_bytes(int64_t n, int c, int kt) {
  if (c != 256) return 256;  // dW_att stays in TMEM
  return 16 + (int64_t)lfa_tc256_bwd_stream_bytes(n, kt) + (int64_t)accumulate_at_b_workspace_bytes(c, c, n * kt);
}

// ws: lfa_tc_bwd_workspace_bytes(n, c, kt) bytes of device scratch
int lfa_tc_bwd_dispatch(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                        const float* att_w, const float* att_wt, const float* go, float* gx, float* gew, float* geb, float* gaw, void* ws, int64_t n,
                        int c, int kt, cudaStream_t st) {
  if (!lfa_tc_supported(c, kt)) return B200_E_UNSUPPORTED;
  uint32_t* absmax = static_cast<uint32_t*>(ws);
  cudaError_t e = cudaMemsetAsync(absmax, 0, sizeof(uint32_t), st);
  if (e != cudaSuccess) return cuda_fail(e, "lfa_tc absmax memset");
  {
    int64_t blocks = ceil_div(n * c / 4 + 1, 256);
    if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
    lfa_absmax_kernel<<<(unsigned)blocks, 256, 0, st>>>(go, n * c, absmax);
    B200_CHECK_LAUNCH("lfa_absmax_kernel");
  }
  if (c == 256)
    return lfa_tc256_bwd(x, pos, nbr, enc_w, enc_b, att_w, att_wt, go, gx, gew, geb, gaw, absmax,
                         reinterpret_cast<float*>(static_cast<char*>(ws) + 16), (size_t)lfa_tc_bwd_workspace_bytes(n, c, kt) - 16, n,
                         kt, st);
#define X(C_, KT_, NEF_, NEB_) \
  if (c == C_ && kt == KT_)    \
    return launch_lfa_tc<C_, NEB_, KT_, true>(x, pos, nbr, enc_w, enc_b, att_w, att_wt, nullptr, go, gx, gew, geb, gaw, absmax, n, st);
  B200_LFA_TC_CASES(X)
#undef X
  return B200_E_UNSUPPORTED;
}

bool lfa_tc_supported(int c, int kt) {
  if (!tc_path_enabled(16)) return false;
  if (c == 256 && (kt == 16 || kt == 32)) return true;  // lfa_tc256.cu
#define X(C_, KT_, NEF_, NEB_) \
  if (c == C_ && kt == KT_) return true;
  B200_LFA_TC_CASES(X)
#undef X
  return false;
}

}  // namespace b200
