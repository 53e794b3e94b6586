// Fused LocSE + attentive pooling, FORWARD and BACKWARD, on the 5th-generation tensor cores for the widest level,
// c = 256 (block 4 of the network), K = 16 / 32 neighbour tables.  Same formulation and numerics as lfa_tc.cu (fp16 x 2
// split operands, three cross products, W_att staged as 16 * W, power-of-two scaled softmax gradient): see there.
//
// What differs from lfa_tc.cu is where W_att lives.  At c = 256 its fp16 x 2 planes are 256 KB: all 512 TMEM columns and
// more than the shared memory of an SM.  So W_att is STREAMED from L2 for every tile, in chunks of KC rows of the K
// dimension, through a two-deep ring in shared memory:
//   * every thread loads its part of chunk c + 1 into registers (fp32, two 16-byte loads per row it owns) while the
//     tensor core multiplies chunk c; the split into fp16 hi / lo and the 16-byte shared-memory stores follow when the
//     ring slot is free again (the MMAs of chunk c - 1 have completed: one mbarrier per ring slot, tcgen05.commit);
//   * a chunk is stored MN-major (rows = K index, 8 consecutive M indices per 16-byte vector), which is the layout
//     both fp32 sources already have row-contiguously: att_wt[m][n] for MMA1 (M = n, K = m) and att_w[n][m] for MMA3
//     (M = m, K = n).  Rows are padded to KC + 1 vectors so that the 32 lanes of a warp (= 32 consecutive M blocks)
//     store conflict-free.
// Channels sit on TMEM lanes in two M = 128 HALVES, edges on columns (the lfa_tc orientation: softmax and pooling stay
// thread-local).  Warp w owns lane quadrant w % 4 of half w / 4, i.e. channel ch = 128 * (w / 4) + 32 * (w % 4) + lane:
// the first four warps own the gathered x channels, the last four the encoding channels.  Each thread handles every
// centre of the tile for its channel.
//     MMA1  S [n][e]  = sum_m W[n][m]  F[e][m]      A = W chunk (smem, MN-major), B = F  (K-major)
//     MMA3  dF[m][e] += sum_n W[n][m] dA[e][n]      A = W chunk (smem, MN-major), B = dA (MN-major), accumulator
//                                                   pre-loaded with s * go by tcgen05.st
// S and dF share the 2 * NE TMEM columns of the tile.  The attention-weight gradient dW = dA^T F stays on the split-K
// GEMM of the FMA path (accumulate_at_b): a TMEM-resident 256 x 256 fp32 dW would need all 512 columns.  The epilogue
// streams the tile's fp32 dA and F rows ([E, 256] each, the layout of lfa.cu's launch_lfa_bwd<..., true>) to the
// workspace, coalesced (32 lanes = 32 consecutive channels of one edge).
//
// Per tile (backward): B1 ids / geometry -> build F -> MMA1 (NK chunks) -> E1: softmax, dA -> smem + workspace, s*go -> TMEM
// -> MMA3 (NK chunks) -> E3: encoder gradients in registers, x-gradients transposed through shared memory (aliasing the
// dA planes, dead once MMA3 has completed) and scattered with 16-byte vector reductions.
#include <math_constants.h>

#include <type_traits>

#include "lfa_tc.cuh"

namespace b200 {

long long* tc_debug_buffer();  // runtime.cu

constexpr int L256_THREADS = 256;
constexpr int L256_C = 256;

template <int NE, int KT, int KC, bool BWD>
struct L256Plan {
  static constexpr int C = L256_C, H = C / 2, H8 = H / 8, TC = NE / KT;
  static constexpr int NK = C / KC;                    // ring chunks per contraction
  static constexpr int NCHUNK = BWD ? 2 * NK : NK;     // per tile: MMA1 chunks, then (backward) MMA3 chunks
  static constexpr int ROWS_PER_THREAD = KC / 8;       // a warp stages 1 row per 8 (8 warps), lane = 8-wide M block
  static constexpr size_t W_PLANE = (size_t)(C / 8) * (KC + 1) * 16;  // [C/8 M blocks][KC K-rows + 1 pad][8]
  static constexpr size_t W_SLOT = 2 * W_PLANE;                        // hi | lo
  static constexpr uint32_t W_HALF_BYTES = 16u * (KC + 1) * 16u;       // 16 M blocks = one M = 128 half
  static constexpr size_t F_PLANE = (size_t)(C / 8) * (NE + 1) * 16;   // rows e, chunked along m
  static constexpr size_t DA_PLANE = BWD ? (size_t)(NE / 8) * (C + 1) * 16 : 0;  // rows n, chunked along e
  static constexpr size_t T_BYTES = tc::operand_floats(NE, H) * 4;     // fp32 [H/4][NE+1][4]
  static constexpr size_t OFF_W = 0;
  static constexpr size_t OFF_F = OFF_W + 2 * W_SLOT;
  static constexpr size_t OFF_DA = OFF_F + 2 * F_PLANE;  // T aliases the dA planes (backward)
  static constexpr size_t OFF_EW = OFF_DA + 2 * DA_PLANE;
  static constexpr size_t OFF_Q = OFF_EW + 16 * 17 * (size_t)H8;
  static constexpr size_t OFF_P = OFF_Q + 16 * (size_t)NE;
  static constexpr size_t OFF_NB = OFF_P + 16 * (size_t)TC;
  static constexpr size_t OFF_DEG = OFF_NB + 4 * (size_t)NE;
  static constexpr size_t SMEM_BYTES = OFF_DEG + 16 * ((TC + 3) / 4);
  static constexpr uint32_t TMEM_COLS = (2 * NE <= 64) ? 64 : (2 * NE <= 128) ? 128 : 256;
  static_assert(KT == 16 || KT == 32, "neighbour slots");
  static_assert(KC % 16 == 0 && C % KC == 0, "ring chunk: whole K = 16 steps");
  static_assert(NE % 32 == 0 && NE >= KT && NE <= L256_THREADS && NE <= 128, "tile shape");
  static_assert(!BWD || T_BYTES <= 2 * DA_PLANE, "the x-gradient transposition fits the dA planes");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
  static_assert(W_SLOT % 16 == 0 && F_PLANE % 16 == 0 && DA_PLANE % 16 == 0, "alignment");
};


template <int NE, int KT, int KC, bool BWD>
__global__ void __launch_bounds__(L256_THREADS, 1)
lfa_tc256_kernel(const float* __restrict__ x, const float* __restrict__ pos, const int32_t* __restrict__ nbr,
                 const float* __restrict__ enc_w, const float* __restrict__ enc_b,
                 const float* __restrict__ att_w /* backward: W_att [n][m] */,
                 const float* __restrict__ att_wt /* att_wt [m][n] = W_att[n][m] */,
                 float* __restrict__ out,                                                    // forward
                 const float* __restrict__ grad_out, float* __restrict__ grad_x,             // backward
                 float* __restrict__ grad_enc_w, float* __restrict__ grad_enc_b,
                 float* __restrict__ da_out, float* __restrict__ f_out /* [n * KT][C] each, for the dW GEMM */,
                 const uint32_t* __restrict__ absmax_bits /* backward: max |grad_out| as float bits */,
                 int64_t n, int64_t ntiles, long long* __restrict__ dbg) {
  using Plan = L256Plan<NE, KT, KC, BWD>;
  constexpr int C = Plan::C, H = Plan::H, H8 = Plan::H8, TC = Plan::TC, NK = Plan::NK;
  // power-of-two scale of the softmax gradient (backward), as in lfa_tc.cu
  float gscale = 1.f, inv_gscale = 1.f;
  if constexpr (BWD) {
    const uint32_t e = (*absmax_bits) >> 23;
    if (e >= 24u && e <= 250u) {
      gscale = __uint_as_float((255u - e) << 23);
      inv_gscale = __uint_as_float((e - 1u) << 23);
    }
  }
  const float dscale = gscale * kWScale;                      // dA planes carry kWScale * gscale
  const float inv_dscale = inv_gscale / (kWScale * kWScale);  // dF accumulator carries gscale * kWScale^2
  (void)dscale, (void)inv_dscale;
  extern __shared__ __align__(128) unsigned char l256_smem[];
  __shared__ __align__(8) uint64_t wbar[2];  // ring slot s is free again: the MMAs of its last chunk completed
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned char* Wring = l256_smem + Plan::OFF_W;
  unsigned char* Fp = l256_smem + Plan::OFF_F;
  unsigned char* dAp = l256_smem + Plan::OFF_DA;
  float* T = reinterpret_cast<float*>(l256_smem + Plan::OFF_DA);
  float4* EW = reinterpret_cast<float4*>(l256_smem + Plan::OFF_EW);  // [H/8][17] float4, as in lfa_tc.cu
  float4* Q = reinterpret_cast<float4*>(l256_smem + Plan::OFF_Q);
  float4* P = reinterpret_cast<float4*>(l256_smem + Plan::OFF_P);
  int* NB = reinterpret_cast<int*>(l256_smem + Plan::OFF_NB);
  int* DEG = reinterpret_cast<int*>(l256_smem + Plan::OFF_DEG);

  int nts = 0;
#define L256_TS()                                                                           \
  do {                                                                                      \
    if (dbg != nullptr && blockIdx.x == 0 && tid == 0 && nts < 120) dbg[nts++] = clock64(); \
  } while (0)
  L256_TS();

  for (int idx = tid; idx < H; idx += L256_THREADS) {
    const float* w = enc_w + idx * 7;
    EW[17 * (idx >> 3) + 2 * (idx & 7)] = make_float4(__ldg(w), __ldg(w + 1), __ldg(w + 2), __ldg(w + 3));
    EW[17 * (idx >> 3) + 2 * (idx & 7) + 1] = make_float4(__ldg(w + 4), __ldg(w + 5), __ldg(w + 6), __ldg(enc_b + idx));
  }
  if (warp == 0) tc::tmem_alloc(&tmem_slot, Plan::TMEM_COLS);
  if (tid == 0) {
    mbar_init(&wbar[0], 1);
    mbar_init(&wbar[1], 1);
    mbar_fence_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();

  // epilogue role: TMEM lane quadrant q = warp % 4 of half hh = warp / 4
  const int q = warp & 3, hh = warp >> 2;
  const int ch = hh * 128 + q * 32 + lane;
  const uint32_t lane_base = (uint32_t)(q * 32) << 16;
  const uint32_t tmem_base = tmem_slot;
  const uint32_t tmem_acc = tmem_base + (uint32_t)(hh * NE);  // this thread's half: S, then dF (backward)
  float4 mw0 = make_float4(0.f, 0.f, 0.f, 0.f), mw1 = mw0;    // encoder weights of this thread's channel (ch >= H)
  if (ch >= H) {
    mw0 = EW[17 * ((ch - H) >> 3) + 2 * ((ch - H) & 7)];
    mw1 = EW[17 * ((ch - H) >> 3) + 2 * ((ch - H) & 7) + 1];
  }
  float gw[8];  // encoder-gradient partials of channel ch (>= H), carried across tiles
#pragma unroll
  for (int t = 0; t < 8; ++t) gw[t] = 0.f;

  // ---- W ring.  Chunk `seq` of a tile: seq < NK -> rows [seq * KC, +KC) of att_wt (MMA1), else rows of att_w (MMA3).
  // Thread (warp, lane) stages rows warp + 8 i of the chunk, M block `lane`.
  float4 wr[Plan::ROWS_PER_THREAD][2];
  auto load_chunk = [&](int seq) {
    const float* src = (BWD && seq >= NK) ? att_w : att_wt;
    const int k0 = (seq % NK) * KC;
#pragma unroll
    for (int i = 0; i < Plan::ROWS_PER_THREAD; ++i) {
      const float4* p = reinterpret_cast<const float4*>(src + (int64_t)(k0 + warp + 8 * i) * C + 8 * lane);
      wr[i][0] = __ldg(p);
      wr[i][1] = __ldg(p + 1);
    }
  };
  uint32_t cc = 0;  // chunks staged so far by this CTA: ring slot cc & 1, use cc >> 1 of that slot
  // stage chunk `seq` (already in wr) into the ring, fetch the next one, and issue its MMAs
  auto stage_and_issue = [&](int seq) {
    const uint32_t s = cc & 1u;
    if (cc >= 2) tc::mbar_wait_or_trap(&wbar[s], ((cc >> 1) - 1u) & 1u);
    unsigned char* slot = Wring + s * Plan::W_SLOT;
#pragma unroll
    for (int i = 0; i < Plan::ROWS_PER_THREAD; ++i) {
      const float v[8] = {kWScale * wr[i][0].x, kWScale * wr[i][0].y, kWScale * wr[i][0].z, kWScale * wr[i][0].w,
                          kWScale * wr[i][1].x, kWScale * wr[i][1].y, kWScale * wr[i][1].z, kWScale * wr[i][1].w};
      uint4 p1, p2;
      tc::split8_f16x2(v, p1, p2);
      const size_t off = ((size_t)lane * (KC + 1) + warp + 8 * i) * 16;
      *reinterpret_cast<uint4*>(slot + off) = p1;
      *reinterpret_cast<uint4*>(slot + Plan::W_PLANE + off) = p2;
    }
    load_chunk(seq + 1 < Plan::NCHUNK ? seq + 1 : 0);  // in flight while these MMAs run (the next tile starts at 0)
    tc::fence_smem_to_async();
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) {
      if (tc::elect_one_sync()) {
        tc::fence_after_sync();
        const bool mma3 = BWD && seq >= NK;
        const int k0 = (seq % NK) * KC;
        const uint64_t wd0 = tc::plane_desc_mn_base(smem_u32(slot), KC);
        const uint64_t bd0 = mma3 ? tc::plane_desc_mn_base(smem_u32(dAp), C) : tc::plane_desc_k_base(smem_u32(Fp), NE);
        const size_t b_plane = mma3 ? Plan::DA_PLANE : Plan::F_PLANE;
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint64_t ad = tc::desc_advance(wd0, (uint32_t)(tc::f16x2_term_a(pass) * Plan::W_PLANE));
          const uint64_t bd = tc::desc_advance(bd0, (uint32_t)(tc::f16x2_term_b(pass) * b_plane));
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int ks = 0; ks < KC / 16; ++ks) {
              const int kk = k0 + 16 * ks;
              const uint64_t a = tc::desc_advance(ad, (uint32_t)h * Plan::W_HALF_BYTES + (uint32_t)ks * tc::kPlaneMnStepBytes);
              if (mma3) {
                constexpr uint32_t idesc = tc::idesc_f16(128, NE, /*a_mn=*/true, /*b_mn=*/true);
                tc::mma_bf16(tmem_base + (uint32_t)(h * NE), a, tc::desc_advance(bd, (uint32_t)kk * 16u), idesc, true);
              } else {
                constexpr uint32_t idesc = tc::idesc_f16(128, NE, /*a_mn=*/true, /*b_mn=*/false);
                tc::mma_bf16(tmem_base + (uint32_t)(h * NE), a, tc::desc_advance(bd, (uint32_t)(kk / 16) * tc::plane_k_step_bytes(NE)),
                             idesc, (seq | pass | ks) != 0);
              }
            }
        }
        tc::mma_commit(&wbar[s]);
      }
      __syncwarp();
    }
    ++cc;
  };
  // all MMAs issued so far have completed (the commit of the last chunk tracks every earlier MMA)
  auto wait_all_mma = [&]() {
    tc::mbar_wait_or_trap(&wbar[(cc - 1u) & 1u], ((cc - 1u) >> 1) & 1u);
    tc::fence_after_sync();
  };

  const int64_t tile_stride = gridDim.x;
  // thread e < NE keeps the neighbour id and the centre position of edge e of the NEXT tile in registers
  int pf_j = -1;
  float4 pf_p = make_float4(0.f, 0.f, 0.f, 0.f);
  auto prefetch = [&](int64_t t) {
    pf_j = -1;
    pf_p = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t i = t * TC + tid / KT;
    if (t < ntiles && i < n) {
      pf_j = __ldg(nbr + i * KT + tid % KT);
      pf_p = make_float4(__ldg(pos + 3 * i), __ldg(pos + 3 * i + 1), __ldg(pos + 3 * i + 2), 0.f);
    }
  };
  if (tid < NE) prefetch(blockIdx.x);
  load_chunk(0);
  L256_TS();

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += tile_stride) {
    const int64_t tile_base = tile * TC;
    // ---- B1: neighbour ids (prefetched during the previous tile), geometry, degrees
    if (tid < NE) {
      const int e = tid, g = e / KT, kk = e % KT;
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
    __syncthreads();
    L256_TS();
    // ---- B2 / B3: F = [x_j ; lrelu(enc_w . q + enc_b)]
    ltc_build_f<NE, KT, H, L256_THREADS>(tid, x, NB, P, Q, EW, Fp, Plan::F_PLANE);
    L256_TS();  // (the F planes are published by the first chunk's barrier)

    // ---- MMA1: S[n][e] = sum_m W[n][m] F[e][m], both halves, W streamed through the ring
#pragma unroll 1
    for (int seq = 0; seq < NK; ++seq) stage_and_issue(seq);
    wait_all_mma();
    L256_TS();

    // ---- E1: thread = channel; softmax over the neighbourhood, pooled output, (backward) softmax gradient
    auto e1_centre = [&](const int g, const int deg, auto full_tag) {
      constexpr bool FULL = decltype(full_tag)::value;
      const int64_t i = tile_base + g;
      float a[KT], f[KT];
      float go_v = 0.f;  // (backward) issued first: its latency hides behind the softmax
      if constexpr (BWD) {
        if (i < n) go_v = __ldg(grad_out + i * C + ch);
      }
      (void)go_v;
#pragma unroll
      for (int k0 = 0; k0 < KT; k0 += 16) {
        float v[16];
        tc::tmem_ld16(tmem_acc + lane_base + (uint32_t)(g * KT + k0), v);
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k0 + k] = v[k];
      }
      // the fp32 feature of (edge, this channel), bit-identical to the value the build split
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
          const float4 qq = Q[g * KT + k];
          float s = sp;
          s = fmaf(mw0.w, qq.x, s), s = fmaf(mw1.x, qq.y, s), s = fmaf(mw1.y, qq.z, s);
          s = fmaf(mw1.z, qq.w, s);
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
        const float gi = inv * go_v;
#pragma unroll
        for (int k8 = 0; k8 < KT; k8 += 8) {
          float da[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int k = k8 + u;
            const float sg = a[k] * gi;            // s * go (0 for invalid edges: p = 0)
            const float d = sg * (f[k] - o);       // gradient w.r.t. the score
            if (i < n) {                           // the edge rows of the dW GEMM
              da_out[(i * KT + k) * C + ch] = d;
              f_out[(i * KT + k) * C + ch] = f[k];
            }
            da[u] = d * dscale;
            a[k] = sg * (dscale * kWScale);        // direct term of dF at the accumulator's scale kWScale^2 * gscale
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
          tc::tmem_st16(tmem_acc + lane_base + (uint32_t)(g * KT + k0), v);  // dF accumulator <- s * go
        }
      }
    };
#pragma unroll 1
    for (int g = 0; g < TC; ++g) {
      const int deg = DEG[g];
      if (deg == KT)
        e1_centre(g, deg, std::true_type{});
      else
        e1_centre(g, deg, std::false_type{});
    }
    if constexpr (!BWD) {
      tc::fence_before_sync();
      __syncthreads();  // TMEM, NB / Q / P / DEG and the F tile are free for the next tile
      tc::fence_after_sync();
      L256_TS();
    } else {
      tc::tmem_st_wait();
      L256_TS();  // (dA planes and the pre-loaded accumulator are published by the first MMA3 chunk's barrier)

      // ---- MMA3: dF[m][e] += sum_n W[n][m] dA[e][n]
#pragma unroll 1
      for (int seq = NK; seq < 2 * NK; ++seq) stage_and_issue(seq);
      wait_all_mma();
      L256_TS();

      // ---- E3: thread = channel m; encoder gradients stay in registers, x-gradients go through T
      auto e3_centre = [&](const int g, const int deg, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        float d[KT];
#pragma unroll
        for (int k0 = 0; k0 < KT; k0 += 16) {
          float v[16];
          tc::tmem_ld16(tmem_acc + lane_base + (uint32_t)(g * KT + k0), v);
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
              const float4 qq = Q[g * KT + k];
              float s = sp;  // lrelu'(z) from the recomputed pre-activation
              s = fmaf(mw0.w, qq.x, s), s = fmaf(mw1.x, qq.y, s), s = fmaf(mw1.y, qq.z, s);
              s = fmaf(mw1.z, qq.w, s);
              const float dz = d[k] * (s > 0.f ? inv_dscale : inv_dscale * kLReluSlope);
              gw[3] = fmaf(dz, qq.x, gw[3]);
              gw[4] = fmaf(dz, qq.y, gw[4]);
              gw[5] = fmaf(dz, qq.z, gw[5]);
              gw[6] = fmaf(dz, qq.w, gw[6]);
              gsum += dz;
            }
          gw[0] = fmaf(gsum, p.x, gw[0]);
          gw[1] = fmaf(gsum, p.y, gw[1]);
          gw[2] = fmaf(gsum, p.z, gw[2]);
          gw[7] += gsum;
        }
      };
#pragma unroll 1
      for (int g = 0; g < TC; ++g) {
        const int deg = DEG[g];
        if (deg == KT)
          e3_centre(g, deg, std::true_type{});
        else
          e3_centre(g, deg, std::false_type{});
      }
      tc::fence_before_sync();
      __syncthreads();
      tc::fence_after_sync();
      L256_TS();
      // ---- scatter the x-gradients
      ltc_scatter_x<NE, H, L256_THREADS>(tid, T, NB, grad_x);
      // the next tile's B1 writes NB / Q / P / DEG and E1 the dA planes (= T), all of which the scatter still reads
      __syncthreads();
      L256_TS();
    }
  }

  if constexpr (BWD) {
    if (ch >= H) {
#pragma unroll
      for (int t = 0; t < 7; ++t) atomicAdd(grad_enc_w + (ch - H) * 7 + t, gw[t]);  // zeros if this CTA had no tile
      atomicAdd(grad_enc_b + (ch - H), gw[7]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_slot, Plan::TMEM_COLS);
  L256_TS();
  if (dbg != nullptr && blockIdx.x == 0 && tid == 0) {
    dbg[127] = nts;
    dbg[126] = gridDim.x;
  }
#undef L256_TS
}

// (NE, KC) per direction: one CTA per SM (the 256 threads need up to 255 registers each), 64- / 128-edge tiles, 32-row
// chunks.  Forward: F planes 132 KB + ring 68 KB; backward: F and dA planes 132 KB + ring 68 KB.
constexpr int L256_NE_FWD = 128, L256_KC_FWD = 32;
constexpr int L256_NE_BWD = 64, L256_KC_BWD = 32;

template <int NE, int KT, int KC, bool BWD>
static int launch_lfa_tc256(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                            const float* att_w, const float* att_wt, float* out, const float* go, float* gx, float* gew,
                            float* geb, float* da_out, float* f_out, const uint32_t* absmax, int64_t n, cudaStream_t st) {
  using Plan = L256Plan<NE, KT, KC, BWD>;
  auto kern = lfa_tc256_kernel<NE, KT, KC, BWD>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Plan::SMEM_BYTES);
  if (e != cudaSuccess) return cuda_fail(e, "lfa_tc256 smem attribute");
  const int64_t ntiles = ceil_div(n, Plan::TC);
  const int grid = persistent_grid(reinterpret_cast<const void*>(kern), L256_THREADS, Plan::SMEM_BYTES, ntiles);
  kern<<<(unsigned)grid, L256_THREADS, Plan::SMEM_BYTES, st>>>(x, pos, nbr, enc_w, enc_b, att_w, att_wt, out, go, gx, gew, geb,
                                                               da_out, f_out, absmax, n, ntiles, tc_debug_buffer());
  B200_CHECK_LAUNCH("lfa_tc256_kernel");
  return B200_OK;
}

int lfa_tc256_fwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                  const float* att_wt, float* out, int64_t n, int kt, cudaStream_t st) {
  if (kt == 16)
    return launch_lfa_tc256<L256_NE_FWD, 16, L256_KC_FWD, false>(x, pos, nbr, enc_w, enc_b, nullptr, att_wt, out, nullptr, nullptr,
                                                                 nullptr, nullptr, nullptr, nullptr, nullptr, n, st);
  if (kt == 32)
    return launch_lfa_tc256<L256_NE_FWD, 32, L256_KC_FWD, false>(x, pos, nbr, enc_w, enc_b, nullptr, att_wt, out, nullptr, nullptr,
                                                                 nullptr, nullptr, nullptr, nullptr, nullptr, n, st);
  return B200_E_UNSUPPORTED;
}

size_t lfa_tc256_bwd_stream_bytes(int64_t n, int kt) { return 2 * (size_t)n * kt * L256_C * sizeof(float); }

int lfa_tc256_bwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b, const float* att_w,
                  const float* att_wt, const float* go, float* gx, float* gew, float* geb, float* gaw, const uint32_t* absmax,
                  float* ws, size_t ws_bytes, int64_t n, int kt, cudaStream_t st) {
  float* da_out = ws;
  float* f_out = ws + n * kt * L256_C;
  int rc = B200_E_UNSUPPORTED;
  if (kt == 16)
    rc = launch_lfa_tc256<L256_NE_BWD, 16, L256_KC_BWD, true>(x, pos, nbr, enc_w, enc_b, att_w, att_wt, nullptr, go, gx, gew, geb,
                                                             da_out, f_out, absmax, n, st);
  if (kt == 32)
    rc = launch_lfa_tc256<L256_NE_BWD, 32, L256_KC_BWD, true>(x, pos, nbr, enc_w, enc_b, att_w, att_wt, nullptr, go, gx, gew, geb,
                                                             da_out, f_out, absmax, n, st);
  if (rc != B200_OK) return rc;
  // dW_att[n][m] += sum_e dA[e][n] F[e][m]: split-K GEMM over the streamed edge rows
  const size_t streams = lfa_tc256_bwd_stream_bytes(n, kt);
  return accumulate_at_b(da_out, L256_C, f_out, L256_C, gaw, n * kt, reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + streams),
                         ws_bytes - streams, st);
}

}  // namespace b200
