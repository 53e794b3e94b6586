// Per-tile pieces shared by the two tensor-core LFA kernels (lfa_tc.cu: c in {32, 64, 128}; lfa_tc256.cu: c = 256).
// A "slot" is the ST threads (local id stid) that own one tile of NE edges = NE / KT centres.
#pragma once
#include "tc.cuh"

namespace b200 {

// F planes of the tile (tc.cuh plane layout: rows = edge e, chunked along the channel m, hi plane then lo plane f_plane
// bytes later): F[:, 0:H) = x_j (gathered, zeros for empty slots), F[:, H:2H) = lrelu(enc_w . q + enc_b), 8 channels
// per item.  The gathers are issued first and consumed after the encoding, so their latency hides behind it.
// EW: encoder weights [H/8][17] float4 ((w0..w3), (w4, w5, w6, bias) per channel, one pad), NB / Q / P: the tile's
// neighbour ids, (p_j, dist) per edge and p_i per centre.
template <int NE, int KT, int H, int ST>
__device__ __forceinline__ void ltc_build_f(int stid, const float* __restrict__ x, const int* NB, const float4* P, const float4* Q,
                                            const float4* EW, unsigned char* Fp, size_t f_plane) {
  constexpr int H8 = H / 8;
  constexpr int BUILD_ITERS = (NE * H8 + ST - 1) / ST;
  float4 xa[BUILD_ITERS], xb[BUILD_ITERS];
#pragma unroll
  for (int it = 0; it < BUILD_ITERS; ++it) {
    const int t = it * ST + stid;
    xa[it] = xb[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    if ((NE * H8) % ST == 0 || t < NE * H8) {
      const int j = NB[t / H8];
      if (j >= 0) {
        xa[it] = __ldg(reinterpret_cast<const float4*>(x + (int64_t)j * H + 8 * (t % H8)));
        xb[it] = __ldg(reinterpret_cast<const float4*>(x + (int64_t)j * H + 8 * (t % H8) + 4));
      }
    }
  }
#pragma unroll
  for (int it = 0; it < BUILD_ITERS; ++it) {
    const int t = it * ST + stid;
    if ((NE * H8) % ST == 0 || t < NE * H8) {
      const int e = t / H8, c8 = t % H8;
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (NB[e] >= 0) {
        const float4 p = P[e / KT], q = Q[e];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const float4 w0 = EW[17 * c8 + 2 * u], w1 = EW[17 * c8 + 2 * u + 1];
          float s = fmaf(w0.z, p.z, fmaf(w0.y, p.y, fmaf(w0.x, p.x, w1.w)));
          s = fmaf(w0.w, q.x, s), s = fmaf(w1.x, q.y, s), s = fmaf(w1.y, q.z, s);
          s = fmaf(w1.z, q.w, s);
          v[u] = lrelu(s, kLReluSlope);
        }
      }
      uint4 p1, p2;
      tc::split8_f16x2(v, p1, p2);
      const size_t off = ((size_t)(H8 + c8) * (NE + 1) + e) * 16;
      *reinterpret_cast<uint4*>(Fp + off) = p1;
      *reinterpret_cast<uint4*>(Fp + f_plane + off) = p2;
    }
  }
#pragma unroll
  for (int it = 0; it < BUILD_ITERS; ++it) {
    const int t = it * ST + stid;
    if ((NE * H8) % ST == 0 || t < NE * H8) {
      const int e = t / H8, m8 = t % H8;
      const float v[8] = {xa[it].x, xa[it].y, xa[it].z, xa[it].w, xb[it].x, xb[it].y, xb[it].z, xb[it].w};
      uint4 p1, p2;
      tc::split8_f16x2(v, p1, p2);
      const size_t off = ((size_t)m8 * (NE + 1) + e) * 16;
      *reinterpret_cast<uint4*>(Fp + off) = p1;
      *reinterpret_cast<uint4*>(Fp + f_plane + off) = p2;
    }
  }
}

// scatter the tile's x-gradients from the transposition buffer T (fp32 [H/4][NE+1][4]): thread = (edge, 4 channels),
// 16-byte vector reductions
template <int NE, int H, int ST>
__device__ __forceinline__ void ltc_scatter_x(int stid, const float* T, const int* NB, float* __restrict__ grad_x) {
  constexpr int H4 = H / 4;
#pragma unroll
  for (int t0 = 0; t0 < NE * H4; t0 += ST) {
    const int t = t0 + stid;
    if ((NE * H4) % ST == 0 || t < NE * H4) {
      const int e = t / H4, m4 = t % H4;
      const int j = NB[e];
      if (j >= 0) {
        const float4 v = *reinterpret_cast<const float4*>(T + (m4 * (NE + 1) + e) * 4);
        atomicAdd(reinterpret_cast<float4*>(grad_x + (int64_t)j * H) + m4, v);
      }
    }
  }
}

}  // namespace b200
