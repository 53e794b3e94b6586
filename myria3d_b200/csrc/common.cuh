// Shared helpers of libb200randla.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/b200randla.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libb200randla is written for sm_100a (B200) only"
#endif

namespace b200 {

// ---- error reporting (thread-local message, no global mutable state besides the counter)
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
void count_launch(int n = 1);
int num_sms();

#define B200_REQUIRE(cond, code, ...)            \
  do {                                           \
    if (!(cond)) {                               \
      ::b200::set_error(__VA_ARGS__);            \
      return (code);                             \
    }                                            \
  } while (0)

#define B200_CHECK_LAUNCH(what)                                   \
  do {                                                            \
    cudaError_t e__ = cudaPeekAtLastError();                      \
    if (e__ != cudaSuccess) return ::b200::cuda_fail(e__, what);  \
    ::b200::count_launch();                                       \
  } while (0)

// out[m][k] += sum_i a[i][m] * b[i][k]  (a: [n, ca], b: [n, cb], out: [ca, cb]; split-K over n).  The attention-weight
// gradient of the fused LFA backward: n = E edges, up to ~10^6 rows.
int accumulate_at_b(const float* a, int ca, const float* b, int cb, float* out, int64_t n, float* ws, size_t ws_bytes,
                    cudaStream_t st);
size_t accumulate_at_b_workspace_bytes(int ca, int cb, int64_t n);

// tensor-core (tcgen05, 3xTF32) version of the same contraction, two-segment activation rows + bias column
// `ws` (optional, tc_tn_workspace_bytes()): per-split partial tiles + a reduction kernel instead of atomics
// (the rows one CTA accumulates are bounded for accuracy of long reductions: tc_gemm.cu)
int launch_tc_tn(const float* gy, int cout, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2,
                 float* gw, float* gb, int64_t n, float* ws, size_t ws_bytes, cudaStream_t st);
size_t tc_tn_workspace_bytes(int cout, int ncols, int64_t n);
// the same contraction for NARROW layers (<= 64 channels, not 64 x 64) on tcgen05 with bf16 x 3 operands read MN-major
// straight from their row-major layout (tc_skinny.cu)
bool tc_skinny_tn_ok(int cout, int ktot, bool has_bias, int64_t n);
int launch_tc_skinny_tn(const float* gy, int cout, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2,
                        float* gw, float* gb, int64_t n, cudaStream_t st);
// fused LFA forward / backward with every contraction on tcgen05 (lfa_tc.cu); B200_E_UNSUPPORTED -> use the FMA kernel
int lfa_tc_fwd_dispatch(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                        const float* att_wt, float* out, int64_t n, int c, int kt, cudaStream_t st);
int lfa_tc_bwd_dispatch(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                        const float* att_w, const float* att_wt, const float* go, float* gx, float* gew, float* geb, float* gaw,
                        void* ws, int64_t n, int c, int kt, cudaStream_t st);
bool lfa_tc_supported(int c, int kt);
int64_t lfa_tc_bwd_workspace_bytes(int64_t n, int c, int kt);  // when lfa_tc_supported(c, kt)
// c = 256 (lfa_tc256.cu): W_att streamed from L2 per tile.  The backward writes the fp32 dA and F edge rows
// (lfa_tc256_bwd_stream_bytes) to ws and reduces dW_att from them with accumulate_at_b, whose partials follow in ws.
int lfa_tc256_fwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b,
                  const float* att_wt, float* out, int64_t n, int kt, cudaStream_t st);
int lfa_tc256_bwd(const float* x, const float* pos, const int32_t* nbr, const float* enc_w, const float* enc_b, const float* att_w,
                  const float* att_wt, const float* go, float* gx, float* gew, float* geb, float* gaw, const uint32_t* absmax,
                  float* ws, size_t ws_bytes, int64_t n, int kt, cudaStream_t st);
size_t lfa_tc256_bwd_stream_bytes(int64_t n, int kt);
// row-streaming NT GEMM on tcgen05 (tc_nt.cu): out[i][m] = sum_k [a1|a2][i][k] * wm[m][k] + bias[m], channels of the
// output split over two destination segments; colstats: fp64 (sum, sum of squares) per row tile [tiles][2 * mrows]
bool tc_nt_shape_ok(int64_t n, int c1, int c2, int mrows);
int tc_nt_rows_per_tile(int64_t n, int mrows);
int launch_tc_nt(const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2, const float* wm, int mrows,
                 const float* bias, float* o1, int64_t old1, int oc1, float* o2, int64_t old2, double* colstats, int64_t n,
                 cudaStream_t st);
int launch_transpose(const float* w, float* wt, int rows, int cols, cudaStream_t st);
// linear_rows.cu: one thread per row, narrow layers of levels 0-1
bool linear_rows_ok(int64_t n, int k, int co);
int linear_rows_grid(int64_t n);
int launch_linear_rows(const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2, const float* w, int w_ld,
                       bool w_out_major, const float* bias, float* o1, int64_t old1, int oc1, float* o2, int64_t old2, int oc2,
                       int64_t n, double* colstats, cudaStream_t st);
// tma_rows.cu: TMA-fed row-streaming kernels for the 16/32/64-channel layers on >= 8192 rows.  NN serves the forward
// (w_out_major: w is [mcols][K]) and the input gradient (w is [K][mcols]); num_partials = rows of the caller's colstats
// buffer (one per CTA is written, the rest zero-filled).  TN is the weight / bias gradient (gw, gb accumulate).
bool tma_rows_enabled(int bit);  // runtime.cu: b200_set_option("tma_rows", mask): 1 forward, 2 input gradient, 4 weight gradient
bool tma_rows_nn_ok(int64_t n, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2, int mcols,
                    const float* o1, int64_t old1, int oc1, const float* o2, int64_t old2);
int launch_tma_rows_nn(const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2, const float* w, int w_ld,
                       bool w_out_major, const float* bias, float* o1, int64_t old1, int oc1, float* o2, int64_t old2,
                       int mcols, int64_t n, double* colstats, int num_partials, cudaStream_t st);
bool tma_rows_tn_ok(int64_t n, const float* gy, int cout, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2,
                    int c2);
int launch_tma_rows_tn(const float* gy, int cout, const float* a1, int64_t ld1, int c1, const float* a2, int64_t ld2, int c2,
                       float* gw, float* gb, int64_t n, cudaStream_t st);
void set_grid_points_per_cell(int v);  // knn_grid.cu (tuning knob, b200_set_option("knn_points_per_cell"))
int get_grid_points_per_cell();
bool bn_backward_fused_enabled();  // runtime.cu: b200_set_option("bn_backward_fused", 0/1)
bool tc_path_enabled(int bit);  // runtime.cu: b200_set_option("tensor_core_paths", mask) -- per-kernel-family A/B switch
bool tensor_cores_enabled();  // runtime.cu: b200_set_option("tensor_cores", 0) selects the FMA kernels (A/B switch)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
// lfa.cu: CTAs of a persistent kernel (resident CTAs per SM x SMs, at most ntiles, at least 1)
int persistent_grid(const void* kernel, int threads, size_t smem, int64_t ntiles);

constexpr float kLReluSlope = 0.2f;  // pyg_randla_net.py:92

// ---- device helpers
__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }

// fp32 squared distance with the reference's rounding sequence: separate products,
// ((dx*dx + dy*dy) + dz*dz), no FMA contraction (SURVEY.md App. D-9).
__device__ __forceinline__ float dist2_rn(float px, float py, float pz, float qx, float qy, float qz) {
  float dx = __fsub_rn(px, qx), dy = __fsub_rn(py, qy), dz = __fsub_rn(pz, qz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// Two independent fp32 FMAs in one instruction (fma.rn.f32x2, SASS FFMA2): d.x = a.x * b.x + c.x, d.y = a.y * b.y + c.y.
// On sm_100a the three-register FFMA issues every second cycle per scheduler; the packed form carries the second half
// of the chip's fp32 rate (measured: the c = 256 LFA kernels sat exactly at the scalar rate, 37 TFLOP/s).  Same IEEE
// result as two fmaf() calls.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}

// (c0, c1) += a * (b0, b1): the scalar operand uses FFMA2's broadcast form (R.F32), no register copy
__device__ __forceinline__ void ffma2_bc(float a, float b0, float b1, float& c0, float& c1) {
  const float2 d = ffma2(make_float2(a, a), make_float2(b0, b1), make_float2(c0, c1));
  c0 = d.x, c1 = d.y;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + 1-D TMA bulk copy (cp.async.bulk, SASS UBLKCP)
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace b200
