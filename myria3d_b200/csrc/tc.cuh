// tcgen05 / TMEM building blocks for sm_100a (inline PTX; bit layouts follow the CUTLASS sm100 headers:
// cute/arch/mma_sm100_desc.hpp `SmemDescriptor` / `InstrDescriptor`, cute/atom/mma_traits_sm100.hpp
// `make_umma_desc`).
//
// Operand layout used throughout: K-major, NO swizzle ("interleave") canonical layout.  In 16-byte units
// (= 4 fp32 / tf32 values) an [R rows x K] operand is stored as
//       chunk(r, j) = (r % 8) + (r / 8) * SBO + j * LBO          j = k / 4
// i.e. 8-row x 16-byte core matrices; we choose SBO = 8 units (128 B: row groups back to back) and
// LBO = R + 1 units (one k-chunk of ALL rows, padded by 16 B so that lanes reading the same row at different
// k-chunks hit different banks).  The array is therefore  float smem[K/4][R+1][4].
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include "common.cuh"

namespace b200 {

// fused LFA kernels (lfa_tc.cu, lfa_tc256.cu): W_att is staged as 16 * W (exact), so that typical weights land in fp16's
// normal range; the scores then carry the factor 16
constexpr float kWScale = 16.f;
constexpr float kLog2eOverWScale = 1.4426950408889634f / kWScale;

namespace tc {

__device__ __forceinline__ uint32_t lbo_bytes(int rows) { return (uint32_t)(rows + 1) * 16u; }
constexpr uint32_t kSboBytes = 128u;

// float offset of element (row r, k) inside an operand tile of `rows` rows
__device__ __forceinline__ int operand_offset(int rows, int r, int k) { return ((k >> 2) * (rows + 1) + r) * 4 + (k & 3); }
__host__ __device__ constexpr size_t operand_floats(int rows, int k) { return (size_t)(k / 4) * (rows + 1) * 4; }

// shared-memory matrix descriptor (K-major, no swizzle, descriptor version 1 = Blackwell)
__device__ __forceinline__ uint64_t smem_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// instruction descriptor: D fp32, A/B tf32, dense.  a_mn / b_mn select the MN-major ("transposed") reading of
// an operand (bits 15 / 16, cute::UMMA::InstrDescriptor::a_major_/b_major_).
__host__ __device__ constexpr uint32_t idesc_tf32(int m, int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ------------------------------------------------------------------------------------------------------------
// 16-bit operands (kind::f16, bf16 x 3 split) and the MN-major ("transposed") reading of a buffer.
//
// tf32 operands can be read MN-major only from the SWIZZLE_128B_BASE32B layout (cutlass sm100_common.inl:
// "for mn-major tf32 operands, SW128_32B is the only available smem layout"; a no-swizzle MN-major tf32 descriptor
// multiplies by zero -- measured), so one tf32 buffer cannot serve both readings.  16-bit operands can: a plane
//       uint16 smem[chunks][R+1][8]          (16-byte vector = 8 consecutive elements of the CHUNKED dimension)
// is, without moving a byte,
//   * K-major  (rows = M/N index, chunks along K):  ((8,n),2):((1,SBO),LBO) in 16-byte units with SBO = 8 (rows are
//     contiguous), LBO = R+1 (chunk stride); one MMA (K = 16) reads 2 chunks; K += 16 adds 2 chunk strides;
//   * MN-major (rows = K index, chunks along M/N):  ((1,n),(8,k)):((X,SBO),(1,LBO)) with LBO = 8 (the next group of
//     8 K-rows follows directly), SBO = R+1 (stride between 8-wide M/N blocks); one MMA reads 16 rows; K += 16 adds
//     256 bytes.  (cute::make_umma_desc<Major::MN>, LayoutType::INTERLEAVE.)
// The fused LFA kernels (lfa_tc.cu) read W_att, F and dA both ways.
// one lane of a converged warp (the tensor core instructions of a CTA are issued by a single thread; electing it
// with elect.sync lets the compiler keep the descriptors in uniform registers without a per-instruction
// uniformisation loop)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
// descriptor of a plane with the start address left out: add (byte offset >> 4) to the low word per instruction
__device__ __forceinline__ uint64_t plane_desc_k_base(uint32_t plane_addr, int rows) {
  return smem_desc(plane_addr, lbo_bytes(rows), 128u);
}
__device__ __forceinline__ uint64_t plane_desc_mn_base(uint32_t plane_addr, int rows) {
  return smem_desc(plane_addr, 128u, lbo_bytes(rows));
}
// advance a descriptor by a byte offset (multiple of 16; the 14-bit start-address field cannot overflow inside
// the 227 KB of shared memory)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }
__host__ __device__ constexpr uint32_t plane_k_step_bytes(int rows) { return 2u * (uint32_t)(rows + 1) * 16u; }  // K += 16, K-major
constexpr uint32_t kPlaneMnStepBytes = 256u;                                                                     // K += 16, MN-major

__host__ __device__ constexpr size_t plane_halves(int rows, int chunked_dim) { return (size_t)(chunked_dim / 8) * (rows + 1) * 8; }
// uint16 offset of element (row r, position c along the chunked dimension) inside a plane of `rows` rows
__device__ __forceinline__ int plane_offset(int rows, int r, int c) { return ((c >> 3) * (rows + 1) + r) * 8 + (c & 7); }
__device__ __forceinline__ uint64_t plane_desc_k(uint32_t plane_addr, int rows, int k0 /* multiple of 16 */) {
  return smem_desc(plane_addr + (uint32_t)(k0 >> 3) * lbo_bytes(rows), lbo_bytes(rows), 128u);
}
__device__ __forceinline__ uint64_t plane_desc_mn(uint32_t plane_addr, int rows, int k0 /* row index, multiple of 16 */) {
  return smem_desc(plane_addr + (uint32_t)k0 * 16u, /*lbo: next 8 K-rows*/ 128u, /*sbo: next 8-wide M/N block*/ lbo_bytes(rows));
}
// instruction descriptor: D fp32, A/B bf16, dense
__host__ __device__ constexpr uint32_t idesc_bf16(int m, int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// instruction descriptor: D fp32, A/B fp16, dense
__host__ __device__ constexpr uint32_t idesc_f16(int m, int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// fp16 x 2 split (round to nearest): v = hi + lo + r, hi = fp16(v), lo = fp16(v - hi) (v - hi is exact in fp32).  Three
// products hi*hi', lo*hi', hi*lo' reproduce the fp32 product to ~2^-22 for operands in fp16's NORMAL range
// (6.1e-5 <= |v| <= 65504; the caller keeps them there: O(1) data, power-of-two pre-scaling); below it the absolute
// error is bounded by the subnormal spacing (<= 3e-8).  Half the planes and half the instructions of bf16 x 3.
// Two values at a time: the packed words hold (v0 | v1 << 16).
__device__ __forceinline__ void split_f16x2_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  v0 = fminf(fmaxf(v0, -60000.f), 60000.f);
  v1 = fminf(fmaxf(v1, -60000.f), 60000.f);
  const __half2 h = __floats2half2_rn(v0, v1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void split8_f16x2(const float (&v)[8], uint4& ph, uint4& pl) {
  split_f16x2_pair(v[0], v[1], ph.x, pl.x);
  split_f16x2_pair(v[2], v[3], ph.y, pl.y);
  split_f16x2_pair(v[4], v[5], ph.z, pl.z);
  split_f16x2_pair(v[6], v[7], ph.w, pl.w);
}
// which part (0 = hi, 1 = lo) of A / B the p-th of the three passes multiplies
__device__ __forceinline__ constexpr int f16x2_term_a(int p) { return p == 1 ? 1 : 0; }
__device__ __forceinline__ constexpr int f16x2_term_b(int p) { return p == 2 ? 1 : 0; }

// bf16 x 3 split by truncation: v = t1 + t2 + t3 + r with |r| <= 2^-24 |v|; every t_i is exactly a bf16 (the high
// half of an fp32 word), every residual is exact in fp32.  The six products t1t1', t1t2', t2t1', t2t2', t1t3', t3t1'
// reproduce the fp32 product to ~2^-23 (dropped: t2t3', t3t2' ~ 2^-24, t3t3' ~ 2^-32).
__device__ __forceinline__ void split_bf16x3(float v, uint32_t& t1, uint32_t& t2, uint32_t& t3) {
  t1 = __float_as_uint(v) & 0xFFFF0000u;
  const float r1 = v - __uint_as_float(t1);
  t2 = __float_as_uint(r1) & 0xFFFF0000u;
  const float r2 = r1 - __uint_as_float(t2);
  t3 = __float_as_uint(r2) & 0xFFFF0000u;
}
// pack the bf16 (= high halves) of two fp32-word terms: low 16 bits <- a, high 16 bits <- b
__device__ __forceinline__ uint32_t pack_hi16(uint32_t a, uint32_t b) { return __byte_perm(a, b, 0x7632); }
// which term of A / B the p-th of the six passes multiplies
__device__ __forceinline__ constexpr int bf16x3_term_a(int p) { return p == 2 || p == 3 ? 1 : (p == 5 ? 2 : 0); }
__device__ __forceinline__ constexpr int bf16x3_term_b(int p) { return p == 1 || p == 3 ? 1 : (p == 4 ? 2 : 0); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// make generic-proxy shared-memory writes visible to the async proxy (the tensor core reads smem through it)
__device__ __forceinline__ void fence_smem_to_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, one elected thread issues
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// the same with the A operand in TENSOR MEMORY (lane = row of A, every 32-bit column = two consecutive K elements,
// the even one in the low half): only B travels from shared memory
__device__ __forceinline__ void mma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: false on timeout (a wrong descriptor must not hang the GPU box)
__device__ __forceinline__ bool mbar_wait_bounded(uint64_t* bar, uint32_t parity, uint32_t max_polls = 4000000u) {
  for (uint32_t i = 0; i < max_polls; ++i) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) return true;
  }
  return false;
}

// the waits of the fused LFA kernels: a wrong descriptor or a lost commit must not hang the GPU
__device__ __forceinline__ void mbar_wait_or_trap(uint64_t* bar, uint32_t parity) {
  if (!mbar_wait_bounded(bar, parity, 20000000u)) __trap();
}

// 16 consecutive fp32 columns of this thread's TMEM lane (warp w of the CTA owns lanes 32*(w%4) .. +31)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 16 consecutive fp32 columns of this thread's TMEM lane <- registers (accumulator pre-initialisation)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_st16u(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
// one row of a bf16 x 3 A operand in tensor memory: 32 fp32 values (K = 32) -> 16 columns in each of the 3 planes
// (plane t at column offset t * plane_cols from taddr)
__device__ __forceinline__ void tmem_st_row32_bf16x3(uint32_t taddr, uint32_t plane_cols, const float (&v)[32]) {
  uint32_t w[3][16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    uint32_t a1, a2, a3, b1, b2, b3;
    split_bf16x3(v[2 * i], a1, a2, a3);
    split_bf16x3(v[2 * i + 1], b1, b2, b3);
    w[0][i] = pack_hi16(a1, b1), w[1][i] = pack_hi16(a2, b2), w[2][i] = pack_hi16(a3, b3);
  }
  tmem_st16u(taddr, w[0]);
  tmem_st16u(taddr + plane_cols, w[1]);
  tmem_st16u(taddr + 2 * plane_cols, w[2]);
}
// the same for fp16 x 2 operands: 2 planes
__device__ __forceinline__ void tmem_st_row32_f16x2(uint32_t taddr, uint32_t plane_cols, const float (&v)[32]) {
  uint32_t w[2][16];
#pragma unroll
  for (int i = 0; i < 16; ++i) split_f16x2_pair(v[2 * i], v[2 * i + 1], w[0][i], w[1][i]);
  tmem_st16u(taddr, w[0]);
  tmem_st16u(taddr + plane_cols, w[1]);
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// the same load without the wait: up to two of them in flight hide the TMEM read latency behind the previous block's
// processing.  tmem_ld_wait takes the destination registers as in/out operands so that no use can be scheduled
// above it.
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// 3xTF32 split: v ~= hi + lo, hi exactly representable in tf32 (round-to-nearest on the 13 dropped mantissa
// bits, done with integer ops: `cvt.rna.tf32.f32` compiles to a branchy NaN/Inf-aware sequence on sm_100a and made
// the operand conversion 5x more expensive than the MMAs it feeds).  lo = v - hi is exact in fp32; the tensor core
// ignores its low 13 bits (relative error <= 2^-10 of lo, i.e. ~2^-21 of v).  Inf/NaN inputs are not special-cased.
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
  lo = v - hi;
}

}  // namespace tc
}  // namespace b200
