// tcgen05 / TMEM / mbarrier building blocks (sm_100a inline PTX) shared by the tensor-core
// kernels.  Operands are FP32 values split into two terms (hi + lo), either two TF32 values or
// two scaled FP16 values; a product is evaluated as hi*hi + hi*lo + lo*hi with FP32
// accumulation in TMEM, which keeps the result within ~1e-6 relative of the FP32 reference --
// a plain TF32 or FP16 operand (10-bit mantissa) cannot meet the 1e-4 tolerance of the path.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>

namespace srcnn {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- operand split -------------------------------------------------------------------------
// hi = x rounded to TF32 (10 explicit mantissa bits, round-half-away on the magnitude: add half
// an ulp to the bit pattern, clear the 13 low bits), lo = x - hi (exact in FP32).  The tensor
// core ignores the 13 low mantissa bits of a TF32 operand, so lo needs no rounding of its own:
// |x - (hi + trunc(lo))| <= 2^-21 |x|.  `cvt.rna.tf32.f32` is NOT used: sm_100a has no such
// instruction, ptxas expands each one to VIADD + FSETP + SEL + LOP3 (9 instructions per split
// instead of 3), and the split is the inner loop of every SIMT role of the fused kernels.
// Non-finite inputs are not preserved (inf becomes NaN); the path never produces them.
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
  lo = x - hi;
}

// FP16 split: x*s = hi + lo with s a power of two that puts the operand range at ~2^14
__device__ __forceinline__ float pow2_scale(float bound) {   // 2^14 / pow2ceil(bound)
  if (!(bound > 0.f) || !(bound < 1e30f)) return 1.f;
  int e;
  frexpf(bound, &e);                 // bound = f * 2^e, f in [0.5, 1)
  return ldexpf(1.f, 14 - e);
}
// xs = hi + lo (raw half bits)
__device__ __forceinline__ void split_h(float xs, unsigned short& hi, unsigned short& lo) {
  const __half h = __float2half_rn(xs);
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(__float2half_rn(xs - __half2float(h)));
}
// two values -> packed pairs (element 0 in the low half: K index order)
__device__ __forceinline__ void split_h2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ uint32_t pack2(unsigned short a, unsigned short b) {
  return (uint32_t)a | ((uint32_t)b << 16);
}

// ---- canonical K-major, no-swizzle operand layout ------------------------------------------
// A [rows][K] operand (K = reduction dim, 32-bit elements) is stored as 8-row x 16-byte core
// matrices (128 contiguous bytes each).  Core matrices that are neighbours along K are 128 B
// apart (LBO), 8-row groups are 128*K/4 bytes apart (SBO).  Returns the FLOAT offset of (r,k).
__host__ __device__ __forceinline__ int kmajor_offset(int r, int k, int K) {
  return (r >> 3) * (32 * (K >> 2)) + (k >> 2) * 32 + (r & 7) * 4 + (k & 3);
}
// K-major canonical layout for 16-bit elements: core matrix = 8 rows x 16 bytes (8 halves);
// returns the offset in halves of (row r, element k) of a [rows][K] operand
__host__ __device__ __forceinline__ int kmajor16(int r, int k, int K) {
  return (r >> 3) * (64 * (K >> 3)) + (k >> 3) * 64 + (r & 7) * 8 + (k & 7);
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address, LBO, SBO in
// 16-byte units, version 1 (Blackwell), layout type 0 = SWIZZLE_NONE
__device__ __forceinline__ uint64_t make_desc_kmajor(const void* base, uint32_t byte_offset,
                                                     uint32_t lbo_bytes, uint32_t sbo_bytes) {
  const uint32_t addr = smem_u32(base) + byte_offset;
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// instruction descriptor (cute::UMMA::InstrDescriptor) for kind::tf32, FP32 accumulate,
// A and B both K-major, dense
__host__ __device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N) {
  uint32_t d = 0;
  d |= 1u << 4;                    // c_format = F32
  d |= 2u << 7;                    // a_format = TF32
  d |= 2u << 10;                   // b_format = TF32
  d |= (uint32_t)(N >> 3) << 17;   // n_dim
  d |= (uint32_t)(M >> 4) << 24;   // m_dim
  return d;
}
__host__ __device__ __forceinline__ uint32_t make_idesc_f16(int Mm, int Nn) {
  // c_format = F32, a_format = b_format = F16, both K-major
  return (1u << 4) | ((uint32_t)(Nn >> 3) << 17) | ((uint32_t)(Mm >> 4) << 24);
}

// ---- TMEM ------------------------------------------------------------------------------------
// one full warp; ncols power of two >= 32; the base address lands in *slot (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(slot)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols)
               : "memory");
}

// warp-collective: lane i receives 8 consecutive columns of TMEM lane (lane_base + i);
// taddr = (lane_base << 16) | column, lane_base = 32 * (warp_id % 4)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float v[8]) {
  uint32_t r[8];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float v[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, "
      "%12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
// the same without the wait: several loads in flight, then one tmem_ld_wait
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float v[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, "
      "%12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// warp-collective: lane i writes 8 consecutive columns of TMEM lane (lane_base + i)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float v[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
      "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
      "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
      : "memory");
}
// the same for 32-bit payloads (packed half pairs)
__device__ __forceinline__ void tmem_st8u(uint32_t taddr, const uint32_t v[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// make generic-proxy shared-memory writes visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- MMA issue / completion -----------------------------------------------------------------
// D[tmem] (+)= A[smem desc] * B[smem desc]^T ; issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// same with the A operand in TMEM (lane = row, one 32-bit column per K element)
__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// kind::f16 versions: A in shared memory (ss) or in TMEM (ts)
__device__ __forceinline__ void mma_f16_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc,
                                           uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d),
      "l"(a), "l"(b), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void mma_f16_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc,
                                           uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d),
      "r"(a), "l"(b), "r"(idesc), "r"(acc)
      : "memory");
}

// one lane of the (converged) warp; ptxas then knows the guarded tcgen05.mma sequence is
// executed by a single thread and does not wrap every instruction in an ELECT/branch loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "@px mov.s32 %0, 1;\n\t"
      "}\n"
      : "+r"(pred));
  return pred != 0;
}

// arrives on the mbarrier when all previously issued MMAs of this thread have completed
// (implicitly performs tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)
               : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// The suspend-time hint lets the hardware park the waiting thread until the phase completes
// (or the hint expires) instead of returning early and spinning: the fused kernels keep ~15
// warps waiting per SM, and their retry loops take issue slots from the single threads that
// issue the MMAs.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(0x989680u)
      : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// named barrier (0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace tc
}  // namespace srcnn
