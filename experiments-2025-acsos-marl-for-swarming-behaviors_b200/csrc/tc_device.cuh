// tc_device.cuh -- tcgen05 (5th-gen tensor core) building blocks for the dense contractions of the Q-network
// (7->32 projection, 32->32 and 32->9 MLP layers).
//
// One CTA of 128 threads = 128 node rows = one UMMA tile: D[128 x N] (TMEM, fp32) = A[128 x K] (TMEM, written by the
// row owners with tcgen05.st) * B[N x K]^T (smem, K-major in the no-swizzle canonical layout: 8-row x 16-byte core
// matrices; LBO = byte stride between the 16-byte K chunks, SBO = byte stride between 8-row groups), kind::tf32.
// TMEM lane r holds row r, so after tcgen05.ld (32x32b) thread r owns exactly its node's output vector -- the same
// "thread = agent" ownership as the CUDA-core path.
//
// Precision: float32 operands are split x = hi + lo with hi = round-to-nearest-TF32(x) and lo = x - hi (exact), and
// the product is accumulated as lo*hi + hi*lo + hi*hi (small terms first).  Measured on B200 (scripts/tc_probe.cu):
// max abs error 2.95e-6 on |ref| <= 19 for K = 32, vs 4.4e-6 for a sequential float32 FFMA chain -- i.e. float32-level,
// which is what keeps Q within 1e-5 relative and greedy actions inside the oracle's tolerance band.
#ifndef SWARM_TC_DEVICE_CUH
#define SWARM_TC_DEVICE_CUH

#include <cuda_runtime.h>
#include <stdint.h>

namespace swarm {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 64-bit shared-memory matrix descriptor (no swizzle, version 1)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// instruction descriptor: D = F32, A = B = TF32, both K-major, M = 128
__device__ __forceinline__ uint32_t make_idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// hi = x rounded to nearest TF32 (ties away from zero, like cvt.rna.tf32.f32), lo = x - hi (exact).  The rounding is
// done on the bit pattern -- add half a TF32 ulp, clear the 13 low mantissa bits -- in two integer instructions;
// cvt.rna.tf32.f32 itself compiles to four (it also screens Inf / NaN, which adding 0x1000 maps to themselves anyway).
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
  lo = x - hi;
}

__device__ __forceinline__ void split4(const float4& v, float4& hi, float4& lo) {
  hi.x = __uint_as_float((__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u);
  hi.y = __uint_as_float((__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u);
  hi.z = __uint_as_float((__float_as_uint(v.z) + 0x1000u) & 0xFFFFE000u);
  hi.w = __uint_as_float((__float_as_uint(v.w) + 0x1000u) & 0xFFFFE000u);
  // lo = v - hi, two lanes per FADD2
  const float2 l0 = __fadd2_rn(make_float2(v.x, v.y), make_float2(-hi.x, -hi.y));
  const float2 l1 = __fadd2_rn(make_float2(v.z, v.w), make_float2(-hi.z, -hi.w));
  lo = make_float4(l0.x, l0.y, l1.x, l1.y);
}

// byte offset of (row r, k-chunk c) inside a K-major operand tile with `rows` rows
__device__ __forceinline__ int tile_off(int rows, int r, int c) { return c * rows * 16 + (r >> 3) * 128 + (r & 7) * 16; }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(done)
               : "r"(smem_u32(bar)), "r"(parity)
               : "memory");
  return done;
}

// bounded wait (a lost arrival traps instead of hanging the GPU).  The first try_wait sits outside the counted loop:
// it suspends the thread until the phase completes or a hardware time limit passes, which covers the usual wait, so
// the counter and the trap test stay off the common path.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t done = 0;
  for (int it = 0; it < (1 << 26) && !done; ++it) done = mbar_try_wait(bar, parity);
  if (!done) __trap();
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, int cols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, int cols) {     // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
  uint32_t e = 0;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(e));
  return e != 0;
}

__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// D = A * B^T with A in TENSOR MEMORY (lane = row, one 32-bit column per k) and B in shared memory (b_hi / b_lo = tile
// base addresses in the shared window, b_rows = N), 3xTF32 split: lo*hi + hi*lo + hi*hi, small terms first.  a_hi / a_lo
// are TMEM column addresses of the two halves; a k-step of 8 advances A by 8 columns and B by two 16-byte K chunks.
// Issued by one elected thread.
__device__ __forceinline__ void mma_tf32_tmem_a(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate ? 1u : 0u)
      : "memory");
}

__device__ __forceinline__ void mma_3xtf32_tmem_a(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                                  int b_rows, int ksteps, uint32_t idesc) {
  const uint32_t b_lbo = (uint32_t)b_rows * 16;
  const uint64_t db_hi = make_desc(b_hi, b_lbo, 128), db_lo = make_desc(b_lo, b_lbo, 128);
  const uint64_t b_step = (uint64_t)((2 * b_lbo) >> 4);
  bool acc = false;
#pragma unroll
  for (int term = 0; term < 3; ++term) {
    const uint32_t ta = (term == 0) ? a_lo : a_hi;         // lo*hi, hi*lo, hi*hi (small terms first)
    const uint64_t db = (term == 1) ? db_lo : db_hi;
#pragma unroll 4
    for (int j = 0; j < ksteps; ++j) {
      mma_tf32_tmem_a(tmem_d, ta + 8u * j, db + j * b_step, idesc, acc);
      acc = true;
    }
  }
}

// this thread's row (TMEM lane) <- 32 / 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

}  // namespace tc
}  // namespace swarm
#endif
