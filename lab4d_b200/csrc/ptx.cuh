// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA bulk copy, tcgen05 (UMMA + TMEM).
// Bit layouts of the shared-memory matrix descriptor and the instruction descriptor follow the
// PTX ISA "tcgen05" chapter (cross-checked against cute/arch/mma_sm100_desc.hpp field tables).
#pragma once
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

namespace b200r {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
#ifndef B200R_WATCHDOG
#define B200R_WATCHDOG 1
#endif
#if B200R_WATCHDOG == 2
static __device__ int g_b200r_abort;  // debugging: a timed-out wait reports itself and every wait of the kernel gives up
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#if B200R_WATCHDOG == 2
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (((++spins) & 0xFFFFu) == 0) {
      if (*(volatile int*)&g_b200r_abort) return;
      if (spins > (1u << 23)) {
        printf("b200r: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x,
               smem_u32(bar), parity);
        *(volatile int*)&g_b200r_abort = 1;
        __threadfence();
        return;
      }
    }
  }
#elif B200R_WATCHDOG == 3
  // debugging: report the wait that timed out, then trap
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) {
      printf("b200r: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
#elif B200R_WATCHDOG
  // A protocol bug would otherwise hang the GPU box: trap after ~seconds of spinning.  No printf here: its call site (stack
  // frame, argument set-up) in every inlined wait cost 3 % of the training step (A/B on the B200: 6.01 -> 5.83 ms without it).
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) __trap();
  }
#else
  while (!mbar_try_wait(bar, parity)) {
  }
#endif
}

// ---------------------------------------------------------------- proxies / fences
// generic-proxy st.shared -> async-proxy readers (tcgen05.mma operand fetch, TMA)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- TMA (bulk, 1-D)
// global -> shared::cta, completion counted in bytes on an mbarrier.  SASS: UBLKCP.
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// multicast variant: the bytes land at the same CTA-relative offset in every CTA of `mask`, and each
// destination CTA's mbarrier (same offset) receives the complete_tx.
__device__ __forceinline__ void tma_bulk_g2s_mcast(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                                   uint16_t mask) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "h"(mask)
      : "memory");
}

// ---------------------------------------------------------------- cluster
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// producer side of a named barrier: signals (releasing this thread's prior writes) without waiting
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// one elected lane of a converged warp (elect.sync); cheaper for the issuing warp than `lane == 0`
// predication: tools/mma_probe.cu measures 67 vs 102 cycles per N=128 MMA on B200
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- TMEM allocation
// One full warp executes; the base address (lane<<16 | column) lands in *smem_slot.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---------------------------------------------------------------- UMMA descriptors
// K-major operand tile in shared memory, 128-byte swizzle: rows of 64 x 16-bit (128 B), 8-row
// groups are 1024 B apart (SBO), tile base 1024-B aligned.  Bits: [0,14) addr>>4, [16,30) LBO>>4,
// [32,46) SBO>>4, [46,48) version=1, [61,64) layout (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;            // LBO (ignored for swizzled K-major; canonical value)
  d |= (uint64_t)(1024 >> 4) << 32;  // SBO
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;            // SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: D=f32, A/B = f16 (0) or bf16 (1), both K-major, M=128.
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t ab_fmt, uint32_t N, uint32_t M = 128) {
  return (1u << 4)            // c_format = F32
         | (ab_fmt << 7)      // a_format
         | (ab_fmt << 10)     // b_format
         | (0u << 15)         // a_major = K
         | (0u << 16)         // b_major = K
         | ((N >> 3) << 17)   // n_dim
         | ((M >> 4) << 24);  // m_dim
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread.  SASS: UTCHMMA.
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TS form: the A operand is read from TMEM (lane = row, one 32-bit column = two consecutive K elements),
// written there by the previous layer's epilogue with tcgen05.st.
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives when all tcgen05 ops previously issued by this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// same, arriving on the barrier at this offset in every CTA of `mask` (2-CTA weight multicast)
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ---------------------------------------------------------------- TMEM -> registers
// 32 lanes x N consecutive 32-bit columns: thread i of the warp gets lane (base+i).  SASS: LDTM.
// The wait names the destination registers as read-write operands so no use can be scheduled above it.
#define B200R_R8(r, o) "=r"(r[o + 0]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]), "=r"(r[o + 6]), "=r"(r[o + 7])
#define B200R_W8(r, o) "+r"(r[o + 0]), "+r"(r[o + 1]), "+r"(r[o + 2]), "+r"(r[o + 3]), "+r"(r[o + 4]), "+r"(r[o + 5]), "+r"(r[o + 6]), "+r"(r[o + 7])
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,"
      "%28,%29,%30,%31}, [%32];"
      : B200R_R8(r, 0), B200R_R8(r, 8), B200R_R8(r, 16), B200R_R8(r, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait32(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : B200R_W8(r, 0), B200R_W8(r, 8), B200R_W8(r, 16), B200R_W8(r, 24)::"memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  tmem_ld32_issue(taddr, r);
  tmem_ld_wait32(r);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// registers -> TMEM: 16 consecutive 32-bit columns of this thread's lane.  SASS: STTM.
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
#define B200R_I8(r, o) "r"(r[o + 0]), "r"(r[o + 1]), "r"(r[o + 2]), "r"(r[o + 3]), "r"(r[o + 4]), "r"(r[o + 5]), "r"(r[o + 6]), "r"(r[o + 7])
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
      "%29,%30,%31,%32};" ::"r"(taddr),
      B200R_I8(r, 0), B200R_I8(r, 8), B200R_I8(r, 16), B200R_I8(r, 24)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), B200R_I8(r, 0) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16u_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : B200R_R8(r, 0), B200R_R8(r, 8)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : B200R_W8(r, 0), B200R_W8(r, 8)::"memory");
}
__device__ __forceinline__ void tmem_ld16u(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : B200R_R8(r, 0), B200R_R8(r, 8)
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" : B200R_W8(r, 0), B200R_W8(r, 8)::"memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : B200R_R8(r, 0), B200R_R8(r, 8)
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" : B200R_W8(r, 0), B200R_W8(r, 8)::"memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---------------------------------------------------------------- tape stores
// 32 operand columns (16 packed registers = four 16-B groups g0..g0+3, g0 in {0, 4}) of tile row `row` into a
// [128 x 64] SWIZZLE_128B chunk image in global memory: group g lives in 16-B slot g ^ (row & 7) of the row's 128 B, so
// groups (g, g+1) share one aligned 32-B sector (swapped when the row is odd) -> two 256-bit stores (STG.256) per call,
// each a full sector.
__device__ __forceinline__ void stg256(void* a, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3, uint32_t r4, uint32_t r5, uint32_t r6,
                                       uint32_t r7) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(a), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(r4), "r"(r5), "r"(r6), "r"(r7)
               : "memory");
}
// Tape layout of one tile with n_chunks chunks: [64-row half][chunk][64 rows x 128 B] - every chunk keeps the swizzled image
// (a 64-row half of it is 8 KB, 1024-B aligned), and the chunks of one half are adjacent, so the weight-gradient kernel
// fetches the G operand and the A operand of a half-tile stage with ONE contiguous bulk copy each.
__host__ __device__ __forceinline__ size_t tape_row_off(int n_chunks, int chunk, uint32_t row) {
  return ((size_t)(row >> 6) * (size_t)n_chunks + (size_t)chunk) * 8192u + (size_t)(row & 63u) * 128u;
}
// rowp = the 128 B of tile row `row` inside its chunk
__device__ __forceinline__ void chunk_st32(uint8_t* rowp, uint32_t row, uint32_t g0, const uint32_t (&o)[16]) {
  const uint32_t r = row & 7u;
  const bool odd = (r & 1u) != 0;
#pragma unroll
  for (int pr = 0; pr < 2; ++pr) {
    const uint32_t slot = ((g0 + 2u * pr) ^ r) & ~1u;
    const uint32_t* a = o + 8 * pr;
    stg256(rowp + (slot << 4), odd ? a[4] : a[0], odd ? a[5] : a[1], odd ? a[6] : a[2], odd ? a[7] : a[3], odd ? a[0] : a[4], odd ? a[1] : a[5],
           odd ? a[2] : a[6], odd ? a[3] : a[7]);
  }
}

// ---------------------------------------------------------------- 16-bit operand formats
struct OpF16 {
  static constexpr uint32_t kFmt = 0;
  // relu(a), relu(b) -> packed f16x2 in one instruction (cvt.rn.relu.f16x2.f32; low half = second operand)
  __device__ static __forceinline__ uint32_t pack2_relu(float a, float b) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
  __device__ static __forceinline__ uint32_t pack2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ static __forceinline__ uint16_t cvt(float a) {
    __half h = __float2half_rn(a);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __device__ static __forceinline__ float2 unpack2(uint32_t v) { return __half22float2(*reinterpret_cast<__half2*>(&v)); }
  __device__ static __forceinline__ float f32(uint16_t v) { return __half2float(*reinterpret_cast<__half*>(&v)); }
  // saturating pack (gradient operands: an overflow clamps to +-65504 instead of becoming inf / NaN downstream)
  __device__ static __forceinline__ uint32_t pack2_sat(float a, float b) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
};
struct OpBF16 {
  static constexpr uint32_t kFmt = 1;
  __device__ static __forceinline__ uint32_t pack2_relu(float a, float b) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
  __device__ static __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ static __forceinline__ uint16_t cvt(float a) {
    __nv_bfloat16 h = __float2bfloat16_rn(a);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __device__ static __forceinline__ float2 unpack2(uint32_t v) { return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v)); }
  __device__ static __forceinline__ float f32(uint16_t v) { return __bfloat162float(*reinterpret_cast<__nv_bfloat16*>(&v)); }
  __device__ static __forceinline__ uint32_t pack2_sat(float a, float b) {
    uint32_t r;
    asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
};

// Byte offset of the 16-byte group `g` (8 halves, g in [0,8)) of row `row` inside a
// [rows x 64] K-major SWIZZLE_128B operand tile.
__host__ __device__ __forceinline__ uint32_t sw128_off(uint32_t row, uint32_t g) {
  return row * 128u + ((g ^ (row & 7u)) << 4);
}

}  // namespace b200r
