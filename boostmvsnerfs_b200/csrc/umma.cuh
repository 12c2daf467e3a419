// tcgen05 (UMMA) / TMEM / mbarrier PTX wrappers shared by the 5th-generation tensor-core kernels of libbmv
// (render_multi_umma.cu, mvs_render_umma.cu, conv3d_umma.cu).  Field layouts: cute/arch/mma_sm100_desc.hpp (CUTLASS,
// vendored with the toolkit image) — restated here, nothing is included from it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bmv {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor: start address, leading (K-chunk) and stride (8-row group) byte offsets in
// 16-byte units, descriptor version 1 (Blackwell), SWIZZLE_NONE
// layout: 0 = SWIZZLE_NONE, 6 = SWIZZLE_32B, 4 = SWIZZLE_64B, 2 = SWIZZLE_128B (bits 61..63)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout = 0) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46) |
         ((uint64_t)layout << 61);
}
// instruction descriptor, kind::f16: D fp32, A/B fp16, both K-major, M = 128
__device__ __forceinline__ uint32_t umma_idesc(int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24); }

__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
               ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// same with the descriptors given as (low, high) 32-bit halves and a compile-time accumulate flag: an issue loop
// that only advances the low words by constants costs two integer adds per MMA
template <bool ACC>
__device__ __forceinline__ void umma_f16_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc) {
  asm volatile("{\n .reg .pred p;\n .reg .b64 da, db;\n setp.ne.b32 p, %6, 0;\n mov.b64 da, {%1, %2};\n mov.b64 db, {%3, %4};\n"
               " tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n}\n"
               ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "n"(ACC ? 1 : 0) : "memory");
}
// the TS form: A from tensor memory (K-major; kind::f16: one 32-bit column holds two consecutive K values of a row, low
// half first, so one K = 16 slab of A is 8 columns starting at a_tmem), B from shared memory as above
template <bool ACC>
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc) {
  asm volatile("{\n .reg .pred p;\n .reg .b64 db;\n setp.ne.b32 p, %5, 0;\n mov.b64 db, {%2, %3};\n"
               " tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n}\n"
               ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "n"(ACC ? 1 : 0) : "memory");
}
// one K = 16 step of a split product: D (+)= A_lo B_hi + A_hi B_lo + A_hi B_hi
__device__ __forceinline__ void umma_kstep(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lbo, uint32_t a_lo_off, uint32_t b_hi,
                                           uint32_t b_lbo, uint32_t b_lo_off, uint32_t idesc, uint32_t acc) {
  const uint64_t ah = umma_desc(a_hi, a_lbo, 128), al = umma_desc(a_hi + a_lo_off, a_lbo, 128);
  const uint64_t bh = umma_desc(b_hi, b_lbo, 128), bl = umma_desc(b_hi + b_lo_off, b_lbo, 128);
  umma_f16(d_tmem, al, bh, idesc, acc);
  umma_f16(d_tmem, ah, bl, idesc, 1u);
  umma_f16(d_tmem, ah, bh, idesc, 1u);
}
// true in exactly one (elected) lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void bar_sync_named(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// A broken pipeline must fault, not hang the GPU: a wait that lasts longer than 20 s of wall clock traps.  (Wall clock,
// not a spin count: under compute-sanitizer a kernel runs hundreds of times slower while try_wait returns at once.)
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t done = 0;
  uint64_t t0 = 0;
  for (uint32_t spins = 0; !done; ++spins) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
    if ((spins & 0xFFFu) == 0xFFFu) {
      const uint64_t now = global_timer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 20000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}

// non-blocking probe of a phase (an issuer polling several barriers must not park on one of them)
__device__ __forceinline__ uint32_t mbar_test(uint32_t mbar, uint32_t parity) {
  uint32_t done;
  asm volatile("{\n .reg .pred p;\n mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
  return done;
}
// 8 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               "tcgen05.wait::ld.sync.aligned;"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// 16 consecutive fp32 columns of this thread's TMEM lane (32 lanes x 32 bit, repeated 16 times)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  // load and wait in ONE asm statement: the registers are not defined for the compiler before the wait
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
               "tcgen05.wait::ld.sync.aligned;"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// 4 / 16 consecutive 32-bit columns of this thread's TMEM lane.  Unlike the loads these do not wait: a writer issues
// all its stores and then tmem_wait_st() once, before it tells another thread (or the tensor core) about them.
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                 "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// one warp allocates `cols` (power of two >= 32) TMEM columns; the base address lands in shared memory
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_alloc_512(uint32_t smem_dst) { tmem_alloc(smem_dst, 512u); }
__device__ __forceinline__ void tmem_dealloc_512(uint32_t taddr) { tmem_dealloc(taddr, 512u); }

// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
               "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n"
               "tcgen05.wait::ld.sync.aligned;"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                 "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                 "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

}  // namespace bmv
