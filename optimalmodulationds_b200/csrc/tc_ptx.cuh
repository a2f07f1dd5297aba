// PTX wrappers shared by the tcgen05 kernels (the prefilter tc_pass1.cu and the scoring kernel tc_exact.cu): mbarriers,
// bulk (TMA) copies, TMEM allocation / loads / stores, UMMA descriptors and the cta_group::2 MMA forms, plus the host
// helpers that lay out their fp16 weight images.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include <cstring>
#include <utility>

namespace tcx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin with a watchdog: a protocol bug must surface as a trapped kernel, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
// acquire at cluster scope: the waiter goes on to hand shared memory written by the PEER CTA to the tensor core
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (clock64() - t0 > 2000000000LL) __trap();
  }
}
// arrive (release at cluster scope) on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote_release(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(bar),
      "r"(rank)
      : "memory");
}
// same with the default .release.cta semantics: what CUTLASS's ClusterBarrier::arrive(cta_id) issues for the
// epilogue -> MMA hand-over of 2-SM kernels (the writer runs fence.proxy.async first); no MEMBAR per arrival
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(bar),
      "r"(rank)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// generic-proxy writes to shared memory (st.shared) -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc_512_2cta(uint32_t dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(dst_smem) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free_512_2cta(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(taddr) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// D[tmem] (+)= A[smem] * B[smem]^T over the CTA pair (M = 256), issued by one thread of the leader CTA
__device__ __forceinline__ void mma_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T, M = 256 over the CTA pair, issued by one thread of the leader CTA
__device__ __forceinline__ void mma_ts_2cta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all MMAs issued so far by this thread -> arrive on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void mma_commit_2cta(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}

#define R8(v, o) "=r"(v[o + 0]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), "=r"(v[o + 7])
#define W8(v, o) "r"(v[o + 0]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3]), "r"(v[o + 4]), "r"(v[o + 5]), "r"(v[o + 6]), "r"(v[o + 7])
// 32 / 16 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : R8(v, 0), R8(v, 8), R8(v, 16), R8(v, 24)
      : "r"(taddr)
      : "memory");
}
// 64 consecutive columns holding one fp16 accumulator element each (32-bit containers), two per register
__device__ __forceinline__ void tmem_ld32p(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : R8(v, 0), R8(v, 8), R8(v, 16), R8(v, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : R8(v, 0), R8(v, 8)
      : "r"(taddr)
      : "memory");
}
template <int OFF, int N>
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[N]) {
  static_assert(OFF + 32 <= N, "out of range");
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31};" ::
          W8(v, OFF + 0), W8(v, OFF + 8), W8(v, OFF + 16), W8(v, OFF + 24), "r"(taddr)
      : "memory");
}

// K-major, no-swizzle UMMA shared-memory descriptor (version 1): 8-row x 16-byte core matrices, consecutive row
// groups SBO = 128 bytes apart, consecutive 8-element K chunks LBO bytes apart
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
  const uint32_t lo = ((smem_addr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
  const uint32_t hi = (128u >> 4) | (1u << 14);
  return ((uint64_t)hi << 32) | lo;
}
// the same descriptor as two 32-bit words: the low word carries the address and LBO (advancing the operand by `bytes`
// adds bytes >> 4 to it), the high word is the constant SBO / version part
__device__ __forceinline__ uint32_t make_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);
// host: byte offset of element (n, k) of a `rows`-row slab in the layout of make_desc -- the 8-row x 16-byte core
// matrices of a K-chunk are contiguous, so row n starts n * 16 bytes into it; K-chunks are rows * 16 bytes apart (LBO)
inline size_t canon(int n, int k, int rows) {
  return (size_t)(k / 8) * rows * 16 + (size_t)n * 16 + (size_t)(k % 8) * 2;
}
// host: fp16 conversions (round to nearest even), no device needed
inline uint16_t f2h(float f) {
  __half h = __float2half_rn(f);
  uint16_t u;
  std::memcpy(&u, &h, 2);
  return u;
}
inline float h2f(uint16_t u) {
  __half h;
  std::memcpy(&h, &u, 2);
  return __half2float(h);
}
// the issuer's form of mma_ss_2cta: descriptors assembled inside the asm block from their low words, so the compiler
// has no 64-bit descriptor tables to precompute (and spill) ahead of the first MMA of a stage
__device__ __forceinline__ void mma_ss_2cta_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 ad, bd;\n\t"
      "mov.b64 ad, {%1, %5};\n\t"
      "mov.b64 bd, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], ad, bd, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "n"(DESC_HI)
      : "memory");
}
// The issuer's form of mma_ts_2cta: everything that is known at compile time (TMEM column offsets, the descriptor's
// offset from the start of shared memory, LBO, the instruction descriptor, the accumulate flag) is an immediate inside
// the asm block, so per MMA only two adds feed the instruction and the compiler has nothing to hoist out of the
// tile loop (a first unrolled version precomputed 240 descriptors and spilled them).
//   sb4      = shared-memory base address >> 4
//   DESC_IMM = (byte offset of the B slab >> 4) + (LBO >> 4 << 16), added to sb4 -> low descriptor word
template <uint32_t D_COL, uint32_t A_COL, uint32_t DESC_IMM, uint32_t IDESC, bool ACC>
__device__ __forceinline__ void mma_ts_2cta_imm(uint32_t tmem_base, uint32_t sb4) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 bd;\n\t.reg .b32 dl, td, ta;\n\t"
      "add.u32 td, %0, %2;\n\t"
      "add.u32 ta, %0, %3;\n\t"
      "add.u32 dl, %1, %4;\n\t"
      "mov.b64 bd, {dl, %5};\n\t"
      "setp.ne.b32 p, %7, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [td], [ta], bd, %6, p;\n\t}" ::"r"(tmem_base),
      "r"(sb4), "n"(D_COL), "n"(A_COL), "n"(DESC_IMM), "n"(DESC_HI), "n"(IDESC), "n"(ACC ? 1 : 0)
      : "memory");
}
// The same MMA, issued only when KS < nk (one warp-uniform compare per K-step; nk is a kernel argument)
template <uint32_t D_COL, uint32_t A_COL, uint32_t DESC_IMM, uint32_t IDESC, uint32_t KS>
__device__ __forceinline__ void mma_ts_2cta_imm_if(uint32_t tmem_base, uint32_t sb4, uint32_t nk) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t.reg .b64 bd;\n\t.reg .b32 dl, td, ta;\n\t"
      "setp.lt.u32 q, %7, %8;\n\t"
      "add.u32 td, %0, %2;\n\t"
      "add.u32 ta, %0, %3;\n\t"
      "add.u32 dl, %1, %4;\n\t"
      "mov.b64 bd, {dl, %5};\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [td], [ta], bd, %6, 1;\n\t}" ::"r"(tmem_base),
      "r"(sb4), "n"(D_COL), "n"(A_COL), "n"(DESC_IMM), "n"(DESC_HI), "n"(IDESC), "n"(KS), "r"(nk)
      : "memory");
}
// The K-steps KS of one accumulator group.  K-steps from FIXED on are issued only while KS < nk: the last 16 - nk
// K-steps multiply input features that the calibration found never active (tc_pass1.cu, dead-feature skip).
template <uint32_t D_COL, uint32_t A_COL, uint32_t B_OFF, uint32_t LBO, uint32_t IDESC, int FIXED, int... KS>
__device__ __forceinline__ void mma_group(uint32_t tmem_base, uint32_t sb4, uint32_t nk,
                                          std::integer_sequence<int, KS...>) {
  auto one = [&](auto K) {
    constexpr int k = decltype(K)::value;
    constexpr uint32_t desc = (B_OFF >> 4) + ((LBO >> 4) << 16) + k * ((2 * LBO) >> 4);
    if constexpr (k < FIXED) mma_ts_2cta_imm<D_COL, A_COL + k * 8, desc, IDESC, (k > 0)>(tmem_base, sb4);
    else mma_ts_2cta_imm_if<D_COL, A_COL + k * 8, desc, IDESC, k>(tmem_base, sb4, nk);
  };
  (one(std::integral_constant<int, KS>{}), ...);
}

// kind::f16 instruction descriptor: fp16 (fmt 0) or bf16 (fmt 1) A and B (K-major), fp32 (or fp16) accumulate, dense
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int M, int N, bool acc_f32 = true) {
  return (acc_f32 ? (1u << 4) : 0u) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

}  // namespace tcx
