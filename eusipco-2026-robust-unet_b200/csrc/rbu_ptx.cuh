// Inline-PTX wrappers for the Blackwell (sm_100a) async machinery used by the GEMM kernels:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA) + TMEM.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug must trap (sticky CUDA error on the host) instead of hanging the GPU.
static __device__ __noinline__ void mbar_timeout() {
  printf("rbunet: mbarrier wait timeout (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) mbar_timeout();
  }
}
// Wait with back-off for waiters that are far ahead of their partner (a TMA producer waiting for a free stage):
// the polling loop otherwise takes issue slots from the warps sharing its scheduler.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(64);
    if (++spins > (1u << 24)) mbar_timeout();
  }
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_shared_b32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
// same, addressed by a 32-bit shared address (no generic->shared conversion in hot loops)
__device__ __forceinline__ uint32_t mbar_try_wait_s(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait_s(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait_s(bar, parity)) {
    if (++spins > (1u << 26)) mbar_timeout();
  }
}
__device__ __forceinline__ void umma_commit_s(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t pack_desc(uint32_t lo, uint32_t hi) {
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
// upper / lower 32 bits of a SWIZZLE_128B shared-memory matrix descriptor (see make_smem_desc below)
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);
}
// same for SWIZZLE_64B operands (layout type 4; MN-major: 64 B = 32 bf16 of M/N per K-row, 8-row atoms of 512 B)
__device__ __forceinline__ uint32_t desc_hi_sw64(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (4u << 29);
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}

// ----------------------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "r"(c4)
      : "memory");
}

// TMA stores (shared -> global, bulk async-group completion) and the group bookkeeping of the issuing thread.
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3,
                                             int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
// the same three, addressed by 32-bit shared addresses
__device__ __forceinline__ void tma_store_4d_s(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_5d_s(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3,
                                               int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_load_4d_s(uint32_t dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                              int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {   // at most N groups still reading their shared-memory source
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {        // at most N groups not yet complete
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all tcgen05 ops previously issued by this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i = TMEM lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }


// ----------------------------------------------------------------------------- CTA pairs (cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(smem_u32(bar)), "r"(rank)
      : "memory");
}
// wait for a phase completed by arrivals from the peer CTA / the tensor core of the pair (cluster-scope acquire)
__device__ __forceinline__ uint32_t mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t b = smem_u32(bar);
  if (mbar_try_wait_cluster(b, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait_cluster(b, parity)) {
    if (++spins > (1u << 26)) mbar_timeout();
  }
}
__device__ __forceinline__ void mbar_wait_cluster_s(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (++spins > (1u << 26)) mbar_timeout();
  }
}
__device__ __forceinline__ void mbar_wait_cluster_backoff(uint64_t* bar, uint32_t parity) {
  const uint32_t b = smem_u32(bar);
  if (mbar_try_wait_cluster(b, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait_cluster(b, parity)) {
    __nanosleep(64);
    if (++spins > (1u << 24)) mbar_timeout();
  }
}
// TMA load issued by either CTA of a pair into its OWN shared memory; the bytes are counted on the LEADER's mbarrier
// (the barrier at the same offset in the even CTA: peer bit 24 of the shared::cluster address cleared)
__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B over the CTA pair: M = 256 (128 rows per CTA, each from its own shared memory), B's N
// columns split in halves between the two CTAs' shared memory; issued by ONE thread of the leader CTA.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarriers at this offset in the CTAs of `mask` once the pair's previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}
// SWIZZLE_32B operands (layout type 6; MN-major: 32 B = 16 bf16 of M/N per K-row, 8-row atoms of 256 B)
__device__ __forceinline__ uint32_t desc_hi_sw32(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (6u << 29);
}

// The same step in a kernel instantiated for one CTA (PAIR = false) or for a CTA pair (PAIR = true, cta_group::2):
// barrier wait (the pair's with cluster-scope acquire), TMA load (the pair's counted on the leader's barrier), MMA issue,
// and commit (the pair's multicast to the barrier at the same offset in both CTAs).
template <bool PAIR> __device__ __forceinline__ void bar_wait_remote(uint64_t* b, uint32_t par) {
  if (PAIR) mbar_wait_cluster(b, par); else mbar_wait(b, par);
}
template <bool PAIR> __device__ __forceinline__ void load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  if (PAIR) tma_load_4d_pair(dst, m, bar, c0, c1, c2, c3); else tma_load_4d(dst, m, bar, c0, c1, c2, c3);
}
template <bool PAIR> __device__ __forceinline__ void load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  if (PAIR) tma_load_2d_pair(dst, m, bar, c0, c1); else tma_load_2d(dst, m, bar, c0, c1);
}
template <bool PAIR> __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  if (PAIR) umma_bf16_pair(d, a, b, idesc, acc); else umma_bf16(d, a, b, idesc, acc);
}
template <bool PAIR> __device__ __forceinline__ void commit_s(uint32_t bar) {
  if (PAIR) umma_commit_pair(bar, 3); else umma_commit_s(bar);
}

// ----------------------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, SWIZZLE_128B, sm_100 version field = 1.
//   K-major operand  (rows = M/N index, 128 B = 64 bf16 of K per row): SBO = 1024 B (8-row group), LBO unused.
//   MN-major operand (rows = K index,   128 B = 64 bf16 of M/N per row): SBO = 1024 B (8 K-rows),
//                                                                      LBO = byte distance between 64-wide M/N blocks.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16, A/B = bf16, D = fp32.
__host__ __device__ __forceinline__ uint32_t make_idesc_bf16(int m, int n, int a_mn_major, int b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;   // D format: F32
  d |= 1u << 7;   // A format: BF16
  d |= 1u << 10;  // B format: BF16
  d |= static_cast<uint32_t>(a_mn_major & 1) << 15;
  d |= static_cast<uint32_t>(b_mn_major & 1) << 16;
  d |= static_cast<uint32_t>(n >> 3) << 17;
  d |= static_cast<uint32_t>(m >> 4) << 24;
  return d;
}

}  // namespace ptx
