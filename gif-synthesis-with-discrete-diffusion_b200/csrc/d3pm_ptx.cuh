// Inline-PTX wrappers for the Blackwell (sm_100a) asynchronous units: mbarriers, 1-D bulk TMA, the 5th-gen tensor cores
// (tcgen05: MMA, commit, tensor-memory allocation and loads) and CTA clusters.  Every kernel that talks to those units - the
// stream step, the training stream, the fused head and the decoder GEMM - uses these and no inline PTX of its own for them.
// Also the operand formats the MMAs are issued with: the tf32 instruction descriptor and the shared-memory descriptor.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace d3pm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarriers ------------------------------------------------------------------------------------------------
// fence_mbarrier_init() makes the inits before it visible to the async proxy and to the other CTAs of the cluster; it goes
// between the inits and the thread or cluster barrier that publishes them.
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(unsigned long long* bar, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
}
__device__ __forceinline__ bool mbar_test(unsigned long long* bar, uint32_t parity) {  // non-blocking
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
// Two waits, each measured in the kernels that use it; changing a kernel's wait is a performance change of that kernel.
// mbar_wait (the fused head, the decoder GEMM): lets the hardware suspend the thread until the phase completes (time-limit
// hint ~10 ms) instead of polling: the single-lane control warps would otherwise burn issue slots the epilogue warps need.
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity), "r"(0x989680)
      : "memory");
}
// mbar_wait_spin (the stream step, the training stream): try_wait without a time-limit hint in a polling loop.  There every
// thread of a group waits for a row whose copy was issued one row earlier; the stream kernels were tuned with this loop.
__device__ __forceinline__ void mbar_wait_spin(unsigned long long* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// the suspending wait with cluster-scope acquire: for barriers that the partner CTA of a pair arrives on
__device__ __forceinline__ void mbar_wait_cluster(unsigned long long* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity), "r"(0x989680)
      : "memory");
}

// ---- bulk TMA and the async proxy -------------------------------------------------------------------------------
// 1-D bulk copy global -> shared, completion bytes counted on the mbarrier.  (An L2 evict-first hint was measured ~4 %
// slower on B200 for the stream kernel's read-once rows, so the copies carry no cache hint.)
__device__ __forceinline__ void tma_load(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// orders this thread's generic-proxy accesses to shared memory before later async-proxy ones (TMA writes, MMA reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05: MMA and commit --------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(unsigned long long* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(unsigned long long* bar) {  // arrives on `bar` in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(static_cast<unsigned short>(3))
               : "memory");
}
// instruction descriptor of a kind::tf32 MMA: D = f32, A = B = tf32, both K-major, M x N (cute::UMMA::InstrDescriptor bit layout);
// M counts the rows of all CTAs of the MMA (256 for a pair)
constexpr uint32_t idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((static_cast<uint32_t>(N) >> 3) << 17) | ((static_cast<uint32_t>(M) >> 4) << 24);
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// issued by the leader CTA of a pair over both CTAs' shared memory and tensor memory
__device__ __forceinline__ void tc_mma_tf32_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// shared-memory descriptor of a K-major operand, 128-byte swizzle: rows at 128 B, 8-row groups at SBO = 1024 B, descriptor
// version 1 (sm_100).  The operand is 1024-byte aligned; `addr` may step by 32 B (K = 8 tf32) inside its 128-byte rows.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
  return static_cast<uint64_t>((addr >> 4) & 0x3fffu) | (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// ---- tcgen05: tensor memory -----------------------------------------------------------------------------------------
// CTAS = 1: this CTA's tensor memory (cta_group::1); CTAS = 2: the same warp of both CTAs of a pair allocates (cta_group::2).
// NCOLS: a power of two >= 32.  The address of the allocation is written to shared memory at `slot`.
template <int CTAS, int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  static_assert(CTAS == 1 || CTAS == 2, "cta_group::1 or ::2");
  if constexpr (CTAS == 2)
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(NCOLS) : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(NCOLS) : "memory");
}
// this CTA allocates no more tensor memory: lets other CTAs on the SM allocate without waiting for it
template <int CTAS>
__device__ __forceinline__ void tmem_relinquish() {
  static_assert(CTAS == 1 || CTAS == 2, "cta_group::1 or ::2");
  if constexpr (CTAS == 2) asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  else asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int CTAS, int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  static_assert(CTAS == 1 || CTAS == 2, "cta_group::1 or ::2");
  if constexpr (CTAS == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// 32 lanes x 32 bit: lane l of the warp reads TMEM lane (taddr >> 16) + l, 16 or 32 consecutive columns from (taddr & 0xffff)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- clusters -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}

}  // namespace d3pm
