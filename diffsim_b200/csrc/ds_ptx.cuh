// Thin inline-PTX wrappers for the sm_100a features the kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / st)
// and the UMMA shared-memory / instruction descriptors.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace ds {

// ---------------------------------------------------------------------------
// addresses
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ void prefetch_l1(const void* p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make mbarrier.init visible to the async proxy (TMA / tcgen05.commit)
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// generic-proxy smem writes -> visible to async-proxy readers (UMMA, TMA store)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// The suspend-time hint lets the hardware park the thread until the phase completes (it is woken by the arrival) or
// the time limit passes: without it a waiting warp re-issues the try_wait every few dozen clocks -- 41% of all
// instructions the v6 attention kernel executed were such spins, paid for in issue slots and, under the power cap,
// in SM clock.
constexpr uint32_t kTryWaitHintNs = 10000000;   // 10 ms
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kTryWaitHintNs)
      : "memory");
  return ok != 0;
}

// non-blocking probe of a phase
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
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
#ifndef DS_WATCHDOG_NS
#define DS_WATCHDOG_NS 4000000000ull  // 4 s: a stuck pipeline traps instead of hanging the GPU
#endif

// Blocking wait with a watchdog.  try_wait suspends the thread in hardware for a bounded time, so the spin is cheap.
// The watchdog is a bare spin counter (three instructions): every wait is inlined into the hot path of some warp
// role, and these kernels live or die by their instruction-cache footprint.  A stuck pipeline traps after 2^10 failed
// try_waits (each may suspend for the hint time: seconds in total); build with -DDS_WATCHDOG_VERBOSE to have it say where.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins == (1u << 10)) {
#ifdef DS_WATCHDOG_VERBOSE
      printf("diffsim_b200: mbarrier watchdog: block %d thread %d bar smem+%u parity %u\n", (int)blockIdx.x,
             (int)threadIdx.x, smem_u32(bar), parity);
#endif
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------
// named barriers (sub-CTA sync)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// barrier + OR-reduction of a predicate over the participating threads
__device__ __forceinline__ bool named_bar_or(uint32_t id, uint32_t nthreads, bool pred) {
  uint32_t out;
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "setp.ne.u32 q, %3, 0;\n\t"
      "bar.red.or.pred p, %1, %2, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(out)
      : "r"(id), "r"(nthreads), "r"((uint32_t)pred)
      : "memory");
  return out != 0;
}

// ---------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "r"(c4)
      : "memory");
}

// TMA prefetch of a 5-D box into L2 (no shared-memory destination, no completion signal)
__device__ __forceinline__ void tma_prefetch_l2_5d(const CUtensorMap* m, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global.tile [%0, {%1, %2, %3, %4, %5}];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}

// TMA store of a 2-D box from shared memory (bulk async group of the issuing thread)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups are still READING their shared-memory source
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------------------
// tcgen05: TMEM allocation
// ---------------------------------------------------------------------------
// Whole-warp call.  ncols: power of two in [32, 512].  The base address is
// written to *dst_smem.
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// Warpgroup register re-allocation (setmaxnreg works on aligned groups of four warps; every warp of the group executes it).
template <int R>
__device__ __forceinline__ void reg_dealloc() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R));
}
template <int R>
__device__ __forceinline__ void reg_alloc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R));
}

// ---------------------------------------------------------------------------
// tcgen05: MMA
// ---------------------------------------------------------------------------
// D[tmem] (+)= A[smem] * B[smem]; single-thread issue.
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once every previously issued tcgen05 op of this thread has
// completed (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------------------
// CTA pairs (cta_group::2): two CTAs of a cluster on the SMs of one TPC execute one M = 256 MMA; each holds its 128
// rows of A, HALF of the B tile and its 128 rows of the accumulator.  Only the leader (cluster rank 0) issues MMAs.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address of the pair
// TMA load into THIS CTA's shared memory; the transaction bytes are counted on the LEADER's mbarrier (same offset)
__device__ __forceinline__ void tma_load_2d_2cta(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_2cta(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                                 int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1),
      "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem], M = 256 over the pair: each CTA supplies its own 128 rows of A from its own TMEM
__device__ __forceinline__ void umma_f16_ts_2cta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at this offset in BOTH CTAs of the pair once the issued MMAs have completed
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"((uint16_t)3)
      : "memory");
}
// ---------------------------------------------------------------------------
// Multicast inside a cluster of independent CTAs (cta_group::1 MMAs): one TMA load lands at the same shared-memory offset
// of every CTA in cta_mask and completes transaction bytes on the mbarrier at the same offset of each; one L2 read serves
// all of them.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_5d_mc(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                               int c3, int c4, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, "
      "%5, %6, %7}], [%2], %8;"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "r"(c4), "h"(cta_mask)
      : "memory");
}
// arrive on the mbarrier at this offset in every CTA of cta_mask once this thread's issued MMAs have completed
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(cta_mask)
      : "memory");
}

// arrive on the LEADER's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, 0;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}\n"
      ::"r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------------------
// tcgen05: TMEM <-> registers.  32x32b: thread i of the warp owns lane
// (lane_base + i) and receives N consecutive 32-bit columns.
// taddr = (lane << 16) | column.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld_x1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  return r;
}
__device__ __forceinline__ void tmem_st_x1(uint32_t taddr, uint32_t v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------
// UMMA descriptors
// ---------------------------------------------------------------------------
// Shared-memory matrix descriptor (tcgen05 "version 1").  Layout types follow
// the hardware encoding: 0 none, 2 = 128B swizzle, 4 = 64B swizzle, 6 = 32B.
enum : uint32_t { UMMA_SW_NONE = 0, UMMA_SW128 = 2, UMMA_SW64 = 4, UMMA_SW32 = 6 };

__host__ __device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                            uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);            // [0,14)  start address >> 4
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;       // [16,30) leading byte offset >> 4
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;       // [32,46) stride byte offset >> 4
  d |= static_cast<uint64_t>(1) << 46;                                // [46,48) descriptor version = 1
  d |= static_cast<uint64_t>(layout & 7u) << 61;                      // [61,64) swizzle mode
  return d;
}

// Instruction descriptor for kind::f16 (fp16 / bf16 inputs, fp32 accumulate).
// fmt: 0 = f16, 1 = bf16.  *_mn_major: 0 = K-major operand, 1 = MN-major operand.
__host__ __device__ __forceinline__ uint32_t umma_idesc_f16_ab(uint32_t fmt_a, uint32_t fmt_b, uint32_t M, uint32_t N,
                                                               uint32_t a_mn_major, uint32_t b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                  // [4,6)   accumulator format: f32
  d |= (fmt_a & 7u) << 7;        // [7,10)  A format
  d |= (fmt_b & 7u) << 10;       // [10,13) B format
  d |= (a_mn_major & 1u) << 15;  // [15]    A major
  d |= (b_mn_major & 1u) << 16;  // [16]    B major
  d |= ((N >> 3) & 63u) << 17;   // [17,23) N / 8
  d |= ((M >> 4) & 31u) << 24;   // [24,29) M / 16
  return d;
}
__host__ __device__ __forceinline__ uint32_t umma_idesc_f16(uint32_t fmt, uint32_t M, uint32_t N, uint32_t a_mn_major,
                                                            uint32_t b_mn_major) {
  return umma_idesc_f16_ab(fmt, fmt, M, N, a_mn_major, b_mn_major);
}

// ---------------------------------------------------------------------------
// packed fp32 pairs (sm_100: FFMA2 / FADD2 / FMUL2 -- two fp32 lanes per issue slot)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t f2_pack_u(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float f2_hsum(uint64_t v) {
  float lo, hi;
  f2_unpack(v, lo, hi);
  return lo + hi;
}

// ---------------------------------------------------------------------------
// small numeric helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// 2^x for two fp32 lanes WITHOUT the MUFU pipe: Cody-Waite split x = j + f (j = round(x), |f| <= 0.5), a degree-3
// minimax polynomial for 2^f (max relative error 7.5e-5 = 2^-13.7, well under the 2^-9 / 2^-12 rounding of 16-bit P)
// on the FMA pipe, and j added straight into the exponent field.  Valid for x in [-126, 127); smaller x is clamped
// (2^-126 is zero in 16 bits anyway), NaN inputs come out as 2^-126.
__device__ __forceinline__ void exp2_poly_f2(float x0, float x1, float& e0, float& e1) {
  x0 = fmaxf(x0, -126.0f);
  x1 = fmaxf(x1, -126.0f);
  const uint64_t x = f2_pack(x0, x1);
  const uint64_t magic = f2_pack(12582912.0f, 12582912.0f);          // 1.5 * 2^23
  const uint64_t r = f2_add(x, magic);                               // low mantissa bits = round(x)
  const uint64_t jf = f2_add(r, f2_pack(-12582912.0f, -12582912.0f));
  const uint64_t f = f2_fma(jf, f2_pack(-1.0f, -1.0f), x);           // x - j
  uint64_t p = f2_fma(f, f2_pack(0.05517144873738289f, 0.05517144873738289f), f2_pack(0.2426108419895172f, 0.2426108419895172f));
  p = f2_fma(p, f, f2_pack(0.6932609677314758f, 0.6932609677314758f));
  p = f2_fma(p, f, f2_pack(0.9999281167984009f, 0.9999281167984009f));
  float p0, p1, r0, r1;
  f2_unpack(p, p0, p1);
  f2_unpack(r, r0, r1);
  e0 = __uint_as_float(__float_as_uint(p0) + (__float_as_uint(r0) << 23));
  e1 = __uint_as_float(__float_as_uint(p1) + (__float_as_uint(r1) << 23));
}

// 2^x for two fp16 lanes in one MUFU op
__device__ __forceinline__ uint32_t ex2_f16x2(uint32_t x) {
  uint32_t y;
  asm("ex2.approx.f16x2 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ uint32_t mul_f16x2(uint32_t a, uint32_t b) {
  uint32_t y;
  asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(y) : "r"(a), "r"(b));
  return y;
}

template <bool kBf16>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  if constexpr (kBf16) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  } else {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
}
template <bool kBf16>
__device__ __forceinline__ float2 unpack2(uint32_t u) {
  if constexpr (kBf16) {
    __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
    return __bfloat1622float2(v);
  } else {
    __half2 v = *reinterpret_cast<__half2*>(&u);
    return __half22float2(v);
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace ds
