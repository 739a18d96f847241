// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma /
// commit / ld), cluster helpers.  Everything here is a 1:1 wrapper around one PTX instruction so the
// kernels read as the hardware protocol they implement.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace scd {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b32 r;\n\t"
      "elect.sync r|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void cluster_arrive_release() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait_acquire() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  cluster_arrive_release();
  cluster_wait_acquire();
}

// named barriers (ids 1..15): a token hand-off between two warps is  arrive  on one side,  sync  on the other
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("barrier.cta.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("barrier.cta.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ uint32_t ld_shared_volatile(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.volatile.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_volatile(uint32_t addr, uint32_t v) {
  asm volatile("st.volatile.shared::cta.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// ------------------------------------------------------------------ mbarrier
// In a 2-CTA pair the leader (cluster rank 0) owns the barriers the tensor core waits on; the
// peer reaches them by clearing bit 24 of its own shared::cta address (the CTA-rank bit of the
// shared::cluster window).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init_cluster() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on a barrier addressed in the shared::cluster window (own or peer CTA)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}
// same, without the cluster-scope release fence (ERRBAR + CGAERRBAR: it drains every outstanding global
// store of the thread first).  Enough when the only thing ordered before the arrive is tcgen05 traffic,
// which tcgen05.wait::ld / tcgen05.fence::before_thread_sync already order.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}
// non-blocking probe (test_wait never suspends the thread): used to look one pipeline stage ahead
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
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
// Two barriers probed by one statement: both try_waits are in flight before either predicate is read, so
// the ~100-cycle barrier round trips overlap (a single-thread issue loop pays the latency once per pair).
__device__ __forceinline__ bool mbar_try_wait2(uint32_t bar0, uint32_t parity0, uint32_t bar1, uint32_t parity1) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 q, [%3], %4;\n\t"
      "and.pred p, p, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar0), "r"(parity0), "r"(bar1), "r"(parity1)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must end in a trap (launch failure the host reports), never in a
// hung GPU.  The bound is wall-clock (globaltimer), 4 s.
// The 64-bit %globaltimer is NOT read atomically (SASS: a CS2R pair on the LO / HI halves; LO wraps every 4.29 s): a read
// that straddles the wrap is off by +-2^32 ns, which a single `now - t0 > 4 s` test takes for a timeout.  Randomised
// stress (tools/estep_stress2.py) hit that about once per 10^4 launches as an "unspecified launch failure" with no
// delay - in every kernel that waits on an mbarrier.  So: signed differences, a torn or backward reading re-arms the
// clock, and the bound must hold on three consecutive probes (a torn reading does not repeat) before the trap.
__device__ __noinline__ void mbar_timeout_trap(uint32_t bar, uint32_t parity, int tag) {
  printf("[scd_b200] mbarrier wait timed out: block %d thread %d tag %d bar 0x%x parity %u\n",
         (int)blockIdx.x, (int)threadIdx.x, tag, bar, parity);
  __trap();
}
// two consecutive readings that agree to within a second: neither is torn
__device__ __forceinline__ uint64_t globaltimer_stable_ns() {
  uint64_t a = globaltimer_ns(), b = globaltimer_ns();
  while ((long long)(b - a) < 0 || b - a > 1000000000ull) { a = b; b = globaltimer_ns(); }
  return b;
}
struct WaitClock {
  uint64_t t0;
  uint32_t spins;
  int over;
  __device__ __forceinline__ WaitClock() : t0(globaltimer_stable_ns()), spins(0), over(0) {}
  // called once per failed probe; true when the wait has really lasted longer than the bound
  __device__ __forceinline__ bool expired() {
    if ((++spins & 0x3FFu) != 0) return false;
    const long long dt = (long long)(globaltimer_ns() - t0);
    if (dt < 0) { over = 0; return false; }                                   // torn / backward reading: ignore it
    if (dt > 4000000000ll && dt < 3600000000000ll) return ++over >= 3;
    over = 0;
    return false;
  }
};
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag = 0) {
  if (mbar_try_wait(bar, parity)) return;
  WaitClock clk;
  while (!mbar_try_wait(bar, parity)) {
    if (clk.expired()) mbar_timeout_trap(bar, parity, tag);
  }
}

// Same bounded wait without a function call on the timeout path: a kernel that moves registers between warp roles
// with setmaxnreg must not call functions (printf is one), or ptxas compiles every role at the launch register count.
// The timed-out wait's tag is left in g_mbar_timeout_tag (best effort: the trap may end the grid before it lands).
__device__ int g_mbar_timeout_tag;
__device__ __forceinline__ void mbar_wait_nocall(uint32_t bar, uint32_t parity, int tag = 0) {
  if (mbar_try_wait(bar, parity)) return;
  WaitClock clk;
  while (!mbar_try_wait(bar, parity)) {
    if (clk.expired()) {
      *reinterpret_cast<volatile int*>(&g_mbar_timeout_tag) = tag;
      __threadfence();
      __trap();
    }
  }
}

// Both barriers of mbar_try_wait2, bounded like mbar_wait_nocall.  Sound only if neither barrier can complete a further
// phase while the waiter spins (each is released by the waiter's own later work).
__device__ __forceinline__ void mbar_wait2_nocall(uint32_t bar0, uint32_t parity0, uint32_t bar1, uint32_t parity1, int tag = 0) {
  if (mbar_try_wait2(bar0, parity0, bar1, parity1)) return;
  WaitClock clk;
  while (!mbar_try_wait2(bar0, parity0, bar1, parity1)) {
    if (clk.expired()) {
      *reinterpret_cast<volatile int*>(&g_mbar_timeout_tag) = tag;
      __threadfence();
      __trap();
    }
  }
}

// ------------------------------------------------------------------ TMA
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void prefetch_tensormap(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
// 2-D tile load, completion bytes signalled on `bar` (a shared::cluster address; with CG==2 the
// leader's barrier).  CG selects the .cta_group qualifier the 2-CTA tensor-core pipeline needs.
template <int CG>
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* desc, uint32_t bar, int c0, int c1,
                                            uint64_t hint) {
  if constexpr (CG == 2) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
  }
}

// 3-D tile load (single-CTA form): used to bring the hi and lo centroid planes in with one instruction
// 1-D bulk copy global -> shared memory of this CTA (no tensor map): `bytes` % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load_1d(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(smem_dst), "l"(gsrc), "r"(bytes), "r"(bar), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const void* desc, uint32_t bar, int c0, int c1, int c2, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(hint)
      : "memory");
}

// ------------------------------------------------------------------ tcgen05
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr, uint32_t ncols) {
  if constexpr (CG == 2)
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "r"(ncols) : "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (CG == 2)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (CG == 2)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate.  One thread issues.
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// Same MMA with the A operand in tensor memory (lane = row, 32-bit column = two consecutive k elements):
// D[tmem] (+)= A[tmem] * B[smem desc].
template <int CG>
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// 32 registers per thread -> 32 lanes x 32 consecutive 32-bit columns (thread = TMEM lane).
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// 16 registers per thread -> 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Completion of every tcgen05 op issued so far by this thread arrives (count 1) on `bar`; with
// CG==2 the arrive is multicast to the barrier at the same offset in every CTA of `cta_mask`.
template <int CG>
__device__ __forceinline__ void umma_commit(uint32_t bar, uint16_t cta_mask) {
  if constexpr (CG == 2) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(cta_mask) : "memory");
  } else {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
  }
}
// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread = TMEM lane).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
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
// 32 lanes x 16 consecutive 32-bit columns -> the first 16 registers (the others are left as they are)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Same wait, but the 32 destination registers of the preceding tcgen05.ld pass through the statement
// as read-write operands: the compiler cannot schedule any use of them above the wait.
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// The 32 registers of a tcgen05.ld that an earlier tcgen05.wait::ld has already covered pass through an empty statement:
// every use of them stays below that wait (one real wait for several loads in flight).
__device__ __forceinline__ void tmem_ld_keep(uint32_t (&r)[32]) {
  asm volatile(""
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// ------------------------------------------------------------------ register reallocation
// Per-thread register budget of the executing warpgroup (all four warps execute the same instruction): .dec hands
// registers back to the CTA's pool, .inc waits until the pool can give them.  N is a multiple of 8 in [24, 256].
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  static_assert(N % 8 == 0 && N >= 24 && N <= 256, "setmaxnreg count");
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  static_assert(N % 8 == 0 && N >= 24 && N <= 256, "setmaxnreg count");
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor, K-major operand, rows densely packed at the swizzle width:
//   bits [0,14) start address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major),
//   [32,46) stride byte offset >> 4 (distance between 8-row groups), [46,48) version = 1 (sm_100),
//   [61,64) layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B, 0 = none.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, uint32_t row_bytes /*128,64,32*/) {
  const uint64_t layout = row_bytes == 128 ? 2ull : (row_bytes == 64 ? 4ull : 6ull);
  const uint64_t sbo = (8u * row_bytes) >> 4;
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (sbo << 32) | (1ull << 46) | (layout << 61);
}
// Instruction descriptor for kind::f16 with bf16 A/B (K-major both), fp32 D:
//   [4,6) D format = 1 (f32), [7,10) A format = 1 (bf16), [10,13) B format = 1 (bf16),
//   [15] A major = 0 (K), [16] B major = 0 (K), [17,23) N >> 3, [24,29) M >> 4.
__host__ __device__ constexpr uint32_t make_idesc_bf16_f32(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace ptx
}  // namespace scd
