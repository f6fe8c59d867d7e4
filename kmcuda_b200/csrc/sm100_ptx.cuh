// sm100_ptx.cuh -- thin inline-PTX wrappers for the Blackwell (sm_100a) features the assignment
// kernel uses: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (TMEM alloc, MMA, commit, ld).
// Nothing here is CUTLASS; descriptor bit layouts follow the PTX ISA "tcgen05" matrix/instruction
// descriptor tables.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace kmb {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// one lane of the (converged) warp is elected; every lane gets the same answer about itself
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// Bounded wait: a stuck pipeline must not hang the GPU box.  Returns false after ~2 s of SM clocks
// or as soon as another thread has published an error in *err (global memory).
// The try_wait carries a suspend-time hint, which ptxas turns into TRYWAIT + NANOSLEEP.SYNCS: a waiting warp
// sleeps until the barrier's phase flips (or the hint expires) instead of competing for issue slots.  Round 1
// spun without a hint: 14 SASS instructions per probe and ~40 % of all issued instructions of the kernel were
// such probes (profiles/r01_tc_assign_v4: 150 M SYNCS + 350 M BRA), stolen from the converter / epilogue warps
// of the same scheduler.
constexpr uint32_t kWaitHintNs = 2000;    // inline probe of every wait
constexpr uint32_t kSlowHintNs = 20000;   // probes of the out-of-line remainder (mbar_wait_slow)
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity, uint32_t hint_ns) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(addr), "r"(parity), "r"(hint_ns)
      : "memory");
  return done != 0;
}
// Out-of-line remainder of every wait: a TIGHT polling loop (round 2's first version re-checked the error word and
// the clock in the loop body: ncu counted 0.9 G warp instructions per pass -- a third of everything the kernel issued --
// in that loop, because a hinted try_wait returns on every update of the barrier, not only when the phase flips).
// `site` names the waiting role; after ~2 s (or as soon as another thread has reported an error) the wait gives up and
// reports 0x1000 + site in *err: a stuck pipeline must not hang the GPU box.
__device__ __noinline__ void mbar_wait_slow(uint32_t addr, uint32_t parity, uint32_t* err, uint32_t site, uint32_t flag_u32) {
  // flag_u32: a word of this CTA's shared memory that is set once any wait of the CTA has given up; from then on every
  // wait returns at once, so a broken pipeline drains in milliseconds instead of timing out wait by wait
  uint32_t dead;
  asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(dead) : "r"(flag_u32));
  if (dead) return;
  const long long t0 = clock64();
  for (;;) {
    uint32_t done;
    // 1024 probes in a loop of 7 SASS instructions (probe, predicated sleep + re-check, counter, compare, branch)
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b32 c;\n\t"
        "mov.u32 c, 0;\n"
        "KMB_WAIT_LOOP_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "@p bra KMB_WAIT_DONE_%=;\n\t"
        "add.u32 c, c, 1;\n\t"
        "setp.lt.u32 q, c, 1024;\n\t"
        "@q bra KMB_WAIT_LOOP_%=;\n"
        "KMB_WAIT_DONE_%=:\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(kSlowHintNs)
        : "memory");
    if (done) return;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(dead) : "r"(flag_u32));
    const bool lost = dead || *reinterpret_cast<volatile uint32_t*>(err);
    if (lost || clock64() - t0 > 4000000000ll) {
      if (!lost) atomicMax(err, 0x1000u + site);
      asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(flag_u32), "r"(1u) : "memory");
      return;
    }
  }
}
// The inline part: one probe (with the suspend hint it may sleep up to the hint while the phase has not flipped).
__device__ __forceinline__ void mbar_wait(uint32_t addr, uint32_t parity, uint32_t* err, uint32_t site, uint32_t flag_u32) {
  if (!mbar_try_wait(addr, parity, kWaitHintNs)) mbar_wait_slow(addr, parity, err, site, flag_u32);
}

// ---------------------------------------------------------------------------- packed fp32 pairs (sm_100: FADD2 / FMUL2 / FFMA2)
// One instruction, two IEEE fp32 operations (same rounding as the scalar forms).  Used where every lane walks a
// whole row: halves the issue slots of the converter and of the epilogue's threshold compare.
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fsub2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
// three-input maximum (FMNMX3); NaN operands are ignored like fmaxf
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// generic-proxy writes to shared memory -> visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tiled load: coordinates {c0 (innermost), c1}
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 1-D bulk copy global -> shared (size multiple of 16, both 16-byte aligned)
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], fp16/bf16 inputs, fp32 accumulate; one thread issues
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand taken from tensor memory (128 lanes x 8 columns of packed fp16 pairs per K=16)
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// One K-block of the TS form in a single statement: four K=16 steps (A: +8 TMEM columns per step; B: +32 bytes along K
// inside the 128-byte swizzle atom = +2 in the descriptor's address field), then a commit that arrives on `bar_u32`
// (shared-space address) when they have retired.  Keeping it one asm block keeps the issue sequence dense.
__device__ __forceinline__ void umma_f16_ts_kblock(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                                   uint32_t accumulate_first, uint32_t bar_u32) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 d1, d2, d3;\n\t.reg .b32 a1, a2, a3;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 q, 0, 0;\n\t"
      "add.u64 d1, %2, 2;\n\tadd.u64 d2, %2, 4;\n\tadd.u64 d3, %2, 6;\n\t"
      "add.u32 a1, %1, 8;\n\tadd.u32 a2, %1, 16;\n\tadd.u32 a3, %1, 24;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [a1], d1, %3, q;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [a2], d2, %3, q;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [a3], d3, %3, q;\n\t"
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate_first), "r"(bar_u32)
      : "memory");
}
__device__ __forceinline__ void umma_commit_u32(uint32_t bar_u32) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_u32) : "memory");
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar_u32) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_u32) : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp receives lane (base_lane + t)
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
// store 32 registers to 32 consecutive columns of this thread's lane (lane = base_lane + thread)
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
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------- CTA pairs (cta_group::2)
// Two CTAs of one cluster (the two SMs of a TPC) run ONE tcgen05.mma of M = 256: each CTA holds its 128 rows of A and
// of the accumulator in its own tensor memory and HALF of the B tile (N / 2 rows) in its own shared memory; the
// leader CTA (cluster rank 0) issues the instruction for both.  Per SM this halves the B traffic: L2 -> shared memory
// copies, shared-memory writes and the tensor core's shared-memory reads.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_u32` (a shared::cta address of this CTA's layout) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_u32, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_u32), "r"(rank));
  return r;
}
// Arrive on a barrier of another CTA of the cluster.  RELAXED: what the waiter (the leader's MMA thread) consumes was
// produced through tensor memory and is ordered by tcgen05.wait::ld / wait::st + tcgen05.fence::before_thread_sync; a
// .release at cluster scope compiles to a cluster-wide memory barrier in front of every arrive (ncu of the first
// CTA-pair build: half of the epilogue warps' time was that barrier).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 2-D tiled load into THIS CTA's shared memory whose completion bytes are counted on the barrier at `leader_bar_u32`
// (a shared::cluster address inside the leader CTA)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst_u32, const void* tmap, int c0, int c1, uint32_t leader_bar_u32) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst_u32), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(leader_bar_u32), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {  // the same warp of BOTH CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// commit of the leader's MMAs: arrives on the barrier at the same shared-memory offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint32_t bar_u32) {
  asm volatile(
      "{\n\t.reg .b16 m;\n\tmov.b16 m, 3;\n\t"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
      ::"r"(bar_u32)
      : "memory");
}
// one K-block (TS form) for the pair: 4 x (M = 256, N = 128, K = 16), then the multicast commit
__device__ __forceinline__ void umma_f16_ts_kblock_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                                        uint32_t accumulate_first, uint32_t bar_u32) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 d1, d2, d3;\n\t.reg .b32 a1, a2, a3;\n\t.reg .b16 m;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 q, 0, 0;\n\t"
      "mov.b16 m, 3;\n\t"
      "add.u64 d1, %2, 2;\n\tadd.u64 d2, %2, 4;\n\tadd.u64 d3, %2, 6;\n\t"
      "add.u32 a1, %1, 8;\n\tadd.u32 a2, %1, 16;\n\tadd.u32 a3, %1, 24;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [a1], d1, %3, q;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [a2], d2, %3, q;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [a3], d3, %3, q;\n\t"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], m;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate_first), "r"(bar_u32)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---------------------------------------------------------------------------- descriptors
// shared-memory matrix descriptor (PTX ISA, tcgen05 "matrix descriptor"):
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4   [46,48) version = 1 (sm_100)
//   [49,52) base offset = 0           [52]    LBO mode = 0
//   [61,64) layout: 0 none, 1 128B(base 32B), 2 128B, 4 64B, 6 32B
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout & 7) << 61;
  return d;
}
// instruction descriptor for kind::f16 (PTX ISA, tcgen05 "instruction descriptor"):
//   [4,6) D format (1 = f32)  [7,10) A format (0 = f16, 1 = bf16)  [10,13) B format
//   [15] A major (0 = K)  [16] B major (0 = K)  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | (0u << 15) | (0u << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

__device__ __forceinline__ float4 ldg_nc_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}

}  // namespace ptx
}  // namespace kmb
