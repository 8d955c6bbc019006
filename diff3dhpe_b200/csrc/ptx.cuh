// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Descriptor bit layouts follow the PTX ISA "tcgen05 shared memory descriptor" / "instruction descriptor"
// tables (cross-checked against cute/arch/mma_sm100_desc.hpp in the image's vendored CUTLASS headers).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace d3d {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
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
// Blocking wait with a watchdog: a protocol bug traps (-> cudaErrorLaunchFailure) instead of hanging the GPU.
// try_wait carries a suspend-time hint, so a waiting warp SLEEPS in hardware (NANOSLEEP.SYNCS) until the barrier's
// phase completes or the hint expires, instead of re-issuing try_wait every ~50 cycles: ncu on the hint-less form
// counted 17 % of all executed instructions of the attention kernel in these spin loops and showed the XU pipe (which
// MUFU.EX2 / RCP and the float conversions of the epilogues need) at 87-120 % in the GEMM kernels
// (profiles/r01zc_full_gemm.md).  D3D_MBAR_SUSPEND_NS = 0 restores the busy spin.
#ifndef D3D_MBAR_SUSPEND_NS
#define D3D_MBAR_SUSPEND_NS 1000000
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
#if D3D_MBAR_SUSPEND_NS > 0
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity), "r"(static_cast<uint32_t>(D3D_MBAR_SUSPEND_NS))
        : "memory");
    if (ok) return;
    if (spin >= 4) {                                  // a handful of expired 1 ms hints: start the clock
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) __trap();   // ~2 s at 2 GHz
    }
#else
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
    if ((spin & 0x3fff) == 0x3fff) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) __trap();   // ~2 s at 2 GHz
    }
#endif
  }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tiled load global -> shared, completion signalled on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                            int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// ---------------------------------------------------------------- thread-block cluster (CTA pair) helpers
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// Arrive on a barrier that may live in another CTA of the cluster.  Default .release.cta semantics (as CUTLASS'
// ClusterBarrier::arrive): the .release.cluster form costs a cluster-scope membar that waits for every in-flight
// global store of the warp -- ncu showed ERRBAR/membar as the top stall of the epilogue warps with it.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load issued by either CTA of a pair; the completion bytes are signalled on `bar_cluster_addr`, which may
// live in the peer (leader) CTA's shared memory.
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr,
                                                int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// Multicast variant: the box is written at the same CTA-relative offset of every CTA in `cta_mask` (bit r = cluster
// rank r); the completion bytes are signalled, per destination CTA, on the barrier at `bar_cta_addr`'s offset in the
// EVEN CTA of that destination's pair (bit 24 of the executing CTA's own shared address cleared, as CUTLASS'
// SM100_TMA_2SM_LOAD_MULTICAST does).
__device__ __forceinline__ void tma_load_2d_cg2_mc(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                                   int32_t c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
      "[%0], [%1, {%4, %5}], [%2], %3;"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "h"(cta_mask),
        "r"(c0), "r"(c1)
      : "memory");
}
// L2 eviction-priority policies for TMA loads: mode 0 normal, 1 evict_last (keep: operands re-read by other CTAs),
// 2 evict_first (streamed once)
__device__ __forceinline__ uint64_t make_l2_policy(int mode) {
  uint64_t pol;
  if (mode == 1) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  else if (mode == 2) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_2d_cg2_hint(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr,
                                                     int32_t c0, int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1),
        "l"(policy)
      : "memory");
}
// streaming (evict-first) 16-byte global accesses for data touched once by this kernel
__device__ __forceinline__ void st_global_cs(void* p, uint4 v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float4 ld_global_cs(const float* p) {
  float4 v;
  asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// Packed fp32 pairs (sm_100 FFMA2 / FMUL2 / FADD2): one fma-pipe issue slot per TWO IEEE-rn operations.  The 3-register
// scalar FFMA issues every other cycle per scheduler, so fp32-heavy epilogues are fma-pipe bound; packing halves that.
using f32x2 = unsigned long long;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ f32x2 splat2(float v) { return pack2(v, v); }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B with M = 256 split over the CTA pair (each CTA: its 128 rows of A and half of
// the N rows of B, at the same shared-memory offsets).  Issued by one thread of the leader CTA.
__device__ __forceinline__ void mma_f16_ss_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once all prior tcgen05.mma of this thread completed) on the barrier at this offset in every CTA of
// `cta_mask` (bit r = CTA rank r of the cluster).
__device__ __forceinline__ void mma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; kind::f16 (fp16/bf16 operands, fp32 accumulate).  One thread issues.
__device__ __forceinline__ void mma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f8f6f4 (here: e5m2 x e5m2, fp32 accumulate; K = 32 per instruction, twice the kind::f16 rate)
__device__ __forceinline__ void mma_f8_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_f8_ss_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers: 32 lanes x 32 consecutive fp32 columns; thread i of the warp gets lane (base+i).
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
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- 4-D TMA (strided token gathers / scatters)
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1,
                                            int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3)
      : "memory");
}
// shared -> global tiled store (bulk async-group completion); rows outside the tensor are clipped by the hardware
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1,
                                             int32_t c2, int32_t c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// L2 prefetch of a tiled box (no shared-memory destination, no completion): HBM -> L2 ahead of the TMA load that needs it
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* m, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1)
               : "memory");
}
// shared-space accesses with 32-bit addresses (a generic pointer costs a 64-bit add and a generic-space LD / ST per access)
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// shared -> global tiled REDUCTION (fp32 add performed by the L2: the destination tile never enters the SM);
// rows / columns outside the tensor are clipped by the hardware
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, uint32_t smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// named barrier among `n_threads` threads (ids 1..15; 0 is __syncthreads)
__device__ __forceinline__ void bar_sync(uint32_t id, uint32_t n_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}

// registers -> TMEM: 32 lanes x 16 consecutive 32-bit columns; thread i of the warp writes lane (base+i)
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]: the A operand (M = 128 rows = lanes, K 16-bit elements packed two per 32-bit
// column) is read from tensor memory -- P of the attention P.V product never touches shared memory.
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Shared-memory matrix descriptor for a K-major operand tile whose rows are 128 bytes (64 fp16) wide and
// stored with the 128-byte swizzle (exactly what a SWIZZLE_128B TMA box of {64, rows} writes):
//   bits [0,14)  start address >> 4          bits [16,30) leading byte offset >> 4 (ignored for SW128 K-major)
//   bits [32,46) stride byte offset >> 4     (8 rows x 128 B = 1024 B between 8-row groups)
//   bits [46,48) descriptor version = 1      bits [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// The same for 64-byte (32 fp16) rows in the 64-byte swizzle (a SWIZZLE_64B TMA box of {32, rows}): 8 rows x 64 B = 512 B
// between 8-row groups, layout type = 4 (SWIZZLE_64B)
__device__ __forceinline__ uint64_t make_desc_k_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(512 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(4) << 61;
  return d;
}

// Shared-memory descriptor of a tcgen05.cp.32x128b source: 32 rows x 16 bytes stored contiguously (row r at 16 r), i.e.
// four 8-row x 16-byte core matrices 128 bytes apart, K-major, no swizzle: SBO = 128 B, LBO unused (one core matrix
// along K), version 1, layout type 0.  This is the 512-byte scale-factor atom of operand.cuh.
__device__ __forceinline__ uint64_t make_desc_sf(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(128 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}
// smem -> TMEM copy of one scale-factor atom: 32 lanes x 128 bits (4 columns), replicated into the four lane quadrants.
// Executes in issue order with the tcgen05.mma of the same thread (no wait in between).  cta_group::2: issued by the
// leader, performed in BOTH CTAs of the pair from the same shared-memory offset to the same TMEM address.
__device__ __forceinline__ void utccp_32x128b_cg2(uint32_t tmem_dst, uint64_t desc) {
  asm volatile("tcgen05.cp.cta_group::2.32x128b.warpx4 [%0], %1;" ::"r"(tmem_dst), "l"(desc) : "memory");
}
// D[tmem of both CTAs] (+)= A * B, kind::mxf4 (packed e2m1 operands in shared memory, K = 64 per instruction, 4x the
// kind::f16 rate) with one ue8m0 scale per 32 elements of K for every row of A and B (scale_vec::2X), read from TMEM:
// sfa / sfb = TMEM addresses of the 4 (A: 128 rows per CTA) / 8 (B: 256 rows) scale columns; which 2 of the 4 bytes of
// a column this MMA uses is the SF id in the instruction descriptor.
__device__ __forceinline__ void mma_mxf4_ss_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                uint32_t sfa, uint32_t sfb, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%5], [%6], p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(sfa), "r"(sfb)
      : "memory");
}
// Block-scaled instruction descriptor, kind::mxf4: A / B format e2m1 (= 1) at bits [7,10) / [10,13), K-major operands,
// N>>3 at [17,23), scale format ue8m0 (bit 23), M>>4 at [24,29), K = 64 (bit 31 = 0); the per-MMA SF ids go to bits
// [4,6) (B) and [29,31) (A).  (cute/arch/mma_sm100_desc.hpp InstrDescriptorBlockScaled.)
__host__ __device__ constexpr uint32_t make_idesc_mxf4(uint32_t M, uint32_t N, uint32_t sf_id) {
  return (sf_id << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | (1u << 23) | ((M >> 4) << 24) | (sf_id << 29);
}

// Instruction descriptor, kind::f16: fp32 accumulate (bits[4,6)=1), A/B format (bits[7,10),[10,13): 0 fp16,
// 1 bf16), both operands K-major (bits 15,16 = 0), N>>3 at bits [17,23), M>>4 at bits [24,29).
// kind::f8f6f4 uses the same layout with A/B format 0 = e4m3, 1 = e5m2.
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N, uint32_t ab_format) {
  return (1u << 4) | (ab_format << 7) | (ab_format << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace ptx
}  // namespace d3d
