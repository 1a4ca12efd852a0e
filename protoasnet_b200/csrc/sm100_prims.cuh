// sm_100a primitives used by the fused prototype-head kernel: mbarrier, cp.async, bulk async copy, tcgen05
// (TMEM alloc / mma / commit / ld / st / fences), UMMA shared-memory + instruction descriptors, and the address
// functions of the canonical operand layouts.  Inline PTX only; field layouts follow the PTX ISA "tcgen05 matrix /
// instruction descriptor" tables (cross-checked against cute/arch/mma_sm100_desc.hpp in the vendored CUTLASS headers).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace pasn {
namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
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
// non-blocking probe (try_wait may suspend the thread for a while; test_wait never does)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug becomes an error code in *err instead of a hung GPU.
#ifndef PASN_MBAR_SPIN_LIMIT
#define PASN_MBAR_SPIN_LIMIT (1u << 26)
#endif
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* err, int code) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > PASN_MBAR_SPIN_LIMIT) {
      if (err) atomicCAS(err, 0, code);
      return false;
    }
  }
  return true;
}

// ----------------------------------------------------------------------------------------------
// async copies
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async_8(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_16(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// streaming 8-byte global load that does not allocate in L1
__device__ __forceinline__ uint2 ldg_nc_na_v2(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ldg_nc_na_v4f(const void* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_shared_v2(uint32_t saddr, uint2 v) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(saddr), "r"(v.x), "r"(v.y) : "memory");
}
// programmatic dependent launch: wait until the preceding grid in the stream has completed and flushed its writes /
// allow the following grid to start launching
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// L2 eviction-priority policies and hinted accesses (createpolicy + .L2::cache_hint)
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void st_global_u16_hint(void* ptr, uint16_t v, uint64_t policy) {
  asm volatile("st.global.L2::cache_hint.u16 [%0], %1, %2;" ::"l"(ptr), "h"(v), "l"(policy) : "memory");
}
__device__ __forceinline__ void cp_async_8_hint(uint32_t dst_smem, const void* src, uint32_t src_bytes, uint64_t policy) {
  asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 8, %2, %3;" ::"r"(dst_smem), "l"(src), "r"(src_bytes), "l"(policy) : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
               : "memory");
}

// arrive on `bar` (without bumping its pending count) once all cp.async issued so far by this thread have landed
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// generic-proxy writes (st.shared / cp.async) -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// TMEM allocation (one warp, .sync.aligned)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// descriptors
// ----------------------------------------------------------------------------------------------
enum : uint32_t { SWZ_NONE = 0, SWZ_128B = 2, SWZ_64B = 4, SWZ_32B = 6 };

// 64-bit shared-memory matrix descriptor: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) |
// base_offset [49,52) = 0 | lbo_mode [52] = 0 | layout_type [61,64)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t swz) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(swz & 7) << 61;
  return d;
}
// advance the start-address field by `bytes` (stays inside the 14-bit field for <256 KB of smem)
__device__ __forceinline__ uint64_t desc_advance(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

// 32-bit instruction descriptor for kind::f16, bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major, uint32_t b_mn_major) {
  return (1u << 4)      // c_format = F32
         | (1u << 7)    // a_format = BF16
         | (1u << 10)   // b_format = BF16
         | ((a_mn_major & 1u) << 15) | ((b_mn_major & 1u) << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// kind::f16 with per-operand element type (F16 = 0, BF16 = 1), fp32 accumulate
__host__ __device__ constexpr uint32_t make_idesc_16(uint32_t M, uint32_t N, uint32_t a_bf16, uint32_t b_bf16, uint32_t a_mn_major,
                                                     uint32_t b_mn_major) {
  return (1u << 4) | ((a_bf16 & 1u) << 7) | ((b_bf16 & 1u) << 10) | ((a_mn_major & 1u) << 15) | ((b_mn_major & 1u) << 16) |
         ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------
// tcgen05.mma / commit
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Lean issue forms for a single elected thread: descriptors travel as (lo, hi) 32-bit halves so that advancing the
// start address is one 32-bit add on the low word (the 14-bit address field never carries for < 256 KB of smem) and the
// constant high word (LBO/SBO/version/swizzle) is folded by the compiler.  ACC = 1 accumulates, 0 overwrites.
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__host__ __device__ constexpr uint32_t desc_hi(uint32_t sbo_bytes, uint32_t swz) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((swz & 7u) << 29);
}
__device__ __forceinline__ void mma_ss_x(uint32_t d_tmem, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
      "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_ts_x(uint32_t d_tmem, uint32_t a_tmem, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit_a(uint32_t bar_saddr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_saddr) : "memory");
}
// one lane of a converged warp (CUTLASS' elect_one_sync); ptxas knows the guarded region runs in a single thread
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ----------------------------------------------------------------------------------------------
// CTA pairs (cta_group::2): one thread of the leader CTA issues MMAs that span both CTAs of a 2-CTA cluster.
// M = 256: each CTA supplies its own 128 rows of A (same smem / TMEM address in both CTAs) and receives its own
// 128 rows of D; each CTA supplies N/2 rows of B at the same smem address.  Every tcgen05 alloc/mma/commit in such a
// kernel uses cta_group::2.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same variable in CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void mma_ss2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_ts2(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// lean single-thread forms (descriptors as 32-bit halves, see mma_ss_x)
__device__ __forceinline__ void mma_ss2_x(uint32_t d_tmem, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
      "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit2_a(uint32_t bar_saddr, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar_saddr),
               "h"(cta_mask)
               : "memory");
}
// arrive (once per listed CTA) on the mbarrier at this smem offset when all prior MMAs of the issuing thread retired
__device__ __forceinline__ void mma_commit2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// TMEM <-> registers (32 lanes x 32-bit; thread i of warp w touches lane 32*(w%4)+i)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// pack two fp32 -> bf16x2 (lo = first / even element)
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// pack two fp32 -> f16x2 (lo = first / even element)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// max(x, 0) folded into the conversion (cvt.rn.relu)
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// ----------------------------------------------------------------------------------------------
// canonical operand layouts (byte offsets inside one operand image; image base 1024-byte aligned)
// ----------------------------------------------------------------------------------------------
// K-major, 128-byte swizzle, one 64-element (128 B) K chunk: row r (M or N index), K element k in [0,64)
//   atoms of 8 rows x 128 B; 16-byte units XOR-swizzled with (r % 8).  Descriptor: SBO = 1024, K-step (+16 el) = +32 B.
__host__ __device__ __forceinline__ uint32_t off_kmajor_sw128(uint32_t r, uint32_t k) {
  return (r >> 3) * 1024u + (r & 7u) * 128u + ((((k >> 3) ^ (r & 7u)) & 7u) << 4) + (k & 7u) * 2u;
}
// MN-major, 128-byte swizzle: mn = M/N index, k = K index.  Atom = 64 mn-elements (128 B) x 8 k-rows (1024 B);
//   k-atoms (8 k) contiguous at SBO = 1024; mn-atoms (64 mn) at LBO = lbo_bytes.  K-step (+16 k) = +2*SBO.
__host__ __device__ __forceinline__ uint32_t off_mnmajor_sw128(uint32_t mn, uint32_t k, uint32_t lbo_bytes) {
  return (mn >> 6) * lbo_bytes + (k >> 3) * 1024u + (k & 7u) * 128u + (((((mn & 63u) >> 3) ^ (k & 7u)) & 7u) << 4) +
         (mn & 7u) * 2u;
}
// MN-major, no swizzle ("interleave"): core matrix = 8 k-rows x 16 B (8 mn-elements) = 128 contiguous bytes;
//   mn-groups (8 mn) at SBO = 128, k-groups (8 k) at LBO = (MN/8)*128.  K-step (+16 k) = +2*LBO.
__host__ __device__ __forceinline__ uint32_t off_mnmajor_nosw(uint32_t mn, uint32_t k, uint32_t mn_extent) {
  return (k >> 3) * (mn_extent >> 3) * 128u + (mn >> 3) * 128u + (k & 7u) * 16u + (mn & 7u) * 2u;
}

}  // namespace sm100
}  // namespace pasn
