// common.cuh -- shared helpers for the sm_100a kernels: error plumbing, PTX wrappers for
// mbarrier / TMA / tcgen05 / TMEM, bf16 packing.  Hand-written; bit layouts follow the PTX ISA
// (tcgen05 matrix/instruction descriptors) -- see DESIGN.md "UMMA descriptors".
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mewzoom_b200.h"

namespace mz {

// ----------------------------------------------------------------------------------------------
// host-side error plumbing
// ----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define MZ_CUDA(expr)                                                        \
  do {                                                                       \
    cudaError_t _e = (expr);                                                 \
    if (_e != cudaSuccess) return ::mz::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define MZ_REQUIRE(cond, ...)          \
  do {                                 \
    if (!(cond)) {                     \
      ::mz::set_error(__VA_ARGS__);    \
      return MZ_ERR_INVALID;           \
    }                                  \
  } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Tensor-map encode through the runtime's driver entry point (no link-time libcuda dependency,
// so the library loads -- and exports its symbols -- on a box without a driver).
int encode_tmap(CUtensorMap* map, CUtensorMapDataType dt, uint32_t rank, void* gaddr, const uint64_t* dims,
                const uint64_t* strides_bytes /*rank-1*/, const uint32_t* box, CUtensorMapSwizzle swz);

int sm_count(int device);

// ----------------------------------------------------------------------------------------------
// device-side PTX wrappers
// ----------------------------------------------------------------------------------------------
#ifdef __CUDACC__

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

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe of a barrier phase.
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded blocking wait.  The retry loop lives INSIDE the asm statement (PTX labels are scoped by the braces):
// to the compiler the wait is one opaque convergent statement, so loop-carried ring state around it stays in
// uniform registers -- a C-level polling loop makes every later value "divergent" and costs an R2UR / ELECT
// waterfall per tcgen05.mma.  A failed try_wait suspends the thread for a hardware-chosen interval and is woken by
// the arrive (an explicit suspend-time hint compiles to NANOSLEEP and adds up to that much latency to every
// wait, so none is given); after MZ_WAIT_LIMIT_TRIES failures a protocol bug traps instead of hanging the GPU.
#ifndef MZ_WAIT_LIMIT_TRIES
#define MZ_WAIT_LIMIT_TRIES 2000000u
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      ".reg .u32 tries;\n\t"
      "mov.u32 tries, 0;\n\t"
      "MZ_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra MZ_DONE;\n\t"
      "add.u32 tries, tries, 1;\n\t"
      "setp.lt.u32 P1, tries, %2;\n\t"
      "@P1 bra MZ_WAIT;\n\t"
      "trap;\n\t"
      "MZ_DONE:\n\t"
      "}\n" ::"r"(bar),
      "r"(parity), "r"(MZ_WAIT_LIMIT_TRIES)
      : "memory");
}

// ---- TMA ----
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// TMA store of a (swizzled) shared-memory box; completion is tracked by the thread's bulk async-group
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// L2 prefetch of a box (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap* m, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still READ their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
// 16-byte chunk index inside a TMA-swizzled row of row_bytes (128 / 64 / 32): the TMA swizzle XORs address bits
// [4, 4+B) with bits [7, 7+B); for a box whose base is aligned to the swizzle period that is a function of the row.
__device__ __forceinline__ uint32_t swz_chunk(uint32_t row, uint32_t chunk, uint32_t row_bytes) {
  return chunk ^ (((row * row_bytes) >> 7) & ((row_bytes >> 4) - 1u));
}

// multicast to every CTA of the cluster named in cta_mask: the box lands at the same CTA-relative offset in each
// destination CTA and completes bytes on the barrier at the same offset there.
__device__ __forceinline__ void tma_load_3d_mcast(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                                  int c2, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, "
      "%5, %6}], [%2], %3;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "h"(cta_mask), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ---- clusters ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- CTA pairs (cta_group::2) ----
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// The same with the default semantics (.release at CTA scope) on a shared::cluster address -- what CUTLASS's
// ClusterBarrier::arrive emits.  The cluster-scope release above costs ~1200 cycles per arrive (measured with the role
// timers of block_fused.cu: it drains the thread's outstanding memory operations cluster-wide); what the waiter
// needs ordered here lives in the ARRIVING CTA's own shared memory / TMEM and is consumed by that CTA's tensor core on a
// command that is issued hundreds of cycles after the arrive is observed (generic -> async proxy ordering is the
// explicit fence.proxy.async before the arrive).
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads of a CTA pair: data lands in the executing CTA, bytes complete on a barrier that may live in the peer
__device__ __forceinline__ void tma2_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1,
                                             int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma2_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1,
                                             int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
      "%5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[each CTA's own 128 rows] * B[N/2 rows from each CTA]; M = 256, issued by the leader CTA
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_acc(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.eq.u32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc)
      : "memory");
}
// arrive (once all previously issued UMMAs of the pair have completed) on the barrier at this offset in the CTAs
// named by cta_mask
__device__ __forceinline__ void umma2_commit_mcast(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(cta_mask)
      : "memory");
}

// ---- programmatic dependent launch ----
// launch_dependents: the next kernel of the stream (launched with programmatic stream serialisation) may start its
// CTAs as soon as every CTA of this grid has executed it (or exited) and resources are free.  wait: blocks until the
// preceding grid has completed and its memory is visible (returns at once when there is no programmatic dependency).
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- tcgen05 / TMEM ----
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the accumulate input hard-wired on (no predicate register to set up per instruction)
__device__ __forceinline__ void umma_acc(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.eq.u32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc)
      : "memory");
}
// mbarrier arrive when all previously issued MMAs of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// same, arriving on the barrier at this offset in every CTA of cta_mask (releases a multicast-filled stage)
__device__ __forceinline__ void umma_commit_mcast(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(cta_mask)
      : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// zero 16 consecutive fp32 columns of this warp's 32 TMEM lanes
__device__ __forceinline__ void tmem_zero16(uint32_t taddr) {
  const uint32_t z = 0u;
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr),
      "r"(z)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---- UMMA descriptors ----
// Shared-memory matrix descriptor, K-major operand, rows of `kc` bf16 (kc = 16/32/64 <=> 32B/64B/128B
// swizzle).  Bits: [0,14) start>>4, [16,30) LBO>>4 (unused for swizzled K-major), [32,46) SBO>>4,
// [46,48) version = 1, [49,52) base offset, [61,64) layout type (2 = 128B, 4 = 64B, 6 = 32B).
__host__ __device__ constexpr uint32_t umma_layout_type(int kc) { return kc == 64 ? 2u : (kc == 32 ? 4u : 6u); }

__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout_type,
                                                   uint32_t base_offset = 0) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;  // LBO (ignored for swizzled K-major; CUTLASS writes 1)
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (sm_100)
  d |= static_cast<uint64_t>(base_offset & 7u) << 49;
  d |= static_cast<uint64_t>(layout_type & 7u) << 61;
  return d;
}
// Instruction descriptor: D fp32 (bits [4,6) = 1), A/B bf16 ([7,10) = [10,13) = 1), both K-major,
// N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
// Same with fp16 operands (A/B format 0): identical tensor-core rate, 10-bit mantissa.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// ---- misc ----
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {  // saturating: never produces inf
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2_rn(float lo, float hi) {  // plain rounding: +-inf beyond the range, as torch
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// MMA-operand element type of the activations / weights: 0 = fp16 (default), 1 = bf16.
__device__ __forceinline__ uint32_t pack_op2(int bf16, float lo, float hi) {
  return bf16 ? pack_bf16x2(lo, hi) : pack_f16x2(lo, hi);
}
// A 16-bit shadow of an fp32 tensor that is not range-tracked: exactly what `x.to(dtype)` gives, so that it can stand in
// for that cast (out-of-range values become inf, not a silently clipped +-65504).
__device__ __forceinline__ uint32_t pack_shadow2(int bf16, float lo, float hi) {
  return bf16 ? pack_bf16x2(lo, hi) : pack_f16x2_rn(lo, hi);
}
// two packed 16-bit operands -> floats (x = low half)
__device__ __forceinline__ float2 unpack_op2(int bf16, uint32_t u) {
  if (bf16) return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
__device__ __forceinline__ float op_to_float(int bf16, uint16_t v) {
  return bf16 ? __uint_as_float(static_cast<uint32_t>(v) << 16) : __half2float(__ushort_as_half(v));
}
// SiLU(v) = v * sigmoid(v) = h + h * tanh(h), h = v / 2: one MUFU (tanh.approx, rel. error ~2^-11, far below the
// bf16 rounding of the stored result) instead of ex2 + rcp.
__device__ __forceinline__ float silu_f(float v) {
  const float h = 0.5f * v;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// The same with the halving folded into the caller's affine transform: silu_h(v / 2) == silu_f(v) bit for bit
// (scaling by 1/2 is exact), one multiply less per value.
__device__ __forceinline__ float silu_h(float h) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

#endif  // __CUDACC__

}  // namespace mz
