// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA, tcgen05 (UMMA) and TMEM.
// Nothing here is generic CUDA; this file only compiles for compute_100a.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>

namespace simstep {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- programmatic dependent launch ------------------------------------------
// Kernels of one env step are launched with programmaticStreamSerialization: a kernel may start while its
// predecessor drains.  grid_dep_wait() blocks until the predecessor has completed and flushed its writes (it
// is a no-op for a normal launch); grid_dep_launch() lets the successor's CTAs be scheduled from here on.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- mbarrier -------------------------------------------------------------

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

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

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Waits for the phase with the given parity to complete.  A barrier that never
// completes is a protocol bug; rather than hanging the GPU (and the box) the
// wait traps after ~2 s so the host sees a launch failure.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("simstep: mbarrier timeout block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}

// ---- TMA ------------------------------------------------------------------

__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

// 2-D tiled load global -> shared of a CTA pair, completion signalled on an mbarrier: the bytes complete on the
// LEADER CTA's barrier (bit 24 of a shared::cluster address selects the CTA of the pair; clearing it addresses the
// even CTA's copy of the barrier).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0,
                                            int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0),
        "r"(c1)
      : "memory");
}

// 1-D bulk copy global -> shared (16-byte aligned addresses, size a multiple of 16), completion on an mbarrier.
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :
               : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// 1-D bulk prefetch global -> L2 (16-byte aligned address, size a multiple of 16).
__device__ __forceinline__ void bulk_prefetch_l2(const void* gmem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes)
               : "memory");
}

// 2-D tiled store shared -> global (bulk async group).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---- TMEM -----------------------------------------------------------------

// Executed by one full warp of EACH CTA of the pair.  Writes the TMEM base address to *smem_result.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(cols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives lane
// (lane_base + i), columns [col, col+32).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// ---- UMMA -----------------------------------------------------------------

// Shared-memory matrix descriptor for a K-major operand tile stored with the
// 128-byte swizzle (rows of 128 B, 8-row groups 1024 B apart).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address, 16-B units
  d |= static_cast<uint64_t>(1) << 16;                      // leading byte offset (unused for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // stride byte offset: next 8-row group
  d |= static_cast<uint64_t>(1) << 46;                      // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B
  return d;
}

// kind: 0 tf32, 1 f16 (fp16 / bf16 operands).  d_tmem (+)= A * B^T, issued by the leader CTA of a pair; A rows
// and B rows (output features) of both CTAs' shared memory form one M 256 x N 256 product.
#define SIMSTEP_UMMA(KINDSTR)                                                                      \
  asm volatile(                                                                                    \
      "{\n\t"                                                                                      \
      ".reg .pred p;\n\t"                                                                          \
      "setp.ne.b32 p, %4, 0;\n\t"                                                                  \
      "tcgen05.mma.cta_group::2.kind::" KINDSTR " [%0], %1, %2, %3, p;\n\t"                       \
      "}\n"                                                                                        \
      :                                                                                            \
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)                         \
      : "memory")
template <int KIND>
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  if constexpr (KIND == 0) SIMSTEP_UMMA("tf32");
  else SIMSTEP_UMMA("f16");
}
#undef SIMSTEP_UMMA

// Arrives on the mbarrier once every previously issued UMMA has completed.  The arrival is multicast to the
// barrier at the same offset in both CTAs of the pair.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(mask)
      : "memory");
}

// ---- clusters ---------------------------------------------------------------

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// Full cluster barrier with release / acquire semantics; every thread of every CTA of the cluster calls it.
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// mbarrier arrive on the barrier at the same offset in CTA `cta_rank` of the cluster.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta_rank) {
  // default semantics (release at cta scope), as CUTLASS's ClusterBarrier::arrive(cta_id): what this arrival hands
  // over is TMEM that the tcgen05 fences already ordered; `.release.cluster` made ptxas emit a gpu-wide MEMBAR +
  // ERRBAR in front of every arrival, the top stall of the short-K epilogues (ncu r02: 27 % of layer 1's samples)
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta_rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t n_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}

__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

}  // namespace ptx
}  // namespace simstep
