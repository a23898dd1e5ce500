// ptx.cuh — thin inline-PTX wrappers (sm_100a): mbarrier, TMA bulk copy, cluster barrier, DSMEM.
#pragma once
#include <stdint.h>

namespace b200rnn {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier -----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make the init visible to the async (TMA) proxy and to the cluster
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// plain arrive (release at CTA scope): used when the producer wrote LOCAL shared memory with ordinary stores
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// one lane of the (fully converged) warp returns true; unlike `lane == 0` the compiler keeps the enclosed code on
// the uniform datapath (tcgen05.mma / commit operands in uniform registers, no per-instruction broadcast loop)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- TMA 1-D bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP) -----------------
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- thread-block cluster -----------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
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
// shared::cta address -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}

// st.async: 16-byte store into a peer CTA's shared memory that also completes 16 bytes of the transaction
// count of an mbarrier in THAT CTA — data and signal travel together, no fence / cluster barrier needed.
// Both addresses are shared::cluster addresses (mapa) of the same target CTA.
__device__ __forceinline__ void st_async_v4(uint32_t cluster_addr, float4 v, uint32_t cluster_mbar) {
  asm volatile(
      "st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
          cluster_addr),
      "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(cluster_mbar)
      : "memory");
}

}  // namespace ptx
}  // namespace b200rnn
