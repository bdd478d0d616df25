// Thread-block cluster and tcgen05 cta_group::2 primitives shared by the fused layer chain (head_chain4.cu) and the batched
// weight-gradient GEMM (gemm2cta.cu). Both run an SM pair {2p, 2p+1} of a cluster as one tensor-core unit:
//   - tcgen05.alloc / dealloc .cta_group::2 are issued by the same warp index in both CTAs, with the same destination offset
//   - the TMA loads of both CTAs complete on the pair LEADER's (even CTA's) barrier of the same offset (kPairLeaderMask)
//   - tcgen05.mma.cta_group::2 is issued by the leader's MMA warp only
//   - tcgen05.commit.cta_group::2 ... multicast::cluster arrives on the barrier of the same offset in every CTA of the mask
// PTX forms follow the vendored CUTLASS headers (cute/arch/copy_sm100_tma.hpp, mma_sm100_umma.hpp, tmem_allocator_sm100.hpp,
// cutlass/arch/barrier.h).
#pragma once
#include "common.cuh"

namespace acez {

#ifdef __CUDACC__
static constexpr uint32_t kPairLeaderMask = 0xFEFFFFFFu;  // clears the pair bit of a shared::cluster address: the even CTA of the pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the shared::cta address `addr` in the CTA of cluster rank `rank`
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote_release(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// plain arrive on the pair leader's barrier of the same offset (executed by the other CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPairLeaderMask) : "memory");
}
// bulk copy shared::cta -> shared::cluster (another CTA's shared memory), completing (bytes) on that CTA's mbarrier
__device__ __forceinline__ void dsmem_copy(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t mbar_cluster) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_cluster),
               "r"(src_cta), "r"(bytes), "r"(mbar_cluster)
               : "memory");
}

__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA load of a CTA of the pair: completes (bytes) on the pair leader's barrier of the same offset
__device__ __forceinline__ void tma_load_3d_pair(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar) & kPairLeaderMask), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// D[tmem of both CTAs] (+)= A[smem desc, per CTA] * B[smem desc, both halves], kind::f16; issued by the pair leader
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior UMMAs of the pair retire) on the barrier of this offset in every CTA of `cta_mask`
__device__ __forceinline__ void tcgen05_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
#endif  // __CUDACC__

}  // namespace acez
