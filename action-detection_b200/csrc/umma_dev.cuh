// Device-side tcgen05 / TMA / mbarrier primitives shared by the tensor-core kernels (inline PTX).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ssnb {
namespace umma {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;             // fp16 elements = 128 B = one SWIZZLE_128B row
constexpr int UMMA_K = 16;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug traps (-> launch error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout_type=2 [61,64)
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                 // leading byte offset (unused for swizzled K-major) = 16 B
  d |= (uint64_t)(1024 >> 4) << 32;       // stride byte offset: 8 rows x 128 B
  d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
  return d;
}

// instruction descriptor, kind::f16: D=f32, A=B=f16, both K-major, M=128, N=n
__device__ __forceinline__ uint32_t make_idesc_f16(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// descriptor words for issue loops that only ever add to the address field
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | (1u << 16); }
__device__ __forceinline__ uint32_t desc_hi_sw128(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (2u << 29); }
__device__ __forceinline__ void umma_f16_lohi(uint32_t tmem_d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
      "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// one lane of a converged warp (warp-uniform role loops: everybody walks the pipeline, this lane issues)
__device__ __forceinline__ bool elect_one_lane() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- CTA pair (cta_group::2) forms ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `saddr` (a shared::cta address of this CTA's layout) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(mapa_shared(smem_u32(bar), rank)) : "memory");
}
// TMA loads issued by either CTA of a pair: data lands in the issuing CTA's shared memory, the transaction bytes are
// counted on `bar_cluster` (a shared::cluster address, normally the leader's barrier)
__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ uint32_t make_idesc_f16_m(int m, int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_f16_lohi_pair(uint32_t tmem_d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                                   uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
      "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at this shared-memory offset in BOTH CTAs of the pair when the prior MMAs retire
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// kind::f16 instruction descriptor with both operands MN-major (a_major bit 15, b_major bit 16)
__device__ __forceinline__ uint32_t make_idesc_f16_mn(int n) {
  return (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
}

}  // namespace umma
}  // namespace ssnb
