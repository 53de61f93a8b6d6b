// sm_100a device primitives used by the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (UMMA issue/commit, TMEM alloc/ld), descriptors.  Thin inline-PTX wrappers only.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cwg { namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
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
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {   // generic-proxy smem writes -> async proxy (TMA / UMMA)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// Wait only until the bulk stores have finished READING shared memory (enough before reusing the
// staging tiles or exiting the CTA; the global writes complete on their own).
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ---------------------------------------------------------------- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// ---------------------------------------------------------------- UMMA
// Shared-memory matrix descriptor for a K-major tile stored as rows of 128 bytes (64 bf16) with
// the 128-byte swizzle (what a TMA box {64, rows} with CU_TENSOR_MAP_SWIZZLE_128B writes):
// 8-row groups are 1024 bytes apart (SBO); LBO is unused for swizzled K-major; version 1 (sm_100).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);          // start address, bits [0,14)
  d |= (uint64_t)(1024 >> 4) << 32;                     // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                               // descriptor version
  d |= (uint64_t)2 << 61;                               // SWIZZLE_128B
  return d;
}
// The same for a K-major tile whose rows are 32 bytes (16 x 16-bit: exactly one K = 16 MMA step) with the 32-byte swizzle
// (a TMA box {16, rows} with CU_TENSOR_MAP_SWIZZLE_32B): 8-row groups are 256 bytes apart.
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;                               // SWIZZLE_32B
  return d;
}
// Instruction descriptor, kind::f16: bf16 x bf16 -> fp32, both operands K-major.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// fp16 x fp16 -> fp32 uses the same kind::f16 instruction with the F16 operand formats.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// kind::f8f6f4, e5m2 x e5m2 -> fp32, both operands K-major (K = 32 per instruction).
__host__ __device__ constexpr uint32_t umma_idesc_e5m2(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// 8 x 32-bit columns of this thread's TMEM lane (warp w may only touch lanes 32*(w%4) .. +31).
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// mbarrier arrives once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------- 2-SM (cta_group::2) forms
// A CTA pair (cluster ranks 2k, 2k+1) executes one MMA with M = 256: the leader (even rank) issues it, each CTA
// supplies its own 128 rows of A and half of the N rows of B from the same shared-memory offsets, and each CTA's
// TMEM receives its 128 rows of D.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {       // every thread of every CTA of the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared-memory object of this CTA's layout) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_dst, uint32_t ncols) {   // same warp id in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA load into this CTA's shared memory whose completion bytes go to an mbarrier given by its shared::cluster
// address (the leader's barrier): the .cta_group::2 form.
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// A operand read from tensor memory ([M lanes] x [K/2 32-bit columns], two bf16 per column, the even-k element in the
// low half): the ".ts" form.
__device__ __forceinline__ void umma_bf16_ts_2sm(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_f8_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive (release, cluster scope) on an mbarrier of another CTA of the cluster, given its shared::cluster address
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {     // acquire at cluster scope
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!ok);
}
// arrives on the mbarrier at this offset in both CTAs of the pair once the 2-SM MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)0x3) : "memory");
}

// ---------------------------------------------------------------- small helpers
__device__ __forceinline__ uint32_t pack_bf16x2(float lo_elem, float hi_elem) {   // lo_elem at the lower address
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo_elem, float hi_elem) {    // lo_elem at the lower address
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
  return r;
}
__device__ __forceinline__ uint32_t pack_e5m2x4(float e0, float e1, float e2, float e3) {   // e0 at the lowest address
  uint16_t a, b;
  asm("cvt.rn.satfinite.e5m2x2.f32 %0, %1, %2;" : "=h"(a) : "f"(e1), "f"(e0));
  asm("cvt.rn.satfinite.e5m2x2.f32 %0, %1, %2;" : "=h"(b) : "f"(e3), "f"(e2));
  return (uint32_t)a | ((uint32_t)b << 16);
}
// Four e5m2 values from two packed fp16 pairs scaled by a power of two: e5m2 is the high byte of fp16, so scale in
// half2 (FMA pipe), round by adding half an e5m2 ulp to each half (ties away from zero; sign-magnitude, so plain
// integer add) and gather the high bytes with one PRMT - no conversion-unit instructions.
__device__ __forceinline__ uint32_t e5m2x4_from_f16x2(uint32_t w0, uint32_t w1, uint32_t scale_f16x2) {
  uint32_t r;
  asm("{\n\t.reg .b32 a, b;\n\t"
      "mul.f16x2 a, %1, %3;\n\tmul.f16x2 b, %2, %3;\n\t"
      "add.u32 a, a, 0x00800080;\n\tadd.u32 b, b, 0x00800080;\n\t"
      "prmt.b32 %0, a, b, 0x7531;\n\t}"
      : "=r"(r) : "r"(w0), "r"(w1), "r"(scale_f16x2));
  return r;
}
constexpr uint32_t F16X2_2P6 = 0x54005400u;    // 64.0 in both halves   (2^F8_P)
constexpr uint32_t F16X2_2M8 = 0x1C001C00u;    // 1/256 in both halves  (2^-F8_Q)
// two packed 16-bit floats -> fp32 (F16: IEEE half, else bf16)
template <bool F16>
__device__ __forceinline__ void unpack2(uint32_t w, float& e0, float& e1) {
  if (F16) {
    asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(e0), "=f"(e1) : "r"(w));
  } else {
    e0 = __uint_as_float(w << 16); e1 = __uint_as_float(w & 0xFFFF0000u);
  }
}
template <bool F16>
__device__ __forceinline__ uint32_t pack2(float lo_elem, float hi_elem) {
  return F16 ? pack_f16x2(lo_elem, hi_elem) : pack_bf16x2(lo_elem, hi_elem);
}
// Byte offset of (row, 16-byte chunk) inside a 128B-swizzled tile whose base is 1024-byte aligned.
__device__ __forceinline__ uint32_t sw128_offset(int row, int chunk) {
  return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4));
}

}}  // namespace cwg::sm100
