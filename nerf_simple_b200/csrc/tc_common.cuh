// Blackwell (sm_100a) primitives used by the fused MLP kernels: mbarrier, bulk-copy TMA,
// tcgen05 MMA / TMEM, UMMA shared-memory and instruction descriptors.  Inline PTX only.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace nb200 {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Bounded wait: a pipeline bug must fail loudly (trap -> launch error), never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = global_timer_ns();
  uint32_t it = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++it & 0xFFFu) == 0u && global_timer_ns() - t0 > 4000000000ull) {
      printf("nb200: mbarrier wait timed out (block %d thread %d tag %d parity %u)\n", blockIdx.x,
             threadIdx.x, tag, parity);
      __trap();
    }
  }
}

// ------------------------------------------------------------------------- TMA bulk copy
// Contiguous global -> shared copy through the TMA engine (SASS UBLKCP); completion is
// signalled as transaction bytes on `bar`.
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
      "l"(src_gmem), "r"(bytes), "r"(bar)
      : "memory");
}

// 2-D tiled TMA load issued by either CTA of a pair; the transaction bytes are signalled on `bar`,
// which may live in the PEER CTA (.cta_group::2) -- the leader's weight barrier counts both halves
// of a slab without a forwarding hop.  `bar` is a shared::cluster address (mapa).
__device__ __forceinline__ void tma_tensor2d_g2s_2cta(uint32_t dst_smem, const void* tmap, int32_t c0, int32_t c1,
                                                      uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst_smem),
      "l"(tmap), "r"(c0), "r"(c1), "r"(bar_cluster)
      : "memory");
}

// Contiguous shared -> global copy through the TMA engine (bulk async-group completion).
__device__ __forceinline__ void tma_bulk_s2g(void* dst_gmem, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(src_smem), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// all bulk stores of this thread have finished READING shared memory (the source may be reused)
__device__ __forceinline__ void tma_bulk_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// L2 cache policy for streamed-out tiles: first to go.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_bulk_s2g_hint(void* dst_gmem, uint32_t src_smem, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst_gmem), "r"(src_smem),
               "r"(bytes), "l"(policy)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

// ----------------------------------------------------------------------------- fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ------------------------------------------------------------------------------- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives row (lane base + i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor, 128-byte swizzle (layout type 2), descriptor version 1.
//   K-major operand  : rows (M or N index) are 128 B apart, 8-row groups SBO = 1024 B apart;
//                      LBO is unused for swizzled K-major (canonical value 1).
//   MN-major operand : 64 contiguous MN elements per 128 B row, rows = K index; 8-row (K) groups
//                      SBO apart; consecutive 64-element MN chunks LBO apart.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // version = 1 (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                       // D format  = F32
         | (1u << 7)                     // A format  = BF16
         | (1u << 10)                    // B format  = BF16
         | ((uint32_t)a_mn_major << 15)  // A major   (0 = K)
         | ((uint32_t)b_mn_major << 16)  // B major   (0 = K)
         | ((uint32_t)(N >> 3) << 17)    // N >> 3
         | ((uint32_t)(M >> 4) << 24);   // M >> 4
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread for the whole CTA.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on `bar` when every tcgen05.mma issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}

// ------------------------------------------------------------- 2-CTA (cta_group::2) variants
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t num_clusters_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (.release at CTA scope), the form CUTLASS uses for cross-CTA pipeline arrives:
  // a cluster-scope release costs a full membar per arrive and sits on the MMA hand-off path
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t dst_smem, uint32_t ncols) {  // one warp in EACH CTA
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// M = 256 across the CTA pair: each CTA supplies its 128 rows of A and half of the N rows of B at
// the SAME shared-memory offsets; issued by one thread of the leader CTA only.
__device__ __forceinline__ void umma_bf16_2cta(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on the barrier at this offset in BOTH CTAs once all prior MMAs of this thread retired.
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}
// fp32 pair -> packed bf16x2 (lo in bits 0..15), optionally fused with ReLU (one F2FP instruction)
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// ReLU bit masks.  flags: 0xFFFF in each half of the result whose bf16 value is > 0 (one HSET2).
__device__ __forceinline__ uint32_t pos_flags_bf16x2(uint32_t w) {
  const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(&w);
  return __hgt2_mask(v, __float2bfloat162_rn(0.f));
}
// pack: pair k (0..7) of a 16-column step contributes bit k (even column) and bit 24+k (odd column) to `acc`;
// fold_mask16 brings the odd-column flags down to bits 8..15.
__device__ __forceinline__ void add_pair_flags(uint32_t& acc, uint32_t w, int k) {
  acc |= pos_flags_bf16x2(w) & ((1u << k) | (1u << (24 + k)));
}
__device__ __forceinline__ uint32_t fold_mask16(uint32_t acc) { return (acc & 0xFFu) | (acc >> 16); }
// unpack: 16-bit field -> 0xFFFF / 0x0000 per half for pair k (shift the two flags to the byte MSBs, PRMT replicates them)
__device__ __forceinline__ uint32_t pair_mask_word(uint32_t field16, int k) {
  uint32_t r;
  asm("prmt.b32 %0, %1, 0, 0x9988;" : "=r"(r) : "r"(field16 << (7 - k)));
  return r;
}

// One lane of a fully converged warp (the MMA warp runs its loops warp-uniformly so that the
// descriptors live in uniform registers; only the tcgen05 instructions are elected).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xFFFFFFFF;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// packed fp32x2 add (Blackwell FADD2): two accumulator columns + two biases per instruction
__device__ __forceinline__ void add_f32x2(float& a0, float& a1, float b0, float b1) {
  uint64_t a, b;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a) : "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(a));
}

// -------------------------------------------------------------------------- small helpers
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// LDS.128 of four floats; at a warp-uniform address it is one broadcast (staged biases, head weights)
__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
// byte offset of 16-byte chunk j (0..7) of row r inside a [rows x 128 B] SWIZZLE_128B image
__host__ __device__ __forceinline__ uint32_t sw128_off(uint32_t r, uint32_t j) {
  return r * 128u + ((j ^ (r & 7u)) << 4);
}

}  // namespace tc
}  // namespace nb200
