// PTX wrappers of the 5th-generation tensor-core kernels: mbarriers, tensor memory (TMEM), tcgen05.mma and its
// descriptors, bulk / TMA copies and the cluster helpers of the CTA-pair schedule.  Every tcgen05 kernel
// (b2n_mlp256.cu: 256-wide decoder; b2n_wgrad256.cu: its weight gradients and those of the fused 128-wide MLPs;
// b2n_mlp64tc.cu / b2n_mlp64.cu: Instant decoder forward and backward weight gradients) issues these instructions
// through this header only, so each one can be checked against the PTX ISA here.
// Suffix 2 = the cta_group::2 form: one instruction spans the two CTAs of an SM pair.
#pragma once
#include <cstdint>
#include "b2n_common.cuh"

namespace b2n {
namespace tc {

__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// byte offset of 16-byte chunk c (0..7) of row r inside a swizzled block of 128-byte rows
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

// ---------------------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// makes the initialised barriers visible to the async proxy and to the other CTA of a cluster
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Remote arrive with the default (.release.cta) semantics, as CUTLASS's ClusterBarrier::arrive(cta_id) does.  What crosses
// the CTA boundary here is shared memory only (the peer's activation tile, read by the leader's tensor core), which no
// cache sits in front of; the explicit `.release.cluster` form compiles to MEMBAR.ALL.GPU and the matching
// `try_wait.acquire.cluster` to CCTL.IVALL (an L1 flush) per wait -- together ~2000 cycles per tile and step (B2N_TRACE).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread for a while; a poller that serves several barriers must not)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded waits: a stalled pipeline raises the error flag instead of hanging the GPU.  The budget of 2^24 tries only
// runs out on a protocol bug; it never bounds a healthy wait.
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, int* err) {
#pragma unroll 1
  for (uint32_t it = 0; it < (1u << 24); ++it)
    if (mbar_try(bar, parity)) return true;
  atomicCAS(err, 0, 7);
  return false;
}
// Form for kernels whose warp roles wait on each other: a time-out raises the CTA's abort flag and stores `code`, and
// every other wait polls that flag (every 1024 tries) so that all roles drain.  false = aborted (this wait timed out or
// another role raised the flag).
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, volatile int* abort_flag, int* err, int code) {
#pragma unroll 1
  for (uint32_t it = 0; it < (1u << 24); ++it) {
    if (mbar_try(bar, parity)) return true;
    if ((it & 1023) == 1023 && *abort_flag) return false;
  }
  *abort_flag = 1;
  atomicCAS(err, 0, code);
  return false;
}

// ---------------------------------------------------------------------------------------- tensor memory
// One warp allocates `cols` columns, writes their base address to shared memory at `slot` and relinquishes the CTA's
// permit to allocate again (every kernel allocates once).
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(cols));
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t tmem, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(cols));
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------- tcgen05 fences, MMA, commit
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the tensor core / TMA (async proxy)
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// D (TMEM) = A B (+ D when acc != 0), kind::f16: fp16 / bf16 operands, fp32 accumulator
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
// CTA pair: M = 256 (128 rows per CTA); each CTA supplies half of B
__device__ __forceinline__ void tc_mma2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
// arrives on `bar` once all prior MMAs of this thread are complete
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrives on the barrier at the same shared-memory offset in BOTH CTAs of the pair once all prior MMAs are complete
__device__ __forceinline__ void tc_commit2(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// ---------------------------------------------------------------------------------------- descriptors
// K-major SWIZZLE_128B shared-memory matrix descriptor: rows of 128 B, 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// MN-major SWIZZLE_128B operand (the contraction index is the ROW of the tile: [rows = K][64 columns = M or N], 128-byte
// rows): 64-column blocks `blk` bytes apart, 8-row groups 1024 B apart; a K step of 16 rows advances the address by 2048 B
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr, uint32_t blk) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((blk >> 4) & 0x3FFF) << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
enum class Fmt { F16, BF16 };   // operand format of kind::f16 (A and B alike)
enum class Major { K, MN };      // operand layout (A and B alike): umma_desc / umma_desc_mn
// kind::f16 instruction descriptor: D = fp32 (bits 4-5), A / B format (7-9 / 10-12), A / B MN-major (15 / 16),
// N >> 3 (17-22), M >> 4 (24-28); M = 256 for a CTA pair
__device__ __forceinline__ uint32_t umma_idesc(Fmt fmt, Major major, int n, int m) {
  const uint32_t ab = fmt == Fmt::BF16 ? (1u << 7) | (1u << 10) : 0u;
  const uint32_t mn = major == Major::MN ? (1u << 15) | (1u << 16) : 0u;
  return (1u << 4) | ab | mn | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---------------------------------------------------------------------------------------- bulk and TMA copies
// 1-D bulk copy global -> shared; the bytes are credited to `bar` (complete_tx)
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* tmap, int c0, int c1, int c2, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
// TMA tile load issued by either CTA of a pair; the transaction bytes are credited to `mbar_cluster`, which may live in
// the other CTA (the leader's "weights landed" barrier)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* tmap, int x, int y, uint32_t mbar_cluster) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(tmap), "r"(x), "r"(y), "r"(mbar_cluster) : "memory");
}
// TMA tensor store smem -> global at coordinates (c0, c1, c2), completed through the bulk group
__device__ __forceinline__ void tma_store_3d(const void* tmap, uint32_t smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(tmap), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the stores issued so far have READ their shared-memory source (it may be overwritten)
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// the stores issued so far are complete
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------------------------------- clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_idx() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_count() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
// shared::cluster address of `saddr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// one lane of a converged warp (warp-uniform control flow keeps descriptors in uniform registers)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

}  // namespace tc
}  // namespace b2n
