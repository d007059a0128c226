// sm100_ptx.cuh -- thin inline-PTX wrappers for the Blackwell (sm_100a) primitives kernel 2 uses:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / fences), clusters; plus the 1-D bulk
// stores kernel 1 writes its C = 3072 rows with.
// Nothing here is generic: shapes and operand forms are exactly the ones k2_sim.cu issues.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#ifndef MV_WATCHDOG
#define MV_WATCHDOG 1  // bounded mbarrier spins: a protocol bug traps instead of hanging the GPU
#endif

namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#if MV_WATCHDOG
  for (uint32_t spin = 0; !mbar_try_wait(bar, parity); ++spin) {
    if (spin > (1u << 26)) {  // seconds; a healthy wait is microseconds
      printf("mvmatch: mbarrier watchdog: block %d thread %d bar 0x%x parity %u\n", (int)blockIdx.x,
             (int)threadIdx.x, bar, parity);
      __trap();
    }
  }
#else
  while (!mbar_try_wait(bar, parity)) {
  }
#endif
}

// ---- TMA --------------------------------------------------------------------------------
// 1-D bulk copy global -> shared (contiguous bytes, 16-byte aligned on both sides, size a multiple of 16), completion on `bar`
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"((uint64_t)src), "r"(bytes), "r"(bar)
               : "memory");
}
// the same with an L2 eviction priority (the fixed policy encodings that createpolicy.fractional.L2::evict_* produces at fraction 1.0)
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull;
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void bulk_load_1d_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
               "l"((uint64_t)src), "r"(bytes), "r"(bar), "l"(policy)
               : "memory");
}
// 1-D bulk copy shared -> global (16-byte aligned on both sides, size a multiple of 16), tracked in the issuing thread's
// bulk groups: that thread commits them and does every wait on them.  Shared memory written through the generic proxy
// needs fence_proxy_async_smem() by its writers (and a barrier to the issuer) before the copy may read it.
__device__ __forceinline__ void bulk_store_1d(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"((uint64_t)dst), "r"(src), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// every committed group has read its shared-memory source: the source may be rewritten
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// every committed group is complete, writes included
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tmap) : "memory");
}
// 2-D tile load global -> shared, completion on `bar` (this CTA)
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"((uint64_t)tmap), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// same, delivered to the same shared offset (and the same barrier offset) of every CTA in `mask`
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, "
      "%5}], [%2], %3;" ::"r"(dst),
      "l"((uint64_t)tmap), "r"(bar), "h"(mask), "r"(c0), "r"(c1)
      : "memory");
}

// ---- clusters ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- tcgen05 ----------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// whole warp; writes the TMEM base address to *dst_smem
__device__ __forceinline__ void tmem_alloc_512(uint32_t dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(dst_smem) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(taddr) : "memory");
}

// K-major operand tile in shared memory written by TMA with CU_TENSOR_MAP_SWIZZLE_128B: rows are 128 B,
// eight rows form one 1024-B swizzle atom (stride byte offset), tile base 1024-B aligned.
//   bits [0,14)  start address >> 4        bits [32,46) stride byte offset >> 4 (1024 -> 64)
//   bits [16,30) leading byte offset (unused for swizzled K-major)      bits [46,48) version = 1 (sm_100)
//   bits [61,64) layout type, 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  const uint32_t lo = (smem_addr & 0x3ffffu) >> 4;
  const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
  return ((uint64_t)hi << 32) | lo;
}

// instruction descriptor: D fp32, A/B K-major, M x N tile.  fmt: 0 = fp16, 1 = bf16 (both kind::f16), 2 = tf32 (kind::tf32)
__host__ __device__ constexpr uint32_t umma_idesc(int fmt, int M, int N) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

template <bool TF32>
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  if (TF32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

// One k-block in a single asm block: four MMAs that walk the 128-byte swizzle row in 32-byte steps (descriptor
// start address + 2 per step), then the commit that releases the shared-memory slot.  Keeping this in one
// block stops the compiler from re-deriving uniform registers (ELECT / R2UR / PLOP3 chains) around every
// instruction -- the issuing thread's own instruction latency was the kernel's bound before (profiles/).
template <bool TF32>
__device__ __forceinline__ void umma_kblock(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate_first, uint32_t empty_bar) {
  if (TF32) {
    asm volatile(
        "{\n\t.reg .pred p, pt;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 6;\n\tadd.u64 db, %2, 6;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p, pt;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 6;\n\tadd.u64 db, %2, 6;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, pt;\n\t"
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar)
        : "memory");
  }
}
// same with the commit multicast to every CTA of `mask`
template <bool TF32>
__device__ __forceinline__ void umma_kblock_mc(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate_first, uint32_t empty_bar, uint16_t mask) {
  if (TF32) {
    asm volatile(
        "{\n\t.reg .pred p, pt;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 6;\n\tadd.u64 db, %2, 6;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar), "h"(mask)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p, pt;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 6;\n\tadd.u64 db, %2, 6;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, pt;\n\t"
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar), "h"(mask)
        : "memory");
  }
}

// ---- CTA pair (cta_group::2): two SMs of a cluster work on one 256-row MMA tile ------------------------
// address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// arrive on a barrier that may live in another CTA of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// one warp of EACH CTA of the pair executes these
__device__ __forceinline__ void tmem_alloc_512_pair(uint32_t dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(dst_smem) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(taddr) : "memory");
}
// tile load into THIS CTA's shared memory, completion signalled on a barrier that may live in the peer CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* tmap, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"((uint64_t)tmap), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}
// one k-block of the 256 x 256 pair tile: 4 MMAs (A: 128 rows per CTA, B: 128 of the 256 columns per CTA), then the
// commit that frees the shared-memory slot in BOTH CTAs
template <bool TF32>
__device__ __forceinline__ void umma_kblock_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate_first, uint32_t empty_bar) {
  if (TF32) {
    asm volatile(
        "{\n\t.reg .pred p, pt;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 6;\n\tadd.u64 db, %2, 6;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], da, db, %3, pt;\n\t"
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar), "h"((uint16_t)3)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p, pt;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, pt;\n\t"
        "add.u64 da, %1, 6;\n\tadd.u64 db, %2, 6;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, pt;\n\t"
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar), "h"((uint16_t)3)
        : "memory");
  }
}

// Last k-block of an operand whose K extent is not a multiple of the 128-byte row: only `steps` (1..3) of the four
// MMAs carry data (the rest of the TMA box is zero fill), so only those are issued.  FORM: 0 = one CTA, 1 = commit
// multicast to `mask`, 2 = CTA pair.
template <bool TF32, int FORM>
__device__ __forceinline__ void umma_kblock_tail(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate_first, uint32_t empty_bar, uint16_t mask, uint32_t steps) {
#define MV_TAIL_BODY(GROUP, KIND, COMMIT)                                                                            \
  asm volatile(                                                                                                      \
      "{\n\t.reg .pred p, pt, q1, q2;\n\t.reg .b64 da, db;\n\t"                                                      \
      "setp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\tsetp.gt.u32 q1, %7, 1;\n\tsetp.gt.u32 q2, %7, 2;\n\t"          \
      "tcgen05.mma.cta_group::" GROUP ".kind::" KIND " [%0], %1, %2, %3, p;\n\t"                                      \
      "add.u64 da, %1, 2;\n\tadd.u64 db, %2, 2;\n\t"                                                                \
      "@q1 tcgen05.mma.cta_group::" GROUP ".kind::" KIND " [%0], da, db, %3, pt;\n\t"                                 \
      "add.u64 da, %1, 4;\n\tadd.u64 db, %2, 4;\n\t"                                                                \
      "@q2 tcgen05.mma.cta_group::" GROUP ".kind::" KIND " [%0], da, db, %3, pt;\n\t" COMMIT "\n\t}" ::"r"(d_tmem),   \
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "r"(empty_bar), "h"(mask), "r"(steps)               \
      : "memory")
#define MV_COMMIT_ONE "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];"
#define MV_COMMIT_MC "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;"
#define MV_COMMIT_PAIR "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;"
  if (FORM == 0) {
    if (TF32) MV_TAIL_BODY("1", "tf32", MV_COMMIT_ONE); else MV_TAIL_BODY("1", "f16", MV_COMMIT_ONE);
  } else if (FORM == 1) {
    if (TF32) MV_TAIL_BODY("1", "tf32", MV_COMMIT_MC); else MV_TAIL_BODY("1", "f16", MV_COMMIT_MC);
  } else {
    if (TF32) MV_TAIL_BODY("2", "tf32", MV_COMMIT_PAIR); else MV_TAIL_BODY("2", "f16", MV_COMMIT_PAIR);
  }
#undef MV_TAIL_BODY
#undef MV_COMMIT_ONE
#undef MV_COMMIT_MC
#undef MV_COMMIT_PAIR
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// arrive on `bar` (this CTA) once every tcgen05 op issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// same, arriving on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (row) t
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
      "tcgen05.wait::ld.sync.aligned;"  // same asm block: no consumer can be scheduled before the wait
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// warp-wide fp32 max in one instruction (CREDUX.MAX.F32 on sm_100a)
__device__ __forceinline__ float warp_max_f32(float v) {
  float m;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(v));
  return m;
}

__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// ---- flags in global memory between CTAs of one grid (stream-K hand-over) ----------------------
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// spin until *p != 0.  The writer is a CTA of the same persistent grid that raises the flag as its first piece of work.
__device__ __forceinline__ void flag_wait(const uint32_t* p) {
#if MV_WATCHDOG
  for (uint32_t spin = 0; ld_acquire_gpu(p) == 0u; ++spin) {
    if (spin > (1u << 24)) {  // seconds
      printf("mvmatch: stream-K flag watchdog: block %d thread %d\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
    __nanosleep(64);
  }
#else
  while (ld_acquire_gpu(p) == 0u) __nanosleep(64);
#endif
}

}  // namespace sm100
