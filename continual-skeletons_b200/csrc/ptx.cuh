// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM).
// Encodings follow the PTX ISA 8.7 tcgen05 chapter; the bit layouts of the shared-memory matrix
// descriptor and the instruction descriptor are the ones documented for sm_100
// (start>>4 | LBO<<16 | SBO<<32 | version(1)<<46 | swizzle<<61 ; c_fmt<<4 | a_fmt<<7 | b_fmt<<10 |
//  N>>3<<17 | M>>4<<24).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cosk {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// make generic-proxy shared-memory writes visible to the async proxy (TMA / UMMA operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
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

// Bounded wait: a pipeline bug must end the kernel with a diagnostic, never hang the GPU.
// Returns false on timeout (about 2 s of SM clock) after recording `code` in *dbg (first wins).
constexpr long long kWaitLimitCycles = 4000000000LL;
__device__ __forceinline__ bool mbar_wait(uint64_t *bar, uint32_t parity, unsigned int *dbg, unsigned int code) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  unsigned int spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xff) == 0) {
      if (dbg != nullptr && *(volatile unsigned int *)dbg != 0) return false;  // someone else already failed
      if (clock64() - t0 > kWaitLimitCycles) {
        if (dbg != nullptr) atomicCAS(dbg, 0u, code);
        return false;
      }
    }
  }
  return true;
}

// ---- TMA ------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap *m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tile load global -> shared, completion counted in bytes on `bar`.  c0 = innermost coordinate.
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap *m, uint64_t *bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(uint32_t smem_dst, const CUtensorMap *m, uint64_t *bar, int c0, int c1,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

// ---- tcgen05 / TMEM -------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major operand tile in shared memory, 128-byte rows (64 bf16 of K), SWIZZLE_128B, rows grouped
// by 8 (1024 B per group).  `saddr` = shared address of the tile start (1024-byte aligned) plus the
// K offset inside the swizzle atom (32 B per UMMA_K = 16 bf16).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;            // leading byte offset: unused for swizzled K-major, canonical 1
  d |= (uint64_t)(1024u >> 4) << 32; // stride byte offset: next 8-row group
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;            // SWIZZLE_128B
  return d;
}
// The same descriptor split into its constant high word and the low word that carries the address, so
// that the single MMA-issuing thread spends one add per operand and K-step instead of rebuilding 64 bits.
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO | version | SWIZZLE_128B
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }

// kind::f16 instruction descriptor: bf16 x bf16 -> fp32, both operands K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same, operands given as descriptor low words (high word = kDescHiSw128)
__device__ __forceinline__ void umma_bf16_lo(uint32_t tmem_d, uint32_t lo_a, uint32_t lo_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "r"(lo_a), "r"(lo_b), "r"(idesc), "r"(accumulate), "r"(kDescHiSw128)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair_lo(uint32_t tmem_d, uint32_t lo_a, uint32_t lo_b, uint32_t idesc, uint32_t accumulate);

// mbarrier arrives once every previously issued tcgen05.mma of this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t).
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
// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM: thread t of the warp writes 16 consecutive 32-bit columns of lane (base_lane + t).  Used to stage
// an A operand in TMEM: a K-major bf16 row of the operand occupies its lane, two K elements per column (even k low).
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]^T : the A operand (128 rows = 128 lanes, K-major, 8 columns per K-step of 16 bf16) is
// read from tensor memory at `tmem_a`; B as a shared-memory descriptor low word (high word = kDescHiSw128).
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t lo_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "r"(tmem_a), "r"(lo_b), "r"(idesc), "r"(accumulate), "r"(kDescHiSw128)
      : "memory");
}

// ---- clusters / CTA pairs (cta_group::2) -----------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA tile load issued by either CTA of a pair; the completion bytes are counted on an mbarrier that
// may live in the peer CTA (`bar_cluster_addr` is a shared::cluster address).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const CUtensorMap *m, uint32_t bar_cluster_addr, int c0,
                                                 int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_hint(uint32_t smem_dst, const CUtensorMap *m, uint32_t bar_cluster_addr, int c0,
                                                      int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t *smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 per CTA] * B[N rows: N/2 per CTA]^T ; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair_lo(uint32_t tmem_d, uint32_t lo_a, uint32_t lo_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "r"(lo_a), "r"(lo_b), "r"(idesc), "r"(accumulate), "r"(kDescHiSw128)
      : "memory");
}
// arrive on the mbarrier at this shared-memory offset in every CTA of `cta_mask` once all prior MMAs completed
__device__ __forceinline__ void umma_commit_pair(uint64_t *bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}

// 128-bit global accesses for the epilogue
__device__ __forceinline__ uint4 ldg_v4(const void *p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_v4(void *p, const uint4 &v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

}  // namespace ptx
}  // namespace cosk
