// Thin inline-PTX wrappers for the sm_100a features the Gram kernel uses: mbarrier, TMA tensor loads,
// tcgen05 (TMEM allocation, MMA issue, commit, TMEM loads).  No library dependency.
#pragma once
#include <cstdint>
#include <cstdio>

namespace tbptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
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
// Bounded wait: a protocol bug traps (the launch reports an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) {  // several seconds at any SM clock
      printf("tblup_b200: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}

// ---- TMA ------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tensormap(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tiled load: c0 = innermost (contiguous) coordinate, c1 = row coordinate.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// 2-D tiled store from shared memory (same box and swizzle as the tensor map's loads); rows outside the tensor are
// clipped.  Completion is tracked per thread with bulk groups.
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// every store committed by this thread has finished READING its shared-memory source (the buffer may be rewritten)
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// every store committed by this thread is complete
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Same, delivered to the same shared-memory offset (and signalled on the same mbarrier offset) of every CTA of the
// cluster whose bit is set in cta_mask.
__device__ __forceinline__ void tma_load_2d_multicast(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1,
                                                      uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5}], [%2], %3;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "h"(cta_mask), "r"(c0), "r"(c1)
      : "memory");
}

// ---- clusters -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}

// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t cta_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
  return r;
}
// arrive on an mbarrier that may live in another CTA of the cluster (address from mapa_u32)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// CTA-pair TMA load: the data lands in THIS CTA's shared memory, the transaction bytes are counted on the mbarrier at
// `bar_cluster_addr` (the pair leader's ring barrier, which the one MMA-issuing thread of the pair waits on)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}

// ---- tcgen05 --------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Whole-warp calls (.sync.aligned).  The allocated base address is written to *smem_slot.
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(kCols) : "memory");
}
// CTA-pair variants: one warp of EACH CTA of the pair executes them; both CTAs receive the same column address
template <int kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(kCols) : "memory");
}

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle, rows of 128 bytes packed densely:
// 8-row groups are 1024 bytes apart (SBO), LBO is unused for swizzled K-major layouts (set to 1),
// descriptor version 1 (Blackwell), layout type 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// Instruction descriptor for kind::i8: s8 x s8 -> s32, both operands K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_s8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread.
__device__ __forceinline__ void umma_s8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::mxf4 (E2M1 operands, UE8M0 block scales, K = 64 per instruction)
__host__ __device__ constexpr uint32_t umma_idesc_mxf4(int m, int n) {
  // block-scaled descriptor: a/b format E2M1 (1), scale format UE8M0 (bit 23), K = 64 (bit 31 = 0), K-major operands
  return (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (1u << 23) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void umma_mxf4(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate, uint32_t tmem_sfa, uint32_t tmem_sfb) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%6], p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(tmem_sfa), "r"(tmem_sfb)
      : "memory");
}
// 32 lanes x 32 columns of one 32-bit value (whole warp; lane i writes TMEM lane base + i)
__device__ __forceinline__ void tmem_fill_32x32(uint32_t taddr, uint32_t v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
      ::"r"(taddr), "r"(v)
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// CTA-pair MMAs (cta_group::2): issued by ONE thread of the pair's leader CTA; M = 256 = 128 rows from each CTA's A tile,
// each CTA's shared memory holds N / 2 rows of B (the pair's tensor cores exchange them), each CTA's TMEM receives its
// own 128 x N accumulator.  Half the shared-memory fill and operand reads per MMA of the single-CTA form.
__device__ __forceinline__ void umma_s8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_mxf4_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate, uint32_t tmem_sfa, uint32_t tmem_sfb) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%6], p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(tmem_sfa), "r"(tmem_sfb)
      : "memory");
}
// completion of the pair's MMAs, signalled on the mbarrier at this offset in the CTAs named by cta_mask
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}

// Arrive on an mbarrier once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// Same arrival on the mbarrier at this offset in every CTA of the cluster named by cta_mask (a stage that the CTAs of a
// cluster fill for each other by TMA multicast is free only when all of them have consumed it).
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives row (lane base + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
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
// 32 lanes x 16 consecutive 32-bit columns (half the registers of the x32 form)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// 16 lanes x 32 consecutive 32-bit columns in the MMA-accumulator register layout (shape .16x256b, 4 repeats):
// lane l = 4 r + p holds, for column group j = 0..3, v[4 j + {0,1}] = row r, columns 8 j + 2 p + {0,1} and
// v[4 j + {2,3}] = row r + 8, same columns -- four lanes own 32 contiguous bytes of a row, so an 8-byte store per
// lane writes whole sectors without a trip through shared memory.
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- coalescing epilogue stores ----------------------------------------------------------------
// After tcgen05.ld.32x32b a thread holds consecutive columns of ONE row, so a direct 16-byte store per thread writes
// 32 rows x 16 B per instruction (half sectors, the slowest pattern the L2 accepts).  These helpers bounce a
// 32-row x 16-word block through a 2 KiB per-warp staging buffer so that each store instruction writes 8 rows x 64
// contiguous bytes (whole sectors).  Granule (16 B) g of row t sits at position g ^ ((t >> 1) & 3): both the
// row-wise write and the transposed read are bank-conflict free.  Callers __syncwarp() between write and read and
// before reusing the buffer.
// (explicit ld/st.shared on a 32-bit shared address: through a generic pointer the compiler emits generic LD/ST)
__device__ __forceinline__ void stage_write16(uint32_t stg_addr, int lane, const uint32_t* v) {
  const uint32_t base = stg_addr + lane * 64;
  const int f = (lane >> 1) & 3;
#pragma unroll
  for (int g = 0; g < 4; ++g)
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + ((g ^ f) << 4)), "r"(v[4 * g]),
                 "r"(v[4 * g + 1]), "r"(v[4 * g + 2]), "r"(v[4 * g + 3])
                 : "memory");
}
// iteration it (0..3): lane reads granule (lane & 3) of row 8 it + (lane >> 2)
__device__ __forceinline__ uint4 stage_read16(uint32_t stg_addr, int lane, int it) {
  const int r = 8 * it + (lane >> 2), g = lane & 3;
  uint4 u;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
               : "r"(stg_addr + ((r * 4 + (g ^ ((r >> 1) & 3))) << 4))
               : "memory");
  return u;
}

}  // namespace tbptx
