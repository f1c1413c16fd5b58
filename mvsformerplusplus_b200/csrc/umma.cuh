// tcgen05 (5th-gen tensor core) building blocks for sm_100a, hand-written PTX.
//   - shared-memory operand descriptors for the canonical K-major, no-swizzle ("interleaved") layout:
//       element (row m, k) of a tile lives at  base + (k/8)*LBO + (m/8)*SBO + (m%8)*16 + (k%8)*2   [fp16]
//     i.e. 8x8 "core matrices" of 128 contiguous bytes (conflict-free for the tensor core's reads);
//   - tcgen05.mma.cta_group::1.kind::f16 (fp16 x fp16 -> fp32 accumulators in TMEM), issued by one thread;
//   - tcgen05.commit -> mbarrier, bounded mbarrier waits (trap instead of hanging the GPU);
//   - bulk copies and TMA tensor-box loads into shared memory that complete on an mbarrier (expect_tx / complete_tx);
//   - TMEM alloc/dealloc and tcgen05.ld (32 lanes x 32 bit, one accumulator row per thread).
// Field layouts follow the PTX ISA / CUTLASS cute/arch/mma_sm100_desc.hpp (SmemDescriptor, InstrDescriptor).
#pragma once
#ifndef MVSF_MBAR_SPIN_LOG2
#define MVSF_MBAR_SPIN_LOG2 26   // bounded mbarrier waits: ~1.5 s of polling before the trap
#endif
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace mvsf {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy shared-memory writes (st.shared / cp.async) -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

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
// non-blocking probe.  An mbarrier query has a latency of 120-260 clk even when the phase completed long ago
// (tools/mbar_microbench.cu): issue the probe EARLY, do independent work, look at the answer later.
__device__ __forceinline__ uint32_t mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// bounded wait: a mis-programmed pipeline traps (sticky CUDA error) instead of hanging the device
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t it = 0; it < (1u << MVSF_MBAR_SPIN_LOG2); ++it)
    if (mbar_try_wait(bar, parity)) return;
#ifdef MVSF_DEBUG_WAIT
  printf("mbarrier wait stuck: block (%d,%d) thread %d bar %x parity %u\n", blockIdx.x, blockIdx.y, threadIdx.x, bar, parity);
  return;   // debug build: carry on (wrong results) so that the printf buffer is flushed at kernel end
#endif
  __trap();
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
// arrive and announce `bytes` of async-proxy writes that have to land before the phase completes
__device__ __forceinline__ void expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// contiguous global -> shared bulk copy (cp.async.bulk); completes `bytes` of the transaction count of `bar`
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// TMA load of one 5-D box at coordinates (c0 .. c4) of `map` (a __grid_constant__ kernel parameter); coordinates outside
// the tensor are filled with zeros
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
// host: the driver's cuTensorMapEncodeTiled (api.cu), nullptr when the driver does not provide it
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn();
// named barrier among a subset of the CTA's warps (id 1..15; id 0 is __syncthreads)
// compile-time id: a run-time id makes ptxas reserve all 16 hardware barriers (and profilers that patch the kernel then
// cannot launch it)
template <int ID>
__device__ __forceinline__ void named_bar_sync_c(int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"n"(ID), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);              // start address            bits [0,14)
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;    // leading byte offset       bits [16,30)  (between the 2 k-chunks)
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;    // stride byte offset        bits [32,46)  (between 8-row groups)
  d |= (uint64_t)1 << 46;                              // descriptor version 1 (Blackwell)
  return d;                                            // base_offset 0, lbo_mode 0, layout_type 0 = SWIZZLE_NONE
}
// kind::f16 instruction descriptor: fp16 A/B (format 0), fp32 accumulate (c_format 1), both K-major, dense
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Converged-warp issue: every lane of a fully converged warp executes this; one elected lane issues the MMA.  Keeps the
// issuing code warp-uniform (descriptors in uniform registers, no per-instruction divergence handling).
__device__ __forceinline__ void mma_f16_ss_elect(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar) : "memory");

}
// Lean issue path for a dedicated, converged MMA warp: the issuing warp is the critical resource of the small-N kernels
// (a tcgen05.mma costs ~50 clk stand-alone, more when its ~20 set-up instructions compete for issue slots).  Descriptors
// are handled as {low word = start address | k-chunk stride, high word = 8-row-group stride | version}: moving a
// descriptor is one 32-bit add on the low word.  `el` (from elect_one()) is non-zero on exactly one lane.
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr >> 4) & 0x3fffu) | ((lbo_bytes >> 4) << 16); }
__host__ __device__ constexpr uint32_t desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3fffu) | (1u << 14); }
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t e;
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(e));
  return e;
}
__device__ __forceinline__ void mma_f16_ss_lh(uint32_t el, uint32_t tmem_d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 q, %0, 0;\n\tsetp.ne.b32 p, %7, 0;\n\t"
      "mov.b64 da, {%2, %3};\n\tmov.b64 db, {%4, %5};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%1], da, db, %6, p;\n\t}"
      ::"r"(el), "r"(tmem_d), "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void commit_el(uint32_t el, uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %0, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%1];\n\t}" ::"r"(el), "r"(bar) : "memory");

}
// one lane polls, the warp reconverges (32 polling lanes steal issue slots and shared-memory bandwidth)
__device__ __forceinline__ void mbar_wait_warp(uint32_t bar, uint32_t parity) {
  if ((threadIdx.x & 31) == 0) mbar_wait(bar, parity);
  __syncwarp();
}
// A operand from tensor memory (128 lanes = rows, K = 16 fp16 packed two per 32-bit column: 8 columns), B from shared memory
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (count 1) on the mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");

}
// one full warp; writes the TMEM base address (lane 0, column c) to *dst_smem
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 16 consecutive fp32 columns of this thread's TMEM lane (lane = 32*(warp%4) + laneid)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld1_nowait(uint32_t taddr, uint32_t& r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
// 32 consecutive fp32 columns, no wait (issue several, then tmem_ld_wait() once)
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
// 16 consecutive 32-bit columns of this thread's TMEM lane <- registers
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void cp_async16_zfill(uint32_t smem_addr, const void* gptr, bool valid) {
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr), "l"(gptr), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// bytes of one K-block tile (64 fp16 = 8 chunks of 16 B per row) of `rows` rows in the padded canonical layout
__host__ __device__ constexpr uint32_t tile_lbo(int rows) { return (uint32_t)(rows / 8) * 128u + 16u; }  // +16: bank-conflict-free fills
__host__ __device__ constexpr uint32_t tile_bytes(int rows) { return 8u * tile_lbo(rows); }
// cooperative fill of one tile from a row-major fp16 matrix: g points at (row 0, k 0) of the tile, ld in elements
template <int NTHREADS>
__device__ __forceinline__ void fill_tile(uint32_t tile_smem, const __half* g, size_t ld, int rows, int valid_rows, int tid) {
  const uint32_t lbo = tile_lbo(rows);
  for (int idx = tid; idx < rows * 8; idx += NTHREADS) {
    int r = idx >> 3, c = idx & 7;
    bool ok = r < valid_rows;
    const __half* src = g + (size_t)(ok ? r : 0) * ld + c * 8;
    cp_async16_zfill(tile_smem + c * lbo + (r >> 3) * 128 + (r & 7) * 16, src, ok);
  }
}

}  // namespace umma
}  // namespace mvsf
