// What the tcgen05 GEMM kernels (joint, dh, dW, linear) share around their own barrier structs and schedules.
#pragma once
#include "common.cuh"

namespace rb {

constexpr int kSmemAlign = 1024;   // 128-byte-swizzled tiles need 1024-byte alignment; launchers add this to a layout

struct AlignedSmem {
  uint32_t addr;   // shared::cta address
  uint8_t* ptr;    // generic pointer to the same byte
};
__device__ __forceinline__ AlignedSmem aligned_smem(uint8_t* smem_raw) {
  const uint32_t addr = (smem_u32(smem_raw) + (kSmemAlign - 1)) & ~static_cast<uint32_t>(kSmemAlign - 1);
  return AlignedSmem{addr, smem_raw + (addr - smem_u32(smem_raw))};
}

// TMEM set-up, tmem_setup = tmem_alloc + tmem_publish: warp 1 allocates `ncols` columns (in both CTAs of the pair when
// kPair) into *slot; then the CTA and the pair synchronise, so the barrier inits done before, shared memory written in
// between and the allocation are visible everywhere before any (remote) arrive.  tmem_publish returns the TMEM base.
// (The joint kernel stages its length tables between the two: staged ahead of the allocation, two of its
// instantiations spill.)
template <bool kPair>
__device__ __forceinline__ void tmem_alloc(int warp, uint32_t* slot, uint32_t ncols) {
  if (warp == 1) {
    if (kPair)
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n\t"
                   "tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
    else
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n\t"
                   "tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
  }
}
template <bool kPair>
__device__ __forceinline__ uint32_t tmem_publish(uint32_t* slot) {
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();
  tc_fence_after();
  return *slot;
}
template <bool kPair>
__device__ __forceinline__ uint32_t tmem_setup(int warp, uint32_t* slot, uint32_t ncols) {
  tmem_alloc<kPair>(warp, slot, ncols);
  return tmem_publish<kPair>(slot);
}

// Mirror image: warp 1 frees the columns once every thread is done with TMEM and the peer CTA is done signalling this
// CTA's barriers and reading its shared memory.
template <bool kPair>
__device__ __forceinline__ void tmem_teardown(int warp, uint32_t base, uint32_t ncols) {
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    if (kPair) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
  }
}

// lane quarter `lane_grp` (the one warp w may access: w & 3), column `col`
__device__ __forceinline__ uint32_t tmem_lane_addr(uint32_t base, int lane_grp, uint32_t col) {
  return base + (static_cast<uint32_t>(lane_grp * 32) << 16) + col;
}

// The kBK / 16 MMAs D[tmem] (+)= A[smem] * B[smem] of one K chunk, issued by one thread; with kPair the leader CTA's
// thread issues M = 256 over both CTAs (each holds 128 rows of A and half of B).  `accumulate` applies to the first MMA
// (the others always accumulate).  Operand tiles:
//   K-major (rows = M or N, 64 16-bit elements of K per 128-byte row, 8-row 1024-byte swizzle atoms):
//     SBO = 1024 (next 8-row group), LBO unused (1).  Advance K by 16 elements = +32 bytes on the start address.
//   MN-major (rows = K, 64 16-bit elements of M/N per 128-byte row):
//     SBO = 1024 (next 8 K-rows), LBO = 8192 = byte stride between 64-element M/N blocks.
//     Advance K by 16 rows = +2048 bytes on the start address.
template <bool kPair, bool kAMn, bool kBMn>
__device__ __forceinline__ void mma_kchunk(uint32_t tmem_d, uint32_t a_addr, uint32_t b_addr, uint32_t idesc,
                                           bool accumulate) {
#pragma unroll
  for (int k = 0; k < kBK / 16; ++k) {
    const uint64_t ad = kAMn ? make_smem_desc(a_addr + k * 2048, 8192, 1024) : make_smem_desc(a_addr + k * 32, 16, 1024);
    const uint64_t bd = kBMn ? make_smem_desc(b_addr + k * 2048, 8192, 1024) : make_smem_desc(b_addr + k * 32, 16, 1024);
    const uint32_t acc = accumulate || k != 0;
    if (kPair)
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                   ::"r"(tmem_d), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
    else
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                   ::"r"(tmem_d), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
  }
}

// Stage barrier `bar` of a CTA pair: the leader's copy expects both CTAs' `bytes_total`, the peer arrives on it.
// Returns the leader's barrier, which both CTAs' TMA loads signal.
__device__ __forceinline__ uint32_t pair_stage_arrive(uint32_t bar, uint32_t rank, uint32_t bytes_total) {
  const uint32_t leader = mapa_shared(bar, 0);
  if (rank == 0) mbar_expect_tx(bar, bytes_total);
  else mbar_arrive_cluster(leader);
  return leader;
}

}  // namespace rb
