// Backward contraction #3:  dW = g^T . h  (K = lattice cells of the current ring chunk).
//
// Replaces the weight-gradient GEMM of joint_ln's autograd backward (rnnt/joint.py:39, SURVEY 8a-8).
// Both operands are read as MN-major views of the row-major rings written by the G-mode joint kernel:
//   A[m=v][k=c] = g_ring[c][v]      B[n=kh][k=c] = h_ring[c][kh]
// A CTA PAIR owns a 256(v) x 512(k_h) block of dW for one K split (tcgen05.mma.cta_group::2, M = 256: each CTA holds
// its 128 classes x 512 hidden units as two TMEM accumulators = all 512 columns, stages its own 128 classes of g^T and
// HALF of each activation box -> 48 instead of 80 bytes of L2 traffic per SM and clock) and adds it into the fp32 dW
// with vector reductions (red.global.add.v4.f32).  The CTAs of the first k_h block also produce db: while the MMAs
// run, their (otherwise idle) epilogue warps sum every A stage over its 64 cells.
#include <algorithm>

#include "kernels.h"
#include "tc_kernel.cuh"

namespace rb {
namespace {

constexpr int kStagesA = 4;
constexpr int kStagesB = 8;
constexpr int kBytesA = kBK * kTileM * 2;       // 16 KB: 64 cells x 128 v  (two 64x64 boxes; this CTA's classes)
constexpr int kBytesB = kBK * (kBN / 2) * 2;    // 16 KB: 64 cells x 128 kh (two 64x64 boxes; this CTA's half of N=256)
constexpr int kNumThreads = 192;
constexpr int kTmemCols = 512;

struct SmemLayout {
  static constexpr int b_ring = 0;
  static constexpr int a_ring = b_ring + kStagesB * kBytesB;
  static constexpr int bars = a_ring + kStagesA * kBytesA;
  static constexpr int db_red = bars + 256;                  // 128 threads x 8 fp32 partial column sums
  static constexpr int total = db_red + 128 * 8 * 4;
};
// b_full: the leader's copy collects both CTAs' boxes (one arrival per CTA).  a_full stays local (the db reducers of each
// CTA read their own A stage); the peer's MMA warp forwards "my A stage landed" to the leader's a_peer.
struct Bars {
  uint64_t b_full[kStagesB], b_empty[kStagesB], a_full[kStagesA], a_empty[kStagesA], tmem_full;
  uint64_t a_peer[kStagesA];   // leader only: the peer CTA's A stage has landed
  uint32_t tmem_slot;
};
static_assert(sizeof(Bars) <= SmemLayout::db_red - SmemLayout::bars, "barrier block overflows its region");

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kNumThreads, 1)
dw_gemm_kernel(const __grid_constant__ CUtensorMap tmGmn, const __grid_constant__ CUtensorMap tmHmn, DwArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const AlignedSmem smem = aligned_smem(smem_raw);
  const uint32_t b_ring = smem.addr + SmemLayout::b_ring;
  const uint32_t a_ring = smem.addr + SmemLayout::a_ring;
  Bars* bars = reinterpret_cast<Bars*>(smem.ptr + SmemLayout::bars);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int total_slots = __ldg(p.n_active);
  const int slot_end = min(total_slots, p.slot_begin + p.slot_cap);
  const int nkc = max(0, slot_end - p.slot_begin);   // K chunks of 64 cells = work-list slots (half-tiles) of this ring chunk

  const int nblk_total = (p.Hp + kBN - 1) / kBN;
  const int nht = (nblk_total + 1) / 2;
  const int nvt = p.Vp / (2 * kTileM);
  int bid = blockIdx.x >> 1;          // pair index
  const int vt = bid % nvt; bid /= nvt;
  const int ht = bid % nht; bid /= nht;
  const int ks = bid;
  const int nblk = min(2, nblk_total - ht * 2);
  const int k_begin = static_cast<int>(static_cast<long long>(nkc) * ks / p.ksplit);
  const int k_end = static_cast<int>(static_cast<long long>(nkc) * (ks + 1) / p.ksplit);
  if (k_begin >= k_end) return;   // uniform over the pair
  const bool do_db = (ht == 0) && p.db != nullptr;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmGmn);
    tma_prefetch_desc(&tmHmn);
    for (int s = 0; s < kStagesB; ++s) { mbar_init(smem_u32(&bars->b_full[s]), 2); mbar_init(smem_u32(&bars->b_empty[s]), 1); }
    for (int s = 0; s < kStagesA; ++s) {
      mbar_init(smem_u32(&bars->a_full[s]), 1);
      mbar_init(smem_u32(&bars->a_empty[s]), do_db ? 5 : 1);
      mbar_init(smem_u32(&bars->a_peer[s]), 1);
    }
    mbar_init(smem_u32(&bars->tmem_full), 1);
    mbar_fence_init();
  }
  const uint32_t tmem_base = tmem_setup<true>(warp, &bars->tmem_slot, kTmemCols);

  if (warp == 0) {
    if (lane == 0) {
      uint32_t ita = 0, itb = 0;
      for (int kc = k_begin; kc < k_end; ++kc, ++ita) {
        const uint32_t sa = ita % kStagesA, pha = (ita / kStagesA) & 1;
        const uint32_t a_full = smem_u32(&bars->a_full[sa]);
        mbar_wait(smem_u32(&bars->a_empty[sa]), pha ^ 1);
        mbar_expect_tx(a_full, kBytesA);
#pragma unroll
        for (int j = 0; j < 2; ++j)
          tma_load_2d(a_ring + sa * kBytesA + j * 8192, &tmGmn, a_full, (vt * 2 + rank) * kTileM + j * 64, kc * kBK);
        // activation rows of this 64-cell chunk: ring rows, or the forward's residual buffer (indexed by half-tile)
        const int hrow = (p.h_map == 0) ? __ldg(p.sub_list + p.slot_begin + kc) * kHalfRows : kc * kBK;
        for (int blk = 0; blk < nblk; ++blk, ++itb) {
          const uint32_t sb = itb % kStagesB, phb = (itb / kStagesB) & 1;
          mbar_wait(smem_u32(&bars->b_empty[sb]), phb ^ 1);
          const uint32_t full_leader = pair_stage_arrive(smem_u32(&bars->b_full[sb]), rank, 2 * kBytesB);
#pragma unroll
          for (int j = 0; j < 2; ++j)
            tma_load_2d_pair(b_ring + sb * kBytesB + j * 8192, &tmHmn, full_leader,
                             (ht * 2 + blk) * kBN + rank * (kBN / 2) + j * 64, hrow);
        }
      }
    }
  } else if (warp == 1 && rank != 0) {
    // peer CTA: tell the leader when this CTA's A stage is in shared memory
    uint32_t ita = 0;
    for (int kc = k_begin; kc < k_end; ++kc, ++ita) {
      const uint32_t sa = ita % kStagesA, pha = (ita / kStagesA) & 1;
      mbar_wait(smem_u32(&bars->a_full[sa]), pha);
      if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&bars->a_peer[sa]), 0));
      __syncwarp();
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(2 * kTileM, kBN, 1, 1, kFmtF16, kFmtF16);
    uint32_t ita = 0, itb = 0;
    for (int kc = k_begin; kc < k_end; ++kc, ++ita) {
      const uint32_t sa = ita % kStagesA, pha = (ita / kStagesA) & 1;
      mbar_wait(smem_u32(&bars->a_full[sa]), pha);
      mbar_wait(smem_u32(&bars->a_peer[sa]), pha);
      for (int blk = 0; blk < nblk; ++blk, ++itb) {
        const uint32_t sb = itb % kStagesB, phb = (itb / kStagesB) & 1;
        mbar_wait(smem_u32(&bars->b_full[sb]), phb);
        tc_fence_after();
        if (lane == 0) {
          mma_kchunk<true, true, true>(tmem_base + blk * kBN, a_ring + sa * kBytesA, b_ring + sb * kBytesB, idesc,
                                       kc > k_begin);
          umma_commit_pair(smem_u32(&bars->b_empty[sb]), 3);
        }
        __syncwarp();
      }
      if (lane == 0) umma_commit_pair(smem_u32(&bars->a_empty[sa]), 3);
      __syncwarp();
    }
    if (lane == 0) umma_commit_pair(smem_u32(&bars->tmem_full), 3);
    __syncwarp();
  } else {
    const int lane_grp = warp & 3;
    const int row = lane_grp * 32 + lane;
    const int v = (vt * 2 + rank) * kTileM + row;
    const float inv_s = __ldg(p.gscale + 1);
    if (do_db) {
      // Column sums of g over the cells of every A stage (MN-major: 64 cell rows of 128 bytes per 64-class box, 16-byte
      // chunks XOR-swizzled by row & 7).  Thread = (16-byte chunk c of the 2 x 8 per row = 8 classes, row group rg): it
      // reads rows rg, rg + 8, ... with one 16-byte load each and keeps 8 fp32 partial sums in registers for the whole
      // kernel; the 8 row groups meet once at the end through shared memory.
      const int et = threadIdx.x - 64;                      // 0 .. 127 over the four epilogue warps
      const int c = et & 15, rg = et >> 4;
      const uint32_t col_off = (c >> 3) * 8192;
      float dacc[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) dacc[e] = 0.f;
      uint32_t ita = 0;
      for (int kc = k_begin; kc < k_end; ++kc, ++ita) {
        const uint32_t sa = ita % kStagesA, pha = (ita / kStagesA) & 1;
        mbar_wait(smem_u32(&bars->a_full[sa]), pha);
        const uint32_t base = a_ring + sa * kBytesA + col_off;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t r = rg + 8 * i;
          uint32_t w0, w1, w2, w3;
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3)
                       : "r"(base + r * 128 + (((c & 7) ^ (r & 7)) << 4)));
          const uint32_t w[4] = {w0, w1, w2, w3};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
            dacc[2 * q] += f.x;
            dacc[2 * q + 1] += f.y;
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bars->a_empty[sa]));
      }
      float* red = reinterpret_cast<float*>(smem.ptr + SmemLayout::db_red);
#pragma unroll
      for (int e = 0; e < 8; ++e) red[(rg * 16 + c) * 8 + e] = dacc[e];
      named_bar_sync(1, 128);
      if (rg == 0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float t = 0.f;
#pragma unroll
          for (int g8 = 0; g8 < 8; ++g8) t += red[(g8 * 16 + c) * 8 + e];      // fixed order
          const int vv = (vt * 2 + rank) * kTileM + (c >> 3) * 64 + (c & 7) * 8 + e;
          if (vv < p.V) {
            if (p.db_fx) fx_add(p.db_fx + vv, t);
            else atomicAdd(p.db + vv, t * inv_s);
          }
        }
      }
    }
    mbar_wait(smem_u32(&bars->tmem_full), 0);
    tc_fence_after();
    for (int c32 = 0; c32 < nblk * (kBN / 32); ++c32) {
      const int col0 = ht * 2 * kBN + c32 * 32;
      if (col0 >= p.H) break;
      float acc[32];
      tmem_ld32(tmem_lane_addr(tmem_base, lane_grp, c32 * 32), acc);
      tmem_ld_wait();
      if (v < p.V && p.dW_fx) {          // deterministic mode: order-independent fixed-point accumulation
        long long* dst = p.dW_fx + static_cast<long long>(v) * p.H + col0;
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (col0 + e < p.H) fx_add(dst + e, acc[e]);
      } else if (v < p.V) {
        float* dst = p.dW + static_cast<long long>(v) * p.H + col0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (col0 + 4 * q + 3 < p.H) {
            red_add_v4(dst + 4 * q, acc[4 * q] * inv_s, acc[4 * q + 1] * inv_s, acc[4 * q + 2] * inv_s,
                       acc[4 * q + 3] * inv_s);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (col0 + 4 * q + e < p.H) atomicAdd(dst + 4 * q + e, acc[4 * q + e] * inv_s);
          }
        }
      }
    }
  }

  tmem_teardown<true>(warp, tmem_base, kTmemCols);
}

}  // namespace

int launch_dw_gemm(const CUtensorMap& tmGmn, const CUtensorMap& tmHmn, const DwArgs& args_in, long long chunk_slots,
                   cudaStream_t stream) {
  ProfScope prof_(kProfDw, stream);
  const size_t smem = SmemLayout::total + kSmemAlign;
  int pairs;
  if (int rc = pair_kernel_setup(reinterpret_cast<const void*>(dw_gemm_kernel), kNumThreads, smem, &pairs)) return rc;
  DwArgs args = args_in;
  const int nblk_total = (args.Hp + kBN - 1) / kBN;
  const int out_blocks = (args.Vp / (2 * kTileM)) * ((nblk_total + 1) / 2);   // 256 x 512 blocks of dW, one pair each
  const long long kchunks = chunk_slots;
  args.ksplit = static_cast<int>(std::max<long long>(1, std::min<long long>(pairs / std::max(1, out_blocks), kchunks)));
  const int grid = 2 * out_blocks * args.ksplit;
  dw_gemm_kernel<<<grid, kNumThreads, smem, stream>>>(tmGmn, tmHmn, args);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace rb
