// Fused joint GEMM kernel (forward "F" and backward "G" modes).
//
// Replaces rnnt/joint.py:32-39 (broadcast add + tanh + joint_ln) fused with the first half of
// torchaudio's rnnt_loss (ReduceMax2D / ReduceLogSumExpGivenMax2D / ComputeLogProbs, reference call
// site rnnt/model.py:35-41) in F mode, and with ComputeGradients in G mode.  The (B,T,U1,V) logit
// tensor only ever exists as fp32 accumulators in TMEM.
//
//   logits[c, v] = sum_k f16(tanh(enc[b,t,k] + pred[b,u,k])) * f16(W[v,k])  (+ bias[v] in the epilogue)
// (fp16 operands: tanh output lies in [-1,1] and joint weights are O(1), so fp16's 11-bit mantissa gives 8x
// finer rounding than bf16 at the same tensor-core rate; accumulation is fp32 in TMEM.)
//
// Structure (persistent CTA PAIRS, one CTA per SM; work unit per CTA = 128 GEMM rows = TWO half-tiles of 16(t) x 4(u)
// lattice cells -- in the forward two consecutive half-tiles, in the backward any two entries of the list of
// half-tiles that carry non-zero gradients; the two 128-row units of a pair form one M=256 tcgen05.mma.cta_group::2
// issued by the pair's leader):
//   * The hidden activations h = tanh(enc+pred) of a tile are produced ONCE, as fp16 rows of a global buffer
//     (the residual the backward re-uses, or a small per-CTA scratch), by 8 producer warps that run one to two
//     tiles AHEAD of the tensor pipe.  They are decoupled from the MMA pipeline: no shared-memory staging, no
//     per-chunk hand-off, their MUFU/ALU work hides under the MMAs of the previous tile.
//   * The GEMM itself is a plain TMA-fed tcgen05 pipeline: per (pass, k-chunk) each CTA loads its own 128x64 h box
//     (just written, so an L2 hit) and HALF of the 256x64 W box (the pair shares the B operand: 64 instead of 96 bytes
//     of L2 traffic per SM and clock) into a 6-stage ring; a pass is one 256-column accumulator, and the two halves
//     of TMEM ping-pong so that the epilogue of pass i overlaps the MMAs of pass i+1.
//   * G mode with saved activations needs no producers at all.
//
// Warp roles: 0 TMA loader | 1 tcgen05.mma issuer (leader CTA only) | 2-9 epilogue (set e = warps 2+4e..5+4e drains accumulator e)
//             | 10-17 (PRODUCE only) activation producers
#include <algorithm>

#include "kernels.h"
#include "tc_kernel.cuh"

namespace rb {

namespace {

constexpr int kStages = 6;
constexpr int kBytesA = kTileM * kBK * 2;       // 16 KB: 128 cells x 64 k
constexpr int kBytesB = (kBN / 2) * kBK * 2;    // 16 KB: this CTA's 128 of the pass's 256 classes x 64 k
constexpr int kStageBytes = kBytesA + kBytesB;
constexpr int kFirstEpiWarp = 2;
constexpr int kNumEpiWarps = 8;
constexpr int kFirstProdWarp = 10;
constexpr int kNumProdWarps = 8;
constexpr int kThreadsNoProd = 32 * kFirstProdWarp;                     // 320
constexpr int kThreadsProd = 32 * (kFirstProdWarp + kNumProdWarps);     // 576
constexpr int kTmemCols = 512;
constexpr int kScratchSlots = 2;   // per-CTA activation scratch (h_map 2): unit n is stored only after unit n-2 is consumed

struct SmemLayout {
  static constexpr int ring = 0;
  static constexpr int xchg = ring + kStages * kStageBytes;   // F: set-1 -> set-0 softmax partials (2 x 128 x 16 B)
  static constexpr int bars = xchg + 2 * kTileM * 16;
  // producers, T-contiguous encoder layout: per half-tile a double-buffered 16(t) x 64(k) fp32 transposing stage
  // epilogue: bias * log2e of the pass a set is draining, double-buffered per set (2 sets x 2 x 256 floats)
  static constexpr int bias_stage = bars + 256;
  static constexpr int len_tab = bias_stage + 2 * 2 * kBN * 4;   // tile_off / T_len / U_len copies (stage_len_tables)
  static constexpr int enc_stage = len_tab + kLenTabBytes;
  // G without producers: per epilogue warp a 32-row x 64-byte transposing stage for the gradient stores (same offset as
  // the producers' stage, which that kernel does not have)
  static constexpr int g_stage = enc_stage;
  static constexpr int total_noprod = g_stage + kNumEpiWarps * 32 * 64;
  static constexpr int total = enc_stage + 2 * 2 * kTileT * kBK * 4;
};
struct Bars {
  uint64_t full[kStages], empty[kStages], tmem_full[2], tmem_empty[2], h_ready[2], tile_done[2];
  uint32_t tmem_slot;
};
static_assert(sizeof(Bars) <= SmemLayout::bias_stage - SmemLayout::bars, "barrier block overflows its region");

__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// v[idx] for a run-time idx in [0, 32) without local memory: a 5-level select tree (31 FSEL).
__device__ __forceinline__ float pick32(const float (&v)[32], int idx) {
  float a[16], b[8], c[4];
  const bool s0 = idx & 1, s1 = idx & 2, s2 = idx & 4, s3 = idx & 8, s4 = idx & 16;
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = s0 ? v[2 * i + 1] : v[2 * i];
#pragma unroll
  for (int i = 0; i < 8; ++i) b[i] = s1 ? a[2 * i + 1] : a[2 * i];
#pragma unroll
  for (int i = 0; i < 4; ++i) c[i] = s2 ? b[2 * i + 1] : b[2 * i];
  const float d0 = s3 ? c[1] : c[0], d1 = s3 ? c[3] : c[2];
  return s4 ? d1 : d0;
}

}  // namespace

int joint_gemm_scratch_tiles(int grid) { return grid * kScratchSlots; }

// MODE 0 = forward (lse + gather), 1 = backward (gradient ring); PRODUCE: activation producer warps present;
// TMAJOR: the producers read T-contiguous encoder features (the (B,T,H) view of a (B,H,T) tensor) instead of H-contiguous
template <int MODE, bool PRODUCE, bool TMAJOR = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PRODUCE ? kThreadsProd : kThreadsNoProd, 1)
joint_gemm_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmH,
                  const __grid_constant__ CUtensorMap tmH2, JointArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const AlignedSmem smem = aligned_smem(smem_raw);
  using SL = SmemLayout;

  const uint32_t ring = smem.addr + SL::ring;
  Bars* bars = reinterpret_cast<Bars*>(smem.ptr + SL::bars);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();          // 0 = leader of the pair (issues the MMAs)
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;

  // work list: slots of 64 rows (half-tiles); identity over all half-tiles in the forward
  const int total_slots = p.n_active ? __ldg(p.n_active) : __ldg(p.tile_off + p.B);
  const int slot_end = min(total_slots, p.slot_begin + p.slot_cap);   // this launch: slots [slot_begin, slot_end)
  const int nunits = (max(0, slot_end - p.slot_begin) + 1) >> 1;      // 128-row units = pairs of consecutive slots
  const int nk = p.Hp / kBK;
  const int npass = p.Vp / kBN;

  // half-tile id of sub-slot s of unit q, or -1 past the end of the list
  auto half_id = [&](int q, int s) -> int {
    const int slot = p.slot_begin + 2 * q + s;
    if (q >= nunits || slot >= slot_end) return -1;
    return p.sub_list ? __ldg(p.sub_list + slot) : slot;
  };
  // first row of the activation buffer that holds sub-slot s of unit q (the cnt-th unit of this CTA)
  auto h_row0 = [&](int q, int s, int hid, uint32_t cnt) -> int {
    if (p.h_map == 0) return hid * kHalfRows;                     // full buffer, indexed by half-tile
    if (p.h_map == 1) return (2 * q + s) * kHalfRows;             // backward ring, indexed by slot of this chunk
    return (static_cast<int>(blockIdx.x) * kScratchSlots + static_cast<int>(cnt % kScratchSlots)) * kTileM + s * kHalfRows;
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmH);
    tma_prefetch_desc(&tmH2);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(smem_u32(&bars->full[s]), 2);        // leader's copy: one expect_tx arrival per CTA of the pair
      mbar_init(smem_u32(&bars->empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bars->tmem_full[a]), 1);
      mbar_init(smem_u32(&bars->tmem_empty[a]), kNumEpiWarps);   // leader's copy: 4 warps of set a in each CTA
      mbar_init(smem_u32(&bars->h_ready[a]), kNumProdWarps);
      mbar_init(smem_u32(&bars->tile_done[a]), 1);
    }
    mbar_fence_init();
  }
  tmem_alloc<true>(warp, &bars->tmem_slot, kTmemCols);
  const LenTables lt = stage_len_tables(reinterpret_cast<int*>(smem.ptr + SL::len_tab), p.tile_off, p.T_len, p.U_len, p.B);
  const uint32_t tmem_base = tmem_publish<true>(&bars->tmem_slot);

// this CTA's units: q = base + rank for base = 2 * (pair + i * npairs); a pair whose second unit is past the end still
// runs (the leader's MMA spans both CTAs) with that CTA's outputs suppressed
#define RB_TILE_LOOP(cntvar) for (int base_ = 2 * pair; base_ < nunits; base_ += 2 * npairs, ++cntvar)

  if (warp == 0) {
    // ===================================================================== TMA loader (W boxes + activation boxes)
    if (lane == 0) {
      uint32_t it = 0, cnt = 0;
      RB_TILE_LOOP(cnt) {
        const int q = base_ + rank;
        int hrow[2];
#pragma unroll
        for (int sh = 0; sh < 2; ++sh) {
          const int hid = half_id(q, sh);
          hrow[sh] = hid >= 0 ? h_row0(q, sh, hid, cnt) : 0;     // nothing there: any resident rows (results unused)
        }
        if (PRODUCE) {
          mbar_wait(smem_u32(&bars->h_ready[cnt & 1]), (cnt >> 1) & 1);
          fence_proxy_async_all();   // the producers' generic-proxy global stores -> TMA (async proxy) reads
        }
        for (int pass = 0; pass < npass; ++pass) {
          for (int kc = 0; kc < nk; ++kc, ++it) {
            const uint32_t s = it % kStages, ph = (it / kStages) & 1;
            mbar_wait(smem_u32(&bars->empty[s]), ph ^ 1);
            // (diagnostics: dbg bit 32 skips every other W load -- stale operands, used to measure what L2 traffic costs)
            const bool skipw = (p.dbg & 32) && (it & 1);
            const uint32_t full_leader =
                pair_stage_arrive(smem_u32(&bars->full[s]), rank, 2 * kStageBytes - (skipw ? 2 * kBytesB : 0));
            if (!skipw)
              tma_load_2d_pair(ring + s * kStageBytes, &tmW, full_leader, kc * kBK, pass * kBN + rank * (kBN / 2));
            if (hrow[1] == hrow[0] + kHalfRows) {     // both halves of one tile / adjacent ring slots: one 128-row box
              tma_load_2d_pair(ring + s * kStageBytes + kBytesB, &tmH2, full_leader, kc * kBK, hrow[0]);
            } else {
              tma_load_2d_pair(ring + s * kStageBytes + kBytesB, &tmH, full_leader, kc * kBK, hrow[0]);
              tma_load_2d_pair(ring + s * kStageBytes + kBytesB + kBytesA / 2, &tmH, full_leader, kc * kBK, hrow[1]);
            }
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===================================================================== MMA issuer (leader CTA of the pair)
    // (diagnostics: dbg bit 16 reinterprets the operands as bf16 -- wrong numbers, used to measure operand-format power)
    const uint32_t idesc = (p.dbg & 16) ? make_idesc(2 * kTileM, kBN, 0, 0, kFmtBF16, kFmtBF16)
                                        : make_idesc(2 * kTileM, kBN, 0, 0, kFmtF16, kFmtF16);
    uint32_t it = 0, pc = 0, cnt = 0;
    RB_TILE_LOOP(cnt) {
      for (int pass = 0; pass < npass; ++pass, ++pc) {
        const uint32_t acc = pc & 1;
        mbar_wait(smem_u32(&bars->tmem_empty[acc]), ((pc >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int kc = 0; kc < nk; ++kc, ++it) {
          const uint32_t s = it % kStages, ph = (it / kStages) & 1;
          mbar_wait(smem_u32(&bars->full[s]), ph);
          tc_fence_after();
          if (lane == 0) {
            const uint32_t b_addr = ring + s * kStageBytes, a_addr = b_addr + kBytesB;
            mma_kchunk<true, false, false>(tmem_base + acc * kBN, a_addr, b_addr, idesc, kc != 0);
            umma_commit_pair(smem_u32(&bars->empty[s]), 3);
          }
          __syncwarp();
        }
        if (lane == 0) umma_commit_pair(smem_u32(&bars->tmem_full[acc]), 3);
        __syncwarp();
      }
      if (PRODUCE) {
        if (lane == 0) umma_commit_pair(smem_u32(&bars->tile_done[cnt & 1]), 3);   // both tiles' activation rows are consumed
        __syncwarp();
      }
    }
  } else if (warp >= kFirstEpiWarp && warp < kFirstEpiWarp + kNumEpiWarps) {
    // ===================================================================== epilogue
    // Set e drains accumulator e, i.e. every pass with (global pass counter & 1) == e.
    const int lane_grp = warp & 3;  // TMEM lane quarter this warp may access
    const int eset = (warp - kFirstEpiWarp) >> 2;
    const int row = lane_grp * 32 + lane;
    const int sub = row >> 6;                     // which of the unit's two half-tiles this row belongs to
    const int ti = (row & 63) >> 2, ui = row & 3;
    float4* xchg = reinterpret_cast<float4*>(smem.ptr + SL::xchg);
    const uint32_t tmem_empty_leader = mapa_shared(smem_u32(&bars->tmem_empty[eset]), 0);
    uint32_t pc = 0, tcount = 0;
    RB_TILE_LOOP(tcount) {
      const int q = base_ + rank;
      const bool mine = q < nunits;
      const int hid = half_id(q, sub);
      const TileCoord tc = decode_half(lt.tile_off, lt.T_len, lt.U_len, p.B, p.T, p.U1, max(hid, 0));
      const int t = tc.t0 + ti, u = tc.u0 + ui;
      const bool valid = hid >= 0 && (t < tc.Tb) && (u <= tc.Ub);
      const long long cell = (static_cast<long long>(tc.b) * p.T + min(t, p.T - 1)) * p.U1 + min(u, p.U1 - 1);
      int tgt = -1;
      if (valid && u < tc.Ub) tgt = __ldg(p.targets + static_cast<long long>(tc.b) * p.tgt_ld + u);
      // F state (log2 units)
      float m = -INFINITY, ssum = 0.f, x_tgt = -INFINITY, x_blank = -INFINITY;
      // G state
      float gam = 0.f, eB = 0.f, eE = 0.f, lse2 = 1e30f, cbound = 0.f;
      float g_blank = 0.f, g_tgt = 0.f;   // G: finished gradient values of the blank / label columns
      if (MODE == 1 && valid) {
        const float4 c4 = __ldg(p.coef + cell);
        gam = c4.x; eB = c4.y; eE = c4.z; lse2 = c4.w * kLog2e;
        const float2 l = __ldg(reinterpret_cast<const float2*>(p.lp) + cell);   // log p(blank), log p(label)
        g_blank = ex2_approx(l.x * kLog2e) * gam - eB;
        g_tgt = ex2_approx(l.y * kLog2e) * gam - eE;
        if (tgt == p.blank) g_tgt -= eB;     // (never the case for valid transcripts)
        if (p.clamp > 0.f) {
          cbound = p.clamp * fabsf(p.dcost ? __ldg(p.dcost + tc.b) : 1.f) * __ldg(p.gscale);
          g_blank = fminf(fmaxf(g_blank, -cbound), cbound);
          g_tgt = fminf(fmaxf(g_tgt, -cbound), cbound);
        }
      }
      __half* g_row = nullptr;
      if (MODE == 1)
        g_row = p.g_ring + (static_cast<long long>(q) * kTileM + row) * p.Vp;

      for (int pass = 0; pass < npass; ++pass, ++pc) {
        if (static_cast<int>(pc & 1) != eset) continue;
        // this pass's 256 bias values -> shared memory (requested before the wait for the accumulator; the L1 is a few
        // KB next to 220 KB of shared memory and the producers stream through it, so per-chunk __ldg's of the bias were
        // L2 round trips on the drain's critical path).  Buffer (pc >> 1) & 1 of this set: the set's barrier of pass
        // j orders every warp's reads of pass j-1 before any write of pass j+1.
        float* bias_s = reinterpret_cast<float*>(smem.ptr + SL::bias_stage) + (eset * 2 + ((pc >> 1) & 1)) * kBN;
        {
          const int i2 = (lane_grp * 32 + lane) * 2;
          *reinterpret_cast<float2*>(bias_s + i2) = __ldg(reinterpret_cast<const float2*>(p.bias2 + pass * kBN + i2));
        }
        named_bar_sync(1 + eset, 128);
        mbar_wait(smem_u32(&bars->tmem_full[eset]), (pc >> 1) & 1);
        tc_fence_after();
        const int nchunk = ((p.dbg & 1) || !mine) ? 0 : (kBN / 32);
        for (int c32 = 0; c32 < nchunk; ++c32) {
          const int col0 = pass * kBN + c32 * 32;  // global column of v[0]
          float v[32];
          tmem_ld32(tmem_lane_addr(tmem_base, lane_grp, eset * kBN + c32 * 32), v);
          tmem_ld_wait();
          const float4* b4 = reinterpret_cast<const float4*>(bias_s + c32 * 32);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 bb = b4[q];
            fma2(v[4 * q + 0], v[4 * q + 1], kLog2e, bb.x, bb.y);
            fma2(v[4 * q + 2], v[4 * q + 3], kLog2e, bb.z, bb.w);
          }
          if (MODE == 0) {
            // online softmax over the chunk: 16 three-input maxima, then (v - m) / sum as packed pairs
            float cmax = max3(v[0], v[1], v[2]);
#pragma unroll
            for (int j = 3; j < 31; j += 2) cmax = max3(cmax, v[j], v[j + 1]);
            const float m_new = fmaxf(m, fmaxf(cmax, v[31]));
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              float e0 = v[j], e1 = v[j + 1];
              add2(e0, e1, -m_new, -m_new);
              add2(s0, s1, ex2_approx(e0), ex2_approx(e1));
            }
            const float acc = s0 + s1;
            ssum = ssum * ex2_approx(m - m_new) + acc;
            m = m_new;
            // label / blank logits: only the one chunk that holds the column pays for the selection
            if (static_cast<unsigned>(tgt - col0) < 32u) x_tgt = pick32(v, tgt - col0);
            if (static_cast<unsigned>(p.blank - col0) < 32u) x_blank = pick32(v, p.blank - col0);
          } else {
            // softmax * gamma = 2^(x - lse) * gamma, as packed pairs around the two MUFU operations
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              add2(v[j], v[j + 1], -lse2, -lse2);
              v[j] = ex2_approx(v[j]);
              v[j + 1] = ex2_approx(v[j + 1]);
              mul2(v[j], v[j + 1], gam);
            }
            if (p.clamp > 0.f) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = fminf(fmaxf(v[j], -cbound), cbound);
            }
            uint4 w4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              w4[q].x = pack_f16x2(v[8 * q + 0], v[8 * q + 1]);
              w4[q].y = pack_f16x2(v[8 * q + 2], v[8 * q + 3]);
              w4[q].z = pack_f16x2(v[8 * q + 4], v[8 * q + 5]);
              w4[q].w = pack_f16x2(v[8 * q + 6], v[8 * q + 7]);
            }
            if (!PRODUCE) {
              // fp16 (scaled by S through the coefficients) to the gradient ring through a per-warp transposing stage:
              // thread = row writes its 64 bytes (16-byte chunk c at c ^ (row >> 1), conflict-free), the one-hot columns
              // are patched in place, then 4 lanes per row store 64 contiguous bytes -- 8 full-sector segments per
              // instruction instead of 32 scattered 16-byte ones.
              uint8_t* gs = smem.ptr + SL::g_stage + (warp - kFirstEpiWarp) * (32 * 64);
              __syncwarp();                                     // the previous chunk's read-back is complete
#pragma unroll
              for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(gs + lane * 64 + ((q ^ (lane >> 1)) & 3) * 16) = w4[q];
              if (static_cast<unsigned>(p.blank - col0) < 32u) {
                const int cc = p.blank - col0;
                *reinterpret_cast<__half*>(gs + lane * 64 + (((cc >> 3) ^ (lane >> 1)) & 3) * 16 + (cc & 7) * 2) = __float2half_rn(g_blank);
              }
              if (static_cast<unsigned>(tgt - col0) < 32u) {
                const int cc = tgt - col0;
                *reinterpret_cast<__half*>(gs + lane * 64 + (((cc >> 3) ^ (lane >> 1)) & 3) * 16 + (cc & 7) * 2) = __float2half_rn(g_tgt);
              }
              __syncwarp();
              __half* g_base = p.g_ring + (static_cast<long long>(q) * kTileM + lane_grp * 32) * p.Vp + col0;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int r = 8 * i + (lane >> 2), c = lane & 3;
                const uint4 val = *reinterpret_cast<const uint4*>(gs + r * 64 + ((c ^ (r >> 1)) & 3) * 16);
                *reinterpret_cast<uint4*>(g_base + static_cast<long long>(r) * p.Vp + c * 8) = val;
              }
            } else {
              // (memory-lean variant, no room for the stage: 64 bytes per row straight from the owning thread)
              uint4* dst = reinterpret_cast<uint4*>(g_row + col0);
#pragma unroll
              for (int q = 0; q < 4; ++q) dst[q] = w4[q];
              // the two columns with one-hot terms are patched afterwards (same thread, program order): their softmax
              // probabilities are exp(lp) from the forward, so no per-element comparison is needed in the loop above
              if (static_cast<unsigned>(p.blank - col0) < 32u) g_row[p.blank] = __float2half_rn(g_blank);
              if (static_cast<unsigned>(tgt - col0) < 32u) g_row[tgt] = __float2half_rn(g_tgt);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tmem_empty_leader);
      }
      if (MODE == 0) {
        // combine the two sets' online-softmax partials: set 1 -> smem -> set 0 writes lp / lse
        float4* xs = xchg + (tcount & 1) * kTileM + row;
        if (eset == 1) *xs = make_float4(m, ssum, x_tgt, x_blank);
        named_bar_sync(3, 32 * kNumEpiWarps);
        if (eset == 0 && valid && !(p.dbg & 1)) {
          const float4 o = *xs;
          const float mm = fmaxf(m, o.x);   // finite: every tile has at least one pass
          const float stot = ssum * ex2_approx(m - mm) + o.y * ex2_approx(o.x - mm);
          const float l2 = mm + lg2_approx(stot);
          p.lse[cell] = l2 * kLn2;
          float2 out;
          out.x = (fmaxf(x_blank, o.w) - l2) * kLn2;
          out.y = (tgt >= 0) ? (fmaxf(x_tgt, o.z) - l2) * kLn2 : 0.f;
          reinterpret_cast<float2*>(p.lp)[cell] = out;
        }
      }
    }
  } else if (PRODUCE && warp >= kFirstProdWarp) {
    // ===================================================================== activation producers
    // Warp rg produces rows rg*16 .. rg*16+15 of the unit = t-rows 4(rg&3) .. +3 x 4 u of half-tile rg>>2.  Lane l owns
    // the 16-byte column chunk c = l & 7 (8 hidden units) of the four rows (t-row 2(rs>>1) + i) x (u = 2(rs&1) + j),
    // rs = l >> 3: (2 + 2) x 8 inputs -> 32 tanh -> four 16-byte global stores; the 8 lanes of one row write 128
    // contiguous bytes.
    //
    // Encoder layout.  H-contiguous features (enc_sh == 1) are read straight into that register tile (two float4 per
    // frame).  The reference hands the joint the (B,T,H) VIEW of the encoder's (B,H,T) output (rnnt/model.py:27-28),
    // i.e. T-contiguous memory (enc_st == 1): the 4 warps of a half-tile then fetch its 64(k) x 16(t) fp32 box with
    // fully used 64-byte row segments (lane = (k row, 4 frames): two float4 loads per chunk), transpose it through a
    // double-buffered, XOR-swizzled shared-memory stage (conflict-free both ways) and read their register tile from
    // there -- no transposed copy of the features in HBM, same number of L1 wavefronts as the H-contiguous path.
    const int rg = warp - kFirstProdWarp;
    const int c = lane & 7, rs = lane >> 3;
    const int sub = rg >> 2, tq = (rg & 3) * 4 + (rs >> 1) * 2, uq = (rs & 1) * 2;
    constexpr bool t_major = TMAJOR;
    const bool vec_ok = ((p.enc_sh | p.enc_sb) & 3) == 0;     // 16-byte aligned rows of the (B,H,T) tensor
    const int wl = rg & 3, kk = lane >> 2, tq4 = lane & 3;    // T-major fetch: k rows 16 wl + 2 kk, + 1; frames 4 tq4 .. +3
    float* stage = reinterpret_cast<float*>(smem.ptr + SL::enc_stage) + sub * (2 * kTileT * kBK);
    uint32_t cnt = 0, cc = 0;                                 // cc: running chunk counter = stage buffer parity
    RB_TILE_LOOP(cnt) {
      const int q = base_ + rank;
      const int hid = half_id(q, sub);
      if (hid < 0) {            // nothing to produce for this half (uniform over its 4 warps): keep the barrier protocol
        if (cnt >= 2) mbar_wait(smem_u32(&bars->tile_done[cnt & 1]), ((cnt >> 1) - 1) & 1);
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bars->h_ready[cnt & 1]));
        continue;
      }
      const TileCoord tc = decode_half(lt.tile_off, lt.T_len, lt.U_len, p.B, p.T, p.U1, hid);
      const int row0 = h_row0(q, sub, hid, cnt);
      const float* e_ptr[2];
      const float* p_ptr[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        e_ptr[i] = p.enc + tc.b * p.enc_sb + static_cast<long long>(min(tc.t0 + tq + i, p.T - 1)) * p.enc_st + 8 * c;
        p_ptr[i] = p.pred + tc.b * p.pred_sb + static_cast<long long>(min(tc.u0 + uq + i, p.U1 - 1)) * p.pred_su + 8 * c;
      }
      float4 e_cur[2][2], p_cur[2][2], g_cur[2];
      auto load_enc = [&](int kc, float4 (&e)[2][2]) {         // H-contiguous: straight into the register tile
        const bool ok = kc * kBK + 8 * c < p.H;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          e[i][0] = ok ? __ldg(reinterpret_cast<const float4*>(e_ptr[i] + kc * kBK)) : make_float4(0.f, 0.f, 0.f, 0.f);
          e[i][1] = ok ? __ldg(reinterpret_cast<const float4*>(e_ptr[i] + kc * kBK) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      auto load_pred = [&](int kc, float4 (&pp)[2][2]) {
        const bool ok = kc * kBK + 8 * c < p.H;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          pp[i][0] = ok ? __ldg(reinterpret_cast<const float4*>(p_ptr[i] + kc * kBK)) : make_float4(0.f, 0.f, 0.f, 0.f);
          pp[i][1] = ok ? __ldg(reinterpret_cast<const float4*>(p_ptr[i] + kc * kBK) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      auto fetch_t = [&](int kc, float4 (&g)[2]) {             // T-contiguous: this lane's 2 (k rows) x 4 frames
        const int t = tc.t0 + 4 * tq4;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int k = kc * kBK + 16 * wl + 2 * kk + h;       // two ADJACENT k rows: their values pair up into 8-byte stores
          g[h] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (k < p.H) {
            const float* src = p.enc + tc.b * p.enc_sb + static_cast<long long>(k) * p.enc_sh;
            if (vec_ok && t + 3 < p.T) {
              g[h] = __ldg(reinterpret_cast<const float4*>(src + t));
            } else {
              g[h].x = __ldg(src + min(t, p.T - 1));
              g[h].y = __ldg(src + min(t + 1, p.T - 1));
              g[h].z = __ldg(src + min(t + 2, p.T - 1));
              g[h].w = __ldg(src + min(t + 3, p.T - 1));
            }
          }
        }
      };
      // stage[buf][t][k ^ ((t >> 2 & 3) << 3)]: writers (fixed frame offset, lanes = 8 k pairs x 4 frame groups, one 8-byte
      // store per frame) and readers (fixed frame, 8 lanes x 8 consecutive k, 16-byte loads) are both bank-conflict free
      auto stage_put = [&](uint32_t buf, const float4 (&g)[2]) {
        float2* dst = reinterpret_cast<float2*>(stage + buf * (kTileT * kBK) + (4 * tq4) * kBK + ((16 * wl + 2 * kk) ^ (tq4 << 3)));
        dst[0] = make_float2(g[0].x, g[1].x);
        dst[kBK / 2] = make_float2(g[0].y, g[1].y);
        dst[kBK] = make_float2(g[0].z, g[1].z);
        dst[3 * kBK / 2] = make_float2(g[0].w, g[1].w);
      };
      auto stage_get = [&](uint32_t buf, float4 (&e)[2][2]) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const float4* src = reinterpret_cast<const float4*>(stage + buf * (kTileT * kBK) + (tq + i) * kBK +
                                                              ((8 * c) ^ (wl << 3)));
          e[i][0] = src[0];
          e[i][1] = src[1];
        }
      };
      if (t_major) fetch_t(0, g_cur); else load_enc(0, e_cur);
      load_pred(0, p_cur);
      // stay at most two units ahead of the tensor pipe: unit cnt-2 must be fully consumed (also keeps the
      // two-phase h_ready / tile_done barriers and the 4-slot scratch unambiguous)
      if (cnt >= 2) mbar_wait(smem_u32(&bars->tile_done[cnt & 1]), ((cnt >> 1) - 1) & 1);
      // row of (t-row tq + i, u = uq + j) inside the half-tile: (tq + i) * 4 + uq + j
      __half* out_base = p.h_out + static_cast<long long>(row0 + tq * 4 + uq) * p.Hp + 8 * c;
      for (int kc = 0; kc < nk; ++kc, ++cc) {
        if (p.dbg & 2) break;   // diagnostics: leave the buffer's previous contents (valid data from an earlier call)
        if (t_major) {
          stage_put(cc & 1, g_cur);
          if (kc + 1 < nk) fetch_t(kc + 1, g_cur);             // next box in flight while this one is consumed
          named_bar_sync(4 + sub, 128);                        // the half-tile's 4 warps: box complete, buffer cc-1 free
          stage_get(cc & 1, e_cur);
        }
        uint4 w[2][2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {        // t-row
#pragma unroll
          for (int j = 0; j < 2; ++j) {      // u
            const float4 a0 = e_cur[i][0], a1 = e_cur[i][1], b0 = p_cur[j][0], b1 = p_cur[j][1];
            w[i][j].x = pack_f16x2(tanh_approx(a0.x + b0.x), tanh_approx(a0.y + b0.y));
            w[i][j].y = pack_f16x2(tanh_approx(a0.z + b0.z), tanh_approx(a0.w + b0.w));
            w[i][j].z = pack_f16x2(tanh_approx(a1.x + b1.x), tanh_approx(a1.y + b1.y));
            w[i][j].w = pack_f16x2(tanh_approx(a1.z + b1.z), tanh_approx(a1.w + b1.w));
          }
        }
        // the inputs of the next chunk are requested before the stores of this one are issued
        if (kc + 1 < nk) {
          if (!t_major) load_enc(kc + 1, e_cur);
          load_pred(kc + 1, p_cur);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j)
            *reinterpret_cast<uint4*>(out_base + static_cast<long long>(i * 4 + j) * p.Hp + kc * kBK) = w[i][j];
      }
      fence_proxy_async_all();   // generic-proxy global writes -> visible to the loader's TMA reads
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->h_ready[cnt & 1]));
    }
  }

#undef RB_TILE_LOOP
  tmem_teardown<true>(warp, tmem_base, kTmemCols);
}

int launch_joint_gemm(int mode, bool produce, const CUtensorMap& tmW, const CUtensorMap& tmH, const CUtensorMap& tmH2,
                      const JointArgs& args, long long max_slots, cudaStream_t stream) {
  ProfScope prof_(mode == 0 ? kProfJointF : kProfJointG, stream);
  RB_REQUIRE(mode != 0 || produce, -30, "forward joint kernel always produces the activations");
  const bool t_major = produce && args.enc_sh != 1;
  void (*const kernel)(CUtensorMap, CUtensorMap, CUtensorMap, JointArgs) =
      !produce    ? joint_gemm_kernel<1, false, false>
      : mode == 0 ? (t_major ? joint_gemm_kernel<0, true, true> : joint_gemm_kernel<0, true, false>)
                  : (t_major ? joint_gemm_kernel<1, true, true> : joint_gemm_kernel<1, true, false>);
  const int threads = produce ? kThreadsProd : kThreadsNoProd;
  const size_t smem = (produce ? SmemLayout::total : SmemLayout::total_noprod) + kSmemAlign;
  int pairs;
  if (int rc = pair_kernel_setup(reinterpret_cast<const void*>(kernel), threads, smem, &pairs)) return rc;
  const long long want_pairs = std::max<long long>(1, (max_slots + 3) / 4);   // 2 slots per CTA, 2 CTAs per pair
  const int grid = 2 * static_cast<int>(std::min<long long>(pairs, want_pairs));
  if (args.dbg & 8)
    fprintf(stderr, "rnnt_b200: joint gemm mode %d produce %d t-major %d grid %d\n", mode, (int)produce, (int)t_major, grid);
  kernel<<<grid, threads, smem, stream>>>(tmW, tmH, tmH2, args);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace rb
