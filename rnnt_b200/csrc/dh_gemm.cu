// Backward contraction #2, transposed:  dh^T[k, c] = sum_v W[v,k] * g[c,v]   (M = hidden unit k, N = lattice cell c),
// fused with the tanh backward and the two broadcast reductions.
//
// Replaces autograd through rnnt/joint.py:32-39 for the activations (SURVEY 8a-8):
//   dz[c,k]       = dh[c,k] * (1 - tanh(enc[b,t,k] + pred[b,u,k])^2)
//   d_enc[b,t,k]  = sum_u dz[b,t,u,k]      d_pred[b,u,k] = sum_t dz[b,t,u,k]
// Putting the hidden unit on the TMEM lane makes a thread own ONE k and 32 consecutive cells (= 8 t x 4 u of a
// half-tile) per tcgen05.ld: both reductions are plain register sums, tanh' is recomputed from 8 enc + 4 pred
// values per thread (MUFU is otherwise idle here), and the fp32 atomics are coalesced over k.
//   A operand: W^T block (128 k x 64 v) = MN-major view of the fp16 W[Vp,Hp] buffer (TMA, two 64x64 boxes)
//   B operand: gradient ring g [ring_rows, Vp] fp16, K-major (TMA, one 64 x 128 box per CTA = two work-list slots)
// Work item of a CTA PAIR = (four half-tiles of the work list = 256 cells, block of 256 hidden units): one tcgen05.mma.cta_group::2
// with M = 256; each CTA stages its own 128 hidden units of W^T and HALF of the gradient box (two half-tiles), so
// the L2 -> shared-memory traffic is 64 instead of 96 bytes per SM and clock.  Accumulators ping-pong between the two
// halves of TMEM so the epilogue of item i overlaps the MMAs of item i+1.
#include <algorithm>

#include "kernels.h"
#include "tc_kernel.cuh"

namespace rb {
namespace {

constexpr int kStages = 6;
constexpr int kBytesA = kBK * 128 * 2;          // 16 KB: 64 v x 128 k (this CTA's hidden units)
constexpr int kBytesB = (kBN / 2) * kBK * 2;    // 16 KB: this CTA's 128 of the item's 256 cells x 64 v
constexpr int kEpiSets = 2;                       // epilogue warp sets; set e handles slots 2e, 2e+1 of the item
constexpr int kNumThreads = 64 + 128 * kEpiSets;
constexpr int kTmemCols = 512;

struct SmemLayout {
  static constexpr int b_ring = 0;
  static constexpr int a_ring = b_ring + kStages * kBytesB;
  static constexpr int bars = a_ring + kStages * kBytesA;
  static constexpr int total = bars + 256;
};
struct Bars {
  uint64_t full[kStages], empty[kStages], tmem_full[2], tmem_empty[2];
  uint32_t tmem_slot;
};
static_assert(sizeof(Bars) <= SmemLayout::total - SmemLayout::bars, "barrier block overflows its region");

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kNumThreads, 1)
dh_gemm_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmWmn, DhArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const AlignedSmem smem = aligned_smem(smem_raw);
  const uint32_t b_ring = smem.addr + SmemLayout::b_ring;
  const uint32_t a_ring = smem.addr + SmemLayout::a_ring;
  Bars* bars = reinterpret_cast<Bars*>(smem.ptr + SmemLayout::bars);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;
  const int total_slots = __ldg(p.n_active);
  const int slot_end = min(total_slots, p.slot_begin + p.slot_cap);   // work-list slots (half-tiles)
  const int nslots = max(0, slot_end - p.slot_begin);
  const int ncb = (nslots + 3) / 4;                 // cell blocks of 4 half-tiles (256 ring rows)
  const int nhb = (p.Hp + 255) / 256;               // hidden blocks of 256 (128 per CTA of the pair)
  const int nitems = ncb * nhb;
  const int nk = p.Vp / kBK;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmG);
    tma_prefetch_desc(&tmWmn);
    for (int s = 0; s < kStages; ++s) { mbar_init(smem_u32(&bars->full[s]), 2); mbar_init(smem_u32(&bars->empty[s]), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(smem_u32(&bars->tmem_full[s]), 1); mbar_init(smem_u32(&bars->tmem_empty[s]), 8 * kEpiSets); }
    mbar_fence_init();
  }
  const uint32_t tmem_base = tmem_setup<true>(warp, &bars->tmem_slot, kTmemCols);

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int item = pair; item < nitems; item += npairs) {
        const int cb = item / nhb, hb = item % nhb;
        const int k0 = hb * 256 + rank * 128;            // this CTA's hidden units
        for (int kc = 0; kc < nk; ++kc, ++it) {
          const uint32_t s = it % kStages, ph = (it / kStages) & 1;
          mbar_wait(smem_u32(&bars->empty[s]), ph ^ 1);
          const uint32_t full_leader = pair_stage_arrive(smem_u32(&bars->full[s]), rank, 2 * (kBytesA + kBytesB));
          tma_load_2d_pair(a_ring + s * kBytesA, &tmWmn, full_leader, k0, kc * kBK);
          tma_load_2d_pair(a_ring + s * kBytesA + 8192, &tmWmn, full_leader, k0 + 64, kc * kBK);
          tma_load_2d_pair(b_ring + s * kBytesB, &tmG, full_leader, kc * kBK, cb * 256 + rank * 128);
        }
      }
    }
  } else if (warp == 1) {
   if (rank == 0) {
    constexpr uint32_t idesc = make_idesc(256, kBN, 1, 0, kFmtF16, kFmtF16);
    uint32_t it = 0, ic = 0;
    for (int item = pair; item < nitems; item += npairs, ++ic) {
      const uint32_t acc = ic & 1, accph = (ic >> 1) & 1;
      mbar_wait(smem_u32(&bars->tmem_empty[acc]), accph ^ 1);
      tc_fence_after();
      for (int kc = 0; kc < nk; ++kc, ++it) {
        const uint32_t s = it % kStages, ph = (it / kStages) & 1;
        mbar_wait(smem_u32(&bars->full[s]), ph);
        tc_fence_after();
        if (lane == 0) {
          // A = W^T (MN-major), B = g (K-major)
          mma_kchunk<true, true, false>(tmem_base + acc * kBN, a_ring + s * kBytesA, b_ring + s * kBytesB, idesc, kc != 0);
          umma_commit_pair(smem_u32(&bars->empty[s]), 3);
        }
        __syncwarp();
      }
      if (lane == 0) umma_commit_pair(smem_u32(&bars->tmem_full[acc]), 3);
      __syncwarp();
    }
   }
  } else {
    const int lane_grp = warp & 3;
    const int eset = (warp - 2) >> 2;
    const int krow = lane_grp * 32 + lane;      // hidden unit within the block = TMEM lane
    const float inv_s = __ldg(p.gscale + 1);
    // vector paths for the T-contiguous layouts (api.cu guarantees 16-byte aligned bases)
    const bool enc_vec = p.enc_st == 1 && p.enc_sh != 1 && ((p.enc_sh | p.enc_sb) & 3) == 0;
    const bool denc_vec = p.denc_st == 1 && p.denc_sh != 1 && ((p.denc_sh | p.denc_sb) & 3) == 0;
    uint32_t ic = 0;
    for (int item = pair; item < nitems; item += npairs, ++ic) {
      const int cb = item / nhb, hb = item % nhb;
      const int k = hb * 256 + rank * 128 + krow;
      const bool k_ok = k < p.H;
      const int kk = k_ok ? k : 0;
      const uint32_t acc = ic & 1, accph = (ic >> 1) & 1;
      mbar_wait(smem_u32(&bars->tmem_full[acc]), accph);
      tc_fence_after();
#pragma unroll 1
      for (int hs = eset * (4 / kEpiSets); hs < (eset + 1) * (4 / kEpiSets); ++hs) {   // this set's half-tiles of the item
        const int slot = p.slot_begin + cb * 4 + hs;
        if (slot >= slot_end) break;            // uniform
        const TileCoord tc = decode_half(p.tile_off, p.T_len, p.U_len, p.B, p.T, p.U1, __ldg(p.sub_list + slot));
        float pv[4], su[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          pv[j] = __ldg(p.pred + tc.b * p.pred_sb + static_cast<long long>(min(tc.u0 + j, p.U1 - 1)) * p.pred_su + kk);
          su[j] = 0.f;
        }
        const float* e_base = p.enc + tc.b * p.enc_sb + static_cast<long long>(kk) * p.enc_sh;
#pragma unroll 1
        for (int q = 0; q < 2; ++q) {           // 32 columns = t-rows 8q .. 8q+7 x 4 u
          float v[32];
          tmem_ld32(tmem_lane_addr(tmem_base, lane_grp, acc * kBN + hs * 64 + q * 32), v);
          const int tb = tc.t0 + q * 8;         // first of this thread's 8 frames
          float ev[8];
          if (enc_vec && tb + 7 < p.T) {        // T-contiguous encoder view: the 8 frames are 32 contiguous bytes
            const float4 a0 = __ldg(reinterpret_cast<const float4*>(e_base + tb));
            const float4 a1 = __ldg(reinterpret_cast<const float4*>(e_base + tb) + 1);
            ev[0] = a0.x; ev[1] = a0.y; ev[2] = a0.z; ev[3] = a0.w; ev[4] = a1.x; ev[5] = a1.y; ev[6] = a1.z; ev[7] = a1.w;
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) ev[i] = __ldg(e_base + static_cast<long long>(min(tb + i, p.T - 1)) * p.enc_st);
          }
          tmem_ld_wait();
          float st[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            st[i] = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float h = tanh_approx(ev[i] + pv[j]);
              const float dz = v[i * 4 + j] * fmaf(-h, h, 1.f);
              st[i] += dz;
              su[j] += dz;
            }
          }
          if (k_ok) {
            if (p.d_enc_fx) {
              long long* dst = p.d_enc_fx + (static_cast<long long>(tc.b) * p.T + tb) * p.H + k;
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (tb + i < tc.Tb) fx_add(dst + static_cast<long long>(i) * p.H, st[i]);
            } else {
              float* dst = p.d_enc + tc.b * p.denc_sb + static_cast<long long>(k) * p.denc_sh;
              if (denc_vec && tb + 7 < tc.Tb) {   // gradient in the encoder's own (B,H,T) layout: two 16-byte reductions
                red_add_v4(dst + tb, st[0] * inv_s, st[1] * inv_s, st[2] * inv_s, st[3] * inv_s);
                red_add_v4(dst + tb + 4, st[4] * inv_s, st[5] * inv_s, st[6] * inv_s, st[7] * inv_s);
              } else {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                  if (tb + i < tc.Tb) atomicAdd(dst + static_cast<long long>(tb + i) * p.denc_st, st[i] * inv_s);
              }
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int u = tc.u0 + j;
          if (k_ok && u <= tc.Ub) {
            const long long o = (static_cast<long long>(tc.b) * p.U1 + u) * p.H + k;
            if (p.d_pred_fx) fx_add(p.d_pred_fx + o, su[j]);
            else atomicAdd(p.d_pred + o, su[j] * inv_s);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&bars->tmem_empty[acc]), 0));
    }
  }

  tmem_teardown<true>(warp, tmem_base, kTmemCols);
}

}  // namespace

int launch_dh_gemm(const CUtensorMap& tmG, const CUtensorMap& tmWmn, const DhArgs& args, long long chunk_slots,
                   cudaStream_t stream) {
  ProfScope prof_(kProfDh, stream);
  const size_t smem = SmemLayout::total + kSmemAlign;
  int pairs;
  if (int rc = pair_kernel_setup(reinterpret_cast<const void*>(dh_gemm_kernel), kNumThreads, smem, &pairs)) return rc;
  const long long items = ((chunk_slots + 3) / 4) * ((args.Hp + 255) / 256);
  const int grid = 2 * static_cast<int>(std::max<long long>(1, std::min<long long>(pairs, items)));
  dh_gemm_kernel<<<grid, kNumThreads, smem, stream>>>(tmG, tmWmn, args);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace rb
