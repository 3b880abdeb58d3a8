// Device helpers shared by the persistent decode kernels (greedy: decode_loop.cu, beam search: beam_loop.cu): block
// reductions and LayerNorm, the batched fixed-order GEMV phase with weights resident in shared memory, the grid barrier
// and the conv1 update from the per-symbol tap table.  Every sum runs in a fixed order, so both kernels are
// deterministic and a row's result does not depend on which rows share the batch.
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace rb {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = (threadIdx.x < kThreads / 32) ? red[threadIdx.x] : 0.f;
  if (w == 0) {
    t = warp_sum(t);
    if (l == 0) red[0] = t;
  }
  __syncthreads();
  return red[0];
}

// dst[i] = LayerNorm(src)[i] * w[i] + b[i] over n elements, by the whole CTA (torch: biased variance, eps 1e-5).
// The row is read ONCE (L2 round trip) into registers when it has at most kLnRegs elements per thread; the sums run in
// the same thread-strided order either way.  `src` may have been written by other CTAs in this kernel: L2 loads only.
constexpr int kLnRegs = 8;
__device__ void block_layer_norm(const float* __restrict__ src, const float* __restrict__ w,
                                 const float* __restrict__ b, float* __restrict__ dst, int n, float* red) {
  const bool cached = n <= kLnRegs * kThreads;
  float x[kLnRegs];
  float s = 0.f;
  if (cached) {
#pragma unroll
    for (int q = 0; q < kLnRegs; ++q) {
      const int i = threadIdx.x + q * kThreads;
      x[q] = i < n ? __ldcg(src + i) : 0.f;
    }
#pragma unroll
    for (int q = 0; q < kLnRegs; ++q) if (threadIdx.x + q * kThreads < n) s += x[q];
  } else {
    for (int i = threadIdx.x; i < n; i += kThreads) s += __ldcg(src + i);
  }
  const float mean = block_sum(s, red) / n;
  float q2 = 0.f;
  if (cached) {
#pragma unroll
    for (int q = 0; q < kLnRegs; ++q) if (threadIdx.x + q * kThreads < n) { const float d = x[q] - mean; q2 += d * d; }
  } else {
    for (int i = threadIdx.x; i < n; i += kThreads) { const float d = __ldcg(src + i) - mean; q2 += d * d; }
  }
  const float var = block_sum(q2, red) / n;
  const float rstd = rsqrtf(var + 1e-5f);
  if (cached) {
#pragma unroll
    for (int q = 0; q < kLnRegs; ++q) {
      const int i = threadIdx.x + q * kThreads;
      if (i < n) dst[i] = (x[q] - mean) * rstd * __ldg(w + i) + __ldg(b + i);
    }
  } else {
    for (int i = threadIdx.x; i < n; i += kThreads) dst[i] = (__ldcg(src + i) - mean) * rstd * __ldg(w + i) + __ldg(b + i);
  }
}

__device__ __forceinline__ void cp_async16(float4* smem_dst, const float4* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }

// ---------------------------------------------------------------------------------------------------------------
// Batched GEMV of one phase: out[r, o] = act(bias[o] + W[o, :] . in_r) for the rows r listed in `rows`, o in the
// CTA's own output range [o_lo, o_hi).  in_r is the concatenation of up to two row segments (lengths multiples of 4).
//
// Every weight matrix is split BY OUTPUT over the CTAs and the CTA's slice stays in shared memory for the whole decode
// (14.7 MB of fp32 weights / 148 SMs = 99 KB per SM at H = V = 1024, E = 512), so a step only moves activations.  A warp
// owns groups of kRG rows: lane l accumulates, for each of its rows and up to kOB outputs, the float4 columns
// l, l + 32, ... of the dot products (activations straight from L2 with coalesced 16-byte loads, weights from shared
// memory), then ONE warp transpose-reduce turns the kRG x kOB per-lane partials into totals -- no block barrier, no
// staging buffer, fixed summation order.
constexpr int kRG = 4;    // rows per warp pass
constexpr int kOB = 8;    // outputs per accumulator block
constexpr int kJ = 4;     // float4 columns per lane and row in flight (K = 512 phases: the whole row)

// v[32] per lane -> lane l returns the sum over the warp's lanes of v[l] (31 shuffles instead of 32 x 5).
__device__ __forceinline__ float warp_transpose_reduce(float (&v)[32]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int step = 16; step >= 1; step >>= 1) {
    const bool up = (lane & step) != 0;
#pragma unroll
    for (int j = 0; j < step; ++j) {
      const float send = up ? v[j] : v[j + step];
      const float keep = up ? v[j + step] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, step);
    }
  }
  return v[0];
}

// EPI 0: out[row][o] = bias[o] + dot            (joint logits, linear)
// EPI 1: causal-conv tap accumulation.  The CTA's outputs are "virtual": vo = (o - o_lo) * taps + j is the dot product of
//        tap j of output channel o (row o of the (E, taps*E) weight, columns [j E, (j+1) E)) with the NEW input vector
//        only.  A causal conv of kernel size `taps` at position n is  y_n = gelu(b + sum_j W_j x_{n-taps+1+j}), so the
//        new vector x_n contributes W_j x_n to position n + taps-1 - j: those partial sums live in a per-utterance
//        ring acc[row][taps][E] (zero-initialised = the left zero padding of rnnt/causalconv.py:29).  The newest tap
//        completes position n: out[row][o] = gelu(bias[o] + acc[row][n % taps][o] + dot) and the slot is cleared for
//        position n + taps.  A step therefore reads E instead of taps*E activations per utterance.
// EPI 2: the tap products themselves, no accumulation: out[row][j * E + o] = dot (the conv1 table: rows = symbols).
struct GemvEpi {
  int mode;                 // 0 / 1 / 2 as above
  int taps;                 // EPI 1
  float* acc;               // EPI 1: [B][taps][E]
  const int* npos;          // EPI 1: position counter source: n = npos[row] - 1
  int E;
};

template <bool GELU>
__device__ void gemv_phase(const float* Wslice /* rows o_lo.. of W, shared or global */, const float* __restrict__ bias,
                           int o_lo, int o_hi, int K, int w_ld, const float* src, int src_stride,
                           const int* rows /* optional: list of row ids; none = rows 0 .. nrows-1 */, int nrows,
                           float* __restrict__ out, long long out_stride, GemvEpi epi, float* xstage) {
  if (o_lo >= o_hi) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kWarps = kThreads / 32;
  constexpr int kBuf = kRG * 32 * kJ;       // float4 per staging buffer
  const int K4 = K >> 2;
  const int nchunks = (K4 + 32 * kJ - 1) / (32 * kJ);
  // This warp's two private staging buffers of kRG rows x (32 kJ) float4.  A chunk of a row group's activations travels
  // L2 -> shared memory with cp.async (no registers held while in flight); every lane copies exactly the elements it
  // reads back itself, so the buffers need no intra-warp synchronisation.  The NEXT chunk / row group is requested
  // before the current one is consumed: one exposed L2 round trip per phase instead of one per chunk.
  float4* xs = reinterpret_cast<float4*>(xstage) + warp * (2 * kBuf);
  const int taps = epi.mode != 0 ? epi.taps : 1;
  const int nvirt = (o_hi - o_lo) * taps;
  int g = warp;
  if (g * kRG >= nrows) return;
  auto load_rows = [&](int gg, int (&rid)[kRG]) {
#pragma unroll
    for (int r = 0; r < kRG; ++r) {
      const int ri = min(gg * kRG + r, nrows - 1);                // tail rows repeat the last one
      rid[r] = rows ? __ldcg(rows + ri) : ri;
    }
  };
  // activations are produced by other CTAs during this kernel: they are read through L2 (cp.async.cg), never L1
  auto issue = [&](const int (&rid)[kRG], int c, int buf) {
#pragma unroll
    for (int r = 0; r < kRG; ++r)
#pragma unroll
      for (int j = 0; j < kJ; ++j) {
        const int f = (c * kJ + j) * 32 + lane;
        if (f < K4)
          cp_async16(xs + buf * kBuf + (r * kJ + j) * 32 + lane,
                     reinterpret_cast<const float4*>(src + static_cast<long long>(rid[r]) * src_stride) + f);
      }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  int rid[kRG], rid_next[kRG];
  load_rows(g, rid);
  issue(rid, 0, 0);
  int buf = 0;
  for (; g * kRG < nrows; g += kWarps) {
    const bool has_next = (g + kWarps) * kRG < nrows;
    if (has_next) load_rows(g + kWarps, rid_next);
    for (int vb = 0; vb < nvirt; vb += kOB) {
      float acc[kRG * kOB];
#pragma unroll
      for (int q = 0; q < kRG * kOB; ++q) acc[q] = 0.f;
      // epilogue operand of this lane's (row, output): requested now, its L2 round trip hides under the FMAs
      const int er = lane / kOB, evo = vb + lane % kOB;
      const bool e_ok = g * kRG + er < nrows && evo < nvirt;
      int erow = rid[0];
#pragma unroll
      for (int r = 1; r < kRG; ++r) erow = (er == r) ? rid[r] : erow;
      float* slot = nullptr;
      float prev = 0.f;
      // (the grid barrier's fences drop the L1 lines, so even the bias is an L2 access once per phase and block)
      const float bias_v = (e_ok && bias) ? __ldg(bias + o_lo + evo / taps) : 0.f;
      if (epi.mode == 1 && e_ok) {
        const int n = __ldcg(epi.npos + erow) - 1;               // position of the new input vector
        slot = epi.acc + (static_cast<long long>(erow) * taps + (n + taps - 1 - evo % taps) % taps) * epi.E + o_lo + evo / taps;
        prev = __ldcg(slot);                                     // only this CTA ever touches (row, *, o)
      }
      for (int c = 0; c < nchunks; ++c) {
        // a new staging buffer becomes current: per chunk when a row spans several chunks (then every output block
        // re-stages), else once per row group; request its successor first, then wait for the current one only
        if (nchunks > 1 || vb == 0) {
          bool pf = true;
          if (nchunks > 1 && c + 1 < nchunks) issue(rid, c + 1, buf ^ 1);
          else if (nchunks > 1 && vb + kOB < nvirt) issue(rid, 0, buf ^ 1);
          else if (has_next) issue(rid_next, 0, buf ^ 1);
          else pf = false;
          if (pf) asm volatile("cp.async.wait_group 1;" ::: "memory");
          else asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        const int f0 = c * 32 * kJ;
        float4 x[kRG][kJ];        // (live inside one output block only: kept across blocks, ptxas spills 4 KB)
#pragma unroll
        for (int r = 0; r < kRG; ++r)
#pragma unroll
          for (int j = 0; j < kJ; ++j) {
            const int f = f0 + j * 32 + lane;
            x[r][j] = f < K4 ? xs[buf * kBuf + (r * kJ + j) * 32 + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
        for (int o = 0; o < kOB; ++o) {
          const int vo = vb + o;
          if (vo < nvirt) {         // uniform
            // virtual output vo -> weight row (vo / taps) of the slice, column block (vo % taps) * K
            const float4* w4 = reinterpret_cast<const float4*>(Wslice + static_cast<long long>(vo / taps) * w_ld +
                                                               static_cast<long long>(vo % taps) * K);
#pragma unroll
            for (int j = 0; j < kJ; ++j) {
              const int f = f0 + j * 32 + lane;
              if (f < K4) {
                const float4 w = w4[f];
#pragma unroll
                for (int r = 0; r < kRG; ++r) {
                  float a = acc[r * kOB + o];
                  a = fmaf(w.x, x[r][j].x, a); a = fmaf(w.y, x[r][j].y, a);
                  a = fmaf(w.z, x[r][j].z, a); a = fmaf(w.w, x[r][j].w, a);
                  acc[r * kOB + o] = a;
                }
              }
            }
          }
        }
        if (nchunks > 1) buf ^= 1;
      }
      const float tot = warp_transpose_reduce(acc);     // lane l: total of partial l = (row l / kOB, output l % kOB)
      if (e_ok) {
        const int o = o_lo + evo / taps;
        if (epi.mode == 0) {
          float v = tot + bias_v;
          if (GELU) v = gelu_erf(v);
          out[erow * out_stride + o] = v;
        } else if (epi.mode == 2) {
          out[erow * out_stride + static_cast<long long>(evo % taps) * epi.E + o] = tot;
        } else if (evo % taps == taps - 1) {                     // newest tap: position n is complete
          float v = prev + tot + bias_v;
          if (GELU) v = gelu_erf(v);
          out[erow * out_stride + o] = v;
          *slot = 0.f;                                           // the slot next collects position n + taps
        } else {
          *slot = prev + tot;
        }
      }
    }
    if (nchunks == 1) buf ^= 1;
#pragma unroll
    for (int r = 0; r < kRG; ++r) rid[r] = rid_next[r];
  }
}

// Grid-wide barrier: cooperative_groups' grid.sync().  Measured on 148 CTAs x 256 threads (scripts/barrier_probe.cu):
// grid.sync 1.21 us, one-counter atomicAdd + acquire spin 1.34 us, 16 spread counters + top counter 1.76 us, per-CTA
// flags gathered by CTA 0 2.02 us -- so the library primitive stays.  (Its fences also drop the SM's L1 lines.)
__device__ __forceinline__ void grid_barrier(unsigned*, unsigned&) { cg::this_grid().sync(); }

// conv1 (kernel size 3) for ONE predictor state whose newest symbol sits at position n, by the whole CTA: tap j of the
// symbol's table row `trow` (3E floats) lands in the accumulator of position n + 2 - j; the newest tap completes position
// n (bias b1 + GELU -> ynew) and clears its slot for position n + 3.  Same arithmetic, in the same order, as the
// tap-accumulating GEMV epilogue (EPI 1) that conv2 uses.  acc / trow are written by other CTAs in other steps: L2 loads
// only.
__device__ __forceinline__ void conv1_update(const float* trow, float* acc, const float* __restrict__ b1,
                                             float* __restrict__ ynew, int E, int n) {
  float* slot[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) slot[j] = acc + ((n + 2 - j) % 3) * E;
  for (int o0 = threadIdx.x; o0 < E; o0 += 2 * kThreads) {
    // all twelve L2 loads of this thread's two channels are in flight before the first store
    float a[2][3], t[2][3], bb[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int o = min(o0 + q * kThreads, E - 1);
      bb[q] = __ldg(b1 + o);
#pragma unroll
      for (int j = 0; j < 3; ++j) { a[q][j] = __ldcg(slot[j] + o); t[q][j] = __ldcg(trow + j * E + o); }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int o = o0 + q * kThreads;
      if (o < E) {
        slot[0][o] = a[q][0] + t[q][0];
        slot[1][o] = a[q][1] + t[q][1];
        ynew[o] = gelu_erf(a[q][2] + t[q][2] + bb[q]);
        slot[2][o] = 0.f;
      }
    }
  }
}

// ---- host side

inline size_t pad4(size_t n) { return (n + 3) & ~static_cast<size_t>(3); }
constexpr size_t kTimerBytes = 128;
constexpr size_t kBarBytes = 128;      // reserved (a counter line for a hand-rolled grid barrier; grid.sync is used)

// Dynamic shared memory of a decode kernel on `grid` CTAs: the resident weight slices, then the per-warp GEMV staging
// buffers (*weight_floats floats of weights first).  Weight residency: each CTA keeps its output slice of a matrix in
// shared memory if it fits the budget, in the order joint (read every step), conv2, conv1, linear; whatever does not
// fit is streamed from L2 every step instead.  Bit i of *resident: matrix i is resident.
inline size_t decode_smem_plan(int grid, int H, int V, int E, int* resident, int* weight_floats) {
  const size_t xstage_bytes = 2 * static_cast<size_t>(kThreads / 32) * kRG * 32 * kJ * sizeof(float4);   // 2 x 64 KB
  const size_t budget = 220 * 1024 - xstage_bytes;
  auto per = [&](int n) { return static_cast<size_t>((n + grid - 1) / grid); };
  const size_t need[4] = {per(V) * H * 4, per(E) * 5 * E * 4, per(E) * 3 * E * 4, per(H) * E * 4};
  size_t smem = 0;
  *resident = 0;
  for (int i = 0; i < 4; ++i) {
    if (i == 2) continue;    // conv1's weights are only read once, for the tap table at kernel start
    if (smem + need[i] <= budget) { smem += need[i]; *resident |= 1 << i; }
  }
  *weight_floats = static_cast<int>(smem / sizeof(float));
  return smem + xstage_bytes;
}

}  // namespace
}  // namespace rb
