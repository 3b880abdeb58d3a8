// Whole batched greedy decode as ONE persistent cooperative kernel (fp32 throughout).
//
// Replaces the host-driven loop of rnnt/model.py:90-128 (`_greedy_decode_conv`): per step
//   joint.single_forward(audio[:, t], pred[:, -1])  (joint.py:44-55)  -> argmax -> blank / 10-emit rule -> append
//   -> ConvPredictor re-run (predictor.py:209-229, model.py:119-123)
// for a whole batch, with every piece of loop state on the device and no host round trip.  The predictor is
// evaluated incrementally: it is causal with a 7-token receptive field, so per utterance the last 2 layer-normed
// embeddings (conv1, k=3) and the last 4 conv1 outputs (conv2, k=5) are kept and one new position is computed per
// emitted token; zero-initialised state is the left zero padding of rnnt/causalconv.py:29.
//
// One CTA per SM, 256 threads, phases separated by grid-wide barriers (the kernel's own counter barrier; the launch is
// cooperative so that all CTAs are co-resident).  Every weight matrix is split by output over the CTAs and each CTA's
// slice lives in shared memory for the whole decode, so a step only moves activations:
//   P1  feats = LayerNorm(lin) for utterances that just emitted; h = tanh(enc[b, t_b] + feats[b])
//   P2  logits[b, v] = W_j[v,:] . h[b,:] + b_j[v]        (CTA = its ~V/148 classes, warp = 4 rows, lanes split K; gemv_phase)
//   P3  argmax (lowest index on ties) + top-2 margin, blank / max-per-frame rule, token append
//       conv1 of an emitted token, inside P3: its tap products W1_j . LN(emb[tok]) depend on the token alone, so they are a
//       (symbols, 3E) TABLE built once at kernel start (1.6 GFLOP, ~3 decode steps' worth) -- the step adds three table
//       rows to the utterance's tap accumulators and applies bias + GELU: no GEMV phase, no grid barrier for conv1
//   P5  z = gelu(conv2) from the tap products of the new conv1 output   P6  lin = linear(z)
// P5-P6 only run in steps where some utterance emitted.  Every dot product is accumulated in a fixed order (thread-
// strided partial sums, then one fixed warp butterfly), so results are deterministic.
//
// Streaming: the per-slot loop state (predictor accumulators, lin / feats, token count, emit flag) and the symbol tables
// live in a caller-owned state buffer, so one launch can continue every slot where the previous one stopped.  A launch
// optionally builds the tables (init), seeds the slots being reset and consumes each slot's frames of this chunk.  The
// one-shot decode is the launch that does all three for every slot; there is one step loop for both.
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"
#include "kernels.h"

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

// per-thread (best, second, index) -> block-wide argmax with lowest index on ties; result in s_*[0]
__device__ __forceinline__ void block_argmax(float best, float second, int idx, float* s_best, float* s_second, int* s_idx) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  auto merge = [&](float b2, float s2, int i2) {
    if (b2 > best || (b2 == best && i2 < idx)) { second = fmaxf(best, s2); best = b2; idx = i2; }
    else second = fmaxf(second, b2);
  };
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const float b2 = __shfl_xor_sync(0xffffffffu, best, o), s2 = __shfl_xor_sync(0xffffffffu, second, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
    merge(b2, s2, i2);
  }
  __syncthreads();
  if (lane == 0) { s_best[warp] = best; s_second[warp] = second; s_idx[warp] = idx; }
  __syncthreads();
  if (warp == 0) {
    const bool have = lane < kThreads / 32;
    best = have ? s_best[lane] : -INFINITY; second = have ? s_second[lane] : -INFINITY; idx = have ? s_idx[lane] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float b2 = __shfl_xor_sync(0xffffffffu, best, o), s2 = __shfl_xor_sync(0xffffffffu, second, o);
      const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
      merge(b2, s2, i2);
    }
    if (lane == 0) { s_best[0] = best; s_second[0] = second; s_idx[0] = idx; }
  }
  __syncthreads();
}

// conv1 (kernel size 3) for ONE utterance whose newest symbol `tok` sits at position n, by the whole CTA: tap j of the
// symbol's table row lands in the accumulator of position n + 2 - j; the newest tap completes position n (bias + GELU ->
// ynew) and clears its slot for position n + 3.  Same arithmetic, in the same order, as the tap-accumulating GEMV
// epilogue (EPI 1) that conv2 uses.  acc1 / t1 are written by other CTAs in other steps: L2 loads only.
__device__ __forceinline__ void conv1_update(const DecodeArgs& p, int b, int tok, int n) {
  const int E = p.E;
  const float* trow = p.t1 + static_cast<long long>(tok) * 3 * E;
  float* acc = p.acc1 + static_cast<long long>(b) * 3 * E;
  float* slot[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) slot[j] = acc + ((n + 2 - j) % 3) * E;
  for (int o0 = threadIdx.x; o0 < E; o0 += 2 * kThreads) {
    // all twelve L2 loads of this thread's two channels are in flight before the first store
    float a[2][3], t[2][3], bb[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int o = min(o0 + q * kThreads, E - 1);
      bb[q] = __ldg(p.b1 + o);
#pragma unroll
      for (int j = 0; j < 3; ++j) { a[q][j] = __ldcg(slot[j] + o); t[q][j] = __ldcg(trow + j * E + o); }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int o = o0 + q * kThreads;
      if (o < E) {
        slot[0][o] = a[q][0] + t[q][0];
        slot[1][o] = a[q][1] + t[q][1];
        p.ynew[static_cast<long long>(b) * E + o] = gelu_erf(a[q][2] + t[q][2] + bb[q]);
        slot[2][o] = 0.f;
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads, 1) greedy_decode_kernel(DecodeArgs p) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float red[kThreads / 32];
  __shared__ float s_best[kThreads / 32];
  __shared__ float s_second[kThreads / 32];
  __shared__ int s_idx[kThreads / 32];
  const int B = p.B, H = p.H, V = p.V, E = p.E;
  const int tid = threadIdx.x;
  const int G = gridDim.x, cta = blockIdx.x;
  int* rows_act = p.rows;          // compacted list of active utterances (P2) ...
  int* rows_emit = p.rows + B;     // ... and of utterances that emitted in this step (P4-P6)
  int* counts = p.flags;           // [0] n_active, [1] n_emit, [2] n_active_next
  unsigned* bar_counter = p.bar;   // zeroed by the launcher
  unsigned bar_target = 0;         // number of barriers passed so far
  const bool timer = (cta == 0 && tid == 0 && p.prof != nullptr);
  long long tmark = timer ? clock64() : 0;
  auto lap = [&](int slot) { if (timer) { const long long now = clock64(); p.prof[slot] += now - tmark; tmark = now; } };
  if (timer) for (int i = 0; i < 8; ++i) p.prof[i] = 0;

  // ---- this CTA's output slices of the four weight matrices; resident in shared memory where the launcher found room
  const int perJ = (V + G - 1) / G, perE = (E + G - 1) / G, perL = (H + G - 1) / G;
  const int j_lo = min(V, cta * perJ), j_hi = min(V, j_lo + perJ);
  const int e_lo = min(E, cta * perE), e_hi = min(E, e_lo + perE);
  const int l_lo = min(H, cta * perL), l_hi = min(H, l_lo + perL);
  const float* Wj_s = p.Wj + static_cast<long long>(j_lo) * H;
  const float* w1_s = p.w1 + static_cast<long long>(e_lo) * 3 * E;
  const float* w2_s = p.w2 + static_cast<long long>(e_lo) * 5 * E;
  const float* wl_s = p.wl + static_cast<long long>(l_lo) * E;
  float* xstage = nullptr;     // per-warp activation staging buffers, after the resident weight slices
  {
    // fixed offsets (every CTA reserves per* rows, so the residency decision is the launcher's alone)
    const long long off_j = 0;
    const long long off_2 = off_j + ((p.resident & 1) ? static_cast<long long>(perJ) * H : 0);
    const long long off_1 = off_2 + ((p.resident & 2) ? static_cast<long long>(perE) * 5 * E : 0);
    const long long off_l = off_1 + ((p.resident & 4) ? static_cast<long long>(perE) * 3 * E : 0);
    auto stage = [&](const float*& w, int nrows, int K, bool resident, long long off) {
      if (!resident) return;
      const float4* src = reinterpret_cast<const float4*>(w);
      float4* d4 = reinterpret_cast<float4*>(smem + off);
      for (int i = tid; i < nrows * (K >> 2); i += kThreads) d4[i] = __ldg(src + i);
      w = smem + off;
    };
    xstage = smem + p.weight_floats;
    stage(Wj_s, j_hi - j_lo, H, p.resident & 1, off_j);
    stage(w2_s, e_hi - e_lo, 5 * E, p.resident & 2, off_2);
    stage(w1_s, e_hi - e_lo, 3 * E, p.resident & 4, off_1);
    stage(wl_s, l_hi - l_lo, E, p.resident & 8, off_l);
  }

  // A slot joins a step while it is live (ntok >= 1), not finished and has frames of this launch left.  Between launches
  // a slot's state sits on a frame boundary: a frame is only left after a blank or the per-frame cap (per = 0), and a
  // slot that finishes mid-frame stays finished until it is reset.  So t_idx and per restart at 0 every launch.
  auto is_reset = [&](int b) { return p.reset_all || (p.reset != nullptr && __ldg(p.reset + b) != 0); };
  auto is_active = [&](int b) {
    const int nt = __ldcg(p.ntok + b);
    return nt >= 1 && nt < p.max_len && __ldcg(p.t_idx + b) < min(__ldg(p.T_len + b), p.T);
  };

  // ---- per launch: frame counters = 0; reset slots get zero conv tap accumulators (the left zero padding), ntok = 1 and
  // "emit" the seed blank so the predictor runs once; init empties the other slots
  if (cta == 0 && tid < 32) {
    int n = 0;
    for (int b0 = 0; b0 < B; b0 += 32) {
      const int b = b0 + tid;
      const bool r = b < B && is_reset(b);
      if (b < B) {
        p.t_idx[b] = 0; p.per[b] = 0;
        if (r) { p.ntok[b] = 1; p.emit[b] = 1; p.last_tok[b] = p.blank; }
        else if (p.init) { p.ntok[b] = 0; p.emit[b] = 0; }
      }
      const unsigned m = __ballot_sync(0xffffffffu, r);
      if (r) rows_emit[n + __popc(m & ((1u << tid) - 1))] = b;
      n += __popc(m);
    }
    if (tid == 0) { counts[0] = 0; counts[1] = n; counts[2] = 0; }
  }
  for (int b = cta; b < B; b += G) {
    if (!is_reset(b)) continue;
    for (int i = tid; i < 3 * E; i += kThreads) p.acc1[static_cast<long long>(b) * 3 * E + i] = 0.f;
    for (int i = tid; i < 5 * E; i += kThreads) p.acc2[static_cast<long long>(b) * 5 * E + i] = 0.f;
  }
  if (p.init) {
    // ---- LayerNorm(embedding) table for every symbol
    for (int v = cta; v < p.NS; v += G)
      block_layer_norm(p.emb + static_cast<long long>(v) * E, p.ln1_w, p.ln1_b, p.emb_ln + static_cast<long long>(v) * E, E, red);
    grid_barrier(bar_counter, bar_target);
    // ---- conv1 tap table: t1[v][j][o] = W1_j[o, :] . LN(emb[v]) for every symbol v (this CTA's output channels)
    {
      GemvEpi epi{2, 3, nullptr, nullptr, E};
      gemv_phase<false>(w1_s, nullptr, e_lo, e_hi, E, 3 * E, p.emb_ln, E, nullptr, p.NS, p.t1, 3 * E, epi, xstage);
    }
    lap(3);
    grid_barrier(bar_counter, bar_target);
  } else {
    __syncthreads();            // this CTA's zeroed accumulators before its own seed updates
  }
  // ---- the seed blank at position 0 of every reset slot
  for (int b = cta; b < B; b += G)
    if (is_reset(b)) conv1_update(p, b, p.blank, 0);
  grid_barrier(bar_counter, bar_target);
  lap(7);

  for (int step = 0;; ++step) {
    const int n_emit = __ldcg(counts + 1);
    if (n_emit > 0) {
      // ---- P5: conv2, tap products of the new conv1 output
      {
        GemvEpi epi{1, 5, p.acc2, p.ntok, E};
        gemv_phase<true>(w2_s, p.b2, e_lo, e_hi, E, 5 * E, p.ynew, E, rows_emit, n_emit, p.z, E, epi, xstage);
      }
      lap(4);
      grid_barrier(bar_counter, bar_target);
      lap(7);
      // ---- P6: linear
      {
        GemvEpi epi{0, 1, nullptr, nullptr, E};
        gemv_phase<false>(wl_s, p.bl, l_lo, l_hi, E, E, p.z, E, rows_emit, n_emit, p.lin, H, epi, xstage);
      }
      lap(5);
      grid_barrier(bar_counter, bar_target);
      lap(7);
    }
    if (step >= p.max_steps) break;

    // ---- P1: refresh predictor features where a token was emitted; joint hidden rows for active utterances
    for (int b = cta; b < B; b += G) {
      if (__ldcg(p.emit + b)) block_layer_norm(p.lin + static_cast<long long>(b) * H, p.ln2_w, p.ln2_b, p.feats + static_cast<long long>(b) * H, H, red);
      __syncthreads();
      if (is_active(b)) {
        const int t = __ldcg(p.t_idx + b);
        const float* e = p.enc + b * p.enc_sb + static_cast<long long>(t) * p.enc_st;
        for (int i = tid; i < H; i += kThreads) p.hbuf[static_cast<long long>(b) * H + i] = tanhf(__ldg(e + i) + p.feats[static_cast<long long>(b) * H + i]);
      }
    }
    if (cta == G - 1) {
      // compact the active list (single warp, order preserved); the last CTA has no utterance of its own when B < G
      if (tid < 32) {
        int n = 0;
        for (int b0 = 0; b0 < B; b0 += 32) {
          const int b = b0 + tid;
          const bool a = b < B && is_active(b);
          const unsigned m = __ballot_sync(0xffffffffu, a);
          if (a) rows_act[n + __popc(m & ((1u << tid) - 1))] = b;
          n += __popc(m);
        }
        if (tid == 0) { counts[0] = n; counts[1] = 0; counts[2] = 0; }
      }
    }
    lap(0);
    grid_barrier(bar_counter, bar_target);
    lap(7);
    const int n_act = __ldcg(counts + 0);
    if (n_act == 0) break;
    if (timer) p.prof[6] += 1;      // joint steps taken (slot 6 of the phase counters)

    // ---- P2: joint logits for the active rows
    {
      GemvEpi epi{0, 1, nullptr, nullptr, E};
      gemv_phase<false>(Wj_s, p.bj, j_lo, j_hi, H, H, p.hbuf, H, rows_act, n_act, p.logits, V, epi, xstage);
    }
    lap(1);
    grid_barrier(bar_counter, bar_target);
    lap(7);

    // ---- P3: argmax + decode rule + embedding layer norm, one CTA per active utterance
    for (int j = cta; j < n_act; j += G) {
      const int b = __ldcg(rows_act + j);
      const float* row = p.logits + static_cast<long long>(b) * V;
      float best = -INFINITY, second = -INFINITY;
      int idx = 0x7fffffff;
      for (int v = tid; v < V; v += kThreads) {
        const float x = __ldcg(row + v);
        if (x > best) { second = best; best = x; idx = v; }
        else if (x > second) second = x;
      }
      block_argmax(best, second, idx, s_best, s_second, s_idx);
      // torch.argmax always returns an in-range index; a row without any finite maximum (all NaN / -inf) maps to 0
      const int tok = static_cast<unsigned>(s_idx[0]) < static_cast<unsigned>(V) ? s_idx[0] : 0;
      const bool advance = (tok == p.blank) || (__ldcg(p.per + b) >= p.max_per_frame);
      const int nt_old = __ldcg(p.ntok + b);        // every thread reads it before thread 0 bumps it
      __syncthreads();
      if (tid == 0) {
        if (p.margins) p.margins[static_cast<long long>(step) * B + b] = s_best[0] - s_second[0];
        if (advance) {
          p.t_idx[b] = __ldcg(p.t_idx + b) + 1; p.per[b] = 0; p.emit[b] = 0;
        } else {
          const int nt = __ldcg(p.ntok + b);
          p.tokens[static_cast<long long>(b) * p.max_len + nt - 1] = tok;
          p.ntok[b] = nt + 1; p.per[b] = __ldcg(p.per + b) + 1; p.emit[b] = 1; p.last_tok[b] = tok;
          rows_emit[atomicAdd(&counts[1], 1)] = b;
        }
      }
      if (!advance) conv1_update(p, b, tok, nt_old);   // the new symbol's position in the predictor's input = old ntok
      __syncthreads();
    }
    // (a finished utterance may keep emit = 1; P1 then recomputes the same feats from an unchanged lin -- harmless)
    lap(2);
    grid_barrier(bar_counter, bar_target);
    lap(7);
  }
  // every exit of the loop follows a grid barrier, so all ntok updates are visible here
  if (cta == 0 && p.n_tokens != nullptr)
    for (int b = tid; b < B; b += kThreads) p.n_tokens[b] = __ldcg(p.ntok + b);
}

}  // namespace

// State / scratch layout: [8 x int64 phase timers | barrier line | float regions, each padded to a multiple of 4 floats
// so that every region starts 16-byte aligned whatever B, V, E are (cp.async / float4 need it) | int regions].  The
// one-shot decode and the streaming decoder share it (include/rnnt_b200.h lists what persists between launches).
namespace {
inline size_t pad4(size_t n) { return (n + 3) & ~static_cast<size_t>(3); }
constexpr size_t kTimerBytes = 128;
constexpr size_t kBarBytes = 128;      // reserved (a counter line for a hand-rolled grid barrier; grid.sync is used)
}  // namespace

size_t greedy_decode_scratch_bytes(int B, int H, int V, int E) {
  const size_t b = static_cast<size_t>(B);
  const size_t floats = 3 * pad4(b * H) /*feats, hbuf, lin*/ + pad4(b * V) /*logits*/ + pad4(b * 3 * E) + pad4(b * 5 * E) +
                        2 * pad4(b * E) /*ynew, z*/ + pad4(static_cast<size_t>(V) * E) /*LayerNorm(embedding) table*/ +
                        pad4(static_cast<size_t>(V) * 3 * E) /*conv1 tap table*/;
  const size_t ints = b * 7 + 16;
  return kTimerBytes + kBarBytes + floats * 4 + ints * 4 + 256;
}

int launch_greedy_decode(DecodeArgs a, float* scratch, cudaStream_t stream) {
  ProfScope prof_(kProfOther, stream);
  RB_REQUIRE(a.B > 0 && a.H > 0 && a.V > 1 && a.E > 0 && a.max_len >= 1, -1, "invalid decode shape");
  RB_REQUIRE(a.H % 4 == 0 && a.E % 4 == 0, -2, "decode kernel needs hidden / embedding sizes that are multiples of 4");
  const int grid = device_sm_count();
  // Weight residency: each CTA keeps its output slice of a matrix in shared memory if it fits the budget, in the order
  // joint (read every step), conv2, conv1, linear; whatever does not fit is streamed from L2 every step instead.
  const size_t xstage_bytes = 2 * static_cast<size_t>(kThreads / 32) * kRG * 32 * kJ * sizeof(float4);   // 2 x 64 KB
  const size_t budget = 220 * 1024 - xstage_bytes;
  auto per = [&](int n) { return static_cast<size_t>((n + grid - 1) / grid); };
  const size_t need[4] = {per(a.V) * a.H * 4, per(a.E) * 5 * a.E * 4, per(a.E) * 3 * a.E * 4, per(a.H) * a.E * 4};
  size_t smem = 0;
  a.resident = 0;
  for (int i = 0; i < 4; ++i) {
    if (i == 2) continue;    // conv1's weights are only read once, for the tap table at kernel start
    if (smem + need[i] <= budget) { smem += need[i]; a.resident |= 1 << i; }
  }
  a.weight_floats = static_cast<int>(smem / sizeof(float));
  smem += xstage_bytes;
  // carve the scratch
  RB_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, -3, "decode scratch must be 16-byte aligned");
  RB_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 127) == 0, -3, "decode scratch must be 128-byte aligned");
  a.prof = reinterpret_cast<long long*>(scratch);          // 8 x int64 at the (aligned) start
  a.bar = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(scratch) + kTimerBytes);
  RB_CUDA_CHECK(cudaMemsetAsync(a.bar, 0, kBarBytes, stream));
  float* f = scratch + (kTimerBytes + kBarBytes) / sizeof(float);
  const int B = a.B, H = a.H, V = a.V, E = a.E;
  const size_t b = static_cast<size_t>(B);
  a.feats = f; f += pad4(b * H);
  a.hbuf = f; f += pad4(b * H);
  a.logits = f; f += pad4(b * V);
  a.acc1 = f; f += pad4(b * 3 * E);
  a.acc2 = f; f += pad4(b * 5 * E);
  a.ynew = f; f += pad4(b * E);
  a.z = f; f += pad4(b * E);
  a.lin = f; f += pad4(b * H);
  a.emb_ln = f; f += pad4(static_cast<size_t>(a.NS) * E);
  a.t1 = f; f += pad4(static_cast<size_t>(a.NS) * 3 * E);
  int* ip = reinterpret_cast<int*>(f);
  a.ntok = ip; ip += B;
  a.t_idx = ip; ip += B;
  a.per = ip; ip += B;
  a.emit = ip; ip += B;
  a.rows = ip; ip += 2 * B;
  a.last_tok = ip; ip += B;
  a.flags = ip; ip += 16;
  RB_CUDA_CHECK(cudaFuncSetAttribute(greedy_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  RB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, greedy_decode_kernel, kThreads, smem));
  RB_REQUIRE(per_sm >= 1, -6, "decode kernel does not fit on an SM");
  void* args[] = {&a};
  // cooperative launch: guarantees that all CTAs are co-resident, which the kernel's own grid barrier relies on
  RB_CUDA_CHECK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(greedy_decode_kernel), dim3(grid), dim3(kThreads),
                                            args, smem, stream));
  return 0;
}

}  // namespace rb
