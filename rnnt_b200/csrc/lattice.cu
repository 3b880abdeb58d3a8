// Small kernels around the GEMMs: tile table, weight conversion, alpha/beta lattice, gradient coefficients,
// and the dense-logits variants of the loss front/back end (for callers that already hold logits).
//
// Lattice = torchaudio ComputeAlphasBetasCosts (reference call site rnnt/model.py:35-41):
//   alpha[0,0]=0; alpha[t,u]=LSE(alpha[t-1,u]+lpB[t-1,u], alpha[t,u-1]+lpE[t,u-1])
//   beta[Tb-1,Ub]=lpB[Tb-1,Ub]; beta[t,u]=LSE(beta[t+1,u]+lpB[t,u], beta[t,u+1]+lpE[t,u]); cost=-beta[0,0]
// One CTA per (utterance, direction); thread u walks anti-diagonals n = t+u.  The neighbour value crosses
// threads through a double-buffered shared array (one __syncthreads per diagonal, no global spin-waits),
// and the log-probs of the next 8 diagonals are prefetched into registers while the current 8 are consumed.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace rb {
namespace {

// Also derives the exact power-of-two scale S that maps max_b |dcost_b| into [2^(kGradShift-1), 2^kGradShift): the backward
// stores logit-gradients in fp16 as g*S (full use of fp16's range whatever the loss scaling) and its epilogues apply 1/S.
__global__ void tile_table_kernel(const int* __restrict__ T_len, const int* __restrict__ U_len, int B, int T, int U1,
                                  int* __restrict__ tile_off, int* __restrict__ status,
                                  int* __restrict__ err_flag, const float* __restrict__ dcost,
                                  float* __restrict__ gscale) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int acc = 0, bad = 0;
  tile_off[0] = 0;
  if (gscale) {
    float mx = 0.f;
    if (dcost) {
      for (int b = 0; b < B; ++b) mx = fmaxf(mx, fabsf(dcost[b]));
    } else {
      mx = 1.f;
    }
    float S = static_cast<float>(1 << kGradShift);
    if (mx > 0.f && mx < INFINITY) {
      int e;
      frexpf(mx, &e);          // mx = m * 2^e, m in [0.5, 1)
      S = ldexpf(1.f, kGradShift - e);     // mx * S in [2^(kGradShift-1), 2^kGradShift)
    }
    gscale[0] = S;
    gscale[1] = 1.f / S;
  }
  for (int b = 0; b < B; ++b) {
    int Tb = T_len[b], Ub = U_len[b];
    if (Tb < 1 || Tb > T || Ub < 0 || Ub > U1 - 1) bad = 1;
    Tb = max(1, min(Tb, T));
    Ub = max(0, min(Ub, U1 - 1));
    acc += ((Tb + kTileT - 1) / kTileT) * ((Ub + 1 + kHalfU - 1) / kHalfU);     // half-tiles of 16(t) x 4(u)
    tile_off[b + 1] = acc;
  }
  *status = bad;                  // the lattice kernel turns the costs into NaN when it is set
  if (err_flag) *err_flag = bad;
}

// W (V,H) fp32 -> fp16 [Vp,Hp] zero-padded, 8 elements (one 16-byte store) per thread; bias * log2(e) with -1e30 padding.
__global__ void convert_weights_kernel(const float* __restrict__ W, const float* __restrict__ bias, int V, int H,
                                       int Vp, int Hp, __half* __restrict__ Wh, float* __restrict__ bias2) {
  const int hp8 = Hp >> 3;                                   // Hp is a multiple of 64, H a multiple of 8
  const long long n = static_cast<long long>(Vp) * hp8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(i / hp8), k = static_cast<int>(i % hp8) * 8;
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (v < V && k < H) {
      const float4* src = reinterpret_cast<const float4*>(W + static_cast<long long>(v) * H + k);
      const float4 a = __ldg(src), b = __ldg(src + 1);
      o.x = pack_f16x2(a.x, a.y); o.y = pack_f16x2(a.z, a.w);
      o.z = pack_f16x2(b.x, b.y); o.w = pack_f16x2(b.z, b.w);
    }
    reinterpret_cast<uint4*>(Wh)[i] = o;
    if (k == 0) bias2[v] = (v < V) ? bias[v] * kLog2e : -1e30f;
  }
}

// log(exp(a) + exp(b)) on the critical path of the wavefront: two MUFU ops (ex2, lg2; relative error ~2^-22 on a
// term bounded by ln 2) instead of the ~50-instruction expf/log1pf pair.
__device__ __forceinline__ float lse2f(float a, float b) {
  const float m = fmaxf(a, b);
  const float t = a - b;                                   // in parallel with the max; NaN only if both are -inf
  const float r = fmaf(lg2_approx(1.f + ex2_approx(fabsf(t) * -kLog2e)), kLn2, m);   // one operand -inf: exp -> 0, r = m
  return m == -INFINITY ? -INFINITY : r;
}

constexpr int kPre = 8;

// Thread u owns lattice column u.  In step s it sits at t = s - u (alpha) or t = Tb-1 - (s - (Ub - u)) (beta), i.e.
// it is active for the Tb consecutive steps starting at s0 = u (alpha) / Ub - u (beta) and walks its column with a
// constant pointer stride, so the per-step work is: one prefetched float2, one smem read, one LSE, two stores.
template <bool BETA>
__device__ __forceinline__ void lattice_walk(const float2* __restrict__ lp2, float* __restrict__ out,
                                             float* __restrict__ costs_b, int Tb, int Ub, int U1, int u, float* sh0,
                                             float* sh1, bool poison) {
  // The step time of this kernel is (instructions per step) x (dependent-issue latency): one warp per scheduler, no
  // other work to hide behind.  So everything that is not the recursion itself is hoisted out of the step: the
  // activity test is one unsigned compare, the store walks a pointer, the emit log-prob of the last column is -inf
  // already when it is fetched, and the corner cell needs no special case (own = 0, side = -inf gives LSE = 0 / lpB).
  const int ndiag = Tb + Ub;
  const bool col_ok = u <= Ub;
  const int s0 = col_ok ? (BETA ? (Ub - u) : u) : 0x40000000;   // first active step (never, for columns past Ub)
  const long long step = BETA ? -static_cast<long long>(U1) : U1;
  const long long first = (BETA ? static_cast<long long>(Tb - 1) * U1 : 0) + min(u, U1 - 1);
  const float2* src = lp2 + first;                           // cell visited at local step 0
  float* dptr = out + first;
  const int nb = BETA ? u + 1 : u - 1;                       // neighbour column feeding this one
  const bool last_col = u >= Ub;
  // shared-memory addresses of the step, computed once: left to the compiler, every step re-derives them from
  // SR_TID / SR_CgaCtaId (two special-register reads on the dependency chain of the wavefront)
  uint32_t rd_addr[2] = {smem_u32(sh1 + nb), smem_u32(sh0 + nb)};          // step parity 0 reads sh1, writes sh0
  uint32_t wr_addr[2] = {smem_u32(sh0 + u), smem_u32(sh1 + u)};
#pragma unroll
  for (int i = 0; i < 2; ++i) {      // opaque to the compiler, so that it keeps them in registers instead of rematerialising
    asm volatile("mov.u32 %0, %0;" : "+r"(rd_addr[i]));
    asm volatile("mov.u32 %0, %0;" : "+r"(wr_addr[i]));
  }

  float2 cur[kPre], nxt[kPre];
  auto fetch = [&](int g, float2 (&d)[kPre]) {
#pragma unroll
    for (int i = 0; i < kPre; ++i) {
      const int rel = g * kPre + i - s0;
      float2 v = make_float2(0.f, 0.f);
      if (static_cast<unsigned>(rel) < static_cast<unsigned>(Tb)) v = __ldg(src + rel * step);
      if (last_col) v.y = -INFINITY;                         // no emission out of the last column
      d[i] = v;
    }
  };
  const int ngroups = (ndiag + kPre - 1) / kPre;
  fetch(0, cur);
  // alpha: own = alpha(t-1,u)+lpB(t-1,u);  beta: own = beta(t+1,u).  The corner cell starts from own = 0.
  float own = ((BETA ? u == Ub : u == 0)) ? 0.f : -INFINITY;
  float last = 0.f;
  for (int g = 0; g < ngroups; ++g) {
    if (g + 1 < ngroups) fetch(g + 1, nxt);
#pragma unroll
    for (int i = 0; i < kPre; ++i) {
      const int s = g * kPre + i;
      if (s < ndiag) {    // uniform over the block
        // (kPre is even: the parity of s is the parity of i.)  Every thread evaluates the step -- inactive ones on
        // harmless operands -- and only the commit is predicated: no divergent branch on the wavefront's critical path.
        const bool act = static_cast<unsigned>(s - s0) < static_cast<unsigned>(Tb);
        const float lpB = cur[i].x, lpE = cur[i].y;
        float side;                                          // guards hold -inf at columns -1 and blockDim.x
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(side) : "r"(rd_addr[i & 1]) : "memory");
        float val, own_next, pub_next;
        if (!BETA) {
          val = lse2f(own, side);                            // own = -inf at t = 0, side = -inf at u = 0
          own_next = val + lpB;                              // feeds alpha(t+1,u)
          pub_next = val + lpE;                              // feeds alpha(t,u+1); -inf out of the last column
        } else {
          val = lse2f(own + lpB, side + lpE);                // own = -inf at t = Tb-1 except in the corner
          own_next = val;
          pub_next = val;
        }
        if (act) {
          *dptr = val;
          dptr += step;
          own = own_next;
          if (BETA) last = val;
        }
        const float pub = act ? pub_next : -INFINITY;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(wr_addr[i & 1]), "f"(pub) : "memory");
        __syncthreads();
      }
    }
#pragma unroll
    for (int i = 0; i < kPre; ++i) cur[i] = nxt[i];
  }
  // beta(0,0) is the last cell column 0 visits.  An out-of-range length anywhere in the batch (status word of the tile
  // table; torchaudio raises for these) turns every cost into NaN, so the error cannot pass silently without a sync.
  if (BETA && u == 0) *costs_b = poison ? __int_as_float(0x7fc00000) : -last;
}

__global__ void lattice_kernel(const float* __restrict__ lp, const int* __restrict__ T_len,
                               const int* __restrict__ U_len, int T, int U1, float* __restrict__ alpha,
                               float* __restrict__ beta, float* __restrict__ costs, const int* __restrict__ status) {
  extern __shared__ float sh[];   // 2 x (blockDim.x + 2)
  const int b = blockIdx.x;
  const int u = threadIdx.x;
  const int Tb = max(1, min(T_len[b], T)), Ub = max(0, min(U_len[b], U1 - 1));
  const int stride = blockDim.x + 2;
  float* sh0 = sh + 1;             // sh0[-1] and sh0[blockDim.x] are -inf guards
  float* sh1 = sh + stride + 1;
  if (u == 0) {
    sh0[-1] = -INFINITY; sh1[-1] = -INFINITY;
    sh0[blockDim.x] = -INFINITY; sh1[blockDim.x] = -INFINITY;
  }
  sh0[u] = -INFINITY;
  sh1[u] = -INFINITY;
  __syncthreads();
  const long long off = static_cast<long long>(b) * T * U1;
  const float2* lp2 = reinterpret_cast<const float2*>(lp) + off;
  const bool poison = status != nullptr && *status != 0;
  if (blockIdx.y == 1) lattice_walk<true>(lp2, beta + off, costs + b, Tb, Ub, U1, u, sh0, sh1, poison);
  else lattice_walk<false>(lp2, alpha + off, costs + b, Tb, Ub, U1, u, sh0, sh1, poison);
}

__global__ void coef_kernel(const float* __restrict__ lp, const float* __restrict__ lse,
                            const float* __restrict__ alpha, const float* __restrict__ beta,
                            const float* __restrict__ dcost, const float* __restrict__ gscale,
                            const int* __restrict__ T_len, const int* __restrict__ U_len, int B, int T, int U1,
                            float4* __restrict__ coef) {
  const long long n = static_cast<long long>(B) * T * U1;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int u = static_cast<int>(i % U1);
    const int t = static_cast<int>((i / U1) % T);
    const int b = static_cast<int>(i / (static_cast<long long>(U1) * T));
    const int Tb = max(1, min(T_len[b], T)), Ub = max(0, min(U_len[b], U1 - 1));
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < Tb && u <= Ub) {
      const float dc = (dcost ? dcost[b] : 1.f) * (gscale ? gscale[0] : 1.f);
      const float logZ = beta[static_cast<long long>(b) * T * U1];
      const float c = alpha[i] - logZ;
      const float2 l = reinterpret_cast<const float2*>(lp)[i];
      o.x = expf(c + beta[i]) * dc;
      if (t < Tb - 1) o.y = expf(c + l.x + beta[i + U1]) * dc;
      else if (u == Ub) o.y = expf(c + l.x) * dc;
      if (u < Ub) o.z = expf(c + l.y + beta[i + 1]) * dc;
      o.w = lse[i];
    }
    coef[i] = o;
  }
}

// ---- occupancy sparsity of the backward.  The logit-gradients of a cell are bounded by max(|gamma'|,|eB'|,|eE'|)
// (coef already carries dcost * S).  A HALF-TILE (16 t x 4 u = 64 cells) whose cells are all at most 2^-25 of the largest
// possible gradient entry max_b |dcost_b| (kSkipBelow; half the resolution fp32 has for that entry) is dropped from the
// backward's work list: what it would add to dh / dW / db is below the rounding of the terms that dominate them.
// One warp per half-tile, then a single-block compaction (order preserved).  In dense mode (RNNT_B200_ALL_TILES) every
// half-tile that holds at least one valid cell stays.
__global__ void tile_activity_kernel(const float4* __restrict__ coef, const int* __restrict__ T_len,
                                     const int* __restrict__ U_len, const int* __restrict__ tile_off, int B, int T,
                                     int U1, int dense, unsigned char* __restrict__ flags) {
  const int total = __ldg(&tile_off[B]);
  const int lane = threadIdx.x & 31;
  const int w0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nw = (gridDim.x * blockDim.x) >> 5;
  for (int hid = w0; hid < total; hid += nw) {
    const TileCoord tc = decode_half(tile_off, T_len, U_len, B, T, U1, hid);
    float mx = 0.f;
    int any_valid = 0;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int r = lane * 2 + i;
      const int t = tc.t0 + (r >> 2), u = tc.u0 + (r & 3);
      if (t < tc.Tb && u <= tc.Ub) {
        const float4 c = __ldg(coef + (static_cast<long long>(tc.b) * T + t) * U1 + u);
        mx = fmaxf(mx, fmaxf(fabsf(c.x), fmaxf(fabsf(c.y), fabsf(c.z))));
        if (!(c.x == c.x) || !(c.y == c.y) || !(c.z == c.z)) mx = INFINITY;   // NaN stays active
        any_valid = 1;
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      any_valid |= __shfl_xor_sync(0xffffffffu, any_valid, o);
    }
    if (lane == 0) flags[hid] = (any_valid && (dense || mx > kSkipBelow)) ? 1 : 0;
  }
}

__global__ void tile_compact_kernel(const unsigned char* __restrict__ flags, const int* __restrict__ tile_off, int B,
                                    int* __restrict__ sub_list, int* __restrict__ n_active) {
  __shared__ int sums[1024];
  const int total = __ldg(&tile_off[B]);
  const int per = (total + blockDim.x - 1) / blockDim.x;
  const int lo = min(total, (int)threadIdx.x * per), hi = min(total, lo + per);
  int cnt = 0;
  for (int i = lo; i < hi; ++i) cnt += flags[i];
  sums[threadIdx.x] = cnt;
  __syncthreads();
  for (int o = 1; o < blockDim.x; o <<= 1) {      // inclusive Hillis-Steele scan
    int v = (threadIdx.x >= o) ? sums[threadIdx.x - o] : 0;
    __syncthreads();
    sums[threadIdx.x] += v;
    __syncthreads();
  }
  int pos = sums[threadIdx.x] - cnt;
  for (int i = lo; i < hi; ++i)
    if (flags[i]) sub_list[pos++] = i;
  if (threadIdx.x == blockDim.x - 1) *n_active = sums[threadIdx.x];
}

// ---- dense-logits front end: one warp per lattice cell (torchaudio ReduceMax2D/ReduceLogSumExp/ComputeLogProbs)
__global__ void dense_logprobs_kernel(const float* __restrict__ logits, const int* __restrict__ targets, int tgt_ld,
                                      const int* __restrict__ T_len, const int* __restrict__ U_len, int B, int T,
                                      int U1, int V, int blank, float* __restrict__ lp, float* __restrict__ lse) {
  const long long ncell = static_cast<long long>(B) * T * U1;
  const int lane = threadIdx.x & 31;
  const long long w0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long nw = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long i = w0; i < ncell; i += nw) {
    const int u = static_cast<int>(i % U1);
    const int t = static_cast<int>((i / U1) % T);
    const int b = static_cast<int>(i / (static_cast<long long>(U1) * T));
    const int Tb = T_len[b], Ub = U_len[b];
    if (t >= Tb || u > Ub) continue;
    const float* row = logits + i * V;
    float m = -INFINITY;
    for (int v = lane; v < V; v += 32) m = fmaxf(m, row[v]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
    for (int v = lane; v < V; v += 32) s += expf(row[v] - m);
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const float l = m + logf(s);
      lse[i] = l;
      float2 o2;
      o2.x = row[blank] - l;
      o2.y = (u < Ub) ? row[targets[static_cast<long long>(b) * tgt_ld + u]] - l : 0.f;
      reinterpret_cast<float2*>(lp)[i] = o2;
    }
  }
}

// ---- dense-logits back end (torchaudio ComputeGradients): grads fully overwritten, zeros on padding
__global__ void dense_grads_kernel(const float* __restrict__ logits, const int* __restrict__ targets, int tgt_ld,
                                   const int* __restrict__ T_len, const int* __restrict__ U_len,
                                   const float4* __restrict__ coef, int B, int T, int U1, int V, int blank,
                                   float clamp, float* __restrict__ grads) {
  const long long ncell = static_cast<long long>(B) * T * U1;
  const int lane = threadIdx.x & 31;
  const long long w0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long nw = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long i = w0; i < ncell; i += nw) {
    const int u = static_cast<int>(i % U1);
    const int t = static_cast<int>((i / U1) % T);
    const int b = static_cast<int>(i / (static_cast<long long>(U1) * T));
    const int Tb = T_len[b], Ub = U_len[b];
    float* out = grads + i * V;
    if (t >= Tb || u > Ub) {
      for (int v = lane; v < V; v += 32) out[v] = 0.f;
      continue;
    }
    const float4 c = coef[i];
    const int tgt = (u < Ub) ? targets[static_cast<long long>(b) * tgt_ld + u] : -1;
    const float* row = logits + i * V;
    for (int v = lane; v < V; v += 32) {
      float g = expf(row[v] - c.w) * c.x;
      if (v == blank) g -= c.y;
      if (v == tgt) g -= c.z;
      if (clamp > 0.f) g = fminf(fmaxf(g, -clamp), clamp);
      out[v] = g;
    }
  }
}

// deterministic mode: 64-bit fixed-point accumulators -> fp32 outputs (possibly strided, e.g. the encoder's (B,H,T) layout)
__global__ void finalize_fixed_kernel(const long long* __restrict__ fx, float* __restrict__ out, long long n0,
                                      long long n1, long long n2, long long s0, long long s1, long long s2,
                                      const float* __restrict__ gscale) {
  const long long n = n0 * n1 * n2;
  const double mul = kFxInv * static_cast<double>(gscale[1]);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long i2 = i % n2, i1 = (i / n2) % n1, i0 = i / (n2 * n1);
    out[i0 * s0 + i1 * s1 + i2 * s2] = static_cast<float>(static_cast<double>(fx[i]) * mul);
  }
}

}  // namespace

int launch_finalize_fixed(const long long* fx, float* out, long long n0, long long n1, long long n2, long long s0,
                          long long s1, long long s2, const float* gscale, cudaStream_t stream) {
  ProfScope prof_(kProfPrep, stream);
  const long long n = n0 * n1 * n2;
  const int grid = static_cast<int>(std::min<long long>((n + 255) / 256, 148 * 16));
  finalize_fixed_kernel<<<grid, 256, 0, stream>>>(fx, out, n0, n1, n2, s0, s1, s2, gscale);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_tile_table(const int* T_len, const int* U_len, int B, int T, int U1, int* tile_off, int* status,
                      int* err_flag, const float* dcost, float* gscale, cudaStream_t stream) {
  ProfScope prof_(kProfPrep, stream);
  tile_table_kernel<<<1, 32, 0, stream>>>(T_len, U_len, B, T, U1, tile_off, status, err_flag, dcost, gscale);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_convert_weights(const float* W, const float* bias, int V, int H, int Vp, int Hp, __half* Wh,
                           float* bias2, cudaStream_t stream) {
  ProfScope prof_(kProfPrep, stream);
  const long long n = static_cast<long long>(Vp) * (Hp / 8);
  const int grid = static_cast<int>(std::min<long long>((n + 255) / 256, 4096));
  convert_weights_kernel<<<grid, 256, 0, stream>>>(W, bias, V, H, Vp, Hp, Wh, bias2);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_lattice(const float* lp, const int* T_len, const int* U_len, int B, int T, int U1, float* alpha,
                   float* beta, float* costs, const int* status, cudaStream_t stream) {
  ProfScope prof_(kProfLattice, stream);
  const int threads = ((U1 + 31) / 32) * 32;
  RB_REQUIRE(threads <= 1024, -5, "lattice kernel supports U+1 <= 1024 (got %d)", U1);
  const size_t smem = 2 * (threads + 2) * sizeof(float);
  lattice_kernel<<<dim3(B, 2), threads, smem, stream>>>(lp, T_len, U_len, T, U1, alpha, beta, costs, status);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_coef(const float* lp, const float* lse, const float* alpha, const float* beta, const float* dcost,
                const float* gscale, const int* T_len, const int* U_len, int B, int T, int U1, float4* coef,
                cudaStream_t stream) {
  ProfScope prof_(kProfPrep, stream);
  const long long n = static_cast<long long>(B) * T * U1;
  const int grid = static_cast<int>(std::min<long long>((n + 255) / 256, 148 * 8));
  coef_kernel<<<grid, 256, 0, stream>>>(lp, lse, alpha, beta, dcost, gscale, T_len, U_len, B, T, U1, coef);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_tile_activity(const float4* coef, const int* T_len, const int* U_len, const int* tile_off, int B, int T,
                         int U1, long long max_tiles, int dense, unsigned char* flags, int* sub_list, int* n_active,
                         cudaStream_t stream) {
  ProfScope prof_(kProfPrep, stream);
  const int grid = static_cast<int>(std::min<long long>((2 * max_tiles + 7) / 8, 148 * 8));
  tile_activity_kernel<<<grid, 256, 0, stream>>>(coef, T_len, U_len, tile_off, B, T, U1, dense, flags);
  tile_compact_kernel<<<1, 1024, 0, stream>>>(flags, tile_off, B, sub_list, n_active);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_dense_logprobs(const float* logits, const int* targets, int tgt_ld, const int* T_len, const int* U_len,
                          int B, int T, int U1, int V, int blank, float* lp, float* lse, cudaStream_t stream) {
  ProfScope prof_(kProfOther, stream);
  const long long ncell = static_cast<long long>(B) * T * U1;
  const int grid = static_cast<int>(std::min<long long>((ncell + 7) / 8, 148 * 16));
  dense_logprobs_kernel<<<grid, 256, 0, stream>>>(logits, targets, tgt_ld, T_len, U_len, B, T, U1, V, blank, lp, lse);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_dense_grads(const float* logits, const int* targets, int tgt_ld, const int* T_len, const int* U_len,
                       const float4* coef, int B, int T, int U1, int V, int blank, float clamp, float* grads,
                       cudaStream_t stream) {
  ProfScope prof_(kProfOther, stream);
  const long long ncell = static_cast<long long>(B) * T * U1;
  const int grid = static_cast<int>(std::min<long long>((ncell + 7) / 8, 148 * 16));
  dense_grads_kernel<<<grid, 256, 0, stream>>>(logits, targets, tgt_ld, T_len, U_len, coef, B, T, U1, V, blank,
                                               clamp, grads);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace rb
