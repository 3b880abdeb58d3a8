// Batched beam-search decode as ONE persistent cooperative kernel (fp32 throughout).
//
// Frame-synchronous "modified" beam search (at most one symbol per frame; include/rnnt_b200.h states the contract): per
// utterance b the beam holds up to K hypotheses, each a token list with a log-score and its own incremental predictor
// state (the conv tap accumulators acc1 / acc2, lin, feats) -- the per-utterance state of the greedy kernel
// (decode_loop.cu), held in B*K hypothesis slots (row b*K + k) instead of B.  Same CTA / thread shape and the same
// shared phases (decode_common.cuh); per frame t:
//   P5  z = gelu(conv2), P6 lin = linear(z)   for the slots extended in the previous frame (and the seed blank)
//   P1  feats = LayerNorm(lin) for those slots; h = tanh(enc[b, t] + feats) for every hypothesis of a live utterance
//   P2  logits = W_j . h + b_j                 (gemv_phase over the live hypothesis rows)
//   P3  one CTA per live utterance, one warp per hypothesis: log-sum-exp, merge test, the top K extensions of the row
//       that no merge takes; then the K(K+1)-candidate selection, the gather of every new hypothesis's state from its
//       parent's slot into the other half of the double-buffered state, and conv1 of the extended ones
//       (+ with token timing: each token's frame and log-probability, gathered with the token lists)
// with a grid barrier after each phase: 5 per frame (P5 / P6 are skipped in a frame that extends nothing).  Every sum
// runs in a fixed order and every selection is a total order, so results are bit-identical run to run and do not
// depend on the batch an utterance sits in.
#include <algorithm>

#include "decode_common.cuh"
#include "kernels.h"

namespace rb {
namespace {

constexpr int kMaxCand = kMaxBeam * (kMaxBeam + 1);     // K blank continuations + K x K extensions
static_assert(kMaxBeam <= kThreads / 32 && kMaxCand <= kThreads, "P3 runs one warp per hypothesis, one thread per candidate");
constexpr unsigned long long kHashMul = 0x100000001b3ull;

// the selection order: score descending, then source hypothesis rank, then token index (ints packed as src * V + tok)
__device__ __forceinline__ bool better(float s1, int k1, float s2, int k2) { return s1 > s2 || (s1 == s2 && k1 < k2); }

__device__ __forceinline__ float log_add_exp(float a, float b) {
  const float m = fmaxf(a, b);
  return m + log1pf(expf(-fabsf(a - b)));
}

// ALIGN: the instance that also keeps each token's frame and log-probability (frames or token_logp requested); the
// plain decode runs the ALIGN = false instance, which has none of that code.
template <bool ALIGN>
__global__ void __launch_bounds__(kThreads, 1) beam_decode_kernel(BeamArgs p) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float red[kThreads / 32];
  // P3, per utterance: the beam (ntok = 1 + tokens, 0 = empty slot; scores; hashes), per hypothesis its log-sum-exp,
  // the slot of its prefix in the beam (-1: none), its last token and its best extensions; then the candidates
  __shared__ int s_nt[kMaxBeam];
  __shared__ float s_sc[kMaxBeam];
  __shared__ unsigned long long s_hash[kMaxBeam];
  __shared__ float s_lse[kMaxBeam];
  __shared__ int s_par[kMaxBeam], s_last[kMaxBeam], s_next[kMaxBeam];
  __shared__ float s_ext[kMaxBeam][kMaxBeam];
  __shared__ int s_extv[kMaxBeam][kMaxBeam];
  __shared__ float c_sc[kMaxCand];
  __shared__ int c_key[kMaxCand];
  __shared__ int c_dom[kMaxCand];       // merged candidates: the slot q whose extension dominates the merge, else -1
  __shared__ int s_sel[kMaxBeam];
  __shared__ int s_nsel;
  const int B = p.B, H = p.H, V = p.V, E = p.E, K = p.K, L = p.max_len;
  const int R = B * K;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x, cta = blockIdx.x;
  int* rows_act = p.rows;          // compacted list of live hypothesis rows (P2) ...
  int* rows_emit = p.rows + R;     // ... and of rows extended in this frame (P5-P6)
  int* counts = p.flags;           // [0] n_live, [1] n_emit
  unsigned* bar_counter = p.bar;
  unsigned bar_target = 0;
  const bool timer = (cta == 0 && tid == 0 && p.prof != nullptr);
  long long tmark = timer ? clock64() : 0;
  auto lap = [&](int slot) { if (timer) { const long long now = clock64(); p.prof[slot] += now - tmark; tmark = now; } };
  if (timer) for (int i = 0; i < 8; ++i) p.prof[i] = 0;

  // ---- this CTA's output slices of the four weight matrices; resident in shared memory where the launcher found room
  // (the same slices and offsets as the greedy kernel)
  const int perJ = (V + G - 1) / G, perE = (E + G - 1) / G, perL = (H + G - 1) / G;
  const int j_lo = min(V, cta * perJ), j_hi = min(V, j_lo + perJ);
  const int e_lo = min(E, cta * perE), e_hi = min(E, e_lo + perE);
  const int l_lo = min(H, cta * perL), l_hi = min(H, l_lo + perL);
  const float* Wj_s = p.Wj + static_cast<long long>(j_lo) * H;
  const float* w1_s = p.w1 + static_cast<long long>(e_lo) * 3 * E;
  const float* w2_s = p.w2 + static_cast<long long>(e_lo) * 5 * E;
  const float* wl_s = p.wl + static_cast<long long>(l_lo) * E;
  float* xstage = smem + p.weight_floats;
  {
    const long long off_j = 0;
    const long long off_2 = off_j + ((p.resident & 1) ? static_cast<long long>(perJ) * H : 0);
    const long long off_1 = off_2 + ((p.resident & 2) ? static_cast<long long>(perE) * 5 * E : 0);
    const long long off_l = off_1 + ((p.resident & 4) ? static_cast<long long>(perE) * 3 * E : 0);
    auto stage = [&](const float*& w, int nrows, int Kw, bool resident, long long off) {
      if (!resident) return;
      const float4* src = reinterpret_cast<const float4*>(w);
      float4* d4 = reinterpret_cast<float4*>(smem + off);
      for (int i = tid; i < nrows * (Kw >> 2); i += kThreads) d4[i] = __ldg(src + i);
      w = smem + off;
    };
    stage(Wj_s, j_hi - j_lo, H, p.resident & 1, off_j);
    stage(w2_s, e_hi - e_lo, 5 * E, p.resident & 2, off_2);
    stage(w1_s, e_hi - e_lo, 3 * E, p.resident & 4, off_1);
    stage(wl_s, l_hi - l_lo, E, p.resident & 8, off_l);
  }

  // per-parity views of the double-buffered hypothesis state
  auto feats = [&](int par) { return p.feats + static_cast<long long>(par) * R * H; };
  auto acc1 = [&](int par) { return p.acc1 + static_cast<long long>(par) * R * 3 * E; };
  auto acc2 = [&](int par) { return p.acc2 + static_cast<long long>(par) * R * 5 * E; };
  auto ntok = [&](int par) { return p.ntok + par * R; };
  auto score = [&](int par) { return p.score + par * R; };
  auto hash = [&](int par) { return p.hash + par * R; };
  auto hyp = [&](int par, int r) { return p.hyp + (static_cast<long long>(par) * R + r) * L; };
  auto hyp_fr = [&](int par, int r) { return p.hyp_fr + (static_cast<long long>(par) * R + r) * L; };
  auto hyp_lp = [&](int par, int r) { return p.hyp_lp + (static_cast<long long>(par) * R + r) * L; };
  auto frames = [&](int b) { return max(0, min(__ldg(p.T_len + b), p.T)); };

  // ---- the initial beam {(empty, 0)}: slot 0 of every utterance holds the seed blank's predictor state (zero tap
  // accumulators = the left zero padding; its conv1 step below, conv2 / linear in the first frame's P5 / P6), the other
  // slots are empty.  The outputs start as that beam, which is the result of an utterance without frames.
  for (int r = cta * kThreads + tid; r < R; r += G * kThreads) {
    const int k = r % K;
    ntok(0)[r] = k == 0 ? 1 : 0;
    score(0)[r] = 0.f;
    hash(0)[r] = 0ull;
    p.emit[r] = k == 0;
    p.n_tokens[r] = k == 0 ? 1 : 0;
    p.scores[r] = k == 0 ? 0.f : -INFINITY;
  }
  if (cta == 0) {
    for (int b = tid; b < B; b += kThreads) rows_emit[b] = b * K;
    if (tid == 0) { counts[0] = 0; counts[1] = B; }
  }
  for (int b = cta; b < B; b += G) {
    const long long r = static_cast<long long>(b) * K;
    for (int i = tid; i < 3 * E; i += kThreads) acc1(0)[r * 3 * E + i] = 0.f;
    for (int i = tid; i < 5 * E; i += kThreads) acc2(0)[r * 5 * E + i] = 0.f;
  }
  // ---- the two per-symbol tables: LayerNorm(embedding) and conv1's tap products of it
  for (int v = cta; v < p.NS; v += G)
    block_layer_norm(p.emb + static_cast<long long>(v) * E, p.ln1_w, p.ln1_b, p.emb_ln + static_cast<long long>(v) * E, E, red);
  grid_barrier(bar_counter, bar_target);
  {
    GemvEpi epi{2, 3, nullptr, nullptr, E};
    gemv_phase<false>(w1_s, nullptr, e_lo, e_hi, E, 3 * E, p.emb_ln, E, nullptr, p.NS, p.t1, 3 * E, epi, xstage);
  }
  lap(3);
  grid_barrier(bar_counter, bar_target);
  for (int b = cta; b < B; b += G) {
    const long long r = static_cast<long long>(b) * K;
    conv1_update(p.t1 + static_cast<long long>(p.blank) * 3 * E, acc1(0) + r * 3 * E, p.b1, p.ynew + r * E, E, 0);
  }
  grid_barrier(bar_counter, bar_target);
  lap(7);

  int cur = 0;
  for (int t = 0;; ++t, cur ^= 1) {
    const int n_emit = __ldcg(counts + 1);
    if (n_emit > 0) {
      // ---- P5: conv2, tap products of the new conv1 output (the tap ring of the slot's current state)
      {
        GemvEpi epi{1, 5, acc2(cur), ntok(cur), E};
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

    // ---- P1: predictor features of the extended slots; joint hidden rows of every hypothesis of a live utterance
    for (int r = cta; r < R; r += G) {
      const int b = r / K;
      const bool live = t < frames(b) && __ldcg(ntok(cur) + r) > 0;
      if (live && __ldcg(p.emit + r))
        block_layer_norm(p.lin + static_cast<long long>(r) * H, p.ln2_w, p.ln2_b, feats(cur) + static_cast<long long>(r) * H, H, red);
      __syncthreads();
      if (live) {
        const float* e = p.enc + b * p.enc_sb + static_cast<long long>(t) * p.enc_st;
        const float* f = feats(cur) + static_cast<long long>(r) * H;
        for (int i = tid; i < H; i += kThreads) p.hbuf[static_cast<long long>(r) * H + i] = tanhf(__ldg(e + i) + __ldcg(f + i));
      }
    }
    if (cta == G - 1 && tid < 32) {
      // compact the live rows (single warp, order preserved)
      int n = 0;
      for (int r0 = 0; r0 < R; r0 += 32) {
        const int r = r0 + tid;
        const bool a = r < R && t < frames(r / K) && __ldcg(ntok(cur) + r) > 0;
        const unsigned m = __ballot_sync(0xffffffffu, a);
        if (a) rows_act[n + __popc(m & ((1u << tid) - 1))] = r;
        n += __popc(m);
      }
      if (tid == 0) { counts[0] = n; counts[1] = 0; }
    }
    lap(0);
    grid_barrier(bar_counter, bar_target);
    lap(7);
    const int n_act = __ldcg(counts + 0);
    if (n_act == 0) break;
    if (timer) p.prof[6] += 1;      // frames taken (slot 6 of the phase counters)

    // ---- P2: joint logits of the live hypotheses
    {
      GemvEpi epi{0, 1, nullptr, nullptr, E};
      gemv_phase<false>(Wj_s, p.bj, j_lo, j_hi, H, H, p.hbuf, H, rows_act, n_act, p.logits, V, epi, xstage);
    }
    lap(1);
    grid_barrier(bar_counter, bar_target);
    lap(7);

    // ---- P3: selection and gather, one CTA per live utterance
    const int nxt = cur ^ 1;
    for (int b = cta; b < B; b += G) {
      const int Tb = frames(b);
      if (t >= Tb) continue;
      const int r0 = b * K;
      if (tid < K) {
        s_nt[tid] = __ldcg(ntok(cur) + r0 + tid);
        s_sc[tid] = __ldcg(score(cur) + r0 + tid);
        s_hash[tid] = __ldcg(hash(cur) + r0 + tid);
      }
      __syncthreads();
      int nh = 0;                   // the filled slots are a prefix of the beam
      for (int k = 0; k < K; ++k) nh += s_nt[k] > 0;
      const int h = warp;           // one warp per hypothesis (K <= 8 warps)
      if (h < nh) {
        const float* row = p.logits + static_cast<long long>(r0 + h) * V;
        float m = -INFINITY;
        for (int v = lane; v < V; v += 32) m = fmaxf(m, __ldcg(row + v));
        for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float s = 0.f;
        for (int v = lane; v < V; v += 32) s += expf(__ldcg(row + v) - m);
        s = warp_sum(s);
        // merge test: the slot q whose token list is this one's minus its last token (equal lengths and hashes
        // pre-filter, the token lists decide)
        const int len = s_nt[h] - 1;
        const int* th = hyp(cur, r0 + h);
        int par = -1, last = -1;
        if (len >= 1) {
          last = __ldcg(th + len - 1);
          for (int q = 0; q < nh && par < 0; ++q) {
            if (s_nt[q] - 1 != len - 1 || s_hash[q] * kHashMul + static_cast<unsigned long long>(last + 1) != s_hash[h])
              continue;
            const int* tq = hyp(cur, r0 + q);
            bool diff = false;
            for (int i = lane; i < len - 1; i += 32) diff |= __ldcg(tq + i) != __ldcg(th + i);
            if (!__any_sync(0xffffffffu, diff)) par = q;
          }
        }
        if (lane == 0) { s_lse[h] = m + logf(s); s_par[h] = par; s_last[h] = last; }
      }
      __syncthreads();
      if (h < nh) {
        // the best K extensions of hypothesis h by candidate score, skipping blank and the tokens a merge takes
        const float* row = p.logits + static_cast<long long>(r0 + h) * V;
        const float lse = s_lse[h], sh = s_sc[h];
        const bool can_extend = s_nt[h] + 1 <= L;       // 1 + len + 1 <= max_len
        int taken[kMaxBeam];
#pragma unroll
        for (int q = 0; q < kMaxBeam; ++q) taken[q] = (q < nh && s_par[q] == h) ? s_last[q] : -1;
        float tv[kMaxBeam];
        int ti[kMaxBeam];
#pragma unroll
        for (int i = 0; i < kMaxBeam; ++i) { tv[i] = -INFINITY; ti[i] = 0x7fffffff; }
        if (can_extend) {
          for (int v = lane; v < V; v += 32) {
            bool skip = v == p.blank;
#pragma unroll
            for (int q = 0; q < kMaxBeam; ++q) skip |= v == taken[q];
            if (skip) continue;
            const float c = sh + (__ldcg(row + v) - lse);
            if (better(c, v, tv[kMaxBeam - 1], ti[kMaxBeam - 1])) {     // sorted insert into the lane's list
              tv[kMaxBeam - 1] = c; ti[kMaxBeam - 1] = v;
#pragma unroll
              for (int i = kMaxBeam - 1; i > 0; --i)
                if (better(tv[i], ti[i], tv[i - 1], ti[i - 1])) {
                  const float x = tv[i]; tv[i] = tv[i - 1]; tv[i - 1] = x;
                  const int y = ti[i]; ti[i] = ti[i - 1]; ti[i - 1] = y;
                }
            }
          }
        }
        // merge of the 32 sorted lane lists: K rounds of a warp arg-best over the list heads
        int n_ext = 0;
        for (int i = 0; i < K; ++i) {
          float bv = tv[0];
          int bi = ti[0];
          for (int o = 16; o; o >>= 1) {
            const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
            const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(v2, i2, bv, bi)) { bv = v2; bi = i2; }
          }
          if (bi == 0x7fffffff) break;                   // fewer than K tokens left (uniform)
          if (ti[0] == bi) {
#pragma unroll
            for (int j = 0; j < kMaxBeam - 1; ++j) { tv[j] = tv[j + 1]; ti[j] = ti[j + 1]; }
            tv[kMaxBeam - 1] = -INFINITY; ti[kMaxBeam - 1] = 0x7fffffff;
          }
          if (lane == 0) { s_ext[h][i] = bv; s_extv[h][i] = bi; }
          ++n_ext;
        }
        if (lane == 0) s_next[h] = n_ext;
      }
      __syncthreads();
      // candidates: c = h * (K+1) is the blank continuation of h (merged with the extension of its prefix slot when
      // there is one), c = h * (K+1) + 1 + i the i-th extension of h
      const int nc = nh * (K + 1);
      if (tid < nc) {
        const int hh = tid / (K + 1), i = tid % (K + 1) - 1;
        float sc = -INFINITY;
        int key = 0x7fffffff, dom = -1;
        if (i < 0) {
          const float* row = p.logits + static_cast<long long>(r0 + hh) * V;
          sc = s_sc[hh] + (__ldcg(row + p.blank) - s_lse[hh]);
          const int q = s_par[hh];
          if (q >= 0) {
            const float* rq = p.logits + static_cast<long long>(r0 + q) * V;
            const float sq = s_sc[q] + (__ldcg(rq + s_last[hh]) - s_lse[q]);
            if (ALIGN && sq > sc) dom = q;   // the merge keeps the timing of its larger term; a tie keeps the blank's
            sc = log_add_exp(sc, sq);
          }
          key = hh * V + p.blank;
        } else if (i < s_next[hh]) {
          sc = s_ext[hh][i];
          key = hh * V + s_extv[hh][i];
        }
        c_sc[tid] = sc;
        c_key[tid] = key;
        if (ALIGN) c_dom[tid] = dom;
      }
      __syncthreads();
      // rank of each candidate in the selection order = number of candidates before it (a total order: keys differ)
      if (tid < nc && c_key[tid] != 0x7fffffff) {
        int rank = 0;
        for (int j = 0; j < nc; ++j) rank += c_key[j] != 0x7fffffff && better(c_sc[j], c_key[j], c_sc[tid], c_key[tid]);
        if (rank < K) s_sel[rank] = tid;
      }
      if (tid == 0) {
        int n = 0;
        for (int j = 0; j < nc; ++j) n += c_key[j] != 0x7fffffff;
        s_nsel = min(n, K);
      }
      __syncthreads();
      const int nsel = s_nsel;
      // frames and log-probabilities of candidate c's token list: those of the constituent that dominates it (the
      // source hypothesis, or for a merge whose extension term is larger, the extended slot q), plus this frame's token
      auto copy_lists = [&](int c, int* dfr, float* dlp) {
        const int src = c_key[c] / V, v = c_key[c] % V, q = c_dom[c];
        const int base = q >= 0 ? q : src, nb = s_nt[base] - 1;
        const int* sf = hyp_fr(cur, r0 + base);
        const float* sl = hyp_lp(cur, r0 + base);
        for (int i = tid; i < nb; i += kThreads) {
          if (dfr) dfr[i] = __ldcg(sf + i);
          if (dlp) dlp[i] = __ldcg(sl + i);
        }
        if (tid == 0 && (v != p.blank || q >= 0)) {
          const int tok = q >= 0 ? s_last[src] : v;
          if (dfr) dfr[nb] = t;
          if (dlp) dlp[nb] = __ldcg(p.logits + static_cast<long long>(r0 + base) * V + tok) - s_lse[base];
        }
      };
      if (t == Tb - 1) {
        // last frame of the utterance: the new beam, best first, is the output
        for (int j = 0; j < K; ++j) {
          const long long o = static_cast<long long>(r0 + j);
          if (j < nsel) {
            const int c = s_sel[j], src = c_key[c] / V, v = c_key[c] % V;
            const int len = s_nt[src] - 1;
            const int* ts = hyp(cur, r0 + src);
            for (int i = tid; i < len; i += kThreads) p.tokens[o * L + i] = __ldcg(ts + i);
            if (tid == 0) {
              if (v != p.blank) p.tokens[o * L + len] = v;
              p.n_tokens[o] = 1 + len + (v != p.blank);
              p.scores[o] = c_sc[c];
            }
          } else if (tid == 0) {
            p.n_tokens[o] = 0;
            p.scores[o] = -INFINITY;
          }
        }
        if (ALIGN)
          for (int j = 0; j < nsel; ++j) {
            const long long o = static_cast<long long>(r0 + j) * L;
            copy_lists(s_sel[j], p.frames ? p.frames + o : nullptr, p.token_logp ? p.token_logp + o : nullptr);
          }
      } else {
        // gather: new slot j takes its parent's state (always copied: parents may feed several slots), extended slots
        // then run conv1 on their new token; feats only matter for blank continuations (the others recompute it)
        for (int j = 0; j < K; ++j) {
          const int rd = r0 + j;
          if (j >= nsel) {
            if (tid == 0) { ntok(nxt)[rd] = 0; p.emit[rd] = 0; }
            continue;
          }
          const int c = s_sel[j], src = c_key[c] / V, v = c_key[c] % V;
          const bool ext = v != p.blank;
          const int rs = r0 + src, nt = s_nt[src];
          auto copy4 = [&](float* dst, const float* srcp, int n) {
            const float4* s4 = reinterpret_cast<const float4*>(srcp);
            float4* d4 = reinterpret_cast<float4*>(dst);
            for (int i = tid; i < (n >> 2); i += kThreads) d4[i] = __ldcg(s4 + i);
          };
          copy4(acc1(nxt) + static_cast<long long>(rd) * 3 * E, acc1(cur) + static_cast<long long>(rs) * 3 * E, 3 * E);
          copy4(acc2(nxt) + static_cast<long long>(rd) * 5 * E, acc2(cur) + static_cast<long long>(rs) * 5 * E, 5 * E);
          if (!ext) copy4(feats(nxt) + static_cast<long long>(rd) * H, feats(cur) + static_cast<long long>(rs) * H, H);
          const int* ts = hyp(cur, rs);
          int* td = hyp(nxt, rd);
          for (int i = tid; i < nt - 1; i += kThreads) td[i] = __ldcg(ts + i);
          if (tid == 0) {
            if (ext) td[nt - 1] = v;
            ntok(nxt)[rd] = nt + ext;
            score(nxt)[rd] = c_sc[c];
            hash(nxt)[rd] = ext ? s_hash[src] * kHashMul + static_cast<unsigned long long>(v + 1) : s_hash[src];
            p.emit[rd] = ext;
            if (ext) rows_emit[atomicAdd(&counts[1], 1)] = rd;
          }
          if (ext) {
            __syncthreads();        // the copied accumulators before conv1 reads them back
            // the new symbol's position in the predictor's input = 1 + the parent's token count = its ntok
            conv1_update(p.t1 + static_cast<long long>(v) * 3 * E, acc1(nxt) + static_cast<long long>(rd) * 3 * E, p.b1,
                         p.ynew + static_cast<long long>(rd) * E, E, nt);
          }
        }
        if (ALIGN)
          for (int j = 0; j < nsel; ++j) copy_lists(s_sel[j], hyp_fr(nxt, r0 + j), hyp_lp(nxt, r0 + j));
      }
      __syncthreads();
    }
    lap(2);
    grid_barrier(bar_counter, bar_target);
    lap(7);
  }
}

}  // namespace

// Scratch layout: [8 x int64 phase timers | barrier line | hashes [2][B*K] | float regions, each padded to a multiple of
// 4 floats (16-byte aligned, cp.async / float4) | int regions].
size_t beam_decode_scratch_bytes(int B, int K, int H, int V, int E, int max_len) {
  const size_t r = static_cast<size_t>(B) * K;
  const size_t floats = 2 * pad4(r * H) /*feats x2*/ + 2 * pad4(r * H) /*hbuf, lin*/ + pad4(r * V) /*logits*/ +
                        2 * pad4(r * 3 * E) + 2 * pad4(r * 5 * E) + 2 * pad4(r * E) /*ynew, z*/ + pad4(2 * r) /*scores*/ +
                        pad4(static_cast<size_t>(V) * E) + pad4(static_cast<size_t>(V) * 3 * E) /*symbol tables*/;
  const size_t ints = 2 * r /*ntok*/ + r /*emit*/ + 2 * r /*rows*/ + 16 + 2 * r * max_len /*token lists*/ +
                      4 * r * max_len /*their frames and log-probabilities*/;
  return kTimerBytes + kBarBytes + 2 * r * 8 + floats * 4 + ints * 4 + 256;
}

int launch_beam_decode(BeamArgs a, float* scratch, cudaStream_t stream) {
  ProfScope prof_(kProfOther, stream);
  RB_REQUIRE(a.B > 0 && a.H > 0 && a.V > 1 && a.E > 0 && a.max_len >= 1 && a.K >= 1 && a.K <= kMaxBeam, -1,
             "invalid decode shape");
  RB_REQUIRE(a.H % 4 == 0 && a.E % 4 == 0, -2, "decode kernel needs hidden / embedding sizes that are multiples of 4");
  RB_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 127) == 0, -3, "decode scratch must be 128-byte aligned");
  const int grid = device_sm_count();
  const size_t smem = decode_smem_plan(grid, a.H, a.V, a.E, &a.resident, &a.weight_floats);
  // carve the scratch
  a.prof = reinterpret_cast<long long*>(scratch);
  a.bar = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(scratch) + kTimerBytes);
  RB_CUDA_CHECK(cudaMemsetAsync(a.bar, 0, kBarBytes, stream));
  const int H = a.H, V = a.V, E = a.E;
  const size_t r = static_cast<size_t>(a.B) * a.K;
  a.hash = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(scratch) + kTimerBytes + kBarBytes);
  float* f = reinterpret_cast<float*>(a.hash + 2 * r);
  a.feats = f; f += 2 * pad4(r * H);
  a.hbuf = f; f += pad4(r * H);
  a.lin = f; f += pad4(r * H);
  a.logits = f; f += pad4(r * V);
  a.acc1 = f; f += 2 * pad4(r * 3 * E);
  a.acc2 = f; f += 2 * pad4(r * 5 * E);
  a.ynew = f; f += pad4(r * E);
  a.z = f; f += pad4(r * E);
  a.score = f; f += pad4(2 * r);
  a.emb_ln = f; f += pad4(static_cast<size_t>(a.NS) * E);
  a.t1 = f; f += pad4(static_cast<size_t>(a.NS) * 3 * E);
  int* ip = reinterpret_cast<int*>(f);
  a.ntok = ip; ip += 2 * r;
  a.emit = ip; ip += r;
  a.rows = ip; ip += 2 * r;
  a.flags = ip; ip += 16;
  a.hyp = ip; ip += 2 * r * a.max_len;
  a.hyp_fr = ip; ip += 2 * r * a.max_len;
  a.hyp_lp = reinterpret_cast<float*>(ip); ip += 2 * r * a.max_len;
  void (*kernel)(BeamArgs) =
      a.frames != nullptr || a.token_logp != nullptr ? beam_decode_kernel<true> : beam_decode_kernel<false>;
  RB_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  RB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem));
  RB_REQUIRE(per_sm >= 1, -6, "decode kernel does not fit on an SM");
  void* args[] = {&a};
  // cooperative launch: guarantees that all CTAs are co-resident, which the kernel's own grid barrier relies on
  RB_CUDA_CHECK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), dim3(grid), dim3(kThreads),
                                            args, smem, stream));
  return 0;
}

}  // namespace rb
