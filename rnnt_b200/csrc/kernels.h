// Internal launch interface between the C-ABI layer (api.cu) and the kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "host_util.h"

namespace rb {

// What the kernels of the fused loss (joint GEMM, dh, dW) share: the joint's inputs, the batch's lengths and tile table,
// the sizes, the window of work-list slots a launch covers, and the gradient scale.  Not every kernel reads every field.
struct BatchArgs {
  const float* enc;       // (B,T,H) fp32 with element strides (enc_sb, enc_st, enc_sh): H-contiguous (enc_sh == 1) or
  long long enc_sb, enc_st, enc_sh;   // the T-contiguous view of the encoder's (B,H,T) output (enc_st == 1)
  const float* pred;      // (B,U1,H) fp32, H contiguous
  long long pred_sb, pred_su;
  const float* bias2;     // [Vp] bias * log2(e); padding columns hold -1e30
  const int* targets;     // (B,U) int32
  int tgt_ld;
  const int* T_len;
  const int* U_len;
  const int* tile_off;    // [B+1] prefix sum of half-tiles (16 t x 4 u) per utterance; tile_off[B] = total
  int B, T, U1, H, Hp, V, Vp, blank;
  int slot_begin, slot_cap;   // process work-list slots (half-tiles, 64 rows) [slot_begin, min(count, slot_begin + slot_cap))
  const int* sub_list;    // backward: slot -> half-tile id (active ones only), ring rows [64 i, 64 i + 64) hold
                          // sub_list[slot_begin + i]; nullptr (forward) = identity over all half-tiles
  const int* n_active;    // backward: number of slots in sub_list
  const float* gscale;    // backward: {S, 1/S} power-of-two gradient scale
  int h_map;              // rows of a half-tile in the activation buffer: 0 = half_id*64 (saved residual), 1 = ring
                          // slot*64 (backward recompute), 2 = per-CTA scratch (forward without a residual buffer)
};

struct JointArgs : BatchArgs {
  float* lp;              // F: output (B,T,U1,2) log-probs (blank, label); G: the same tensor, read-only
  float* lse;             // F: (B,T,U1) log-sum-exp of the logits (natural log)
  const float4* coef;     // G: (B,T,U1) (gamma*dc*S, eB*dc*S, eE*dc*S, lse)
  const float* dcost;     // G: (B) or nullptr (only used to scale the clamp bound)
  float clamp;            // G: <= 0 disables (torchaudio's clamp argument, rnnt/model.py:40 passes -1)
  __half* h_out;          // producers: activation rows h = tanh(enc+pred) as fp16 [rows, Hp] (same buffer tmH reads)
  __half* g_ring;         // G: gradient ring [ring_tiles*128, Vp] fp16
  int dbg;                // diagnostics only (RNNT_B200_DBG): 1 = skip epilogue math, 2 = skip producer math
};

struct DhArgs : BatchArgs {   // tanh' is recomputed from enc and pred
  float* d_enc;          // (B,T,H) fp32 with element strides (denc_sb, denc_st, denc_sh), accumulated with atomics
  long long denc_sb, denc_st, denc_sh;   // (caller zero-fills)
  float* d_pred;         // (B,U1,H) contiguous
  // deterministic mode: order-independent 64-bit fixed-point accumulators (2^-36 units) instead of fp32 atomics;
  // dense (B,T,H) / (B,U1,H) row-major, converted to d_enc / d_pred by finalize_fixed_kernel
  long long* d_enc_fx;
  long long* d_pred_fx;
};

struct DwArgs : BatchArgs {   // ring rows of a chunk = slots in range * 64; h_map is 0 or 1
  float* dW;             // (V,H) fp32, accumulated with atomics (caller zero-fills)
  float* db;             // (V) fp32, accumulated with atomics (column sums of g, taken from the A stages)
  long long* dW_fx;      // deterministic mode: 64-bit fixed-point accumulators (V,H) / (V), else nullptr
  long long* db_fx;
  int ksplit;
};

// One launch of the persistent greedy decode.  The per-slot decoder state lives in the caller's state buffer (carved by
// the launcher), so a launch continues every live slot where the previous launch on the same buffer stopped:
//   init     build the two per-symbol tables and mark every slot empty (n_tokens 0)
//   reset    slots that start a new utterance before this launch's frames: predictor state zeroed, seed blank run
//   T_len    frames each slot consumes in this launch, clamped to [0, T]
// The one-shot decode is init + every slot reset + T_len = the utterance lengths.
struct DecodeArgs {
  const float* enc;        // (B,T,H) fp32, H contiguous
  long long enc_sb, enc_st;
  const int* T_len;        // (B) frames per slot in this launch (may be null when no slot is live)
  int init;                // 1: build the symbol tables and empty every slot first
  int reset_all;           // 1: every slot is reset (else the slots with reset[b] != 0)
  const int* reset;        // (B) or null
  const float* Wj; const float* bj;                       // joint_ln (V,H), (V)
  const float* emb; const float* ln1_w; const float* ln1_b;   // embedding (NS,E), input LayerNorm (E)
  const float* w1; const float* b1;                       // conv1 as (E, 3E): taps oldest..newest
  const float* w2; const float* b2;                       // conv2 as (E, 5E)
  const float* wl; const float* bl;                       // linear (H,E), (H)
  const float* ln2_w; const float* ln2_b;                 // output LayerNorm (H)
  int B, T, H, V, E, blank, max_len, max_per_frame, max_steps;
  int weight_floats;       // floats of dynamic shared memory taken by the resident weight slices (staging follows)
  int resident;            // bit i: weight matrix i (joint, conv2, conv1, linear) has its per-CTA slice in shared memory
  int* tokens;             // (B, max_len) emitted tokens (seed blank excluded)
  int* n_tokens;           // (B) output copy of ntok at the end of the launch (may be null)
  float* margins;          // (max_steps, B) top-2 logit gap per step (may be null)
  // state (carved by the launcher): kept across launches -- feats, lin, acc1, acc2, emb_ln, t1, ntok, emit, last_tok,
  // frame_base, path_score;
  // per-launch scratch -- hbuf, logits, ynew, z, t_idx, per, rows, flags
  float *feats, *hbuf, *logits, *acc1, *acc2, *ynew, *z, *lin, *emb_ln, *t1 /* conv1 tap table (NS, 3E) */;
  int* ntok;               // (B) 0 = empty slot, else 1 + number of emitted tokens (the predictor's next position)
  int *t_idx, *per, *emit, *rows, *last_tok, *flags;
  unsigned* bar;           // grid-barrier counters (one per 128-byte line)
  int NS;                  // number of symbols = rows of the embedding table
  long long* prof;         // 8 cycle counters (block 0): P1, P2, P3, conv1 table build (once), P5, P6, -, grid barriers
  // token timing and confidence: per emitted token its frame and log-probability, per slot the greedy path's score
  int* frames;             // (B, max_len) frame of each emitted token, counted from the slot's reset (may be null)
  float* token_logp;       // (B, max_len) log-softmax of the emitted token at its step (may be null)
  float* path_scores;      // (B) output copy of path_score at the end of the launch (may be null)
  int want_lp;             // 1: P3 takes each row's log-sum-exp and accumulates path_score (token_logp or path_scores
                           // requested, and every streaming launch)
  int* frame_base;         // state (B): frames consumed since the slot's reset, before this launch
  float* path_score;       // state (B): sum of the step log-probabilities since the slot's reset
};

size_t greedy_decode_scratch_bytes(int B, int H, int V, int E);
int launch_greedy_decode(DecodeArgs a, float* scratch, cudaStream_t stream);

// One launch of the persistent beam-search decode (beam_loop.cu).  Weights, sizes, enc / T_len, blank and max_len are
// the DecodeArgs fields; the rows of the per-row buffers are the B*K hypothesis slots (row b*K + k = slot k of
// utterance b).  feats, acc1, acc2 and ntok are double-buffered by frame parity ([2][B*K][...]): a frame reads one
// copy and gathers each new hypothesis's state from its parent into the other.  lin, hbuf, logits, ynew, z, emit and
// rows are single.  tokens (B,K,max_len) and n_tokens (B,K) are the outputs, as is `scores`.
struct BeamArgs : DecodeArgs {
  int K;                      // beam size, 1..kMaxBeam
  float* scores;              // (B,K) output: log-scores, best first; -inf for slots that never fill
  float* score;               // [2][B*K] running hypothesis scores
  unsigned long long* hash;   // [2][B*K] rolling hash of each token list (pre-filter of the merge test)
  int* hyp;                   // [2][B*K][max_len] token lists (seed blank excluded)
  int* hyp_fr;                // [2][B*K][max_len] frame of each token (read and written only when `frames` or
  float* hyp_lp;              // [2][B*K][max_len] its log-probability   `token_logp` is set)
};
constexpr int kMaxBeam = 8;

size_t beam_decode_scratch_bytes(int B, int K, int H, int V, int E, int max_len);
int launch_beam_decode(BeamArgs a, float* scratch, cudaStream_t stream);

int joint_gemm_scratch_tiles(int grid);   // tiles of per-CTA activation scratch the forward needs when h_map == 2
// tmW: 64(k) x 128(v) boxes (each CTA of a pair loads half of a 256-class block); tmH / tmH2: 64(k) x 64 / 128 (row)
// boxes of the activation buffer (one half-tile / two adjacent ones); max_slots bounds the work-list slots of this launch
int launch_joint_gemm(int mode, bool produce, const CUtensorMap& tmW, const CUtensorMap& tmH, const CUtensorMap& tmH2,
                      const JointArgs& args, long long max_slots, cudaStream_t stream);
// tmG: 64(v) x 128(cell) boxes of the gradient ring; chunk_slots bounds the work-list slots of this ring chunk
int launch_dh_gemm(const CUtensorMap& tmG, const CUtensorMap& tmWmn, const DhArgs& args, long long chunk_slots,
                   cudaStream_t stream);
int launch_dw_gemm(const CUtensorMap& tmGmn, const CUtensorMap& tmHmn, const DwArgs& args, long long chunk_slots,
                   cudaStream_t stream);   // picks args.ksplit itself

// prep / small kernels (prep.cu, lattice.cu, decode.cu)
// status: internal word, non-zero when a length is out of range (read by the lattice); err_flag: optional copy for the
// caller; gscale (optional): {S, 1/S} derived from dcost
int launch_tile_table(const int* T_len, const int* U_len, int B, int T, int U1, int* tile_off, int* status,
                      int* err_flag, const float* dcost, float* gscale, cudaStream_t stream);
int launch_convert_weights(const float* W, const float* bias, int V, int H, int Vp, int Hp, __half* Wh,
                           float* bias2, cudaStream_t stream);
// status (optional): device flag written by the tile table; a non-zero flag turns every cost into NaN
int launch_lattice(const float* lp, const int* T_len, const int* U_len, int B, int T, int U1, float* alpha,
                   float* beta, float* costs, const int* status, cudaStream_t stream);
// Viterbi walk + backtrace (forced alignment), one CTA of round_up(U1, 32) threads per utterance.  Its decision bits
// live in shared memory: viterbi_smem_bytes(T, U1) must not exceed the sm_100a per-block opt-in limit.
constexpr size_t kViterbiSmemLimit = 232448;
size_t viterbi_smem_bytes(int T, int U1);
int launch_viterbi(const float* lp, const int* T_len, const int* U_len, int B, int T, int U1, int* frames,
                   float* scores, cudaStream_t stream);
// deterministic mode: out[i] = fx[i] * 2^-36 * gscale[1]; dst strides in elements (n0 x n1 x n2 logical shape)
int launch_finalize_fixed(const long long* fx, float* out, long long n0, long long n1, long long n2, long long s0,
                          long long s1, long long s2, const float* gscale, cudaStream_t stream);
int launch_coef(const float* lp, const float* lse, const float* alpha, const float* beta, const float* dcost,
                const float* gscale, const int* T_len, const int* U_len, int B, int T, int U1, float4* coef,
                cudaStream_t stream);
// flags / sub_list are indexed by half-tile id
int launch_tile_activity(const float4* coef, const int* T_len, const int* U_len, const int* tile_off, int B, int T,
                         int U1, long long max_tiles, int dense, unsigned char* flags, int* sub_list, int* n_active,
                         cudaStream_t stream);
int launch_dense_logprobs(const float* logits, const int* targets, int tgt_ld, const int* T_len, const int* U_len,
                          int B, int T, int U1, int V, int blank, float* lp, float* lse, cudaStream_t stream);
int launch_dense_grads(const float* logits, const int* targets, int tgt_ld, const int* T_len, const int* U_len,
                       const float4* coef, int B, int T, int U1, int V, int blank, float clamp, float* grads,
                       cudaStream_t stream);
int launch_joint_argmax(const float* enc_rows, long long enc_stride, const float* pred_rows, long long pred_stride,
                        const float* W, const float* bias, int N, int H, int V, int* tokens, float* top2,
                        float* scratch, cudaStream_t stream);
size_t joint_argmax_scratch_bytes(int N, int V);

// pre-projection GEMMs (linear_gemm.cu): y = x W^T + b and its backward, fp16 operands / fp32 accumulate
size_t linear_workspace_bytes(long long M, int K, int N, bool backward, bool deterministic);
int launch_linear_fwd(const float* x, const float* W, const float* bias, long long M, int K, int N, float* y,
                      void* workspace, cudaStream_t stream);
int launch_linear_bwd(const float* x, const float* W, const float* dy, long long M, int K, int N, float* dx, float* dW,
                      float* db, bool deterministic, void* workspace, cudaStream_t stream);

}  // namespace rb
