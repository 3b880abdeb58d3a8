/* rnnt_b200 -- C ABI of the B200 (sm_100a) joint-network + transducer-loss hot path.
 *
 * Drop-in boundary for the reference's Python-level interface (jakepoz/rnnt has no FFI of its own):
 *   rnnt/joint.py:25-39   JointNetwork.forward            -> rnnt_b200_joint_loss_fwd/bwd (fused, no logits)
 *   rnnt/joint.py:44-55   JointNetwork.single_forward     -> rnnt_b200_joint_argmax (decode step)
 *   rnnt/model.py:35-41   torchaudio.functional.rnnt_loss -> rnnt_b200_joint_loss_fwd/bwd, or
 *                                                            rnnt_b200_loss_dense_fwd/bwd when logits exist
 *   rnnt/model.py:66-69, 110-113  joint step + argmax of greedy decode -> rnnt_b200_joint_argmax
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless stated otherwise; the caller owns every buffer, including the
 *     workspace.  The library allocates nothing persistent and keeps no references after a call returns.
 *   - Work is enqueued on `stream` (a cudaStream_t); no call synchronises the device.  Re-entrant.
 *   - Return 0 on success, a negative code for invalid arguments / unsupported shapes (no CPU fallback:
 *     unsupported means error), a positive cudaError_t value for CUDA failures.
 *     rnnt_b200_last_error() returns the message for the calling thread.
 *   - Lattice tensors use the reference layout: (B, T, U1) row-major with U1 = max target length + 1;
 *     targets are (B, U1-1) int32; lengths are int32; blank < 0 means V + blank (the reference passes -1).
 */
#ifndef RNNT_B200_H_
#define RNNT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RNNT_B200_ABI_VERSION 3

/* `flags` of rnnt_b200_joint_loss_bwd / rnnt_b200_workspace_bytes */
#define RNNT_B200_ALL_TILES 1      /* process every half-tile, also those whose fp16 logit-gradients are all zero */
#define RNNT_B200_DETERMINISTIC 2  /* cross-CTA sums in 64-bit fixed point: bit-identical gradients run to run */

int rnnt_b200_abi_version(void);
const char* rnnt_b200_last_error(void);

/* Upper bound on the number of 128-row GEMM units (= pairs of 16(t) x 4(u) half-tiles) of a (B,T,U1) batch. */
int64_t rnnt_b200_max_tiles(int B, int T, int U1);

/* Size in bytes of the optional activation residual `hidden`: h = tanh(enc + pred) as fp16, one 64-row block per
 * half-tile of 16(t) x 4(u) lattice cells (row r = cell (t0 + r/4, u0 + r%4); half-tiles are numbered utterance by
 * utterance, t-block by t-block, u-block by u-block), rows padded to a multiple of 64 hidden units.  The reference's autograd saves the same tensor in fp32
 * (rnnt/joint.py:37).  With it the backward does not recompute the tanh; without it (NULL) it does. */
size_t rnnt_b200_hidden_bytes(int B, int T, int U1, int H);

/* Workspace sizes in bytes.  ring_tiles = number of 128-cell tiles the backward's 16-bit gradient (and, without a
 * hidden residual, activation) ring holds at once (fixed size, independent of B*T*U1); the backward walks the batch in
 * chunks of that size.  have_hidden = 1 if `hidden` will be passed to the calls (smaller workspaces).  flags = the
 * flags the backward will be called with (RNNT_B200_DETERMINISTIC adds 8 bytes per gradient element). */
int rnnt_b200_workspace_bytes(int B, int T, int U1, int H, int V, int64_t ring_tiles, int have_hidden, int flags,
                              size_t* fwd_bytes, size_t* bwd_bytes);

/* Fused joint + loss forward.  Replaces rnnt/joint.py:25-39 followed by rnnt/model.py:35-41 (reduction="none").
 *   enc  (B,T,H) fp32 with element strides (enc_sb, enc_st, enc_sh): either H-contiguous (enc_sh = 1, enc_sb and
 *        enc_st multiples of 4) or T-contiguous (enc_st = 1) -- the permuted view of the encoder's (B,H,T) output
 *        that rnnt/model.py:27-28 hands to the joint; it is read in place, no transposed copy is made
 *   pred (B,U1,H) fp32 contiguous     W (V,H) fp32 (joint_ln.weight)     bias (V) fp32 (joint_ln.bias)
 * Outputs (all fully written for valid cells): costs (B), lp (B,T,U1,2) = log p(blank), log p(label),
 * lse (B,T,U1), alpha (B,T,U1), beta (B,T,U1).  These five are the residuals the backward consumes.
 * hidden (optional, rnnt_b200_hidden_bytes, 128-byte aligned): receives the fp16 activations for the backward; NULL
 * keeps them in a small per-SM scratch inside the workspace (loss-only evaluation, or a recomputing backward).
 * status (optional, may be NULL): device int set to 1 if any length is out of range (T_b outside [1,T], U_b outside
 * [0,U1-1]; torchaudio raises for these).  Independently of `status`, every cost is NaN in that case. */
int rnnt_b200_joint_loss_fwd(const float* enc, int64_t enc_sb, int64_t enc_st, int64_t enc_sh, const float* pred,
                             const float* W, const float* bias, const int32_t* targets, const int32_t* T_len,
                             const int32_t* U_len, int B, int T, int U1, int H, int V, int blank, float* costs,
                             float* lp, float* lse, float* alpha, float* beta, void* hidden, int32_t* status,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Fused backward.  Replaces RnntLoss.backward + autograd through rnnt/joint.py:32-39 (SURVEY 8a-6, 8a-8).
 * dcost (B) = d loss / d cost_b (1/B for reduction="mean"); clamp <= 0 disables gradient clamping.
 * hidden = the buffer the forward filled, or NULL to recompute the activations (memory-lean mode).
 * Outputs are overwritten, all fp32: d_enc = a dense (B,T,H) tensor (strides (T*H, H, 1)) or a dense (B,H,T) tensor
 * viewed as (B,T,H) (strides (T*H, 1, T): the gradient lands in the encoder's own layout), d_pred (B,U1,H), dW (V,H),
 * dbias (V) -- dW / dbias may point into a flat all-reduce bucket.
 * Half-tiles (16 t x 4 u lattice blocks) whose logit-gradients are all at most 2^-25 of max|dcost| are skipped: they
 * are left out of the work list, so they add nothing to d_enc, d_pred, dW and dbias, although their gradients need not
 * be zero.  The work list holds, in order, exactly the half-tiles with a valid cell whose gradient coefficients exceed
 * that bound; RNNT_B200_ALL_TILES disables the skipping.
 * RNNT_B200_DETERMINISTIC replaces the fp32 atomics (d_enc, d_pred, dW, dbias are sums over CTAs) by 64-bit
 * fixed-point accumulation, which is order-independent: gradients are bit-identical from run to run.
 * dw_done_event (optional cudaEvent_t, may be NULL) is recorded on `stream` as soon as dW and dbias are final, before
 * the activation-gradient GEMM of the last chunk is enqueued, so a data-parallel caller can overlap the all-reduce of
 * the weight gradients (rnnt/train.py:67-68 DDP) with the rest of the backward. */
int rnnt_b200_joint_loss_bwd(const float* enc, int64_t enc_sb, int64_t enc_st, int64_t enc_sh, const float* pred,
                             const float* W, const float* bias, const int32_t* targets, const int32_t* T_len,
                             const int32_t* U_len, int B, int T, int U1, int H, int V, int blank, const float* lp,
                             const float* lse, const float* alpha, const float* beta, const void* hidden,
                             const float* dcost, float clamp, float* d_enc, int64_t denc_sb, int64_t denc_st,
                             int64_t denc_sh, float* d_pred, float* dW, float* dbias, int64_t ring_tiles, int flags,
                             void* dw_done_event, void* workspace, size_t workspace_bytes, void* stream);

/* Loss on already materialised logits (B,T,U1,V) fp32 contiguous -- the literal torchaudio.functional.rnnt_loss
 * call of rnnt/model.py:35-41 for callers that hold logits (e.g. eval.py:76 style uses).  fwd writes costs and the
 * residuals; bwd writes grads (B,T,U1,V) = d loss / d logits (zeros on padding).  scratch_coef: (B,T,U1,4) fp32. */
int rnnt_b200_loss_dense_fwd(const float* logits, const int32_t* targets, const int32_t* T_len, const int32_t* U_len,
                             int B, int T, int U1, int V, int blank, float* costs, float* lp, float* lse,
                             float* alpha, float* beta, void* stream);
int rnnt_b200_loss_dense_bwd(const float* logits, const int32_t* targets, const int32_t* T_len, const int32_t* U_len,
                             int B, int T, int U1, int V, int blank, const float* lp, const float* lse,
                             const float* alpha, const float* beta, const float* dcost, float clamp,
                             float* scratch_coef, float* grads, void* stream);

/* Lattice only: alpha/beta/costs from log-probs (B,T,U1,2). */
int rnnt_b200_lattice(const float* lp, const int32_t* T_len, const int32_t* U_len, int B, int T, int U1, float* alpha,
                      float* beta, float* costs, void* stream);

/* Greedy-decode joint step (fp32): tokens[n] = argmax_v(W . tanh(enc_rows[n] + pred_rows[n]) + bias), lowest index
 * on ties; margin[n] (optional) = top1 - top2 logit.  Row n of enc_rows / pred_rows starts at n * stride floats.
 * scratch: rnnt_b200_joint_argmax_scratch_bytes(N, V) bytes. */
size_t rnnt_b200_joint_argmax_scratch_bytes(int N, int V);
int rnnt_b200_joint_argmax(const float* enc_rows, int64_t enc_stride, const float* pred_rows, int64_t pred_stride,
                           const float* W, const float* bias, int N, int H, int V, int32_t* tokens, float* margin,
                           void* scratch, void* stream);

/* Whole batched greedy decode in one persistent cooperative kernel (fp32).  Replaces the host loop of
 * rnnt/model.py:90-128 (_greedy_decode_conv) including the ConvPredictor re-run (rnnt/predictor.py:209-229), evaluated
 * incrementally (the predictor is causal with a 7-token receptive field).  enc (B,T,H) are the encoder features,
 * T_len (B) their lengths; conv1_w / conv2_w are the Conv1d weights re-laid as (E, 3E) / (E, 5E) with taps ordered
 * oldest..newest (weight.permute(0,2,1).reshape(E,-1)); every other parameter is the module's tensor as is.
 * tokens (B, max_len) int32 receives the emitted tokens, n_tokens (B) = 1 + their count (the seed blank is counted,
 * as rnnt/model.py:53,64 does).  margins_out (optional, (T+max_len+2, B) fp32, caller-initialised) receives the top-2
 * logit gap at [step, b] for every step utterance b was active in.  scratch: rnnt_b200_greedy_decode_scratch_bytes
 * bytes, 128-byte aligned (it also holds two per-symbol tables built at kernel start: LayerNorm(embedding), (V, E), and
 * conv1's tap products of it, (V, 3E) floats); its first 64 bytes return eight int64 counters of CTA 0 (cycles of
 * phases P1, P2, P3, the one-off conv1 table build, P5, P6, joint steps taken, cycles in grid barriers). */
size_t rnnt_b200_greedy_decode_scratch_bytes(int B, int H, int V, int E);
int rnnt_b200_greedy_decode(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* T_len,
                            const float* joint_w, const float* joint_b, const float* emb, const float* ln1_w,
                            const float* ln1_b, const float* conv1_w, const float* conv1_b, const float* conv2_w,
                            const float* conv2_b, const float* lin_w, const float* lin_b, const float* ln2_w,
                            const float* ln2_b, int B, int T, int H, int V, int E, int blank, int max_len,
                            int max_per_frame, int32_t* tokens, int32_t* n_tokens, float* margins_out, void* scratch,
                            void* stream);

/* Streaming greedy decode: the loop of rnnt_b200_greedy_decode fed one chunk of encoder frames per call, for B slots
 * (one live stream each) whose decoder state outlives the call.  Decoding an utterance in any sequence of consecutive
 * chunks (zero-length ones included, other slots reset or fed in between, any slot, any B) gives the same tokens and
 * per-step margins, bit for bit, as rnnt_b200_greedy_decode on the whole utterance with the same max_len and
 * max_per_frame.
 *
 * state: rnnt_b200_greedy_decode_state_bytes(B, H, V, E) bytes, caller-owned, 128-byte aligned; its layout is that of
 * the one-shot scratch.  It holds, per slot: the token count n (0 = empty slot, else 1 + tokens emitted, which is the
 * predictor's next input position), the emit flag, the linear output `lin` and LayerNorm'd predictor features `feats`
 * (H each), and the conv tap accumulators of conv1 (3E) and conv2 (5E); plus the two per-symbol tables
 * (LayerNorm(embedding) (V, E) and conv1's tap products (V, 3E)) and the per-call scratch (frame counters, row lists,
 * joint hidden rows, logits, conv outputs).  Its first 64 bytes hold the eight int64 counters of the last call, as for
 * the one-shot scratch.
 *
 * rnnt_b200_greedy_decode_stream_init builds the symbol tables from the weights and empties every slot.  Run it
 * before the first call and again whenever the weights change.
 *
 * rnnt_b200_greedy_decode_stream consumes enc (B, Tc, H) fp32 (strides (enc_sb, enc_st, 1), multiples of 4): slot b
 * takes the first chunk_len[b] frames (clamped to [0, Tc]).  Slots with reset[b] != 0 (reset may be NULL) start a new
 * utterance first: predictor state zeroed, the seed blank run through the predictor, n = 1 (the seed is counted, as
 * rnnt/model.py:53,64 does).  Every other non-empty slot continues where its last call stopped, with the rule of
 * rnnt/model.py:108-123.  A slot is finished when n == max_len and ignores frames until it is reset; empty slots
 * ignore frames too.  A call always leaves a slot on a frame boundary (a frame is only left after a blank or the
 * max_per_frame cap), so no per-frame counter crosses calls.  tokens (B, max_len) int32, caller-owned and kept
 * between calls: the k-th token of the slot's utterance goes to column k-1, so this call added
 * tokens[b, n_before-1 : n_after-1] (n_before = 1 for a reset slot).  n_tokens (B) int32 receives n after the call.
 * margins_out (optional, (Tc + min(Tc * max_per_frame, max_len - 1) + 1, B) fp32, caller-initialised) receives the
 * top-2 logit gap at [step, b] for every step of this call slot b was active in (steps 0, 1, ... of the call).
 * Use the same max_len and max_per_frame for every call of a state. */
size_t rnnt_b200_greedy_decode_state_bytes(int B, int H, int V, int E);
int rnnt_b200_greedy_decode_stream_init(const float* joint_w, const float* joint_b, const float* emb,
                                        const float* ln1_w, const float* ln1_b, const float* conv1_w,
                                        const float* conv1_b, const float* conv2_w, const float* conv2_b,
                                        const float* lin_w, const float* lin_b, const float* ln2_w, const float* ln2_b,
                                        int B, int H, int V, int E, void* state, void* stream);
int rnnt_b200_greedy_decode_stream(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* chunk_len,
                                   const int32_t* reset, const float* joint_w, const float* joint_b, const float* emb,
                                   const float* ln1_w, const float* ln1_b, const float* conv1_w, const float* conv1_b,
                                   const float* conv2_w, const float* conv2_b, const float* lin_w, const float* lin_b,
                                   const float* ln2_w, const float* ln2_b, int B, int Tc, int H, int V, int E,
                                   int blank, int max_len, int max_per_frame, int32_t* tokens, int32_t* n_tokens,
                                   float* margins_out, void* state, void* stream);

/* Optional pre-projections of the joint (rnnt/joint.py:8-12, 26-30: audio_ln / text_ln of the non-"convjs" configs) as
 * tcgen05 GEMMs ahead of the fused call, with their backward.  Row-major contiguous fp32 tensors:
 *   fwd:  y[M,N] = x[M,K] . W[N,K]^T + bias[N]        (M = B*T or B*U1 rows, K = in features, N = hidden_features)
 *   bwd:  dx[M,K] = dy . W,  dW[N,K] = dy^T . x,  db[N] = column sums of dy;  any of dx / dW / db may be NULL (skipped)
 * Operands are rounded to fp16, accumulation is fp32.  K and N must be multiples of 8.  flags: RNNT_B200_DETERMINISTIC.
 * workspace: rnnt_b200_linear_workspace_bytes(M, K, N, backward, flags) bytes, 256-byte aligned. */
size_t rnnt_b200_linear_workspace_bytes(int64_t M, int K, int N, int backward, int flags);
int rnnt_b200_linear_fwd(const float* x, const float* W, const float* bias, int64_t M, int K, int N, float* y,
                         void* workspace, size_t workspace_bytes, void* stream);
int rnnt_b200_linear_bwd(const float* x, const float* W, const float* dy, int64_t M, int K, int N, float* dx,
                         float* dW, float* db, int flags, void* workspace, size_t workspace_bytes, void* stream);

/* Opt-in measurement hook (bench.py): between begin and end every kernel launch of the library is bracketed by
 * CUDA events on its launch stream.  end() synchronises on those events and returns, per kernel family, the summed
 * device time in ms and the number of launches.  HOST pointers.  Families: 0 prep (tile table, weight conversion,
 * gradient coefficients), 1 joint GEMM forward, 2 lattice, 3 joint GEMM backward-recompute, 4 dh GEMM, 5 dW GEMM,
 * 6 db, 7 other (dense-logits kernels, decode). */
int rnnt_b200_profile_begin(void);
int rnnt_b200_profile_end(float* ms /*[8]*/, int64_t* launches /*[8]*/);

/* Test hook: byte offsets of the workspace regions so tests can inspect the rings after a backward call:
 *   offsets[0] tile table: B+1 int32 prefix sums of half-tiles per utterance, status, {S, 1/S} (fp32), n_active half-tiles
 *   offsets[1] W as fp16 [Vp, Hp] (zero padded)       offsets[2] bias * log2(e) [Vp] (padding = -1e30)
 *   offsets[3] gradient coefficients (B,T,U1,4) fp32   offsets[4] gradient ring g [ring_tiles*128, Vp] fp16
 *   offsets[5] activation ring h [ring_tiles*128, Hp] fp16 (-1 with have_hidden)
 *   offsets[6] bytes that satisfy both the forward and the backward call (any flags)
 *   offsets[7] work list of active half-tiles (int32 ids); ring rows [64 i, 64 i + 64) = entry i.
 * Hp / Vp = H / V rounded up to multiples of 64 / 256. */
int rnnt_b200_debug_ws_layout(int B, int T, int U1, int H, int V, int64_t ring_tiles, int have_hidden,
                              int64_t* offsets /*[8]*/, int* Hp, int* Vp);

#ifdef __cplusplus
}
#endif
#endif /* RNNT_B200_H_ */
