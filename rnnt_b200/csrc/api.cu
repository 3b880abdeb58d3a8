// C-ABI entry points (see include/rnnt_b200.h).  Plain pointers and sizes only; every buffer is caller-owned.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>

#include "../../include/rnnt_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace {

using rb::kTileM;

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Diagnostic knobs (read once per process), which exist to measure what parts of a kernel cost:
//   RNNT_B200_DBG      bit mask handed to the joint kernels (1 skip epilogue math, 2 skip producer math, 8 print grids, ...)
//   RNNT_B200_NO_DB    leave db out of the dW kernel (db is then NOT computed)
struct EnvKnobs { int dbg; bool no_db; };
const EnvKnobs& env_knobs() {
  static const EnvKnobs k = [] {
    EnvKnobs e{};
    const char* s = getenv("RNNT_B200_DBG");      e.dbg = s ? atoi(s) : 0;
    e.no_db = getenv("RNNT_B200_NO_DB") != nullptr;
    return e;
  }();
  return k;
}
inline int round_up(int x, int a) { return (x + a - 1) / a * a; }

struct WsLayout {
  size_t tile_off, status, gscale, n_active, wb, bias2, h_scratch, coef, flags, tile_list, g_ring, h_ring, fx, total_fwd,
      total_bwd;
  int Hp, Vp, scratch_tiles;
};

// have_hidden: the caller supplies the activation residual buffer (rnnt_b200_hidden_bytes).  Then the forward needs
// no per-CTA activation scratch and the backward ring holds the logit-gradients only.
WsLayout ws_layout(int B, int T, int U1, int H, int V, int64_t ring_tiles, bool have_hidden, bool deterministic = false) {
  WsLayout w;
  w.Hp = round_up(H, 64);
  w.Vp = round_up(V, 256);
  size_t off = 0;
  // tile-table region (documented in rnnt_b200.h): B+1 prefix sums, then status, {S, 1/S}, n_active and one spare word
  w.tile_off = off;
  w.status = w.tile_off + (static_cast<size_t>(B) + 1) * sizeof(int);
  w.gscale = w.status + sizeof(int);
  w.n_active = w.gscale + 2 * sizeof(float);
  off = align_up(w.n_active + 2 * sizeof(int), 1024);
  w.wb = off;       off = align_up(off + static_cast<size_t>(w.Vp) * w.Hp * 2, 1024);
  w.bias2 = off;    off = align_up(off + static_cast<size_t>(w.Vp) * 4, 1024);
  const size_t common = off;
  w.scratch_tiles = have_hidden ? 0 : rb::joint_gemm_scratch_tiles(rb::device_sm_count());
  w.h_scratch = off; off = align_up(off + static_cast<size_t>(w.scratch_tiles) * kTileM * w.Hp * 2, 1024);
  w.total_fwd = off;
  off = common;      // the backward re-uses the region after the converted weights
  w.coef = off;     off = align_up(off + static_cast<size_t>(B) * T * U1 * 16, 1024);
  const size_t max_tiles = static_cast<size_t>(B) * ((T + rb::kTileT - 1) / rb::kTileT) * ((U1 + rb::kTileU - 1) / rb::kTileU);
  w.flags = off;    off = align_up(off + 2 * max_tiles, 1024);                     // one per half-tile
  w.tile_list = off; off = align_up(off + 2 * max_tiles * sizeof(int), 1024);     // work list of half-tile ids
  const size_t ring_rows = static_cast<size_t>(ring_tiles) * kTileM;
  w.g_ring = off;   off = align_up(off + ring_rows * w.Vp * 2, 1024);
  w.h_ring = off;   off = align_up(off + (have_hidden ? 0 : ring_rows * w.Hp * 2), 1024);
  // deterministic mode: int64 fixed-point accumulators for d_enc (B,T,H), d_pred (B,U1,H), dW (V,H), db (V)
  const size_t fx_elems = static_cast<size_t>(B) * T * H + static_cast<size_t>(B) * U1 * H + static_cast<size_t>(V) * H + V;
  w.fx = off;       off = align_up(off + (deterministic ? fx_elems * 8 : 0), 1024);
  w.total_bwd = off;
  return w;
}

// Encoder-feature layouts the kernels read directly (element strides of the logical (B,T,H) tensor):
//   H-contiguous: (sb, st >= H, 1), sb and st multiples of 4 (16-byte vector loads), or
//   T-contiguous: (sb, 1, sh >= T) -- the permuted view of the encoder's (B,H,T) output, rnnt/model.py:28.
int check_layout(const char* what, int64_t& sb, int64_t& st, int64_t& sh, int B, int T, int H) {
  if (sh == 1) {
    if (T == 1) st = H;                        // strides of size-1 dimensions carry no information
    if (B == 1) sb = static_cast<int64_t>(T) * st;
    RB_REQUIRE(st % 4 == 0 && sb % 4 == 0 && st >= H, -3,
               "%s: H-contiguous layout needs strides (sb, st >= H, 1) that are multiples of 4 elements", what);
    return 0;
  }
  if (T == 1) st = 1;
  if (B == 1) sb = static_cast<int64_t>(H) * sh;
  RB_REQUIRE(st == 1 && sh >= T, -3,
             "%s must be contiguous in the feature dimension (B,T,H) or in the time dimension (view of (B,H,T))", what);
  return 0;
}

int check_common(const void* enc, int64_t& enc_sb, int64_t& enc_st, int64_t& enc_sh, const void* pred, int B, int T,
                 int U1, int H, int V, int* blank) {
  RB_REQUIRE(B > 0 && T > 0 && U1 > 0 && H > 0 && V > 1, -1, "invalid shape B=%d T=%d U1=%d H=%d V=%d", B, T, U1, H, V);
  RB_REQUIRE(H % 8 == 0, -2, "hidden_features must be a multiple of 8 (got %d)", H);
  RB_REQUIRE(U1 <= 1024, -5, "U+1 must be <= 1024 (got %d)", U1);
  RB_REQUIRE((reinterpret_cast<uintptr_t>(enc) & 15) == 0 && (reinterpret_cast<uintptr_t>(pred) & 15) == 0, -3,
             "enc/pred must be 16-byte aligned");
  if (int rc = check_layout("audio features", enc_sb, enc_st, enc_sh, B, T, H)) return rc;
  if (*blank < 0) *blank += V;
  RB_REQUIRE(*blank >= 0 && *blank < V, -4, "blank index out of range");
  return 0;
}

// What the backward passes to the prologue beyond the forward's arguments (check_layout normalises the d_enc strides in
// place, as it does the encoder's).
struct BwdArgs {
  const float* d_enc;
  int64_t &denc_sb, &denc_st, &denc_sh;
  int64_t ring_tiles;
  bool deterministic;
  const float* dcost;
};

// One call of a fused-loss entry as its prologue leaves it: the workspace (offsets: ws_layout) carved into typed
// pointers, the tensor map over the fp16 W, and the batch fields of the kernel arguments.
struct LossCall {
  WsLayout w;
  int* tile_off;          // [B+1] prefix sums of half-tiles per utterance
  int* status;            // non-zero when a length is out of range
  float* gscale;          // backward: {S, 1/S}
  int* n_active;          // backward: number of active half-tiles in sub_list
  __half* Wb;             // W as fp16 [Vp, Hp], zero-padded
  float* bias2;           // [Vp]
  __half* h_scratch;      // forward without a residual buffer: per-CTA activation rows
  float4* coef;           // backward (the regions from here on reuse the forward's h_scratch): (B,T,U1) coefficients
  unsigned char* flags;   // one per half-tile: active in the backward
  int* sub_list;          // work list of active half-tiles, order preserved
  __half* g_ring;         // logit gradients of one chunk of the work list
  __half* h_ring;         // activations of that chunk, recomputed when the caller keeps no residual buffer
  long long *fx_enc, *fx_pred, *fx_w, *fx_b;   // deterministic mode: fixed-point shadows of d_enc, d_pred, dW, db
  CUtensorMap tmW;        // fp16 W, 64(k) x 128(v) boxes
  rb::BatchArgs base;
};

// The part both fused-loss entries share (bwd == nullptr for the forward): check every argument before anything touches
// a device, carve the workspace, enqueue the tile table and the fp16 copy of W, build the tensor map over that copy,
// and fill the batch fields of the kernel arguments.
int loss_prologue(LossCall& c, const float* enc, int64_t enc_sb, int64_t enc_st, int64_t enc_sh, const float* pred,
                  const float* W, const float* bias, const int32_t* targets, const int32_t* T_len,
                  const int32_t* U_len, int B, int T, int U1, int H, int V, int blank, const void* hidden,
                  BwdArgs* bwd, int32_t* err_flag, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  int rc = check_common(enc, enc_sb, enc_st, enc_sh, pred, B, T, U1, H, V, &blank);
  if (rc) return rc;
  RB_REQUIRE((reinterpret_cast<uintptr_t>(W) & 15) == 0, -3, "W must be 16-byte aligned");
  RB_REQUIRE((reinterpret_cast<uintptr_t>(hidden) & 127) == 0, -3, "hidden must be 128-byte aligned");
  if (bwd) {
    rc = check_layout("d_enc", bwd->denc_sb, bwd->denc_st, bwd->denc_sh, B, T, H);
    if (rc) return rc;
    RB_REQUIRE((reinterpret_cast<uintptr_t>(bwd->d_enc) & 15) == 0, -3, "d_enc must be 16-byte aligned");
    const int64_t TH = static_cast<int64_t>(T) * H;
    RB_REQUIRE((bwd->denc_sh == 1 && bwd->denc_st == H && bwd->denc_sb == TH) ||
                   (bwd->denc_st == 1 && bwd->denc_sh == T && bwd->denc_sb == TH),
               -3, "d_enc must be a dense (B,T,H) tensor or a dense (B,H,T) tensor viewed as (B,T,H)");
    RB_REQUIRE(bwd->ring_tiles >= 1 && bwd->ring_tiles * kTileM < (1ll << 30), -8, "ring_tiles out of range");
  }
  const bool deterministic = bwd && bwd->deterministic;
  const WsLayout& w = c.w = ws_layout(B, T, U1, H, V, bwd ? bwd->ring_tiles : 0, hidden != nullptr, deterministic);
  const size_t need = bwd ? w.total_bwd : w.total_fwd;
  RB_REQUIRE(workspace != nullptr && workspace_bytes >= need, -7, "workspace too small: need %zu bytes", need);
  RB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, -7, "workspace must be 256-byte aligned");

  uint8_t* p = static_cast<uint8_t*>(workspace);
  c.tile_off = reinterpret_cast<int*>(p + w.tile_off);
  c.status = reinterpret_cast<int*>(p + w.status);
  c.gscale = reinterpret_cast<float*>(p + w.gscale);
  c.n_active = reinterpret_cast<int*>(p + w.n_active);
  c.Wb = reinterpret_cast<__half*>(p + w.wb);
  c.bias2 = reinterpret_cast<float*>(p + w.bias2);
  c.h_scratch = reinterpret_cast<__half*>(p + w.h_scratch);
  c.coef = reinterpret_cast<float4*>(p + w.coef);
  c.flags = p + w.flags;
  c.sub_list = reinterpret_cast<int*>(p + w.tile_list);
  c.g_ring = reinterpret_cast<__half*>(p + w.g_ring);
  c.h_ring = reinterpret_cast<__half*>(p + w.h_ring);
  if (deterministic) {   // d_enc (B,T,H), d_pred (B,U1,H), dW (V,H), db (V)
    c.fx_enc = reinterpret_cast<long long*>(p + w.fx);
    c.fx_pred = c.fx_enc + static_cast<size_t>(B) * T * H;
    c.fx_w = c.fx_pred + static_cast<size_t>(B) * U1 * H;
    c.fx_b = c.fx_w + static_cast<size_t>(V) * H;
  }

  rc = rb::launch_tile_table(T_len, U_len, B, T, U1, c.tile_off, c.status, err_flag, bwd ? bwd->dcost : nullptr,
                             bwd ? c.gscale : nullptr, stream);
  if (rc) return rc;
  rc = rb::launch_convert_weights(W, bias, V, H, w.Vp, w.Hp, c.Wb, c.bias2, stream);
  if (rc) return rc;
  rc = rb::make_tmap_2d(&c.tmW, c.Wb, 2, w.Hp, w.Vp, static_cast<uint64_t>(w.Hp) * 2, 64, 128);
  if (rc) return rc;

  rb::BatchArgs& a = c.base;
  a.enc = enc; a.enc_sb = enc_sb; a.enc_st = enc_st; a.enc_sh = enc_sh;
  a.pred = pred; a.pred_sb = static_cast<long long>(U1) * H; a.pred_su = H;
  a.bias2 = c.bias2; a.targets = targets; a.tgt_ld = U1 - 1;
  a.T_len = T_len; a.U_len = U_len; a.tile_off = c.tile_off;
  a.B = B; a.T = T; a.U1 = U1; a.H = H; a.Hp = w.Hp; a.V = V; a.Vp = w.Vp; a.blank = blank;
  // the forward covers every half-tile from slot 0 in one launch; the backward walks its work list a ring at a time
  a.slot_cap = bwd ? static_cast<int>(2 * bwd->ring_tiles) : 0x3fffffff;
  a.sub_list = bwd ? c.sub_list : nullptr;
  a.n_active = bwd ? c.n_active : nullptr;
  a.gscale = bwd ? c.gscale : nullptr;
  a.h_map = hidden ? 0 : bwd ? 1 : 2;
  return 0;
}

// An fp16 [rows, cols] buffer of activations (cols = Hp) or logit gradients (cols = Vp) in boxes 64 columns wide: 64 rows
// (one half-tile) and 128 rows (two adjacent ones)
int make_row_maps(CUtensorMap* m64, CUtensorMap* m128, const __half* buf, uint64_t rows, int cols) {
  int rc = rb::make_tmap_2d(m64, buf, 2, cols, rows, static_cast<uint64_t>(cols) * 2, 64, 64);
  if (rc) return rc;
  return rb::make_tmap_2d(m128, buf, 2, cols, rows, static_cast<uint64_t>(cols) * 2, 64, 128);
}

}  // namespace

extern "C" {

int rnnt_b200_abi_version(void) { return RNNT_B200_ABI_VERSION; }
const char* rnnt_b200_last_error(void) { return rb::get_error(); }

int64_t rnnt_b200_max_tiles(int B, int T, int U1) {
  return static_cast<int64_t>(B) * ((T + rb::kTileT - 1) / rb::kTileT) * ((U1 + rb::kTileU - 1) / rb::kTileU);
}

size_t rnnt_b200_hidden_bytes(int B, int T, int U1, int H) {
  if (B <= 0 || T <= 0 || U1 <= 0 || H <= 0) return 0;
  return static_cast<size_t>(rnnt_b200_max_tiles(B, T, U1)) * kTileM * round_up(H, 64) * 2;
}

int rnnt_b200_workspace_bytes(int B, int T, int U1, int H, int V, int64_t ring_tiles, int have_hidden, int flags,
                              size_t* fwd_bytes, size_t* bwd_bytes) {
  RB_REQUIRE(B > 0 && T > 0 && U1 > 0 && H > 0 && V > 1 && ring_tiles >= 0, -1, "invalid shape");
  const WsLayout w = ws_layout(B, T, U1, H, V, ring_tiles, have_hidden != 0, (flags & RNNT_B200_DETERMINISTIC) != 0);
  if (fwd_bytes) *fwd_bytes = w.total_fwd;
  if (bwd_bytes) *bwd_bytes = w.total_bwd;
  return 0;
}

int rnnt_b200_debug_ws_layout(int B, int T, int U1, int H, int V, int64_t ring_tiles, int have_hidden,
                              int64_t* offsets, int* Hp, int* Vp) {
  const WsLayout w = ws_layout(B, T, U1, H, V, ring_tiles, have_hidden != 0, true);
  offsets[0] = w.tile_off; offsets[1] = w.wb; offsets[2] = w.bias2; offsets[3] = w.coef;
  offsets[4] = w.g_ring; offsets[5] = have_hidden ? -1 : static_cast<int64_t>(w.h_ring);
  offsets[6] = std::max(w.total_fwd, w.total_bwd); offsets[7] = w.tile_list;
  if (Hp) *Hp = w.Hp;
  if (Vp) *Vp = w.Vp;
  return 0;
}

int rnnt_b200_lattice(const float* lp, const int32_t* T_len, const int32_t* U_len, int B, int T, int U1, float* alpha,
                      float* beta, float* costs, void* stream) {
  RB_REQUIRE(B > 0 && T > 0 && U1 > 0, -1, "invalid shape");
  return rb::launch_lattice(lp, T_len, U_len, B, T, U1, alpha, beta, costs, nullptr, static_cast<cudaStream_t>(stream));
}

int rnnt_b200_viterbi(const float* lp, const int32_t* T_len, const int32_t* U_len, int B, int T, int U1,
                      int32_t* frames, float* scores, void* stream) {
  RB_REQUIRE(B > 0 && T > 0 && U1 > 0, -1, "invalid shape");
  RB_REQUIRE(scores != nullptr && (frames != nullptr || U1 == 1), -1,
             "viterbi: scores and (for U+1 > 1) frames are required");
  return rb::launch_viterbi(lp, T_len, U_len, B, T, U1, frames, scores, static_cast<cudaStream_t>(stream));
}

int rnnt_b200_joint_loss_fwd(const float* enc, int64_t enc_sb, int64_t enc_st, int64_t enc_sh, const float* pred,
                             const float* W, const float* bias, const int32_t* targets, const int32_t* T_len,
                             const int32_t* U_len, int B, int T, int U1, int H, int V, int blank, float* costs,
                             float* lp, float* lse, float* alpha, float* beta, void* hidden, int32_t* status,
                             void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  LossCall c{};
  int rc = loss_prologue(c, enc, enc_sb, enc_st, enc_sh, pred, W, bias, targets, T_len, U_len, B, T, U1, H, V, blank,
                         hidden, nullptr, status, workspace, workspace_bytes, stream);
  if (rc) return rc;

  const int64_t max_tiles = rnnt_b200_max_tiles(B, T, U1);
  // activation rows h = tanh(enc+pred): the caller's residual buffer (one 64-row block per half-tile) or a
  // small per-CTA scratch when no backward will follow
  __half* hbuf = hidden ? static_cast<__half*>(hidden) : c.h_scratch;
  const uint64_t hrows = static_cast<uint64_t>(hidden ? max_tiles : c.w.scratch_tiles) * kTileM;
  CUtensorMap tmH, tmH2;
  rc = make_row_maps(&tmH, &tmH2, hbuf, hrows, c.w.Hp);
  if (rc) return rc;

  rb::JointArgs a{c.base};
  a.lp = lp; a.lse = lse; a.h_out = hbuf;
  a.dbg = env_knobs().dbg;
  rc = rb::launch_joint_gemm(0, true, c.tmW, tmH, tmH2, a, 2 * max_tiles, stream);
  if (rc) return rc;
  return rb::launch_lattice(lp, T_len, U_len, B, T, U1, alpha, beta, costs, c.status, stream);
}

int rnnt_b200_joint_loss_bwd(const float* enc, int64_t enc_sb, int64_t enc_st, int64_t enc_sh, const float* pred,
                             const float* W, const float* bias, const int32_t* targets, const int32_t* T_len,
                             const int32_t* U_len, int B, int T, int U1, int H, int V, int blank, const float* lp,
                             const float* lse, const float* alpha, const float* beta, const void* hidden,
                             const float* dcost, float clamp, float* d_enc, int64_t denc_sb, int64_t denc_st,
                             int64_t denc_sh, float* d_pred, float* dW, float* dbias, int64_t ring_tiles, int flags,
                             void* dw_done_event, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool deterministic = (flags & RNNT_B200_DETERMINISTIC) != 0;
  BwdArgs bwd{d_enc, denc_sb, denc_st, denc_sh, ring_tiles, deterministic, dcost};
  LossCall c{};
  int rc = loss_prologue(c, enc, enc_sb, enc_st, enc_sh, pred, W, bias, targets, T_len, U_len, B, T, U1, H, V, blank,
                         hidden, &bwd, nullptr, workspace, workspace_bytes, stream);
  if (rc) return rc;

  // accumulation targets: the fp32 outputs themselves (atomics), or 64-bit fixed-point shadows (deterministic mode)
  const size_t n_enc = static_cast<size_t>(B) * T * H, n_pred = static_cast<size_t>(B) * U1 * H;
  const size_t n_w = static_cast<size_t>(V) * H;
  if (deterministic) {
    RB_CUDA_CHECK(cudaMemsetAsync(c.fx_enc, 0, (n_enc + n_pred + n_w + V) * 8, stream));
  } else {
    RB_CUDA_CHECK(cudaMemsetAsync(d_enc, 0, n_enc * 4, stream));
    RB_CUDA_CHECK(cudaMemsetAsync(d_pred, 0, n_pred * 4, stream));
    RB_CUDA_CHECK(cudaMemsetAsync(dW, 0, n_w * 4, stream));
    RB_CUDA_CHECK(cudaMemsetAsync(dbias, 0, static_cast<size_t>(V) * 4, stream));
  }

  const int64_t max_tiles = rnnt_b200_max_tiles(B, T, U1);
  rc = rb::launch_coef(lp, lse, alpha, beta, dcost, c.gscale, T_len, U_len, B, T, U1, c.coef, stream);
  if (rc) return rc;
  rc = rb::launch_tile_activity(c.coef, T_len, U_len, c.tile_off, B, T, U1, max_tiles,
                                (flags & RNNT_B200_ALL_TILES) ? 1 : 0, c.flags, c.sub_list, c.n_active, stream);
  if (rc) return rc;

  // activations: the forward's residual buffer (rows = half-tile id * 64) or, recomputed, a ring like g's
  const __half* h_src = hidden ? static_cast<const __half*>(hidden) : c.h_ring;
  const uint64_t ring_rows = static_cast<uint64_t>(ring_tiles) * kTileM;
  const uint64_t h_rows = hidden ? static_cast<uint64_t>(max_tiles) * kTileM : ring_rows;
  const int Hp = c.w.Hp, Vp = c.w.Vp;
  CUtensorMap tmWmn, tmHk, tmHk2, tmGmn, tmG128;
  // W [Vp, Hp]: MN-major boxes (64 k_h x 64 v) for dh.  Activations: the 64-row boxes serve as the K-major operand of
  // the logit recompute and the MN-major operand of dW.  Gradient ring: 64 x 128 K-major boxes for dh (two work-list
  // slots per CTA of a pair), 64 x 64 boxes for the MN-major dW operand
  rc = rb::make_tmap_2d(&tmWmn, c.Wb, 2, Hp, Vp, static_cast<uint64_t>(Hp) * 2, 64, 64);
  if (rc) return rc;
  rc = make_row_maps(&tmHk, &tmHk2, h_src, h_rows, Hp);
  if (rc) return rc;
  rc = make_row_maps(&tmGmn, &tmG128, c.g_ring, ring_rows, Vp);
  if (rc) return rc;

  // The work list is walked in chunks of as many slots (half-tiles of 64 rows) as the ring holds.  Per chunk: G (logit
  // recompute -> gradient ring), then dW/db, then dh -- the weight gradients come first so that, after the last chunk,
  // `dw_done_event` lets the caller start their all-reduce while the dh GEMM of that chunk is still running.
  const int64_t max_slots = 2 * max_tiles, ring_slots = 2 * ring_tiles;
  const int64_t nchunks = (max_slots + ring_slots - 1) / ring_slots;
  for (int64_t k = 0; k < nchunks; ++k) {
    c.base.slot_begin = static_cast<int>(k * ring_slots);
    const int64_t chunk_slots = std::min<int64_t>(ring_slots, max_slots - k * ring_slots);
    rb::JointArgs a{c.base};
    a.lp = const_cast<float*>(lp); a.coef = c.coef; a.dcost = dcost; a.clamp = clamp;
    a.h_out = const_cast<__half*>(h_src); a.g_ring = c.g_ring;
    a.dbg = env_knobs().dbg;
    rc = rb::launch_joint_gemm(1, hidden == nullptr, c.tmW, tmHk, tmHk2, a, chunk_slots, stream);
    if (rc) return rc;

    rb::DwArgs g{c.base};
    g.dW = dW; g.db = env_knobs().no_db ? nullptr : dbias; g.dW_fx = c.fx_w; g.db_fx = c.fx_b;
    rc = rb::launch_dw_gemm(tmGmn, tmHk, g, chunk_slots, stream);
    if (rc) return rc;
    if (k == nchunks - 1) {
      if (deterministic) {
        rc = rb::launch_finalize_fixed(c.fx_w, dW, 1, V, H, 0, H, 1, c.gscale, stream);
        if (rc) return rc;
        rc = rb::launch_finalize_fixed(c.fx_b, dbias, 1, 1, V, 0, 0, 1, c.gscale, stream);
        if (rc) return rc;
      }
      if (dw_done_event) RB_CUDA_CHECK(cudaEventRecord(static_cast<cudaEvent_t>(dw_done_event), stream));
    }

    rb::DhArgs d{c.base};
    d.d_enc = d_enc; d.denc_sb = denc_sb; d.denc_st = denc_st; d.denc_sh = denc_sh; d.d_pred = d_pred;
    d.d_enc_fx = c.fx_enc; d.d_pred_fx = c.fx_pred;
    rc = rb::launch_dh_gemm(tmG128, tmWmn, d, chunk_slots, stream);
    if (rc) return rc;
  }
  if (deterministic) {
    rc = rb::launch_finalize_fixed(c.fx_enc, d_enc, B, T, H, denc_sb, denc_st, denc_sh, c.gscale, stream);
    if (rc) return rc;
    rc = rb::launch_finalize_fixed(c.fx_pred, d_pred, 1, static_cast<long long>(B) * U1, H, 0, H, 1, c.gscale,
                                   stream);
    if (rc) return rc;
  }
  return 0;
}

int rnnt_b200_loss_dense_fwd(const float* logits, const int32_t* targets, const int32_t* T_len, const int32_t* U_len,
                             int B, int T, int U1, int V, int blank, float* costs, float* lp, float* lse,
                             float* alpha, float* beta, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  RB_REQUIRE(B > 0 && T > 0 && U1 > 0 && V > 1, -1, "invalid shape");
  RB_REQUIRE(U1 <= 1024, -5, "U+1 must be <= 1024 (got %d)", U1);
  if (blank < 0) blank += V;
  RB_REQUIRE(blank >= 0 && blank < V, -4, "blank index out of range");
  int rc = rb::launch_dense_logprobs(logits, targets, U1 - 1, T_len, U_len, B, T, U1, V, blank, lp, lse, stream);
  if (rc) return rc;
  return rb::launch_lattice(lp, T_len, U_len, B, T, U1, alpha, beta, costs, nullptr, stream);
}

int rnnt_b200_loss_dense_bwd(const float* logits, const int32_t* targets, const int32_t* T_len, const int32_t* U_len,
                             int B, int T, int U1, int V, int blank, const float* lp, const float* lse,
                             const float* alpha, const float* beta, const float* dcost, float clamp,
                             float* scratch_coef, float* grads, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  RB_REQUIRE(B > 0 && T > 0 && U1 > 0 && V > 1, -1, "invalid shape");
  if (blank < 0) blank += V;
  RB_REQUIRE(blank >= 0 && blank < V, -4, "blank index out of range");
  RB_REQUIRE((reinterpret_cast<uintptr_t>(scratch_coef) & 15) == 0, -3, "scratch_coef must be 16-byte aligned");
  // clamp acts on d cost / d logits before the dcost scaling (torchaudio ComputeGradients).
  RB_REQUIRE(!(clamp > 0.f && dcost != nullptr), -9,
             "dense backward: clamp > 0 requires dcost == NULL (scale the returned gradients by dcost instead)");
  float4* coef = reinterpret_cast<float4*>(scratch_coef);
  int rc = rb::launch_coef(lp, lse, alpha, beta, dcost, nullptr, T_len, U_len, B, T, U1, coef, stream);
  if (rc) return rc;
  return rb::launch_dense_grads(logits, targets, U1 - 1, T_len, U_len, coef, B, T, U1, V, blank, clamp, grads, stream);
}

size_t rnnt_b200_greedy_decode_scratch_bytes(int B, int H, int V, int E) {
  return rb::greedy_decode_scratch_bytes(B, H, V, E);
}

size_t rnnt_b200_greedy_decode_state_bytes(int B, int H, int V, int E) {
  if (B <= 0 || H <= 0 || V <= 1 || E <= 0) return 0;
  return rb::greedy_decode_scratch_bytes(B, H, V, E);
}

namespace {

// Arguments of the decode entries that are checked before anything touches a device.
int check_decode(int B, int T, int H, int V, int E, int blank, int max_len, int max_per_frame, int64_t enc_sb,
                 int64_t enc_st, const void* state) {
  RB_REQUIRE(B > 0 && T >= 0 && H > 0 && V > 1 && E > 0 && max_len >= 1 && max_per_frame >= 0, -1, "invalid shape");
  RB_REQUIRE(blank >= 0 && blank < V, -4, "blank index out of range");
  RB_REQUIRE(H % 4 == 0 && E % 4 == 0 && enc_st % 4 == 0 && enc_sb % 4 == 0, -2,
             "decode kernel needs hidden / embedding sizes and strides that are multiples of 4");
  RB_REQUIRE(state != nullptr && (reinterpret_cast<uintptr_t>(state) & 127) == 0, -3,
             "decode scratch must be 128-byte aligned");
  return 0;
}

rb::DecodeArgs decode_args(const float* joint_w, const float* joint_b, const float* emb, const float* ln1_w,
                           const float* ln1_b, const float* conv1_w, const float* conv1_b, const float* conv2_w,
                           const float* conv2_b, const float* lin_w, const float* lin_b, const float* ln2_w,
                           const float* ln2_b, int B, int H, int V, int E) {
  rb::DecodeArgs a{};
  a.Wj = joint_w; a.bj = joint_b; a.emb = emb; a.ln1_w = ln1_w; a.ln1_b = ln1_b;
  a.w1 = conv1_w; a.b1 = conv1_b; a.w2 = conv2_w; a.b2 = conv2_b; a.wl = lin_w; a.bl = lin_b;
  a.ln2_w = ln2_w; a.ln2_b = ln2_b;
  a.B = B; a.H = H; a.V = V; a.E = E; a.NS = V;
  return a;
}

}  // namespace

int rnnt_b200_greedy_decode_aligned(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* T_len,
                                    const float* joint_w, const float* joint_b, const float* emb, const float* ln1_w,
                                    const float* ln1_b, const float* conv1_w, const float* conv1_b,
                                    const float* conv2_w, const float* conv2_b, const float* lin_w, const float* lin_b,
                                    const float* ln2_w, const float* ln2_b, int B, int T, int H, int V, int E,
                                    int blank, int max_len, int max_per_frame, int32_t* tokens, int32_t* n_tokens,
                                    float* margins_out, void* scratch, void* stream, int32_t* frames,
                                    float* token_logp, float* scores) {
  RB_REQUIRE(T > 0, -1, "invalid shape");
  if (int rc = check_decode(B, T, H, V, E, blank, max_len, max_per_frame, enc_sb, enc_st, scratch)) return rc;
  // one launch: build the tables, reset every slot, consume the whole utterance
  rb::DecodeArgs a = decode_args(joint_w, joint_b, emb, ln1_w, ln1_b, conv1_w, conv1_b, conv2_w, conv2_b, lin_w, lin_b,
                                 ln2_w, ln2_b, B, H, V, E);
  a.enc = enc; a.enc_sb = enc_sb; a.enc_st = enc_st; a.T_len = T_len; a.T = T;
  a.init = 1; a.reset_all = 1; a.reset = nullptr;
  a.blank = blank; a.max_len = max_len; a.max_per_frame = max_per_frame; a.max_steps = T + max_len + 1;
  a.tokens = tokens; a.n_tokens = n_tokens; a.margins = margins_out;
  a.frames = frames; a.token_logp = token_logp; a.path_scores = scores;
  a.want_lp = token_logp != nullptr || scores != nullptr;
  return rb::launch_greedy_decode(a, static_cast<float*>(scratch), static_cast<cudaStream_t>(stream));
}

int rnnt_b200_greedy_decode(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* T_len,
                            const float* joint_w, const float* joint_b, const float* emb, const float* ln1_w,
                            const float* ln1_b, const float* conv1_w, const float* conv1_b, const float* conv2_w,
                            const float* conv2_b, const float* lin_w, const float* lin_b, const float* ln2_w,
                            const float* ln2_b, int B, int T, int H, int V, int E, int blank, int max_len,
                            int max_per_frame, int32_t* tokens, int32_t* n_tokens, float* margins_out, void* scratch,
                            void* stream) {
  return rnnt_b200_greedy_decode_aligned(enc, enc_sb, enc_st, T_len, joint_w, joint_b, emb, ln1_w, ln1_b, conv1_w,
                                         conv1_b, conv2_w, conv2_b, lin_w, lin_b, ln2_w, ln2_b, B, T, H, V, E, blank,
                                         max_len, max_per_frame, tokens, n_tokens, margins_out, scratch, stream,
                                         nullptr, nullptr, nullptr);
}

int rnnt_b200_greedy_decode_stream_init(const float* joint_w, const float* joint_b, const float* emb,
                                        const float* ln1_w, const float* ln1_b, const float* conv1_w,
                                        const float* conv1_b, const float* conv2_w, const float* conv2_b,
                                        const float* lin_w, const float* lin_b, const float* ln2_w, const float* ln2_b,
                                        int B, int H, int V, int E, void* state, void* stream) {
  if (int rc = check_decode(B, 0, H, V, E, 0, 1, 0, 0, 0, state)) return rc;
  rb::DecodeArgs a = decode_args(joint_w, joint_b, emb, ln1_w, ln1_b, conv1_w, conv1_b, conv2_w, conv2_b, lin_w, lin_b,
                                 ln2_w, ln2_b, B, H, V, E);
  a.init = 1; a.reset_all = 0; a.reset = nullptr;
  a.T = 0; a.max_len = 1; a.max_per_frame = 0; a.max_steps = 0;      // no slot is live: the step loop exits at once
  return rb::launch_greedy_decode(a, static_cast<float*>(state), static_cast<cudaStream_t>(stream));
}

int rnnt_b200_greedy_decode_stream_aligned(const float* enc, int64_t enc_sb, int64_t enc_st,
                                           const int32_t* chunk_len, const int32_t* reset, const float* joint_w,
                                           const float* joint_b, const float* emb, const float* ln1_w,
                                           const float* ln1_b, const float* conv1_w, const float* conv1_b,
                                           const float* conv2_w, const float* conv2_b, const float* lin_w,
                                           const float* lin_b, const float* ln2_w, const float* ln2_b, int B, int Tc,
                                           int H, int V, int E, int blank, int max_len, int max_per_frame,
                                           int32_t* tokens, int32_t* n_tokens, float* margins_out, void* state,
                                           void* stream, int32_t* frames, float* token_logp, float* scores) {
  if (int rc = check_decode(B, Tc, H, V, E, blank, max_len, max_per_frame, enc_sb, enc_st, state)) return rc;
  RB_REQUIRE(chunk_len != nullptr && tokens != nullptr && n_tokens != nullptr, -1,
             "decode stream: chunk_len, tokens and n_tokens are required");
  rb::DecodeArgs a = decode_args(joint_w, joint_b, emb, ln1_w, ln1_b, conv1_w, conv1_b, conv2_w, conv2_b, lin_w, lin_b,
                                 ln2_w, ln2_b, B, H, V, E);
  a.enc = enc; a.enc_sb = enc_sb; a.enc_st = enc_st; a.T_len = chunk_len; a.T = Tc;
  a.init = 0; a.reset_all = 0; a.reset = reset;
  a.blank = blank; a.max_len = max_len; a.max_per_frame = max_per_frame;
  // steps of one launch: every step of a slot either consumes a frame or emits a token
  a.max_steps = static_cast<int>(Tc + std::min<int64_t>(static_cast<int64_t>(Tc) * max_per_frame, max_len - 1) + 1);
  a.tokens = tokens; a.n_tokens = n_tokens; a.margins = margins_out;
  // the running path score lives in the state: every call keeps it, so plain and aligned calls can share a state
  a.frames = frames; a.token_logp = token_logp; a.path_scores = scores; a.want_lp = 1;
  return rb::launch_greedy_decode(a, static_cast<float*>(state), static_cast<cudaStream_t>(stream));
}

int rnnt_b200_greedy_decode_stream(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* chunk_len,
                                   const int32_t* reset, const float* joint_w, const float* joint_b, const float* emb,
                                   const float* ln1_w, const float* ln1_b, const float* conv1_w, const float* conv1_b,
                                   const float* conv2_w, const float* conv2_b, const float* lin_w, const float* lin_b,
                                   const float* ln2_w, const float* ln2_b, int B, int Tc, int H, int V, int E,
                                   int blank, int max_len, int max_per_frame, int32_t* tokens, int32_t* n_tokens,
                                   float* margins_out, void* state, void* stream) {
  return rnnt_b200_greedy_decode_stream_aligned(enc, enc_sb, enc_st, chunk_len, reset, joint_w, joint_b, emb, ln1_w,
                                                ln1_b, conv1_w, conv1_b, conv2_w, conv2_b, lin_w, lin_b, ln2_w, ln2_b,
                                                B, Tc, H, V, E, blank, max_len, max_per_frame, tokens, n_tokens,
                                                margins_out, state, stream, nullptr, nullptr, nullptr);
}

size_t rnnt_b200_beam_decode_scratch_bytes(int B, int K, int H, int V, int E, int max_len) {
  if (B <= 0 || K < 1 || K > rb::kMaxBeam || H <= 0 || V <= 1 || E <= 0 || max_len < 1) return 0;
  return rb::beam_decode_scratch_bytes(B, K, H, V, E, max_len);
}

int rnnt_b200_beam_decode_aligned(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* T_len,
                                  const float* joint_w, const float* joint_b, const float* emb, const float* ln1_w,
                                  const float* ln1_b, const float* conv1_w, const float* conv1_b, const float* conv2_w,
                                  const float* conv2_b, const float* lin_w, const float* lin_b, const float* ln2_w,
                                  const float* ln2_b, int B, int T, int H, int V, int E, int blank, int beam,
                                  int max_len, int32_t* tokens, int32_t* n_tokens, float* scores, void* scratch,
                                  void* stream, int32_t* frames, float* token_logp) {
  RB_REQUIRE(T > 0, -1, "invalid shape");
  if (int rc = check_decode(B, T, H, V, E, blank, max_len, 0, enc_sb, enc_st, scratch)) return rc;
  RB_REQUIRE(beam >= 1 && beam <= rb::kMaxBeam, -1, "beam size must be in [1, %d] (got %d)", rb::kMaxBeam, beam);
  RB_REQUIRE(tokens != nullptr && n_tokens != nullptr && scores != nullptr, -1,
             "beam decode: tokens, n_tokens and scores are required");
  rb::BeamArgs a{};
  static_cast<rb::DecodeArgs&>(a) = decode_args(joint_w, joint_b, emb, ln1_w, ln1_b, conv1_w, conv1_b, conv2_w, conv2_b,
                                                lin_w, lin_b, ln2_w, ln2_b, B, H, V, E);
  a.enc = enc; a.enc_sb = enc_sb; a.enc_st = enc_st; a.T_len = T_len; a.T = T;
  a.blank = blank; a.max_len = max_len; a.K = beam;
  a.tokens = tokens; a.n_tokens = n_tokens; a.scores = scores;
  a.frames = frames; a.token_logp = token_logp;
  return rb::launch_beam_decode(a, static_cast<float*>(scratch), static_cast<cudaStream_t>(stream));
}

int rnnt_b200_beam_decode(const float* enc, int64_t enc_sb, int64_t enc_st, const int32_t* T_len,
                          const float* joint_w, const float* joint_b, const float* emb, const float* ln1_w,
                          const float* ln1_b, const float* conv1_w, const float* conv1_b, const float* conv2_w,
                          const float* conv2_b, const float* lin_w, const float* lin_b, const float* ln2_w,
                          const float* ln2_b, int B, int T, int H, int V, int E, int blank, int beam, int max_len,
                          int32_t* tokens, int32_t* n_tokens, float* scores, void* scratch, void* stream) {
  return rnnt_b200_beam_decode_aligned(enc, enc_sb, enc_st, T_len, joint_w, joint_b, emb, ln1_w, ln1_b, conv1_w,
                                       conv1_b, conv2_w, conv2_b, lin_w, lin_b, ln2_w, ln2_b, B, T, H, V, E, blank,
                                       beam, max_len, tokens, n_tokens, scores, scratch, stream, nullptr, nullptr);
}

size_t rnnt_b200_linear_workspace_bytes(int64_t M, int K, int N, int backward, int flags) {
  if (M <= 0 || K <= 0 || N <= 0) return 0;
  return rb::linear_workspace_bytes(M, K, N, backward != 0, (flags & RNNT_B200_DETERMINISTIC) != 0);
}

namespace {
int check_linear(const void* x, const void* W, int64_t M, int K, int N, const void* workspace, size_t workspace_bytes,
                 size_t need) {
  RB_REQUIRE(M > 0 && M < (1ll << 31) && K > 0 && N > 0, -1, "invalid shape M=%lld K=%d N=%d", (long long)M, K, N);
  RB_REQUIRE(K % 8 == 0 && N % 8 == 0, -2, "pre-projection: in/out features must be multiples of 8 (got %d, %d)", K, N);
  RB_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(W)) & 15) == 0, -3,
             "pre-projection: x / W must be 16-byte aligned");
  RB_REQUIRE(workspace != nullptr && workspace_bytes >= need && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, -7,
             "pre-projection: workspace must be 256-byte aligned and hold %zu bytes", need);
  return 0;
}
}  // namespace

int rnnt_b200_linear_fwd(const float* x, const float* W, const float* bias, int64_t M, int K, int N, float* y,
                         void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_linear(x, W, M, K, N, workspace, workspace_bytes, rb::linear_workspace_bytes(M, K, N, false, false));
  if (rc) return rc;
  RB_REQUIRE((reinterpret_cast<uintptr_t>(y) & 15) == 0, -3, "pre-projection: y must be 16-byte aligned");
  return rb::launch_linear_fwd(x, W, bias, M, K, N, y, workspace, static_cast<cudaStream_t>(stream));
}

int rnnt_b200_linear_bwd(const float* x, const float* W, const float* dy, int64_t M, int K, int N, float* dx,
                         float* dW, float* db, int flags, void* workspace, size_t workspace_bytes, void* stream) {
  const bool det = (flags & RNNT_B200_DETERMINISTIC) != 0;
  int rc = check_linear(x, W, M, K, N, workspace, workspace_bytes, rb::linear_workspace_bytes(M, K, N, true, det));
  if (rc) return rc;
  RB_REQUIRE(((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dW)) & 15) == 0,
             -3, "pre-projection: dy / dx / dW must be 16-byte aligned");
  return rb::launch_linear_bwd(x, W, dy, M, K, N, dx, dW, db, det, workspace, static_cast<cudaStream_t>(stream));
}

int rnnt_b200_profile_begin(void) { return rb::prof_begin(); }
int rnnt_b200_profile_end(float* ms, int64_t* launches) {
  long long l[rb::kProfFamilies];
  const int rc = rb::prof_end(ms, l);
  for (int i = 0; i < rb::kProfFamilies; ++i) launches[i] = l[i];
  return rc;
}

size_t rnnt_b200_joint_argmax_scratch_bytes(int N, int V) { return rb::joint_argmax_scratch_bytes(N, V); }

int rnnt_b200_joint_argmax(const float* enc_rows, int64_t enc_stride, const float* pred_rows, int64_t pred_stride,
                           const float* W, const float* bias, int N, int H, int V, int32_t* tokens, float* margin,
                           void* scratch, void* stream) {
  RB_REQUIRE(N >= 0 && H > 0 && V > 0, -1, "invalid shape");
  return rb::launch_joint_argmax(enc_rows, enc_stride, pred_rows, pred_stride, W, bias, N, H, V, tokens, margin,
                                 static_cast<float*>(scratch), static_cast<cudaStream_t>(stream));
}

}  // extern "C"
