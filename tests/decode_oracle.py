"""fp64 checker of the persistent greedy decode kernel (decode_loop.cu on decode_common.cuh), for the tests.

The kernel is observed along its own path: the streaming decoder is fed one frame per call and its state buffer is
read after every call (`state_regions`).  `check` then compares every observable element by element with fp64:

  * a stage whose input is in the state is checked locally -- the kernel's own fp32 input pushed through the stage in
    fp64 -- so errors do not compound and each bound covers one stage's rounding only;
  * the predictor features are also checked end to end against `oracle.rnnt_oracle.conv_predictor` on the last 7 tokens
    of [blank] + y, with a bound propagated through every stage (`Chain`);
  * every step's decision and top-2 margin is checked against fp64 logits teacher-forced on the kernel's own token
    prefix, so a near-tie may go either way but nothing else may.

Bounds (u = 2^-24, gamma(n) = n u / (1 - n u), the classical bound of n sequential fp32 roundings):

  GEMV (gemv_phase): a lane accumulates its float4 columns l, l+32, ... with 4 ceil(K/128) sequential FMAs, then 5
      butterfly levels and the bias add: depth 4 ceil(K/128) + 6, |err| <= gamma(depth) (sum|w_i x_i| + |b|).  The conv2
      ring adds up to 5 such dot products and the bias in a fixed order: depth + 5.
  conv1 (conv1_update): three table entries and the bias, three fp32 adds: gamma(3) (sum|t| + |b1|).
  GELU (gelu_erf): |gelu'| <= 1.13 carries the input error; erff is within 2 ulp (2^-22 absolute, |erf| <= 1), its
      argument x * fp32(1/sqrt 2) within 2u relative (erf' <= 1.13), and 1 + erf, the final product one rounding each.
  tanh (tanhf of an fp32 add): u |s| for the add, 2 ulp (2^-22 |tanh|) for tanhf, Lipschitz 1.
  LayerNorm (block_layer_norm): sums of ceil(n/256) strided terms, 5 + 3 butterfly levels (d1 = ceil(n/256) + 8);
      mean within gamma(d1) sum|x| / n + u |mean|; each x - mean within that plus u |x - mean|; the variance within
      gamma(d1 + 1) of the rounded squares plus their deviation from the exact squares; rsqrtf within 2 ulp (4u
      relative); two products and the bias add one rounding each.
  LayerNorm input sensitivity (end to end only): an input error dx moves output i by at most
      |w_i| r (dx_i + mean dx + |x_i - mean| r max dx), r = 1 / sqrt(var + eps).

  Propagated bounds are first order; SLACK = 1 + 2^-10 covers the second-order terms (products of two errors that are
  each below 1e-4 relative).  A bound of 2^-126 is added everywhere for subnormal results.

  Decisions: with delta_v the bound of logit v (its GEMV term plus sum_k |W_vk| (tanh bound + end-to-end feats bound)),
      a chosen token v satisfies l64[v] >= max l64 - (delta_v + delta_top) (the kernel's l32[v] >= l32[top]); a margin,
      a difference of the two largest values, is within 2 max delta of fp64's plus u |margin| for its fp32 subtraction.
"""
import math

import numpy as np
from scipy.special import erf

from oracle.rnnt_oracle import conv_predictor

U = 2.0 ** -24
TINY = 2.0 ** -126
SLACK = 1.0 + 2.0 ** -10
THREADS = 256
CHUNK = 512                                  # floats of one GEMV K-chunk: 32 lanes x kJ = 4 float4
LN_CACHED = 8 * THREADS                      # block_layer_norm keeps rows of up to 2048 elements in registers
XSTAGE_BYTES = 2 * (THREADS // 32) * 4 * 32 * 4 * 16
SMEM_BUDGET = 220 * 1024 - XSTAGE_BYTES      # 92 KB of resident weight slices per CTA


def gamma(n):
    return n * U / (1.0 - n * U)


def gemv_chunks(K):
    return -(-(K // 4) // (CHUNK // 4))


def gemv_depth(K):
    return 4 * -(-K // 128) + 6


# ------------------------------------------------------------------------------------------------ launch plan, layout

JOINT, CONV2, CONV1, LINEAR = 1, 2, 4, 8


def smem_plan(grid, H, V, E):
    """Mirror of decode_smem_plan: bit i set = matrix i (joint, conv2, conv1, linear) resident in shared memory.
    conv1's weights are read once (the tap table) and never resident; the others in that order while they fit."""
    per = lambda n: -(-n // grid)
    need = {JOINT: per(V) * H * 4, CONV2: per(E) * 5 * E * 4, LINEAR: per(H) * E * 4}
    used, resident = 0, 0
    for bit in (JOINT, CONV2, LINEAR):
        if used + need[bit] <= SMEM_BUDGET:
            used += need[bit]
            resident |= bit
    return resident


FLOAT_REGIONS = ("feats", "hbuf", "logits", "acc1", "acc2", "ynew", "z", "lin", "emb_ln", "t1")
INT_REGIONS = ("ntok", "t_idx", "per", "emit", "rows", "last_tok", "flags")
HEADER_BYTES = 256                           # 8 int64 phase counters, then the barrier line


def state_layout(B, H, V, E):
    """Mirror of the carving in launch_greedy_decode: name -> (offset in 4-byte words, count), and the end in bytes.
    Float regions are padded to multiples of 4 floats; the symbol tables have one row per class."""
    sizes = dict(feats=B * H, hbuf=B * H, logits=B * V, acc1=B * 3 * E, acc2=B * 5 * E, ynew=B * E, z=B * E,
                 lin=B * H, emb_ln=V * E, t1=V * 3 * E, ntok=B, t_idx=B, per=B, emit=B, rows=2 * B, last_tok=B,
                 flags=16)
    off, out = HEADER_BYTES // 4, {}
    for name in FLOAT_REGIONS + INT_REGIONS:
        out[name] = (off, sizes[name])
        off += (sizes[name] + 3) // 4 * 4 if name in FLOAT_REGIONS else sizes[name]
    return out, off * 4


SLOT_SHAPES = dict(feats=("H",), hbuf=("H",), logits=("V",), acc1=(3, "E"), acc2=(5, "E"), ynew=("E",), z=("E",),
                   lin=("H",))


def split_regions(words_f32, words_i32, B, H, V, E, names=tuple(SLOT_SHAPES) + ("ntok",)):
    """Per-slot views of a state read as flat float32 / int32 numpy arrays."""
    lay, _ = state_layout(B, H, V, E)
    dims = dict(H=H, V=V, E=E)
    out = {}
    for name in names:
        off, n = lay[name]
        if name in SLOT_SHAPES:
            shape = (B,) + tuple(dims.get(d, d) for d in SLOT_SHAPES[name])
            out[name] = words_f32[off:off + n].reshape(shape).copy()
        else:
            out[name] = words_i32[off:off + n].copy()
    return out


def tables(words_f32, B, H, V, E):
    lay, _ = state_layout(B, H, V, E)
    (oe, ne), (ot, nt) = lay["emb_ln"], lay["t1"]
    return words_f32[oe:oe + ne].reshape(V, E).copy(), words_f32[ot:ot + nt].reshape(V, 3 * E).copy()


# ------------------------------------------------------------------------------------------------ stage references

def layer_norm(x, w, b, eps=1e-5):
    """fp64 LayerNorm of the last axis of x, and the bound of block_layer_norm's fp32 result from the same x."""
    n = x.shape[-1]
    mu = x.mean(-1, keepdims=True)
    d = x - mu
    var = (d * d).mean(-1, keepdims=True)
    r = 1.0 / np.sqrt(var + eps)
    y = d * r * w + b
    d1 = -(-n // THREADS) + 8
    dmu = gamma(d1) * np.abs(x).sum(-1, keepdims=True) / n
    dmu = dmu + U * (np.abs(mu) + dmu)
    e = dmu + U * (np.abs(d) + dmu)                                  # |fl(x - mean^) - (x - mean)|
    sq = (d * d).sum(-1, keepdims=True)
    dsq = (e * (2 * np.abs(d) + e)).sum(-1, keepdims=True)           # rounded differences, squared
    dvar = (gamma(d1 + 1) * (sq + dsq) + dsq) / n
    dvar = dvar + U * (var + dvar) + U * (var + dvar + eps)          # the division, then + eps
    rv = dvar / (var + eps)
    rel_r = 0.5 * rv / (1 - rv) ** 1.5 + 4 * U                       # rsqrtf: 2 ulp
    core = np.abs(w) * r * (e * (1 + rel_r) + np.abs(d) * (rel_r + 2 * U * (1 + rel_r))) * (1 + U) ** 2
    return y, core + U * (np.abs(y) + core) + TINY


def layer_norm_propagated(x, w, dx, eps=1e-5):
    """First-order bound of LayerNorm's output change for an input change of at most dx (elementwise)."""
    mu = x.mean(-1, keepdims=True)
    d = x - mu
    r = 1.0 / np.sqrt((d * d).mean(-1, keepdims=True) + eps)
    mx = dx.max(-1, keepdims=True)
    return np.abs(w) * r * (dx + dx.mean(-1, keepdims=True) + np.abs(d) * r * mx)


def gelu(x, dx):
    """fp64 GELU (erf form) at x, and the bound of gelu_erf's fp32 result at an fp32 input within dx of x."""
    g = 0.5 * x * (1.0 + erf(x / math.sqrt(2.0)))
    ax = np.abs(x) + dx
    rnd = 0.5 * ax * (2.0 ** -22 + 1.6 * U * ax + 2 * U) + U * (np.abs(g) + 1.13 * dx)
    return g, 1.13 * dx + rnd + TINY


def tanh_add(a, f):
    """fp64 tanh(a + f) and the bound of tanhf(fl(a + f)) from the same fp32 a, f."""
    s = a + f
    h = np.tanh(s)
    return h, U * np.abs(s) + 2.0 ** -22 * np.abs(h) + TINY


# ------------------------------------------------------------------------------------------------ the model in fp64

class Model:
    """fp64 weights in the kernel's layout: conv taps (k, E_out, E_in), oldest tap first."""

    def __init__(self, joint_w, joint_b, predictor, blank, max_len, max_per_frame):
        f = lambda t: t.detach().cpu().double().numpy()
        self.Wj, self.bj = f(joint_w), f(joint_b)
        self.sd = {k: f(v) for k, v in predictor.state_dict().items()}
        sd = self.sd
        self.emb, self.ln1_w, self.ln1_b = sd["embedding.weight"], sd["input_layer_norm.weight"], sd["input_layer_norm.bias"]
        self.W1, self.b1 = sd["conv1.conv.weight"].transpose(2, 0, 1).copy(), sd["conv1.conv.bias"]
        self.W2, self.b2 = sd["conv2.conv.weight"].transpose(2, 0, 1).copy(), sd["conv2.conv.bias"]
        self.Wl, self.bl = sd["linear.weight"], sd["linear.bias"]
        self.ln2_w, self.ln2_b = sd["output_layer_norm.weight"], sd["output_layer_norm.bias"]
        self.aWj, self.aW1, self.aW2, self.aWl = (np.abs(a) for a in (self.Wj, self.W1, self.W2, self.Wl))
        self.V, self.H = self.Wj.shape
        self.E = self.emb.shape[1]
        self.blank, self.max_len, self.max_per_frame = int(blank), int(max_len), int(max_per_frame)


class Chain:
    """The predictor evaluated in fp64 from the weights (the tap-table formulation the kernel uses), with a first-order
    bound of the kernel's fp32 error at every stage; the features are cross-checked against conv_predictor."""

    def __init__(self, m):
        self.m = m
        self._sym, self._y, self._f = {}, {}, {}

    def symbol(self, v):
        """(t1 row (3, E), its bound) of symbol v: LayerNorm(embedding) then the three conv1 taps."""
        if v not in self._sym:
            m = self.m
            x, ex = layer_norm(m.emb[v], m.ln1_w, m.ln1_b)
            t = m.W1 @ x
            et = gamma(gemv_depth(m.E)) * (m.aW1 @ np.abs(x)) + m.aW1 @ ex
            self._sym[v] = (t, et * SLACK)
        return self._sym[v]

    def y(self, full, n):
        key = tuple(full[max(0, n - 2):n + 1])
        if key not in self._y:
            m = self.m
            pre, apre, epre = m.b1.copy(), np.abs(m.b1), 0.0
            for j in range(3):
                p = n - 2 + j
                if p >= 0:
                    t, et = self.symbol(full[p])
                    pre, apre, epre = pre + t[j], apre + np.abs(t[j]), epre + et[j]
            self._y[key] = gelu(pre, gamma(3) * apre + epre)
        return self._y[key]

    def feats(self, full, n):
        """(feats64, bound) at predictor position n of `full` ([blank] + tokens)."""
        key = tuple(full[max(0, n - 6):n + 1])
        if key not in self._f:
            m = self.m
            pre, apre, epre = m.b2.copy(), np.abs(m.b2), 0.0
            for j in range(5):
                p = n - 4 + j
                if p >= 0:
                    y, ey = self.y(full, p)
                    pre, apre, epre = pre + m.W2[j] @ y, apre + m.aW2[j] @ np.abs(y), epre + m.aW2[j] @ ey
            z, ez = gelu(pre, gamma(gemv_depth(m.E) + 5) * apre + epre)
            lin = m.Wl @ z + m.bl
            elin = gamma(gemv_depth(m.E)) * (m.aWl @ np.abs(z) + np.abs(m.bl)) + m.aWl @ ez
            f, ef = layer_norm(lin, m.ln2_w, m.ln2_b)
            ef = (ef + layer_norm_propagated(lin, m.ln2_w, elin)) * SLACK
            ref = conv_predictor(list(key), m.sd)[-1]
            assert np.abs(ref - f).max() <= 1e-9 * (1 + np.abs(ref).max()), "tap-table chain != conv_predictor"
            self._f[key] = (ref, ef)
        return self._f[key]

    def logits(self, a, full, n):
        """Teacher-forced fp64 logits at frame features a and position n, and each logit's bound delta."""
        m = self.m
        f, ef = self.feats(full, n)
        h, eh = tanh_add(a, f)
        l64 = m.Wj @ h + m.bj
        delta = gamma(gemv_depth(m.H)) * (m.aWj @ np.abs(h) + np.abs(m.bj)) + m.aWj @ (eh + ef)
        return l64, delta * SLACK + TINY


# ------------------------------------------------------------------------------------------------ the checker

class Checker:
    def __init__(self, m, report=None):
        self.m, self.chain = m, Chain(m)
        self.fails, self.report = [], ({} if report is None else report)
        self._yk = {}

    def obs(self, name, got, ref, bound, where):
        """Every element of `got` within `bound` of `ref`; records the largest err / bound."""
        got = np.asarray(got, np.float64)
        err = np.abs(got - ref)
        bad = ~(err <= bound)
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            self.fails.append(f"{name}: {where}: {int(bad.sum())} of {bad.size} out of bound; first flat index {i}: got "
                              f"{got.flat[i]!r}, want {float(np.broadcast_to(ref, got.shape).flat[i])!r}, "
                              f"bound {float(np.broadcast_to(bound, got.shape).flat[i])!r}")
        elif err.size:
            self.report[name] = max(self.report.get(name, 0.0), float((err / bound).max()))

    def fail(self, name, msg):
        self.fails.append(f"{name}: {msg}")

    # -- symbol tables, once
    def tables(self, emb_ln, t1):
        m = self.m
        ref, bound = layer_norm(m.emb, m.ln1_w, m.ln1_b)
        self.obs("emb_ln", emb_ln, ref, bound, "table")
        x = emb_ln.astype(np.float64)
        t = np.einsum("joi,vi->vjo", m.W1, x).reshape(m.V, 3 * m.E)
        bt = gamma(gemv_depth(m.E)) * np.einsum("joi,vi->vjo", m.aW1, np.abs(x)).reshape(m.V, 3 * m.E)
        self.obs("t1", t1, t, bt + TINY, "table")
        self.t1k = t1.astype(np.float64).reshape(m.V, 3, m.E)

    def y_kernel(self, full, p):
        """conv1 output at position p from the kernel's own tap table, and the bound of the kernel's fp32 value."""
        key = tuple(full[max(0, p - 2):p + 1])
        if key not in self._yk:
            pre, apre = self.m.b1.copy(), np.abs(self.m.b1)
            for j in range(3):
                q = p - 2 + j
                if q >= 0:
                    t = self.t1k[full[q], j]
                    pre, apre = pre + t, apre + np.abs(t)
            self._yk[key] = gelu(pre, gamma(3) * apre)
        return self._yk[key]

    # -- the predictor state of one slot at its newest position n
    def predictor_state(self, R, full, where):
        m = self.m
        n = len(full) - 1
        self.obs("ynew", R["ynew"], *self.y_kernel(full, n), where)
        ring1 = R["acc1"].astype(np.float64)
        for p in range(n + 1, n + 3):
            ref, a = 0.0, 0.0
            for q in range(max(0, p - 2), n + 1):
                t = self.t1k[full[q], q - p + 2]
                ref, a = ref + t, a + np.abs(t)
            self.obs("acc1", ring1[p % 3], ref, gamma(2) * a + TINY, where + f" position {p}")
        if np.any(ring1[n % 3] != 0):
            self.fail("acc1", f"{where}: the slot of position {n + 3} is not zero")
        ring2 = R["acc2"].astype(np.float64)
        ys = {q: self.y_kernel(full, q) for q in range(max(0, n - 4), n + 1)}
        d2 = gamma(gemv_depth(m.E) + 5)
        for p in range(n, n + 5):
            pre, apre, epre = 0.0, 0.0, 0.0
            for q in range(max(0, p - 4), n + 1):
                y, ey = ys[q]
                W, aW = m.W2[q - p + 4], m.aW2[q - p + 4]
                pre, apre, epre = pre + W @ y, apre + aW @ np.abs(y), epre + aW @ ey
            if p == n:
                self.obs("z", R["z"], *gelu(pre + m.b2, (d2 * (apre + np.abs(m.b2)) + epre) * SLACK), where)
            else:
                self.obs("acc2", ring2[p % 5], pre, (d2 * apre + epre) * SLACK + TINY, where + f" position {p}")
        if np.any(ring2[n % 5] != 0):
            self.fail("acc2", f"{where}: the slot of position {n + 5} is not zero")
        z = R["z"].astype(np.float64)
        self.obs("lin", R["lin"], m.Wl @ z + m.bl,
                 gamma(gemv_depth(m.E)) * (m.aWl @ np.abs(z) + np.abs(m.bl)) + TINY, where)
        self.obs("feats", R["feats"], *layer_norm(R["lin"].astype(np.float64), m.ln2_w, m.ln2_b), where)
        f64, ef = self.chain.feats(full, n)
        self.obs("feats_e2e", R["feats"], f64, ef, where)

    def joint_state(self, R, a, where, hbuf_current):
        m = self.m
        if hbuf_current:
            self.obs("hbuf", R["hbuf"], *tanh_add(a, R["feats"].astype(np.float64)), where)
        h = R["hbuf"].astype(np.float64)
        self.obs("logits", R["logits"], m.Wj @ h + m.bj,
                 gamma(gemv_depth(m.H)) * (m.aWj @ np.abs(h) + np.abs(m.bj)) + TINY, where)

    # -- the decisions of one frame
    def frame_steps(self, a, full, new, margins, where):
        m = self.m
        n = len(new)
        finished = len(full) + n >= m.max_len
        if n > m.max_per_frame:
            self.fail("cap", f"{where}: {n} emits in one frame, max_per_frame {m.max_per_frame}")
        if len(margins) != n + (0 if finished else 1):
            self.fail("steps", f"{where}: {len(margins)} steps for {n} emits (finished: {finished})")
            return
        for i, mg in enumerate(margins):
            l64, delta = self.chain.logits(a, full + new[:i], len(full) + i - 1)
            top = int(np.argmax(l64))
            s = np.sort(l64)
            dm = 2 * delta.max() + U * abs(mg)
            err = abs(mg - (s[-1] - s[-2]))
            if not err <= dm:
                self.fail("margin", f"{where} step {i}: margin {mg!r}, fp64 {s[-1] - s[-2]!r}, bound {dm!r}")
            else:
                self.report["margin"] = max(self.report.get("margin", 0.0), err / dm)
            if i < n:
                v = new[i]
                gap, tol = l64[top] - l64[v], delta[v] + delta[top]
                if v == m.blank or not gap <= tol:
                    self.fail("token", f"{where} step {i}: emitted {v}, fp64 best {top} by {gap!r} (bound {tol!r})")
                elif tol > 0:
                    self.report["token"] = max(self.report.get("token", 0.0), gap / tol)
            elif n < m.max_per_frame:        # the frame's advance, not forced by the cap: blank won
                gap, tol = l64[top] - l64[m.blank], delta[m.blank] + delta[top]
                if not gap <= tol:
                    self.fail("advance", f"{where}: advanced with blank {gap!r} below the best {top} (bound {tol!r})")
                elif tol > 0:
                    self.report["advance"] = max(self.report.get("advance", 0.0), gap / tol)


def check(m, trace, report=None):
    """Checks a decode trace (see `trace_from_frames`): returns the failures ("observable: where: what"); with `report`,
    records the largest err / bound per observable."""
    c = Checker(m, report)
    c.tables(trace["emb_ln"], trace["t1"])
    enc, lens = trace["enc"], trace["lens"]
    B = len(lens)
    for b in range(B):
        full, prev = [m.blank], None
        for t, fr in enumerate(trace["frames"]):
            R = {k: v[b] for k, v in fr["regions"].items()}
            new, margins = fr["new"][b], fr["margins"][b]
            where = f"slot {b} frame {t}"
            live = t < lens[b] and len(full) < m.max_len
            if not live:
                if new or margins:
                    c.fail("idle", f"{where}: {len(margins)} steps and tokens {new} after its end")
                if prev is not None:
                    for k in SLOT_SHAPES:
                        if not np.array_equal(R[k].view(np.uint32), prev[k].view(np.uint32)):
                            c.fail("idle", f"{where}: {k} changed after its end")
            else:
                c.frame_steps(enc[b, t].astype(np.float64), full, list(new), list(margins), where)
            full = full + list(new)
            if int(R["ntok"]) != len(full):
                c.fail("ntok", f"{where}: state holds {int(R['ntok'])}, the tokens give {len(full)}")
            if live or t == 0:
                c.predictor_state(R, full, where)
                if margins:
                    c.joint_state(R, enc[b, t].astype(np.float64), where, hbuf_current=len(margins) > len(new))
            prev = R
    return c.fails


# ------------------------------------------------------------------------------------------------ fp32 emulation

class Emulator:
    """The kernel's decode on the CPU: the tap-accumulator predictor (ConvPredictorStepper's incremental evaluation
    in the kernel's ring form) and the step rule, each stage computed in fp64 from fp32 operands and stored in fp32,
    as the kernel stores it.  `defect` plants one fault."""

    def __init__(self, m, B, defect=None):
        self.m, self.defect = m, defect
        r = lambda a: np.asarray(a, np.float64).astype(np.float32)
        self.r = r
        self.emb_ln = r(layer_norm(m.emb, m.ln1_w, m.ln1_b)[0])
        self.t1 = r(np.einsum("joi,vi->vjo", m.W1, self.emb_ln.astype(np.float64)).reshape(m.V, 3 * m.E))
        H, V, E = m.H, m.V, m.E
        self.S = dict(feats=np.zeros((B, H), np.float32), hbuf=np.zeros((B, H), np.float32),
                      logits=np.zeros((B, V), np.float32), acc1=np.zeros((B, 3, E), np.float32),
                      acc2=np.zeros((B, 5, E), np.float32), ynew=np.zeros((B, E), np.float32),
                      z=np.zeros((B, E), np.float32), lin=np.zeros((B, H), np.float32), ntok=np.zeros(B, np.int32))
        self.full = [[m.blank] for _ in range(B)]

    def _conv1(self, b, tok, n):
        S, r, m = self.S, self.r, self.m
        rows = self.t1[tok].reshape(3, m.E).astype(np.float64)
        acc = S["acc1"][b]
        acc[(n + 2) % 3] = r(acc[(n + 2) % 3] + rows[0])
        acc[(n + 1) % 3] = r(acc[(n + 1) % 3] + rows[1])
        S["ynew"][b] = r(gelu(r(r(acc[n % 3] + rows[2]) + m.b1).astype(np.float64), 0.0)[0])
        acc[n % 3] = 0.0

    def _predict(self, b, n, refresh=True):
        S, r, m = self.S, self.r, self.m
        y = S["ynew"][b].astype(np.float64)
        acc = S["acc2"][b]
        for j in range(4):
            k = (n + 5 - j) % 5 if self.defect == "conv2_ring_rotated" else (n + 4 - j) % 5
            acc[k] = r(acc[k] + r(m.W2[j] @ y))
        pre = r(r(acc[n % 5] + r(m.W2[4] @ y)) + m.b2)
        S["z"][b] = r(gelu(pre.astype(np.float64), 0.0)[0])
        acc[n % 5] = 0.0
        S["lin"][b] = r(m.Wl @ S["z"][b].astype(np.float64) + m.bl)
        if refresh:
            lin = S["lin"][b].astype(np.float64)
            if self.defect == "ln_first_2048":
                S["feats"][b, :LN_CACHED] = r(layer_norm(lin[:LN_CACHED], m.ln2_w[:LN_CACHED], m.ln2_b[:LN_CACHED])[0])
            else:
                S["feats"][b] = r(layer_norm(lin, m.ln2_w, m.ln2_b)[0])

    def _argmax(self, l):
        best = int(np.argmax(l))
        rest = np.delete(l, best)
        if self.defect == "margin_other_warps":        # second best of the winning warp's threads only
            warp = np.arange(len(l)) % THREADS // 32
            rest = np.delete(np.where(warp == warp[best], l, -np.inf), best)
        second = rest.max() if rest.size else -np.inf
        return best, float(np.float32(l[best]) - np.float32(second))

    def reset(self, b):
        S, m = self.S, self.m
        S["acc1"][b] = 0.0
        S["acc2"][b] = 0.0
        S["ntok"][b] = 1
        self.full[b] = [m.blank]
        self._conv1(b, m.blank, 0)
        self._predict(b, 0)

    def frame(self, b, a):
        """One frame of slot b at encoder features a: (new tokens, margins)."""
        S, r, m = self.S, self.r, self.m
        new, margins, per = [], [], 0
        cap = m.max_per_frame + (1 if self.defect == "cap_plus_one" else 0)
        while S["ntok"][b] < m.max_len:
            S["hbuf"][b] = r(np.tanh(r(a + S["feats"][b]).astype(np.float64)))
            h = S["hbuf"][b].astype(np.float64)
            if self.defect == "joint_last_chunk_dropped":
                k0 = CHUNK * (gemv_chunks(m.H) - 1)
                S["logits"][b] = r(m.Wj[:, :k0] @ h[:k0] + m.bj)
            else:
                S["logits"][b] = r(m.Wj @ h + m.bj)
            tok, margin = self._argmax(S["logits"][b])
            margins.append(margin)
            if tok == m.blank or per >= cap:
                break
            n = int(S["ntok"][b])
            new.append(tok)
            self.full[b].append(tok)
            self._conv1(b, tok, n)
            S["ntok"][b] = n + 1
            per += 1
            self._predict(b, n, refresh=self.defect != "feats_not_refreshed")
        return new, margins


def emulate(m, enc, lens, defect=None):
    """The trace `check` reads, produced by the emulator: enc (B, T, H) fp32 numpy, lens per slot."""
    B, T = enc.shape[:2]
    em = Emulator(m, B, defect)
    frames = []
    for b in range(B):
        em.reset(b)
    for t in range(T):
        new, margins = [], []
        for b in range(B):
            live = t < lens[b] and em.S["ntok"][b] < m.max_len
            nw, mg = em.frame(b, enc[b, t].astype(np.float64)) if live else ([], [])
            new.append(nw)
            margins.append(mg)
        frames.append(dict(new=new, margins=margins, regions={k: v.copy() for k, v in em.S.items()}))
    return dict(enc=enc, lens=list(lens), emb_ln=em.emb_ln, t1=em.t1, frames=frames)
