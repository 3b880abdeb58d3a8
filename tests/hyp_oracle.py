"""fp64 references of the decoders' token timing and confidence (the *_aligned entries, include/rnnt_b200.h), for the
tests: greedy frames / token log-probabilities / path score, the lattice path sum along (tokens, frames), beam search
with per-token frames and log-probabilities and the merge's dominance rule, and the bounds of the kernel's fp32
log-probabilities along its own decisions.

Bounds (u = 2^-24, gamma as in tests/decode_oracle.py).  The kernel takes logp[v] = fl(x_v - fl(mx + logf(S))),
S = the fixed-order sum of expf(x_i - mx) over the V logits of the step (ceil(V/256) thread-strided terms, 5 warp and 3
block butterfly levels: depth d = ceil(V/256) + 8):
  * from the logits: x_v is within delta_v of fp64 (decode_oracle.Chain.logits) and log-sum-exp is 1-Lipschitz in the
    max norm, so the exact logp moves by at most delta_v + max(delta);
  * S: each term x_i - mx rounds once (u |x_i - mx| relative after expf), expf is within 2 ulp (2^-22 relative), and
    each of the d additions on a term's path rounds once (u); the terms are positive, so S's relative error is at most
    d (2^-22 + 2u + u max|x_i - mx|) (first order, a superset of gamma(d) + 2^-22 + u max|x_i - mx|); log turns it
    into an absolute error of the same size, logf adds 2 ulp (2^-22 |log S|), the add mx + log S and the final
    subtraction one rounding each (u |lse|, u |logp|).
The path score is the fp32 left-to-right sum of n step terms of one sign: each term's bound plus gamma(n - 1) times the
sum of their magnitudes."""
import math

import numpy as np

from decode_oracle import SLACK, TINY, U, gamma
from oracle.rnnt_oracle import conv_predictor, joint_logits, log_probs, single_forward


def _logp(logits):
    m = logits.max()
    return logits - (m + np.log(np.sum(np.exp(logits - m))))


def greedy_hypothesis(enc, T_b, W, b, pred_sd, blank, max_length=200, max_per_frame=10):
    """fp64 greedy decode (oracle.rnnt_oracle.greedy_decode's rule) with, per token, its frame and log-probability,
    and the path score: the sum of logp[token] over emitting steps and logp[blank] over advancing steps."""
    enc = np.asarray(enc, np.float64)
    tokens, frames, lps, score = [blank], [], [], 0.0
    t, per = 0, 0
    feats = conv_predictor(tokens, pred_sd)[-1]
    while t < T_b and len(tokens) < max_length:
        lp = _logp(single_forward(enc[t], feats, W, b))
        tok = int(np.argmax(lp))
        if tok == blank or per >= max_per_frame:
            score += lp[blank]
            t, per = t + 1, 0
        else:
            score += lp[tok]
            tokens.append(tok)
            frames.append(t)
            lps.append(float(lp[tok]))
            feats = conv_predictor(tokens[-7:], pred_sd)[-1]
            per += 1
    return tokens[1:], frames, lps, float(score)


def path_sum(enc, T_b, W, b, pred_sd, blank, tokens, frames):
    """Log-probability of the lattice path that emits tokens[u] at frame frames[u] and takes a blank step everywhere
    else, final blank at (T_b - 1, U) included: the loss oracle's lattice log-probabilities (log_probs on the full
    (T, U+1) joint) summed along it."""
    U_ = len(tokens)
    pred = conv_predictor([blank] + list(tokens), pred_sd)
    logits = joint_logits(np.asarray(enc, np.float64)[None, :T_b], pred[None], W, b)
    _, lpB, lpE = log_probs(logits, np.asarray(tokens, np.int64)[None], blank)
    s, t = 0.0, 0
    for u in range(U_ + 1):
        stop = frames[u] if u < U_ else T_b          # row U: blank steps up to and including the final one
        for tt in range(t, stop):
            s += lpB[0, tt, u]
        t = stop
        if u < U_:
            s += lpE[0, t, u]
    return float(s)


def steps_of(tokens, frames, T_b, max_len, blank):
    """The step sequence a greedy decode with these outputs took: (frame, emitted token or None for an advance)."""
    out, k, full = [], 0, 1
    for t in range(T_b):
        while k < len(tokens) and frames[k] == t:
            out.append((t, tokens[k]))
            k, full = k + 1, full + 1
        if full >= max_len:
            break
        out.append((t, None))
    assert k == len(tokens), "frames not non-decreasing or past T_b"
    return out


def lse_bound(x64, delta):
    """Bound on |logp32[v] - logp64[v]| except for delta_v (see the module text), for all v at once."""
    V = x64.shape[0]
    d = -(-V // 256) + 8
    m = x64.max()
    lse = m + math.log(np.exp(x64 - m).sum())
    rng = float((x64 - x64.min()).max() + 2 * delta.max())
    es = d * (2.0 ** -22 + 2 * U + U * rng)
    return delta.max() + es + 2.0 ** -22 * abs(lse - m) + U * (abs(lse) + es) + U * (np.abs(x64 - lse) + es) + TINY


def check_greedy_along(m, chain, a_rows, T_b, tokens, frames, logps, score):
    """The kernel's (tokens, frames, token log-probs, score) of one utterance against fp64 logits teacher-forced on its
    own decisions.  Every decision must be admissible (within the logits' bounds of fp64's best, or the cap);
    log-probs and score within the bounds above.  Returns (failures, worst err / bound of logp and score)."""
    fails, worst = [], {"logp": 0.0, "score": 0.0}
    full, per, k = [m.blank], 0, 0
    s64, sbound, mags, n = 0.0, 0.0, 0.0, 0
    for t, tok in steps_of(tokens, frames, T_b, m.max_len, m.blank):
        l64, delta = chain.logits(a_rows[t], full, len(full) - 1)
        top = int(np.argmax(l64))
        lp64 = l64 - (l64.max() + math.log(np.exp(l64 - l64.max()).sum()))
        bnd = (delta + lse_bound(l64, delta)) * SLACK
        v = m.blank if tok is None else tok
        if tok is None:
            if per < m.max_per_frame and not l64[top] - l64[m.blank] <= delta[top] + delta[m.blank]:
                fails.append(f"frame {t}: advanced with blank {l64[top] - l64[m.blank]!r} below the best")
            per = 0
        else:
            if per >= m.max_per_frame or tok == m.blank or not l64[top] - l64[tok] <= delta[top] + delta[tok]:
                fails.append(f"frame {t}: emitted {tok}, fp64 best {top}, per-frame count {per}")
            err = abs(logps[k] - lp64[tok])
            if not err <= bnd[tok]:
                fails.append(f"token {k}: logp {logps[k]!r}, fp64 {lp64[tok]!r}, bound {bnd[tok]!r}")
            worst["logp"] = max(worst["logp"], err / bnd[tok])
            full, per, k = full + [tok], per + 1, k + 1
        s64, sbound, mags, n = s64 + lp64[v], sbound + bnd[v], mags + abs(lp64[v]) + bnd[v], n + 1
    sb = sbound + gamma(max(n - 1, 0)) * mags + TINY
    err = abs(score - s64)
    if not err <= sb:
        fails.append(f"score {score!r}, fp64 {s64!r}, bound {sb!r}")
    worst["score"] = err / sb
    return fails, worst, s64


def beam_search_aligned(enc, T_b, W, b, pred_sd, blank, beam, max_length=200):
    """tests/beam_oracle.py::beam_search with, per hypothesis token, its frame and log-probability, and the merge's
    dominance rule: a merged candidate takes the lists of its larger term (blank continuation s_h + logp_h[blank]
    against extension s_q + logp_q[v]), the blank continuation's on a tie.

    Returns (nbest, gaps, dom_gaps): nbest = up to `beam` (tokens, frames, log_probs, score), best first; gaps as
    beam_search's; dom_gaps[t] = the smallest |blank term - extension term| over the merges kept at frame t (inf if
    none)."""
    W = np.asarray(W, np.float64)
    b = np.asarray(b, np.float64)
    enc = np.asarray(enc, np.float64)
    T_b = max(0, min(int(T_b), enc.shape[0]))
    V = W.shape[0]
    cache = {}

    def feats(y):
        win = tuple(([blank] + list(y))[-7:])
        if win not in cache:
            cache[win] = conv_predictor(list(win), pred_sd)[-1]
        return cache[win]

    hyps = [((), (), (), 0.0)]
    gaps, dom_gaps = [], []
    for t in range(T_b):
        cand = {}          # token list -> [score, source rank, token, frames, log-probs, term, merge gap]

        def add(y, s, rank, tok, fr, lp):
            if y in cand:
                c = cand[y]
                gap = abs(s - c[5])
                if tok == blank:            # c is an extension: the blank continuation keeps its lists unless beaten
                    if not c[5] > s:
                        c[3], c[4] = fr, lp
                    c[1], c[2] = rank, tok
                elif s > c[5]:              # c is a blank continuation: the extension takes over only if larger
                    c[3], c[4] = fr, lp
                c[0] = float(np.logaddexp(c[0], s))
                c[5], c[6] = max(c[5], s), gap
            else:
                cand[y] = [s, rank, tok, fr, lp, s, math.inf]

        in_beam = {y for y, _, _, _ in hyps}
        for rank, (y, fr, lps, s) in enumerate(hyps):
            logp = _logp(single_forward(enc[t], feats(y), W, b))
            add(y, s + logp[blank], rank, blank, fr, lps)
            if 1 + len(y) + 1 <= max_length:
                order = [v for v in np.argsort(-logp, kind="stable") if v != blank][: 2 * beam + 1]
                merged = [v for v in range(V) if v != blank and y + (v,) in in_beam]
                for v in sorted(set(int(v) for v in order) | set(merged)):
                    add(y + (v,), s + logp[v], rank, v, fr + (t,), lps + (float(logp[v]),))
        ranked = sorted(cand.items(), key=lambda kv: (-kv[1][0], kv[1][1], kv[1][2]))
        kept = ranked[:beam]
        sc = [c[0] for _, c in ranked[: beam + 1]]
        gaps.append(min((sc[i] - sc[i + 1] for i in range(len(sc) - 1)), default=float("inf")))
        dom_gaps.append(min((c[6] for _, c in kept), default=float("inf")))
        hyps = [(y, c[3], c[4], c[0]) for y, c in kept]
    return [(list(y), list(fr), list(lp), float(s)) for y, fr, lp, s in hyps], gaps, dom_gaps
