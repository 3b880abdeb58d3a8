"""fp64 reference of the batched beam-search decode (rnnt_b200_beam_decode, include/rnnt_b200.h), for the tests.

Built on the oracle's ConvPredictor and joint step (oracle/rnnt_oracle.py), one utterance at a time."""
import numpy as np

from oracle.rnnt_oracle import conv_predictor, single_forward


def beam_search(enc, T_b, W, b, pred_sd, blank, beam, max_length=200):
    """Frame-synchronous "modified" beam search (at most one symbol per frame) in fp64 -- the contract of
    rnnt_b200_beam_decode (include/rnnt_b200.h).  enc (T,H) for ONE utterance.

    Returns (nbest, gaps): nbest = up to `beam` (tokens, score) pairs, best first; gaps[t] = the smallest selection gap
    of frame t: between the beam-th kept and the best dropped candidate, and between adjacent kept ones (inf if none).
    The predictor runs on the last 7 tokens of [blank] + y (its receptive field)."""
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

    hyps = [((), 0.0)]
    gaps = []
    for t in range(T_b):
        cand = {}          # token list -> [score, source rank, token]

        def add(y, s, rank, tok):
            if y in cand:  # the blank continuation of one hypothesis = the extension of another: merge
                c = cand[y]
                c[0] = float(np.logaddexp(c[0], s))
                if tok == blank:
                    c[1], c[2] = rank, tok
            else:
                cand[y] = [s, rank, tok]

        in_beam = {y for y, _ in hyps}
        for rank, (y, s) in enumerate(hyps):
            logits = single_forward(enc[t], feats(y), W, b)
            m = logits.max()
            logp = logits - (m + np.log(np.sum(np.exp(logits - m))))
            add(y, s + logp[blank], rank, blank)
            if 1 + len(y) + 1 <= max_length:
                # every extension that can be kept, merged or be the best dropped one: the 2*beam+1 best tokens and
                # those that reproduce a hypothesis of the beam
                order = [v for v in np.argsort(-logp, kind="stable") if v != blank][: 2 * beam + 1]
                merged = [v for v in range(V) if v != blank and y + (v,) in in_beam]
                for v in sorted(set(int(v) for v in order) | set(merged)):
                    add(y + (v,), s + logp[v], rank, v)
        ranked = sorted(cand.items(), key=lambda kv: (-kv[1][0], kv[1][1], kv[1][2]))
        kept = ranked[:beam]
        sc = [c[0] for _, c in ranked[: beam + 1]]
        gaps.append(min((sc[i] - sc[i + 1] for i in range(len(sc) - 1)), default=float("inf")))
        hyps = [(y, c[0]) for y, c in kept]
    return [(list(y), float(s)) for y, s in hyps], gaps
