"""fp64 and fp32 references of the forced alignment (rnnt_b200_viterbi, include/rnnt_b200.h), for the tests.

`viterbi_f64` is the contract in fp64 and also reports how clearly the path was decided: the smallest gap
|blank - label| between the two predecessor values at the decisions along its backtrace.  `viterbi_f32` restates the
kernel's arithmetic exactly (one fp32 add per edge, compare-select with the tie rule), so the kernel must reproduce it
bit for bit."""
import numpy as np


def _viterbi(lpB, lpE, Tb, Ub, dtype):
    """One utterance: lpB, lpE (T, U1) of which the cells t < Tb, u <= Ub are read (lpE not in column Ub).
    Returns (score, frames (Ub,) list, gap floor)."""
    ninf = dtype(-np.inf)
    B_ = np.asarray(lpB)[:Tb, :Ub + 1].astype(dtype)
    E_ = np.asarray(lpE)[:Tb, :Ub + 1].astype(dtype)
    E_[:, Ub] = ninf                                          # no emission out of the last column
    delta = np.full((Tb, Ub + 1), ninf, dtype)
    left = np.zeros((Tb, Ub + 1), bool)
    gap = np.full((Tb, Ub + 1), np.inf)
    delta[0, 0] = dtype(0)
    for n in range(1, Tb + Ub):
        u = np.arange(max(0, n - Tb + 1), min(n, Ub) + 1)
        t = n - u
        tp, up = np.maximum(t - 1, 0), np.maximum(u - 1, 0)
        own = np.where(t > 0, delta[tp, u] + B_[tp, u], ninf)     # from (t-1, u): blank step
        side = np.where(u > 0, delta[t, up] + E_[t, up], ninf)    # from (t, u-1): label step
        lf = side > own                                           # an exact tie goes to the blank predecessor
        delta[t, u] = np.where(lf, side, own)
        left[t, u] = lf
        gap[t, u] = np.where((t > 0) & (u > 0), np.abs(side.astype(np.float64) - own.astype(np.float64)), np.inf)
    score = delta[Tb - 1, Ub] + B_[Tb - 1, Ub]
    frames = [-1] * Ub
    floor = np.inf
    t, u = Tb - 1, Ub
    while u > 0:
        floor = min(floor, gap[t, u])
        if t == 0 or left[t, u]:
            u -= 1
            frames[u] = t
        else:
            t -= 1
    return float(score), frames, float(floor)


def viterbi_f64(lpB, lpE, Tb, Ub):
    """(score, frames, gap floor) of one utterance in fp64."""
    return _viterbi(lpB, lpE, Tb, Ub, np.float64)


def viterbi_f32(lpB, lpE, Tb, Ub):
    """(score, frames, gap floor) of one utterance with the kernel's fp32 arithmetic."""
    return _viterbi(lpB, lpE, Tb, Ub, np.float32)


def align_batch(lp, T_len, U_len, fn=viterbi_f32):
    """The kernel's outputs for a batch: scores (B,) fp32 / fp64, frames (B, U1-1) int32 with -1 padding, gap floors (B,).
    lp (B,T,U1,2); out-of-range lengths give NaN and a row of -1."""
    lp = np.asarray(lp)
    B, T, U1, _ = lp.shape
    dt = np.float32 if fn is viterbi_f32 else np.float64
    scores = np.full(B, np.nan, dt)
    frames = np.full((B, U1 - 1), -1, np.int32)
    floors = np.full(B, np.inf)
    for b in range(B):
        Tb, Ub = int(T_len[b]), int(U_len[b])
        if not (1 <= Tb <= T and 0 <= Ub <= U1 - 1):
            continue
        s, f, g = fn(lp[b, :, :, 0], lp[b, :, :, 1], Tb, Ub)
        scores[b], frames[b, :Ub], floors[b] = s, f, g
    return scores, frames, floors


def path_log_prob(lpB, lpE, frames, Tb):
    """fp64 log-probability of the path whose label steps are at `frames` (one utterance)."""
    lpB = np.asarray(lpB, np.float64)
    lpE = np.asarray(lpE, np.float64)
    Ub = len(frames)
    total, t, u = 0.0, 0, 0
    for u, f in enumerate(frames):
        total += lpB[t:f, u].sum()
        total += lpE[f, u]
        t = f
    return total + lpB[t:Tb, Ub].sum()
