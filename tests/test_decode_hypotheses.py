"""Token timing and confidence of the decoders: rnnt_b200_greedy_decode_aligned, rnnt_b200_greedy_decode_stream_aligned,
rnnt_b200_beam_decode_aligned, and the `return_hypotheses` / `DecodedHypothesis` surfaces on top of them.

CPU tests: the fp64 references of tests/hyp_oracle.py (the greedy path score equals the loss oracle's lattice path sum
along the decoded (tokens, frames); the aligned beam reference keeps beam_oracle's n-best lists and at K = 1 gives
greedy's frames with one symbol per frame) and the argument checks of the new C entries.
GPU tests (-m gpu): the plain outputs are unchanged by the new ones; greedy frames, log-probabilities and scores
against fp64 along the kernel's own decisions in every shared-memory plan; streaming bit-identical to one shot for
every split; beam against the aligned fp64 reference; the greedy score against the Viterbi kernel and the loss; bit
identity across runs and batch positions; the Python surfaces against the functional calls."""
import math

import numpy as np
import pytest
import torch

import decode_oracle as do
import hyp_oracle as ho
from beam_oracle import beam_search

gpu = pytest.mark.gpu


def _model(seed, H, V, E, scale=3.0, blank=None, blank_bias=0.0):
    import rnnt_b200
    torch.manual_seed(seed)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.weight.mul_(scale)
        joint.joint_ln.bias[V - 1 if blank is None else blank] += blank_bias
    if blank is not None:
        joint.blank_idx = blank
    return joint, rnnt_b200.ConvPredictor(V, H, E, 0.3).eval()


def _np(joint, pred):
    return (joint.joint_ln.weight.detach().cpu().double().numpy(), joint.joint_ln.bias.detach().cpu().double().numpy(),
            {k: v.detach().cpu().numpy() for k, v in pred.state_dict().items()})


def _feats(seed, B, T, H):
    return torch.randn(B, T, H, generator=torch.Generator().manual_seed(seed))


# ---------------------------------------------------------------------------------------------------------- CPU tests

@pytest.mark.parametrize("blank,max_len,mpf,bias", [(11, 200, 10, 0.5), (0, 200, 10, 0.5), (11, 200, 2, -3.0),
                                                    (0, 7, 10, 0.0), (11, 200, 1, 0.5)])
def test_greedy_reference_score_is_the_lattice_path_sum(blank, max_len, mpf, bias):
    from oracle import rnnt_oracle as orc
    H, V, E, T = 16, 12, 8, 14
    for seed in range(3):
        joint, pred = _model(seed, H, V, E, scale=2.0, blank=blank, blank_bias=bias)
        W, b, sd = _np(joint, pred)
        enc = _feats(seed, 1, T, H)[0].numpy()
        for T_b in (T, 5, 0):
            toks, frames, lps, score = ho.greedy_hypothesis(enc, T_b, W, b, sd, blank, max_len, mpf)
            assert toks == orc.greedy_decode(enc, T_b, W, b, sd, blank, max_len, mpf)[0]
            assert frames == sorted(frames) and all(0 <= f < T_b for f in frames)
            assert all(frames[i:i + mpf + 1] != [frames[i]] * (mpf + 1) for i in range(len(frames)))
            if T_b == 0:
                assert (toks, score) == ([], 0.0)
            elif 1 + len(toks) < max_len:            # ran to T_b: the whole lattice path
                want = ho.path_sum(enc, T_b, W, b, sd, blank, toks, frames)
                assert abs(score - want) <= 1e-10 * (1 + abs(want)), (seed, T_b, score, want)
            assert score <= sum(lps) + 1e-12


@pytest.mark.parametrize("blank,K,max_len", [(11, 1, 200), (0, 1, 5), (11, 2, 200), (0, 4, 200), (11, 8, 6)])
def test_aligned_beam_reference(blank, K, max_len):
    H, V, E, T = 16, 12, 8, 12
    merges = 0
    for seed in range(3):
        joint, pred = _model(seed + 40, H, V, E, scale=2.0, blank=blank, blank_bias=0.3)
        W, b, sd = _np(joint, pred)
        enc = _feats(seed + 40, 1, T, H)[0].numpy()
        got, gaps, dgaps = ho.beam_search_aligned(enc, T, W, b, sd, blank, K, max_len)
        want, wgaps = beam_search(enc, T, W, b, sd, blank, K, max_len)
        assert [(y, s) for y, _, _, s in got] == want and gaps == wgaps
        merges += sum(g < math.inf for g in dgaps)
        for y, fr, lp, s in got:
            assert len(fr) == len(lp) == len(y)
            assert all(fr[i] < fr[i + 1] for i in range(len(fr) - 1))     # one symbol per frame
            assert all(x <= 0 for x in lp)
        if K == 1:
            toks, frames, lps, _ = ho.greedy_hypothesis(enc, T, W, b, sd, blank, max_len, 1)
            assert got[0][:3] == (toks, frames, lps)
    assert K == 1 or merges > 0


# (entry family, keyword) pairs that the plain entry's host checks reject, so no call below reaches a launcher: the
# pointers are made up and never dereferenced.  mpf is not an argument of the beam entries, beam not one of the greedy
# ones, and the one-shot greedy entry takes NULL outputs.
REJECTED = {
    "greedy": [dict(B=0), dict(T=0), dict(V=1), dict(E=0), dict(max_len=0), dict(mpf=-1), dict(H=18), dict(E=10),
               dict(blank=-1), dict(blank=8), dict(scratch=None), dict(scratch=4096 + 64)],
    "stream": [dict(B=0), dict(T=-1), dict(V=1), dict(E=0), dict(max_len=0), dict(mpf=-1), dict(H=18), dict(E=10),
               dict(blank=-1), dict(blank=8), dict(scratch=None), dict(scratch=4096 + 64), dict(out=None)],
    "beam": [dict(B=0), dict(T=0), dict(V=1), dict(E=0), dict(max_len=0), dict(H=18), dict(E=10), dict(blank=-1),
             dict(blank=8), dict(scratch=None), dict(scratch=4096 + 64), dict(beam=0), dict(beam=9), dict(out=None)],
}


def _calls(L, family, out=4096, scratch=4096, **kw):
    """(plain code, aligned code) of one family's entries on made-up pointers."""
    B, T, H, V, E = kw.get("B", 2), kw.get("T", 4), kw.get("H", 16), kw.get("V", 8), kw.get("E", 8)
    blank, max_len, mpf, beam = kw.get("blank", 7), kw.get("max_len", 10), kw.get("mpf", 10), kw.get("beam", 4)
    if family == "greedy":
        a = (None, T * H, H, None, *([None] * 13), B, T, H, V, E, blank, max_len, mpf, out, out, None, scratch, None)
        return L.rnnt_b200_greedy_decode(*a), L.rnnt_b200_greedy_decode_aligned(*a, out, out, out)
    if family == "stream":
        a = (None, T * H, H, out, None, *([None] * 13), B, T, H, V, E, blank, max_len, mpf, out, out, None, scratch,
             None)
        return L.rnnt_b200_greedy_decode_stream(*a), L.rnnt_b200_greedy_decode_stream_aligned(*a, out, out, out)
    a = (None, T * H, H, None, *([None] * 13), B, T, H, V, E, blank, beam, max_len, out, out, out, scratch, None)
    return L.rnnt_b200_beam_decode(*a), L.rnnt_b200_beam_decode_aligned(*a, out, out)


@pytest.mark.parametrize("family,kw", [(f, kw) for f, kws in REJECTED.items() for kw in kws])
def test_aligned_entries_check_like_their_plain_entries(family, kw):
    from rnnt_b200 import _lib
    L = _lib.lib()
    plain, aligned = _calls(L, family, **kw)
    assert plain < 0 and aligned == plain, (family, kw, plain, aligned)


def test_return_hypotheses_is_rejected_where_there_is_no_kernel():
    import rnnt_b200
    from helpers import TinyStatefulPredictor
    H, V, E = 16, 12, 8
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    feats, lens = torch.randn(2, 5, H), torch.tensor([5, 3])
    lstm = rnnt_b200.RNNTModel(TinyStatefulPredictor(V, H, E), torch.nn.Identity(), joint)
    with pytest.raises(ValueError, match="return_hypotheses"):
        lstm.greedy_decode_features(feats.cuda() if torch.cuda.is_available() else _Cudaish(feats), lens,
                                    return_hypotheses=True)


class _Cudaish:
    """A stand-in that passes the decode's is_cuda check on a machine without a GPU, to reach the dispatch errors."""
    def __init__(self, t):
        self.t, self.is_cuda, self.shape, self.device = t, True, t.shape, t.device


# ---------------------------------------------------------------------------------------------------------- GPU tests

def _greedy(joint, pred, feats, lens, max_len, mpf, aligned, margins=True):
    """Direct C calls: (tokens, n_tokens, margins, frames, token_logp, scores) as numpy, the last three None for the
    plain entry."""
    import rnnt_b200.functional as RF
    from rnnt_b200 import _lib
    L = _lib.lib()
    dev = feats.device
    B, T, H = feats.shape
    V, E = joint.joint_ln.weight.shape[0], pred.embedding.embedding_dim
    params = RF._decode_params(joint.joint_ln.weight, joint.joint_ln.bias, pred, dev)
    lens_t = torch.as_tensor(lens).to(dev, torch.int32).contiguous()
    tok = torch.full((B, max_len), -7, dtype=torch.int32, device=dev)
    nt = torch.zeros(B, dtype=torch.int32, device=dev)
    mg = torch.full((T + max_len + 2, B), float("inf"), device=dev) if margins else None
    fr = torch.full((B, max_len), -7, dtype=torch.int32, device=dev)
    lp = torch.full((B, max_len), 7.0, device=dev)
    sc = torch.full((B,), 7.0, device=dev)
    scratch = torch.empty(L.rnnt_b200_greedy_decode_scratch_bytes(B, H, V, E), dtype=torch.uint8, device=dev)
    args = (feats.data_ptr(), feats.stride(0), feats.stride(1), lens_t.data_ptr(), *[t.data_ptr() for t in params], B,
            T, H, V, E, int(joint.blank_idx) % V, max_len, mpf, tok.data_ptr(), nt.data_ptr(),
            mg.data_ptr() if margins else None, scratch.data_ptr(), RF._stream_ptr(dev))
    if aligned:
        _lib.check(L.rnnt_b200_greedy_decode_aligned(*args, fr.data_ptr(), lp.data_ptr(), sc.data_ptr()), "aligned")
    else:
        _lib.check(L.rnnt_b200_greedy_decode(*args), "plain")
    out = [tok.cpu().numpy(), nt.cpu().numpy(), mg.cpu().numpy() if margins else None]
    return out + ([fr.cpu().numpy(), lp.cpu().numpy(), sc.cpu().numpy()] if aligned else [None] * 3)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32) if a.dtype == np.float32 else a


def _case(name):
    from test_decode_oracle import CASES, case_inputs
    joint, pred, enc, lens, m = case_inputs(name)
    return joint, pred, enc, lens, m, CASES[name][5], CASES[name][6]


GREEDY_CASES = ["resident", "joint_streamed", "conv2_streamed", "linear_streamed", "wide_H", "wide_E", "small_odd",
                "small_odd_blank0", "many_rows"]


@gpu
@pytest.mark.parametrize("name", GREEDY_CASES)
def test_greedy_aligned_keeps_the_plain_outputs_and_matches_fp64(name, capsys):
    joint, pred, enc, lens, m, max_len, mpf = _case(name)
    joint, pred, feats = joint.cuda(), pred.cuda(), enc.cuda()
    plain = _greedy(joint, pred, feats, lens, max_len, mpf, False)
    got = _greedy(joint, pred, feats, lens, max_len, mpf, True)
    for i in range(3):
        assert np.array_equal(_bits(plain[i]), _bits(got[i])), i
    tok, nt, _, fr, lp, sc = got
    chain = do.Chain(m)
    enc64 = enc.double().numpy()
    worst, fails = {"logp": 0.0, "score": 0.0}, []
    for b, T_b in enumerate(lens):
        n = int(nt[b]) - 1
        assert (fr[b, n:] == -7).all() and (lp[b, n:] == 7.0).all()
        if T_b == 0:
            assert n == 0 and sc[b] == 0.0
            continue
        f, w, _ = ho.check_greedy_along(m, chain, enc64[b], T_b, tok[b, :n].tolist(), fr[b, :n].tolist(),
                                        lp[b, :n].tolist(), float(sc[b]))
        fails += [f"utterance {b}: {x}" for x in f]
        worst = {k: max(v, w[k]) for k, v in worst.items()}
    assert not fails, "\n".join(fails[:20])
    with capsys.disabled():
        print(f"\n[hyp-oracle] {name}: largest err / bound: logp {worst['logp']:.3g}, score {worst['score']:.3g}")


def _stream_aligned(model, feats, splits, max_len, plain_calls=()):
    """Feed slot b the frames of feats[b] in pieces splits[b]; calls listed in plain_calls use the plain C entry on the
    decoder's state, which writes no frames or log-probabilities.  Returns the decoder and, per slot, the token indices
    an aligned call emitted."""
    import rnnt_b200.functional as RF
    from rnnt_b200 import _lib
    S, H = len(splits), feats.shape[2]
    dec = model.streaming_decoder(S, max_length=max_len)
    dec.reset(range(S))
    pos, aligned_idx = [0] * S, [set() for _ in range(S)]
    for c in range(max(len(s) for s in splits)):
        before = dec.n_tokens.tolist()
        takes = [s[c] if c < len(s) else 0 for s in splits]
        chunk = torch.randn(S, max(takes) + 1, H, device="cuda")
        for b in range(S):
            chunk[b, :takes[b]] = feats[b, pos[b]:pos[b] + takes[b]]
            pos[b] += takes[b]
        if c in plain_calls:
            L = _lib.lib()
            lens = torch.tensor(takes, dtype=torch.int32, device="cuda")
            _lib.check(L.rnnt_b200_greedy_decode_stream(
                chunk.data_ptr(), chunk.stride(0), chunk.stride(1), lens.data_ptr(), dec._reset_mask.data_ptr(),
                *[t.data_ptr() for t in dec._params], S, chunk.shape[1], H, dec.V, dec.E, dec.blank, dec.max_length,
                dec.max_outputs_per_step, dec.tokens.data_ptr(), dec.n_tokens.data_ptr(), None, dec.state.data_ptr(),
                RF._stream_ptr(chunk.device)), "plain stream")
            dec._reset_mask.zero_()
            dec._pending.clear()
            dec._n_host = dec.n_tokens.tolist()
        else:
            dec.decode_chunk(chunk, takes)
            for b, (n0, n1) in enumerate(zip(before, dec.n_tokens.tolist())):
                aligned_idx[b].update(range(max(n0 - 1, 0) if c else 0, n1 - 1))
    return dec, aligned_idx


def _uniform(lens, k):
    return [[k] * (n // k) + ([n % k] if n % k else []) for n in lens]


def _ragged(lens, seed, top=9):
    import random
    rng = random.Random(seed)
    out = []
    for n in lens:
        s, left = [], n
        while left > 0:
            k = min(rng.randint(0, top), left)
            s.append(k)
            left -= k
        out.append(s + [0] * rng.randint(0, 2))
    return out


def _stream_model(seed, H, V, E, blank_bias=1.2):
    import rnnt_b200
    joint, pred = _model(seed, H, V, E, blank_bias=blank_bias)
    return rnnt_b200.RNNTModel(pred, torch.nn.Identity(), joint).cuda().eval()


def _assert_hyp_equal(dec, slot, want, b=None, only=None):
    """The slot's hypothesis equals the one-shot aligned outputs `want` = (tok, nt, _, fr, lp, sc) of utterance b
    (default: b = slot); with `only`, frames and log-probabilities at those token indices only."""
    b = slot if b is None else b
    h = dec.hypothesis(slot)
    n = int(want[1][b]) - 1
    keep = sorted(range(n) if only is None else only)
    assert h.tokens == want[0][b, :n].tolist(), slot
    assert [h.frames[k] for k in keep] == want[3][b, keep].tolist(), slot
    assert np.array_equal(_bits(np.float32([h.log_probs[k] for k in keep])), _bits(want[4][b, keep])), slot
    assert np.float32(h.score).view(np.uint32) == want[5][b:b + 1].view(np.uint32)[0], slot


@gpu
@pytest.mark.parametrize("split", ["1", "3", "7", "ragged0", "ragged1", "mixed"])
def test_streaming_aligned_is_bit_identical_to_one_shot(split):
    model = _stream_model(3, 96, 301, 72)
    B, T, max_len = 9, 24, 30
    feats = _feats(5, B, T, 96).cuda()
    lens = [24, 0, 1, 17, 9, 24, 3, 20, 12]
    want = _greedy(model.joint, model.predictor, feats, lens, max_len, 10, True)
    assert sum(int(x) - 1 for x in want[1]) > B
    if split == "mixed":                  # plain and aligned calls on one state; the last call is aligned
        dec, idx = _stream_aligned(model, feats, _uniform(lens, 2), max_len, plain_calls=(1, 2, 5, 9))
        assert sum(map(len, idx)) < sum(int(x) - 1 for x in want[1])
    else:
        splits = _ragged(lens, int(split[-1])) if split.startswith("ragged") else _uniform(lens, int(split))
        dec, idx = _stream_aligned(model, feats, splits, max_len)
    for b in range(B):
        _assert_hyp_equal(dec, b, want, only=idx[b])


@gpu
def test_streaming_aligned_reset_refresh_and_new_tokens():
    model = _stream_model(21, 128, 64, 64)
    S, T = 4, 48
    A = _feats(1, S, T, 128).cuda()
    X = _feats(2, 1, 30, 128).cuda()
    dec = model.streaming_decoder(S, max_length=60)
    dec.reset(range(S))
    seen = [[] for _ in range(S)]
    for c in range(6):
        feats, lens = A[:, 8 * c: 8 * c + 8].clone(), [8] * S
        if c == 2:
            dec.reset([2])
            seen[2] = []
        if c >= 2:
            n = min(8, 30 - 8 * (c - 2))
            feats[2, :max(n, 0)] = X[0, 8 * (c - 2): 8 * (c - 2) + max(n, 0)]
            lens[2] = max(n, 0)
        new = dec.decode_chunk(feats, lens, return_hypotheses=True)
        for b in range(S):
            assert new[b].score == dec.hypothesis(b).score
            seen[b].append(new[b])
    whole = _greedy(model.joint, model.predictor, A, [T] * S, 60, 10, True)
    for b in (0, 1, 3):
        _assert_hyp_equal(dec, b, whole)
        h = dec.hypothesis(b)
        assert sum((x.tokens for x in seen[b]), []) == h.tokens
        assert sum((x.frames for x in seen[b]), []) == h.frames
        assert sum((x.log_probs for x in seen[b]), []) == h.log_probs
    _assert_hyp_equal(dec, 2, _greedy(model.joint, model.predictor, X, [30], 60, 10, True), b=0)
    # refresh empties every slot: a new session starts from frame 0 and score 0
    dec.refresh()
    dec.reset(range(S))
    dec.decode_chunk(A[:, :20], [20] * S)
    dec.decode_chunk(A[:, 20:], [T - 20] * S)
    for b in range(S):
        _assert_hyp_equal(dec, b, whole)


def _beam_aligned(joint, pred, feats, lens, K, max_len, blank):
    import rnnt_b200
    return rnnt_b200.beam_decode(feats, torch.as_tensor(lens), joint.joint_ln.weight, joint.joint_ln.bias, pred, blank,
                                 beam_size=K, max_length=max_len, return_hypotheses=True)


BEAM_CASES = {   # (H, V, E, blank, K, T, lens, max_len, seed, scale, blank_bias)
    "v29_k1": (36, 29, 36, 28, 1, 12, [12, 0, 1, 9, 5], 40, 1, 3.0, 0.0),
    "v29_k2": (36, 29, 36, 28, 2, 12, [12, 0, 1, 9, 5], 40, 1, 3.0, 0.0),
    "v33_k4_blank0": (36, 33, 36, 0, 4, 12, [12, 1, 0, 7, 11], 40, 7, 3.0, 0.0),
    "v29_k8_blank0_cap": (36, 29, 36, 0, 8, 12, [12, 10, 1, 0, 6], 5, 6, 3.0, -1.0),
    "v33_k8_cap": (36, 33, 36, 32, 8, 10, [10, 0, 3, 8, 1], 6, 47, 3.0, -1.0),
    "full_k4": (1024, 1024, 512, 1023, 4, 16, [16, 12, 9], 200, 6, 3.0, 2.5),
}
GAP_FLOOR = 1e-3
SCORE_ATOL, SCORE_RTOL = 2e-4, 2e-5          # those of tests/test_beam_decode.py


@gpu
@pytest.mark.parametrize("name", sorted(BEAM_CASES))
def test_beam_aligned_matches_fp64_and_keeps_the_plain_outputs(name, capsys):
    import rnnt_b200
    H, V, E, blank, K, T, lens, max_len, seed, scale, bb = BEAM_CASES[name]
    joint, pred = _model(seed, H, V, E, scale=scale, blank=blank, blank_bias=bb)
    feats = _feats(seed, len(lens), T, H)
    W, b, sd = _np(joint, pred)
    ref = [ho.beam_search_aligned(feats[i].numpy(), n, W, b, sd, blank, K, max_len) for i, n in enumerate(lens)]
    gap = min([math.inf] + [g for _, gs, _ in ref for g in gs])
    dgap = min([math.inf] + [g for _, _, ds in ref for g in ds])
    assert gap > GAP_FLOOR, f"near-tie in the reference's selections ({gap:.3g}): not a test case"
    joint, pred, feats = joint.cuda(), pred.cuda(), feats.cuda()
    got = _beam_aligned(joint, pred, feats, lens, K, max_len, blank)
    plain = rnnt_b200.beam_decode(feats, torch.as_tensor(lens), joint.joint_ln.weight, joint.joint_ln.bias, pred, blank,
                                  beam_size=K, max_length=max_len)
    assert [[(h.tokens, h.score) for h in nb] for nb in got] == plain
    worst = 0.0
    for i, (g, (w, _, dg)) in enumerate(zip(got, ref)):
        assert [h.tokens for h in g] == [y for y, _, _, _ in w], i
        for h, (_, wf, wl, ws) in zip(g, w):
            assert len(h.frames) == len(h.log_probs) == len(h.tokens)
            if min(dg, default=math.inf) > GAP_FLOOR:
                assert h.frames == wf, i
            for x, y in zip(h.log_probs, wl):
                assert abs(x - y) <= SCORE_ATOL + SCORE_RTOL * abs(y), (i, x, y)
                worst = max(worst, abs(x - y))
    with capsys.disabled():
        print(f"\n[hyp-oracle] beam {name}: smallest selection gap {gap:.3g}, smallest dominance gap {dgap:.3g}, "
              f"max |logp - fp64| {worst:.3g}")


@gpu
def test_beam_one_frames_are_greedy_one_symbol_per_frame():
    joint, pred = _model(0, 1024, 1024, 512, scale=1.0, blank_bias=1.0)
    joint, pred = joint.cuda(), pred.cuda()
    feats = _feats(1, 64, 200, 1024).cuda()
    lens = torch.randint(100, 201, (64,), generator=torch.Generator().manual_seed(2))
    lens[0] = 200
    lens = lens.tolist()
    beam = _beam_aligned(joint, pred, feats, lens, 1, 200, 1023)
    g = _greedy(joint, pred, feats, lens, 200, 1, True)
    margins = g[2]
    exact = 0
    for b in range(64):
        n = int(g[1][b]) - 1
        toks, frames = g[0][b, :n].tolist(), g[3][b, :n].tolist()
        steps = margins[:, b][np.isfinite(margins[:, b])]
        safe = int(np.argmax(steps < 1e-4)) if (steps < 1e-4).any() else None
        h = beam[b][0]
        if safe is None:
            assert (h.tokens, h.frames) == (toks, frames), b
            exact += 1
        else:       # up to the token count before the first near-tie step
            k = _tokens_before_step(frames, safe, lens[b])
            assert (h.tokens[:k], h.frames[:k]) == (toks[:k], frames[:k]), b
    assert exact >= 32


def _tokens_before_step(frames, step, T_b):
    """Tokens a greedy decode with one symbol per frame emitted before its step `step` (each frame: an emit and an
    advance, or an advance)."""
    steps, k = 0, 0
    for t in range(T_b):
        if k < len(frames) and frames[k] == t:
            if steps >= step:
                return k
            steps, k = steps + 1, k + 1
        if steps >= step:
            return k
        steps += 1
    return k


@gpu
def test_greedy_score_against_viterbi_loss_and_fp64_path_sum():
    import rnnt_b200
    H, V, E, T = 64, 40, 32, 24
    joint, pred = _model(31, H, V, E, scale=2.0, blank_bias=0.8)
    feats = _feats(32, 6, T, H)
    lens = [24, 20, 13, 24, 7, 1]
    W, b, sd = _np(joint, pred)
    jc, pc = joint.cuda(), pred.cuda()
    hyps = rnnt_b200.greedy_decode(feats.cuda(), torch.tensor(lens), jc.joint_ln.weight, jc.joint_ln.bias, pc, V - 1,
                                   200, 10, return_hypotheses=True)
    assert sum(len(h.tokens) for h in hyps) > 6
    ran = 0
    for i, h in enumerate(hyps):
        U_ = len(h.tokens)
        if 1 + U_ >= 200:               # stopped by max_length: the score covers the steps taken, not a whole path
            continue
        ran += 1
        want = ho.path_sum(feats[i].numpy(), lens[i], W, b, sd, V - 1, h.tokens, h.frames)
        assert abs(h.score - want) <= 1e-4 * (1 + abs(want)), (i, h.score, want)
        if U_ == 0:
            continue
        # the decoded transcript through the fused joint: Viterbi (best path) and the loss (all paths)
        enc = feats[i:i + 1, :lens[i]].cuda()
        with torch.no_grad():
            pfe = pc(torch.tensor([[V - 1] + h.tokens], device="cuda"))
        tg = torch.tensor([h.tokens], dtype=torch.int32, device="cuda")
        al = rnnt_b200.joint_forced_align(enc, pfe, jc.joint_ln.weight, jc.joint_ln.bias, tg,
                                          torch.tensor([lens[i]], dtype=torch.int32, device="cuda"),
                                          torch.tensor([U_], dtype=torch.int32, device="cuda"), blank=V - 1)
        vit, logp = float(al.score[0]), float(al.log_prob[0])
        tol = 1e-4 * (1 + abs(vit))
        assert h.score <= vit + tol and vit <= logp + tol, (i, h.score, vit, logp)
    assert ran >= 4


@gpu
def test_bit_identical_across_runs_and_batch_positions():
    import rnnt_b200
    H, V, E = 256, 300, 128
    joint, pred = _model(11, H, V, E, scale=2.0, blank_bias=0.5)
    joint, pred = joint.cuda(), pred.cuda()
    feats = _feats(12, 64, 40, H).cuda()
    lens = torch.randint(0, 41, (64,), generator=torch.Generator().manual_seed(13))
    lens[5] = 40
    w, bias = joint.joint_ln.weight, joint.joint_ln.bias

    def run(f, n):
        g = rnnt_b200.greedy_decode(f, n, w, bias, pred, V - 1, 30, 10, return_hypotheses=True)
        bm = rnnt_b200.beam_decode(f, n, w, bias, pred, V - 1, 4, 30, return_hypotheses=True)
        return g, bm

    first = run(feats, lens)
    assert run(feats, lens) == first
    assert sum(len(h.tokens) for h in first[0]) > 64
    for pos in (0, 37, 63):
        f, n = feats.clone(), lens.clone()
        f[pos], n[pos] = feats[5], lens[5]
        g, bm = run(f, n)
        assert g[pos] == first[0][5] and bm[pos] == first[1][5], pos


@gpu
def test_python_surfaces_equal_the_functional_calls():
    import rnnt_b200
    from helpers import StubEncoder
    H, V, E = 64, 40, 32
    joint, pred = _model(21, H, V, E, blank_bias=1.0)
    torch.manual_seed(22)
    model = rnnt_b200.RNNTModel(pred, StubEncoder(20, H), joint).cuda().eval()
    mel = torch.randn(3, 20, 30, device="cuda")
    mel_lens = torch.tensor([30, 21, 8])
    with torch.no_grad():
        enc = model.encoder(mel).permute(0, 2, 1)
    lens = model.encoder.calc_output_lens(mel_lens)
    w, b = model.joint.joint_ln.weight, model.joint.joint_ln.bias
    hyps = rnnt_b200.greedy_decode(enc, lens, w, b, model.predictor, V - 1, 25, 10, return_hypotheses=True)
    assert all(isinstance(h, rnnt_b200.DecodedHypothesis) for h in hyps)
    assert [h.tokens for h in hyps] == rnnt_b200.greedy_decode(enc, lens, w, b, model.predictor, V - 1, 25, 10)
    assert model.greedy_decode_features(enc, lens, 25, return_hypotheses=True) == hyps
    got, mg = model.greedy_decode_features(enc, lens, 25, return_margins=True, return_hypotheses=True)
    assert got == hyps and mg == model.greedy_decode_features(enc, lens, 25, return_margins=True)[1]
    for h, T_b in zip(hyps, lens.tolist()):
        assert len(h.frames) == len(h.log_probs) == len(h.tokens)
        assert all(0 <= f < T_b for f in h.frames) and h.frames == sorted(h.frames)
        assert h.score <= sum(h.log_probs) and all(x <= 0 for x in h.log_probs)
    nb = rnnt_b200.beam_decode(enc, lens, w, b, model.predictor, V - 1, 4, 25, return_hypotheses=True)
    assert model.beam_search_features(enc, lens, 4, 25, return_hypotheses=True) == nb
    assert model.beam_search(mel, mel_lens, 4, 25, return_hypotheses=True) == nb
    assert [[(h.tokens, h.score) for h in x] for x in nb] == model.beam_search_features(enc, lens, 4, 25)
    with pytest.raises(ValueError, match="return_hypotheses"):
        model.greedy_decode_features(enc, lens, 25, engine="graph", return_hypotheses=True)
