"""Batched beam-search decode (rnnt_b200_beam_decode / functional.beam_decode / RNNTModel.beam_search*).

CPU tests: argument validation of the C entries (negative codes, no device touched), the Python dispatch errors, and
the fp64 reference of tests/beam_oracle.py itself (K = 1 is greedy search with one symbol per frame; with a beam wide
enough for every distinct token list, its scores are the exact sequence probabilities).  GPU tests (-m gpu): K = 1
against the greedy kernel, K in {2, 4, 8} against the fp64 reference (identical n-best lists, scores within
SCORE_ATOL + SCORE_RTOL |score|), bit-identical results run to run and whatever batch position an utterance sits in."""
import itertools
import math
import os

import numpy as np
import pytest
import torch

from beam_oracle import beam_search

gpu = pytest.mark.gpu

# |kernel - oracle| score tolerance: fp32 logits and a fp32 running sum of one log-probability per frame
# (DESIGN.md section 5 records the errors measured on a B200)
SCORE_ATOL, SCORE_RTOL = 2e-4, 2e-5
GAP_FLOOR = 1e-3          # every oracle selection must be decided by more than this, or the case is not a test


def _model(seed, H, V, E, scale=3.0, blank=None, blank_bias=0.0):
    """Seeded joint weights / ConvPredictor on the CPU generator (identical on every machine)."""
    import rnnt_b200
    torch.manual_seed(seed)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.weight.mul_(scale)
        joint.joint_ln.bias[V - 1 if blank is None else blank] += blank_bias
    return joint, rnnt_b200.ConvPredictor(V, H, E, 0.3).eval()


def _sd(predictor):
    return {k: v.detach().cpu().numpy() for k, v in predictor.state_dict().items()}


def _feats(seed, B, T, H):
    return torch.randn(B, T, H, generator=torch.Generator().manual_seed(seed))


# ---------------------------------------------------------------------------------------------------------- CPU tests

def _beam_call(L, B=2, T=4, H=16, V=8, E=8, blank=7, beam=4, max_len=10, scratch=4096, out=4096):
    return L.rnnt_b200_beam_decode(None, T * H, H, None, *([None] * 13), B, T, H, V, E, blank, beam, max_len,
                                   out, out, out, scratch, None)


def test_beam_entries_reject_bad_arguments_without_device():
    from rnnt_b200 import _lib
    L = _lib.lib()
    assert L.rnnt_b200_beam_decode_scratch_bytes(2, 4, 16, 8, 8, 10) > 0
    assert (L.rnnt_b200_beam_decode_scratch_bytes(2, 8, 16, 8, 8, 10)
            > L.rnnt_b200_beam_decode_scratch_bytes(2, 4, 16, 8, 8, 10))
    for args in ((0, 4, 16, 8, 8, 10), (2, 0, 16, 8, 8, 10), (2, 9, 16, 8, 8, 10), (2, 4, 0, 8, 8, 10),
                 (2, 4, 16, 1, 8, 10), (2, 4, 16, 8, 0, 10), (2, 4, 16, 8, 8, 0)):
        assert L.rnnt_b200_beam_decode_scratch_bytes(*args) == 0, args

    def err():
        return L.rnnt_b200_last_error()

    for kw in (dict(B=0), dict(T=0), dict(V=1), dict(E=0), dict(max_len=0)):
        assert _beam_call(L, **kw) == -1 and b"invalid shape" in err(), kw
    for kw in (dict(H=18), dict(E=10)):
        assert _beam_call(L, **kw) == -2 and b"multiples of 4" in err(), kw
    for blank in (-1, 8):
        assert _beam_call(L, blank=blank) == -4 and b"blank index out of range" in err()
    for scratch in (None, 4096 + 64):
        assert _beam_call(L, scratch=scratch) == -3 and b"128-byte aligned" in err()
    for beam in (0, 9, -1):
        assert _beam_call(L, beam=beam) == -1 and b"beam size must be in [1, 8]" in err(), beam
    assert _beam_call(L, out=None) == -1 and b"required" in err()


def test_beam_search_rejects_unsupported_modules():
    import rnnt_b200
    from helpers import StubEncoder, TinyStatefulPredictor
    H, V, E = 16, 12, 8
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    conv = rnnt_b200.ConvPredictor(V, H, E, 0.3)
    feats, lens = torch.randn(2, 5, H), torch.tensor([5, 3])
    with pytest.raises(ValueError, match="ConvPredictor"):
        rnnt_b200.RNNTModel(TinyStatefulPredictor(V, H, E), torch.nn.Identity(), joint).beam_search_features(feats, lens)
    with pytest.raises(ValueError, match="Unknown predictor type"):
        rnnt_b200.RNNTModel(torch.nn.Linear(2, 2), torch.nn.Identity(), joint).beam_search_features(feats, lens)
    for pre in (rnnt_b200.JointNetwork(20, -1, H, V), rnnt_b200.JointNetwork(-1, 20, H, V)):
        with pytest.raises(ValueError, match="audio_ln / text_ln"):
            rnnt_b200.RNNTModel(conv, torch.nn.Identity(), pre).beam_search_features(feats, lens)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.RNNTModel(conv, torch.nn.Identity(), joint).beam_search_features(feats, lens)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.RNNTModel(conv, StubEncoder(6, H), joint).beam_search(torch.randn(2, 6, 10), torch.tensor([10, 7]))
    for k in (0, 9):
        with pytest.raises(ValueError, match="beam_size"):
            rnnt_b200.beam_decode(feats, lens, joint.joint_ln.weight, joint.joint_ln.bias, conv, V - 1, beam_size=k)


@pytest.mark.parametrize("blank,max_len", [(11, 200), (0, 200), (11, 5), (0, 3)])
def test_oracle_beam_one_is_greedy_with_one_symbol_per_frame(blank, max_len):
    from oracle import rnnt_oracle as orc
    H, V, E = 16, 12, 8
    for seed in range(3):
        joint, pred = _model(seed, H, V, E, scale=2.0, blank=blank, blank_bias=0.5)
        W, b = joint.joint_ln.weight.detach().numpy(), joint.joint_ln.bias.detach().numpy()
        enc = _feats(seed, 1, 14, H)[0].numpy()
        want, _ = orc.greedy_decode(enc, 14, W, b, _sd(pred), blank, max_len, max_per_frame=1)
        nbest, gaps = beam_search(enc, 14, W, b, _sd(pred), blank, 1, max_len)
        assert len(nbest) == 1 and nbest[0][0] == want, seed
        assert len(gaps) == 14


def _brute_force(enc, T, W, b, sd, blank, max_len):
    """log P(y) of every token list y: all emission patterns of at most one symbol per frame, log-added."""
    from oracle import rnnt_oracle as orc
    V = W.shape[0]
    feats = {}
    out = {}
    for pattern in itertools.product(range(V), repeat=T):
        y, lp = [], 0.0
        for t, v in enumerate(pattern):
            key = tuple(y)
            if key not in feats:
                feats[key] = orc.conv_predictor([blank] + y, sd)[-1]        # the whole sequence, no window
            logits = orc.single_forward(enc[t], feats[key], W, b)
            lp += logits[v] - np.log(np.exp(logits - logits.max()).sum()) - logits.max()
            if v != blank:
                if 1 + len(y) + 1 > max_len:
                    lp = -np.inf
                    break
                y = y + [v]
        if lp > -np.inf:
            key = tuple(y)
            out[key] = np.logaddexp(out.get(key, -np.inf), lp)
    return out


@pytest.mark.parametrize("T,blank,max_len", [(1, 2, 200), (3, 0, 200), (4, 2, 200), (4, 1, 3)])
def test_oracle_scores_are_sequence_probabilities_with_a_wide_beam(T, blank, max_len):
    H, V, E = 8, 3, 8
    joint, pred = _model(T + blank, H, V, E, scale=1.5, blank=blank)
    W, b = joint.joint_ln.weight.detach().numpy(), joint.joint_ln.bias.detach().numpy()
    enc = _feats(T, 1, T, H)[0].numpy()
    want = _brute_force(enc, T, W, b, _sd(pred), blank, max_len)
    nbest, _ = beam_search(enc, T, W, b, _sd(pred), blank, 64, max_len)
    assert len(nbest) == len(want)
    got = {tuple(y): s for y, s in nbest}
    assert got.keys() == want.keys()
    for y, s in want.items():
        assert abs(got[y] - s) <= 1e-12, (y, got[y], s)
    scores = [s for _, s in nbest]
    assert scores == sorted(scores, reverse=True)
    assert abs(np.logaddexp.reduce(scores)) < 1e-12 or max_len < T + 1     # all paths: total probability 1


# ---------------------------------------------------------------------------------------------------------- GPU tests

def _beam(joint, pred, feats, lens, K, max_len, blank=None):
    import rnnt_b200
    V = joint.joint_ln.weight.shape[0]
    return rnnt_b200.beam_decode(feats, torch.as_tensor(lens), joint.joint_ln.weight, joint.joint_ln.bias, pred,
                                 V - 1 if blank is None else blank, beam_size=K, max_length=max_len)


def _check_well_formed(nbest, V, blank, K):
    assert 1 <= len(nbest) <= K
    scores = [s for _, s in nbest]
    assert scores == sorted(scores, reverse=True)
    assert all(math.isfinite(s) for s in scores)
    for toks, _ in nbest:
        assert all(0 <= v < V and v != blank for v in toks)
    assert len({tuple(t) for t, _ in nbest}) == len(nbest)


def _greedy_frame_by_frame(joint, pred, feats, lens, max_len):
    """Greedy decode with one symbol per frame, fed one frame per call so that every token is tied to its frame:
    per utterance the tokens and the number of them emitted before the first frame whose decision (the frame's first
    step) has a top-2 logit margin below 1e-4 (None: no such frame)."""
    import rnnt_b200
    B, T = feats.shape[:2]
    dec = rnnt_b200.StreamingGreedyDecoder(joint, pred, B, max_length=max_len, max_outputs_per_step=1)
    dec.reset(range(B))
    toks, safe = [[] for _ in range(B)], [None] * B
    for t in range(T):
        new, mg = dec.decode_chunk(feats[:, t:t + 1], [int(t < n) for n in lens], return_margins=True)
        for b in range(B):
            if safe[b] is None and mg[b] and mg[b][0] < 1e-4:
                safe[b] = len(toks[b])
            toks[b] += new[b]
    return toks, safe


def _one_shot_greedy(joint, pred, feats, lens, max_len):
    import rnnt_b200
    V = joint.joint_ln.weight.shape[0]
    return rnnt_b200.greedy_decode(feats, torch.as_tensor(lens), joint.joint_ln.weight, joint.joint_ln.bias, pred,
                                   V - 1, max_len, 1)


def _compare_with_greedy(joint, pred, feats, lens, max_len, beam):
    """The best hypothesis of K = 1 against greedy with one symbol per frame: equal token lists, or equal up to the
    first near-tie of greedy's decisions."""
    greedy, safe = _greedy_frame_by_frame(joint, pred, feats, lens, max_len)
    assert greedy == _one_shot_greedy(joint, pred, feats, lens, max_len)
    exact = 0
    for i, (want, n) in enumerate(zip(greedy, safe)):
        got = beam[i][0][0]
        if n is None:
            assert got == want, i
            exact += 1
        else:
            assert got[:n] == want[:n], (i, n)
    assert exact >= len(greedy) // 2
    assert sum(len(x) for x in greedy) > len(greedy)


@gpu
def test_beam_one_matches_greedy_on_the_full_golden_setup(golden_dir):
    from helpers import decode_full_setup
    g = np.load(os.path.join(golden_dir, "decode_full.npz"))
    model, feats, T_len = decode_full_setup(g)
    model = model.cuda().eval()
    feats = feats.cuda()
    max_len = int(g["max_length"])
    beam = model.beam_search_features(feats, T_len, beam_size=1, max_length=max_len)
    _compare_with_greedy(model.joint, model.predictor, feats, T_len.tolist(), max_len, beam)


@gpu
def test_beam_one_matches_greedy_at_full_width():
    """B=64, T=400, H=V=1024, E=512, ConvPredictor at default init, max_length 200, ragged lengths."""
    joint, pred = _model(0, 1024, 1024, 512, scale=1.0, blank_bias=1.0)
    joint, pred = joint.cuda(), pred.cuda()
    feats = _feats(1, 64, 400, 1024).cuda()
    lens = torch.randint(200, 401, (64,), generator=torch.Generator().manual_seed(2))
    lens[0] = 400
    lens = lens.tolist()
    _compare_with_greedy(joint, pred, feats, lens, 200, _beam(joint, pred, feats, lens, 1, 200))


# (H, V, E, blank, K, T, lens, max_len, seed, scale, blank_bias): small odd sizes, blank at either end, ragged lengths
# with T_b = 0 and 1, and max_length reached mid-utterance; then a few utterances at full width, and two shapes whose
# weights do not all fit in shared memory on 148 SMs (tests/decode_oracle.py::smem_plan): the joint read from L2
# (V = 4096), and conv2 read from L2 with its tap GEMV and the conv1 table over two K-chunks (E = 1024)
ORACLE_CASES = {
    "v29_k2": (36, 29, 36, 28, 2, 12, [12, 0, 1, 9, 5], 40, 1, 3.0, 0.0),
    "v33_k4_blank0": (36, 33, 36, 0, 4, 12, [12, 1, 0, 7, 11], 40, 7, 3.0, 0.0),
    "v29_k8_blank0_cap": (36, 29, 36, 0, 8, 12, [12, 10, 1, 0, 6], 5, 6, 3.0, -1.0),
    "v33_k8_cap": (36, 33, 36, 32, 8, 10, [10, 0, 3, 8, 1], 6, 47, 3.0, -1.0),
    "v33_k2_cap": (36, 33, 36, 32, 2, 12, [12, 11, 0, 1, 4], 4, 5, 3.0, -2.0),
    "full_k4": (1024, 1024, 512, 1023, 4, 16, [16, 12, 9], 200, 6, 3.0, 2.5),
    "joint_streamed_k4": (1024, 4096, 512, 4095, 4, 12, [12, 10, 7], 200, 27, 3.0, 2.5),
    "conv2_streamed_k4": (1024, 1024, 1024, 1023, 4, 12, [12, 10, 7], 200, 22, 3.0, 2.5),
}


def oracle_case(name):
    """The case's model, features and the oracle's n-best lists and smallest selection gap over every utterance."""
    H, V, E, blank, K, T, lens, max_len, seed, scale, bb = ORACLE_CASES[name]
    joint, pred = _model(seed, H, V, E, scale=scale, blank=blank, blank_bias=bb)
    feats = _feats(seed, len(lens), T, H)
    W, b, sd = joint.joint_ln.weight.detach().numpy(), joint.joint_ln.bias.detach().numpy(), _sd(pred)
    want, gap = [], math.inf
    for i, n in enumerate(lens):
        nbest, gaps = beam_search(feats[i].numpy(), n, W, b, sd, blank, K, max_len)
        want.append(nbest)
        gap = min([gap] + gaps)
    return joint, pred, feats, want, gap


@gpu
@pytest.mark.parametrize("name", sorted(ORACLE_CASES))
def test_beam_matches_fp64_oracle(name):
    H, V, E, blank, K, T, lens, max_len, _, _, _ = ORACLE_CASES[name]
    joint, pred, feats, want, gap = oracle_case(name)
    assert gap > GAP_FLOOR, f"near-tie in the oracle's selections ({gap:.3g}): not a test case"
    got = _beam(joint.cuda(), pred.cuda(), feats.cuda(), lens, K, max_len, blank)
    worst = 0.0
    for i, (g, w) in enumerate(zip(got, want)):
        _check_well_formed(g, V, blank, K)
        assert [t for t, _ in g] == [t for t, _ in w], i
        for (_, gs), (_, ws) in zip(g, w):
            assert abs(gs - ws) <= SCORE_ATOL + SCORE_RTOL * abs(ws), (i, gs, ws)
            worst = max(worst, abs(gs - ws))
        if lens[i] == 0:
            assert g == [([], 0.0)]
    print(f"{name}: max |score - oracle| = {worst:.3g}")


@gpu
@pytest.mark.parametrize("K", [1, 3, 8])
def test_bit_identical_across_runs_and_batch_positions(K):
    H, V, E = 256, 300, 128
    joint, pred = _model(11, H, V, E, scale=2.0, blank_bias=0.5)
    joint, pred = joint.cuda(), pred.cuda()
    feats = _feats(12, 64, 48, H).cuda()
    lens = torch.randint(0, 49, (64,), generator=torch.Generator().manual_seed(13))
    lens[5] = 48
    first = _beam(joint, pred, feats, lens, K, 30)
    assert _beam(joint, pred, feats, lens, K, 30) == first
    for got in first:
        _check_well_formed(got, V, V - 1, K)
    assert sum(len(t) for nb in first for t, _ in nb) > 64
    solo = _beam(joint, pred, feats[5:6], lens[5:6], K, 30)[0]
    for pos in (0, 5, 37, 63):
        f, n = feats.clone(), lens.clone()
        f[pos], n[pos] = feats[5], lens[5]
        assert _beam(joint, pred, f, n, K, 30)[pos] == solo, pos


@gpu
def test_model_beam_search_runs_the_encoder_first():
    import rnnt_b200
    from helpers import StubEncoder
    H, V, E = 64, 40, 32
    joint, pred = _model(21, H, V, E)
    torch.manual_seed(22)
    model = rnnt_b200.RNNTModel(pred, StubEncoder(20, H), joint).cuda().eval()
    mel = torch.randn(3, 20, 30, device="cuda")
    mel_lens = torch.tensor([30, 21, 8])
    got = model.beam_search(mel, mel_lens, beam_size=4, max_length=25)
    with torch.no_grad():
        enc = model.encoder(mel)
    lens = model.encoder.calc_output_lens(mel_lens)
    assert got == model.beam_search_features(enc.permute(0, 2, 1), lens, beam_size=4, max_length=25)
    assert got == model.beam_search_features(enc.permute(0, 2, 1).contiguous(), lens, beam_size=4, max_length=25)
    for nb in got:
        _check_well_formed(nb, V, V - 1, 4)
