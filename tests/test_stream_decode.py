"""Streaming greedy decode (rnnt_b200_greedy_decode_stream / StreamingGreedyDecoder).

CPU tests: argument validation of the C entries (negative codes, no device touched) and the Python decoder's dispatch
errors.  GPU tests (-m gpu): an utterance decoded in any split into chunks gives exactly the tokens and per-step
margins of the one-shot kernel on the whole utterance, whatever slot it sits in and whatever the other slots do."""
import ctypes as C
import os
import random

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------- CPU tests

def _stream_call(L, B=2, Tc=4, H=16, V=8, E=8, blank=7, state=4096, max_len=10, mpf=10):
    return L.rnnt_b200_greedy_decode_stream(None, Tc * H, H, None, None, *([None] * 13), B, Tc, H, V, E, blank,
                                            max_len, mpf, None, None, None, state, None)


def _init_call(L, B=2, H=16, V=8, E=8, state=4096):
    return L.rnnt_b200_greedy_decode_stream_init(*([None] * 13), B, H, V, E, state, None)


def test_stream_entries_reject_bad_arguments_without_device():
    from rnnt_b200 import _lib
    L = _lib.lib()
    assert L.rnnt_b200_greedy_decode_state_bytes(2, 16, 8, 8) == L.rnnt_b200_greedy_decode_scratch_bytes(2, 16, 8, 8) > 0
    assert L.rnnt_b200_greedy_decode_state_bytes(0, 16, 8, 8) == 0

    def err():
        return L.rnnt_b200_last_error()

    for kw in (dict(B=0), dict(Tc=-1), dict(V=1), dict(E=0), dict(max_len=0), dict(mpf=-1)):
        assert _stream_call(L, **kw) == -1 and b"invalid shape" in err(), kw
    for kw in (dict(H=18), dict(E=10)):
        assert _stream_call(L, **kw) == -2 and b"multiples of 4" in err(), kw
        assert _init_call(L, **kw) == -2, kw
    for blank in (-1, 8):
        assert _stream_call(L, blank=blank) == -4 and b"blank index out of range" in err()
    for state in (None, 4096 + 64):
        assert _stream_call(L, state=state) == -3 and b"128-byte aligned" in err()
        assert _init_call(L, state=state) == -3
    assert _init_call(L, B=0) == -1
    # the one-shot entry shares the checks (null scratch included)
    rc = L.rnnt_b200_greedy_decode(None, 64, 16, None, *([None] * 13), 2, 4, 16, 8, 8, 7, 10, 10, None, None, None,
                                   None, None)
    assert rc == -3 and b"128-byte aligned" in err()
    rc = L.rnnt_b200_greedy_decode(None, 64, 16, None, *([None] * 13), 2, 0, 16, 8, 8, 7, 10, 10, None, None, None,
                                   4096, None)
    assert rc == -1


def test_streaming_decoder_rejects_unsupported_modules():
    import rnnt_b200
    from helpers import TinyStatefulPredictor
    H, V, E = 16, 12, 8
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with pytest.raises(ValueError, match="ConvPredictor"):
        rnnt_b200.StreamingGreedyDecoder(joint, TinyStatefulPredictor(V, H, E), 2)
    with pytest.raises(ValueError, match="Unknown predictor type"):
        rnnt_b200.StreamingGreedyDecoder(joint, torch.nn.Linear(2, 2), 2)
    conv = rnnt_b200.ConvPredictor(V, H, E, 0.3)
    with pytest.raises(ValueError, match="audio_ln / text_ln"):
        rnnt_b200.StreamingGreedyDecoder(rnnt_b200.JointNetwork(20, -1, H, V), conv, 2)
    with pytest.raises(ValueError, match="audio_ln / text_ln"):
        rnnt_b200.RNNTModel(conv, torch.nn.Identity(), rnnt_b200.JointNetwork(-1, 20, H, V)).streaming_decoder(2)
    with pytest.raises(RuntimeError, match="hidden size must agree"):
        rnnt_b200.StreamingGreedyDecoder(rnnt_b200.JointNetwork(-1, -1, 2 * H, V), conv, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.RNNTModel(conv, torch.nn.Identity(), joint).streaming_decoder(2)


# ---------------------------------------------------------------------------------------------------------- GPU tests

def _model(seed, H, V, E, scale=3.0, blank_bias=1.2):
    import rnnt_b200
    torch.manual_seed(seed)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.weight.mul_(scale)
        joint.joint_ln.bias[V - 1] += blank_bias
    return rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.3), torch.nn.Identity(), joint).cuda().eval()


def _one_shot(model, feats, lens, max_length, mpf=10):
    import rnnt_b200
    return rnnt_b200.greedy_decode(feats, torch.as_tensor(lens), model.joint.joint_ln.weight, model.joint.joint_ln.bias,
                                   model.predictor, model.joint.blank_idx, max_length, mpf, return_margins=True)


def _uniform(lens, k):
    return [[k] * (n // k) + ([n % k] if n % k else []) for n in lens]


def _ragged(lens, seed, top=9):
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


def _stream(dec, feats, splits, pad=1):
    """Feed slot b the frames of feats[b] in pieces splits[b] (one piece per call; slots with fewer pieces take 0
    frames).  Frames past a slot's piece are random: the decoder must ignore them.  Returns tokens and margins."""
    S, H = dec.slots, feats.shape[2]
    pos, toks, mgs = [0] * S, [[] for _ in range(S)], [[] for _ in range(S)]
    for c in range(max(len(s) for s in splits)):
        takes = [s[c] if c < len(s) else 0 for s in splits]
        chunk = torch.randn(S, max(takes) + pad, H, device="cuda")
        for b in range(S):
            chunk[b, :takes[b]] = feats[b, pos[b]:pos[b] + takes[b]]
            pos[b] += takes[b]
        new, mg = dec.decode_chunk(chunk, torch.tensor(takes), return_margins=True)
        for b in range(S):
            toks[b] += new[b]
            mgs[b] += mg[b]
    return toks, mgs


def _fresh(model, S, max_length):
    dec = model.streaming_decoder(S, max_length=max_length)
    dec.reset(range(S))
    return dec


def _assert_same(got, want):
    (gt, gm), (wt, wm) = got, want
    for b in range(len(wt)):
        assert gt[b] == wt[b], b
        assert gm[b] == wm[b], b          # bit-identical margins, step for step


def _small_golden(golden_dir):
    import rnnt_b200
    g = np.load(os.path.join(golden_dir, "decode_small.npz"))
    V, H = g["W"].shape
    E = g["pred.embedding.weight"].shape[1]
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    joint.load_state_dict({"joint_ln.weight": torch.from_numpy(g["W"]), "joint_ln.bias": torch.from_numpy(g["b"])})
    pred = rnnt_b200.ConvPredictor(V, H, E, 0.3)
    pred.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("pred.")})
    model = rnnt_b200.RNNTModel(pred, torch.nn.Identity(), joint).cuda().eval()
    return g, model, torch.from_numpy(g["feats"]).cuda()


@gpu
@pytest.mark.parametrize("split", ["1", "3", "7", "ragged0", "ragged1"])
def test_small_golden_through_chunks(golden_dir, split):
    g, model, feats = _small_golden(golden_dir)
    lens = [int(x) for x in g["T_len"]]
    max_len = int(g["max_length"])
    splits = _ragged(lens, int(split[-1])) if split.startswith("ragged") else _uniform(lens, int(split))
    got = _stream(_fresh(model, len(lens), max_len), feats, splits)
    off = 0
    for i, n in enumerate(g["tok_len"]):
        assert got[0][i] == g["tok_flat"][off:off + n].tolist(), i
        off += n
    _assert_same(got, _one_shot(model, feats, lens, max_len))


@gpu
def test_full_golden_in_16_frame_chunks(golden_dir):
    from helpers import decode_full_setup
    g = np.load(os.path.join(golden_dir, "decode_full.npz"))
    model, feats, T_len = decode_full_setup(g)
    model = model.cuda().eval()
    feats = feats.cuda()
    lens = T_len.tolist()
    max_len = int(g["max_length"])
    got = _stream(_fresh(model, len(lens), max_len), feats, _uniform(lens, 16), pad=0)
    off, exact = 0, 0
    for i, n in enumerate(g["tok_len"]):
        want = g["tok_flat"][off:off + n].tolist()
        off += n
        safe = int(g["safe_len"][i])
        assert got[0][i][:safe] == want[:safe], (i, safe)
        if safe == n:
            assert got[0][i] == want, i
            exact += 1
    assert exact >= 8
    _assert_same(got, _one_shot(model, feats, lens, max_len))


@gpu
@pytest.mark.parametrize("k", [16, 1])
def test_full_size_workload_bit_identical_to_one_shot(k):
    """B=64, T=400, H=V=1024, E=512, ConvPredictor at default init, max_length 200, ragged lengths."""
    model = _model(0, 1024, 1024, 512, scale=1.0, blank_bias=1.0)
    feats = torch.randn(64, 400, 1024, device="cuda")
    lens = torch.randint(200, 401, (64,)).tolist()
    lens[0] = 400
    want = _one_shot(model, feats, lens, 200)
    assert sum(len(x) for x in want[0]) > 64
    # the permuted view of an encoder's (B,H,T) output is accepted as is
    dec = _fresh(model, 64, 200)
    toks, mgs = [[] for _ in range(64)], [[] for _ in range(64)]
    enc_bht = feats.permute(0, 2, 1).contiguous()
    for t0 in range(0, 400, k):
        chunk = enc_bht[:, :, t0:t0 + k].permute(0, 2, 1)
        new, mg = dec.decode_chunk(chunk, [min(max(n - t0, 0), k) for n in lens], return_margins=True)
        for b in range(64):
            toks[b] += new[b]
            mgs[b] += mg[b]
    _assert_same((toks, mgs), want)
    assert [dec.transcript(b) for b in range(64)] == want[0]


@gpu
def test_slot_reset_mid_session_is_independent():
    import rnnt_b200
    model = _model(21, 128, 64, 64)
    S, T = 4, 48
    A = torch.randn(S, T, 128, device="cuda")
    X = torch.randn(1, 30, 128, device="cuda")

    def session(reset_at):
        """6 calls of 8 frames of A per slot; with reset_at, slot 2 is reset before call reset_at and fed X instead."""
        dec = _fresh(model, S, 60)
        outs = [[[], []] for _ in range(S)]          # per slot: (tokens, margins) per call, before / after the reset
        pos_x = 0
        for c in range(6):
            feats = A[:, 8 * c: 8 * c + 8].clone()
            lens = [8] * S
            part = 0
            if reset_at is not None and c >= reset_at:
                if c == reset_at:
                    dec.reset([2])
                n = min(8, 30 - pos_x)
                feats[2, :n] = X[0, pos_x:pos_x + n]
                lens[2] = n
                pos_x += n
                part = 1
            new, mg = dec.decode_chunk(feats, lens, return_margins=True)
            for b in range(S):
                key = part if b == 2 else 0
                outs[b][key] += [(new[b], mg[b])]
        return outs

    plain, with_reset = session(None), session(2)
    for b in (0, 1, 3):
        assert with_reset[b] == plain[b], b
    assert with_reset[2][0] == plain[2][0][:2]                    # before the reset: unchanged
    after_t = sum((t for t, _ in with_reset[2][1]), [])
    after_m = sum((m for _, m in with_reset[2][1]), [])
    solo = rnnt_b200.StreamingGreedyDecoder(model.joint, model.predictor, 1, max_length=60)
    solo.reset(0)
    st, sm = solo.decode_chunk(X, return_margins=True)
    assert (after_t, after_m) == (st[0], sm[0])
    assert (st, sm) == tuple(_one_shot(model, X, [30], 60))


@gpu
def test_max_length_finishes_a_slot_until_reset():
    model = _model(5, 64, 32, 32, blank_bias=-20.0)         # blank never wins: every frame emits max_per_frame tokens
    S, max_len = 3, 6
    feats = torch.randn(S, 12, 64, device="cuda")
    dec = model.streaming_decoder(S, max_length=max_len)
    dec.reset([0, 1])
    new = dec.decode_chunk(feats[:, :2])
    assert [len(x) for x in new] == [max_len - 1, max_len - 1, 0]       # finished inside the first frame
    assert dec.finished.tolist() == [True, True, False]
    want = _one_shot(model, feats[:2, :2], [2, 2], max_len)[0]
    assert new[:2] == want
    for c in range(1, 4):
        assert dec.decode_chunk(feats[:, 2 * c: 2 * c + 2]) == [[], [], []]
    assert dec.transcript(0) == want[0] and dec.transcript(2) == []
    assert dec.n_tokens.tolist() == [max_len, max_len, 0]
    dec.reset(0)
    again = dec.decode_chunk(feats[:, 8:12])
    assert again[0] == _one_shot(model, feats[:1, 8:12], [4], max_len)[0][0] and again[1:] == [[], []]
    assert dec.finished.tolist() == [True, True, False]


@gpu
def test_refresh_after_weight_change_and_interleaved_decoders():
    m1, m2 = _model(7, 96, 48, 40), _model(8, 96, 48, 40)
    feats = torch.randn(3, 20, 96, device="cuda")
    lens = [20, 17, 9]
    d1, d2 = _fresh(m1, 3, 50), _fresh(m2, 3, 50)
    _assert_same(_stream(d1, feats, _uniform(lens, 5)), _one_shot(m1, feats, lens, 50))
    # new weights: tables and re-laid copies are rebuilt by refresh()
    with torch.no_grad():
        m1.joint.joint_ln.weight.mul_(1.3)
        m1.predictor.conv1.conv.weight.add_(0.05 * torch.randn_like(m1.predictor.conv1.conv.weight))
        m1.predictor.embedding.weight.add_(0.1 * torch.randn_like(m1.predictor.embedding.weight))
    d1.refresh()
    assert d1.n_tokens.tolist() == [0, 0, 0]
    d1.reset(range(3))
    # two decoders with different weights, calls interleaved on one stream
    s1, s2 = _uniform(lens, 4), _uniform(lens, 3)
    out1, out2 = ([[] for _ in range(3)], [[] for _ in range(3)]), ([[] for _ in range(3)], [[] for _ in range(3)])
    pos1, pos2 = [0] * 3, [0] * 3
    for c in range(max(len(s) for s in s2)):
        for dec, splits, pos, out in ((d1, s1, pos1, out1), (d2, s2, pos2, out2)):
            takes = [s[c] if c < len(s) else 0 for s in splits]
            chunk = torch.zeros(3, max(max(takes), 1), 96, device="cuda")
            for b in range(3):
                chunk[b, :takes[b]] = feats[b, pos[b]:pos[b] + takes[b]]
                pos[b] += takes[b]
            new, mg = dec.decode_chunk(chunk, takes, return_margins=True)
            for b in range(3):
                out[0][b] += new[b]
                out[1][b] += mg[b]
    _assert_same(out1, _one_shot(m1, feats, lens, 50))
    _assert_same(out2, _one_shot(m2, feats, lens, 50))


@gpu
@pytest.mark.parametrize("shape", [(1, 30, 64, 29, 32, 3, 40), (150, 24, 96, 301, 72, 11, 30)])
def test_odd_sizes(shape):
    B, T, H, V, E, seed, max_len = shape
    model = _model(seed, H, V, E, blank_bias=2.0 if B == 1 else 1.2)
    feats = torch.randn(B, T, H, device="cuda")
    lens = torch.randint(1, T + 1, (B,)).tolist()
    lens[0] = T
    want = _one_shot(model, feats, lens, max_len)
    assert B == 1 or sum(len(x) for x in want[0]) > B
    _assert_same(_stream(_fresh(model, B, max_len), feats, _ragged(lens, seed)), want)
    _assert_same(_stream(_fresh(model, B, max_len), feats, _uniform(lens, 3)), want)
