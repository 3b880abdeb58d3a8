"""Forced alignment (rnnt_b200_viterbi / functional.viterbi, forced_align, joint_forced_align / JointNetwork.align /
RNNTModel.align).

CPU tests: the fp64 reference of tests/align_oracle.py against brute-force enumeration of every path, its fp32
restatement against it, the single-path cases against the oracle's lattice, argument validation of the C entry (no
device touched) and the Python checks.  GPU tests (-m gpu): the kernel alone bit for bit against the fp32 restatement
(ragged lengths, ties, garbage in the cells it must not read, batch position, out-of-range lengths, the shared-memory
limit); the fused and dense paths against the fp32 restatement on their own log-probs and against fp64."""
import itertools

import numpy as np
import pytest
import torch

from align_oracle import align_batch, path_log_prob, viterbi_f32, viterbi_f64

gpu = pytest.mark.gpu

LOSS_RTOL = 1e-4           # log_prob against the golden costs (the loss tests' tolerance)
SCORE_RTOL = 1e-4          # kernel score (and its path scored in fp64) against the fp64 optimum
# Fused path: the kernel's frames must equal the fp64 path for every utterance whose fp64 decisions along that path are
# all decided by more than this (log-prob units).  The fused log-probs differ from fp64 by at most 5.6e-4 per cell
# (fp16 GEMM operands; measured on a B200, DESIGN.md section 5); a decision compares sums of such terms over the two
# competing sub-paths, so the floor is ~18x that per-cell error.
GAP_FLOOR = 0.01
GAP_FLOOR_DENSE = 1e-3     # dense front end: fp32 log-softmax of the given logits, errors ~1e-6


def _rand_lp(rng, B, T, U1, quantised=False):
    lp = np.log(rng.uniform(0.02, 0.95, size=(B, T, U1, 2))).astype(np.float32)
    if quantised:                                            # multiples of 1/8: exact ties are frequent
        lp = (np.round(lp * 8) / 8).astype(np.float32)
    return lp


# ---------------------------------------------------------------------------------------------------------- CPU tests

def _brute_force(lpB, lpE, Tb, Ub):
    """Every path by enumeration (fp64): the best score, and the best path's frames under the tie rule (among equal
    scores, the smallest frame for the last token, then for the one before, ...)."""
    best = None
    for pos in itertools.combinations(range(Tb - 1 + Ub), Ub):   # positions of the label steps among all steps
        t = u = 0
        s = 0.0
        frames = []
        for k in range(Tb - 1 + Ub):
            if k in pos:
                s += lpE[t, u]
                frames.append(t)
                u += 1
            else:
                s += lpB[t, u]
                t += 1
        s += lpB[Tb - 1, Ub]
        key = (s, tuple(-f for f in reversed(frames)))
        if best is None or key > best[0]:
            best = (key, s, frames)
    return best[1], best[2]


@pytest.mark.parametrize("quantised", [False, True])
def test_oracle_equals_brute_force_on_tiny_lattices(quantised):
    rng = np.random.default_rng(7)
    for Tb in range(1, 6):
        for Ub in range(0, 4):
            for _ in range(3):
                lp = _rand_lp(rng, 1, Tb, Ub + 1, quantised)[0].astype(np.float64)
                s, f, _ = viterbi_f64(lp[..., 0], lp[..., 1], Tb, Ub)
                s_bf, f_bf = _brute_force(lp[..., 0], lp[..., 1], Tb, Ub)
                assert abs(s - s_bf) <= 1e-12, (Tb, Ub, s, s_bf)
                assert f == f_bf, (Tb, Ub, f, f_bf)
                assert all(0 <= a <= b <= Tb - 1 for a, b in zip(f, f[1:] + [Tb - 1]))


def test_f32_restatement_agrees_with_f64_where_decided():
    rng = np.random.default_rng(3)
    decided = 0
    for seed in range(6):
        lp = _rand_lp(rng, 1, 60, 21)[0]
        Tb, Ub = 60 - 7 * seed, 20 - 2 * seed
        s64, f64, floor = viterbi_f64(lp[..., 0], lp[..., 1], Tb, Ub)
        s32, f32, _ = viterbi_f32(lp[..., 0], lp[..., 1], Tb, Ub)
        assert abs(s32 - s64) <= 1e-5 * abs(s64)
        if floor > 1e-3:
            decided += 1
            assert f32 == f64, seed
    assert decided >= 3


def test_single_path_score_is_minus_cost():
    from oracle import rnnt_oracle as orc
    rng = np.random.default_rng(5)
    lp = _rand_lp(rng, 4, 9, 6).astype(np.float64)
    T_len, U_len = np.array([9, 1, 1, 4]), np.array([0, 5, 0, 0])
    _, _, costs = orc.lattice(lp[..., 0], lp[..., 1], T_len, U_len)
    scores, frames, _ = align_batch(lp, T_len, U_len, viterbi_f64)
    np.testing.assert_allclose(scores, -costs, rtol=1e-12)
    assert frames[1].tolist() == [0] * 5 and (frames[[0, 2, 3]] == -1).all()


def test_viterbi_entry_rejects_bad_arguments_without_device():
    from rnnt_b200 import _lib
    L = _lib.lib()
    out = 4096                                               # never dereferenced: every call fails its host checks

    def call(B=2, T=8, U1=5, frames=out, scores=out):
        return L.rnnt_b200_viterbi(None, None, None, B, T, U1, frames, scores, None)

    def err():
        return L.rnnt_b200_last_error()

    for kw in (dict(B=0), dict(T=0), dict(U1=0), dict(B=-1)):
        assert call(**kw) == -1 and b"invalid shape" in err(), kw
    assert call(scores=None) == -1 and b"required" in err()
    assert call(frames=None) == -1 and b"required" in err()
    assert call(U1=1025) == -5 and b"U+1 <= 1024" in err()
    assert call(T=1729, U1=1024) == -5 and b"T <= 1728" in err()
    assert call(T=14433, U1=101) == -5 and b"T <= 14432" in err()
    assert call(T=1 << 30, U1=32) == -5 and b"shared memory" in err()


def test_python_align_checks_mirror_the_loss():
    import rnnt_b200
    B, T, U, H, V = 2, 6, 3, 16, 8
    enc, pred = torch.randn(B, T, H), torch.randn(B, U + 1, H)
    W, b = torch.randn(V, H), torch.randn(V)
    tg = torch.zeros(B, U, dtype=torch.int32)
    tl, ul = torch.full((B,), T, dtype=torch.int32), torch.full((B,), U, dtype=torch.int32)
    fa = rnnt_b200.joint_forced_align
    with pytest.raises(RuntimeError, match="targets must be int32"):
        fa(enc, pred, W, b, tg.long(), tl, ul)
    with pytest.raises(RuntimeError, match="logit_lengths must be int32"):
        fa(enc, pred, W, b, tg, tl.long(), ul)
    with pytest.raises(RuntimeError, match="joint inputs must be float32"):
        fa(enc.double(), pred, W, b, tg, tl, ul)
    with pytest.raises(RuntimeError, match="input length mismatch"):
        fa(enc, pred, W, b, tg, tl - 1, ul)
    with pytest.raises(RuntimeError, match="output length mismatch"):
        fa(enc, pred, W, b, tg, tl, ul - 1)
    with pytest.raises(RuntimeError, match="blank must be within"):
        fa(enc, pred, W, b, tg, tl, ul, blank=V)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fa(enc, pred, W, b, tg, tl, ul)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.JointNetwork(-1, -1, H, V).align(enc, pred, tg, tl, ul)
    logits = torch.randn(B, T, U + 1, V)
    with pytest.raises(RuntimeError, match="logits must be float32"):
        rnnt_b200.forced_align(logits.double(), tg, tl, ul)
    with pytest.raises(RuntimeError, match="logits must be contiguous"):
        rnnt_b200.forced_align(logits.transpose(1, 2).contiguous().transpose(1, 2), tg, tl, ul)
    with pytest.raises(RuntimeError, match="target_lengths must be int32"):
        rnnt_b200.forced_align(logits, tg, tl, ul.long())
    with pytest.raises(RuntimeError, match="input length mismatch"):
        rnnt_b200.forced_align(logits, tg, tl - 1, ul)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.forced_align(logits, tg, tl, ul)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.viterbi(torch.zeros(B, T, U + 1, 2), tl, ul)
    with pytest.raises(RuntimeError, match="int32"):
        rnnt_b200.viterbi(torch.zeros(B, T, U + 1, 2), tl.long(), ul)


# ---------------------------------------------------------------------------------------------------------- GPU tests

def _kernel(lp, T_len, U_len):
    import rnnt_b200
    frames, score = rnnt_b200.viterbi(torch.from_numpy(lp).cuda(), torch.from_numpy(T_len).cuda(),
                                      torch.from_numpy(U_len).cuda())
    return frames.cpu().numpy(), score.cpu().numpy()


def _same(kernel, want):
    frames, score = kernel
    s_want, f_want, _ = want
    np.testing.assert_array_equal(frames, f_want)
    np.testing.assert_array_equal(score.view(np.int32), s_want.view(np.int32))     # bit for bit (NaN included)


# (B, T, U1): ragged lengths with U_b = 0 and T_b = 1, 32 .. 1024 threads, T at the shared-memory limit of 1024 and
# of 101 columns
KERNEL_SHAPES = [(5, 37, 9), (4, 50, 33), (3, 200, 101), (3, 64, 1024), (2, 1728, 1024), (1, 14432, 101)]


def _lengths(rng, B, T, U1):
    T_len = rng.integers(1, T + 1, B).astype(np.int32)
    U_len = rng.integers(0, U1, B).astype(np.int32)
    T_len[0], U_len[0] = T, U1 - 1
    if B > 2:
        U_len[1] = 0
        T_len[2] = 1
    return T_len, U_len


@gpu
@pytest.mark.parametrize("quantised", [False, True])
@pytest.mark.parametrize("shape", KERNEL_SHAPES)
def test_kernel_is_bit_identical_to_the_f32_restatement(shape, quantised):
    B, T, U1 = shape
    rng = np.random.default_rng(B * 7919 + T * 31 + U1 + quantised)
    lp = _rand_lp(rng, B, T, U1, quantised)
    T_len, U_len = _lengths(rng, B, T, U1)
    want = align_batch(lp, T_len, U_len)
    got = _kernel(lp, T_len, U_len)
    _same(got, want)
    # cells outside each utterance, and lpE in its last column, are never read
    lp_nan = lp.copy()
    for b in range(B):
        lp_nan[b, T_len[b]:] = np.nan
        lp_nan[b, :, U_len[b] + 1:] = np.nan
        lp_nan[b, :, U_len[b], 1] = np.nan
    _same(_kernel(lp_nan, T_len, U_len), want)
    # every utterance gets the same bits alone, at another batch position, and in a second run
    perm = rng.permutation(B)
    f_p, s_p = _kernel(np.ascontiguousarray(lp[perm]), T_len[perm], U_len[perm])
    np.testing.assert_array_equal(f_p, got[0][perm])
    np.testing.assert_array_equal(s_p.view(np.int32), got[1][perm].view(np.int32))
    f_1, s_1 = _kernel(np.ascontiguousarray(lp[-1:]), T_len[-1:], U_len[-1:])
    np.testing.assert_array_equal(f_1[0], got[0][-1])
    assert s_1.view(np.int32)[0] == got[1].view(np.int32)[-1]
    _same(_kernel(lp, T_len, U_len), want)


@gpu
def test_out_of_range_lengths_poison_only_their_row():
    rng = np.random.default_rng(11)
    B, T, U1 = 5, 30, 12
    lp = _rand_lp(rng, B, T, U1)
    T_len, U_len = _lengths(rng, B, T, U1)
    T_len[1], U_len[3], T_len[4] = T + 1, U1, 0
    frames, score = _kernel(lp, T_len, U_len)
    s, f, _ = align_batch(lp, T_len, U_len)
    for b in (1, 3, 4):
        assert np.isnan(score[b]) and (frames[b] == -1).all()
    _same((frames, score), (s, f, None))


@gpu
def test_single_column_needs_no_frames_buffer():
    import rnnt_b200
    rng = np.random.default_rng(2)
    lp = _rand_lp(rng, 3, 10, 1)
    T_len, U_len = np.array([10, 4, 1], np.int32), np.zeros(3, np.int32)
    frames, score = rnnt_b200.viterbi(torch.from_numpy(lp).cuda(), torch.from_numpy(T_len).cuda(),
                                      torch.from_numpy(U_len).cuda())
    assert frames.shape == (3, 0)
    np.testing.assert_array_equal(score.cpu().numpy(), align_batch(lp, T_len, U_len)[0])


def _lp_f64(enc, pred, W, b, targets, blank, audio_ln=None, text_ln=None):
    """(B,T,U1,2) fp64 log-probs of the joint on the GPU in fp64, one utterance at a time."""
    d = lambda x: x.detach().to("cuda", torch.float64)
    enc, pred, W, b = d(enc), d(pred), d(W), d(b)
    if audio_ln is not None:
        enc = enc @ d(audio_ln[0]).T + d(audio_ln[1])
    if text_ln is not None:
        pred = pred @ d(text_ln[0]).T + d(text_ln[1])
    V = W.shape[0]
    blank = blank % V
    out = []
    for i in range(enc.shape[0]):
        logits = torch.tanh(enc[i].unsqueeze(1) + pred[i].unsqueeze(0)) @ W.T + b
        lsm = torch.log_softmax(logits, -1)
        tg = targets[i].long().to("cuda")
        lpE = torch.full(lsm.shape[:2], float("-inf"), dtype=torch.float64, device="cuda")
        lpE[:, :-1] = lsm[:, :-1].gather(2, tg.view(1, -1, 1).expand(lsm.shape[0], -1, 1)).squeeze(2)
        out.append(torch.stack([lsm[..., blank], lpE], -1))
    return torch.stack(out).cpu().numpy()


def _check_against_fp64(al, lp32, lp64, T_len, U_len, gap_floor, log_prob_want=None):
    """The fused / dense alignment `al` against the fp32 restatement on the same log-probs and against fp64."""
    frames, score, log_prob = (x.cpu().numpy() for x in al)
    _same((frames, score), align_batch(lp32, T_len, U_len))
    s64, f64, floors = align_batch(lp64, T_len, U_len, viterbi_f64)
    if log_prob_want is not None:
        assert np.abs(log_prob - log_prob_want).max() <= LOSS_RTOL * np.abs(log_prob_want).max()
    assert (score <= log_prob + 1e-5 * np.abs(log_prob)).all(), (score, log_prob)
    assert (np.abs(score - s64) <= SCORE_RTOL * np.abs(s64)).all(), (score, s64)
    decided = 0
    for b in range(len(T_len)):
        Tb, Ub = int(T_len[b]), int(U_len[b])
        mine = path_log_prob(lp64[b, :, :, 0], lp64[b, :, :, 1], frames[b, :Ub].tolist(), Tb)
        assert abs(mine - s64[b]) <= SCORE_RTOL * abs(s64[b]), (b, mine, s64[b])
        if floors[b] > gap_floor:
            decided += 1
            np.testing.assert_array_equal(frames[b], f64[b])
    assert decided >= 1, floors
    return dict(score_err=float(np.max(np.abs(score - s64) / np.abs(s64))), floors=floors.tolist())


def _fused_case(enc, pred, W, b, targets, T_len, U_len, blank, log_prob_want):
    import rnnt_b200
    al = rnnt_b200.joint_forced_align(enc, pred, W, b, targets, T_len, U_len, blank=blank)
    assert all(not x.requires_grad for x in al)
    assert al.frames.dtype == torch.int32 and al.frames.shape == targets.shape
    with torch.no_grad():
        _, res = rnnt_b200.joint_rnnt_loss(enc, pred, W, b, targets, T_len, U_len, blank=blank, reduction="none",
                                           return_residuals=True)
    lp32 = res["lp"].cpu().numpy()
    lp64 = _lp_f64(enc, pred, W, b, targets, blank)
    if log_prob_want is None:
        from oracle import rnnt_oracle as orc
        log_prob_want = -orc.lattice_fast(lp64[..., 0], lp64[..., 1], T_len.cpu().numpy(), U_len.cpu().numpy())[2]
    rec = _check_against_fp64(al, lp32, lp64, T_len.cpu().numpy(), U_len.cpu().numpy(), GAP_FLOOR, log_prob_want)
    again = rnnt_b200.joint_forced_align(enc, pred, W, b, targets, T_len, U_len, blank=blank)
    for x, y in zip(al, again):
        assert torch.equal(x, y)
    return rec


@gpu
@pytest.mark.parametrize("name", ["loss_tiny", "loss_mid", "loss_wide"])
def test_fused_alignment_on_golden_cases(golden_dir, name):
    from helpers import load_loss_golden
    g = load_loss_golden(golden_dir, name)
    t = lambda k, dt=None: torch.from_numpy(g[k]).cuda() if dt is None else torch.from_numpy(g[k]).to(dt).cuda()
    # the encoder features as the (B,T,H) view of a (B,H,T) tensor, as the model hands them over
    enc = t("enc").permute(0, 2, 1).contiguous().permute(0, 2, 1)
    _fused_case(enc, t("pred"), t("W"), t("b"), t("targets", torch.int32), t("T_len", torch.int32),
                t("U_len", torch.int32), -1, -g["costs"])


@gpu
@pytest.mark.parametrize("blank", [-1, 0])
def test_fused_alignment_full_width(blank):
    from helpers import make_inputs
    inp = make_inputs(4, 400, 100, 1024, 1024, seed=77, ragged=True)
    enc = inp["enc"].permute(0, 2, 1).contiguous().permute(0, 2, 1)     # (B,H,T) storage
    targets = inp["targets"] if blank == -1 else inp["targets"] + 1     # labels never equal the blank
    _fused_case(enc, inp["pred"], inp["W"], inp["b"], targets, inp["T_len"], inp["U_len"], blank, None)


@gpu
def test_dense_alignment(golden_dir):
    import rnnt_b200
    from helpers import load_loss_golden
    from rnnt_b200.functional import _dense_forward
    g = load_loss_golden(golden_dir, "loss_tiny")
    rng = np.random.default_rng(4)
    B, T, U, V = 3, 60, 20, 64
    cases = [(g["logits"], g["targets"], g["T_len"], g["U_len"], -g["costs"]),
             ((rng.standard_normal((B, T, U + 1, V)) * 2).astype(np.float32),
              rng.integers(0, V - 1, (B, U)).astype(np.int32), np.array([T, 41, 1], np.int32),
              np.array([U, 0, 7], np.int32), None)]
    for logits, targets, T_len, U_len, want in cases:
        c = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
        lg, tg, tl, ul = (c(logits), c(targets).to(torch.int32), c(T_len).to(torch.int32),
                          c(U_len).to(torch.int32))
        al = rnnt_b200.forced_align(lg, tg, tl, ul)
        lp32 = _dense_forward(lg, tg, tl, ul, -1)[1].cpu().numpy()
        from oracle import rnnt_oracle as orc
        _, lpB, lpE = orc.log_probs(logits.astype(np.float64), targets, -1)
        lp64 = np.stack([lpB, lpE], -1)
        if want is None:
            want = -orc.lattice_fast(lpB, lpE, T_len, U_len)[2]
        _check_against_fp64(al, lp32, lp64, T_len, U_len, GAP_FLOOR_DENSE, want)
        for x, y in zip(al, rnnt_b200.forced_align(lg, tg, tl, ul)):
            assert torch.equal(x, y)


@gpu
def test_lazy_handle_aligns_through_the_fused_path():
    import rnnt_b200
    from helpers import make_inputs
    inp = make_inputs(2, 30, 8, 64, 256, ragged=True)
    lazy = rnnt_b200.LazyJointLogits(inp["enc"], inp["pred"], inp["W"], inp["b"])
    a = rnnt_b200.forced_align(lazy, inp["targets"], inp["T_len"], inp["U_len"])
    b = rnnt_b200.joint_forced_align(inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"],
                                     inp["U_len"])
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@gpu
def test_model_align_equals_the_fused_call_on_its_features():
    import rnnt_b200
    from helpers import StubEncoder
    torch.manual_seed(3)
    n_mels, H, V, E, B, L, U = 12, 64, 40, 32, 3, 50, 9
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.3), StubEncoder(n_mels, H),
                                rnnt_b200.JointNetwork(-1, -1, H, V)).cuda().eval()
    mel = torch.randn(B, n_mels, L, device="cuda")
    mel_lens = torch.tensor([L, 37, 20], device="cuda")
    ids = torch.randint(0, V - 1, (B, U), device="cuda")
    id_lens = torch.tensor([U, 4, 0], device="cuda")
    al = model.align(mel, mel_lens, ids, id_lens, V - 1)
    with torch.no_grad():
        feats = model.predictor(torch.cat([torch.full((B, 1), V - 1, device="cuda", dtype=ids.dtype), ids], 1))
        audio = model.encoder(mel).permute(0, 2, 1)
        lens = model.encoder.calc_output_lens(mel_lens)
    want = rnnt_b200.joint_forced_align(audio, feats, model.joint.joint_ln.weight, model.joint.joint_ln.bias,
                                        ids.int(), lens.int(), id_lens.int())
    for x, y in zip(al, want):
        assert torch.equal(x, y)
    assert (al.frames[2] == -1).all() and (al.frames[1, 4:] == -1).all() and (al.frames[1, :4] >= 0).all()
    assert (al.score <= al.log_prob + 1e-5 * al.log_prob.abs()).all()


@gpu
def test_joint_align_with_preprojections():
    import rnnt_b200
    from rnnt_b200.functional import linear
    torch.manual_seed(5)
    B, T, U, Fa, Ft, H, V = 2, 40, 10, 48, 24, 64, 128
    joint = rnnt_b200.JointNetwork(Fa, Ft, H, V).cuda()
    a, p = torch.randn(B, T, Fa, device="cuda"), torch.randn(B, U + 1, Ft, device="cuda")
    tg = torch.randint(0, V - 1, (B, U), dtype=torch.int32, device="cuda")
    tl, ul = torch.tensor([T, 25], dtype=torch.int32, device="cuda"), torch.tensor([U, 6], dtype=torch.int32,
                                                                                     device="cuda")
    al = joint.align(a, p, tg, tl, ul)
    with torch.no_grad():
        want = rnnt_b200.joint_forced_align(linear(a, joint.audio_ln.weight, joint.audio_ln.bias),
                                            linear(p, joint.text_ln.weight, joint.text_ln.bias),
                                            joint.joint_ln.weight, joint.joint_ln.bias, tg, tl, ul)
    for x, y in zip(al, want):
        assert torch.equal(x, y)
    lp64 = _lp_f64(a, p, joint.joint_ln.weight, joint.joint_ln.bias, tg, -1,
                   (joint.audio_ln.weight, joint.audio_ln.bias), (joint.text_ln.weight, joint.text_ln.bias))
    s64, _, _ = align_batch(lp64, tl.cpu().numpy(), ul.cpu().numpy(), viterbi_f64)
    score = al.score.cpu().numpy()
    # fp16 operands in the two pre-projections as well as in the joint
    assert (np.abs(score - s64) <= 10 * SCORE_RTOL * np.abs(s64)).all(), (score, s64)
