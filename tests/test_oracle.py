"""Pin the CPU oracle against golden vectors produced by the reference itself (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

from helpers import load_loss_golden
from oracle import rnnt_oracle as orc


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


@pytest.mark.parametrize("name", ["loss_tiny", "loss_mid", "loss_wide"])
def test_oracle_costs_and_grads_match_reference(golden_dir, name):
    g = load_loss_golden(golden_dir, name)
    out = orc.loss_and_grads(g["enc"], g["pred"], g["W"], g["b"], g["targets"], g["T_len"], g["U_len"], blank=-1)
    out["dW"] = out["dW"][g["dW_rows"]]
    np.testing.assert_allclose(out["costs"], g["costs"], rtol=2e-6, atol=2e-5)
    assert abs(out["costs"].mean() - float(g["loss_mean"])) < 1e-4 * abs(float(g["loss_mean"]))
    for k in ("d_enc", "d_pred", "dW", "db"):
        ref = g[k]
        err = np.abs(out[k] - ref).max()
        assert err <= 1e-4 * max(1.0, np.abs(ref).max()), (k, err)   # fp32 reference rounding


def test_oracle_slow_and_fast_lattice_agree(golden_dir):
    g = _load(golden_dir, "loss_tiny")
    logits = orc.joint_logits(g["enc"], g["pred"], g["W"], g["b"])
    lse, lpB, lpE = orc.log_probs(logits, g["targets"], -1)
    a1, b1, c1 = orc.lattice(lpB, lpE, g["T_len"], g["U_len"])
    a2, b2, c2 = orc.lattice_fast(lpB, lpE, g["T_len"], g["U_len"])
    np.testing.assert_allclose(c1, c2, rtol=1e-12)
    m = np.isfinite(a1)
    np.testing.assert_allclose(a1[m], a2[m], rtol=1e-12, atol=1e-12)
    m = np.isfinite(b1)
    np.testing.assert_allclose(b1[m], b2[m], rtol=1e-12, atol=1e-12)


def test_oracle_logits_and_logit_grads(golden_dir):
    g = _load(golden_dir, "loss_tiny")
    logits = orc.joint_logits(g["enc"], g["pred"], g["W"], g["b"])
    np.testing.assert_allclose(logits, g["logits"], rtol=0, atol=5e-6)
    lse, lpB, lpE = orc.log_probs(logits, g["targets"], -1)
    al, be, _ = orc.lattice(lpB, lpE, g["T_len"], g["U_len"])
    dl = orc.logit_grads(logits, g["targets"], g["T_len"], g["U_len"], -1, lse, lpB, lpE, al, be)
    np.testing.assert_allclose(dl, g["dlogits"], rtol=0, atol=3e-6)
    # padded cells: exactly zero gradient; valid cells: rows sum to ~0
    B, T, U1, V = dl.shape
    for b in range(B):
        Tb, Ub = int(g["T_len"][b]), int(g["U_len"][b])
        assert not dl[b, Tb:].any() and not dl[b, :, Ub + 1:].any()
        assert np.abs(dl[b, :Tb, :Ub + 1].sum(-1)).max() < 1e-12


def test_oracle_known_answers():
    rng = np.random.default_rng(0)
    # U_b = 0: the only path is all blanks -> cost = -sum_t lpB[t,0]
    T, V = 5, 7
    logits = rng.normal(size=(1, T, 1, V))
    lse, lpB, lpE = orc.log_probs(logits, np.zeros((1, 0), np.int32), -1)
    _, _, c = orc.lattice(lpB, lpE, [T], [0])
    assert abs(c[0] + lpB[0, :, 0].sum()) < 1e-12
    # T_b = 1: emit all U labels then one blank
    U = 3
    logits = rng.normal(size=(1, 1, U + 1, V))
    tg = rng.integers(0, V - 1, size=(1, U))
    lse, lpB, lpE = orc.log_probs(logits, tg, -1)
    _, _, c = orc.lattice(lpB, lpE, [1], [U])
    assert abs(c[0] + lpE[0, 0, :U].sum() + lpB[0, 0, U]) < 1e-12


def test_oracle_greedy_decode_matches_reference(golden_dir):
    g = _load(golden_dir, "decode_small")
    sd = {k[5:]: g[k] for k in g.files if k.startswith("pred.")}
    V = g["W"].shape[0]
    off = 0
    for i, n in enumerate(g["tok_len"]):
        want = g["tok_flat"][off:off + n].tolist()
        off += n
        got, margins = orc.greedy_decode(g["feats"][i], int(g["T_len"][i]), g["W"], g["b"], sd, blank=V - 1,
                                         max_length=int(g["max_length"]))
        assert got == want, (i, min(margins))


def test_oracle_preprojection_joint_matches_reference(golden_dir):
    """audio_ln / text_ln variant (rnnt/joint.py:8-12,26-30), vectors from the reference module."""
    g = _load(golden_dir, "loss_proj")
    P = lambda k: g["param." + k]
    out = orc.loss_and_grads(g["audio"], g["text"], P("joint_ln.weight"), P("joint_ln.bias"), g["targets"], g["T_len"],
                             g["U_len"], blank=-1, audio_ln=(P("audio_ln.weight"), P("audio_ln.bias")),
                             text_ln=(P("text_ln.weight"), P("text_ln.bias")))
    np.testing.assert_allclose(out["costs"], g["costs"], rtol=2e-6, atol=2e-5)
    pairs = [("d_enc", "d_audio"), ("d_pred", "d_text"), ("dW", "grad.joint_ln.weight"), ("db", "grad.joint_ln.bias"),
             ("dWa", "grad.audio_ln.weight"), ("dba", "grad.audio_ln.bias"), ("dWt", "grad.text_ln.weight"),
             ("dbt", "grad.text_ln.bias")]
    for mine, ref in pairs:
        err = np.abs(out[mine] - g[ref]).max()
        assert err <= 1e-4 * max(1.0, np.abs(g[ref]).max()), (mine, err)


def test_oracle_model_forward_glue_matches_reference(golden_dir):
    """rnnt/model.py:17-43: blank prepend (:20-21), permuted encoder view (:28), calc_output_lens (:29), .int() casts
    (:36-38), reduction="mean".  Encoder / predictor features come from this repo's module mirrors loaded with the
    golden parameters; the oracle supplies joint + loss; the scalar must equal the reference's."""
    import torch
    import rnnt_b200
    from helpers import StubEncoder
    g = _load(golden_dir, "model_forward")
    V, H = g["param.joint.joint_ln.weight"].shape
    E = g["param.predictor.embedding.weight"].shape[1]
    pred_m = rnnt_b200.ConvPredictor(V, H, E, 0.0)
    pred_m.load_state_dict({k[16:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("param.predictor.")})
    enc_m = StubEncoder(g["mel"].shape[1], H)
    enc_m.load_state_dict({k[14:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("param.encoder.")})
    ids = torch.from_numpy(g["input_ids"])
    with torch.no_grad():
        prepended = torch.cat([torch.full((ids.shape[0], 1), V - 1, dtype=ids.dtype), ids], 1)
        dec = pred_m(prepended).numpy()
        audio = enc_m(torch.from_numpy(g["mel"])).permute(0, 2, 1).numpy()
        lens = enc_m.calc_output_lens(torch.from_numpy(g["mel_lens"])).numpy()
    out = orc.loss_and_grads(audio, dec, g["param.joint.joint_ln.weight"], g["param.joint.joint_ln.bias"],
                             g["input_ids"].astype(np.int32), lens, g["id_lens"], blank=-1)
    assert abs(out["costs"].mean() - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))


def test_oracle_greedy_decode_full_width_matches_reference(golden_dir):
    """H = V = 1024, E = 512 (BASELINE configs[4] width): the fp64 oracle loop reproduces the reference's tokens up to the
    first near-tie (top-2 gap < 1e-4) of each utterance.  Three utterances (the fp64 full re-run is slow)."""
    from helpers import decode_full_setup
    g = _load(golden_dir, "decode_full")
    model, feats, T_len = decode_full_setup(g)
    sd = {k: v.numpy() for k, v in model.predictor.state_dict().items()}
    W = model.joint.joint_ln.weight.detach().numpy()
    b = model.joint.joint_ln.bias.detach().numpy()
    offs = np.concatenate([[0], np.cumsum(g["tok_len"])])
    for i in (3, 7, 1):
        want = g["tok_flat"][offs[i]:offs[i + 1]].tolist()
        got, margins = orc.greedy_decode(feats[i].numpy(), int(T_len[i]), W, b, sd, blank=int(g["V"]) - 1,
                                         max_length=int(g["max_length"]))
        safe = int(g["safe_len"][i])
        assert got[:safe] == want[:safe], (i, min(margins))
        if safe == len(want):
            assert got == want
