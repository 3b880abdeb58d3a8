"""GPU parity tests (-m gpu): the CUDA path, called through the C-ABI / public API, against the oracle.

Tolerances (stated once):
  * per-utterance loss: relative 1e-4 vs the fp32 reference (north_star bar); fp16-operand tensor-core GEMM inside;
  * gradients (fp16 activations / weights / logit-gradients, fp32 accumulation): relative Frobenius error <= 2e-3 vs the
    fp32 reference and <= 1e-3 vs a reference whose joint GEMM operands are rounded to fp16 (measured at H=V=1024:
    2.5e-4 / 1.5e-4; the same path run by torch in bf16 is ~10x worse -- test_full_size_vs_reference prints both);
  * lattice / dense-logits kernels (fp32 throughout): 1e-5 relative;  decode tokens: exact.
"""
import os

import numpy as np
import pytest
import torch

from helpers import fused_raw, load_loss_golden, make_inputs, rel_err, torch_reference

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-4
GRAD_TOL_FP32 = 2e-3     # vs the fp32 reference
GRAD_TOL_F16 = 1e-3      # vs a reference whose GEMM operands are rounded to fp16 like the kernels' (isolates kernel bugs)
GRAD_TOL_TINY = 6e-3     # shapes with H < 64: a handful of products per logit, fp16 rounding does not average out


def _golden(golden_dir, name):
    g = load_loss_golden(golden_dir, name)
    t = lambda k, dt=None: torch.from_numpy(g[k]).cuda() if dt is None else torch.from_numpy(g[k]).to(dt).cuda()
    inp = dict(enc=t("enc"), pred=t("pred"), W=t("W"), b=t("b"), targets=t("targets", torch.int32),
               T_len=t("T_len", torch.int32), U_len=t("U_len", torch.int32))
    return g, inp


@pytest.mark.parametrize("name", ["loss_tiny", "loss_mid", "loss_wide"])
def test_fused_matches_reference_golden(golden_dir, name):
    """Committed vectors produced by the reference itself (JointNetwork + torchaudio rnnt_loss, fp32 CPU)."""
    g, inp = _golden(golden_dir, name)
    out = fused_raw(inp)
    assert out["status"] == 0
    out["dW"] = out["dW"][torch.from_numpy(g["dW_rows"]).long().cuda()]
    costs = out["costs"].cpu().numpy()
    assert np.abs(costs - g["costs"]).max() <= LOSS_RTOL * np.abs(g["costs"]).max(), (costs, g["costs"])
    for k in ("d_enc", "d_pred", "dW", "db"):
        r, _ = rel_err(out[k].cpu(), torch.from_numpy(g[k]))
        assert r <= GRAD_TOL_FP32, (k, r)


@pytest.mark.parametrize("shape", [(2, 20, 9, 64, 256, True), (3, 37, 13, 128, 512, True),
                                   (2, 33, 17, 1024, 1024, False), (4, 200, 40, 1024, 1024, False)])
def test_fused_vs_oracle_same_device(shape):
    """Config (i) of BASELINE.json (B=4,T=200,U=40,H=V=1024) and smaller ragged cases vs the torchaudio path."""
    B, T, U, H, V, ragged = shape
    inp = make_inputs(B, T, U, H, V, ragged=ragged)
    ref = torch_reference(inp)
    refq = torch_reference(inp, emulate_bf16=True)
    out = fused_raw(inp)
    r, _ = rel_err(out["costs"], ref["costs"])
    assert (out["costs"] - ref["costs"]).abs().max() <= LOSS_RTOL * ref["costs"].abs().max()
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert rel_err(out[k], ref[k])[0] <= GRAD_TOL_FP32, (k, rel_err(out[k], ref[k]))
        assert rel_err(out[k], refq[k])[0] <= GRAD_TOL_F16, (k, rel_err(out[k], refq[k]))


def test_fuzz_small_ragged_shapes_vs_cpu_reference():
    """Random small shapes (odd V, H not a multiple of 64, T=1, U=0, single utterance ...) against torchaudio's CPU path."""
    rng = np.random.default_rng(2024)
    cases = [(1, 1, 0, 8, 2), (2, 1, 3, 16, 5), (3, 9, 0, 24, 37), (1, 40, 20, 72, 300)]
    for _ in range(8):
        cases.append((int(rng.integers(1, 6)), int(rng.integers(1, 41)), int(rng.integers(0, 21)),
                      int(rng.choice([8, 16, 40, 64, 72, 128])), int(rng.choice([2, 3, 37, 256, 257, 300]))))
    for i, (B, T, U, H, V) in enumerate(cases):
        inp = make_inputs(B, T, U, H, V, ragged=True, seed=100 + i)
        ref = torch_reference(inp, device="cpu")
        out = fused_raw(inp)
        assert out["status"] == 0
        err = (out["costs"].cpu() - ref["costs"]).abs()
        # absolute floor: on a lattice of a few cells one cell's fp16 / tanh.approx rounding (~1e-4) is the whole error
        assert (err <= LOSS_RTOL * ref["costs"].abs() + 3e-4).all(), ((B, T, U, H, V), out["costs"], ref["costs"])
        for k in ("d_enc", "d_pred", "dW", "db"):
            r, a = rel_err(out[k].cpu(), ref[k])
            assert r <= GRAD_TOL_FP32 or a < 1e-5, ((B, T, U, H, V), k, r, a)


def test_many_utterances_fall_back_to_global_tile_tables():
    """B above the shared-memory tile-table capacity (340 utterances): the kernels walk the global tables instead."""
    inp = make_inputs(400, 6, 3, 64, 40, ragged=True, seed=77)
    ref = torch_reference(inp, device="cpu")
    out = fused_raw(inp)
    assert out["status"] == 0
    err = (out["costs"].cpu() - ref["costs"]).abs()
    assert (err <= LOSS_RTOL * ref["costs"].abs() + 3e-4).all()
    for k in ("d_enc", "d_pred", "dW", "db"):
        r, a = rel_err(out[k].cpu(), ref[k])
        assert r <= GRAD_TOL_FP32 or a < 1e-5, (k, r, a)


def test_multi_chunk_backward_equals_single_chunk():
    inp = make_inputs(2, 40, 20, 256, 1024, ragged=True)
    one = fused_raw(inp)
    many = fused_raw(inp, ring_tiles=7)
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert rel_err(many[k], one[k])[0] < 1e-5, k


def test_recompute_mode_equals_saved_activation_mode():
    """hidden = NULL: per-SM activation scratch in the forward, producers inside the backward kernel.  Same numbers."""
    import rnnt_b200
    for shape, kw in (((2, 40, 20, 256, 1024), {}), ((3, 50, 11, 72, 300), dict(ring_tiles=5)),
                      ((2, 130, 30, 64, 256), {})):
        inp = make_inputs(*shape, ragged=True, seed=11)
        saved = fused_raw(inp, **kw)
        lean = fused_raw(inp, save_hidden=False, **kw)
        assert torch.equal(saved["costs"], lean["costs"])
        assert torch.equal(saved["lp"], lean["lp"])
        for k in ("d_enc", "d_pred", "dW", "db"):
            assert rel_err(lean[k], saved[k])[0] < 1e-5, (shape, k, rel_err(lean[k], saved[k]))
    # public API: loss-only evaluation (no grad -> no residual buffer) and the save_hidden switch
    inp = make_inputs(2, 40, 20, 256, 1024, ragged=True, seed=11)
    args = (inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"], inp["U_len"])
    with torch.no_grad():
        plain = rnnt_b200.joint_rnnt_loss(inp["enc"], *args, reduction="none")
    grads = []
    for save in (True, False):
        enc = inp["enc"].clone().requires_grad_(True)
        costs = rnnt_b200.joint_rnnt_loss(enc, *args, reduction="none", save_hidden=save)
        assert torch.equal(costs.detach(), plain)
        costs.sum().backward()
        grads.append(enc.grad)
    assert rel_err(grads[1], grads[0])[0] < 1e-5


def test_saved_activations_are_the_fp16_tanh():
    """The residual buffer holds h = tanh(enc+pred) in fp16, one 64-row block per 16(t) x 4(u) half-tile."""
    from helpers import tile_rows
    inp = make_inputs(2, 21, 9, 64, 256, ragged=True, seed=5)
    out = fused_raw(inp)
    h = out["hidden"].view(torch.float16).view(-1, out["Hp"]).float()
    rows = tile_rows(inp["T_len"].cpu(), inp["U_len"].cpu())
    assert h.shape[0] >= len(rows)
    want = torch.tanh(inp["enc"].unsqueeze(2) + inp["pred"].unsqueeze(1))
    for r in range(0, len(rows), 7):
        b, t, u, valid = rows[r]
        if valid:
            assert (h[r, :64] - want[b, t, u]).abs().max() < 2e-3


def test_zero_tile_skipping_is_exact():
    """Tiles dropped from the backward hold only zeros in the fp16 gradient ring: results equal the all-tiles run."""
    inp = make_inputs(2, 160, 40, 128, 512, ragged=True, seed=17)
    dense = fused_raw(inp, flags=1)
    sparse = fused_raw(inp, flags=0)
    assert dense["active_halves"] == dense["total_halves"]   # every half-tile of the lattice
    assert 0 < sparse["active_halves"] < dense["active_halves"]
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert rel_err(sparse[k], dense[k])[0] < 1e-5, (k, rel_err(sparse[k], dense[k]))
    ref = torch_reference(inp)
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert rel_err(sparse[k], ref[k])[0] <= GRAD_TOL_FP32, k


def test_padded_cells_have_zero_gradient_and_edge_lengths():
    # U_b = 0 (pure blank path), T_b = 1, and a fully ragged batch; padded frames / labels get exactly zero grads
    inp = make_inputs(4, 18, 6, 64, 256, ragged=True, seed=7)
    inp["T_len"] = torch.tensor([18, 1, 9, 5], dtype=torch.int32, device="cuda")
    inp["U_len"] = torch.tensor([6, 3, 0, 6], dtype=torch.int32, device="cuda")
    ref = torch_reference(inp, device="cpu")   # torchaudio's CUDA kernels mishandle T_b=1 / U_b=0 rows; its CPU path is the oracle
    out = fused_raw(inp)
    assert ((out["costs"].cpu() - ref["costs"]).abs() <= LOSS_RTOL * ref["costs"].abs()).all(), (out["costs"], ref["costs"])
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert rel_err(out[k].cpu(), ref[k])[0] <= GRAD_TOL_FP32, k
    for b in range(4):
        Tb, Ub = int(inp["T_len"][b]), int(inp["U_len"][b])
        assert not out["d_enc"][b, Tb:].any()
        assert not out["d_pred"][b, Ub + 1:].any()
    # known answer: U_b = 0 -> cost = -sum_t lpB[t, 0]
    b = 2
    assert abs(float(out["costs"][b]) + float(out["lp"][b, :9, 0, 0].sum())) < 1e-3


def test_linearity_in_dcost_and_mean_reduction():
    import rnnt_b200
    inp = make_inputs(3, 25, 7, 64, 256, ragged=True, seed=3)
    one = fused_raw(inp)
    dc = torch.tensor([0.5, -2.0, 3.0], device="cuda")
    scaled = fused_raw(inp, dcost=dc)
    # d_enc rows scale per utterance exactly like dcost (same kernels, same order -> tight tolerance)
    for b in range(3):
        assert rel_err(scaled["d_enc"][b], one["d_enc"][b] * dc[b])[0] < 2e-3
    enc = inp["enc"].clone().requires_grad_(True)
    loss = rnnt_b200.joint_rnnt_loss(enc, inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"],
                                     inp["U_len"], reduction="mean")
    assert abs(float(loss.detach()) - float(one["costs"].mean())) < 1e-4 * abs(float(loss.detach()))
    loss.backward()
    assert rel_err(enc.grad, one["d_enc"] / 3)[0] < 2e-3


def test_clamp_matches_torchaudio(capsys):
    """clamp > 0 (rnnt/optuna.py wanted it; rnnt/model.py:40 passes -1): d cost / d logits clamped to [-clamp, clamp] before
    the dcost scaling.  The oracle is torchaudio's CPU path (the reference arm of this repo)."""
    import torchaudio
    import rnnt_b200
    inp = make_inputs(2, 12, 5, 64, 256, ragged=False, seed=5)
    enc = inp["enc"].clone().requires_grad_(True)
    loss = rnnt_b200.joint_rnnt_loss(enc, inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"],
                                     inp["U_len"], clamp=0.01, reduction="sum")
    loss.backward()
    errs = {}
    for dev in ("cpu", "cuda"):
        cp = {k: v.to(dev) for k, v in inp.items()}
        enc2 = cp["enc"].clone().requires_grad_(True)
        logits = torch.nn.functional.linear(torch.tanh(enc2.unsqueeze(2) + cp["pred"].unsqueeze(1)), cp["W"], cp["b"])
        ref = torchaudio.functional.rnnt_loss(logits, cp["targets"], cp["T_len"], cp["U_len"], clamp=0.01,
                                              reduction="sum")
        ref.backward()
        errs[dev] = rel_err(enc.grad.cpu(), enc2.grad.cpu())[0]
    with capsys.disabled():
        print(f"\n[clamp] d_enc rel err vs torchaudio CPU {errs['cpu']:.2e}, vs torchaudio CUDA {errs['cuda']:.2e}")
    assert errs["cpu"] < GRAD_TOL_FP32, errs


def test_dense_loss_matches_torchaudio_and_golden(golden_dir):
    import torchaudio
    import rnnt_b200
    g, inp = _golden(golden_dir, "loss_tiny")
    logits = torch.from_numpy(g["logits"]).cuda().requires_grad_(True)
    costs = rnnt_b200.rnnt_loss(logits, inp["targets"], inp["T_len"], inp["U_len"], reduction="none")
    costs.sum().backward()
    np.testing.assert_allclose(costs.detach().cpu().numpy(), g["costs"], rtol=1e-5)
    np.testing.assert_allclose(logits.grad.cpu().numpy(), g["dlogits"], atol=2e-6)
    for (B, T, U, V) in [(4, 50, 20, 1024), (2, 400, 100, 64)]:
        i2 = make_inputs(B, T, U, 16, V, ragged=True)
        lg = torch.randn(B, T, U + 1, V, device="cuda").requires_grad_(True)
        l2 = lg.detach().clone().requires_grad_(True)
        mine = rnnt_b200.rnnt_loss(lg, i2["targets"], i2["T_len"], i2["U_len"], reduction="mean")
        ref = torchaudio.functional.rnnt_loss(l2, i2["targets"], i2["T_len"], i2["U_len"], reduction="mean")
        mine.backward(); ref.backward()
        assert abs(float(mine.detach()) - float(ref.detach())) < 1e-5 * abs(float(ref.detach()))
        assert rel_err(lg.grad, l2.grad)[0] < 2e-4


@pytest.mark.parametrize("shape", [(3, 23, 9), (3, 40, 33), (2, 37, 64), (3, 50, 101), (2, 30, 128), (2, 25, 150)])
def test_lattice_kernel_vs_numpy_oracle(shape):
    """Block sizes of 32 .. 160 threads (one thread per lattice column), ragged lengths incl. U_b = 0 and T_b = 1."""
    import rnnt_b200
    from oracle import rnnt_oracle as orc
    rng = np.random.default_rng(0)
    B, T, U1 = shape
    lp = np.log(rng.uniform(0.05, 0.9, size=(B, T, U1, 2))).astype(np.float32)
    T_len = np.array([T, max(1, T // 2), 1][:B], np.int32)
    U_len = np.array([U1 - 1, 0, min(5, U1 - 1)][:B], np.int32)
    al, be, co = rnnt_b200.lattice(torch.from_numpy(lp).cuda(), torch.from_numpy(T_len).cuda(),
                                   torch.from_numpy(U_len).cuda())
    a_ref, b_ref, c_ref = orc.lattice(lp[..., 0].astype(np.float64), lp[..., 1].astype(np.float64), T_len, U_len)
    np.testing.assert_allclose(co.cpu().numpy(), c_ref, rtol=1e-5)
    for b in range(B):
        sl = (b, slice(0, T_len[b]), slice(0, U_len[b] + 1))
        np.testing.assert_allclose(al.cpu().numpy()[sl], a_ref[sl], rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(be.cpu().numpy()[sl], b_ref[sl], rtol=1e-5, atol=1e-4)
        # the two recursions agree on the total: -beta(0,0) == -(alpha(Tb-1,Ub) + lpB(Tb-1,Ub))
        tail = al.cpu().numpy()[b, T_len[b] - 1, U_len[b]] + lp[b, T_len[b] - 1, U_len[b], 0]
        assert abs(tail + co.cpu().numpy()[b]) < 1e-3 * max(1.0, abs(tail))


def test_error_behaviour_mirrors_torchaudio():
    import rnnt_b200
    inp = make_inputs(2, 10, 4, 64, 256)
    with pytest.raises(RuntimeError, match="targets must be int32"):
        rnnt_b200.joint_rnnt_loss(inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"].long(), inp["T_len"],
                                  inp["U_len"])
    bad_T = inp["T_len"].clone(); bad_T[:] = 9
    with pytest.raises(RuntimeError, match="input length mismatch"):
        rnnt_b200.joint_rnnt_loss(inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"], bad_T, inp["U_len"])
    bad_U = inp["U_len"].clone(); bad_U[:] = 3
    with pytest.raises(RuntimeError, match="output length mismatch"):
        rnnt_b200.joint_rnnt_loss(inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"], bad_U)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rnnt_b200.joint_rnnt_loss(inp["enc"].cpu(), inp["pred"].cpu(), inp["W"].cpu(), inp["b"].cpu(),
                                  inp["targets"].cpu(), inp["T_len"].cpu(), inp["U_len"].cpu())
    logits = torch.randn(2, 10, 5, 7, device="cuda")
    with pytest.raises(RuntimeError, match="logits must be contiguous"):
        rnnt_b200.rnnt_loss(logits.transpose(1, 2).contiguous().transpose(1, 2), inp["targets"], inp["T_len"],
                            inp["U_len"])


def test_joint_module_dropin_and_zero_edit_mode():
    """JointNetwork keeps the reference's state_dict keys; the unmodified model.py:32-41 call pattern runs fused."""
    import torchaudio
    import rnnt_b200
    torch.manual_seed(1)
    joint = rnnt_b200.JointNetwork(-1, -1, 64, 256).cuda()
    assert sorted(joint.state_dict().keys()) == ["joint_ln.bias", "joint_ln.weight"]
    full = rnnt_b200.JointNetwork(32, 48, 64, 256).cuda()
    assert "audio_ln.weight" in full.state_dict() and "text_ln.bias" in full.state_dict()
    inp = make_inputs(2, 14, 6, 64, 256)
    dense = joint(inp["enc"], inp["pred"])
    assert dense.shape == (2, 14, 7, 256)
    ref = torchaudio.functional.rnnt_loss(dense, inp["targets"], inp["T_len"], inp["U_len"], blank=-1, clamp=-1,
                                          reduction="mean")
    rnnt_b200.enable_zero_edit_mode(joint)
    lazy = joint(inp["enc"], inp["pred"])                       # what rnnt/model.py:32 receives
    assert isinstance(lazy, rnnt_b200.LazyJointLogits) and lazy.shape == dense.shape
    loss = torchaudio.functional.rnnt_loss(logits=lazy, targets=inp["targets"], logit_lengths=inp["T_len"],
                                           target_lengths=inp["U_len"], blank=-1, clamp=-1, reduction="mean")
    assert abs(float(loss) - float(ref)) < LOSS_RTOL * abs(float(ref))
    loss.backward()
    assert joint.joint_ln.weight.grad is not None and joint.joint_ln.bias.grad is not None
    # pre-projection variant (non-"convjs" configs, joint.py:8-12): grads reach audio_ln / text_ln
    a = torch.randn(2, 14, 32, device="cuda"); t = torch.randn(2, 7, 48, device="cuda")
    l2 = full.loss(a, t, inp["targets"], inp["T_len"], inp["U_len"])
    l2.backward()
    assert all(p.grad is not None for p in full.parameters())
    with torch.no_grad():
        d2 = full(a, t)
    r2 = torchaudio.functional.rnnt_loss(d2, inp["targets"], inp["T_len"], inp["U_len"], reduction="mean")
    assert abs(float(l2) - float(r2)) < LOSS_RTOL * abs(float(r2))


def test_greedy_decode_matches_reference_golden(golden_dir):
    """Token sequences produced by the reference's RNNTModel._greedy_decode_conv (fp32 CPU) -- must be exact."""
    import rnnt_b200
    g = np.load(os.path.join(golden_dir, "decode_small.npz"))
    V, H = g["W"].shape
    E = g["pred.embedding.weight"].shape[1]
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    joint.load_state_dict({"joint_ln.weight": torch.from_numpy(g["W"]), "joint_ln.bias": torch.from_numpy(g["b"])})
    pred = rnnt_b200.ConvPredictor(V, H, E, 0.3)
    pred.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("pred.")})
    model = rnnt_b200.RNNTModel(pred, torch.nn.Identity(), joint).cuda().eval()
    feats = torch.from_numpy(g["feats"]).cuda()
    got, margins = model.greedy_decode_features(feats, torch.from_numpy(g["T_len"]), max_length=int(g["max_length"]),
                                                return_margins=True)
    off = 0
    for i, n in enumerate(g["tok_len"]):
        want = g["tok_flat"][off:off + n].tolist()
        off += n
        assert got[i] == want, (i, min(margins[i]))
    # the torch-op device loop (CUDA graph replay and eager) and the host-driven loop agree with the persistent kernel
    for graph in (True, False):
        assert model.greedy_decode_features(feats, torch.from_numpy(g["T_len"]), max_length=int(g["max_length"]),
                                            use_cuda_graph=graph, engine="graph") == got
    assert model._greedy_decode_features_hostloop(feats, torch.from_numpy(g["T_len"]),
                                                  max_length=int(g["max_length"])) == got
    # reference-signature entry: batch of one through an (identity) encoder, list[int] out
    one = model.greedy_decode(feats[:1, : int(g["T_len"][0])].permute(0, 2, 1), torch.tensor([int(g["T_len"][0])]),
                              max_length=int(g["max_length"]))
    assert one == got[0]


def test_decode_step_full_width_vs_fp64():
    import rnnt_b200
    torch.manual_seed(0)
    N, H, V = 64, 1024, 1024
    a, p = torch.randn(N, H, device="cuda"), torch.randn(N, H, device="cuda")
    W, b = torch.randn(V, H, device="cuda") / 32, torch.randn(V, device="cuda") * 0.1
    tok, mg = rnnt_b200.joint_argmax(a, p, W, b, return_margin=True)
    ref = torch.tanh(a.double() + p.double()) @ W.double().T + b.double()
    bad = tok.long() != ref.argmax(-1)
    # a flip is only tolerable at a numerical tie; report the margin if it ever happens
    assert not bad.any(), mg[bad]


def test_full_size_properties():
    """BASELINE configs[1] size (B=32,T=400,U=100,H=V=1024): size-independent checks, no dense reference."""
    inp = make_inputs(32, 400, 100, 1024, 1024, ragged=False, seed=99)
    out = fused_raw(inp)
    costs = out["costs"]
    assert torch.isfinite(costs).all() and (costs > 0).all()
    # -beta[0,0] == -(alpha[T-1,U] + lpB[T-1,U])  (both directions of the lattice agree)
    tail = -(out["alpha"][:, -1, -1] + out["lp"][:, -1, -1, 0])
    assert (tail - costs).abs().max() <= 2e-5 * costs.abs().max()
    # sum_v dlogits = 0 for every cell  =>  sum(db) == 0 up to bf16 rounding of ~1.3M gradient rows
    assert abs(float(out["db"].sum())) < 1e-2 * float(out["db"].abs().sum())
    # a second run is bit-identical in the forward and close in the (atomic-order dependent) backward
    again = fused_raw(inp)
    assert torch.equal(again["costs"], costs)
    assert rel_err(again["dW"], out["dW"])[0] < 1e-5
    # utterance 0 alone gives the same cost and the same d_enc row block
    sub = {k: (v[:1].contiguous() if k in ("enc", "pred", "targets", "T_len", "U_len") else v) for k, v in inp.items()}
    solo = fused_raw(sub)
    assert torch.equal(solo["costs"][0], costs[0])
    assert rel_err(solo["d_enc"][0], out["d_enc"][0])[0] < 1e-5


def test_stress_shape_properties_and_sampled_parity():
    """BASELINE configs[3]: B=8, T=1500, U=300, V=4096 (ragged).  The reference would need ~110 GiB for logits and their
    gradients at this size, so the whole batch is checked through size-independent properties and ONE (short) utterance
    against the torch + torchaudio path."""
    B, T, U, H, V = 8, 1500, 300, 1024, 4096
    inp = make_inputs(B, T, U, H, V, ragged=True, seed=5)
    inp["T_len"][3] = 300; inp["U_len"][3] = 60            # the utterance the dense reference can afford
    out = fused_raw(inp)
    assert out["status"] == 0
    costs = out["costs"]
    assert torch.isfinite(costs).all() and (costs > 0).all()
    for b in range(B):
        Tb, Ub = int(inp["T_len"][b]), int(inp["U_len"][b])
        tail = -(out["alpha"][b, Tb - 1, Ub] + out["lp"][b, Tb - 1, Ub, 0])
        assert abs(float(tail - costs[b])) <= 2e-5 * abs(float(costs[b]))
        assert not out["d_enc"][b, Tb:].any() and not out["d_pred"][b, Ub + 1:].any()
    assert abs(float(out["db"].sum())) < 1e-2 * float(out["db"].abs().sum())
    assert 0 < out["active_halves"] < out["total_halves"]
    # memory-lean mode gives the same numbers at this size too
    lean = fused_raw(inp, save_hidden=False)
    assert torch.equal(lean["costs"], costs)
    # (different ring chunking -> different fp32 summation order over ~2M cells)
    assert rel_err(lean["dW"], out["dW"])[0] < 1e-3
    del lean
    # one utterance against the reference path (dense logits: 300 x 61 x 4096 fp32 = 0.3 GB)
    b, Tb, Ub = 3, 300, 60
    sub = dict(enc=inp["enc"][b:b + 1, :Tb].contiguous(), pred=inp["pred"][b:b + 1, :Ub + 1].contiguous(), W=inp["W"],
               b=inp["b"], targets=inp["targets"][b:b + 1, :Ub].contiguous(),
               T_len=inp["T_len"][b:b + 1], U_len=inp["U_len"][b:b + 1])
    ref = torch_reference(sub)
    assert abs(float(ref["costs"][0] - costs[b])) <= LOSS_RTOL * abs(float(ref["costs"][0]))
    assert rel_err(out["d_enc"][b, :Tb], ref["d_enc"][0])[0] <= GRAD_TOL_FP32
    assert rel_err(out["d_pred"][b, :Ub + 1], ref["d_pred"][0])[0] <= GRAD_TOL_FP32


def test_decode_config_full_size_engines_agree():
    """BASELINE configs[4]: batched greedy decode at B=64, T=400 (max_length 200, ConvPredictor at default init).  The
    persistent kernel, the captured-graph torch-op loop and the reference's per-utterance algorithm (host loop on the
    same features) must emit identical token sequences."""
    import rnnt_b200
    torch.manual_seed(0)
    H = V = 1024
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += 1.0          # make blank competitive so utterances both emit and advance
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, 512, 0.3), torch.nn.Identity(), joint).cuda().eval()
    feats = torch.randn(64, 400, H, device="cuda")
    lens = torch.randint(200, 401, (64,)); lens[0] = 400
    got, margins = model.greedy_decode_features(feats, lens, max_length=200, return_margins=True)
    assert len(got) == 64 and all(len(x) <= 199 for x in got) and sum(len(x) for x in got) > 64
    assert model.greedy_decode_features(feats, lens, max_length=200, engine="graph") == got
    # the reference's loop (rnnt/model.py:90-128) for a few utterances, one at a time
    for b in (0, 17, 63):
        one = model._greedy_decode_features_hostloop(feats[b:b + 1, : int(lens[b])], lens[b:b + 1], max_length=200)
        assert one[0] == got[b], (b, min(margins[b]))


def test_data_parallel_shards_reproduce_the_global_batch():
    """Sharding by utterance (SURVEY 8e): per-shard mean losses with equal shard sizes average to the global mean
    loss, and the averaged weight gradients equal the global ones -- what DDP / GradAllReducer compute."""
    import rnnt_b200
    inp = make_inputs(8, 30, 9, 64, 256, ragged=True, seed=41)
    def run(sl):
        W = inp["W"].clone().requires_grad_(True); b = inp["b"].clone().requires_grad_(True)
        enc = inp["enc"][sl].contiguous().requires_grad_(True)
        # every shard keeps the global padded shape, so lengths need not hit the maxima
        loss = rnnt_b200.joint_rnnt_loss(enc, inp["pred"][sl].contiguous(), W, b, inp["targets"][sl].contiguous(),
                                         inp["T_len"][sl].contiguous(), inp["U_len"][sl].contiguous(),
                                         reduction="mean", validate=False)
        loss.backward()
        return loss.detach(), W.grad, b.grad, enc.grad
    full = run(slice(0, 8))
    shards = [run(slice(0, 4)), run(slice(4, 8))]
    assert abs(float(full[0]) - float((shards[0][0] + shards[1][0]) / 2)) < 1e-5 * abs(float(full[0]))
    assert rel_err((shards[0][1] + shards[1][1]) / 2, full[1])[0] < 1e-5
    assert rel_err((shards[0][2] + shards[1][2]) / 2, full[2])[0] < 1e-5
    assert rel_err(torch.cat([shards[0][3], shards[1][3]]) / 2, full[3])[0] < 1e-5


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import rnnt_b200
from rnnt_b200.parallel import GradAllReducer, WeightGradBucket, shard_bounds
from helpers import make_inputs
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
inp = make_inputs(8, 30, 9, 64, 256, ragged=True, seed=41, device=f"cuda:{rank}")
lo, hi = shard_bounds(8, world, rank)
W = inp["W"].clone().requires_grad_(True); b = inp["b"].clone().requires_grad_(True)
loss = rnnt_b200.joint_rnnt_loss(inp["enc"][lo:hi].contiguous(), inp["pred"][lo:hi].contiguous(), W, b,
                                 inp["targets"][lo:hi].contiguous(), inp["T_len"][lo:hi].contiguous(),
                                 inp["U_len"][lo:hi].contiguous(), reduction="mean", validate=False)
loss.backward()
GradAllReducer([], average=True).all_reduce_grads([W.grad, b.grad])
W2 = inp["W"].clone().requires_grad_(True); b2 = inp["b"].clone().requires_grad_(True)
full = rnnt_b200.joint_rnnt_loss(inp["enc"], inp["pred"], W2, b2, inp["targets"], inp["T_len"], inp["U_len"],
                                 reduction="mean", validate=False)
full.backward()
err = float((W.grad - W2.grad).norm() / W2.grad.norm())
assert err < 1e-5, err
# overlapped variant: dW / db written straight into the flat bucket, all-reduce gated by the dW-done event
bucket = WeightGradBucket(256, 64, 100, torch.device("cuda", rank), average=True)
rnnt_b200.functional.set_weight_grad_sink(bucket)
W3 = inp["W"].clone().requires_grad_(True); b3 = inp["b"].clone().requires_grad_(True)
loss = rnnt_b200.joint_rnnt_loss(inp["enc"][lo:hi].contiguous(), inp["pred"][lo:hi].contiguous(), W3, b3,
                                 inp["targets"][lo:hi].contiguous(), inp["T_len"][lo:hi].contiguous(),
                                 inp["U_len"][lo:hi].contiguous(), reduction="mean", validate=False)
bucket.extra_slice.fill_(float(rank + 1))
loss.backward()
bucket.finish()
rnnt_b200.functional.set_weight_grad_sink(None)
torch.cuda.synchronize()
assert W3.grad.data_ptr() == bucket.flat.data_ptr(), "dW must live in the bucket (no flatten copy)"
err2 = float((W3.grad - W2.grad).norm() / W2.grad.norm())
err3 = float((b3.grad - b2.grad).norm() / b2.grad.norm())
assert err2 < 1e-5 and err3 < 1e-5, (err2, err3)
assert abs(float(bucket.extra_slice[0]) - (world + 1) / 2) < 1e-6
dist.destroy_process_group()
print("ok", rank, err, err2)
"""


def test_two_gpu_gradient_allreduce_nccl(tmp_path):
    """N>1 on real GPUs (skipped on a single-GPU box; the gloo world_size-2 test covers the host logic on CPU)."""
    import subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(_NCCL_WORKER)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29633", str(script), root]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ok") == 2


# ------------------------------------------------------------------------------------------------ round 2 additions
def _bf16_torch_baseline(inp):
    """The same path as torch would run it in bf16 (activations and weights rounded to bf16, bf16 matmul with fp32
    accumulation, bf16 logits) -- only used to put this repo's gradient error into scale (SURVEY 8c)."""
    import torchaudio
    enc = inp["enc"].detach().clone().requires_grad_(True)
    pred = inp["pred"].detach().clone().requires_grad_(True)
    W = inp["W"].detach().clone().requires_grad_(True)
    b = inp["b"].detach().clone().requires_grad_(True)
    h = torch.tanh(enc.unsqueeze(2) + pred.unsqueeze(1)).to(torch.bfloat16)
    logits = torch.nn.functional.linear(h, W.to(torch.bfloat16), b.to(torch.bfloat16)).float()
    costs = torchaudio.functional.rnnt_loss(logits, inp["targets"], inp["T_len"], inp["U_len"], blank=-1, clamp=-1,
                                            reduction="none")
    costs.sum().backward()
    return dict(costs=costs.detach(), d_enc=enc.grad, d_pred=pred.grad, dW=W.grad, db=b.grad)


def test_full_size_vs_reference(capsys):
    """BASELINE configs[1] at FULL size (B=32,T=400,U=100,H=V=1024): the public API, fed the permuted (B,H,T) encoder
    view that rnnt/model.py:28 produces, against the reference's own call path (torch fp32 linear+tanh + torchaudio
    rnnt_loss, ~20 GiB) on the same GPU.  Also reports the error a bf16 torch run of the same path makes."""
    import rnnt_b200
    B, T, U, H, V = 32, 400, 100, 1024, 1024
    inp = make_inputs(B, T, U, H, V, ragged=False, seed=2026)
    ref = torch_reference(inp)
    ref = {k: v for k, v in ref.items() if k != "logits"}
    torch.cuda.empty_cache()
    enc_bht = inp["enc"].permute(0, 2, 1).contiguous()
    view = enc_bht.permute(0, 2, 1).requires_grad_(True)            # (B,T,H) view, T-contiguous
    pred = inp["pred"].clone().requires_grad_(True)
    W = inp["W"].clone().requires_grad_(True)
    b = inp["b"].clone().requires_grad_(True)
    costs = rnnt_b200.joint_rnnt_loss(view, pred, W, b, inp["targets"], inp["T_len"], inp["U_len"], reduction="none")
    costs.sum().backward()
    ours = dict(costs=costs.detach(), d_enc=view.grad, d_pred=pred.grad, dW=W.grad, db=b.grad)
    cost_rel = float(((ours["costs"] - ref["costs"]).abs() / ref["costs"].abs()).max())
    assert cost_rel <= LOSS_RTOL, cost_rel
    errs = {k: rel_err(ours[k], ref[k])[0] for k in ("d_enc", "d_pred", "dW", "db")}
    for k, e in errs.items():
        assert e <= GRAD_TOL_FP32, (k, e)
    del costs, view, pred, W, b
    torch.cuda.empty_cache()
    small = {k: (v[:8].contiguous() if k in ("enc", "pred", "targets", "T_len", "U_len") else v) for k, v in inp.items()}
    ref8, bf8 = torch_reference(small), _bf16_torch_baseline(small)
    bf_errs = {k: rel_err(bf8[k], ref8[k])[0] for k in ("d_enc", "d_pred", "dW", "db")}
    bf_cost = float(((bf8["costs"] - ref8["costs"]).abs() / ref8["costs"].abs()).max())
    with capsys.disabled():
        print(f"\n[full-size parity] cost rel err: ours {cost_rel:.2e} (bar 1e-4), bf16 torch {bf_cost:.2e}")
        for k in errs:
            print(f"[full-size parity] {k}: rel-Frobenius ours {errs[k]:.2e}  bf16 torch (B=8 slice) {bf_errs[k]:.2e}")
    for k in errs:
        assert errs[k] < bf_errs[k], (k, errs[k], bf_errs[k])      # fp16 operands beat the bf16 torch baseline


def test_trained_scale_inputs_stay_in_fp16_range():
    """Large-magnitude activations (|enc|, |pred| ~ 4 sigma = 16) and weights up to |W| ~ 1 (32x the init range), i.e. a
    sharp, trained-looking softmax: fp16 operands (tanh in [-1,1], W, S-scaled gradients) must not overflow or lose
    the loss / gradient parity."""
    B, T, U, H, V = 2, 60, 20, 1024, 1024
    inp = make_inputs(B, T, U, H, V, ragged=True, seed=77, scale=4.0)
    inp["W"] = inp["W"] * 32.0
    inp["b"] = inp["b"] * 32.0
    ref = torch_reference(inp)
    out = fused_raw(inp)
    assert torch.isfinite(out["costs"]).all()
    assert ((out["costs"] - ref["costs"]).abs() <= LOSS_RTOL * ref["costs"].abs()).all(), (out["costs"], ref["costs"])
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert torch.isfinite(out[k]).all()
        assert rel_err(out[k], ref[k])[0] <= GRAD_TOL_FP32, (k, rel_err(out[k], ref[k]))


def test_strided_encoder_view_is_read_in_place():
    """f-2: the (B,T,H) view of the encoder's (B,H,T) output (rnnt/model.py:27-28) is consumed without a transposed copy
    (the tensor saved for the backward IS the view), gives bit-identical costs, and its gradient comes back in the
    encoder's own layout."""
    import rnnt_b200
    for (B, T, U, H, V) in [(2, 16, 5, 64, 256), (3, 37, 9, 72, 300), (2, 50, 12, 128, 256), (1, 33, 4, 64, 64)]:
        inp = make_inputs(B, T, U, H, V, ragged=True, seed=3)
        enc_bht = inp["enc"].permute(0, 2, 1).contiguous()
        view = enc_bht.permute(0, 2, 1).requires_grad_(True)
        assert not view.is_contiguous() or T == 1
        dense = inp["enc"].clone().requires_grad_(True)
        args = (inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"], inp["U_len"])
        a = rnnt_b200.joint_rnnt_loss(view, *args, reduction="none")
        b = rnnt_b200.joint_rnnt_loss(dense, *args, reduction="none")
        saved = a.grad_fn.saved_tensors[0]
        assert saved.data_ptr() == view.data_ptr() and saved.stride() == view.stride()
        assert torch.equal(a.detach(), b.detach())
        a.sum().backward(); b.sum().backward()
        assert view.grad.shape == view.shape
        assert rel_err(view.grad, dense.grad)[0] < 1e-5, (B, T, U, H, V)
        out_view = fused_raw(dict(inp, enc=view.detach()))
        assert out_view["d_enc"].stride(1) == 1 or T == 1                       # gradient in (B,H,T) memory order
        assert rel_err(out_view["d_enc"], dense.grad)[0] < 1e-5
        for b_ in range(B):
            assert not out_view["d_enc"][b_, int(inp["T_len"][b_]):].any()


def test_deterministic_mode_is_bit_identical():
    """RNNT_B200_DETERMINISTIC: cross-CTA sums in 64-bit fixed point -> gradients identical bit for bit from run to run
    (the default mode uses fp32 atomics, whose order varies), and equal to the default mode up to fp32 rounding."""
    inp = make_inputs(4, 120, 30, 256, 512, ragged=True, seed=21)
    a = fused_raw(inp, flags=2)
    b = fused_raw(inp, flags=2)
    d = fused_raw(inp, flags=0)
    for k in ("d_enc", "d_pred", "dW", "db"):
        assert torch.equal(a[k], b[k]), k
        assert rel_err(a[k], d[k])[0] < 1e-5, (k, rel_err(a[k], d[k]))
    view = inp["enc"].permute(0, 2, 1).contiguous().permute(0, 2, 1)
    c = fused_raw(dict(inp, enc=view), flags=2)
    assert torch.equal(c["d_enc"], a["d_enc"]) and torch.equal(c["dW"], a["dW"])
    import rnnt_b200
    enc = inp["enc"].clone().requires_grad_(True)
    g = []
    for _ in range(2):
        enc.grad = None
        rnnt_b200.joint_rnnt_loss(enc, inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"], inp["U_len"],
                                  deterministic=True).backward()
        g.append(enc.grad.clone())
    assert torch.equal(g[0], g[1])


def test_out_of_range_lengths_poison_the_costs():
    """validate=False skips the host-side checks (no sync); lengths torchaudio would raise for must not pass silently:
    the kernels clamp them (no out-of-bounds access) and every cost of the batch becomes NaN."""
    import rnnt_b200
    inp = make_inputs(3, 12, 5, 64, 256, seed=9)
    args = (inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"])
    ok = rnnt_b200.joint_rnnt_loss(*args, inp["T_len"], inp["U_len"], reduction="none", validate=False)
    assert torch.isfinite(ok).all()
    for bad_T, bad_U in ((torch.tensor([12, 13, 12]), None), (torch.tensor([12, 0, 12]), None),
                         (None, torch.tensor([5, 9, 5])), (None, torch.tensor([5, -1, 5]))):
        tl = inp["T_len"] if bad_T is None else bad_T.int().cuda()
        ul = inp["U_len"] if bad_U is None else bad_U.int().cuda()
        out = rnnt_b200.joint_rnnt_loss(*args, tl, ul, reduction="none", validate=False)
        assert torch.isnan(out).all(), (tl, ul, out)
    out = fused_raw(dict(inp, T_len=torch.tensor([12, 40, 12], dtype=torch.int32, device="cuda")))
    assert out["status"] == 1 and torch.isnan(out["costs"]).all()


def test_preprojection_joint_matches_reference_golden(golden_dir):
    """f-4: JointNetwork with audio_ln / text_ln (rnnt/joint.py:8-12,26-30) -- costs and every gradient, including the
    projections' weights and the raw (unprojected) inputs, against vectors produced by the reference module."""
    import rnnt_b200
    g = np.load(os.path.join(golden_dir, "loss_proj.npz"))
    Fa, Ft = g["audio"].shape[2], g["text"].shape[2]
    V, H = g["param.joint_ln.weight"].shape
    joint = rnnt_b200.JointNetwork(Fa, Ft, H, V)
    joint.load_state_dict({k[6:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("param.")})
    joint = joint.cuda()
    audio = torch.from_numpy(g["audio"]).cuda().requires_grad_(True)
    text = torch.from_numpy(g["text"]).cuda().requires_grad_(True)
    t = lambda k: torch.from_numpy(g[k]).to(torch.int32).cuda()
    costs = joint.loss(audio, text, t("targets"), t("T_len"), t("U_len"), reduction="none")
    costs.sum().backward()
    assert np.abs(costs.detach().cpu().numpy() - g["costs"]).max() <= LOSS_RTOL * np.abs(g["costs"]).max()
    assert rel_err(audio.grad.cpu(), torch.from_numpy(g["d_audio"]))[0] <= GRAD_TOL_TINY
    assert rel_err(text.grad.cpu(), torch.from_numpy(g["d_text"]))[0] <= GRAD_TOL_TINY
    for name, p in joint.named_parameters():
        assert rel_err(p.grad.cpu(), torch.from_numpy(g["grad." + name]))[0] <= GRAD_TOL_TINY, name


def test_model_forward_matches_reference_golden(golden_dir):
    """a-7: RNNTModel.forward end to end (the call train.py:133 makes) against the reference's RNNTModel.forward
    (rnnt/model.py:17-43): blank prepend, predictor, encoder + permuted view, calc_output_lens, .int() casts, mean loss,
    and the gradients autograd carries back into joint, predictor and encoder."""
    import rnnt_b200
    from helpers import StubEncoder
    g = np.load(os.path.join(golden_dir, "model_forward.npz"))
    V, H = g["param.joint.joint_ln.weight"].shape
    E = g["param.predictor.embedding.weight"].shape[1]
    n_mels = g["mel"].shape[1]
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.0), StubEncoder(n_mels, H),
                                rnnt_b200.JointNetwork(-1, -1, H, V))
    model.load_state_dict({k[6:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("param.")})
    model = model.cuda().train()
    loss = model(torch.from_numpy(g["mel"]).cuda(), torch.from_numpy(g["mel_lens"]).cuda(),
                 torch.from_numpy(g["input_ids"]).cuda(), torch.from_numpy(g["id_lens"]).cuda(), blank_idx=V - 1)
    assert loss.dim() == 0
    assert abs(float(loss.detach()) - float(g["loss"])) <= LOSS_RTOL * abs(float(g["loss"]))
    loss.backward()
    for name, p in model.named_parameters():
        want = torch.from_numpy(g["grad." + name])
        assert p.grad is not None, name
        r, a = rel_err(p.grad.cpu(), want)
        assert r <= GRAD_TOL_TINY or a < 1e-6, (name, r, a)


def test_greedy_decode_full_size_matches_reference_golden(golden_dir):
    """BASELINE configs[4] width (H=V=1024, E=512, T up to 400, max_length 200): tokens of the persistent decode kernel
    against the reference's own loop (rnnt/model.py:90-128, fp32 CPU), for 12 seeded utterances.  The weights and
    features are re-created from the stored seed (checksums verified).  Decisions whose reference top-2 gap is below
    1e-4 may legitimately depend on fp32 summation order, so exactness is required up to the first such decision of
    an utterance (its position is stored in the fixture) and for whole utterances without one."""
    import rnnt_b200
    from helpers import decode_full_setup
    g = np.load(os.path.join(golden_dir, "decode_full.npz"))
    model, feats, T_len = decode_full_setup(g)
    model = model.cuda().eval()
    got, margins = model.greedy_decode_features(feats.cuda(), T_len, max_length=int(g["max_length"]),
                                                return_margins=True)
    off, exact = 0, 0
    for i, n in enumerate(g["tok_len"]):
        want = g["tok_flat"][off:off + n].tolist()
        off += n
        safe = int(g["safe_len"][i])
        assert got[i][:safe] == want[:safe], (i, safe, min(margins[i]))
        if safe == n:
            assert got[i] == want, (i, min(margins[i]))
            exact += 1
    assert exact >= 8                                   # at least 8 utterances are pinned token for token


def test_decode_single_utterance_odd_vocab():
    """B = 1 with an odd vocabulary (the reference-signature greedy_decode case): scratch regions stay aligned."""
    import rnnt_b200
    torch.manual_seed(3)
    H, V, E = 64, 29, 32
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.weight.mul_(3.0)
        joint.joint_ln.bias[V - 1] += 2.0
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.3), torch.nn.Identity(), joint).cuda().eval()
    feats = torch.randn(1, 30, H, device="cuda")
    lens = torch.tensor([30])
    got = model.greedy_decode_features(feats, lens, max_length=40)
    assert got == model._greedy_decode_features_hostloop(feats, lens, max_length=40)
    assert got == model.greedy_decode_features(feats, lens, max_length=40, engine="graph")
    assert rnnt_b200.functional._last_decode_phase_cycles is not None


def test_decode_wide_batch_odd_sizes():
    """More utterances than one pass of row groups (several prefetched groups per warp), an embedding width that does
    not fill a staging chunk, more symbols than CTAs (tail groups in the conv1 table build), ragged lengths."""
    import rnnt_b200
    torch.manual_seed(11)
    B, T, H, V, E = 150, 24, 96, 301, 72
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.weight.mul_(3.0)
        joint.joint_ln.bias[V - 1] += 1.2
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.3), torch.nn.Identity(), joint).cuda().eval()
    feats = torch.randn(B, T, H, device="cuda")
    lens = torch.randint(1, T + 1, (B,)); lens[0] = T
    got = model.greedy_decode_features(feats, lens, max_length=30)
    assert got == model.greedy_decode_features(feats, lens, max_length=30, engine="graph")
    assert sum(len(x) for x in got) > B          # the workload does emit


def test_greedy_decode_dispatches_on_predictor_shape():
    """RNNTModel.greedy_decode (rnnt/model.py:130-139) accepts any ConvPredictor-SHAPED module (e.g. the reference's own
    class when only joint._target_ is swapped), runs LSTMPredictor-shaped ones through the stateful loop
    (rnnt/model.py:46-87) and raises the reference's ValueError otherwise."""
    import rnnt_b200
    from helpers import TinyStatefulPredictor
    torch.manual_seed(5)
    H, V, E = 64, 32, 32
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.weight.mul_(3.0)
        joint.joint_ln.bias[V - 1] += 1.5

    class Wrapped(torch.nn.Module):                     # not a rnnt_b200.ConvPredictor instance, same attributes
        def __init__(self, inner):
            super().__init__()
            for name in ("embedding", "input_layer_norm", "conv1", "conv2", "linear", "output_layer_norm"):
                setattr(self, name, getattr(inner, name))
            self.inner = inner

        def forward(self, ids):
            return self.inner(ids)

    conv = rnnt_b200.ConvPredictor(V, H, E, 0.3)
    feats = torch.randn(2, 20, H, device="cuda")
    lens = torch.tensor([20, 13])
    a = rnnt_b200.RNNTModel(conv, torch.nn.Identity(), joint).cuda().eval().greedy_decode_features(feats, lens, 30)
    b = rnnt_b200.RNNTModel(Wrapped(conv), torch.nn.Identity(), joint).cuda().eval().greedy_decode_features(feats, lens, 30)
    assert a == b and sum(len(x) for x in a) > 0
    # stateful (LSTM-shaped) predictor: this repo's joint kernel inside the reference's loop vs plain torch
    lstm = TinyStatefulPredictor(V, H, E)
    model = rnnt_b200.RNNTModel(lstm, torch.nn.Identity(), joint).cuda().eval()
    got = model.greedy_decode_features(feats, lens, 30)
    for i in range(2):
        tokens, t, per = [V - 1], 0, 0
        f, _, st = lstm(torch.tensor([tokens], device="cuda"), torch.tensor([1], device="cuda"))
        while t < int(lens[i]) and len(tokens) < 30:
            tok = int(joint.single_forward(feats[i, t:t + 1], f[:, -1, :]).argmax(-1))
            if tok == V - 1 or per >= 10:
                t += 1; per = 0
            else:
                tokens.append(tok)
                f, _, st = lstm(torch.tensor([[tok]], device="cuda"), torch.tensor([len(tokens)], device="cuda"), st)
                per += 1
        assert got[i] == tokens[1:], i
    one = model.greedy_decode(feats[:1].permute(0, 2, 1), torch.tensor([20]), max_length=30)
    assert one == got[0]
    with pytest.raises(ValueError, match="Unknown predictor type"):
        rnnt_b200.RNNTModel(torch.nn.Linear(2, 2), torch.nn.Identity(), joint).cuda().greedy_decode_features(feats, lens)


@pytest.mark.parametrize("shape", [(12800, 1024, 1024), (404, 1024, 1024), (300, 72, 136), (1, 8, 8), (77, 40, 264),
                                   (2600, 256, 128)])
def test_preprojection_gemm_matches_torch(shape):
    """rnnt_b200_linear_fwd/bwd (tcgen05, fp16 operands) vs torch fp32 linear: y, dx, dW, db; ragged tile edges."""
    from rnnt_b200.functional import linear
    M, K, N = shape
    g = torch.Generator().manual_seed(M + K)
    x = torch.randn(M, K, generator=g).cuda().requires_grad_(True)
    W = ((torch.rand(N, K, generator=g) * 2 - 1) / K ** 0.5).cuda().requires_grad_(True)
    b = ((torch.rand(N, generator=g) * 2 - 1) / K ** 0.5).cuda().requires_grad_(True)
    dy = torch.randn(M, N, generator=g).cuda()
    y = linear(x, W, b)
    y.backward(dy)
    got = [y.detach(), x.grad.clone(), W.grad.clone(), b.grad.clone()]
    x.grad = W.grad = b.grad = None
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        y2 = torch.nn.functional.linear(x, W, b)
        y2.backward(dy)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    for name, a, r in zip(("y", "dx", "dW", "db"), got, (y2.detach(), x.grad, W.grad, b.grad)):
        assert rel_err(a, r)[0] < 1e-3, (shape, name, rel_err(a, r))
    # deterministic variant of the split-K weight gradient
    torch.use_deterministic_algorithms(True)
    try:
        outs = []
        for _ in range(2):
            x.grad = W.grad = b.grad = None
            linear(x, W, b).backward(dy)
            outs.append((W.grad.clone(), b.grad.clone()))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        assert rel_err(outs[0][0], got[2])[0] < 1e-5
    finally:
        torch.use_deterministic_algorithms(False)


def test_preprojection_joint_full_width_vs_reference():
    """f-4 at the reference's width: JointNetwork(audio_features=1024, text_features=1024, 1024, 1024) -- the joint of the
    non-"convjs" configs -- loss and every gradient (raw inputs, audio_ln, text_ln, joint_ln) vs the same modules run
    the reference's way (torch fp32 linear + tanh + torchaudio rnnt_loss) on the same device."""
    import torchaudio
    import rnnt_b200
    torch.manual_seed(7)
    B, T, U, F_, H, V = 4, 120, 30, 1024, 1024, 1024
    joint = rnnt_b200.JointNetwork(F_, F_, H, V).cuda()
    audio = torch.randn(B, T, F_, device="cuda")
    text = torch.randn(B, U + 1, F_, device="cuda")
    targets = torch.randint(0, V - 1, (B, U), dtype=torch.int32, device="cuda")
    T_len = torch.tensor([T, T - 7, T // 2, T], dtype=torch.int32, device="cuda")
    U_len = torch.tensor([U, U // 2, U, 3], dtype=torch.int32, device="cuda")

    def run(fused):
        a = audio.clone().requires_grad_(True)
        t = text.clone().requires_grad_(True)
        joint.zero_grad()
        if fused:
            costs = joint.loss(a, t, targets, T_len, U_len, reduction="none")
        else:
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            try:
                costs = torchaudio.functional.rnnt_loss(joint(a, t), targets, T_len, U_len, blank=-1, clamp=-1,
                                                        reduction="none")
            finally:
                torch.backends.cuda.matmul.allow_tf32 = prev
        costs.sum().backward()
        grads = {n: p.grad.clone() for n, p in joint.named_parameters()}
        grads["audio"], grads["text"] = a.grad, t.grad
        return costs.detach(), grads

    c_ref, g_ref = run(False)
    c_our, g_our = run(True)
    assert ((c_our - c_ref).abs() <= LOSS_RTOL * c_ref.abs()).all(), (c_our, c_ref)
    for k in g_ref:
        assert rel_err(g_our[k], g_ref[k])[0] <= GRAD_TOL_FP32, (k, rel_err(g_our[k], g_ref[k]))


def test_train_loop_guard_shapes_fit_in_bounded_memory():
    """f-3: rnnt/train.py:120-130 halves any batch with max(U) * max(mel frames) > max_joint_size (160,000 in the shipped
    configs) because the (B,T,U+1,V) logits, their gradients and the fp32 activations would not fit a 24 GB card.
    A batch 5.6x over that limit (U=300, 3000 mel frames -> T=1500, B=8: the reference would need 14.8 GB logits +
    14.8 GB logit-gradients + 14.8 GB activations) runs fused forward+backward in a few GiB, so the guard (and its two
    `.item()` syncs per step) can be dropped by the owner."""
    import rnnt_b200
    B, T, U, H, V = 8, 1500, 300, 1024, 1024
    assert U * (2 * T) > 160000 * 5
    inp = make_inputs(B, T, U, H, V, ragged=True, seed=8)
    peaks = {}
    for save_hidden in (True, False):
        enc = inp["enc"].clone().requires_grad_(True)
        W = inp["W"].clone().requires_grad_(True)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        loss = rnnt_b200.joint_rnnt_loss(enc, inp["pred"], W, inp["b"], inp["targets"], inp["T_len"], inp["U_len"],
                                         reduction="mean", save_hidden=save_hidden)
        loss.backward()
        torch.cuda.synchronize()
        peaks[save_hidden] = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
        assert torch.isfinite(loss.detach()) and torch.isfinite(enc.grad).all() and torch.isfinite(W.grad).all()
        del loss, enc, W
    reference_need = 3 * B * T * (U + 1) * V * 4 / 2 ** 30      # logits + logit-gradients + fp32 activations (H = V)
    assert reference_need > 40 and peaks[True] < 12 and peaks[False] < 5, (reference_need, peaks)


def test_fuzz_layouts_modes_and_chunking():
    """Random small problems through random combinations of the code paths: encoder layout (dense / (B,H,T) view),
    backward flags (all tiles, deterministic), saved or recomputed activations, single- or multi-chunk gradient ring."""
    rng = np.random.default_rng(7)
    for i in range(14):
        B, T, U = int(rng.integers(1, 5)), int(rng.integers(1, 70)), int(rng.integers(0, 25))
        H, V = int(rng.choice([8, 64, 72, 128, 256])), int(rng.choice([5, 64, 256, 300, 520]))
        inp = make_inputs(B, T, U, H, V, ragged=True, seed=500 + i)
        ref = torch_reference(inp, device="cpu")
        view = bool(rng.integers(0, 2)) and T > 1
        if view:
            inp = dict(inp, enc=inp["enc"].permute(0, 2, 1).contiguous().permute(0, 2, 1))
        flags = int(rng.integers(0, 4))
        save_hidden = bool(rng.integers(0, 2))
        ring = None if rng.integers(0, 2) else int(rng.integers(1, 6))
        out = fused_raw(inp, flags=flags, save_hidden=save_hidden, ring_tiles=ring)
        tag = (B, T, U, H, V, view, flags, save_hidden, ring)
        assert out["status"] == 0, tag
        err = (out["costs"].cpu() - ref["costs"]).abs()
        assert (err <= LOSS_RTOL * ref["costs"].abs() + 3e-4).all(), (tag, out["costs"], ref["costs"])
        tol = GRAD_TOL_TINY if H < 64 else GRAD_TOL_FP32
        for k in ("d_enc", "d_pred", "dW", "db"):
            r, a = rel_err(out[k].cpu(), ref[k])
            assert r <= tol or a < 1e-5, (tag, k, r, a)
