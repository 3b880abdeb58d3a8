"""Generate golden vectors by running the UNMODIFIED reference in the build container.

    python tests/golden/make_golden.py          # needs /root/reference (absent on the GPU box)

Imports rnnt.joint.JointNetwork / rnnt.model.RNNTModel / rnnt.predictor.ConvPredictor from
/root/reference and torchaudio.functional.rnnt_loss (the call at rnnt/model.py:35-41), runs them in
fp32 on CPU with fixed seeds, and writes small .npz fixtures next to this script.  The fixtures are
committed; tests never read /root/reference.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, "/root/reference")
import torchaudio  # noqa: E402
from rnnt.joint import JointNetwork  # noqa: E402
from rnnt.model import RNNTModel  # noqa: E402
from rnnt.predictor import ConvPredictor  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def loss_case(name, B, T, U, H, V, T_len, U_len, seed, dW_rows=None):
    """dW_rows=n keeps the file of a wide case under 1 MB: the float inputs are replaced by the seed and their checksums
    (tests/helpers.py::load_loss_golden re-creates them), only a seeded choice of n rows of dW and no dense logits are
    stored."""
    torch.manual_seed(seed)
    joint = JointNetwork(-1, -1, H, V)
    enc = torch.randn(B, H, T).permute(0, 2, 1).contiguous().requires_grad_(True)   # model.py:28 layout, made dense
    pred = torch.randn(B, U + 1, H, requires_grad=True)
    targets = torch.randint(0, V - 1, (B, U), dtype=torch.int32)
    T_len = torch.tensor(T_len, dtype=torch.int32)
    U_len = torch.tensor(U_len, dtype=torch.int32)
    logits = joint(enc, pred)                                                     # joint.py:25-39
    logits.retain_grad()
    costs = torchaudio.functional.rnnt_loss(logits=logits, targets=targets, logit_lengths=T_len,
                                            target_lengths=U_len, blank=-1, clamp=-1, reduction="none")
    costs.sum().backward()
    mean = torchaudio.functional.rnnt_loss(logits=logits.detach(), targets=targets, logit_lengths=T_len,
                                           target_lengths=U_len, blank=-1, clamp=-1, reduction="mean")
    out = dict(
        enc=enc.detach().numpy(), pred=pred.detach().numpy(),
        W=joint.joint_ln.weight.detach().numpy(), b=joint.joint_ln.bias.detach().numpy(),
        targets=targets.numpy(), T_len=T_len.numpy(), U_len=U_len.numpy(),
        costs=costs.detach().numpy(), loss_mean=mean.numpy(),
        d_enc=enc.grad.numpy(), d_pred=pred.grad.numpy(),
        dW=joint.joint_ln.weight.grad.numpy(), db=joint.joint_ln.bias.grad.numpy(),
        logits=logits.detach().numpy().astype(np.float32) if logits.numel() < 200000 else np.zeros(0, np.float32),
        dlogits=logits.grad.numpy() if logits.numel() < 200000 else np.zeros(0, np.float32),
    )
    if dW_rows is not None:
        for k in ("enc", "pred", "W", "b"):
            out["chk." + k] = np.abs(out.pop(k).astype(np.float64)).sum()
        rows = np.sort(np.random.default_rng(seed).choice(V, dW_rows, replace=False)).astype(np.int32)
        out.update(seed=np.int64(seed), B=np.int32(B), T=np.int32(T), U=np.int32(U), H=np.int32(H), V=np.int32(V),
                   dW=out["dW"][rows], dW_rows=rows)
        del out["logits"], out["dlogits"]
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "costs", costs.detach().numpy())


class FixedEncoder(torch.nn.Module):
    """Stands in for AudioEncoder: returns the given (N,C,L) features (model.py:93-95 consumes them)."""
    def __init__(self, feats):
        super().__init__()
        self.feats = feats
        self.p = torch.nn.Parameter(torch.zeros(1))

    def forward(self, mel):
        return self.feats

    def calc_output_lens(self, lens):
        return lens


def decode_case(name, n_utt, T, H, V, E, seed, max_length, scale, blank_bias):
    torch.manual_seed(seed)
    joint = JointNetwork(-1, -1, H, V)
    predictor = ConvPredictor(V, H, E, 0.3).eval()
    # make non-blank emissions likely enough that the loop exercises emits and the 10-per-frame cap
    with torch.no_grad():
        joint.joint_ln.weight.mul_(scale)
        joint.joint_ln.bias[V - 1] += blank_bias
    feats = torch.randn(n_utt, T, H)
    T_len = torch.randint(T // 2, T + 1, (n_utt,))
    T_len[0] = T
    tokens = []
    for i in range(n_utt):
        f = feats[i, : int(T_len[i])].t().unsqueeze(0).contiguous()                # (1,C,L)
        model = RNNTModel(predictor, FixedEncoder(f), joint).eval()
        toks = model.greedy_decode(torch.zeros(1, 1, 1), torch.tensor([int(T_len[i])]), max_length=max_length)
        tokens.append(np.asarray(toks, np.int32))
        print(name, i, int(T_len[i]), len(toks), toks[:12])
    sd = {("pred." + k): v.numpy() for k, v in predictor.state_dict().items()}
    flat = np.concatenate(tokens) if tokens else np.zeros(0, np.int32)
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"), feats=feats.numpy(), T_len=T_len.numpy().astype(np.int32),
        W=joint.joint_ln.weight.detach().numpy(), b=joint.joint_ln.bias.detach().numpy(),
        tok_flat=flat, tok_len=np.asarray([len(t) for t in tokens], np.int32),
        max_length=np.int32(max_length), **sd)


def proj_case(name, B, T, U, Fa, Ft, H, V, T_len, U_len, seed):
    """Non-"convjs" joint (rnnt/joint.py:8-12,26-30): audio_ln / text_ln pre-projections in front of the joint."""
    torch.manual_seed(seed)
    joint = JointNetwork(Fa, Ft, H, V)
    audio = torch.randn(B, T, Fa, requires_grad=True)
    text = torch.randn(B, U + 1, Ft, requires_grad=True)
    targets = torch.randint(0, V - 1, (B, U), dtype=torch.int32)
    T_len = torch.tensor(T_len, dtype=torch.int32)
    U_len = torch.tensor(U_len, dtype=torch.int32)
    logits = joint(audio, text)
    costs = torchaudio.functional.rnnt_loss(logits=logits, targets=targets, logit_lengths=T_len,
                                            target_lengths=U_len, blank=-1, clamp=-1, reduction="none")
    costs.sum().backward()
    out = dict(audio=audio.detach().numpy(), text=text.detach().numpy(), targets=targets.numpy(), T_len=T_len.numpy(),
               U_len=U_len.numpy(), costs=costs.detach().numpy(), d_audio=audio.grad.numpy(), d_text=text.grad.numpy())
    for k, v in joint.state_dict().items():
        out["param." + k] = v.numpy()
    for k, v in joint.named_parameters():
        out["grad." + k] = v.grad.numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "costs", costs.detach().numpy())


def model_forward_case(name, B, n_mels, L, U, H, V, E, mel_lens, id_lens, seed):
    """The drop-in call train.py:133 makes: RNNTModel.forward (rnnt/model.py:17-43) -- blank prepend, predictor,
    encoder + permute, calc_output_lens, joint, rnnt_loss(reduction="mean") -- with a small stand-in encoder."""
    sys.path.insert(0, os.path.join(os.path.dirname(HERE)))
    from helpers import StubEncoder
    torch.manual_seed(seed)
    model = RNNTModel(ConvPredictor(V, H, E, 0.0), StubEncoder(n_mels, H), JointNetwork(-1, -1, H, V))
    mel = torch.randn(B, n_mels, L)
    mel_lens = torch.tensor(mel_lens, dtype=torch.int64)
    id_lens = torch.tensor(id_lens, dtype=torch.int64)
    input_ids = torch.randint(0, V - 1, (B, U), dtype=torch.int64)
    for b in range(B):
        input_ids[b, int(id_lens[b]):] = 0                     # zero padding as dataset.py:76-80 produces it
    loss = model(mel, mel_lens, input_ids, id_lens, blank_idx=V - 1)
    loss.backward()
    out = dict(mel=mel.numpy(), mel_lens=mel_lens.numpy(), input_ids=input_ids.numpy(), id_lens=id_lens.numpy(),
               loss=loss.detach().numpy())
    for k, v in model.state_dict().items():
        out["param." + k] = v.numpy()
    for k, v in model.named_parameters():
        out["grad." + k] = v.grad.numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "loss", float(loss))


def decode_full_case(name, n_utt, T, H, V, E, seed, max_length, blank_bias, margin_floor=1e-4):
    """BASELINE configs[4] width (H = V = 1024, E = 512): tokens of the reference's own loop (rnnt/model.py:90-128).
    Stored: seed, lengths, tokens, checksums of the seeded weights / features (the test re-creates them from the seed with
    this repo's module mirrors, same construction order), and for every utterance the number of tokens emitted before
    the first decision whose top-2 logit gap is below `margin_floor` (fp32 summation order may legitimately flip a
    decision inside that gap; everything before it must match exactly)."""
    torch.manual_seed(seed)
    joint = JointNetwork(-1, -1, H, V)
    predictor = ConvPredictor(V, H, E, 0.3).eval()
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += blank_bias
    g = torch.Generator().manual_seed(seed + 1)
    feats = torch.randn(n_utt, T, H, generator=g)
    T_len = torch.randint(T * 3 // 4, T + 1, (n_utt,), generator=g)
    T_len[0] = T
    log = []                       # (top-2 gap, argmax) of every joint evaluation of the current utterance
    orig = joint.single_forward

    def recording_single_forward(a, t):
        out = orig(a, t)
        top = out.topk(2, dim=-1).values
        log.append((float(top[0, 0] - top[0, 1]), int(out.argmax(-1))))
        return out

    joint.single_forward = recording_single_forward
    toks_all, safe, min_margin = [], [], []
    for i in range(n_utt):
        f = feats[i, : int(T_len[i])].t().unsqueeze(0).contiguous()
        model = RNNTModel(predictor, FixedEncoder(f), joint).eval()
        log.clear()
        toks = model.greedy_decode(torch.zeros(1, 1, 1), torch.tensor([int(T_len[i])]), max_length=max_length)
        # replay the control flow of rnnt/model.py:113-125 over the log: tokens out before the first near-tie
        n_out, per, first_unsafe = 0, 0, None
        for m, tok in log:
            if m < margin_floor and first_unsafe is None:
                first_unsafe = n_out
            if tok == joint.blank_idx or per >= 10:
                per = 0
            else:
                n_out += 1
                per += 1
        assert n_out == len(toks)
        toks_all.append(np.asarray(toks, np.int32))
        safe.append(len(toks) if first_unsafe is None else first_unsafe)
        min_margin.append(min(m for m, _ in log) if log else np.inf)
        print(name, i, int(T_len[i]), len(toks), "min margin %.3g" % min_margin[-1], "safe prefix", safe[-1])
    joint.single_forward = orig
    cs = lambda v: np.abs(v.detach().numpy().astype(np.float64)).sum()      # numpy pairwise sum: thread-independent
    chk = {("chk." + k): cs(v) for k, v in predictor.state_dict().items()}
    chk["chk.joint_w"] = cs(joint.joint_ln.weight)
    chk["chk.feats"] = cs(feats)
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"), seed=np.int64(seed), n_utt=np.int32(n_utt), T=np.int32(T), H=np.int32(H),
        V=np.int32(V), E=np.int32(E), blank_bias=np.float32(blank_bias), max_length=np.int32(max_length),
        margin_floor=np.float32(margin_floor), T_len=T_len.numpy().astype(np.int32),
        tok_flat=np.concatenate(toks_all), tok_len=np.asarray([len(t) for t in toks_all], np.int32),
        safe_len=np.asarray(safe, np.int32), min_margin=np.asarray(min_margin, np.float32), **chk)


if __name__ == "__main__":
    torch.set_num_threads(4)
    if len(sys.argv) > 1 and sys.argv[1] == "decode_full":     # regenerate only the slow one
        decode_full_case("decode_full", n_utt=12, T=400, H=1024, V=1024, E=512, seed=33, max_length=200, blank_bias=1.8)
        sys.exit(0)
    # tiny ragged case with U_b = 0 and T_b = 1 rows (dense logits + logit grads kept)
    loss_case("loss_tiny", B=4, T=7, U=4, H=16, V=11, T_len=[7, 5, 1, 3], U_len=[4, 0, 2, 4], seed=11)
    # mid case: kernel-tile friendly sizes, ragged
    loss_case("loss_mid", B=3, T=37, U=13, H=128, V=256, T_len=[37, 20, 31], U_len=[13, 9, 4], seed=12)
    # wide case (H=V=512; the full H=V=1024 width is checked against the live oracle), short lattice
    loss_case("loss_wide", B=2, T=19, U=9, H=512, V=512, T_len=[19, 11], U_len=[7, 9], seed=13, dW_rows=384)
    decode_case("decode_small", n_utt=6, T=24, H=64, V=48, E=32, seed=21, max_length=40, scale=3.0, blank_bias=2.2)
    # round 2: pre-projection joint, the RNNTModel.forward glue, and decode at the full BASELINE configs[4] width
    proj_case("loss_proj", B=3, T=21, U=6, Fa=48, Ft=40, H=64, V=32, T_len=[21, 13, 17], U_len=[6, 2, 5], seed=31)
    model_forward_case("model_forward", B=3, n_mels=20, L=50, U=7, H=64, V=32, E=24, mel_lens=[50, 37, 44],
                       id_lens=[7, 3, 5], seed=32)
    decode_full_case("decode_full", n_utt=12, T=400, H=1024, V=1024, E=512, seed=33, max_length=200, blank_bias=1.8)
