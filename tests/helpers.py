"""Shared helpers for the GPU parity tests: input generation, direct C-ABI calls, ring <-> lattice mapping."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch


class StubEncoder(torch.nn.Module):
    """Small stand-in for rnnt.jasper.AudioEncoder with the two members RNNTModel.forward uses (rnnt/model.py:27-29):
    forward(mel (N,F,L)) -> (N,C,L') and calc_output_lens.  One strided Conv1d + tanh; L' = ceil(L / 2)."""

    def __init__(self, n_mels: int, hidden: int):
        super().__init__()
        self.conv = torch.nn.Conv1d(n_mels, hidden, kernel_size=3, stride=2, padding=1)

    def forward(self, mel):
        return torch.tanh(self.conv(mel))

    def calc_output_lens(self, lens):
        return (lens + 1) // 2


class TinyStatefulPredictor(torch.nn.Module):
    """LSTMPredictor-shaped stand-in (rnnt/predictor.py:84-186): `p(ids, lengths, state) -> (out, lengths, state)` with
    a `lstm_layers` list; one LSTMCell layer between an embedding and a linear + LayerNorm."""

    def __init__(self, num_symbols: int, output_dim: int, dim: int):
        super().__init__()
        self.embedding = torch.nn.Embedding(num_symbols, dim)
        self.lstm_layers = torch.nn.ModuleList([torch.nn.LSTMCell(dim, dim)])
        self.linear = torch.nn.Linear(dim, output_dim)
        self.output_layer_norm = torch.nn.LayerNorm(output_dim)

    def forward(self, ids, lengths, state=None):
        x = self.embedding(ids)                                   # (B,U,D)
        h, c = state[0] if state is not None else (x.new_zeros(x.shape[0], x.shape[2]),) * 2
        outs = []
        for u in range(x.shape[1]):
            h, c = self.lstm_layers[0](x[:, u], (h, c))
            outs.append(h)
        out = self.output_layer_norm(self.linear(torch.stack(outs, 1)))
        return out, lengths, [[h, c]]


def decode_full_setup(g):
    """Re-create the seeded model / features of tests/golden/decode_full.npz (make_golden.py::decode_full_case) with
    this repo's module mirrors and verify them against the stored checksums.  Returns (RNNTModel, feats, T_len)."""
    import rnnt_b200
    seed, n_utt, T = int(g["seed"]), int(g["n_utt"]), int(g["T"])
    H, V, E = int(g["H"]), int(g["V"]), int(g["E"])
    torch.manual_seed(seed)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    predictor = rnnt_b200.ConvPredictor(V, H, E, 0.3).eval()
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += float(g["blank_bias"])
    gen = torch.Generator().manual_seed(seed + 1)
    feats = torch.randn(n_utt, T, H, generator=gen)
    T_len = torch.randint(T * 3 // 4, T + 1, (n_utt,), generator=gen)
    T_len[0] = T
    assert T_len.tolist() == g["T_len"].tolist()
    cs = lambda v: float(np.abs(v.detach().numpy().astype(np.float64)).sum())
    for k, v in predictor.state_dict().items():
        assert cs(v) == float(g["chk." + k]), k
    assert cs(joint.joint_ln.weight) == float(g["chk.joint_w"])
    assert cs(feats) == float(g["chk.feats"])
    return rnnt_b200.RNNTModel(predictor, torch.nn.Identity(), joint), feats, T_len


def load_loss_golden(golden_dir, name):
    """Arrays of tests/golden/<name>.npz (make_golden.py::loss_case) as a dict.  A case stored without its float inputs
    is re-created from its seed in loss_case's drawing order and verified against the stored checksums.  Such a case
    may keep only the rows `dW_rows` of dW; for the others `dW_rows` is every row."""
    g = dict(np.load(os.path.join(golden_dir, name + ".npz")))
    if "enc" not in g:
        import rnnt_b200
        B, T, U, H, V = (int(g[k]) for k in ("B", "T", "U", "H", "V"))
        torch.manual_seed(int(g["seed"]))
        joint = rnnt_b200.JointNetwork(-1, -1, H, V)
        g["enc"] = torch.randn(B, H, T).permute(0, 2, 1).contiguous().numpy()
        g["pred"] = torch.randn(B, U + 1, H).numpy()
        g["W"], g["b"] = joint.joint_ln.weight.detach().numpy(), joint.joint_ln.bias.detach().numpy()
        for k in ("enc", "pred", "W", "b"):
            assert float(np.abs(g[k].astype(np.float64)).sum()) == float(g["chk." + k]), k
    g.setdefault("dW_rows", np.arange(g["W"].shape[0]))
    return g


def make_inputs(B, T, U, H, V, seed=1234, ragged=False, device="cuda", scale=1.0):
    g = torch.Generator().manual_seed(seed)
    enc = torch.randn(B, H, T, generator=g).permute(0, 2, 1).contiguous() * scale   # dense copy of the model.py:28 view
    pred = torch.randn(B, U + 1, H, generator=g) * scale
    bound = 1.0 / (H ** 0.5)
    W = (torch.rand(V, H, generator=g) * 2 - 1) * bound       # nn.Linear default init range (joint.py:18)
    b = (torch.rand(V, generator=g) * 2 - 1) * bound
    targets = torch.randint(0, V - 1, (B, U), generator=g, dtype=torch.int32)
    if ragged:
        T_len = torch.randint(max(1, T // 2), T + 1, (B,), generator=g, dtype=torch.int32)
        U_len = torch.randint(U // 2, U + 1, (B,), generator=g, dtype=torch.int32)
        T_len[0] = T
        U_len[B - 1] = U
    else:
        T_len = torch.full((B,), T, dtype=torch.int32)
        U_len = torch.full((B,), U, dtype=torch.int32)
    to = lambda x: x.to(device)
    return dict(enc=to(enc), pred=to(pred), W=to(W), b=to(b), targets=to(targets), T_len=to(T_len), U_len=to(U_len))


def fused_raw(inp, ring_tiles=None, dcost=None, clamp=-1.0, flags=0, save_hidden=True, blank=-1, fill=None):
    """Call the C-ABI forward + backward directly; returns outputs plus the raw workspace and its layout.
    save_hidden=False exercises the memory-lean mode (per-SM scratch in the forward, recomputing backward).
    flags: 1 = RNNT_B200_ALL_TILES, 2 = RNNT_B200_DETERMINISTIC.  inp["enc"] may be H-contiguous or the T-contiguous
    permuted view of a (B,H,T) tensor; d_enc is produced in the same layout.  fill: a byte value the workspace, `hidden`
    and every output are filled with before the calls (default zeros), so a test can vary memory the kernels must
    overwrite."""
    from rnnt_b200 import _lib
    from rnnt_b200.functional import _stream_ptr, pick_ring_tiles
    L = _lib.lib()
    enc, pred, W, b = inp["enc"], inp["pred"], inp["W"], inp["b"]
    targets, T_len, U_len = inp["targets"], inp["T_len"], inp["U_len"]
    B, T, H = enc.shape
    U1 = pred.shape[1]
    V = W.shape[0]
    dev = enc.device
    if ring_tiles is None:
        ring_tiles = pick_ring_tiles(B, T, U1, H, V, have_hidden=save_hidden)
    offs = (C.c_int64 * 8)()
    hp, vp = C.c_int(0), C.c_int(0)
    _lib.check(L.rnnt_b200_debug_ws_layout(B, T, U1, H, V, ring_tiles, int(save_hidden), offs, C.byref(hp),
                                           C.byref(vp)), "layout")
    byte = 0 if fill is None else int(fill)
    raw = lambda n: torch.full((n,), byte, dtype=torch.uint8, device=dev)
    ws = raw(int(offs[6]))
    hidden = raw(L.rnnt_b200_hidden_bytes(B, T, U1, H)) if save_hidden else None
    hptr = hidden.data_ptr() if save_hidden else None
    f = lambda *s: raw(4 * int(np.prod(s))).view(torch.float32).view(*s)
    d_enc = f(B, H, T).permute(0, 2, 1) if (enc.stride(1) == 1 and T > 1) else f(B, T, H)
    out = dict(costs=f(B), lp=f(B, T, U1, 2), lse=f(B, T, U1), alpha=f(B, T, U1), beta=f(B, T, U1),
               d_enc=d_enc, d_pred=f(B, U1, H), dW=f(V, H), db=f(V))
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _stream_ptr(dev)
    _lib.check(L.rnnt_b200_joint_loss_fwd(
        enc.data_ptr(), enc.stride(0), enc.stride(1), enc.stride(2), pred.data_ptr(), W.data_ptr(), b.data_ptr(),
        targets.data_ptr(), T_len.data_ptr(), U_len.data_ptr(), B, T, U1, H, V, blank, out["costs"].data_ptr(),
        out["lp"].data_ptr(), out["lse"].data_ptr(), out["alpha"].data_ptr(), out["beta"].data_ptr(),
        hptr, status.data_ptr(), ws.data_ptr(), ws.numel(), st), "fwd")
    torch.cuda.synchronize()
    if dcost is None:
        dcost = torch.ones(B, dtype=torch.float32, device=dev)
    _lib.check(L.rnnt_b200_joint_loss_bwd(
        enc.data_ptr(), enc.stride(0), enc.stride(1), enc.stride(2), pred.data_ptr(), W.data_ptr(), b.data_ptr(),
        targets.data_ptr(), T_len.data_ptr(), U_len.data_ptr(), B, T, U1, H, V, blank, out["lp"].data_ptr(),
        out["lse"].data_ptr(), out["alpha"].data_ptr(), out["beta"].data_ptr(), hptr, dcost.data_ptr(), float(clamp),
        d_enc.data_ptr(), d_enc.stride(0), d_enc.stride(1), d_enc.stride(2), out["d_pred"].data_ptr(),
        out["dW"].data_ptr(), out["db"].data_ptr(), ring_tiles, flags, None, ws.data_ptr(), ws.numel(), st), "bwd")
    torch.cuda.synchronize()
    meta = ws[int(offs[0]): int(offs[0]) + (B + 5) * 4].view(torch.int32)
    out.update(ws=ws, hidden=hidden, offs=[int(x) for x in offs], Hp=hp.value, Vp=vp.value, ring_tiles=ring_tiles,
               status=int(status.item()), total_halves=int(meta[B]), active_halves=int(meta[B + 4]))
    return out


def ring_views(out):
    """g ring, activation rows (ring when recomputed; else the tile-indexed residual buffer), gradient scale S."""
    ws, offs, Hp, Vp = out["ws"], out["offs"], out["Hp"], out["Vp"]
    rows = out["ring_tiles"] * 128
    g = ws[offs[4]:offs[4] + rows * Vp * 2].view(torch.float16).view(rows, Vp)
    if out["hidden"] is not None:
        h = out["hidden"].view(torch.float16).view(-1, Hp)
    else:
        h = ws[offs[5]:offs[5] + rows * Hp * 2].view(torch.float16).view(rows, Hp)
    B = out["costs"].numel()
    scale = ws[offs[0] + (B + 2) * 4: offs[0] + (B + 4) * 4].view(torch.float32)   # {S, 1/S}
    return g, h, float(scale[0])


def ws_views(out):
    """Typed views of the workspace regions rnnt_b200_debug_ws_layout documents, as a backward call left them: tile_off
    [B+1] (prefix sums of half-tiles), W16 [Vp, Hp] fp16, bias2 [Vp] (bias * log2 e), coef (B,T,U1,4), g ring
    [ring_tiles*128, Vp] fp16, h ring [ring_tiles*128, Hp] fp16 (None with a saved residual), work list [n_active] int32,
    S and 1/S."""
    ws, offs, Hp, Vp = out["ws"], out["offs"], out["Hp"], out["Vp"]
    B, T, U1 = out["lse"].shape
    rows = out["ring_tiles"] * 128
    region = lambda off, n, dt: ws[off: off + n * dt.itemsize].view(dt)
    meta = region(offs[0], B + 5, torch.int32)
    gs = region(offs[0] + (B + 2) * 4, 2, torch.float32)
    return dict(tile_off=meta[:B + 1], W16=region(offs[1], Vp * Hp, torch.float16).view(Vp, Hp),
                bias2=region(offs[2], Vp, torch.float32), coef=region(offs[3], B * T * U1 * 4, torch.float32).view(B, T, U1, 4),
                g=region(offs[4], rows * Vp, torch.float16).view(rows, Vp),
                h=None if offs[5] < 0 else region(offs[5], rows * Hp, torch.float16).view(rows, Hp),
                work_list=region(offs[7], out["active_halves"], torch.int32), S=float(gs[0]), inv_S=float(gs[1]))


def tile_rows(T_len, U_len, out=None):
    """(b, t, u, valid) for every row of the activation buffer: the lattice of each utterance is cut into half-tiles of
    16(t) x 4(u) cells = 64 rows (row r <-> (t0 + r//4, u0 + r%4)), enumerated utterance by utterance, t-block by
    t-block, u-block by u-block.  Mirrors the kernels' map; with `out` (result of fused_raw) only the half-tiles of the
    backward's work list are returned, in ring order."""
    rows = []
    if out is not None:
        n = out["active_halves"]
        lst = out["ws"][out["offs"][7]: out["offs"][7] + n * 4].view(torch.int32).tolist()
        allrows = tile_rows(T_len, U_len)
        for hid in lst:
            rows.extend(allrows[hid * 64:(hid + 1) * 64])
        return rows
    for b, (Tb, Ub) in enumerate(zip(T_len.tolist(), U_len.tolist())):
        nt, nu = (Tb + 15) // 16, (Ub + 1 + 3) // 4
        for it in range(nt):
            for iu in range(nu):
                for r in range(64):
                    t, u = it * 16 + (r >> 2), iu * 4 + (r & 3)
                    rows.append((b, t, u, t < Tb and u <= Ub))
    return rows


def torch_reference(inp, emulate_bf16=False, dcost=None, device=None, blank=-1):
    """fp32 torch restatement on the SAME device (oracle/ref_path.py semantics), optionally with the joint GEMM
    operands (tanh output, W) rounded to fp16 as the kernels do, to separate kernel bugs from precision."""
    import torchaudio
    if device is not None:
        inp = {k: v.to(device) for k, v in inp.items()}
        dcost = None if dcost is None else dcost.to(device)
    enc = inp["enc"].detach().clone().requires_grad_(True)
    pred = inp["pred"].detach().clone().requires_grad_(True)
    W = inp["W"].detach().clone().requires_grad_(True)
    b = inp["b"].detach().clone().requires_grad_(True)
    h = torch.tanh(enc.unsqueeze(2) + pred.unsqueeze(1))
    if emulate_bf16:
        h = h + (h.detach().half().float() - h.detach())
        Wq = W + (W.detach().half().float() - W.detach())
    else:
        Wq = W
    logits = torch.nn.functional.linear(h, Wq, b)
    costs = torchaudio.functional.rnnt_loss(logits, inp["targets"], inp["T_len"], inp["U_len"], blank=blank, clamp=-1,
                                            reduction="none")
    costs.backward(torch.ones_like(costs) if dcost is None else dcost)
    return dict(costs=costs.detach(), d_enc=enc.grad, d_pred=pred.grad, dW=W.grad, db=b.grad,
                logits=logits.detach())


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / max(b.norm(), 1e-30)), float((a - b).abs().max())
