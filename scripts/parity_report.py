"""Print the measured parity errors of the fused path for every shape the tests use (run on the B200 box).
The tolerances in tests/test_gpu_parity.py are set from this report."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import fused_raw, load_loss_golden, make_inputs, rel_err, torch_reference  # noqa: E402


def report(tag, out, ref, refq=None):
    cost = float(((out["costs"].cpu() - ref["costs"].cpu()).abs() / ref["costs"].cpu().abs().clamp_min(1e-6)).max())
    parts = [f"{tag:42s} cost {cost:.1e}"]
    for k in ("d_enc", "d_pred", "dW", "db"):
        r, a = rel_err(out[k].cpu(), ref[k].cpu())
        s = f"{k} {r:.1e}"
        if refq is not None:
            s += f"/{rel_err(out[k].cpu(), refq[k].cpu())[0]:.1e}"
        parts.append(s)
    print("  ".join(parts), flush=True)


def main():
    gd = os.path.join(ROOT, "tests", "golden")
    for name in ("loss_tiny", "loss_mid", "loss_wide"):
        g = load_loss_golden(gd, name)
        t = lambda k, dt=None: torch.from_numpy(g[k]).cuda() if dt is None else torch.from_numpy(g[k]).to(dt).cuda()
        inp = dict(enc=t("enc"), pred=t("pred"), W=t("W"), b=t("b"), targets=t("targets", torch.int32),
                   T_len=t("T_len", torch.int32), U_len=t("U_len", torch.int32))
        ref = {k: torch.from_numpy(g[k]) for k in ("costs", "d_enc", "d_pred", "dW", "db")}
        out = fused_raw(inp)
        out["dW"] = out["dW"][t("dW_rows", torch.long)]
        report("golden " + name, out, ref)
    for shape in [(2, 20, 9, 64, 256, True), (3, 37, 13, 128, 512, True), (2, 33, 17, 1024, 1024, False),
                  (4, 200, 40, 1024, 1024, False), (2, 160, 40, 128, 512, True), (2, 12, 5, 64, 256, False),
                  (4, 18, 6, 64, 256, True)]:
        B, T, U, H, V, ragged = shape
        inp = make_inputs(B, T, U, H, V, ragged=ragged)
        report("same-device " + str(shape), fused_raw(inp), torch_reference(inp), torch_reference(inp, emulate_bf16=True))
    rng = np.random.default_rng(2024)
    cases = [(1, 1, 0, 8, 2), (2, 1, 3, 16, 5), (3, 9, 0, 24, 37), (1, 40, 20, 72, 300)]
    for _ in range(8):
        cases.append((int(rng.integers(1, 6)), int(rng.integers(1, 41)), int(rng.integers(0, 21)),
                      int(rng.choice([8, 16, 40, 64, 72, 128])), int(rng.choice([2, 3, 37, 256, 257, 300]))))
    for i, (B, T, U, H, V) in enumerate(cases):
        inp = make_inputs(B, T, U, H, V, ragged=True, seed=100 + i)
        report("fuzz " + str((B, T, U, H, V)), fused_raw(inp), torch_reference(inp, device="cpu"))
    inp = make_inputs(2, 60, 20, 1024, 1024, ragged=True, seed=77, scale=4.0)
    inp["W"] = inp["W"] * 32.0
    inp["b"] = inp["b"] * 32.0
    report("trained-scale (x4 inputs, x32 weights)", fused_raw(inp), torch_reference(inp),
           torch_reference(inp, emulate_bf16=True))


if __name__ == "__main__":
    main()
