"""Beam-search decode cost on the GPU box: B=64 utterances of up to T=400 frames (lengths 200..400), H=V=1024, E=512,
ConvPredictor at default init, blank bias +1.0, max_length 200 -- the greedy workload of scripts/decode_bench.py --
decoded by the beam kernel with K = 1, 2, 4, 8 and by the greedy kernel (max_outputs_per_step 10) on the same inputs,
in the same process, the variants alternating pass by pass.

Prints one JSON line: per variant the device time of the decode kernel per batch (CUDA events around every launch:
the library's profiling hook; median over the passes after one warm-up pass each), frames per second (the batch's
frames over that time), the whole Python call (host clock, ends in a synchronise as the results are returned as host
lists), and the tokens of the best hypotheses.  The card's name and power limit are read in the same run."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rnnt_b200  # noqa: E402
from rnnt_b200 import _lib  # noqa: E402

B, T, H, V, E, MAX_LEN = 64, 400, 1024, 1024, 512, 200
BEAMS = (1, 2, 4, 8)
PASSES = 5


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + [""])[:2] if r.returncode == 0 else ("?", "?")
    return name, power


def measured(fn):
    """(result, device ms of the library's decode kernel inside fn(), host ms of fn() up to a synchronise)."""
    L = _lib.lib()
    torch.cuda.synchronize()
    _lib.check(L.rnnt_b200_profile_begin(), "profile_begin")
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) * 1e3
    ms, n = (C.c_float * 8)(), (C.c_int64 * 8)()
    _lib.check(L.rnnt_b200_profile_end(ms, n), "profile_end")
    assert n[7] == 1, n[7]
    return out, ms[7], host


def main():
    if not torch.cuda.is_available():
        raise SystemExit("beam_decode_bench.py needs a CUDA device")
    name, power = gpu_info()
    torch.manual_seed(0)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += 1.0
    pred = rnnt_b200.ConvPredictor(V, H, E, 0.3)
    joint, pred = joint.cuda(), pred.cuda().eval()
    feats = torch.randn(B, T, H, device="cuda")
    lens = torch.randint(200, T + 1, (B,))
    lens[0] = T
    frames = int(lens.sum())
    w, bias = joint.joint_ln.weight, joint.joint_ln.bias
    variants = {"greedy": lambda: rnnt_b200.greedy_decode(feats, lens, w, bias, pred, V - 1, MAX_LEN, 10)}
    for k in BEAMS:
        variants[f"beam{k}"] = (lambda k=k: rnnt_b200.beam_decode(feats, lens, w, bias, pred, V - 1, k, MAX_LEN))
    for fn in variants.values():
        fn()                                                       # warm-up: module load, symbol tables, allocator
    dev, host, tokens = {k: [] for k in variants}, {k: [] for k in variants}, {}
    for _ in range(PASSES):
        for key, fn in variants.items():
            out, d, h = measured(fn)
            dev[key].append(d)
            host[key].append(h)
            tokens[key] = sum(len(x) for x in out) if key == "greedy" else sum(len(nb[0][0]) for nb in out)
    rec = {}
    for key in variants:
        d = statistics.median(dev[key])
        rec[key] = dict(device_ms=round(d, 3), device_ms_min=round(min(dev[key]), 3),
                        device_ms_max=round(max(dev[key]), 3), frames_per_s=round(frames / d * 1e3),
                        call_ms=round(statistics.median(host[key]), 3), tokens=tokens[key])
    out = dict(bench="beam_decode", gpu=name, power_limit=power, B=B, T=T, H=H, V=V, E=E, max_length=MAX_LEN,
               frames=frames, passes=PASSES, variants=rec)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
