"""Forced-alignment cost on the GPU box: `joint_forced_align` (fused forward without a residual + the Viterbi kernel)
against `joint_rnnt_loss` under no_grad (the same forward without the Viterbi kernel), on
  - the bench shape B=32, T=400, U=100, H=V=1024, encoder features as the (B,T,H) view of a (B,H,T) tensor, and
  - the ragged stress shape B=8, T=1500, U=300, H=1024, V=4096 (lengths T/2..T, U/2..U).
The two calls alternate pass by pass after one warm-up call each.

Prints one JSON line: per shape and call the medians over the passes of the device time per kernel family (CUDA events
around every launch: the library's profiling hook; joint F, lattice, Viterbi = family 7 "other", prep), of the whole
call (host clock up to a synchronise), and lattice cells per second (valid cells sum T_b (U_b + 1) over the call).
The card's name and power limit are read in the same run."""
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

SHAPES = {"bench_B32_T400_U100_V1024": (32, 400, 100, 1024, 1024, False),
          "stress_B8_T1500_U300_V4096_ragged": (8, 1500, 300, 1024, 4096, True)}
PASSES = 7
FAMILIES = {"prep": 0, "joint_f": 1, "lattice": 2, "viterbi": 7}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + [""])[:2] if r.returncode == 0 else ("?", "?")
    return name, power


def inputs(B, T, U, H, V, ragged):
    g = torch.Generator().manual_seed(77)
    enc = torch.randn(B, H, T, generator=g).cuda().permute(0, 2, 1)       # the model's (B,T,H) view of (B,H,T)
    pred = torch.randn(B, U + 1, H, generator=g).cuda()
    bound = 1.0 / (H ** 0.5)
    W = ((torch.rand(V, H, generator=g) * 2 - 1) * bound).cuda()
    bias = ((torch.rand(V, generator=g) * 2 - 1) * bound).cuda()
    tg = torch.randint(0, V - 1, (B, U), generator=g, dtype=torch.int32).cuda()
    if ragged:
        tl = torch.randint(T // 2, T + 1, (B,), generator=g, dtype=torch.int32); tl[0] = T
        ul = torch.randint(U // 2, U + 1, (B,), generator=g, dtype=torch.int32); ul[-1] = U
    else:
        tl = torch.full((B,), T, dtype=torch.int32); ul = torch.full((B,), U, dtype=torch.int32)
    cells = int((tl.long() * (ul.long() + 1)).sum())
    return (enc, pred, W, bias, tg, tl.cuda(), ul.cuda()), cells


def measured(fn):
    """(per-family device ms, launches per family, host ms of fn() up to a synchronise)."""
    L = _lib.lib()
    torch.cuda.synchronize()
    _lib.check(L.rnnt_b200_profile_begin(), "profile_begin")
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) * 1e3
    ms, n = (C.c_float * 8)(), (C.c_int64 * 8)()
    _lib.check(L.rnnt_b200_profile_end(ms, n), "profile_end")
    return list(ms), list(n), host


def main():
    if not torch.cuda.is_available():
        raise SystemExit("align_bench.py needs a CUDA device")
    name, power = gpu_info()
    out = dict(bench="forced_align", gpu=name, power_limit=power, passes=PASSES, shapes={})
    for key, (B, T, U, H, V, ragged) in SHAPES.items():
        args, cells = inputs(B, T, U, H, V, ragged)
        calls = {"align": lambda: rnnt_b200.joint_forced_align(*args, validate=False),
                 "loss_no_grad": lambda: rnnt_b200.joint_rnnt_loss(*args, reduction="none", validate=False)}
        with torch.no_grad():
            for fn in calls.values():
                fn()                                                   # warm-up: module load, allocator
            rec = {k: dict(dev=[], n=None, host=[]) for k in calls}
            for _ in range(PASSES):
                for k, fn in calls.items():
                    ms, n, host = measured(fn)
                    rec[k]["dev"].append(ms)
                    rec[k]["n"] = n
                    rec[k]["host"].append(host)
        res = dict(B=B, T=T, U=U, H=H, V=V, ragged=ragged, valid_cells=cells)
        for k, r in rec.items():
            fam = {f: round(statistics.median(p[i] for p in r["dev"]), 4) for f, i in FAMILIES.items()}
            call = statistics.median(r["host"])
            res[k] = dict(device_ms=fam, launches={f: r["n"][i] for f, i in FAMILIES.items()},
                          call_ms=round(call, 3), call_ms_min=round(min(r["host"]), 3),
                          cells_per_s=round(cells / (call * 1e-3)))
        res["viterbi_over_call"] = round(res["align"]["device_ms"]["viterbi"] / res["align"]["call_ms"], 4)
        out["shapes"][key] = res
        del args
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
