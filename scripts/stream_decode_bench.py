"""Streaming decode cost on the GPU box: the workloads of scripts/decode_bench.py (B=64, T=400, H=V=1024, E=512,
ConvPredictor at default init, max_length 200; blank bias +1.0 with lengths 200..400 and +1.8 with 300..400) decoded
once in one shot and then through StreamingGreedyDecoder in chunks of 1, 4, 16, 64 and 400 frames per call.

Prints one JSON line: per workload the one-shot pass, and per chunk size the total time of a pass (host clock, every
call ends in a synchronise as decode_chunk returns host lists), the per-call latency a server sees (median, p90), the
device time of the decode kernel per call (CUDA events of the library's profiling hook), the fixed cost per call
((chunked total - one-shot total) / calls, host and device) and whether tokens and per-step margins are identical to
the one-shot decode.  The card's name and power limit are read in the same run."""
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
CHUNKS = (1, 4, 16, 64, 400)
PASSES = 5


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + [""])[:2] if r.returncode == 0 else ("?", "?")
    return name, power


def kernel_ms(fn):
    """Device time of the library's decode kernels inside fn() and their launch count (CUDA events per launch)."""
    L = _lib.lib()
    _lib.check(L.rnnt_b200_profile_begin(), "profile_begin")
    fn()
    ms, n = (C.c_float * 8)(), (C.c_int64 * 8)()
    _lib.check(L.rnnt_b200_profile_end(ms, n), "profile_end")
    return ms[7], n[7]


def one_shot(model, feats, lens, margins=False):
    return rnnt_b200.greedy_decode(feats, lens, model.joint.joint_ln.weight, model.joint.joint_ln.bias,
                                   model.predictor, model.joint.blank_idx, MAX_LEN, 10, return_margins=margins)


def chunked(dec, feats, lens, k, margins=False, lat=None):
    dec.reset(range(B))
    toks, mgs = [[] for _ in range(B)], [[] for _ in range(B)]
    for t0 in range(0, T, k):
        n = [min(max(x - t0, 0), k) for x in lens]
        t1 = time.perf_counter()
        out = dec.decode_chunk(feats[:, t0:t0 + k], n, return_margins=margins)
        if lat is not None:
            lat.append(time.perf_counter() - t1)
        new, mg = out if margins else (out, None)
        for b in range(B):
            toks[b] += new[b]
            if margins:
                mgs[b] += mg[b]
    return toks, mgs


def timed(fn, passes=PASSES):
    times = []
    for _ in range(passes):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return statistics.median(times) * 1e3


def workload(bias, lo):
    torch.manual_seed(0)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += bias
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.3), torch.nn.Identity(), joint).cuda().eval()
    feats = torch.randn(B, T, H, device="cuda")
    lens_t = torch.randint(lo, T + 1, (B,))
    lens_t[0] = T
    lens = lens_t.tolist()
    ref_tok, ref_mg = one_shot(model, feats, lens_t, margins=True)
    one_ms = timed(lambda: one_shot(model, feats, lens_t))
    one_dev, _ = kernel_ms(lambda: one_shot(model, feats, lens_t))
    rec = dict(blank_bias=bias, lengths=[lo, T], tokens=sum(len(x) for x in ref_tok), one_shot_ms=round(one_ms, 3),
               one_shot_device_ms=round(one_dev, 3), chunks={})
    dec = model.streaming_decoder(B, max_length=MAX_LEN)
    for k in CHUNKS:
        calls = (T + k - 1) // k
        tok, mg = chunked(dec, feats, lens, k, margins=True)       # warm-up and the identity check
        identical = tok == ref_tok and mg == ref_mg
        lat = []
        total = timed(lambda: chunked(dec, feats, lens, k, lat=lat))
        dev_ms, launches = kernel_ms(lambda: chunked(dec, feats, lens, k))
        lat_us = sorted(x * 1e6 for x in lat)
        rec["chunks"][str(k)] = dict(
            calls=calls, total_ms=round(total, 3), vs_one_shot=round(total / one_ms, 3),
            call_latency_us_median=round(statistics.median(lat_us), 1),
            call_latency_us_p90=round(lat_us[int(0.9 * (len(lat_us) - 1))], 1),
            device_us_per_call=round(dev_ms * 1e3 / max(launches, 1), 1), device_total_ms=round(dev_ms, 3),
            fixed_cost_us_per_call_host=round((total - one_ms) * 1e3 / calls, 1),
            fixed_cost_us_per_call_device=round((dev_ms - one_dev) * 1e3 / calls, 1),
            identical_tokens_and_margins=identical)
    return rec


def main():
    if not torch.cuda.is_available():
        raise SystemExit("stream_decode_bench.py needs a CUDA device")
    name, power = gpu_info()
    out = dict(bench="stream_decode", gpu=name, power_limit=power, B=B, T=T, H=H, V=V, E=E, max_length=MAX_LEN,
               passes=PASSES, workloads=[workload(1.0, 200), workload(1.8, 300)])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
