"""Cost of token timing and confidence on the GPU box: each decode entry against its _aligned entry, in one process,
the two variants alternating pass by pass, on the workloads of the three decode benchmarks:
  greedy   scripts/decode_bench.py: B=64, T<=400, H=V=1024, E=512, ConvPredictor at default init, max_length 200,
           blank bias +1.0 (lengths 200..400) and +1.8 (300..400)
  stream   scripts/stream_decode_bench.py: the +1.0 workload through one stream state in chunks of 1, 4, 16, 64, 400
           frames (plain: rnnt_b200_greedy_decode_stream, aligned: rnnt_b200_greedy_decode_stream_aligned)
  beam     scripts/beam_decode_bench.py: the +1.0 workload with K = 1, 2, 4, 8

Prints one JSON line: per workload and variant the device time of the decode kernels of one pass (CUDA events around
every launch: the library's profiling hook; median, min and max over the passes after one warm-up pass), the aligned
cost relative to plain, and whether the plain outputs of the two variants are identical.  The card's name and power
limit are read in the same run."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rnnt_b200  # noqa: E402
import rnnt_b200.functional as RF  # noqa: E402
from rnnt_b200 import _lib  # noqa: E402

B, T, H, V, E, MAX_LEN = 64, 400, 1024, 1024, 512, 200
CHUNKS = (1, 4, 16, 64, 400)
BEAMS = (1, 2, 4, 8)
PASSES = int(os.environ.get("PASSES", "5"))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + [""])[:2] if r.returncode == 0 else ("?", "?")
    return name, power


def device_ms(fn):
    """(fn(), device ms of the library's decode kernels inside fn())."""
    L = _lib.lib()
    torch.cuda.synchronize()
    _lib.check(L.rnnt_b200_profile_begin(), "profile_begin")
    out = fn()
    torch.cuda.synchronize()
    ms, n = (C.c_float * 8)(), (C.c_int64 * 8)()
    _lib.check(L.rnnt_b200_profile_end(ms, n), "profile_end")
    return out, ms[7]


def alternate(variants):
    """{name: fn} -> {name: (device ms per pass list, last output)}, the variants alternating pass by pass."""
    for fn in variants.values():
        fn()                                                       # warm-up
    times, outs = {k: [] for k in variants}, {}
    for _ in range(PASSES):
        for k, fn in variants.items():
            outs[k], ms = device_ms(fn)
            times[k].append(ms)
    return times, outs


def summary(times):
    p, a = statistics.median(times["plain"]), statistics.median(times["aligned"])
    return dict(plain_ms=round(p, 3), plain_min_max=[round(min(times["plain"]), 3), round(max(times["plain"]), 3)],
                aligned_ms=round(a, 3),
                aligned_min_max=[round(min(times["aligned"]), 3), round(max(times["aligned"]), 3)],
                aligned_cost_pct=round(100 * (a / p - 1), 2))


def model_for(bias):
    torch.manual_seed(0)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += bias
    return joint.cuda(), rnnt_b200.ConvPredictor(V, H, E, 0.3).cuda().eval()


def inputs(lo):
    feats = torch.randn(B, T, H, device="cuda")
    lens = torch.randint(lo, T + 1, (B,))
    lens[0] = T
    return feats, lens


def greedy(bias, lo):
    joint, pred = model_for(bias)
    feats, lens = inputs(lo)
    w, b = joint.joint_ln.weight, joint.joint_ln.bias
    times, outs = alternate({
        "plain": lambda: rnnt_b200.greedy_decode(feats, lens, w, b, pred, V - 1, MAX_LEN, 10),
        "aligned": lambda: rnnt_b200.greedy_decode(feats, lens, w, b, pred, V - 1, MAX_LEN, 10, return_hypotheses=True),
    })
    same = outs["plain"] == [h.tokens for h in outs["aligned"]]
    return dict(blank_bias=bias, lengths=[lo, T], tokens=sum(len(x) for x in outs["plain"]), identical_tokens=same,
                **summary(times))


def stream(bias, lo):
    joint, pred = model_for(bias)
    feats, lens = inputs(lo)
    lens = lens.tolist()
    dec = rnnt_b200.StreamingGreedyDecoder(joint, pred, B, max_length=MAX_LEN)
    L = _lib.lib()
    out = {}
    for k in CHUNKS:
        chunks = []
        for t0 in range(0, T, k):
            c = feats[:, t0:t0 + k].contiguous()
            chunks.append((c, torch.tensor([min(max(x - t0, 0), k) for x in lens], dtype=torch.int32, device="cuda")))

        def run(aligned):
            dec.reset(range(B))
            stream_ptr = RF._stream_ptr(feats.device)
            for i, (c, n) in enumerate(chunks):
                args = (c.data_ptr(), c.stride(0), c.stride(1), n.data_ptr(), dec._reset_mask.data_ptr(),
                        *[t.data_ptr() for t in dec._params], B, c.shape[1], H, V, E, dec.blank, dec.max_length,
                        dec.max_outputs_per_step, dec.tokens.data_ptr(), dec.n_tokens.data_ptr(), None,
                        dec.state.data_ptr(), stream_ptr)
                if aligned:
                    _lib.check(L.rnnt_b200_greedy_decode_stream_aligned(*args, dec.frames.data_ptr(),
                                                                         dec.token_logp.data_ptr(),
                                                                         dec.scores.data_ptr()), "stream aligned")
                else:
                    _lib.check(L.rnnt_b200_greedy_decode_stream(*args), "stream")
                if i == 0:
                    dec._reset_mask.zero_()
            return dec.tokens.clone(), dec.n_tokens.clone()

        times, outs = alternate({"plain": lambda: run(False), "aligned": lambda: run(True)})
        same = all(torch.equal(x, y) for x, y in zip(outs["plain"], outs["aligned"]))
        out[str(k)] = dict(calls=len(chunks), identical_tokens=same, **summary(times))
    return dict(blank_bias=bias, lengths=[lo, T], chunks=out)


def beam(bias, lo):
    joint, pred = model_for(bias)
    feats, lens = inputs(lo)
    w, b = joint.joint_ln.weight, joint.joint_ln.bias
    out = {}
    for K in BEAMS:
        times, outs = alternate({
            "plain": lambda: rnnt_b200.beam_decode(feats, lens, w, b, pred, V - 1, K, MAX_LEN),
            "aligned": lambda: rnnt_b200.beam_decode(feats, lens, w, b, pred, V - 1, K, MAX_LEN,
                                                     return_hypotheses=True),
        })
        same = outs["plain"] == [[(h.tokens, h.score) for h in nb] for nb in outs["aligned"]]
        out[f"K{K}"] = dict(identical_nbest=same, **summary(times))
    return dict(blank_bias=bias, lengths=[lo, T], beams=out)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("aligned_decode_bench.py needs a CUDA device")
    name, power = gpu_info()
    res = dict(bench="aligned_decode", gpu=name, power_limit=power, B=B, T=T, H=H, V=V, E=E, max_length=MAX_LEN,
               passes=PASSES, greedy=[greedy(1.0, 200), greedy(1.8, 300)], stream=stream(1.0, 200),
               beam=beam(1.0, 200))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
