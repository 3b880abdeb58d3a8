"""Device time of rnnt_b200_linear_bwd (linear_gemm.cu) per output combination, for one or more builds of the library.

  python scripts/linear_bwd_time.py [--lib PATH ...] [--iters N] [--det]

At the reference width (K = N = 1024) and M = 12800 (B T) and 3232 (B (U+1)): dx only (K-major x MN-major), dW only
(MN-major x MN-major, split-K), db only, and all three.  Each call is timed alone with CUDA events after a 256 MB
write that evicts L2, so every call reads its operands from HBM.  The builds (default: the in-tree library) are
alternated call by call, so that they share the machine's state; the median over the calls is printed, in ms.
"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rnnt_b200 import _lib  # noqa: E402


def load(path):
    h = C.CDLL(path)
    for name in ("rnnt_b200_linear_workspace_bytes", "rnnt_b200_linear_bwd", "rnnt_b200_last_error"):
        res, args = _lib._SIGNATURES[name]
        fn = getattr(h, name)
        fn.restype, fn.argtypes = res, args
    return h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=None)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--det", action="store_true", help="RNNT_B200_DETERMINISTIC")
    a = ap.parse_args()
    paths = a.lib or [_lib.LIB_PATH]
    libs = [load(p) for p in paths]
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("device:", q[0] if q else torch.cuda.get_device_name(0))
    flags = _lib.FLAG_DETERMINISTIC if a.det else 0
    st = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    K = N = 1024
    for M in (12800, 3232):
        g = torch.Generator(device="cuda").manual_seed(M)
        x = torch.randn(M, K, device="cuda", generator=g)
        W = torch.randn(N, K, device="cuda", generator=g) / 32
        dy = torch.randn(M, N, device="cuda", generator=g) * 1e-4
        dx, dW, db = (torch.empty(M, K, device="cuda"), torch.empty(N, K, device="cuda"),
                      torch.empty(N, device="cuda"))
        ws = [torch.empty(L.rnnt_b200_linear_workspace_bytes(M, K, N, 1, flags), dtype=torch.uint8, device="cuda")
              for L in libs]
        for label, outs in (("dx", (dx, None, None)), ("dW", (None, dW, None)), ("db", (None, None, db)),
                            ("dx+dW+db", (dx, dW, db))):
            ptrs = [t.data_ptr() if t is not None else None for t in outs]
            times = [[] for _ in libs]
            for it in range(a.iters + 3):
                for i, L in enumerate(libs):
                    flush.fill_(it & 0xFF)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    rc = L.rnnt_b200_linear_bwd(x.data_ptr(), W.data_ptr(), dy.data_ptr(), M, K, N, *ptrs, flags,
                                                ws[i].data_ptr(), ws[i].numel(), st)
                    e1.record()
                    assert rc == 0, L.rnnt_b200_last_error()
                    torch.cuda.synchronize()
                    if it >= 3:
                        times[i].append(e0.elapsed_time(e1))
            meds = [statistics.median(t) for t in times]
            row = "  ".join(f"{os.path.basename(p)} {m:.4f} ms (spread {min(t):.4f}-{max(t):.4f})"
                            for p, m, t in zip(paths, meds, times))
            print(f"M={M:5d} K={K} N={N} {'det ' if a.det else ''}{label:9s} {row}")


if __name__ == "__main__":
    main()
