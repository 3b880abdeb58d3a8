"""In-tree build of the CUDA extension: nvcc -> rnnt_b200/_C/librnnt_b200.so (sm_100a only)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB_PATH = os.path.join(OUT_DIR, "librnnt_b200.so")
SOURCES = ["host_util.cu", "joint_gemm.cu", "dh_gemm.cu", "dw_gemm.cu", "linear_gemm.cu", "lattice.cu", "decode.cu", "decode_loop.cu", "beam_loop.cu", "api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build rnnt_b200's CUDA extension")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "rnnt_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_extension(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into one shared library.  Returns the library path."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(OUT_DIR, exist_ok=True)
    extra = os.environ.get("RNNT_B200_NVCC_EXTRA", "").split()
    cmd = [_nvcc()] + NVCC_FLAGS + extra + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH + ".tmp"]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    if verbose:
        print(proc.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build_extension(force=True, verbose=True))
