"""ctypes binding of the C-ABI in include/rnnt_b200.h.  There is no fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

_lib = None
ABI_VERSION = 3
FLAG_ALL_TILES = 1        # RNNT_B200_ALL_TILES
FLAG_DETERMINISTIC = 2    # RNNT_B200_DETERMINISTIC

_i32p = C.c_void_p   # device pointers are passed as integers
_f32p = C.c_void_p
_ptr = C.c_void_p

_SIGNATURES = {
    "rnnt_b200_abi_version": (C.c_int, []),
    "rnnt_b200_last_error": (C.c_char_p, []),
    "rnnt_b200_max_tiles": (C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "rnnt_b200_hidden_bytes": (C.c_size_t, [C.c_int] * 4),
    "rnnt_b200_workspace_bytes": (C.c_int, [C.c_int] * 5 + [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_size_t),
                                                           C.POINTER(C.c_size_t)]),
    "rnnt_b200_joint_loss_fwd": (C.c_int, [_f32p, C.c_int64, C.c_int64, C.c_int64, _f32p, _f32p, _f32p, _i32p, _i32p,
                                           _i32p] + [C.c_int] * 6 + [_f32p] * 5
                                 + [_ptr, _i32p, _ptr, C.c_size_t, _ptr]),
    "rnnt_b200_joint_loss_bwd": (C.c_int, [_f32p, C.c_int64, C.c_int64, C.c_int64, _f32p, _f32p, _f32p, _i32p, _i32p,
                                           _i32p] + [C.c_int] * 6 + [_f32p] * 4 + [_ptr, _f32p, C.c_float]
                                 + [_f32p, C.c_int64, C.c_int64, C.c_int64] + [_f32p] * 3
                                 + [C.c_int64, C.c_int, _ptr, _ptr, C.c_size_t, _ptr]),
    "rnnt_b200_loss_dense_fwd": (C.c_int, [_f32p, _i32p, _i32p, _i32p] + [C.c_int] * 5 + [_f32p] * 5 + [_ptr]),
    "rnnt_b200_loss_dense_bwd": (C.c_int, [_f32p, _i32p, _i32p, _i32p] + [C.c_int] * 5 + [_f32p] * 5
                                 + [C.c_float, _f32p, _f32p, _ptr]),
    "rnnt_b200_lattice": (C.c_int, [_f32p, _i32p, _i32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p, _ptr]),
    "rnnt_b200_joint_argmax_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "rnnt_b200_joint_argmax": (C.c_int, [_f32p, C.c_int64, _f32p, C.c_int64, _f32p, _f32p, C.c_int, C.c_int, C.c_int,
                                         _i32p, _f32p, _ptr, _ptr]),
    "rnnt_b200_greedy_decode_scratch_bytes": (C.c_size_t, [C.c_int] * 4),
    "rnnt_b200_greedy_decode": (C.c_int, [_f32p, C.c_int64, C.c_int64, _i32p] + [_f32p] * 13 + [C.c_int] * 8
                                + [_i32p, _i32p, _f32p, _ptr, _ptr]),
    "rnnt_b200_greedy_decode_state_bytes": (C.c_size_t, [C.c_int] * 4),
    "rnnt_b200_greedy_decode_stream_init": (C.c_int, [_f32p] * 13 + [C.c_int] * 4 + [_ptr, _ptr]),
    "rnnt_b200_greedy_decode_stream": (C.c_int, [_f32p, C.c_int64, C.c_int64, _i32p, _i32p] + [_f32p] * 13
                                       + [C.c_int] * 8 + [_i32p, _i32p, _f32p, _ptr, _ptr]),
    "rnnt_b200_linear_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int]),
    "rnnt_b200_linear_fwd": (C.c_int, [_f32p, _f32p, _f32p, C.c_int64, C.c_int, C.c_int, _f32p, _ptr, C.c_size_t, _ptr]),
    "rnnt_b200_linear_bwd": (C.c_int, [_f32p, _f32p, _f32p, C.c_int64, C.c_int, C.c_int, _f32p, _f32p, _f32p, C.c_int,
                                       _ptr, C.c_size_t, _ptr]),
    "rnnt_b200_profile_begin": (C.c_int, []),
    "rnnt_b200_profile_end": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int64)]),
    "rnnt_b200_debug_ws_layout": (C.c_int, [C.c_int] * 5 + [C.c_int64, C.c_int, C.POINTER(C.c_int64),
                                                           C.POINTER(C.c_int), C.POINTER(C.c_int)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib() -> C.CDLL:
    """Load librnnt_b200.so (built in-tree by rnnt_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            # first use in a fresh checkout: compile in-tree if a CUDA toolchain is present, otherwise fail loudly
            try:
                from .build import build_extension
                build_extension()
            except Exception as exc:
                raise RuntimeError(
                    f"rnnt_b200: CUDA extension not built ({LIB_PATH} missing) and building it failed: {exc}. "
                    "Run `python -m rnnt_b200.build` (needs nvcc); there is no CPU or PyTorch fallback for this "
                    "path.") from exc
        # RNNT_B200_LIB: load another build of the same ABI (A/B timing of kernel variants); the default is the in-tree one
        handle = C.CDLL(os.environ.get("RNNT_B200_LIB") or LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if handle.rnnt_b200_abi_version() != ABI_VERSION:
            raise RuntimeError("rnnt_b200: ABI version mismatch between Python host code and librnnt_b200.so")
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().rnnt_b200_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"rnnt_b200: {what} failed (code {rc}): {msg}")
