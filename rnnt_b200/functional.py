"""Host-side mirror of the reference's loss call (rnnt/model.py:35-41) on top of the C-ABI.

`joint_rnnt_loss` is the fused entry (joint + loss, no logits tensor); `rnnt_loss` has the exact signature of
`torchaudio.functional.rnnt_loss` and accepts either dense logits or the lazy handle `JointNetwork.forward`
returns in zero-edit mode.  PyTorch is used for device memory, streams and autograd plumbing only.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _lib

_DEFAULT_RING_BYTES = int(os.environ.get("RNNT_B200_RING_BYTES", str(3 << 30)))
# Keep h = tanh(enc + pred) (fp16, 2*H bytes per lattice cell) from the forward for the backward (default), or
# recompute it there (RNNT_B200_SAVE_HIDDEN=0: residuals shrink to 20 bytes per cell, the backward runs ~10 % slower).
_SAVE_HIDDEN = os.environ.get("RNNT_B200_SAVE_HIDDEN", "1") != "0"
# Bit-identical gradients from run to run (64-bit fixed-point accumulation instead of fp32 atomics); also switched on
# by torch.use_deterministic_algorithms(True) or per call (deterministic=True).
_DETERMINISTIC = os.environ.get("RNNT_B200_DETERMINISTIC", "0") != "0"

# Optional bookkeeping for bench.py / tests: when enabled, every fused backward leaves a 2-element device tensor
# (active half-tiles, total half-tiles) here.  Off by default (costs two tiny copies per step).
COLLECT_BACKWARD_STATS = False
_last_backward_stats = None
_last_decode_phase_cycles = None   # int64[8] cycle counters of the last decode kernel (P1..P6, -, grid barriers)

# Data-parallel hook (rnnt_b200.parallel.WeightGradBucket): when set, the fused backward writes dW / db straight into the
# sink's flat bucket and tells it the moment they are final, so the all-reduce overlaps the activation-gradient GEMM.
_weight_grad_sink = None


def set_weight_grad_sink(sink) -> None:
    global _weight_grad_sink
    _weight_grad_sink = sink


def last_backward_stats():
    """(active, total) half-tiles (16 t x 4 u lattice blocks) of the most recent fused backward, or None.  Synchronises."""
    if _last_backward_stats is None:
        return None
    a, t = _last_backward_stats.tolist()
    return int(a), int(t)


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError("rnnt_b200 runs on CUDA (sm_100a) tensors only; there is no CPU fallback")


def _validate_lengths(T, U1, logit_lengths, target_lengths):
    """Same checks (and messages) torchaudio's rnnt_loss raises (SURVEY appendix A8).  Synchronises."""
    if int(logit_lengths.max()) != T:
        raise RuntimeError("input length mismatch")
    if int(target_lengths.max()) + 1 != U1:
        raise RuntimeError("output length mismatch")


def _check_index_tensors(targets, logit_lengths, target_lengths):
    if targets.dtype != torch.int32:
        raise RuntimeError("targets must be int32 type")
    if logit_lengths.dtype != torch.int32:
        raise RuntimeError("logit_lengths must be int32 type")
    if target_lengths.dtype != torch.int32:
        raise RuntimeError("target_lengths must be int32 type")
    if not targets.is_contiguous():
        raise RuntimeError("targets must be contiguous")


def _check_blank(blank, V):
    """torchaudio's check and message: blank < 0 counts from the end of the vocabulary."""
    if not -V <= int(blank) < V:
        raise RuntimeError("blank must be within [0, logits.shape[-1])")


def pick_ring_tiles(B: int, T: int, U1: int, H: int, V: int, ring_bytes: Optional[int] = None,
                    have_hidden: bool = False) -> int:
    """Tiles per backward chunk: the batch's tile bound split into equal chunks of at most `ring_bytes`."""
    ring_bytes = _DEFAULT_RING_BYTES if ring_bytes is None else ring_bytes
    max_tiles = int(_lib.lib().rnnt_b200_max_tiles(B, T, U1))
    hp = (H + 63) // 64 * 64
    vp = (V + 255) // 256 * 256
    per_tile = 128 * (vp if have_hidden else hp + vp) * 2
    cap = max(1, ring_bytes // per_tile)
    nchunks = (max_tiles + cap - 1) // cap
    return (max_tiles + nchunks - 1) // nchunks


def workspace_bytes(B, T, U1, H, V, ring_tiles, have_hidden=False, flags=0):
    fwd, bwd = C.c_size_t(0), C.c_size_t(0)
    _lib.check(_lib.lib().rnnt_b200_workspace_bytes(B, T, U1, H, V, ring_tiles, int(bool(have_hidden)), int(flags),
                                                    C.byref(fwd), C.byref(bwd)), "workspace_bytes")
    return fwd.value, bwd.value


def _kernel_layout(x):
    """`x` itself if the kernels can read its (B,T,H) layout in place -- H-contiguous, or the T-contiguous permuted view
    of a dense (B,H,T) tensor (what rnnt/model.py:27-28 passes to the joint) -- else a contiguous copy."""
    B, T, H = x.shape
    if x.data_ptr() % 16 == 0:
        if x.stride(2) == 1 and x.stride(1) % 4 == 0 and x.stride(0) % 4 == 0 and x.stride(1) >= H:
            return x
        if x.stride(1) == 1 and x.stride(2) >= T:
            return x
    return x.contiguous()


def _grad_like(x):
    """Gradient buffer for the (B,T,H) input `x`: same memory layout when that layout is dense (a dense (B,H,T) tensor
    viewed as (B,T,H) gets its gradient in (B,H,T) order, so the encoder's backward sees a contiguous tensor)."""
    B, T, H = x.shape
    if x.stride(1) == 1 and x.stride(2) == T and (B == 1 or x.stride(0) == H * T) and T > 1:
        return torch.empty(B, H, T, dtype=torch.float32, device=x.device).permute(0, 2, 1)
    return torch.empty(B, T, H, dtype=torch.float32, device=x.device)


class _FusedJointLoss(torch.autograd.Function):
    """costs[B] = transducer loss of joint_ln(tanh(enc + pred)); residuals are 5 lattice-sized fp32 tensors."""

    @staticmethod
    def forward(ctx, enc, pred, weight, bias, targets, logit_lengths, target_lengths, blank, clamp, ring_bytes,
                skip_zero_tiles=True, save_hidden=None, deterministic=None):
        L = _lib.lib()
        B, T, H = enc.shape
        U1 = pred.shape[1]
        V = weight.shape[0]
        dev = enc.device
        enc_c = _kernel_layout(enc)          # no copy for the (B,H,T)-view layout of rnnt/model.py:28
        pred_c = pred.contiguous()
        weight_c = weight.contiguous()
        bias_c = bias.contiguous()
        costs = torch.empty(B, dtype=torch.float32, device=dev)
        lp = torch.empty(B, T, U1, 2, dtype=torch.float32, device=dev)
        lse = torch.empty(B, T, U1, dtype=torch.float32, device=dev)
        alpha = torch.empty(B, T, U1, dtype=torch.float32, device=dev)
        beta = torch.empty(B, T, U1, dtype=torch.float32, device=dev)
        needs_grad = any(ctx.needs_input_grad[:4])
        save_hidden = (_SAVE_HIDDEN if save_hidden is None else bool(save_hidden)) and needs_grad
        hidden = (torch.empty(L.rnnt_b200_hidden_bytes(B, T, U1, H), dtype=torch.uint8, device=dev)
                  if save_hidden else None)
        fwd_bytes, _ = workspace_bytes(B, T, U1, H, V, 0, save_hidden)
        ws = torch.empty(fwd_bytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            # out-of-range lengths (torchaudio raises for them) need no sync here: the kernels clamp them and turn
            # every cost of the batch into NaN
            _lib.check(L.rnnt_b200_joint_loss_fwd(
                enc_c.data_ptr(), enc_c.stride(0), enc_c.stride(1), enc_c.stride(2), pred_c.data_ptr(),
                weight_c.data_ptr(), bias_c.data_ptr(), targets.data_ptr(), logit_lengths.data_ptr(),
                target_lengths.data_ptr(), B, T, U1, H, V, blank, costs.data_ptr(), lp.data_ptr(), lse.data_ptr(),
                alpha.data_ptr(), beta.data_ptr(), hidden.data_ptr() if save_hidden else None, None, ws.data_ptr(),
                fwd_bytes, _stream_ptr(dev)), "joint_loss_fwd")
        ctx.save_for_backward(enc_c, pred_c, weight_c, bias_c, targets, logit_lengths, target_lengths,
                              lp, lse, alpha, beta, *([hidden] if save_hidden else []))
        ctx.have_hidden = save_hidden
        ctx.blank, ctx.clamp, ctx.ring_bytes = blank, clamp, ring_bytes
        if deterministic is None:
            deterministic = _DETERMINISTIC or torch.are_deterministic_algorithms_enabled()
        ctx.flags = (0 if skip_zero_tiles else _lib.FLAG_ALL_TILES) | (_lib.FLAG_DETERMINISTIC if deterministic else 0)
        ctx.mark_non_differentiable(lp, lse, alpha, beta)
        return costs, lp, lse, alpha, beta

    @staticmethod
    def backward(ctx, dcost, *_unused):
        L = _lib.lib()
        enc, pred, weight, bias, targets, logit_lengths, target_lengths, lp, lse, alpha, beta = ctx.saved_tensors[:11]
        hidden = ctx.saved_tensors[11] if ctx.have_hidden else None
        B, T, H = enc.shape
        U1 = pred.shape[1]
        V = weight.shape[0]
        dev = enc.device
        dcost = dcost.contiguous().float()
        d_enc = _grad_like(enc)
        d_pred = torch.empty(B, U1, H, dtype=torch.float32, device=dev)
        sink = _weight_grad_sink
        event = None
        if sink is not None and sink.accepts(V, H, dev):
            dW, db, event = sink.weight_grad_views(V, H)     # slices of the flat all-reduce bucket
        else:
            sink = None
            dW = torch.empty(V, H, dtype=torch.float32, device=dev)
            db = torch.empty(V, dtype=torch.float32, device=dev)
        ring_tiles = pick_ring_tiles(B, T, U1, H, V, ctx.ring_bytes, ctx.have_hidden)
        _, bwd_bytes = workspace_bytes(B, T, U1, H, V, ring_tiles, ctx.have_hidden, ctx.flags)
        ws = torch.empty(bwd_bytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.rnnt_b200_joint_loss_bwd(
                enc.data_ptr(), enc.stride(0), enc.stride(1), enc.stride(2), pred.data_ptr(), weight.data_ptr(),
                bias.data_ptr(), targets.data_ptr(), logit_lengths.data_ptr(), target_lengths.data_ptr(),
                B, T, U1, H, V, ctx.blank, lp.data_ptr(), lse.data_ptr(), alpha.data_ptr(), beta.data_ptr(),
                hidden.data_ptr() if ctx.have_hidden else None, dcost.data_ptr(), float(ctx.clamp),
                d_enc.data_ptr(), d_enc.stride(0), d_enc.stride(1), d_enc.stride(2), d_pred.data_ptr(),
                dW.data_ptr(), db.data_ptr(), ring_tiles, ctx.flags, event, ws.data_ptr(), bwd_bytes,
                _stream_ptr(dev)), "joint_loss_bwd")
            if sink is not None:
                sink.weight_grads_enqueued()      # starts the all-reduce on its side stream, gated by the event
        if COLLECT_BACKWARD_STATS:
            global _last_backward_stats
            meta = ws[: (B + 5) * 4].view(torch.int32)     # tile table region starts at offset 0
            _last_backward_stats = torch.stack([meta[B + 4], meta[B]])
        return d_enc, d_pred, dW, db, None, None, None, None, None, None, None, None, None


class _Linear(torch.autograd.Function):
    """y = x W^T + b through the library's tcgen05 GEMM (fp16 operands, fp32 accumulate), with its backward."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        L = _lib.lib()
        K, N = weight.shape[1], weight.shape[0]
        x2 = x.reshape(-1, K).contiguous()
        w = weight.contiguous()
        M = x2.shape[0]
        y = torch.empty(M, N, dtype=torch.float32, device=x.device)
        nbytes = L.rnnt_b200_linear_workspace_bytes(M, K, N, 0, 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(L.rnnt_b200_linear_fwd(x2.data_ptr(), w.data_ptr(), bias.contiguous().data_ptr(), M, K, N,
                                              y.data_ptr(), ws.data_ptr(), nbytes, _stream_ptr(x.device)), "linear_fwd")
        ctx.save_for_backward(x2, w)
        ctx.x_shape = x.shape
        return y.view(*x.shape[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        L = _lib.lib()
        x2, w = ctx.saved_tensors
        M, K = x2.shape
        N = w.shape[0]
        dy2 = dy.reshape(M, N).contiguous().float()
        flags = _lib.FLAG_DETERMINISTIC if (_DETERMINISTIC or torch.are_deterministic_algorithms_enabled()) else 0
        dx = torch.empty(M, K, dtype=torch.float32, device=dy.device) if ctx.needs_input_grad[0] else None
        dW = torch.empty(N, K, dtype=torch.float32, device=dy.device) if ctx.needs_input_grad[1] else None
        db = torch.empty(N, dtype=torch.float32, device=dy.device) if ctx.needs_input_grad[2] else None
        nbytes = L.rnnt_b200_linear_workspace_bytes(M, K, N, 1, flags)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dy.device)
        ptr = lambda t: t.data_ptr() if t is not None else None
        with torch.cuda.device(dy.device):
            _lib.check(L.rnnt_b200_linear_bwd(x2.data_ptr(), w.data_ptr(), dy2.data_ptr(), M, K, N, ptr(dx), ptr(dW),
                                              ptr(db), flags, ws.data_ptr(), nbytes, _stream_ptr(dy.device)),
                       "linear_bwd")
        return (dx.view(ctx.x_shape) if dx is not None else None), dW, db


def linear(x, weight, bias):
    """The joint's pre-projection (rnnt/joint.py:26-30 `audio_ln` / `text_ln`) as a tcgen05 GEMM of this library.
    fp32 CUDA tensors with in / out features that are multiples of 8 run the kernels; anything else is not part of
    the hot path and goes through torch's own linear."""
    if (x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32 and bias is not None
            and weight.shape[0] % 8 == 0 and weight.shape[1] % 8 == 0 and x.numel() > 0):
        return _Linear.apply(x, weight, bias)
    return torch.nn.functional.linear(x, weight, bias)


def _reduce(costs, reduction):
    if reduction == "none":
        return costs
    if reduction == "mean":
        return costs.mean()
    if reduction == "sum":
        return costs.sum()
    raise ValueError('reduction should be one of "none", "mean", "sum"')


def _check_joint_inputs(audio_frame, text_frame, weight, targets, logit_lengths, target_lengths, blank, validate):
    """The fused entries' checks on dtypes, shapes, blank and (validate=True) lengths, with torchaudio's messages."""
    if audio_frame.dtype != torch.float32 or text_frame.dtype != torch.float32:
        raise RuntimeError("joint inputs must be float32 (the fused kernels convert to fp16 operands internally)")
    if audio_frame.dim() != 3 or text_frame.dim() != 3 or audio_frame.shape[0] != text_frame.shape[0] \
            or audio_frame.shape[2] != text_frame.shape[2] or weight.shape[1] != audio_frame.shape[2]:
        raise RuntimeError("expected audio (B,T,H), text (B,U+1,H) and weight (V,H)")
    _check_index_tensors(targets, logit_lengths, target_lengths)
    if targets.shape[0] != audio_frame.shape[0] or targets.shape[1] != text_frame.shape[1] - 1:
        raise RuntimeError("output length mismatch")
    _check_blank(blank, weight.shape[0])
    if validate:
        _validate_lengths(audio_frame.shape[1], text_frame.shape[1], logit_lengths, target_lengths)


def joint_rnnt_loss(audio_frame, text_frame, weight, bias, targets, logit_lengths, target_lengths, blank: int = -1,
                    clamp: float = -1, reduction: str = "mean", validate: bool = True,
                    ring_bytes: Optional[int] = None, return_residuals: bool = False,
                    skip_zero_tiles: bool = True, save_hidden: Optional[bool] = None,
                    deterministic: Optional[bool] = None):
    """Fused replacement for `joint_ln(tanh(a.unsqueeze(2) + p.unsqueeze(1)))` (rnnt/joint.py:32-39) followed by
    `torchaudio.functional.rnnt_loss(..., blank, clamp, reduction)` (rnnt/model.py:35-41).

    audio_frame (B,T,H) and text_frame (B,U+1,H) are the (already projected) joint inputs; weight (V,H) / bias (V)
    are joint_ln's parameters.  Per-utterance costs when reduction="none".  validate=True performs torchaudio's
    host-side length checks (one device sync, as the reference does); pass False on the hot loop.
    skip_zero_tiles=False makes the backward process every half-tile (16 t x 4 u lattice block), including those whose fp16 logit-gradients
    are identically zero (same result, more work).  save_hidden: keep the fp16 activations tanh(a+p) from the forward
    for the backward (default; the reference's autograd keeps them in fp32) or recompute them there (False: the saved
    state shrinks to 20 bytes per lattice cell).  deterministic=True makes the gradients bit-identical from run to run
    (64-bit fixed-point accumulation instead of fp32 atomics; default: RNNT_B200_DETERMINISTIC or
    torch.use_deterministic_algorithms).  audio_frame may be the permuted (B,T,H) view of the encoder's (B,H,T) output
    (rnnt/model.py:27-28): it is read in place, and its gradient is produced in the same layout.
    With validate=False, lengths outside [1,T] / [0,U] (for which torchaudio raises) make every cost NaN instead.
    """
    _require_cuda(audio_frame, text_frame, weight, bias, targets, logit_lengths, target_lengths)
    _check_joint_inputs(audio_frame, text_frame, weight, targets, logit_lengths, target_lengths, blank, validate)
    costs, lp, lse, alpha, beta = _FusedJointLoss.apply(audio_frame, text_frame, weight.float(), bias.float(),
                                                        targets, logit_lengths, target_lengths, int(blank),
                                                        float(clamp), ring_bytes, bool(skip_zero_tiles), save_hidden,
                                                        deterministic)
    out = _reduce(costs, reduction)
    if return_residuals:
        return out, dict(lp=lp, lse=lse, alpha=alpha, beta=beta)
    return out


def _dense_forward(logits, targets, logit_lengths, target_lengths, blank):
    """rnnt_b200_loss_dense_fwd: costs and the residuals lp, lse, alpha, beta of dense fp32 logits (B,T,U+1,V)."""
    L = _lib.lib()
    B, T, U1, V = logits.shape
    dev = logits.device
    costs = torch.empty(B, dtype=torch.float32, device=dev)
    lp = torch.empty(B, T, U1, 2, dtype=torch.float32, device=dev)
    lse = torch.empty(B, T, U1, dtype=torch.float32, device=dev)
    alpha = torch.empty(B, T, U1, dtype=torch.float32, device=dev)
    beta = torch.empty(B, T, U1, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.rnnt_b200_loss_dense_fwd(
            logits.data_ptr(), targets.data_ptr(), logit_lengths.data_ptr(), target_lengths.data_ptr(),
            B, T, U1, V, blank, costs.data_ptr(), lp.data_ptr(), lse.data_ptr(), alpha.data_ptr(),
            beta.data_ptr(), _stream_ptr(dev)), "loss_dense_fwd")
    return costs, lp, lse, alpha, beta


class _DenseLoss(torch.autograd.Function):
    """torchaudio.functional.rnnt_loss on materialised logits: log-softmax gather, lattice, gradient kernel."""

    @staticmethod
    def forward(ctx, logits, targets, logit_lengths, target_lengths, blank, clamp):
        costs, lp, lse, alpha, beta = _dense_forward(logits, targets, logit_lengths, target_lengths, blank)
        ctx.save_for_backward(logits, targets, logit_lengths, target_lengths, lp, lse, alpha, beta)
        ctx.blank, ctx.clamp = blank, clamp
        return costs

    @staticmethod
    def backward(ctx, dcost):
        L = _lib.lib()
        logits, targets, logit_lengths, target_lengths, lp, lse, alpha, beta = ctx.saved_tensors
        B, T, U1, V = logits.shape
        dev = logits.device
        grads = torch.empty_like(logits)
        coef = torch.empty(B, T, U1, 4, dtype=torch.float32, device=dev)
        dcost = dcost.contiguous().float()
        clamped = ctx.clamp > 0
        with torch.cuda.device(dev):
            _lib.check(L.rnnt_b200_loss_dense_bwd(
                logits.data_ptr(), targets.data_ptr(), logit_lengths.data_ptr(), target_lengths.data_ptr(),
                B, T, U1, V, ctx.blank, lp.data_ptr(), lse.data_ptr(), alpha.data_ptr(), beta.data_ptr(),
                None if clamped else dcost.data_ptr(), float(ctx.clamp), coef.data_ptr(), grads.data_ptr(),
                _stream_ptr(dev)), "loss_dense_bwd")
        if clamped:
            grads = grads * dcost.view(-1, 1, 1, 1)
        return grads, None, None, None, None, None


def _check_dense_inputs(logits, targets, logit_lengths, target_lengths, blank):
    """The dense entries' checks (torchaudio's messages): fp32 contiguous 4-D logits, int32 indices, lengths, blank."""
    if logits.dtype != torch.float32:
        raise RuntimeError("logits must be float32 or float16 (half) type" if logits.dtype not in
                           (torch.float16,) else "rnnt_b200 dense loss supports float32 logits only")
    if not logits.is_contiguous():
        raise RuntimeError("logits must be contiguous")
    if logits.dim() != 4:
        raise RuntimeError("logits must be 4-D (batch, time, target, class)")
    _check_index_tensors(targets, logit_lengths, target_lengths)
    _validate_lengths(logits.shape[1], logits.shape[2], logit_lengths, target_lengths)
    _check_blank(blank, logits.shape[-1])


def rnnt_loss(logits, targets, logit_lengths, target_lengths, blank: int = -1, clamp: float = -1,
              reduction: str = "mean", fused_log_softmax: bool = True):
    """Same signature and error behaviour as torchaudio.functional.rnnt_loss (call site rnnt/model.py:35-41).

    `logits` may be the lazy handle a zero-edit-mode JointNetwork returns; the call then runs the fused kernels and
    no (B,T,U+1,V) tensor is ever created.  Dense fp32 logits run the dense CUDA kernels.
    """
    from .joint import LazyJointLogits
    if isinstance(logits, LazyJointLogits):
        return joint_rnnt_loss(logits.audio, logits.text, logits.weight, logits.bias, targets, logit_lengths,
                               target_lengths, blank=blank, clamp=clamp, reduction=reduction)
    if not fused_log_softmax:
        raise RuntimeError("rnnt_b200.rnnt_loss only implements fused_log_softmax=True (what the reference uses)")
    _require_cuda(logits, targets, logit_lengths, target_lengths)
    _check_dense_inputs(logits, targets, logit_lengths, target_lengths, blank)
    costs = _DenseLoss.apply(logits, targets, logit_lengths, target_lengths, int(blank), float(clamp))
    return _reduce(costs, reduction)


def lattice(lp, logit_lengths, target_lengths):
    """alpha, beta, costs from log-probs (B,T,U+1,2) -- the lattice kernel alone."""
    _require_cuda(lp, logit_lengths, target_lengths)
    B, T, U1, _ = lp.shape
    lp = lp.contiguous().float()
    alpha = torch.full((B, T, U1), float("-inf"), dtype=torch.float32, device=lp.device)
    beta = torch.full((B, T, U1), float("-inf"), dtype=torch.float32, device=lp.device)
    costs = torch.empty(B, dtype=torch.float32, device=lp.device)
    with torch.cuda.device(lp.device):
        _lib.check(_lib.lib().rnnt_b200_lattice(lp.data_ptr(), logit_lengths.data_ptr(), target_lengths.data_ptr(),
                                                B, T, U1, alpha.data_ptr(), beta.data_ptr(), costs.data_ptr(),
                                                _stream_ptr(lp.device)), "lattice")
    return alpha, beta, costs


class Alignment(NamedTuple):
    """Forced alignment of a batch (`forced_align`, `joint_forced_align`), device tensors without grad.
    frames (B,U) int32: frame of each target token on the best path, -1 past U_b.  score (B) fp32: the best path's
    log-probability.  log_prob (B) fp32: log P(targets | audio) = -cost of the same forward, so exp(score - log_prob)
    is the best path's posterior."""
    frames: torch.Tensor
    score: torch.Tensor
    log_prob: torch.Tensor


def viterbi(lp, logit_lengths, target_lengths):
    """frames (B,U) int32 and score (B) fp32 of the best lattice path from log-probs (B,T,U+1,2) -- the Viterbi kernel
    alone (`rnnt_b200_viterbi`; include/rnnt_b200.h states the recursion and the tie rule).  An utterance whose lengths
    are out of range gets score NaN and frames -1."""
    if lp.dim() != 4 or lp.shape[-1] != 2:
        raise RuntimeError("expected log-probs of shape (B,T,U+1,2)")
    if logit_lengths.dtype != torch.int32:
        raise RuntimeError("logit_lengths must be int32 type")
    if target_lengths.dtype != torch.int32:
        raise RuntimeError("target_lengths must be int32 type")
    _require_cuda(lp, logit_lengths, target_lengths)
    B, T, U1, _ = lp.shape
    lp = lp.contiguous().float()
    T_len, U_len = logit_lengths.contiguous(), target_lengths.contiguous()
    frames = torch.empty(B, U1 - 1, dtype=torch.int32, device=lp.device)
    score = torch.empty(B, dtype=torch.float32, device=lp.device)
    with torch.cuda.device(lp.device):
        _lib.check(_lib.lib().rnnt_b200_viterbi(lp.data_ptr(), T_len.data_ptr(), U_len.data_ptr(), B, T, U1,
                                                frames.data_ptr() if U1 > 1 else None, score.data_ptr(),
                                                _stream_ptr(lp.device)), "viterbi")
    return frames, score


def joint_forced_align(audio_frame, text_frame, weight, bias, targets, logit_lengths, target_lengths,
                       blank: int = -1, validate: bool = True) -> Alignment:
    """Forced alignment through the fused joint: the inputs, checks and messages of `joint_rnnt_loss`, the fused forward
    without an activation residual (no logits, no autograd), then the Viterbi kernel on its log-probs.  audio_frame may
    be the permuted (B,T,H) view of the encoder's (B,H,T) output; it is read in place.  With validate=False, lengths
    outside [1,T] / [0,U] give that utterance score NaN and frames -1, and every log_prob NaN (as the loss's costs)."""
    _check_joint_inputs(audio_frame, text_frame, weight, targets, logit_lengths, target_lengths, blank, validate)
    _require_cuda(audio_frame, text_frame, weight, bias, targets, logit_lengths, target_lengths)
    with torch.no_grad():
        costs, lp, _, _, _ = _FusedJointLoss.apply(audio_frame.detach(), text_frame.detach(), weight.detach().float(),
                                                   bias.detach().float(), targets, logit_lengths, target_lengths,
                                                   int(blank), -1.0, None, True, False, None)
        frames, score = viterbi(lp, logit_lengths, target_lengths)
    return Alignment(frames, score, -costs)


def forced_align(logits, targets, logit_lengths, target_lengths, blank: int = -1) -> Alignment:
    """Forced alignment with the inputs of `rnnt_loss`: dense fp32 logits (B,T,U+1,V) go through the dense front end,
    the lazy handle of a zero-edit-mode JointNetwork through `joint_forced_align`."""
    from .joint import LazyJointLogits
    if isinstance(logits, LazyJointLogits):
        return joint_forced_align(logits.audio, logits.text, logits.weight, logits.bias, targets, logit_lengths,
                                  target_lengths, blank=blank)
    _check_dense_inputs(logits, targets, logit_lengths, target_lengths, blank)
    _require_cuda(logits, targets, logit_lengths, target_lengths)
    with torch.no_grad():
        costs, lp, _, _, _ = _dense_forward(logits.detach(), targets, logit_lengths, target_lengths, int(blank))
        frames, score = viterbi(lp, logit_lengths, target_lengths)
    return Alignment(frames, score, -costs)


def joint_argmax_scratch(N: int, V: int, device):
    """Reusable scratch for `joint_argmax(..., scratch=...)` (lets a decode loop run allocation-free)."""
    n = max(1, _lib.lib().rnnt_b200_joint_argmax_scratch_bytes(N, V))
    return torch.empty(n, dtype=torch.uint8, device=device)


def joint_argmax(audio_rows, text_rows, weight, bias, return_margin: bool = False, out=None, margin_out=None,
                 scratch=None):
    """tokens[n] = argmax(joint.single_forward(audio_rows[n], text_rows[n])) in fp32 (rnnt/model.py:110-113)."""
    _require_cuda(audio_rows, text_rows, weight, bias)
    N, H = audio_rows.shape
    V = weight.shape[0]
    if audio_rows.stride(1) != 1:
        audio_rows = audio_rows.contiguous()
    if text_rows.stride(1) != 1:
        text_rows = text_rows.contiguous()
    weight = weight.contiguous()
    bias = bias.contiguous()
    dev = audio_rows.device
    tokens = torch.empty(N, dtype=torch.int32, device=dev) if out is None else out
    margin = None
    if return_margin:
        margin = torch.empty(N, dtype=torch.float32, device=dev) if margin_out is None else margin_out
    L = _lib.lib()
    if scratch is None:
        scratch = torch.empty(max(1, L.rnnt_b200_joint_argmax_scratch_bytes(N, V)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.rnnt_b200_joint_argmax(
            audio_rows.data_ptr(), audio_rows.stride(0), text_rows.data_ptr(), text_rows.stride(0),
            weight.data_ptr(), bias.data_ptr(), N, H, V, tokens.data_ptr(),
            margin.data_ptr() if return_margin else None, scratch.data_ptr(), _stream_ptr(dev)), "joint_argmax")
    return (tokens, margin) if return_margin else tokens


def _check_decode_sizes(predictor, joint_weight, H):
    if predictor.linear.out_features != H or joint_weight.shape[1] != H:
        raise RuntimeError("predictor output, encoder features and joint hidden size must agree")
    if predictor.conv1.conv.kernel_size[0] != 3 or predictor.conv2.conv.kernel_size[0] != 5:
        raise RuntimeError("decode kernel expects ConvPredictor's kernel sizes 3 and 5")


def _decode_params(joint_weight, joint_bias, p, dev):
    """The 13 weight tensors of the decode entries, fp32 contiguous on `dev`, conv weights re-laid as (E, k*E) with
    taps ordered oldest..newest."""
    E = p.embedding.embedding_dim
    f = lambda t: t.detach().to(dev, torch.float32).contiguous()
    w1 = f(p.conv1.conv.weight.detach().permute(0, 2, 1).reshape(E, -1))
    w2 = f(p.conv2.conv.weight.detach().permute(0, 2, 1).reshape(E, -1))
    return [f(joint_weight), f(joint_bias), f(p.embedding.weight), f(p.input_layer_norm.weight),
            f(p.input_layer_norm.bias), w1, f(p.conv1.conv.bias), w2, f(p.conv2.conv.bias), f(p.linear.weight),
            f(p.linear.bias), f(p.output_layer_norm.weight), f(p.output_layer_norm.bias)]


class DecodedHypothesis(NamedTuple):
    """One decoded hypothesis as host values: tokens (list[int]), frames (list[int], the encoder frame at which each
    token was emitted), log_probs (list[float], each token's log-probability at its step) and score (float).  For greedy
    decode the score is the log-probability of the greedy path through the transducer lattice, its blank steps
    included; for beam search it is the hypothesis's beam score.  Seconds are frame * the encoder's frame shift."""
    tokens: list
    frames: list
    log_probs: list
    score: float


def greedy_decode(audio_features, audio_feature_lens, joint_weight, joint_bias, predictor, blank: int,
                  max_length: int = 200, max_outputs_per_step: int = 10, return_margins: bool = False,
                  return_hypotheses: bool = False):
    """Batched greedy decode (rnnt/model.py:90-128 for every utterance of a batch) in ONE persistent CUDA kernel.

    audio_features (B,T,H) fp32, audio_feature_lens (B); `predictor` is a ConvPredictor-shaped module (embedding,
    input_layer_norm, conv1.conv, conv2.conv, linear, output_layer_norm).  Returns list[list[int]] (and, optionally,
    per-utterance lists of top-2 logit margins for every step the utterance was active in).  With return_hypotheses,
    one `DecodedHypothesis` per utterance replaces its token list (`rnnt_b200_greedy_decode_aligned`)."""
    _require_cuda(audio_features, joint_weight, joint_bias)
    L = _lib.lib()
    dev = audio_features.device
    B, T, H = audio_features.shape
    V = joint_weight.shape[0]
    _check_decode_sizes(predictor, joint_weight, H)
    E = predictor.embedding.embedding_dim
    enc = audio_features.detach().to(dev, torch.float32).contiguous()
    params = _decode_params(joint_weight, joint_bias, predictor, dev)
    lens = audio_feature_lens.to(dev, torch.int32).clamp(max=T).contiguous()
    max_len = max(int(max_length), 1)
    tokens = torch.zeros(B, max_len, dtype=torch.int32, device=dev)
    ntok = torch.ones(B, dtype=torch.int32, device=dev)
    margins = torch.full((T + max_len + 2, B), float("inf"), device=dev) if return_margins else None
    scratch = torch.empty(L.rnnt_b200_greedy_decode_scratch_bytes(B, H, V, E), dtype=torch.uint8, device=dev)
    args = (enc.data_ptr(), enc.stride(0), enc.stride(1), lens.data_ptr(), *[t.data_ptr() for t in params],
            B, T, H, V, E, int(blank), max_len, int(max_outputs_per_step), tokens.data_ptr(), ntok.data_ptr(),
            margins.data_ptr() if return_margins else None, scratch.data_ptr(), _stream_ptr(dev))
    with torch.cuda.device(dev):
        if return_hypotheses:
            frames = torch.zeros(B, max_len, dtype=torch.int32, device=dev)
            logp = torch.zeros(B, max_len, dtype=torch.float32, device=dev)
            scores = torch.zeros(B, dtype=torch.float32, device=dev)
            _lib.check(L.rnnt_b200_greedy_decode_aligned(*args, frames.data_ptr(), logp.data_ptr(),
                                                         scores.data_ptr()), "greedy_decode_aligned")
        else:
            _lib.check(L.rnnt_b200_greedy_decode(*args), "greedy_decode")
    global _last_decode_phase_cycles
    _last_decode_phase_cycles = scratch[:64].view(torch.int64)
    n = (ntok - 1).tolist()
    toks = tokens.tolist()
    result = [toks[b][: n[b]] for b in range(B)]
    if return_hypotheses:
        fr, lp, sc = frames.tolist(), logp.tolist(), scores.tolist()
        result = [DecodedHypothesis(result[b], fr[b][: n[b]], lp[b][: n[b]], sc[b]) for b in range(B)]
    if return_margins:
        ml = margins.t().tolist()
        return result, [[x for x in ml[b] if x != float("inf")] for b in range(B)]
    return result


MAX_BEAM = 8


def beam_decode(audio_features, audio_feature_lens, joint_weight, joint_bias, predictor, blank: int,
                beam_size: int = 4, max_length: int = 200, return_hypotheses: bool = False):
    """Batched frame-synchronous beam search (at most one symbol per frame, equal token lists merged with logaddexp) in
    ONE persistent CUDA kernel (`rnnt_b200_beam_decode`; include/rnnt_b200.h states the exact rule).

    audio_features (B,T,H) fp32 (any strides), audio_feature_lens (B); `predictor` is ConvPredictor-shaped, as for
    `greedy_decode`; beam_size in [1, 8]; max_length counts the seed blank.  Returns, per utterance, its n-best list:
    up to beam_size (tokens, log-score) pairs, best first (fewer when fewer distinct token lists exist).  With
    return_hypotheses the pairs are `DecodedHypothesis` objects carrying each token's frame and log-probability too
    (`rnnt_b200_beam_decode_aligned`)."""
    K = int(beam_size)
    if not 1 <= K <= MAX_BEAM:
        raise ValueError(f"beam_size must be in [1, {MAX_BEAM}] (got {beam_size})")
    _require_cuda(audio_features, joint_weight, joint_bias)
    L = _lib.lib()
    dev = audio_features.device
    B, T, H = audio_features.shape
    V = joint_weight.shape[0]
    _check_decode_sizes(predictor, joint_weight, H)
    E = predictor.embedding.embedding_dim
    enc = audio_features.detach().to(dev, torch.float32).contiguous()
    params = _decode_params(joint_weight, joint_bias, predictor, dev)
    lens = audio_feature_lens.to(dev, torch.int32).clamp(0, T).contiguous()
    max_len = max(int(max_length), 1)
    tokens = torch.zeros(B, K, max_len, dtype=torch.int32, device=dev)
    ntok = torch.zeros(B, K, dtype=torch.int32, device=dev)
    scores = torch.empty(B, K, dtype=torch.float32, device=dev)
    scratch = torch.empty(L.rnnt_b200_beam_decode_scratch_bytes(B, K, H, V, E, max_len), dtype=torch.uint8, device=dev)
    args = (enc.data_ptr(), enc.stride(0), enc.stride(1), lens.data_ptr(), *[t.data_ptr() for t in params],
            B, T, H, V, E, int(blank), K, max_len, tokens.data_ptr(), ntok.data_ptr(), scores.data_ptr(),
            scratch.data_ptr(), _stream_ptr(dev))
    with torch.cuda.device(dev):
        if return_hypotheses:
            frames = torch.zeros(B, K, max_len, dtype=torch.int32, device=dev)
            logp = torch.zeros(B, K, max_len, dtype=torch.float32, device=dev)
            _lib.check(L.rnnt_b200_beam_decode_aligned(*args, frames.data_ptr(), logp.data_ptr()),
                       "beam_decode_aligned")
        else:
            _lib.check(L.rnnt_b200_beam_decode(*args), "beam_decode")
    global _last_decode_phase_cycles
    _last_decode_phase_cycles = scratch[:64].view(torch.int64)
    n, toks, sc = ntok.tolist(), tokens.tolist(), scores.tolist()
    if return_hypotheses:
        fr, lp = frames.tolist(), logp.tolist()
        return [[DecodedHypothesis(toks[b][k][: n[b][k] - 1], fr[b][k][: n[b][k] - 1], lp[b][k][: n[b][k] - 1],
                                   sc[b][k]) for k in range(K) if n[b][k] > 0] for b in range(B)]
    return [[(toks[b][k][: n[b][k] - 1], sc[b][k]) for k in range(K) if n[b][k] > 0] for b in range(B)]


def _check_kernel_decode_modules(joint, predictor, what: str) -> None:
    """The modules the persistent decode kernels accept: a ConvPredictor-shaped predictor, a joint without
    pre-projections."""
    from .model import _is_conv_predictor, _is_lstm_predictor
    if _is_lstm_predictor(predictor):
        raise ValueError(f"{what} needs a ConvPredictor; decode an LSTM predictor with "
                         "RNNTModel.greedy_decode_features")
    if not _is_conv_predictor(predictor):
        raise ValueError("Unknown predictor type")
    if hasattr(joint, "audio_ln") or hasattr(joint, "text_ln"):
        raise ValueError(f"{what} does not support a joint with audio_ln / text_ln pre-projections")


class StreamingGreedyDecoder:
    """Greedy decode of `slots` live streams whose encoder frames arrive chunk by chunk, in the persistent decode kernel
    (`rnnt_b200_greedy_decode_stream`).  The decoder state of every slot stays on the device between calls.

    `reset(slots)` makes slots start a new utterance at the next `decode_chunk`; every other live slot continues where
    its previous call stopped.  However an utterance's frames are split into chunks, its tokens (and per-step margins)
    are bit-identical to `greedy_decode` on the whole utterance with the same max_length / max_outputs_per_step.  The
    weights are re-laid for the kernel once and the per-symbol tables are built from them: call `refresh()` after the
    weights change (it empties every slot).

    Every call also records each new token's frame (counted from the slot's reset) and log-probability, and the slot's
    running path score (`rnnt_b200_greedy_decode_stream_aligned`): `hypothesis(slot)` returns them, and
    `decode_chunk(..., return_hypotheses=True)` returns the new tokens with theirs."""

    def __init__(self, joint, predictor, slots: int, max_length: int = 200, max_outputs_per_step: int = 10):
        _check_kernel_decode_modules(joint, predictor, "streaming decode")
        if int(slots) < 1:
            raise ValueError("slots must be >= 1")
        weight = joint.joint_ln.weight
        _check_decode_sizes(predictor, weight, weight.shape[1])
        _require_cuda(weight)
        self.joint, self.predictor = joint, predictor
        self.slots = int(slots)
        self.max_length = max(int(max_length), 1)
        self.max_outputs_per_step = int(max_outputs_per_step)
        self.blank = int(joint.blank_idx)
        self.dev = weight.device
        self.V, self.H = weight.shape
        self.E = predictor.embedding.embedding_dim
        L = _lib.lib()
        S = self.slots
        i32 = dict(dtype=torch.int32, device=self.dev)
        self.state = torch.empty(L.rnnt_b200_greedy_decode_state_bytes(S, self.H, self.V, self.E), dtype=torch.uint8,
                                 device=self.dev)
        self.tokens = torch.zeros(S, self.max_length, **i32)     # column k-1 = k-th token of the slot's utterance
        self.n_tokens = torch.zeros(S, **i32)                    # 0 = empty slot, else 1 + tokens (seed blank counted)
        self.frames = torch.zeros(S, self.max_length, **i32)     # frame of each token, counted from the slot's reset
        self.token_logp = torch.zeros(S, self.max_length, dtype=torch.float32, device=self.dev)
        self.scores = torch.zeros(S, dtype=torch.float32, device=self.dev)   # running path score since the reset
        self._reset_mask = torch.zeros(S, **i32)
        self._pending = set()                                    # host copy of the reset mask
        self._n_host = [0] * S                                   # host copy of n_tokens
        self.refresh()

    def refresh(self) -> None:
        """Re-read the joint and predictor weights and rebuild the per-symbol tables.  Empties every slot (resets
        already requested stay pending)."""
        self._params = _decode_params(self.joint.joint_ln.weight, self.joint.joint_ln.bias, self.predictor, self.dev)
        with torch.cuda.device(self.dev):
            _lib.check(_lib.lib().rnnt_b200_greedy_decode_stream_init(
                *[t.data_ptr() for t in self._params], self.slots, self.H, self.V, self.E, self.state.data_ptr(),
                _stream_ptr(self.dev)), "greedy_decode_stream_init")
        self.n_tokens.zero_()
        self.scores.zero_()
        self._n_host = [0] * self.slots

    def reset(self, slots) -> None:
        """Start a new utterance in each of `slots` (an int or an iterable of ints) at the next decode_chunk."""
        idx = [int(slots)] if isinstance(slots, int) else [int(s) for s in slots]
        if any(s < 0 or s >= self.slots for s in idx):
            raise IndexError(f"slot index out of range [0, {self.slots})")
        if idx:
            self._reset_mask[torch.tensor(idx, device=self.dev)] = 1
            self._pending.update(idx)

    @property
    def finished(self) -> torch.Tensor:
        """(slots,) bool: the slot's utterance reached max_length tokens (seed blank counted) and ignores frames."""
        return self.n_tokens >= self.max_length

    def transcript(self, slot: int) -> list:
        """Every token the slot's current utterance has emitted so far."""
        return self.tokens[slot, : max(self._n_host[slot] - 1, 0)].tolist()

    def hypothesis(self, slot: int) -> DecodedHypothesis:
        """Everything the slot's current utterance has emitted so far: tokens, their frames (counted from the slot's
        reset) and log-probabilities, and the running path score (log-probability of the greedy path so far).  Like
        `transcript`, after `reset(slot)` it keeps returning the previous utterance until the next `decode_chunk`."""
        n = max(self._n_host[slot] - 1, 0)
        return DecodedHypothesis(self.tokens[slot, :n].tolist(), self.frames[slot, :n].tolist(),
                                 self.token_logp[slot, :n].tolist(), float(self.scores[slot]))

    def decode_chunk(self, features, lens=None, return_margins: bool = False, return_hypotheses: bool = False):
        """Feed the next chunk of encoder frames: features (slots, Tc, H) (any strides, e.g. the permuted view of the
        encoder's (slots, H, Tc) output), lens (slots,) = frames of the chunk each slot takes (default Tc, clamped to
        [0, Tc]).  Returns the tokens this call added per slot (and, optionally, the top-2 logit margins of every step
        the slot took in this call).  With return_hypotheses, each slot's entry is a `DecodedHypothesis` of the new
        tokens, their frames and log-probabilities, and the slot's running path score.  Synchronises once, to return
        the tokens."""
        _require_cuda(features)
        S, H = self.slots, self.H
        if features.dim() != 3 or features.shape[0] != S or features.shape[2] != H:
            raise RuntimeError(f"expected features (slots={S}, Tc, H={H}), got {tuple(features.shape)}")
        Tc = features.shape[1]
        enc = features.detach().to(self.dev, torch.float32).contiguous()
        if lens is None:
            chunk = torch.full((S,), Tc, dtype=torch.int32, device=self.dev)
        else:
            chunk = torch.as_tensor(lens).to(self.dev, torch.int32).clamp(0, Tc).contiguous()
            if chunk.shape != (S,):
                raise RuntimeError(f"expected lens of shape ({S},), got {tuple(chunk.shape)}")
        most = min(Tc * self.max_outputs_per_step, self.max_length - 1)     # tokens one call can add to a slot
        margins = (torch.full((Tc + most + 1, S), float("inf"), device=self.dev) if return_margins else None)
        start = [0 if b in self._pending else max(n - 1, 0) for b, n in enumerate(self._n_host)]
        L = _lib.lib()
        with torch.cuda.device(self.dev):
            _lib.check(L.rnnt_b200_greedy_decode_stream_aligned(
                enc.data_ptr(), enc.stride(0), enc.stride(1), chunk.data_ptr(), self._reset_mask.data_ptr(),
                *[t.data_ptr() for t in self._params], S, Tc, H, self.V, self.E, self.blank, self.max_length,
                self.max_outputs_per_step, self.tokens.data_ptr(), self.n_tokens.data_ptr(),
                margins.data_ptr() if return_margins else None, self.state.data_ptr(), _stream_ptr(self.dev),
                self.frames.data_ptr(), self.token_logp.data_ptr(), self.scores.data_ptr()), "greedy_decode_stream")
            self._reset_mask.zero_()
            self._pending.clear()
            # the columns this call can have written, gathered on the device: one copy to the host
            cols = (torch.tensor(start, dtype=torch.int64, device=self.dev).view(S, 1)
                    + torch.arange(most, device=self.dev)).clamp(max=self.max_length - 1)
            parts = [self.n_tokens.view(S, 1), self.tokens.gather(1, cols)]
            if return_hypotheses:   # the same single copy: frames, then log-probs and scores as their fp32 bits
                parts += [self.frames.gather(1, cols), self.token_logp.gather(1, cols).view(torch.int32),
                          self.scores.view(S, 1).view(torch.int32)]
            host = torch.cat(parts, 1).cpu().numpy()
            rows = host[:, : 1 + most].tolist()
        global _last_decode_phase_cycles
        _last_decode_phase_cycles = self.state[:64].view(torch.int64)
        self._n_host = [r[0] for r in rows]
        new = [rows[b][1: 1 + max(rows[b][0] - 1, 0) - start[b]] for b in range(S)]
        if return_hypotheses:
            fr = host[:, 1 + most: 1 + 2 * most].tolist()
            lp = host[:, 1 + 2 * most: 1 + 3 * most].view(np.float32).tolist()
            sc = host[:, 1 + 3 * most].view(np.float32).tolist()
            new = [DecodedHypothesis(new[b], fr[b][: len(new[b])], lp[b][: len(new[b])], sc[b]) for b in range(S)]
        if return_margins:
            ml = margins.t().tolist()
            return new, [[x for x in ml[b] if x != float("inf")] for b in range(S)]
        return new
