"""Drop-in for the reference's joint network (rnnt/joint.py:4-55): same constructor, attributes and state_dict keys.

Select it from the reference's YAML by `joint._target_: rnnt_b200.joint.JointNetwork`.  `forward` keeps returning
dense logits (eval.py:76, export_onnx.py use it on tiny shapes) unless zero-edit mode is on; `loss` is the fused
joint + transducer loss the training step calls instead of materialising (B,T,U+1,V) logits.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


class LazyJointLogits:
    """What `JointNetwork.forward` returns in zero-edit mode while grad is enabled: the operands of the joint, not
    its output.  `rnnt_b200.functional.rnnt_loss` consumes it with the fused kernels; anything else that needs
    real numbers calls `materialize()`."""

    def __init__(self, audio, text, weight, bias):
        self.audio, self.text, self.weight, self.bias = audio, text, weight, bias

    @property
    def shape(self):
        return torch.Size((self.audio.shape[0], self.audio.shape[1], self.text.shape[1], self.weight.shape[0]))

    @property
    def device(self):
        return self.audio.device

    @property
    def dtype(self):
        return self.audio.dtype

    def materialize(self) -> torch.Tensor:
        joint = torch.tanh(self.audio.unsqueeze(2) + self.text.unsqueeze(1))
        return F.linear(joint, self.weight, self.bias)


class JointNetwork(torch.nn.Module):
    def __init__(self, audio_features: int, text_features: int, hidden_features: int, num_classes: int):
        super().__init__()
        # same optional pre-projections and parameter names as rnnt/joint.py:8-18
        if audio_features > 0:
            self.audio_ln = torch.nn.Linear(audio_features, hidden_features)
        if text_features > 0:
            self.text_ln = torch.nn.Linear(text_features, hidden_features)
        self.activation = F.tanh
        self.joint_ln = torch.nn.Linear(hidden_features, num_classes)
        self.blank_idx = num_classes - 1
        self.zero_edit_mode = False

    def _project(self, audio_frame, text_frame, fused: bool = False):
        """rnnt/joint.py:26-30.  fused=True (the loss path): the projections run as tcgen05 GEMMs of the library."""
        if fused:
            from .functional import linear
        else:
            linear = F.linear
        if hasattr(self, "audio_ln"):
            audio_frame = linear(audio_frame, self.audio_ln.weight, self.audio_ln.bias)
        if hasattr(self, "text_ln"):
            text_frame = linear(text_frame, self.text_ln.weight, self.text_ln.bias)
        return audio_frame, text_frame

    def forward(self, audio_frame, text_frame):
        """(B,T,F) x (B,U+1,F) -> logits (B,T,U+1,V), as rnnt/joint.py:25-39.

        In zero-edit mode with grad enabled this returns a LazyJointLogits handle for the patched
        torchaudio.functional.rnnt_loss; the dense result is only meant for small shapes."""
        lazy = self.zero_edit_mode and torch.is_grad_enabled() and audio_frame.is_cuda
        audio_frame, text_frame = self._project(audio_frame, text_frame, fused=lazy)
        if lazy:
            return LazyJointLogits(audio_frame, text_frame, self.joint_ln.weight, self.joint_ln.bias)
        joint_frames = self.activation(audio_frame.unsqueeze(2) + text_frame.unsqueeze(1))
        return self.joint_ln(joint_frames)

    def single_forward(self, audio_frame, text_frame):
        """Aligned rows, no broadcasting (rnnt/joint.py:44-55).  Kept as plain scriptable torch for ONNX export."""
        audio_frame, text_frame = self._project(audio_frame, text_frame)
        return self.joint_ln(self.activation(audio_frame + text_frame))

    def loss(self, audio_frame, text_frame, targets, logit_lengths, target_lengths, blank: int = -1,
             clamp: float = -1, reduction: str = "mean", validate: bool = True):
        """Fused forward + transducer loss: replaces `joint(...)` + `torchaudio.functional.rnnt_loss(...)`
        (rnnt/model.py:32-41) without creating the logits.  Gradients reach every parameter through autograd."""
        from .functional import joint_rnnt_loss
        audio_frame, text_frame = self._project(audio_frame, text_frame, fused=True)
        return joint_rnnt_loss(audio_frame, text_frame, self.joint_ln.weight, self.joint_ln.bias, targets,
                               logit_lengths, target_lengths, blank=blank, clamp=clamp, reduction=reduction,
                               validate=validate)

    def align(self, audio_frame, text_frame, targets, logit_lengths, target_lengths, blank: int = -1,
              validate: bool = True):
        """Forced alignment of `targets` (`functional.joint_forced_align`): the fused pre-projections, then the fused
        forward and the Viterbi kernel.  Returns an `Alignment` (frames, score, log_prob) without grad."""
        from .functional import joint_forced_align
        with torch.no_grad():
            audio_frame, text_frame = self._project(audio_frame, text_frame, fused=True)
        return joint_forced_align(audio_frame, text_frame, self.joint_ln.weight, self.joint_ln.bias, targets,
                                  logit_lengths, target_lengths, blank=blank, validate=validate)

    def argmax_step(self, audio_rows, text_rows, return_margin: bool = False, **kw):
        """argmax(single_forward(audio_rows, text_rows), -1) for a batch of rows in fp32 (decode step)."""
        from .functional import joint_argmax
        audio_rows, text_rows = self._project(audio_rows, text_rows)
        return joint_argmax(audio_rows, text_rows, self.joint_ln.weight, self.joint_ln.bias, return_margin, **kw)
