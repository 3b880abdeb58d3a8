"""rnnt_b200: B200-native (sm_100a) RNN-T joint network + transducer loss hot path behind the reference's API."""
from .joint import JointNetwork, LazyJointLogits  # noqa: F401
from .model import RNNTModel, enable_zero_edit_mode  # noqa: F401
from .predictor import ConvPredictor  # noqa: F401
from .functional import (joint_rnnt_loss, rnnt_loss, joint_argmax, lattice, greedy_decode,  # noqa: F401
                         StreamingGreedyDecoder)

__all__ = ["JointNetwork", "LazyJointLogits", "RNNTModel", "ConvPredictor", "enable_zero_edit_mode",
           "joint_rnnt_loss", "rnnt_loss", "joint_argmax", "lattice", "greedy_decode", "StreamingGreedyDecoder"]
