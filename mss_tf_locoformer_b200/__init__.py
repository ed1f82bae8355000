"""B200-native (sm_100a) implementation of the TF-Locoformer separation forward path.

Drop-in for chynggi/mss-tf-locoformer's ``TFLocoformerMSS`` / ``TFLocoformerSeparator`` /
``BSLocoformerSeparator``: same constructors, forward signatures and state_dict layout;
every arithmetic step runs in the hand-written CUDA kernels of ``csrc/`` behind the C ABI
declared in ``include/tfl.h``.  No CPU path, no Triton, no multi-backend dispatch: importing
works anywhere, running needs the built library and a CUDA device.
"""
from .models import BSLocoformerSeparator, TFLocoformerMSS, TFLocoformerSeparator, strip_prefix  # noqa: F401
from .modules import (  # noqa: F401
    ConvDeconv1d, LocoformerBlock, MSSTransform, MultiHeadSelfAttention, RMSGroupNorm, RotaryEmbedding,
    SwiGLUConvDeconv1d, TFLocoformerBlock,
)
from .engine import Engine, segment_ola, segment_ola_hop  # noqa: F401

__all__ = ["TFLocoformerMSS", "TFLocoformerSeparator", "BSLocoformerSeparator", "strip_prefix", "Engine", "segment_ola",
           "segment_ola_hop"]
