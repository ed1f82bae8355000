"""ESPnet `AbsSeparator` adapter -- espnet2/enh/separator/tflocoformer_separator.py:22-189 on the B200 path.

Same constructor (leading positional ``input_dim``), ``forward(input, ilens, additional) -> (list of num_spk complex
[B, T, F] tensors, ilens, OrderedDict())`` and ``num_spk`` property as the reference class, same parameter names, so an
ESPnet checkpoint (keys prefixed ``separator.``; see ``strip_prefix``) loads with ``strict=True``.  When ``espnet2`` is
importable the class derives from ``espnet2.enh.separator.abs_separator.AbsSeparator`` (so ``espnet2.tasks.enh`` can
register it exactly as espnet2/tasks/enh.patch:14,22 does for the reference); otherwise from ``torch.nn.Module``.
The arithmetic is the standalone separator's (models.TFLocoformerSeparator): conv + gLN, Locoformer blocks, deconv.
"""
from collections import OrderedDict
from typing import Dict, List, Optional, Tuple, Union

import torch

from .models import TFLocoformerSeparator as _Standalone

try:  # pragma: no cover - espnet2 is not installed in the build image
    from espnet2.enh.separator.abs_separator import AbsSeparator as _Base
    HAVE_ESPNET = True
except Exception:  # noqa: BLE001
    _Base = torch.nn.Module
    HAVE_ESPNET = False


class TFLocoformerSeparator(_Standalone, _Base):
    """TF-Locoformer separator with the ESPnet interface."""

    def __init__(self, input_dim, num_spk: int = 2, n_layers: int = 6, emb_dim: int = 128,
                 norm_type: str = "rmsgrouporm", num_groups: int = 4, tf_order: str = "ft", n_heads: int = 4,
                 flash_attention: bool = False, attention_dim: int = 128, pos_enc: str = "rope",
                 ffn_type: Union[str, list] = "swiglu_conv1d", ffn_hidden_dim: Union[int, list] = 384,
                 conv1d_kernel: int = 4, conv1d_shift: int = 1, dropout: float = 0.0, eps: float = 1.0e-5,
                 differentiable: bool = False):
        # input_dim is accepted and unused, as in the reference (:66-89).  differentiable (not in the reference; an
        # ESPnet separator_conf key): train through torch autograd -- ESPnet's own loss, DDP and optimiser (autograd.py)
        _Standalone.__init__(self, num_spk=num_spk, n_layers=n_layers, emb_dim=emb_dim, norm_type=norm_type,
                             num_groups=num_groups, tf_order=tf_order, n_heads=n_heads, flash_attention=flash_attention,
                             attention_dim=attention_dim, pos_enc=pos_enc, ffn_type=ffn_type,
                             ffn_hidden_dim=ffn_hidden_dim, conv1d_kernel=conv1d_kernel, conv1d_shift=conv1d_shift,
                             dropout=dropout, eps=eps)
        self.differentiable = bool(differentiable)

    def forward(self, input: torch.Tensor, ilens: torch.Tensor, additional: Optional[Dict] = None
                ) -> Tuple[List[torch.Tensor], torch.Tensor, OrderedDict]:
        """input: complex [B, T, F] (or [B, T, 1, F]: ESPnet's channel axis follows time) -> ([B, T, F] x num_spk, ilens, {})."""
        if input.ndim == 4:
            # the reference asserts on shape[1] before its transpose (:160-162); what it means -- and what ESPnet
            # feeds, [B, T, C, F] -- is a single channel
            assert input.shape[2] == 1 or input.shape[1] == 1, "Only monaural input is supported."
            input = input[:, :, 0] if input.shape[2] == 1 else input[:, 0]
        est = _Standalone.forward(self, input)                    # [B, num_spk, T, F] complex64
        return [est[:, src] for src in range(self._num_spk)], ilens, OrderedDict()

    @property
    def num_spk(self):
        return self._num_spk

    @num_spk.setter
    def num_spk(self, value):      # the standalone constructor assigns the attribute; ESPnet reads the property
        object.__setattr__(self, "_num_spk", value)
