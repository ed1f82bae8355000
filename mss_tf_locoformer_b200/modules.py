"""Drop-in module surface of the reference, backed by the sm_100a C-ABI library.

Same class names, constructor kwargs, assertions, forward signatures and state_dict
layout as /root/reference/models/mss_tflocoformer.py and
/root/reference/standalone/tflocoformer_separator.py, so existing checkpoints load with
``strict=True`` and callers (inference/separate.py:95-104,148) switch by changing one
import.  The torch.nn layers below are PARAMETER CONTAINERS ONLY (they give the reference's
key names, shapes and default initialisation); none of their forward methods is ever
called -- all arithmetic runs in csrc/ kernels.  Forward-only: no autograd, no CPU path.
"""
from typing import Dict, List, Optional, Union

import torch
import torch.nn as nn

from .engine import Engine, PRECISIONS

SOURCE_NAMES = ["vocals", "drums", "bass", "other"]  # models/mss_tflocoformer.py:242


def _resolve_precision(owner) -> int:
    """'fp32' | 'bf16' | 'tf32' | None (auto: bf16 iff the caller is inside torch.autocast(cuda, bfloat16),
    which is how the reference enters its bf16 mode -- SURVEY.md F9; fp32 otherwise).  'tf32' is opt-in only: it is
    never chosen from torch.backends.cudnn.allow_tf32, whose default is True."""
    p = getattr(owner, "precision", None)
    if p is None:
        auto = torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16
        return PRECISIONS["bf16" if auto else "fp32"]
    if p not in PRECISIONS:
        raise ValueError(f"precision must be one of {list(PRECISIONS)} or None, got {p!r}")
    return PRECISIONS[p]


def _no_training_dropout(module: nn.Module):
    if module.training and getattr(module, "_dropout_p", 0.0) > 0.0:
        raise NotImplementedError(
            "training-mode dropout is not implemented by the B200 forward path; call .eval() "
            "(parity with the reference is defined for eval mode only)")


def _forward_only(module: nn.Module, *tensors):
    _no_training_dropout(module)
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise NotImplementedError("mss_tf_locoformer_b200 is forward-only (no autograd); run under torch.no_grad() "
                                  "with inputs that do not require grad")


class RotaryEmbedding(nn.Module):
    """Holds the ``freqs`` parameter of rotary_embedding_torch.RotaryEmbedding(dim) so state_dicts keep the
    ``...attn.rope.freqs`` key (models/mss_tflocoformer.py:153-154).  The rotation itself is applied inside
    the attention kernels (interleaved pairs, theta = 10000, positions from 0)."""

    def __init__(self, dim: int, theta: float = 10000.0):
        super().__init__()
        idx = torch.arange(0, dim, 2)[: dim // 2].float()
        self.freqs = nn.Parameter(1.0 / (theta ** (idx / dim)), requires_grad=False)


class MSSTransform(nn.Module):
    """models/mss_tflocoformer.py:20-75.  STFT / iSTFT run as kernels of the owning model's engine."""

    def __init__(self, n_fft: int = 2048, hop_length: int = 1024, win_length: Optional[int] = None, window: str = "hann"):
        super().__init__()
        self.n_fft = n_fft
        self.hop_length = hop_length
        self.win_length = win_length or n_fft
        self.window = window
        if self.win_length != n_fft or window != "hann":
            raise NotImplementedError("only win_length == n_fft with a Hann window is supported (the reference's use)")
        self._owner = None

    def _engine(self) -> Engine:
        if self._owner is None:
            raise RuntimeError("MSSTransform must belong to a TFLocoformerMSS to run")
        return self._owner()._ready()

    def stft(self, audio: torch.Tensor) -> torch.Tensor:
        """audio [B, T] -> complex [B, F, Tf] (:36-54)."""
        ri = self._engine().stft(audio.to(torch.float32))
        return torch.view_as_complex(ri).transpose(-1, -2)

    def istft(self, spec: torch.Tensor, length: Optional[int] = None) -> torch.Tensor:
        """complex [B, F, Tf] -> audio [B, T] (:56-75)."""
        eng = self._engine()
        B, F, Tf = spec.shape
        if length is None:
            length = self.hop_length * (Tf - 1)
        ri = torch.view_as_real(spec.transpose(-1, -2).contiguous()).unsqueeze(1)  # [B, 1, Tf, F, 2]
        if eng.cfg["n_src"] != 1:
            ri = ri.expand(B, eng.cfg["n_src"], Tf, F, 2).contiguous()
        return eng.istft(ri, length)[0]


class RMSGroupNorm(nn.Module):
    """models/mss_tflocoformer.py:658-706."""

    def __init__(self, num_groups: int, dim: int, eps: float = 1e-8, bias: bool = False):
        super().__init__()
        assert dim % num_groups == 0, (dim, num_groups)
        self.num_groups = num_groups
        self.dim_per_group = dim // self.num_groups
        self.gamma = nn.Parameter(torch.ones(dim, dtype=torch.float32))
        self.bias = bias
        if self.bias:
            raise NotImplementedError("RMSGroupNorm(bias=True) is never used by the reference models")
        self.eps = eps
        self._site = None  # (owner weakref, layer, axis, which)

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        if self._site is None:
            raise RuntimeError("RMSGroupNorm must belong to a separator model to run")
        owner, layer, axis, which = self._site
        return owner()._ready().rms_group_norm(layer, axis, which, input.to(torch.float32))


class SwiGLUConvDeconv1d(nn.Module):
    """models/mss_tflocoformer.py:603-655 (parameters only; the fused norm+FFN+residual kernel is reached
    through LocoformerBlock / the model forward)."""

    def __init__(self, dim: int, dim_inner: int, conv1d_kernel: int, conv1d_shift: int, dropout: float = 0.0, **kwargs):
        super().__init__()
        if conv1d_shift != 1:
            raise NotImplementedError("conv1d_shift != 1 is not supported (no reference config or test uses it)")
        self.conv1d = nn.Conv1d(dim, dim_inner * 2, conv1d_kernel, stride=conv1d_shift)
        self.swish = nn.SiLU()
        self.deconv1d = nn.ConvTranspose1d(dim_inner, dim, conv1d_kernel, stride=conv1d_shift)
        self.dropout = nn.Dropout(dropout)
        self.dim_inner = dim_inner
        self.diff_ks = conv1d_kernel - conv1d_shift
        self.conv1d_kernel = conv1d_kernel
        self.conv1d_shift = conv1d_shift


class ConvDeconv1d(nn.Module):
    """models/mss_tflocoformer.py:562-600.  Raises: the reference's own forward fails for the default
    kernel 4 / shift 1 (SURVEY.md a8) and no config or test selects it."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        raise NotImplementedError("ffn_type='conv1d' is not supported; use 'swiglu_conv1d'")


class MultiHeadSelfAttention(nn.Module):
    """models/mss_tflocoformer.py:467-559 (parameters only)."""

    def __init__(self, emb_dim: int, attention_dim: int, n_heads: int = 8, dropout: float = 0.0, rope=None,
                 flash_attention: bool = False):
        super().__init__()
        self.n_heads = n_heads
        self.dropout = dropout
        self.rope = rope
        self.qkv = nn.Linear(emb_dim, attention_dim * 3, bias=False)
        self.aggregate_heads = nn.Sequential(nn.Linear(attention_dim, emb_dim, bias=False), nn.Dropout(dropout))
        self.flash_attention = flash_attention


class LocoformerBlock(nn.Module):
    """models/mss_tflocoformer.py:356-464."""

    def __init__(self, rope, emb_dim: int = 128, norm_type: str = "rmsgroupnorm", num_groups: int = 4, n_heads: int = 4,
                 flash_attention: bool = False, attention_dim: int = 128, ffn_type: Union[str, list] = "swiglu_conv1d",
                 ffn_hidden_dim: Union[int, list] = 384, conv1d_kernel: int = 4, conv1d_shift: int = 1,
                 dropout: float = 0.0, eps: float = 1.0e-5):
        super().__init__()
        FFN = {"conv1d": ConvDeconv1d, "swiglu_conv1d": SwiGLUConvDeconv1d}
        Norm = {"layernorm": nn.LayerNorm, "rmsgroupnorm": RMSGroupNorm}
        assert norm_type in Norm, norm_type
        if norm_type != "rmsgroupnorm":
            raise NotImplementedError("norm_type='layernorm' is not supported (unused by every reference config/test)")
        self.macaron_style = isinstance(ffn_type, list) and len(ffn_type) == 2
        if self.macaron_style:
            assert isinstance(ffn_hidden_dim, list) and len(ffn_hidden_dim) == 2
            ffn_type_list = ffn_type[::-1]
            ffn_dim_list = ffn_hidden_dim[::-1]
        else:
            ffn_type_list = [ffn_type]
            ffn_dim_list = [ffn_hidden_dim]
        self.ffn_norm = nn.ModuleList([])
        self.ffn = nn.ModuleList([])
        for f_type, f_dim in zip(ffn_type_list, ffn_dim_list):
            assert f_type in FFN, f_type
            self.ffn_norm.append(RMSGroupNorm(num_groups, emb_dim, eps=eps))
            self.ffn.append(FFN[f_type](emb_dim, f_dim, conv1d_kernel, conv1d_shift, dropout=dropout))
        self.attn_norm = RMSGroupNorm(num_groups, emb_dim, eps=eps)
        self.attn = MultiHeadSelfAttention(emb_dim, attention_dim=attention_dim, n_heads=n_heads, rope=rope,
                                           dropout=dropout, flash_attention=flash_attention)
        self._site = None  # (owner weakref, layer, axis)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [B, S1, S2, C] -> same, sequences along S2 (:430-464).  freq_path: S2 = F; frame_path: S2 = Tf."""
        if self._site is None:
            raise RuntimeError("LocoformerBlock must belong to a separator model to run")
        owner, layer, axis = self._site
        model = owner()
        _forward_only(model, x)
        eng, prec = model._ready(), _resolve_precision(model)
        # channels-last canonical buffer [B, Tf, F, C]; the time path sees it as [B, F, Tf, C] (:342)
        xc = x.to(torch.float32)
        xc = (xc.transpose(1, 2) if axis == 1 else xc).contiguous().clone()
        if self.macaron_style:
            eng.ffn_(layer, axis, 1, xc, prec)
        eng.attn_(layer, axis, xc, prec)
        eng.ffn_(layer, axis, 0, xc, prec)
        return xc.transpose(1, 2) if axis == 1 else xc


class TFLocoformerBlock(nn.Module):
    """models/mss_tflocoformer.py:261-353."""

    def __init__(self, rope_freq, rope_time, emb_dim: int = 128, norm_type: str = "rmsgroupnorm", num_groups: int = 4,
                 tf_order: str = "ft", n_heads: int = 4, flash_attention: bool = False, attention_dim: int = 128,
                 ffn_type: Union[str, list] = "swiglu_conv1d", ffn_hidden_dim: Union[int, list] = 384,
                 conv1d_kernel: int = 4, conv1d_shift: int = 1, dropout: float = 0.0, eps: float = 1.0e-5):
        super().__init__()
        assert tf_order in ["tf", "ft"], tf_order
        self.tf_order = tf_order
        self.conv1d_kernel = conv1d_kernel
        self.conv1d_shift = conv1d_shift
        kw = dict(emb_dim=emb_dim, norm_type=norm_type, num_groups=num_groups, n_heads=n_heads,
                  flash_attention=flash_attention, attention_dim=attention_dim, ffn_type=ffn_type,
                  ffn_hidden_dim=ffn_hidden_dim, conv1d_kernel=conv1d_kernel, conv1d_shift=conv1d_shift,
                  dropout=dropout, eps=eps)
        self.freq_path = LocoformerBlock(rope_freq, **kw)
        self.frame_path = LocoformerBlock(rope_time, **kw)

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        """input [B, C, T, F] -> [B, C, T, F] (:323-353)."""
        x = input.movedim(1, -1)  # [B, T, F, C]
        if self.tf_order == "ft":
            x = self.freq_path(x)
            x = self.frame_path(x.transpose(1, 2)).transpose(1, 2)
        else:
            x = self.frame_path(x.transpose(1, 2)).transpose(1, 2)
            x = self.freq_path(x)
        return x.movedim(-1, 1)
