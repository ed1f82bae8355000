"""Top-level separators with the reference's constructors, forward signatures and state_dict keys."""
import weakref
from typing import Dict, Optional, Union

import torch
import torch.nn as nn

from .engine import Engine
from .autograd import BSFunction, MSSFunction, SeparatorFunction, bs_band_params, wants_autograd
from .engine import _require_cuda
from .modules import (MSSTransform, RotaryEmbedding, TFLocoformerBlock, SOURCE_NAMES, _forward_only,
                      _no_training_dropout, _resolve_precision)


class _SeparatorBase(nn.Module):
    """Shared plumbing: engine creation, lazy weight packing, sub-module call sites."""

    precision: Optional[str] = None  # None = follow torch.autocast (bf16) else fp32; or "fp32" / "bf16"
    # True: in training mode with grad enabled, forward builds an autograd graph over the parameters and, for
    # TFLocoformerMSS and TFLocoformerSeparator, the input (autograd.py).  training.Trainer does not need it.
    differentiable: bool = False

    def _init_engine_cfg(self, **cfg):
        self._engine_cfg = cfg
        self._engine: Optional[Engine] = None
        self._dropout_p = float(cfg.pop("dropout"))

    def _attach_sites(self):
        ref = weakref.ref(self)
        for i, blk in enumerate(self.blocks):
            for axis, path in enumerate((blk.freq_path, blk.frame_path)):
                path._site = (ref, i, axis)
                for j, norm in enumerate(path.ffn_norm):
                    norm._site = (ref, i, axis, j)
                path.attn_norm._site = (ref, i, axis, 2)

    def _ready(self) -> Engine:
        if self._engine is None:
            self._engine = Engine(self._engine_cfg)
        refs = getattr(self, "_param_refs", None)
        if refs is None:            # parameter objects by state_dict key, collected once (not once per forward)
            refs = dict(self.state_dict(keep_vars=True))
            self._param_refs = refs
        self._engine.ensure_packed(refs)
        return self._engine

    def repack(self):
        """Re-read the parameters into the packed weight image at the next forward.

        The image is refreshed automatically when a parameter's storage or version counter changes (``load_state_dict``,
        ``.to()``, optimiser steps); call this after writes that bypass the version counter (``p.data.copy_(ema)``) or
        after replacing a parameter object."""
        self._param_refs = None
        if self._engine is not None:
            self._engine.invalidate()

    def _build_blocks(self, n_layers, rope_freq, rope_time, **kw):
        self.blocks = nn.ModuleList([])
        for _ in range(n_layers):
            self.blocks.append(TFLocoformerBlock(rope_freq, rope_time, **kw))


def _engine_cfg(n_fft, hop, n_src, n_layers, emb_dim, num_groups, tf_order, n_heads, attention_dim, pos_enc, ffn_type,
                ffn_hidden_dim, conv1d_kernel, dropout, eps, enc_in_ch):
    macaron = isinstance(ffn_type, list) and len(ffn_type) == 2
    if macaron:
        hid0, hid1 = ffn_hidden_dim[1], ffn_hidden_dim[0]  # lists are stored reversed (:391-392)
    else:
        hid0, hid1 = (ffn_hidden_dim[0] if isinstance(ffn_hidden_dim, list) else ffn_hidden_dim), 0
    return dict(n_fft=n_fft, hop=hop, n_src=n_src, n_layers=n_layers, emb_dim=emb_dim, num_groups=num_groups,
                tf_order=0 if tf_order == "ft" else 1, n_heads=n_heads, attention_dim=attention_dim,
                rope=1 if pos_enc == "rope" else 0, macaron=int(macaron), ffn_hidden0=int(hid0), ffn_hidden1=int(hid1),
                conv_kernel=conv1d_kernel, enc_in_ch=enc_in_ch, eps=float(eps), dropout=dropout)


class TFLocoformerMSS(_SeparatorBase):
    """TF-Locoformer for music source separation -- models/mss_tflocoformer.py:78-258.

    ``forward(mixture[B, T], return_time_domain=True) -> {'vocals','drums','bass','other'}[:n_sources]``.
    """

    def __init__(self, n_fft: int = 2048, hop_length: int = 1024, n_sources: int = 4, n_layers: int = 6,
                 emb_dim: int = 128, norm_type: str = "rmsgroupnorm", num_groups: int = 4, tf_order: str = "ft",
                 n_heads: int = 4, flash_attention: bool = False, attention_dim: int = 128, pos_enc: str = "rope",
                 ffn_type: Union[str, list] = "swiglu_conv1d", ffn_hidden_dim: Union[int, list] = 384,
                 conv1d_kernel: int = 4, conv1d_shift: int = 1, dropout: float = 0.0, eps: float = 1.0e-5):
        super().__init__()
        self.n_fft = n_fft
        self.hop_length = hop_length
        self.n_sources = n_sources
        self.n_layers = n_layers
        self.transform = MSSTransform(n_fft=n_fft, hop_length=hop_length)
        t_ksize = 3
        ks, padding = (t_ksize, 3), (t_ksize // 2, 1)
        self.conv = nn.Sequential(nn.Conv2d(2, emb_dim, ks, padding=padding), nn.GroupNorm(1, emb_dim, eps=eps))
        assert attention_dim % n_heads == 0, (attention_dim, n_heads)
        if pos_enc == "nope":
            rope_freq = rope_time = None
        elif pos_enc == "rope":
            rope_freq = RotaryEmbedding(attention_dim // n_heads)
            rope_time = RotaryEmbedding(attention_dim // n_heads)
        else:
            raise ValueError(f"Unsupported positional encoding: {pos_enc}")
        self._build_blocks(n_layers, rope_freq, rope_time, emb_dim=emb_dim, norm_type=norm_type, num_groups=num_groups,
                           tf_order=tf_order, n_heads=n_heads, flash_attention=flash_attention,
                           attention_dim=attention_dim, ffn_type=ffn_type, ffn_hidden_dim=ffn_hidden_dim,
                           conv1d_kernel=conv1d_kernel, conv1d_shift=conv1d_shift, dropout=dropout, eps=eps)
        self.deconv = nn.ConvTranspose2d(emb_dim, n_sources * 2, ks, padding=padding)
        self._init_engine_cfg(**_engine_cfg(n_fft, hop_length, n_sources, n_layers, emb_dim, num_groups, tf_order,
                                            n_heads, attention_dim, pos_enc, ffn_type, ffn_hidden_dim, conv1d_kernel,
                                            dropout, eps, enc_in_ch=2))
        self.transform._owner = weakref.ref(self)
        self._attach_sites()

    def forward(self, mixture: torch.Tensor, return_time_domain: bool = True) -> Dict[str, torch.Tensor]:
        _no_training_dropout(self)
        if wants_autograd(self, list(self.parameters()), mixture):
            _require_cuda(mixture, "mixture")
            eng = self._ready()
            eng.check_mixture(mixture)
            out = MSSFunction.apply(self, mixture.to(torch.float32).contiguous(), return_time_domain,
                                    *[self._param_refs[k] for k in eng.keys])
            audio, spec = (out, None) if return_time_domain else (None, out)
        else:
            _forward_only(self, mixture)
            eng, prec = self._ready(), _resolve_precision(self)
            audio, spec = eng.mss_forward(mixture, prec, want_audio=return_time_domain, want_spec=not return_time_domain)
        if return_time_domain:
            return {name: audio[i] for i, name in enumerate(SOURCE_NAMES[: self.n_sources])}
        est = torch.view_as_complex(spec)  # [B, S, Tf, F]
        # the reference hard-codes four names here (:253-258) and raises IndexError for n_sources < 4
        return {name: est[:, i].transpose(-1, -2) for i, name in enumerate(SOURCE_NAMES)}


class TFLocoformerSeparator(_SeparatorBase):
    """standalone/tflocoformer_separator.py:17-171.  complex [B, T, F] (or [B, 1, T, F]) -> [B, num_spk, T, F]."""

    def __init__(self, num_spk: int = 2, n_layers: int = 6, emb_dim: int = 128, norm_type: str = "rmsgrouporm",
                 num_groups: int = 4, tf_order: str = "ft", n_heads: int = 4, flash_attention: bool = False,
                 attention_dim: int = 128, pos_enc: str = "rope", ffn_type: Union[str, list] = "swiglu_conv1d",
                 ffn_hidden_dim: Union[int, list] = 384, conv1d_kernel: int = 4, conv1d_shift: int = 1,
                 dropout: float = 0.0, eps: float = 1.0e-5):
        super().__init__()
        self.num_spk = num_spk
        self.n_layers = n_layers
        t_ksize = 3
        ks, padding = (t_ksize, 3), (t_ksize // 2, 1)
        self.conv = nn.Sequential(nn.Conv2d(2, emb_dim, ks, padding=padding), nn.GroupNorm(1, emb_dim, eps=eps))
        assert attention_dim % n_heads == 0, (attention_dim, n_heads)
        if pos_enc == "nope":
            pe_freq = pe_time = None
        elif pos_enc == "rope":
            pe_freq = RotaryEmbedding(attention_dim // n_heads)
            pe_time = RotaryEmbedding(attention_dim // n_heads)
        else:
            raise ValueError(f"Unsupported positional encoding: {pos_enc}")
        self._build_blocks(n_layers, pe_freq, pe_time, emb_dim=emb_dim, norm_type=norm_type, num_groups=num_groups,
                           tf_order=tf_order, n_heads=n_heads, flash_attention=flash_attention,
                           attention_dim=attention_dim, ffn_type=ffn_type, ffn_hidden_dim=ffn_hidden_dim,
                           conv1d_kernel=conv1d_kernel, conv1d_shift=conv1d_shift, dropout=dropout, eps=eps)
        self.deconv = nn.ConvTranspose2d(emb_dim, num_spk * 2, ks, padding=padding)
        self._init_engine_cfg(**_engine_cfg(0, 0, num_spk, n_layers, emb_dim, num_groups, tf_order, n_heads,
                                            attention_dim, pos_enc, ffn_type, ffn_hidden_dim, conv1d_kernel, dropout,
                                            eps, enc_in_ch=2))
        self._attach_sites()

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        _no_training_dropout(self)
        grad = wants_autograd(self, list(self.parameters()), input)
        if not grad:
            _forward_only(self, input)
        if input.ndim == 4:
            assert input.shape[1] == 1, "Only monaural input is supported."
            input = input[:, 0]
        if not input.is_complex() or input.ndim != 3:
            raise ValueError("input must be a complex spectrogram [B, T, F] or [B, 1, T, F]")
        if grad:
            _require_cuda(input, "input")
            eng = self._ready()
            # not detached: autograd carries d spec back through view_as_real (torch's complex-gradient convention)
            ri = torch.view_as_real(input.to(torch.complex64).contiguous())
            return torch.view_as_complex(SeparatorFunction.apply(self, ri, *[self._param_refs[k] for k in eng.keys]))
        eng, prec = self._ready(), _resolve_precision(self)
        ri = torch.view_as_real(input.to(torch.complex64).contiguous())
        return torch.view_as_complex(eng.separator_forward(ri, prec))


def strip_prefix(state_dict: Dict[str, torch.Tensor], prefix: str = "separator.") -> Dict[str, torch.Tensor]:
    """ESPnet checkpoints carry a ``separator.`` prefix (tests/test_tflocoformer_load_pretrained_weights.py:68-73)."""
    return {k[len(prefix):]: v for k, v in state_dict.items() if k.startswith(prefix)}


# same configuration as BS-Roformer (standalone/bslocoformer_separator.py:20): (frequency range): bins per band
BAND_SPLIT = {(0, 1000): 2, (1000, 2000): 4, (2000, 4000): 12, (4000, 8000): 24, (8000, 16000): 48}


class BandSplitModule(nn.Module):
    """Parameter container with the reference's layout (standalone/bslocoformer_separator.py:186-239); the
    band-split / band-wise decoding arithmetic runs in csrc/kernels_bs.cuh."""

    def __init__(self, num_src: int, emb_dim: int, stft_size: int, sample_rate: int, stereo: bool = False):
        super().__init__()
        import math
        from itertools import accumulate
        self.num_src = num_src
        num_freq_bins = stft_size // 2 + 1
        self.bands = []
        freq_each_bin = sample_rate // 2 / num_freq_bins
        for freq_range, num_bins in BAND_SPLIT.items():
            start, end = freq_range
            num_band = math.ceil((end - start) / (num_bins * freq_each_bin))
            self.bands.extend([num_bins] * num_band)
        rest = num_freq_bins - sum(self.bands)
        if sample_rate == 48000:
            self.bands.extend([rest // 4, rest // 4, rest // 4, rest // 4 + rest % 4])
        else:
            self.bands.extend([math.floor(rest / 2), math.ceil(rest / 2)])
        assert sum(self.bands) == num_freq_bins, (sum(self.bands), num_freq_bins, self.bands)
        print(f"Band-split module has {len(self.bands)} bands", flush=True)
        self.stereo = stereo
        coef = 4 if self.stereo else 2
        self.band_split_module = nn.ModuleList([])
        for band in self.bands:
            self.band_split_module.append(nn.Sequential(nn.GroupNorm(1, band * coef),
                                                        nn.Conv1d(band * coef, emb_dim, kernel_size=1)))
        self.bandwise_decoding_module = nn.ModuleList([])
        for band in self.bands:
            self.bandwise_decoding_module.append(nn.Sequential(
                nn.GroupNorm(1, emb_dim), nn.Conv1d(emb_dim, emb_dim * 4, kernel_size=1), nn.Tanh(),
                nn.Conv1d(emb_dim * 4, emb_dim * 4, kernel_size=1),
                nn.Conv1d(emb_dim * 4, band * num_src * coef * 2, kernel_size=1), nn.GLU(dim=1)))
        self.band_idx = list(accumulate([0] + self.bands))


class BSLocoformerSeparator(_SeparatorBase):
    """BS-Locoformer -- standalone/bslocoformer_separator.py:23-183.  complex [B, (M), T, F] -> [B, num_spk, (M), T, F]."""

    def __init__(self, num_spk: int = 2, n_layers: int = 6, emb_dim: int = 128, norm_type: str = "rmsgrouporm",
                 num_groups: int = 4, tf_order: str = "ft", n_heads: int = 4, flash_attention: bool = False,
                 attention_dim: int = 128, pos_enc: str = "rope", ffn_type: Union[str, list] = "swiglu_conv1d",
                 ffn_hidden_dim: Union[int, list] = 384, conv1d_kernel: int = 4, conv1d_shift: int = 1,
                 dropout: float = 0.0, sample_rate: int = 44100, stft_size: int = 2048, eps: float = 1.0e-5,
                 masking: bool = True, stereo: bool = False):
        super().__init__()
        self.num_spk = num_spk
        self.n_layers = n_layers
        assert attention_dim % n_heads == 0, (attention_dim, n_heads)
        if pos_enc == "nope":
            pe_freq = pe_time = None
        elif pos_enc == "rope":
            pe_freq = RotaryEmbedding(attention_dim // n_heads)
            pe_time = RotaryEmbedding(attention_dim // n_heads)
        else:
            raise ValueError(f"Unsupported positional encoding: {pos_enc}")
        self._build_blocks(n_layers, pe_freq, pe_time, emb_dim=emb_dim, norm_type=norm_type, num_groups=num_groups,
                           tf_order=tf_order, n_heads=n_heads, flash_attention=flash_attention,
                           attention_dim=attention_dim, ffn_type=ffn_type, ffn_hidden_dim=ffn_hidden_dim,
                           conv1d_kernel=conv1d_kernel, conv1d_shift=conv1d_shift, dropout=dropout, eps=eps)
        self.band_split_module = BandSplitModule(num_spk, emb_dim, stft_size, sample_rate, stereo=stereo)
        self.masking = masking
        self.stereo = stereo
        self.emb_dim = emb_dim
        self._init_engine_cfg(**_engine_cfg(0, 0, num_spk, n_layers, emb_dim, num_groups, tf_order, n_heads,
                                            attention_dim, pos_enc, ffn_type, ffn_hidden_dim, conv1d_kernel, dropout,
                                            eps, enc_in_ch=0))
        self._attach_sites()
        self._bs_pack = None

    def _bs_packed(self, device):
        """One fp32 weight buffer + int64 index table for tfl_bs_band_split / tfl_bs_band_decode (layout: include/tfl.h)."""
        bsm = self.band_split_module
        tensors = [p for p in bsm.parameters()]
        fp = tuple((t.data_ptr(), t._version) for t in tensors)
        if self._bs_pack is not None and self._bs_pack[0] == fp:
            return self._bs_pack[1], self._bs_pack[2]
        chunks, table, off, where = [], [], 0, {}

        def add(t, src=None):
            nonlocal off
            flat = t.detach().to(device=device, dtype=torch.float32).reshape(-1)
            chunks.append(flat)
            start = off
            off += flat.numel()
            where[id(t if src is None else src)] = (start, src is not None)
            return start

        for b, width in enumerate(bsm.bands):
            sp, de = bsm.band_split_module[b], bsm.bandwise_decoding_module[b]
            row = [bsm.band_idx[b], width,
                   add(sp[0].weight), add(sp[0].bias), add(sp[1].weight[:, :, 0].t().contiguous(), sp[1].weight),
                   add(sp[1].bias), add(de[0].weight), add(de[0].bias),
                   add(de[1].weight[:, :, 0].t().contiguous(), de[1].weight), add(de[1].bias),
                   add(de[3].weight[:, :, 0].t().contiguous(), de[3].weight), add(de[3].bias),
                   add(de[4].weight[:, :, 0].t().contiguous(), de[4].weight), add(de[4].bias), 0, 0]
            table.append(row)
        wbuf = torch.cat(chunks)
        tab = torch.tensor(table, dtype=torch.int64, device=device)
        # per parameter (bs_band_params order): (offset in wbuf, stored transposed) -- where its gradient lands
        self._bs_pack = (fp, wbuf, tab, [where[id(t)] for t in tensors])
        return wbuf, tab

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        from .engine import _stream
        from ._lib import check
        _forward_only(self, input)
        if input.ndim == 3:
            assert not self.stereo
            spec = input.unsqueeze(1)
        else:
            spec = input
        if not spec.is_complex() or spec.ndim != 4:
            raise ValueError("input must be a complex spectrogram [B, T, F] or [B, M, T, F]")
        _require_cuda(spec, "input")
        B, M, T, F = spec.shape
        assert M == (2 if self.stereo else 1), (M, self.stereo)
        if wants_autograd(self, list(self.parameters())):
            eng = self._ready()
            ri = torch.view_as_real(spec.detach().to(torch.complex64).contiguous())
            params = [self._param_refs[k] for k in eng.keys] + bs_band_params(self)
            out = torch.view_as_complex(BSFunction.apply(self, ri, *params))    # [B, S, M, T, F]
            return out if self.stereo else out[:, :, 0]
        eng, prec = self._ready(), _resolve_precision(self)
        bsm = self.band_split_module
        nb, C, S = len(bsm.bands), self.emb_dim, self.num_spk
        ri = torch.view_as_real(spec.to(torch.complex64).contiguous())            # [B, M, T, F, 2]
        wbuf, tab = self._bs_packed(spec.device)
        x = torch.empty((B, T, nb, C), dtype=torch.float32, device=spec.device)
        est = torch.empty((B, S, M, T, F, 2), dtype=torch.float32, device=spec.device)
        lib = eng.lib
        with torch.cuda.device(spec.device):
            check(lib.tfl_bs_band_split(ri.data_ptr(), B, M, T, F, C, nb, max(bsm.bands), tab.data_ptr(), wbuf.data_ptr(),
                                        x.data_ptr(), _stream()))
        eng.blocks(x, prec)                                                       # frames = T, "bins" = bands
        with torch.cuda.device(spec.device):
            check(lib.tfl_bs_band_decode(x.data_ptr(), ri.data_ptr(), B, M, T, F, C, nb, S, tab.data_ptr(), wbuf.data_ptr(),
                                         est.data_ptr(), 1 if self.masking else 0, _stream()))
        out = torch.view_as_complex(est)                                          # [B, S, M, T, F]
        return out if self.stereo else out[:, :, 0]
