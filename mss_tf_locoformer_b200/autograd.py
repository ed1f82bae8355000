"""Training of the models through torch autograd (DESIGN.md section 8b).

``TFLocoformerMSS``, ``TFLocoformerSeparator`` (and its ESPnet adapter) and ``BSLocoformerSeparator`` run their forward
as a ``torch.autograd.Function`` when the model is built or set with ``differentiable = True``, is in training mode, grad
is enabled and some parameter requires grad (for ``TFLocoformerMSS`` and ``TFLocoformerSeparator``: or the input does).
The forward keeps its activations in a workspace of its own (one per call, so two forwards before one backward do not
share saved state); the backward is CUDA (include/tfl.h: ``tfl_mss_train_backward``, ``tfl_sep_train_backward[_input]``,
``tfl_blocks_train_backward``, ``tfl_bs_band_decode_bwd``, ``tfl_bs_band_split_bwd``) and returns every parameter's
gradient in the reference's tensor layout, so any torch loss, optimiser, gradient clipping or DDP wrapper drives the
model as it would the reference.

Arithmetic follows ``TFL_OPT_TRAIN_MODE`` exactly as the MSS training step (``training.Trainer``) does: fp32, tf32, or
(the default) mixed -- the sub-block forward on the bf16 tcgen05 kernels, encoder / decoder and backward on tf32.  The
model's ``precision`` attribute selects the inference arithmetic only.  ``TFLocoformerMSS`` returns a gradient for the
mixture and ``TFLocoformerSeparator`` one for its complex input spectrogram; ``BSLocoformerSeparator`` refuses an input
that requires grad, as the inference path does.

Under ``torch.use_deterministic_algorithms(True)``, as read at the forward and recorded for its backward, every
reduction of the backward pass runs in a fixed order (``TFL_OPT_DETERMINISTIC``): two identical forward + backward
passes return bitwise-identical gradients.
"""
import ctypes as C
from typing import List

import torch
from torch.autograd.function import once_differentiable

from ._lib import check, deterministic_option
from .engine import _stream


def wants_autograd(model, params: List[torch.Tensor], *inputs: torch.Tensor) -> bool:
    """True when ``model``'s forward must build a graph: opted in, training mode, grad enabled, and a parameter or one of
    ``inputs`` requires grad."""
    return (bool(getattr(model, "differentiable", False)) and model.training and torch.is_grad_enabled()
            and any(t.requires_grad for t in list(params) + list(inputs)))


def _grad_layout(eng):
    """(offsets, sizes, total) of the flat gradient buffer (tfl_train_grad_layout), cached on the engine."""
    lay = getattr(eng, "_grad_layout", None)
    if lay is None:
        n = len(eng.keys)
        offs, sizes = (C.c_int64 * n)(), (C.c_int64 * n)()
        total = eng.lib.tfl_train_grad_layout(eng.plan, offs, sizes, n)
        if total < 0:
            check(-1)
        lay = (list(offs), list(sizes), int(total))
        eng._grad_layout = lay
    return lay


def _weights_array(params):
    return (C.c_void_p * len(params))(*[p.data_ptr() for p in params])


def _raw(params):
    """The fp32 contiguous device tensors the data-gradient GEMMs read in place (views of the parameters)."""
    out = []
    for p in params:
        if p.dtype != torch.float32 or not p.is_contiguous():
            raise RuntimeError("differentiable separators need float32 contiguous parameters")
        out.append(p.detach())
    return out


def _unflatten(eng, grads: torch.Tensor, params, needs=None) -> List:
    """Per-parameter views of the flat buffer; None where the tensor is not trainable or (``needs``) wants no gradient."""
    offs, sizes, _ = _grad_layout(eng)
    needs = [True] * len(params) if needs is None else needs
    return [None if o < 0 or not w else grads[o:o + n].view(p.shape) for p, o, n, w in zip(params, offs, sizes, needs)]


class MSSFunction(torch.autograd.Function):
    """mixture [B, T] -> audio [S, B, T] (``want_audio``) or est [B, S, Tf, F, 2] of a TFLocoformerMSS; differentiable in
    the parameters and the mixture."""

    @staticmethod
    def forward(ctx, model, mixture, want_audio, *params):
        eng = model._engine
        lib = eng.lib
        B, T = mixture.shape
        S, n_fft, hop = eng.cfg["n_src"], eng.cfg["n_fft"], eng.cfg["hop"]
        dev = mixture.device
        det = torch.are_deterministic_algorithms_enabled()
        shape = (S, B, T) if want_audio else (B, S, 1 + T // hop, n_fft // 2 + 1, 2)
        out = torch.empty(shape, dtype=torch.float32, device=dev)
        packed = eng.packed
        with deterministic_option(det), torch.cuda.device(dev):
            ws = torch.empty(max(256, lib.tfl_mss_train_workspace_bytes(eng.plan, B, T)), dtype=torch.uint8, device=dev)
            check(lib.tfl_mss_train_forward(eng.plan, packed.data_ptr(), mixture.data_ptr(), B, T,
                                            out.data_ptr() if want_audio else None,
                                            None if want_audio else out.data_ptr(), ws.data_ptr(), ws.numel(),
                                            _stream()))
        ctx.eng, ctx.want_audio, ctx.shape, ctx.deterministic = eng, want_audio, (B, T), det
        ctx.save_for_backward(packed, ws, *params)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_out):
        eng = ctx.eng
        packed, ws, *params = ctx.saved_tensors
        raw = _raw(params)
        B, T = ctx.shape
        dev = ws.device
        grads = torch.empty(_grad_layout(eng)[2], dtype=torch.float32, device=dev)
        d_out = d_out.to(torch.float32).contiguous()
        d_mix = torch.empty((B, T), dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        with deterministic_option(ctx.deterministic), torch.cuda.device(dev):
            check(eng.lib.tfl_mss_train_backward(eng.plan, packed.data_ptr(), _weights_array(raw), len(raw),
                                                 d_out.data_ptr() if ctx.want_audio else None,
                                                 None if ctx.want_audio else d_out.data_ptr(), B, T, grads.data_ptr(),
                                                 None if d_mix is None else d_mix.data_ptr(), ws.data_ptr(), ws.numel(),
                                                 _stream()))
        return (None, d_mix, None, *_unflatten(eng, grads, params, ctx.needs_input_grad[3:]))


class SeparatorFunction(torch.autograd.Function):
    """spec [B, Tf, F, 2] -> est [B, S, Tf, F, 2] of a TFLocoformerSeparator; differentiable in the parameters and spec."""

    @staticmethod
    def forward(ctx, model, spec_ri, *params):
        eng = model._engine
        lib = eng.lib
        B, Tf, F, _ = spec_ri.shape
        dev = spec_ri.device
        det = torch.are_deterministic_algorithms_enabled()
        est = torch.empty((B, eng.cfg["n_src"], Tf, F, 2), dtype=torch.float32, device=dev)
        packed = eng.packed
        with deterministic_option(det), torch.cuda.device(dev):
            ws = torch.empty(max(256, lib.tfl_sep_train_workspace_bytes(eng.plan, B, Tf, F)), dtype=torch.uint8, device=dev)
            check(lib.tfl_sep_train_forward(eng.plan, packed.data_ptr(), spec_ri.data_ptr(), B, Tf, F, est.data_ptr(),
                                            ws.data_ptr(), ws.numel(), _stream()))
        ctx.eng, ctx.deterministic = eng, det
        ctx.save_for_backward(spec_ri, packed, ws, *params)
        return est

    @staticmethod
    @once_differentiable
    def backward(ctx, d_est):
        eng = ctx.eng
        spec_ri, packed, ws, *params = ctx.saved_tensors
        raw = _raw(params)
        B, Tf, F, _ = spec_ri.shape
        grads = torch.empty(_grad_layout(eng)[2], dtype=torch.float32, device=spec_ri.device)
        d_est = d_est.to(torch.float32).contiguous()
        args = (eng.plan, packed.data_ptr(), _weights_array(raw), len(raw), d_est.data_ptr(), spec_ri.data_ptr(), B, Tf, F,
                grads.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
        d_spec = torch.empty_like(spec_ri) if ctx.needs_input_grad[1] else None
        with deterministic_option(ctx.deterministic), torch.cuda.device(spec_ri.device):
            if d_spec is None:
                check(eng.lib.tfl_sep_train_backward(*args))
            else:
                check(eng.lib.tfl_sep_train_backward_input(*args, d_spec.data_ptr()))
        return (None, d_spec, *_unflatten(eng, grads, params, ctx.needs_input_grad[2:]))


def bs_band_params(model) -> List[torch.Tensor]:
    """The band-split module's parameters, in ``BandSplitModule.parameters()`` order (the order ``_bs_packed`` reads)."""
    return list(model.band_split_module.parameters())


class BSFunction(torch.autograd.Function):
    """spec [B, M, T, F, 2] -> est [B, S, M, T, F, 2] of a BSLocoformerSeparator; differentiable in the parameters.
    ``params`` = the Locoformer block parameters (engine key order), then ``bs_band_params(model)``."""

    @staticmethod
    def forward(ctx, model, ri, *params):
        eng = model._engine
        lib = eng.lib
        bsm = model.band_split_module
        B, M, T, F, _ = ri.shape
        nb, Cd, S, wmax = len(bsm.bands), model.emb_dim, model.num_spk, max(bsm.bands)
        dev = ri.device
        wbuf, tab = model._bs_packed(dev)
        packed = eng.packed
        det = torch.are_deterministic_algorithms_enabled()
        x0 = torch.empty((B, T, nb, Cd), dtype=torch.float32, device=dev)
        x1 = torch.empty_like(x0)
        est = torch.empty((B, S, M, T, F, 2), dtype=torch.float32, device=dev)
        with deterministic_option(det), torch.cuda.device(dev):
            ws = torch.empty(max(256, lib.tfl_sep_train_workspace_bytes(eng.plan, B, T, nb)), dtype=torch.uint8, device=dev)
            check(lib.tfl_bs_band_split(ri.data_ptr(), B, M, T, F, Cd, nb, wmax, tab.data_ptr(), wbuf.data_ptr(),
                                        x0.data_ptr(), _stream()))
            check(lib.tfl_blocks_train_forward(eng.plan, packed.data_ptr(), x0.data_ptr(), B, T, nb, x1.data_ptr(),
                                               ws.data_ptr(), ws.numel(), _stream()))
            check(lib.tfl_bs_band_decode(x1.data_ptr(), ri.data_ptr(), B, M, T, F, Cd, nb, S, tab.data_ptr(),
                                         wbuf.data_ptr(), est.data_ptr(), 1 if model.masking else 0, _stream()))
        del x0
        ctx.eng, ctx.model_cfg, ctx.deterministic = eng, (nb, Cd, S, wmax, bool(model.masking), len(eng.keys)), det
        ctx.band_map = model._bs_pack[3]
        ctx.save_for_backward(ri, packed, wbuf, tab, ws, x1, *params)
        return est

    @staticmethod
    @once_differentiable
    def backward(ctx, d_est):
        eng = ctx.eng
        lib = eng.lib
        ri, packed, wbuf, tab, ws, x1, *params = ctx.saved_tensors
        nb, Cd, S, wmax, masking, n_blk = ctx.model_cfg
        B, M, T, F, _ = ri.shape
        dev = ri.device
        d_est = d_est.to(torch.float32).contiguous()
        dx1 = torch.empty_like(x1)
        dx0 = torch.empty_like(x1)
        gw = torch.empty_like(wbuf)
        grads = torch.empty(_grad_layout(eng)[2], dtype=torch.float32, device=dev)
        blk_params = params[:n_blk]
        raw = _raw(blk_params)
        n_bws = lib.tfl_bs_band_bwd_workspace_bytes(B, M, T, F, Cd, nb, S, wmax)
        bws = torch.empty(max(256, n_bws), dtype=torch.uint8, device=dev)
        with deterministic_option(ctx.deterministic), torch.cuda.device(dev):
            check(lib.tfl_bs_band_decode_bwd(x1.data_ptr(), ri.data_ptr(), d_est.data_ptr(), B, M, T, F, Cd, nb, S, wmax,
                                             tab.data_ptr(), wbuf.data_ptr(), 1 if masking else 0, dx1.data_ptr(),
                                             gw.data_ptr(), bws.data_ptr(), bws.numel(), _stream()))
            check(lib.tfl_blocks_train_backward(eng.plan, packed.data_ptr(), _weights_array(raw), len(raw),
                                                dx1.data_ptr(), B, T, nb, dx0.data_ptr(), grads.data_ptr(), ws.data_ptr(),
                                                ws.numel(), _stream()))
            check(lib.tfl_bs_band_split_bwd(ri.data_ptr(), dx0.data_ptr(), B, M, T, F, Cd, nb, wmax, tab.data_ptr(),
                                            wbuf.data_ptr(), gw.data_ptr(), bws.data_ptr(), bws.numel(), _stream()))
        out = _unflatten(eng, grads, blk_params)
        for p, (off, transposed) in zip(params[n_blk:], ctx.band_map):
            g = gw[off:off + p.numel()]
            if transposed:                       # stored as W^T [in][out]; the parameter is conv.weight [out, in, 1]
                g = g.view(p.shape[1], p.shape[0]).t().contiguous()
            out.append(g.view(p.shape))
        return (None, None, *out)
