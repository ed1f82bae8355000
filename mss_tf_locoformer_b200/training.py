"""Training step of TFLocoformerMSS on the CUDA kernels of csrc/ (SURVEY.md section 8(f) row N1).

Mirrors /root/reference/training/train.py:68-172 for one process per GPU: forward -> ``MSSLoss`` (``loss_type='combined'``,
/root/reference/models/mss_loss.py:18-109) -> backward -> ``clip_grad_norm_(5.0)`` -> ``AdamW`` (train.py:141-146, :351-357).
Every arithmetic step is a kernel reached through include/tfl.h (``tfl_train_forward_backward``, ``tfl_grad_clip_norm``,
``tfl_adamw_step``); torch holds the buffers and, when ``torch.distributed`` is initialised, all-reduces the ONE flat
gradient buffer (NCCL over NVLink; the reference itself has no multi-GPU training, SURVEY F2).

Arithmetic (``tfl_debug_set_option(TFL_OPT_TRAIN_MODE, m)``): 0 = exact fp32 on CUDA cores (the gradient-parity mode),
1 = tf32 ``mma.sync`` GEMMs, 2 (default) = forward of the sub-blocks on the bf16 tcgen05 inference kernels and bf16 / tf32
``mma.sync`` backward (DESIGN.md section 8b).  Dropout is not applied (parity is defined for p = 0): a model built with
``dropout > 0`` is refused.

Under ``torch.use_deterministic_algorithms(True)`` (read at every ``forward_backward`` / ``step``) the backward pass
reduces in a fixed order (``TFL_OPT_DETERMINISTIC``), so the same step from the same state gives bitwise-identical
gradients, and clipping and AdamW, which are fixed-order already, keep them so.  The all-reduce across ranks is NCCL's.
"""
import ctypes as C
from typing import Dict, Optional, Union

import torch

from . import _lib
from ._lib import TflLossConfig, check, deterministic_option
from .engine import _require_cuda, _stream
from .modules import SOURCE_NAMES


def allreduce_mean_(flat: torch.Tensor) -> torch.Tensor:
    """Average the flat gradient buffer over the ranks in place (one collective; no-op without a process group)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return flat
    if dist.get_backend() == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG)
    else:                                   # gloo (CPU tests) has no AVG
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.div_(dist.get_world_size())
    return flat


class Trainer:
    """One optimiser over one ``TFLocoformerMSS`` on one GPU.

    The model's trainable parameters are re-pointed at slices of one flat fp32 buffer (``self.params``) laid out by
    ``tfl_train_grad_layout``; ``self.grads``, ``self.exp_avg`` and ``self.exp_avg_sq`` share that layout, so
    ``state_dict()`` / checkpoints of the model keep working unchanged while the optimiser is two kernels.
    """

    def __init__(self, model, lr: float = 3e-4, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01,
                 max_grad_norm: float = 5.0, si_sdr_weight: float = 1.0, l1_weight: float = 0.1,
                 spectral_weight: float = 0.1, loss_eps: float = 1e-8, spec_n_fft: int = 2048, spec_hop: int = 1024,
                 gradient_accumulation_steps: int = 1):
        if getattr(model, "_dropout_p", 0.0) > 0.0:
            raise NotImplementedError("training kernels do not apply dropout: construct the model with dropout=0.0")
        self.model = model
        self.lib = _lib.load()
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), tuple(betas), float(eps), float(weight_decay)
        self.max_grad_norm = float(max_grad_norm)
        self.loss_cfg = TflLossConfig(si_sdr_weight, l1_weight, spectral_weight, loss_eps, spec_n_fft, spec_hop)
        self.step_count = 0
        eng = model._ready()
        self.engine = eng
        refs = model._param_refs
        self.tensors = [refs[k] for k in eng.keys]
        dev = self.tensors[0].device
        _require_cuda(self.tensors[0], "model parameters")
        n = len(self.tensors)
        offs, sizes = (C.c_int64 * n)(), (C.c_int64 * n)()
        total = self.lib.tfl_train_grad_layout(eng.plan, offs, sizes, n)
        if total < 0:
            check(-1)
        self.offsets, self.sizes, self.total = list(offs), list(sizes), int(total)
        self.params = torch.zeros(self.total, dtype=torch.float32, device=dev)
        for t, off, size in zip(self.tensors, self.offsets, self.sizes):
            assert t.numel() == size, (tuple(t.shape), size)
            if off < 0:
                continue
            view = self.params[off:off + size].view(t.shape)
            view.copy_(t.detach())
            t.data = view                      # the parameter now lives in the flat buffer
        self.grads = torch.zeros_like(self.params)
        self.exp_avg = torch.zeros_like(self.params)
        self.exp_avg_sq = torch.zeros_like(self.params)
        self.norm = torch.zeros(2, dtype=torch.float32, device=dev)
        self._scratch = torch.zeros(592, dtype=torch.float64, device=dev)
        self._ws: Optional[torch.Tensor] = None
        self._ws_key = None
        self.gradient_accumulation_steps = int(gradient_accumulation_steps)
        self._accum: Optional[torch.Tensor] = None
        self._micro = 0
        model.repack()

    # ---- pieces of a step -----------------------------------------------------------------------------------------
    def _weights_array(self):
        return (C.c_void_p * len(self.tensors))(*[t.data_ptr() for t in self.tensors])

    def forward_backward(self, mixture: torch.Tensor, targets: Union[torch.Tensor, Dict[str, torch.Tensor]],
                         want_audio: bool = False):
        """-> (loss [1 + 3 S] device tensor: total, then (si_sdr, l1, spectral) per source; est audio [S, B, T] or None).
        ``self.grads`` holds d total_loss / d parameters afterwards (local, before any all-reduce)."""
        _require_cuda(mixture, "mixture")
        S = self.engine.cfg["n_src"]
        if isinstance(targets, dict):
            targets = torch.stack([targets[name] for name in SOURCE_NAMES[:S]], 0)
        mixture = mixture.detach().to(torch.float32).contiguous()
        targets = targets.detach().to(torch.float32).contiguous()
        B, T = mixture.shape
        if tuple(targets.shape) != (S, B, T):
            raise ValueError(f"targets must be [{S}, {B}, {T}] (sources, batch, samples), got {tuple(targets.shape)}")
        eng = self.model._ready()
        det = torch.are_deterministic_algorithms_enabled()
        loss = torch.empty(1 + 3 * S, dtype=torch.float32, device=mixture.device)
        audio = torch.empty((S, B, T), dtype=torch.float32, device=mixture.device) if want_audio else None
        with deterministic_option(det), torch.cuda.device(mixture.device):
            key = (B, T, det)
            if self._ws_key != key:
                n = self.lib.tfl_train_workspace_bytes(eng.plan, B, T, self.loss_cfg.spec_n_fft, self.loss_cfg.spec_hop)
                self._ws = None
                self._ws = torch.empty(n, dtype=torch.uint8, device=mixture.device)
                self._ws_key = key
            check(self.lib.tfl_train_forward_backward(
                eng.plan, eng.packed.data_ptr(), self._weights_array(), len(self.tensors), mixture.data_ptr(),
                targets.data_ptr(), B, T, C.byref(self.loss_cfg), self.grads.data_ptr(), loss.data_ptr(),
                None if audio is None else audio.data_ptr(), self._ws.data_ptr(), self._ws.numel(), _stream()))
        return loss, audio

    def optimizer_step(self):
        """clip_grad_norm_(max_grad_norm) + AdamW over the flat buffers; the packed weight image is refreshed lazily."""
        self.step_count += 1
        with torch.cuda.device(self.params.device):
            check(self.lib.tfl_grad_clip_norm(self.grads.data_ptr(), self.total, self.max_grad_norm, self.norm.data_ptr(),
                                              self._scratch.data_ptr(), self._scratch.numel() * 8, _stream()))
            check(self.lib.tfl_adamw_step(self.params.data_ptr(), self.grads.data_ptr(), self.exp_avg.data_ptr(),
                                          self.exp_avg_sq.data_ptr(), self.total, self.norm.data_ptr(), self.lr,
                                          self.betas[0], self.betas[1], self.eps, self.weight_decay, self.step_count,
                                          _stream()))
        self.engine.invalidate()             # the kernels wrote the parameters behind torch's version counters

    def step(self, mixture: torch.Tensor, targets) -> torch.Tensor:
        """One training step (train.py:115-146).  Data parallel: every rank calls it on its own batch.

        With ``gradient_accumulation_steps = N > 1`` (train.py:117-146) the gradients of N consecutive calls are averaged
        (``loss / N``) and the all-reduce + clip + AdamW run on every N-th call only."""
        loss, _ = self.forward_backward(mixture, targets)
        n = self.gradient_accumulation_steps
        if n > 1:
            if self._accum is None:
                self._accum = torch.zeros_like(self.grads)
            with torch.cuda.device(self.params.device):
                check(self.lib.tfl_grad_accumulate(self._accum.data_ptr(), self.grads.data_ptr(), self.total, 1.0 / n,
                                                   1 if self._micro == 0 else 0, _stream()))
            self._micro += 1
            if self._micro < n:
                return loss
            self._micro = 0
            self.grads, self._accum = self._accum, self.grads      # the optimiser reads self.grads
        allreduce_mean_(self.grads)
        self.optimizer_step()
        return loss

    # ---- checkpoint / resume (train.py: `save_optimizer: true`) ----------------------------------------------------
    def state_dict(self) -> dict:
        """Optimiser state per state_dict key, in the reference's tensor shapes (like torch.optim's per-parameter state)."""
        def views(flat):
            return {k: flat[o:o + n].view(t.shape).detach().clone()
                    for k, t, o, n in zip(self.engine.keys, self.tensors, self.offsets, self.sizes) if o >= 0}
        return {"step": self.step_count, "lr": self.lr, "betas": self.betas, "eps": self.eps, "weight_decay": self.weight_decay,
                "exp_avg": views(self.exp_avg), "exp_avg_sq": views(self.exp_avg_sq)}

    def load_state_dict(self, state: dict):
        self.step_count = int(state["step"])
        self.lr, self.betas = float(state["lr"]), tuple(state["betas"])
        self.eps, self.weight_decay = float(state["eps"]), float(state["weight_decay"])
        for name, flat in (("exp_avg", self.exp_avg), ("exp_avg_sq", self.exp_avg_sq)):
            for k, t, o, n in zip(self.engine.keys, self.tensors, self.offsets, self.sizes):
                if o >= 0:
                    flat[o:o + n].view(t.shape).copy_(state[name][k])

    def set_lr(self, lr: float):
        """Learning-rate schedulers (ReduceLROnPlateau, warm-up: train.py:360-371) drive the step size through this."""
        self.lr = float(lr)

    def grad_of(self, key: str) -> torch.Tensor:
        """Gradient of the state_dict tensor ``key`` (a view of the flat buffer, in the reference's layout)."""
        i = self.engine.keys.index(key)
        if self.offsets[i] < 0:
            raise KeyError(f"{key} is not trainable")
        return self.grads[self.offsets[i]:self.offsets[i] + self.sizes[i]].view(self.tensors[i].shape)


# ---- stage-level backward calls (used by the per-kernel parity tests) ------------------------------------------------
def _stage_setup(model, x_in: torch.Tensor):
    lib = _lib.load()
    eng = model._ready()
    tensors = [model._param_refs[k] for k in eng.keys]
    n = len(tensors)
    offs, sizes = (C.c_int64 * n)(), (C.c_int64 * n)()
    total = lib.tfl_train_grad_layout(eng.plan, offs, sizes, n)
    B, Tf, F, _ = x_in.shape
    ws = torch.empty(lib.tfl_train_stage_workspace_bytes(eng.plan, B, Tf, F), dtype=torch.uint8, device=x_in.device)
    grads = torch.zeros(int(total), dtype=torch.float32, device=x_in.device)
    staged = [t.detach().to(torch.float32).contiguous() for t in tensors]
    arr = (C.c_void_p * n)(*[t.data_ptr() for t in staged])

    def grad_of(key):
        i = eng.keys.index(key)
        return grads[offs[i]:offs[i] + sizes[i]].view(tensors[i].shape)

    return lib, eng, arr, n, ws, grads, grad_of, staged


def ffn_backward(model, layer: int, axis: int, index: int, x_in: torch.Tensor, dy: torch.Tensor):
    """x_out = x_in + FFN(norm(x_in)) along ``axis`` on channels-last [B, Tf, F, C]: returns (dL/dx_in, grad_of(key))."""
    _require_cuda(x_in, "x_in")
    B, Tf, F, _ = x_in.shape
    dx = dy.detach().to(torch.float32).contiguous().clone()
    xc = x_in.detach().to(torch.float32).contiguous()
    with deterministic_option(torch.are_deterministic_algorithms_enabled()), torch.cuda.device(x_in.device):
        lib, eng, arr, n, ws, grads, grad_of, staged = _stage_setup(model, x_in)
        check(lib.tfl_conv_swiglu_ffn_bwd(eng.plan, eng.packed.data_ptr(), arr, n, layer, axis, index, xc.data_ptr(),
                                          dx.data_ptr(), B, Tf, F, grads.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
        torch.cuda.synchronize()
    return dx, grad_of


def attn_backward(model, layer: int, axis: int, x_in: torch.Tensor, dy: torch.Tensor):
    """x_out = x_in + MHSA(norm(x_in)) along ``axis``: returns (dL/dx_in, grad_of(key))."""
    _require_cuda(x_in, "x_in")
    B, Tf, F, _ = x_in.shape
    dx = dy.detach().to(torch.float32).contiguous().clone()
    xc = x_in.detach().to(torch.float32).contiguous()
    with deterministic_option(torch.are_deterministic_algorithms_enabled()), torch.cuda.device(x_in.device):
        lib, eng, arr, n, ws, grads, grad_of, staged = _stage_setup(model, x_in)
        check(lib.tfl_rope_attn_bwd(eng.plan, eng.packed.data_ptr(), arr, n, layer, axis, xc.data_ptr(), dx.data_ptr(),
                                    B, Tf, F, grads.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
        torch.cuda.synchronize()
    return dx, grad_of
