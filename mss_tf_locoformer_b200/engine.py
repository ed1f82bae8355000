"""Host-side driver of the C-ABI library: plan, weight packing, workspace, launches.

PyTorch is used for device memory, streams and parameter storage only; every arithmetic
step of the forward path is a kernel of csrc/ reached through include/tfl.h.
"""
import ctypes as C
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib
from ._lib import TflConfig, check

PRECISIONS = {"fp32": 0, "bf16": 1}
AXIS = {"freq": 0, "time": 1}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: mss_tf_locoformer_b200 has no CPU path (got {t.device})")


def weight_keys(cfg: dict) -> List[str]:
    """state_dict keys in the order tfl_pack_weights expects (include/tfl.h)."""
    n_ffn = 2 if cfg["macaron"] else 1
    keys = []
    if cfg["enc_in_ch"]:
        keys += ["conv.0.weight", "conv.0.bias", "conv.1.weight", "conv.1.bias"]
    for i in range(cfg["n_layers"]):
        for path in ("freq_path", "frame_path"):
            p = f"blocks.{i}.{path}."
            keys += [p + f"ffn_norm.{j}.gamma" for j in range(n_ffn)]
            for j in range(n_ffn):
                keys += [p + f"ffn.{j}.conv1d.weight", p + f"ffn.{j}.conv1d.bias",
                         p + f"ffn.{j}.deconv1d.weight", p + f"ffn.{j}.deconv1d.bias"]
            keys.append(p + "attn_norm.gamma")
            if cfg["rope"]:
                keys.append(p + "attn.rope.freqs")
            keys += [p + "attn.qkv.weight", p + "attn.aggregate_heads.0.weight"]
    if cfg["enc_in_ch"]:
        keys += ["deconv.weight", "deconv.bias"]
    return keys


class Engine:
    """One per model instance.  Owns the tfl_plan, the packed weight image and workspaces."""

    def __init__(self, cfg: dict):
        self.cfg = dict(cfg)
        self.lib = _lib.load()
        c = TflConfig(**{k: v for k, v in self.cfg.items()})
        handle = C.c_void_p()
        check(self.lib.tfl_plan_create(C.byref(c), C.byref(handle)))
        self.plan = handle
        self.keys = weight_keys(self.cfg)
        assert len(self.keys) == self.lib.tfl_num_weight_tensors(self.plan)
        self.packed: Optional[torch.Tensor] = None
        self._fingerprint = None
        self._ws: Dict[Tuple, torch.Tensor] = {}
        self._staging: List[torch.Tensor] = []

    def __del__(self):
        try:
            if getattr(self, "plan", None):
                self.lib.tfl_plan_destroy(self.plan)
                self.plan = None
        except Exception:
            pass

    # ---- weights -------------------------------------------------------------------
    @staticmethod
    def _version_of(t: torch.Tensor) -> int:
        try:
            return t._version
        except RuntimeError:          # inference-mode tensors do not track versions: repack on every data_ptr change only
            return -1

    def invalidate(self):
        """Force a re-pack at the next forward (after in-place writes the fingerprint cannot see, e.g. ``p.data.copy_``)."""
        self._fingerprint = None

    def ensure_packed(self, params: Dict[str, torch.Tensor]):
        tensors = [params[k] for k in self.keys]
        fp = tuple((t.data_ptr(), self._version_of(t), t.device) for t in tensors)
        if fp == self._fingerprint and self.packed is not None:
            return
        dev = tensors[0].device
        for k, t in zip(self.keys, tensors):
            _require_cuda(t, k)
            if t.device != dev:
                raise RuntimeError("all parameters must live on one CUDA device")
        staged = [t.detach().to(torch.float32).contiguous() for t in tensors]
        nbytes = self.lib.tfl_packed_bytes(self.plan)
        packed = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        arr = (C.c_void_p * len(staged))(*[t.data_ptr() for t in staged])
        with torch.cuda.device(dev):
            check(self.lib.tfl_pack_weights(self.plan, arr, len(staged), packed.data_ptr(), nbytes, _stream()))
        self._staging = staged  # keep alive until the pack kernels have run
        self.packed = packed
        self._fingerprint = fp
        self._ws.clear()

    def workspace(self, B: int, Tf: int, F: int, precision: int, device) -> torch.Tensor:
        key = (B, Tf, F, precision, str(device))
        ws = self._ws.get(key)
        if ws is None:
            n = self.lib.tfl_workspace_bytes(self.plan, B, Tf, F, precision)
            if len(self._ws) >= 4:
                self._ws.clear()
            ws = torch.empty(max(n, 256), dtype=torch.uint8, device=device)
            self._ws[key] = ws
        return ws

    # ---- whole-model calls ---------------------------------------------------------
    def check_mixture(self, mixture: torch.Tensor):
        """The mixture checks of TFLocoformerMSS.forward: a [B, T] CUDA tensor longer than the reflect padding."""
        _require_cuda(mixture, "mixture")
        if mixture.ndim != 2:
            raise ValueError(f"mixture must be [B, T], got {tuple(mixture.shape)}")
        B, T = mixture.shape
        n_fft = self.cfg["n_fft"]
        if T <= n_fft // 2:  # same failure mode as torch.stft's reflect pad in the reference
            raise RuntimeError(f"Argument #4: Padding size should be less than the corresponding input dimension, "
                               f"but got: padding ({n_fft // 2}, {n_fft // 2}) at dimension 2 of input {[1, B, T]}")

    def mss_forward(self, mixture: torch.Tensor, precision: int, want_audio: bool, want_spec: bool):
        """mixture [B, T] fp32 CUDA -> (audio [S, B, T] or None, est_spec [B, S, Tf, F, 2] or None)."""
        self.check_mixture(mixture)
        B, T = mixture.shape
        n_fft, hop, S = self.cfg["n_fft"], self.cfg["hop"], self.cfg["n_src"]
        x = mixture.detach().to(torch.float32).contiguous()
        Tf, F = 1 + T // hop, n_fft // 2 + 1
        dev = x.device
        ws = self.workspace(B, Tf, F, precision, dev)
        audio = torch.empty((S, B, T), dtype=torch.float32, device=dev) if want_audio else None
        spec = torch.empty((B, S, Tf, F, 2), dtype=torch.float32, device=dev) if want_spec else None
        with torch.cuda.device(dev):
            check(self.lib.tfl_forward(self.plan, self.packed.data_ptr(), x.data_ptr(), B, T, _ptr(audio), _ptr(spec),
                                       ws.data_ptr(), ws.numel(), precision, _stream()))
        return audio, spec

    def separator_forward(self, spec_ri: torch.Tensor, precision: int) -> torch.Tensor:
        """spec_ri [B, T, F, 2] fp32 CUDA -> est [B, S, T, F, 2]."""
        _require_cuda(spec_ri, "input")
        B, Tf, F, _ = spec_ri.shape
        dev = spec_ri.device
        ws = self.workspace(B, Tf, F, precision, dev)
        est = torch.empty((B, self.cfg["n_src"], Tf, F, 2), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(self.lib.tfl_separator_forward(self.plan, self.packed.data_ptr(), spec_ri.data_ptr(), B, Tf, F,
                                                 est.data_ptr(), ws.data_ptr(), ws.numel(), precision, _stream()))
        return est

    def blocks(self, x: torch.Tensor, precision: int) -> torch.Tensor:
        """All Locoformer blocks, in place on x [B, Tf, F, C] fp32 (channels-last)."""
        _require_cuda(x, "x")
        B, Tf, F, _ = x.shape
        ws = self.workspace(B, Tf, F, precision, x.device)
        with torch.cuda.device(x.device):
            check(self.lib.tfl_blocks(self.plan, self.packed.data_ptr(), x.data_ptr(), B, Tf, F, ws.data_ptr(),
                                      ws.numel(), precision, _stream()))
        return x

    # ---- stage calls (used by the sub-module forwards and the per-kernel tests) ------
    def stft(self, audio: torch.Tensor) -> torch.Tensor:
        _require_cuda(audio, "audio")
        B, T = audio.shape
        Tf, F = 1 + T // self.cfg["hop"], self.cfg["n_fft"] // 2 + 1
        spec = torch.empty((B, Tf, F, 2), dtype=torch.float32, device=audio.device)
        with torch.cuda.device(audio.device):
            check(self.lib.tfl_stft(self.plan, self.packed.data_ptr(), audio.contiguous().data_ptr(), B, T,
                                    spec.data_ptr(), _stream()))
        return spec

    def istft(self, est: torch.Tensor, n_samples: int) -> torch.Tensor:
        """est [B, S, Tf, F, 2] -> audio [S, B, n_samples]."""
        _require_cuda(est, "est")
        B, S, Tf, F, _ = est.shape
        audio = torch.empty((S, B, n_samples), dtype=torch.float32, device=est.device)
        with torch.cuda.device(est.device):
            check(self.lib.tfl_istft_ola(self.plan, self.packed.data_ptr(), est.contiguous().data_ptr(), B, Tf,
                                         n_samples, audio.data_ptr(), _stream()))
        return audio

    def enc_conv_gln(self, spec_ri: torch.Tensor, precision: int = 0) -> torch.Tensor:
        """spec_ri [B, Tf, F, 2] -> x [B, Tf, F, C]; ``precision`` 1 is the tf32 encoder of the bf16 mode."""
        _require_cuda(spec_ri, "spec")
        B, Tf, F, _ = spec_ri.shape
        x = torch.empty((B, Tf, F, self.cfg["emb_dim"]), dtype=torch.float32, device=spec_ri.device)
        ws = self.workspace(B, Tf, F, 0, x.device)
        with torch.cuda.device(x.device):
            check(self.lib.tfl_enc_conv_gln_mode(self.plan, self.packed.data_ptr(), spec_ri.contiguous().data_ptr(), B,
                                                 Tf, F, x.data_ptr(), ws.data_ptr(), ws.numel(), precision, _stream()))
        return x

    def dec_conv(self, x: torch.Tensor, precision: int = 0) -> torch.Tensor:
        _require_cuda(x, "x")
        B, Tf, F, _ = x.shape
        est = torch.empty((B, self.cfg["n_src"], Tf, F, 2), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            check(self.lib.tfl_dec_conv_mode(self.plan, self.packed.data_ptr(), x.contiguous().data_ptr(), B, Tf, F,
                                             est.data_ptr(), precision, _stream()))
        return est

    def rms_group_norm(self, layer: int, axis: int, which: int, x: torch.Tensor) -> torch.Tensor:
        _require_cuda(x, "x")
        xc = x.contiguous()
        y = torch.empty_like(xc)
        rows = xc.numel() // self.cfg["emb_dim"]
        with torch.cuda.device(x.device):
            check(self.lib.tfl_rms_group_norm(self.plan, self.packed.data_ptr(), layer, axis, which, xc.data_ptr(),
                                              y.data_ptr(), rows, _stream()))
        return y

    def ffn_(self, layer: int, axis: int, index: int, x: torch.Tensor, precision: int) -> torch.Tensor:
        """In place on channels-last x [B, Tf, F, C]: x += FFN(norm(x)) along ``axis``."""
        _require_cuda(x, "x")
        B, Tf, F, _ = x.shape
        ws = self.workspace(B, Tf, F, precision, x.device)
        with torch.cuda.device(x.device):
            check(self.lib.tfl_conv_swiglu_ffn(self.plan, self.packed.data_ptr(), layer, axis, index, x.data_ptr(), B,
                                               Tf, F, ws.data_ptr(), ws.numel(), precision, _stream()))
        return x

    def ffn_out(self, layer: int, axis: int, index: int, x: torch.Tensor, y: torch.Tensor, precision: int) -> torch.Tensor:
        """Out of place on channels-last [B, Tf, F, C]: y = x + FFN(norm(x)) along ``axis`` (x, y distinct)."""
        _require_cuda(x, "x")
        _require_cuda(y, "y")
        if not (x.is_contiguous() and y.is_contiguous()) or x.shape != y.shape:
            raise ValueError("x and y must be contiguous tensors of the same shape")
        B, Tf, F, _ = x.shape
        ws = self.workspace(B, Tf, F, precision, x.device)
        with torch.cuda.device(x.device):
            check(self.lib.tfl_conv_swiglu_ffn_out(self.plan, self.packed.data_ptr(), layer, axis, index, x.data_ptr(),
                                                   y.data_ptr(), B, Tf, F, ws.data_ptr(), ws.numel(), precision, _stream()))
        return y

    def attn_(self, layer: int, axis: int, x: torch.Tensor, precision: int) -> torch.Tensor:
        """In place on channels-last x [B, Tf, F, C]: x += MHSA(norm(x)) along ``axis``."""
        _require_cuda(x, "x")
        B, Tf, F, _ = x.shape
        ws = self.workspace(B, Tf, F, precision, x.device)
        with torch.cuda.device(x.device):
            check(self.lib.tfl_rope_attn(self.plan, self.packed.data_ptr(), layer, axis, x.data_ptr(), B, Tf, F,
                                         ws.data_ptr(), ws.numel(), precision, _stream()))
        return x


def segment_ola(seg_audio: torch.Tensor, seg_index0: int, n_seg_total: int, track: torch.Tensor, track_origin: int = 0):
    """track[S, n] += window * seg_audio[S, B, seg_len] for segments seg_index0.. (tfl_segment_ola); ``track`` holds the
    samples [track_origin, track_origin + n) of the full track."""
    _require_cuda(seg_audio, "seg_audio")
    S, B, L = seg_audio.shape
    lib = _lib.load()
    with torch.cuda.device(track.device):
        check(lib.tfl_segment_ola(seg_audio.contiguous().data_ptr(), S, B, L, seg_index0, n_seg_total, track.data_ptr(),
                                  track.shape[-1], track_origin, _stream()))
    return track


def tc_selftest(A: torch.Tensor, B: torch.Tensor, taps: int, mode: int) -> torch.Tensor:
    """Diagnostic for the tcgen05 plumbing (tfl_tc_selftest).  mode 0: A [128+taps-1, Kd], B [taps, N, Kd];
    mode 1: A [128, Kd], B [Kd, N].  Returns D [128, N] fp32."""
    _require_cuda(A, "A")
    lib = _lib.load()
    Kd = A.shape[1]
    N = B.shape[1] if mode == 0 else B.shape[1]
    D = torch.empty((128, N), dtype=torch.float32, device=A.device)
    scratch = torch.empty(max(256, taps * N * Kd * 2), dtype=torch.uint8, device=A.device)
    with torch.cuda.device(A.device):
        check(lib.tfl_tc_selftest(A.contiguous().data_ptr(), B.contiguous().data_ptr(), D.data_ptr(),
                                  scratch.data_ptr(), N, Kd, taps, mode, _stream()))
    return D


def debug_timeout(reset: bool = True):
    """(timed_out, block, thread, barrier smem address, parity) of the first expired mbarrier wait (tfl_debug_timeout)."""
    lib = _lib.load()
    out = (C.c_uint32 * 5)()
    check(lib.tfl_debug_timeout(out, 1 if reset else 0))
    return tuple(int(v) for v in out)
