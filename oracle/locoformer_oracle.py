"""CPU restatement of the reference forward path -- TEST INFRASTRUCTURE ONLY.

See oracle/__init__.py for who may import this.  Citations are into /root/reference/.
All functions are pure: weights come in as a ``state_dict``-style mapping with the
reference's key names (SURVEY.md section 8b), activations are channels-last
``[B, Tf, F, C]`` torch CPU tensors.  ``dtype`` may be float32 (the parity oracle) or
float64 (a tighter "truth" used to judge which of two fp32 results is closer).
"""
import math
from typing import Dict, List, Optional, Sequence, Union

import torch

from .rope import rope_rotate

SOURCE_NAMES = ["vocals", "drums", "bass", "other"]  # models/mss_tflocoformer.py:242


# --------------------------------------------------------------------------------------
# STFT / iSTFT  (models/mss_tflocoformer.py:36-75 -> torch.stft / torch.istft semantics)
# --------------------------------------------------------------------------------------
def hann_periodic(n: int, dtype=torch.float32) -> torch.Tensor:
    """torch.hann_window(n) (periodic): 0.5 - 0.5 cos(2 pi k / n).  :45, :66"""
    k = torch.arange(n, dtype=torch.float64)
    return (0.5 - 0.5 * torch.cos(2.0 * math.pi * k / n)).to(dtype)


def stft(audio: torch.Tensor, n_fft: int, hop: int) -> torch.Tensor:
    """models/mss_tflocoformer.py:36-54.  audio [B, T] -> complex [B, Tf, F].

    center=True, reflect pad n_fft/2, periodic Hann, onesided, unnormalised;
    frame t = padded[t*hop : t*hop + n_fft]; Tf = 1 + T // hop.  (The reference's
    [B, F, Tf] is this transposed; it transposes right back at :214.)
    """
    pad = n_fft // 2
    if audio.shape[-1] <= pad:
        raise RuntimeError("reflect padding needs more than n_fft/2 samples")  # torch's own error
    left = audio[:, 1:pad + 1].flip(-1)
    right = audio[:, -pad - 1:-1].flip(-1)
    padded = torch.cat([left, audio, right], dim=-1)
    n_frames = 1 + audio.shape[-1] // hop
    idx = torch.arange(n_frames)[:, None] * hop + torch.arange(n_fft)[None, :]
    frames = padded[:, idx] * hann_periodic(n_fft, audio.dtype)
    return torch.fft.rfft(frames, dim=-1)


def istft(spec: torch.Tensor, n_fft: int, hop: int, length: int) -> torch.Tensor:
    """models/mss_tflocoformer.py:56-75.  complex [B, Tf, F] -> [B, length].

    irfft per frame (imaginary parts of DC / Nyquist ignored), times window,
    overlap-add, divide by the sum of squared windows, drop the first n_fft/2
    samples, cut (or zero-extend) to ``length``.
    """
    b, n_frames, _ = spec.shape
    rdtype = torch.float64 if spec.dtype == torch.complex128 else torch.float32
    win = hann_periodic(n_fft, rdtype)
    frames = torch.fft.irfft(spec, n=n_fft, dim=-1) * win
    total = n_fft + hop * (n_frames - 1)
    y = torch.zeros(b, total, dtype=rdtype)
    env = torch.zeros(total, dtype=rdtype)
    wsq = win * win
    for t in range(n_frames):
        y[:, t * hop:t * hop + n_fft] += frames[:, t]
        env[t * hop:t * hop + n_fft] += wsq
    start = n_fft // 2
    y = y[:, start:start + length]
    env = env[start:start + length]
    y = y / env
    if y.shape[-1] < length:
        y = torch.nn.functional.pad(y, (0, length - y.shape[-1]))
    return y


# --------------------------------------------------------------------------------------
# Encoder / decoder  (models/mss_tflocoformer.py:141-146,218-219 and :182,229-237)
# --------------------------------------------------------------------------------------
def encoder(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, gw: torch.Tensor,
            gb: torch.Tensor, eps: float) -> torch.Tensor:
    """Conv2d(Cin, C, 3x3, padding 1) + GroupNorm(1, C).  x [B, Tf, F, Cin] -> [B, Tf, F, C].

    Kernel dim 0 runs over frames, dim 1 over bins (:142-144).  gLN statistics are over
    (C, Tf, F) per sample, biased variance, eps inside the sqrt (:145).
    """
    bsz, tf, nf, cin = x.shape
    xp = torch.zeros(bsz, tf + 2, nf + 2, cin, dtype=x.dtype)
    xp[:, 1:-1, 1:-1] = x
    y = b.to(x.dtype).expand(bsz, tf, nf, -1).clone()
    for dt in range(3):
        for df in range(3):
            y = y + xp[:, dt:dt + tf, df:df + nf] @ w[:, :, dt, df].to(x.dtype).t()
    mean = y.mean(dim=(1, 2, 3), keepdim=True)
    var = ((y - mean) ** 2).mean(dim=(1, 2, 3), keepdim=True)
    return (y - mean) / torch.sqrt(var + eps) * gw.to(x.dtype) + gb.to(x.dtype)


def decoder(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """ConvTranspose2d(C, 2S, 3x3, padding 1), stride 1 (:182).  [B,Tf,F,C] -> [B,Tf,F,2S].

    out[t, f, o] = b[o] + sum_{dt,df,c} x[t + 1 - dt, f + 1 - df, c] * w[c, o, dt, df].
    """
    bsz, tf, nf, c = x.shape
    xp = torch.zeros(bsz, tf + 2, nf + 2, c, dtype=x.dtype)
    xp[:, 1:-1, 1:-1] = x
    y = b.to(x.dtype).expand(bsz, tf, nf, -1).clone()
    for dt in range(3):
        for df in range(3):
            y = y + xp[:, 2 - dt:2 - dt + tf, 2 - df:2 - df + nf] @ w[:, :, dt, df].to(x.dtype)
    return y


# --------------------------------------------------------------------------------------
# Block internals
# --------------------------------------------------------------------------------------
def rms_group_norm(x: torch.Tensor, gamma: torch.Tensor, groups: int, eps: float) -> torch.Tensor:
    """models/mss_tflocoformer.py:682-706.  eps is added to the RMS, outside the sqrt."""
    c = x.shape[-1]
    d = c // groups
    xg = x.reshape(x.shape[:-1] + (groups, d))
    rms = torch.sqrt((xg * xg).sum(-1, keepdim=True)) * d ** -0.5
    return (xg / (rms + eps)).reshape(x.shape) * gamma.to(x.dtype)


def swiglu_conv_deconv(xn: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor,
                       w2: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """models/mss_tflocoformer.py:626-655 with conv1d_shift == 1.

    xn [Nseq, S, C] (already normalised).  Zero-pad K-1 both sides (:640-644);
    h[j] = b1 + sum_k W1[:, :, k] xp[j + k], j < S + K - 1 (:647);
    g = h[:, :hid] * silu(h[:, hid:]) (:648-649);
    out[i] = b2 + sum_k W2[:, :, k]^T g[i + (K - 1) - k]  (ConvTranspose1d :651, crop :654).
    """
    nseq, s, c = xn.shape
    two_h, _, k = w1.shape
    hid = two_h // 2
    dt = xn.dtype
    xp = torch.zeros(nseq, s + 2 * (k - 1), c, dtype=dt)
    xp[:, k - 1:k - 1 + s] = xn
    hlen = s + k - 1
    h = b1.to(dt).expand(nseq, hlen, -1).clone()
    for kk in range(k):
        h = h + xp[:, kk:kk + hlen] @ w1[:, :, kk].to(dt).t()
    gate = h[..., hid:]
    g = h[..., :hid] * (gate * torch.sigmoid(gate))
    out = b2.to(dt).expand(nseq, s, -1).clone()
    for kk in range(k):
        out = out + g[:, (k - 1) - kk:(k - 1) - kk + s] @ w2[:, :, kk].to(dt)
    return out


def attention(xn: torch.Tensor, wqkv: torch.Tensor, wo: torch.Tensor, n_heads: int,
              freqs: Optional[torch.Tensor]) -> torch.Tensor:
    """models/mss_tflocoformer.py:504-559.  xn [Nseq, L, C] -> [Nseq, L, C].

    qkv rows are [q ; k ; v], each head-major (:545-547); RoPE on q and k (:557-558);
    softmax(q k^T / sqrt(hd)) v, no mask (:525-531); heads merged head-major (:536-537);
    bias-free output projection (:487, :538).
    """
    nseq, length, _ = xn.shape
    dt = xn.dtype
    qkv = xn @ wqkv.to(dt).t()
    a = qkv.shape[-1] // 3
    hd = a // n_heads
    qkv = qkv.reshape(nseq, length, 3, n_heads, hd).permute(2, 0, 3, 1, 4)  # [3, Nseq, H, L, hd]
    q, k, v = qkv[0], qkv[1], qkv[2]
    if freqs is not None:
        q = rope_rotate(q, freqs)
        k = rope_rotate(k, freqs)
    scores = (q @ k.transpose(-1, -2)) * (1.0 / math.sqrt(hd))
    p = torch.softmax(scores, dim=-1)
    o = (p @ v).permute(0, 2, 1, 3).reshape(nseq, length, a)
    return o @ wo.to(dt).t()


def locoformer_path(x: torch.Tensor, sd: Dict[str, torch.Tensor], prefix: str, cfg: dict) -> torch.Tensor:
    """LocoformerBlock.forward, models/mss_tflocoformer.py:430-464.  x [B, S1, S2, C].

    ffn / ffn_norm lists are stored in REVERSED config order (:391-392): index -1 is the
    pre-attention (macaron) FFN, index 0 the post-attention one.  No 1/2 scaling.
    """
    b, s1, s2, c = x.shape
    groups, eps, heads = cfg["num_groups"], cfg["eps"], cfg["n_heads"]
    macaron = isinstance(cfg["ffn_type"], (list, tuple)) and len(cfg["ffn_type"]) == 2

    def ffn(x, j):
        p = f"{prefix}.ffn.{j}."
        xn = rms_group_norm(x, sd[f"{prefix}.ffn_norm.{j}.gamma"], groups, eps)
        y = swiglu_conv_deconv(xn.reshape(b * s1, s2, c), sd[p + "conv1d.weight"], sd[p + "conv1d.bias"],
                               sd[p + "deconv1d.weight"], sd[p + "deconv1d.bias"])
        return x + y.reshape(b, s1, s2, c)

    if macaron:
        x = ffn(x, 1)                                                         # :443-447 (index -1)
    xn = rms_group_norm(x, sd[f"{prefix}.attn_norm.gamma"], groups, eps)     # :452-453
    freqs = sd.get(f"{prefix}.attn.rope.freqs") if cfg.get("pos_enc", "rope") == "rope" else None
    y = attention(xn.reshape(b * s1, s2, c), sd[f"{prefix}.attn.qkv.weight"],
                  sd[f"{prefix}.attn.aggregate_heads.0.weight"], heads, freqs)
    x = x + y.reshape(b, s1, s2, c)                                           # :456
    return ffn(x, 0)                                                          # :459-462


def tf_block(x: torch.Tensor, sd, prefix: str, cfg: dict) -> torch.Tensor:
    """TFLocoformerBlock, models/mss_tflocoformer.py:323-353.  x [B, Tf, F, C] channels-last."""
    def freq(x):   # batch B*Tf, sequence along F
        return locoformer_path(x, sd, prefix + ".freq_path", cfg)

    def time(x):   # batch B*F, sequence along Tf
        return locoformer_path(x.transpose(1, 2).contiguous(), sd, prefix + ".frame_path", cfg).transpose(1, 2).contiguous()

    if cfg.get("tf_order", "ft") == "ft":
        return time(freq(x))
    return freq(time(x))


def blocks_forward(x, sd, cfg, prefix="blocks"):
    for i in range(cfg["n_layers"]):
        x = tf_block(x, sd, f"{prefix}.{i}", cfg)
    return x


# --------------------------------------------------------------------------------------
# Whole models
# --------------------------------------------------------------------------------------
def _cast(sd, dtype):
    """Weights in the compute dtype; a weight that requires grad keeps its autograd graph (the training tests
    differentiate the oracle forward with respect to the state_dict)."""
    return {k: v.to(dtype) if v.is_floating_point() else v for k, v in sd.items()}


def separator_forward(sd, cfg: dict, spec: torch.Tensor, dtype=torch.float32) -> torch.Tensor:
    """standalone/tflocoformer_separator.py:131-171.  complex [B, T, F] -> complex [B, S, T, F]."""
    sd = _cast(sd, dtype)
    if spec.ndim == 4:
        assert spec.shape[1] == 1, "Only monaural input is supported."
        spec = spec[:, 0]
    x = torch.stack([spec.real, spec.imag], dim=-1).to(dtype)                 # [B, T, F, 2]
    x = encoder(x, sd["conv.0.weight"], sd["conv.0.bias"], sd["conv.1.weight"], sd["conv.1.bias"], cfg["eps"])
    x = blocks_forward(x, sd, cfg)
    y = decoder(x, sd["deconv.weight"], sd["deconv.bias"])                    # [B, T, F, 2S]
    b, t, f, _ = y.shape
    y = y.reshape(b, t, f, -1, 2).permute(0, 3, 1, 2, 4)                      # [B, S, T, F, 2]
    return torch.complex(y[..., 0].contiguous(), y[..., 1].contiguous())


def mss_forward(sd, cfg: dict, mixture: torch.Tensor, return_time_domain: bool = True,
                dtype=torch.float32) -> Dict[str, torch.Tensor]:
    """TFLocoformerMSS.forward, models/mss_tflocoformer.py:184-258.  mixture [B, T]."""
    n_fft, hop, n_src = cfg["n_fft"], cfg["hop_length"], cfg["n_sources"]
    spec = stft(mixture.to(dtype), n_fft, hop)                                # [B, Tf, F]
    est = separator_forward(sd, cfg, spec, dtype)                             # [B, S, Tf, F]
    out = {}
    for i, name in enumerate(SOURCE_NAMES[:n_src]):
        if return_time_domain:
            out[name] = istft(est[:, i], n_fft, hop, mixture.shape[-1])
        else:
            out[name] = est[:, i].transpose(-1, -2)                           # [B, F, Tf] (:237)
    return out


def bs_bands(sample_rate: int, stft_size: int) -> List[int]:
    """standalone/bslocoformer_separator.py:191-207."""
    table = {(0, 1000): 2, (1000, 2000): 4, (2000, 4000): 12, (4000, 8000): 24, (8000, 16000): 48}
    nbins = stft_size // 2 + 1
    per_bin = sample_rate // 2 / nbins
    bands: List[int] = []
    for (lo, hi), width in table.items():
        bands += [width] * math.ceil((hi - lo) / (width * per_bin))
    rest = nbins - sum(bands)
    if sample_rate == 48000:
        bands += [rest // 4, rest // 4, rest // 4, rest // 4 + rest % 4]
    else:
        bands += [math.floor(rest / 2), math.ceil(rest / 2)]
    assert sum(bands) == nbins, (sum(bands), nbins, bands)
    return bands


def _gn1(x, w, b, eps=1e-5):
    """GroupNorm(1, C) on [B, C, T]: stats over (C, T)."""
    mean = x.mean(dim=(1, 2), keepdim=True)
    var = ((x - mean) ** 2).mean(dim=(1, 2), keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * w[None, :, None] + b[None, :, None]


def bs_forward(sd, cfg: dict, spec: torch.Tensor, dtype=torch.float32) -> torch.Tensor:
    """BSLocoformerSeparator.forward, standalone/bslocoformer_separator.py:142-183.

    spec complex [B, T, F] (mono) or [B, M=2, T, F] (stereo) -> [B, S, (M), T, F].
    """
    sd = _cast(sd, dtype)
    stereo, masking, n_src = cfg.get("stereo", False), cfg.get("masking", True), cfg["num_spk"]
    cdt = torch.complex64 if dtype == torch.float32 else torch.complex128
    inp = spec.to(cdt)
    if inp.ndim == 3:
        assert not stereo
        inp = inp.unsqueeze(1)
    bsz, m, t, f = inp.shape
    coef = 2 * m
    bands = bs_bands(cfg.get("sample_rate", 44100), cfg.get("stft_size", 2048))
    edges = [0]
    for w in bands:
        edges.append(edges[-1] + w)
    # [B, T, F, 2M] with channel order (re_0..re_{M-1}, im_0..im_{M-1})  (:163-164)
    feat = torch.cat([inp.real, inp.imag], dim=1).permute(0, 2, 3, 1)
    cols = []
    for bi, w in enumerate(bands):                                            # :241-254
        sub = feat[:, :, edges[bi]:edges[bi + 1]]                             # [B, T, w, 2M]
        sub = sub.permute(0, 2, 3, 1).reshape(bsz, w * coef, t)               # channel = f_local*2M + ch
        p = f"band_split_module.band_split_module.{bi}."
        sub = _gn1(sub, sd[p + "0.weight"], sd[p + "0.bias"])
        cols.append(torch.einsum("oc,bct->bto", sd[p + "1.weight"][:, :, 0], sub) + sd[p + "1.bias"])
    x = torch.stack(cols, dim=2)                                              # [B, T, nb, C]
    x = blocks_forward(x, sd, cfg)
    outs = []
    for bi, w in enumerate(bands):                                            # :256-270
        p = f"band_split_module.bandwise_decoding_module.{bi}."
        z = x[:, :, bi].transpose(1, 2)                                       # [B, C, T]
        z = _gn1(z, sd[p + "0.weight"], sd[p + "0.bias"])
        z = torch.einsum("oc,bct->bot", sd[p + "1.weight"][:, :, 0], z) + sd[p + "1.bias"][None, :, None]
        z = torch.tanh(z)
        z = torch.einsum("oc,bct->bot", sd[p + "3.weight"][:, :, 0], z) + sd[p + "3.bias"][None, :, None]
        z = torch.einsum("oc,bct->bot", sd[p + "4.weight"][:, :, 0], z) + sd[p + "4.bias"][None, :, None]
        half = z.shape[1] // 2
        z = z[:, :half] * torch.sigmoid(z[:, half:])                          # GLU(dim=1)
        if stereo:
            z = z.reshape(bsz, 2, n_src, 2, w, t)
        else:
            z = z.reshape(bsz, 2, n_src, 1, w, t)
        outs.append(z)
    y = torch.cat(outs, dim=-2).transpose(-1, -2)                             # [B, 2, S, M, T, F]
    y = torch.complex(y[:, 0].contiguous(), y[:, 1].contiguous())             # [B, S, M, T, F]
    if masking:
        y = inp.unsqueeze(1) * y                                              # :179-182
    if not stereo:
        y = y[:, :, 0]
    return y


def si_sdr_db(est: torch.Tensor, ref: torch.Tensor, eps: float = 1e-12) -> float:
    """Scale-invariant SDR in dB of ``est`` against ``ref`` (evaluation/metrics.py:35-56)."""
    est = est.reshape(-1).double()
    ref = ref.reshape(-1).double()
    est = est - est.mean()
    ref = ref - ref.mean()
    alpha = (est @ ref) / (ref @ ref + eps)
    target = alpha * ref
    noise = est - target
    return float(10.0 * torch.log10((target @ target + eps) / (noise @ noise + eps)))
