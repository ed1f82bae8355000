"""float64 restatement of the bf16-mode sub-blocks, rounded where the kernels round -- TEST INFRASTRUCTURE ONLY.

``oracle`` states what the model computes; this module states what the bf16 mode's kernels compute: the same math in
float64, with every operand the kernels hand to a tensor core rounded to bf16 (tcgen05) or tf32 (mma.sync) at the
point where the kernel rounds it.  With ``rounding=False`` every function here is the float64 oracle (checked to
1e-12 by tests/test_bf16_ref_cpu.py).

Rounding points (kernel source, mss_tf_locoformer_b200/csrc/):

* FFN (ffn_tc_kernel, ffn_tc2_kernel)
  - A = bf16(x * inv * gamma), inv = 1 / (sqrt(ss) * D^-1/2 + eps): kernels_tc.cuh:435-436 and :469-470,
    kernels_tc2.cuh:513-514.
  - conv1d / transposed-conv weights: bf16 image, kernels_tc2.cuh:143 (tc_pack_ffn2_kernel) and tc_pack_ffn.
  - hidden = bf16(SwiGLU(acc + b1)): kernels_tc.cuh:621-623 (swiglu_fast), kernels_tc2.cuh:571 (swiglu_pair_bf16).
  - y = acc2 + b2 + x in fp32: kernels_tc2.cuh:644.
* attention (qkv_tc_kernel, attn_tc2_kernel / attn_tc_kernel, proj_tc_kernel)
  - A = bf16(x * inv), no gamma: kernels_attn.cuh:790-793, :827-828, :852-853.
  - q|k|v weight image = bf16(W * gamma * (log2(e) / sqrt(hd) for the q rows)), the products in fp32:
    kernels_attn.cuh:624.
  - RoPE in fp32 on the accumulator, angle = fp32(j * freq) (rope_table_kernel, kernels_attn.cuh:607), then q, k, v
    rounded to bf16: kernels_attn.cuh:898-904.
  - scores are in log2 units (the q image carries log2(e) / sqrt(hd)); p = exp2(s - m); the row sum uses fp32 p, the
    P.V product bf16(p): kernels_attn2.cuh:183-188.
  - O = bf16(P.V / l): kernels_attn2.cuh:607-615.  The projection uses the bf16 Wo image: kernels_attn.cuh:630.
* encoder (enc_conv_mma_kernel) and decoder (dec_conv_mma_kernel, dec_conv_scatter_kernel): spectrogram / activation
  and weights rounded to tf32 with cvt.rna (round to nearest, ties away from zero): kernels_f32.cuh:33-35, :273, :307,
  :770, :807, :863, :915.  The gLN statistics are double sums of the fp32 accumulators (kernels_f32.cuh:326-331).

One rounding point cannot be reproduced: attn_tc2_kernel subtracts a LAZY reference maximum m_ref (raised only when a
later key exceeds it by more than 2^ATT2_TH) before exp2, so the p it rounds to bf16 is p_true * 2^(m - m_ref) and
lands on other bf16 neighbours than the reference's exp2(s - rowmax).  The attn_tc_kernel (true running maximum) and
the tail-row kernels (fp32 p on CUDA cores or mma.sync) round p differently again.  Here p is rounded with the true row
maximum; the difference is an error source of the attention gates, not a modelled quantity.

The remaining differences between a correct kernel and this reference:
  (1) fp32 summation order of the accumulators (K = C * taps <= 2048 terms: ~1e-6 relative);
  (2) tanh.approx in SwiGLU (2^-11 relative), ex2.approx / rcp.approx / sqrt.approx in the attention (~2^-22);
  (3) the non-reproducible bf16 rounding of P above;
  (4) rounding flips: an intermediate that the kernel holds (1)-(3) away from the reference value rounds to the other
      bf16 neighbour with probability ~ (difference / ulp); each flip is one ulp (2^-8 relative) of one element.
(1) and (2) reach the output through (4): hidden elements differ by ~2^-11 before rounding, ~1/8 of them flip, and the
transposed conv averages H * K such independent one-ulp flips, so the branch error is ~ 2^-8 * sqrt(1/8) ~ 1.4e-3 of
the branch's RMS at worst, ~5e-4 typically.  (3) is of the same size for the attention.  So:

  REL_L2 = 2e-3   per-sequence ||got - ref|| / ||ref|| of the branch (half a bf16 ulp of 2^-8 = 3.9e-3)
  MAX_OVER_RMS = 1e-2   per-sequence max |got - ref| / RMS(ref): a sum of many independent roundings is near-Gaussian,
                        and the largest of <= 1e6 Gaussian samples is < 5 standard deviations, 5 * REL_L2.

The attention has one more error source that the estimate above does not cover: (3), the bf16 rounding of P, which
the reference gets wrong by construction whenever attn_tc2's lazy m_ref differs from the row maximum.  Where they agree
(L <= 16: m_ref is taken from the first 16 keys) the reference reproduces the kernels to ~1e-7.  Where they do not, p
carries 2^-9 of rounding noise in the kernel and independent noise in the reference, and O (rounded again to bf16)
inherits it: measured on an NVIDIA B200 (1000 W power limit), every attention shape with L >= 127 lands at 2.0e-3 to
3.2e-3 relative L2 and 1.1e-2 to 1.6e-2 max / RMS, on both attention kernels.  The attention gates are therefore one
bf16 ulp, the most the unmodelled P rounding may cost, and five times that for the maximum:

  REL_L2_ATTN = 4e-3, MAX_OVER_RMS_ATTN = 2e-2

A kernel bug that corrupts a few rows or channels of one sequence moves that sequence's statistics, not a global
maximum that other sequences dominate.
"""
import math
from typing import Optional, Tuple

import torch

REL_L2 = 2e-3
MAX_OVER_RMS = 1e-2
REL_L2_ATTN = 4e-3          # the bf16 rounding of P is not reproducible (see above)
MAX_OVER_RMS_ATTN = 2e-2
F64 = torch.float64


def bf16(x: torch.Tensor, on: bool = True) -> torch.Tensor:
    """Round to bf16 (round to nearest even) as the kernels' __float2bfloat16_rn / cvt.rn.bf16x2.f32 do on an fp32 value."""
    if not on:
        return x.to(F64)
    return x.to(torch.float32).to(torch.bfloat16).to(F64)


def tf32(x: torch.Tensor, on: bool = True) -> torch.Tensor:
    """Round to tf32 (10 explicit mantissa bits) as cvt.rna.tf32.f32 does: to nearest, ties away from zero."""
    if not on:
        return x.to(F64)
    bits = x.to(torch.float32).contiguous().view(torch.int32)
    finite = torch.isfinite(x.to(torch.float32))
    # the sign is the top bit: adding half of the dropped 13 bits to the pattern rounds the magnitude away from zero
    r = torch.where(finite, (bits + 0x1000) & ~0x1FFF, bits)
    return r.view(torch.float32).to(F64)


def _fp32(x):
    return torch.as_tensor(x, dtype=torch.float32)


def _inv_rms(x: torch.Tensor, groups: int, eps: float) -> torch.Tensor:
    """1 / (sqrt(sum of squares) * D^-1/2 + eps) per (row, group), broadcast over the group's channels."""
    c = x.shape[-1]
    d = c // groups
    xg = x.reshape(x.shape[:-1] + (groups, d))
    inv = 1.0 / (torch.sqrt((xg * xg).sum(-1, keepdim=True)) * d ** -0.5 + eps)
    return inv.expand(xg.shape).reshape(x.shape)


def ffn_branch(x: torch.Tensor, gamma, w1, b1, w2, b2, groups: int, eps: float, rounding: bool = True) -> torch.Tensor:
    """ConvSwiGLU(RMSGroupNorm(x)) of x [Nseq, S, C] (the FFN branch, without the residual) as the bf16 kernels
    compute it.  Weights in the reference's layout: w1 [2H, C, K], b1 [2H], w2 [H, C, K], b2 [C]."""
    x = x.to(F64)
    nseq, s, c = x.shape
    two_h, _, k = w1.shape
    hid = two_h // 2
    a = bf16(x * _inv_rms(x, groups, eps) * gamma.to(F64), rounding)
    w1, w2 = bf16(w1, rounding), bf16(w2, rounding)
    xp = torch.zeros(nseq, s + 2 * (k - 1), c, dtype=F64)
    xp[:, k - 1:k - 1 + s] = a
    hlen = s + k - 1
    h = b1.to(F64).expand(nseq, hlen, -1).clone()
    for kk in range(k):
        h = h + xp[:, kk:kk + hlen] @ w1[:, :, kk].t()
    gate = h[..., hid:]
    g = bf16(h[..., :hid] * (gate * torch.sigmoid(gate)), rounding)
    out = b2.to(F64).expand(nseq, s, -1).clone()
    for kk in range(k):
        out = out + g[:, (k - 1) - kk:(k - 1) - kk + s] @ w2[:, :, kk]
    return out


def attention_branch(x: torch.Tensor, gamma, wqkv, wo, n_heads: int, freqs: Optional[torch.Tensor], groups: int,
                     eps: float, rounding: bool = True, positions: Optional[torch.Tensor] = None,
                     drop_last_key: bool = False) -> torch.Tensor:
    """Wo MHSA(RoPE(qkv(RMSGroupNorm(x)))) of x [Nseq, L, C] as qkv_tc -> attn_tc2 -> proj_tc compute it.

    ``positions`` (default 0..L-1) and ``drop_last_key`` exist to build deliberately wrong references."""
    x = x.to(F64)
    nseq, length, c = x.shape
    a_dim = wqkv.shape[0] // 3
    hd = a_dim // n_heads
    a = bf16(x * _inv_rms(x, groups, eps), rounding)
    if rounding:   # the image is built in fp32: (w * gamma) * qscale, qscale = fp32(log2 e) / sqrtf(hd)
        qscale = _fp32(1.4426950408889634) / torch.sqrt(_fp32(hd))
        w = wqkv.to(torch.float32) * gamma.to(torch.float32)[None, :]
        w = torch.cat([w[:a_dim] * qscale, w[a_dim:]], 0)
        w = bf16(w)
    else:
        w = wqkv.to(F64) * gamma.to(F64)[None, :]
        w = torch.cat([w[:a_dim] * (math.log2(math.e) / math.sqrt(hd)), w[a_dim:]], 0)
    qkv = (a @ w.t()).reshape(nseq, length, 3, n_heads, hd).permute(2, 0, 3, 1, 4)   # [3, Nseq, H, L, hd]
    q, k, v = qkv[0], qkv[1], qkv[2]
    if freqs is not None:
        pos = torch.arange(length) if positions is None else positions
        ang = pos.to(torch.float32)[:, None] * freqs.to(torch.float32)[None, :]      # fp32 product and fp32 sincosf,
        cos, sin = ang.cos().to(F64), ang.sin().to(F64)                               # as the table (and the oracle)

        def rot(t):
            out = torch.empty_like(t)
            out[..., 0::2] = t[..., 0::2] * cos - t[..., 1::2] * sin
            out[..., 1::2] = t[..., 1::2] * cos + t[..., 0::2] * sin
            return out
        q, k = rot(q), rot(k)
    q, k, v = bf16(q, rounding), bf16(k, rounding), bf16(v, rounding)
    if drop_last_key:
        k, v = k[..., :-1, :], v[..., :-1, :]
    s = q @ k.transpose(-1, -2)                                   # log2 units
    p = torch.exp2(s - s.max(-1, keepdim=True).values)
    o = (bf16(p, rounding) @ v) / p.sum(-1, keepdim=True)
    o = bf16(o, rounding).permute(0, 2, 1, 3).reshape(nseq, length, a_dim)
    return o @ bf16(wo, rounding).t()


def encoder(spec: torch.Tensor, w, b, gw, gb, eps: float, rounding: bool = True) -> torch.Tensor:
    """Conv2d(2, C, 3x3) + GroupNorm(1, C) of spec [B, Tf, F, 2] as enc_conv_mma_kernel computes it."""
    bsz, tf, nf, cin = spec.shape
    xp = torch.zeros(bsz, tf + 2, nf + 2, cin, dtype=F64)
    xp[:, 1:-1, 1:-1] = tf32(spec, rounding)
    w = tf32(w, rounding)
    y = b.to(F64).expand(bsz, tf, nf, -1).clone()
    for dt in range(3):
        for df in range(3):
            y = y + xp[:, dt:dt + tf, df:df + nf] @ w[:, :, dt, df].t()
    mean = y.mean(dim=(1, 2, 3), keepdim=True)
    var = ((y - mean) ** 2).mean(dim=(1, 2, 3), keepdim=True)
    return (y - mean) / torch.sqrt(var + eps) * gw.to(F64) + gb.to(F64)


def decoder(x: torch.Tensor, w, b, rounding: bool = True) -> torch.Tensor:
    """ConvTranspose2d(C, 2S, 3x3, padding 1) of x [B, Tf, F, C] as the tf32 decoders compute it -> [B, Tf, F, 2S]."""
    bsz, tf, nf, c = x.shape
    xp = torch.zeros(bsz, tf + 2, nf + 2, c, dtype=F64)
    xp[:, 1:-1, 1:-1] = tf32(x, rounding)
    w = tf32(w, rounding)
    y = b.to(F64).expand(bsz, tf, nf, -1).clone()
    for dt in range(3):
        for df in range(3):
            y = y + xp[:, 2 - dt:2 - dt + tf, 2 - df:2 - df + nf] @ w[:, :, dt, df]
    return y


def per_sequence_errors(got: torch.Tensor, ref: torch.Tensor) -> Tuple[float, float, int]:
    """got, ref [Nseq, ...]: worst per-sequence relative L2 error, worst per-sequence max |err| / RMS(ref), and the
    index of the sequence with the worst relative L2."""
    got, ref = got.to(F64).reshape(got.shape[0], -1), ref.to(F64).reshape(ref.shape[0], -1)
    err = got - ref
    ref_norm = ref.norm(dim=1).clamp_min(1e-300)
    rel = err.norm(dim=1) / ref_norm
    rms = ref_norm / math.sqrt(ref.shape[1])
    mx = err.abs().max(dim=1).values / rms
    return float(rel.max()), float(mx.max()), int(rel.argmax())
