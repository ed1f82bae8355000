"""CPU self-tests of tests/bf16_ref.py: without rounding it is the float64 oracle; its roundings are bf16 / tf32."""
import math

import numpy as np
import pytest
import torch

import bf16_ref
import oracle


def _weights(c, hid, k, a_dim, seed):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    return dict(gamma=1 + 0.1 * r(c), w1=r(2 * hid, c, k) / math.sqrt(c * k), b1=0.1 * r(2 * hid),
                w2=r(hid, c, k) / math.sqrt(hid * k), b2=0.1 * r(c), wqkv=r(3 * a_dim, c) / math.sqrt(c),
                wo=r(c, a_dim) / math.sqrt(a_dim))


@pytest.mark.parametrize("c,groups,hid,k", [(32, 4, 64, 4), (48, 1, 32, 1), (64, 8, 64, 8)])
def test_ffn_without_rounding_is_the_oracle(c, groups, hid, k):
    w = _weights(c, hid, k, c, seed=c + k)
    x = torch.randn(3, 11, c, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    xn = oracle.rms_group_norm(x, w["gamma"], groups, 1e-5)
    want = oracle.swiglu_conv_deconv(xn, w["w1"], w["b1"], w["w2"], w["b2"])
    got = bf16_ref.ffn_branch(x, w["gamma"], w["w1"], w["b1"], w["w2"], w["b2"], groups, 1e-5, rounding=False)
    assert float((got - want).abs().max()) < 1e-12


@pytest.mark.parametrize("c,groups,heads,hd,rope", [(32, 4, 2, 16, True), (48, 2, 4, 12, False), (64, 1, 3, 24, True)])
def test_attention_without_rounding_is_the_oracle(c, groups, heads, hd, rope):
    a_dim = heads * hd
    w = _weights(c, 8, 1, a_dim, seed=c + heads)
    freqs = oracle.rope.rope_freqs(hd) if rope else None
    x = torch.randn(2, 130, c, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    xn = oracle.rms_group_norm(x, w["gamma"], groups, 1e-5)
    want = oracle.attention(xn, w["wqkv"], w["wo"], heads, freqs)
    got = bf16_ref.attention_branch(x, w["gamma"], w["wqkv"], w["wo"], heads, freqs, groups, 1e-5, rounding=False)
    assert float((got - want).abs().max()) < 1e-12


def test_encoder_and_decoder_without_rounding_are_the_oracle():
    g = torch.Generator().manual_seed(3)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    spec, w, b, gw, gb = r(2, 5, 17, 2), r(24, 2, 3, 3), r(24), r(24), r(24)
    want = oracle.encoder(spec, w, b, gw, gb, 1e-5)
    assert float((bf16_ref.encoder(spec, w, b, gw, gb, 1e-5, rounding=False) - want).abs().max()) < 1e-12
    x, wd, bd = r(2, 5, 17, 24), r(24, 6, 3, 3), r(6)
    want = oracle.decoder(x, wd, bd)
    assert float((bf16_ref.decoder(x, wd, bd, rounding=False) - want).abs().max()) < 1e-12


def _tie_cases(mant_bits):
    """fp32 values exactly halfway between two representable values of a format with `mant_bits` explicit bits, and
    their neighbours one fp32 ulp away, for both signs."""
    drop = 23 - mant_bits
    base = np.array([0x3F800000, 0x40490000, 0x3A123000, 0x7E000000, 0x00800000], dtype=np.int64)
    base = base & ~((1 << drop) - 1)
    half = 1 << (drop - 1)
    odd = base | (1 << drop)                       # last kept bit set: ties-to-even and ties-away differ here
    bits = np.concatenate([base + half, odd + half, base + half - 1, base + half + 1, odd + half + 1])
    v = bits.astype(np.uint32).view(np.float32)
    return torch.from_numpy(np.concatenate([v, -v]))


def test_bf16_rounding_is_torch_bfloat16():
    g = torch.Generator().manual_seed(4)
    x = torch.cat([torch.randn(10000, generator=g) * 10.0 ** torch.randint(-20, 20, (10000,), generator=g),
                   _tie_cases(7)])
    want = x.to(torch.bfloat16).to(torch.float64)
    assert torch.equal(bf16_ref.bf16(x), want)
    assert torch.equal(bf16_ref.bf16(x.double()), want)          # a float64 operand is first an fp32 value, as in the kernels


def _tf32_by_frexp(v: float) -> float:
    """Nearest value with 11 significant bits, halfway cases away from zero (cvt.rna.tf32.f32)."""
    if v == 0.0:
        return v
    m, e = math.frexp(abs(v))                     # abs(v) = m * 2^e, m in [0.5, 1)
    q = math.floor(m * 2048.0 + 0.5)
    return math.copysign(math.ldexp(q, e - 11), v)


def test_tf32_rounding_is_round_to_nearest_ties_away():
    g = torch.Generator().manual_seed(5)
    x = torch.cat([torch.randn(5000, generator=g) * 10.0 ** torch.randint(-20, 20, (5000,), generator=g),
                   _tie_cases(10)])
    got = bf16_ref.tf32(x)
    want = torch.tensor([_tf32_by_frexp(float(v)) for v in x], dtype=torch.float64)
    assert torch.equal(got, want)
    # tf32 keeps 10 explicit bits: the 13 low bits of the fp32 pattern are zero
    assert int((got.float().view(torch.int32) & 0x1FFF).abs().max()) == 0


def test_per_sequence_errors_see_one_bad_sequence():
    """A corrupted row in one sequence of many moves that sequence's statistics past the gates."""
    g = torch.Generator().manual_seed(6)
    ref = torch.randn(50, 20, 16, generator=g, dtype=torch.float64)
    ref[7] *= 0.01                                  # a quiet sequence: a global maximum would not see its error
    got = ref.clone()
    got[7, 3] += 0.01 * 0.05
    rel, mx, worst = bf16_ref.per_sequence_errors(got, ref)
    assert worst == 7 and rel > 2 * bf16_ref.REL_L2 and mx > 2 * bf16_ref.MAX_OVER_RMS
    rel, mx, _ = bf16_ref.per_sequence_errors(ref, ref)
    assert rel == 0.0 and mx == 0.0
