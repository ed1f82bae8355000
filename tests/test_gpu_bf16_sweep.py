"""The bf16 kernels swept over norm-group widths, head shapes, sequence edges and kernel variants, against the
rounding-aware float64 reference of tests/bf16_ref.py (gates and their derivation: bf16_ref's docstring).

Every sub-block is compared per sequence (relative L2 of the branch and max |error| / RMS of that sequence), so a
fault confined to a few rows, channels or one sequence cannot hide behind the others.  The fp32 mode is checked at the
same shapes with the 1e-4 max-abs gate of test_gpu_parity.py.  Bitwise properties catch what a tolerance cannot:
reads of stale shared memory (run-to-run differences) and dependence on a sequence's place in the batch.
"""
import contextlib
import math
import os

import pytest
import torch

import bf16_ref
import oracle
from bf16_ref import MAX_OVER_RMS, MAX_OVER_RMS_ATTN, REL_L2, REL_L2_ATTN
from conftest import load_golden
from test_gpu_parity import FP32_MAXABS, VARIANT_D, _mixture, _random_model

pytestmark = pytest.mark.gpu

OPT_ATTN, OPT_FFN, OPT_TAIL, OPT_PDL = 0, 1, 3, 4          # include/tfl.h TFL_OPT_*
PATHS = ("freq_path", "frame_path")


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available()
    return m


@contextlib.contextmanager
def option(key, value):
    """tfl_debug_set_option for the duration of a block; the default is restored however the block ends."""
    from mss_tf_locoformer_b200 import _lib
    lib = _lib.load()
    default = (1 if os.environ.get("TFL_PDL") else 0) if key == OPT_PDL else 2
    assert lib.tfl_debug_set_option(key, value) == 0
    try:
        yield
    finally:
        lib.tfl_debug_set_option(key, default)


def _cfg(emb, groups, heads=4, hd=None, hidden=384, k=4, pos="rope"):
    return dict(VARIANT_D, emb_dim=emb, num_groups=groups, n_heads=heads, attention_dim=heads * (hd or emb // heads),
                ffn_hidden_dim=[hidden, hidden], conv1d_kernel=k, pos_enc=pos)


def _model(pkg, cfg, seed=0):
    model = _random_model(pkg, cfg, seed)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.cuda().eval()
    return model._ready(), sd


def _seqs(x, axis):
    """[B, Tf, F, C] -> [Nseq, L, C] in the order the sub-block sees its sequences."""
    b, tf, nf, c = x.shape
    return x.reshape(b * tf, nf, c) if axis == 0 else x.transpose(1, 2).reshape(b * nf, tf, c)


def _ffn_ref(sd, cfg, x, axis, j=0, rounding=True, **over):
    p = f"blocks.0.{PATHS[axis]}"
    w = dict(gamma=sd[f"{p}.ffn_norm.{j}.gamma"], w1=sd[f"{p}.ffn.{j}.conv1d.weight"], b1=sd[f"{p}.ffn.{j}.conv1d.bias"],
             w2=sd[f"{p}.ffn.{j}.deconv1d.weight"], b2=sd[f"{p}.ffn.{j}.deconv1d.bias"], eps=cfg["eps"])
    w.update(over)
    return bf16_ref.ffn_branch(_seqs(x, axis), w["gamma"], w["w1"], w["b1"], w["w2"], w["b2"], cfg["num_groups"],
                               w["eps"], rounding)


def _attn_ref(sd, cfg, x, axis, rounding=True, gamma=None, **kw):
    p = f"blocks.0.{PATHS[axis]}"
    freqs = sd.get(f"{p}.attn.rope.freqs") if cfg["pos_enc"] == "rope" else None
    return bf16_ref.attention_branch(_seqs(x, axis), sd[f"{p}.attn_norm.gamma"] if gamma is None else gamma,
                                     sd[f"{p}.attn.qkv.weight"], sd[f"{p}.attn.aggregate_heads.0.weight"],
                                     cfg["n_heads"], freqs, cfg["num_groups"], cfg["eps"], rounding, **kw)


def _ffn_got(eng, x, axis, j=0, precision=1):
    return _seqs(eng.ffn_(0, axis, j, x.cuda().clone(), precision).cpu().double() - x.double(), axis)


def _attn_got(eng, x, axis, precision=1):
    return _seqs(eng.attn_(0, axis, x.cuda().clone(), precision).cpu().double() - x.double(), axis)


def _gates(what):
    """(relative L2, max / RMS) gates: the attention's are wider by the bf16 rounding of P (bf16_ref docstring)."""
    return (REL_L2_ATTN, MAX_OVER_RMS_ATTN) if what.startswith("attn") else (REL_L2, MAX_OVER_RMS)


def _gate(got, want, what):
    rel, mx, worst = bf16_ref.per_sequence_errors(got, want)
    print(f"{what}: rel L2 {rel:.2e}, max/RMS {mx:.2e} (sequence {worst})")
    g_rel, g_max = _gates(what)
    assert rel <= g_rel and mx <= g_max, (what, rel, mx, worst)
    return rel, mx


def _gate_fp32(got, want, what):
    err = float((got - want).abs().max())
    print(f"{what}: fp32 max-abs {err:.2e}")
    assert err <= FP32_MAXABS, (what, err)


# ---------------------------------------------------------------------------------------------------------------------
# norm-group width D = emb / groups: 4 ... 128 (the 2-CTA FFN takes D <= 32 only; qkv_tc has D == 32, D < 32, D > 32)
GROUP_WIDTHS = [(128, 4), (128, 2), (128, 1), (96, 2), (96, 1), (64, 1), (64, 8), (32, 8), (48, 4), (256, 8), (256, 4)]


def _x(shape, emb, seed=3, scale=1.0):
    return scale * torch.randn(*shape, emb, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("emb,groups", GROUP_WIDTHS)
def test_ffn_group_widths(pkg, emb, groups):
    """Both FFN kernels (TFL_OPT_FFN_KERNEL 1, 2; shapes the 2-CTA kernel does not take run on the 1-CTA one), both
    axes, both FFNs of the macaron block; fp32 mode at the same shape."""
    cfg = _cfg(emb, groups, heads=8 if emb == 256 else 4, hidden=1024 if emb == 256 else 384)
    eng, sd = _model(pkg, cfg)
    x = _x((1, 5, 131), emb)
    for axis in (0, 1):
        for j in (0, 1):
            want = _ffn_ref(sd, cfg, x, axis, j)
            for opt in (1, 2):
                with option(OPT_FFN, opt):
                    _gate(_ffn_got(eng, x, axis, j), want, f"ffn ({emb},{groups}) kernel {opt} axis {axis} j {j}")
            _gate_fp32(_ffn_got(eng, x, axis, j, 0), _ffn_ref(sd, cfg, x, axis, j, rounding=False),
                       f"ffn ({emb},{groups}) axis {axis} j {j}")


@pytest.mark.parametrize("emb,groups", [g for g in GROUP_WIDTHS if g[0] != 256])
def test_attention_group_widths(pkg, emb, groups):
    """qkv_tc's three producer branches (D == 32, D < 32, D > 32) through the whole attention sub-block, both axes
    (L = 131: three tail rows; L = 5), both attention kernels; fp32 mode at the same shape."""
    cfg = _cfg(emb, groups)
    eng, sd = _model(pkg, cfg)
    x = _x((1, 5, 131), emb)
    for axis in (0, 1):
        want = _attn_ref(sd, cfg, x, axis)
        for opt in (2, 1):
            with option(OPT_ATTN, opt):
                _gate(_attn_got(eng, x, axis), want, f"attn ({emb},{groups}) kernel {opt} axis {axis}")
        _gate_fp32(_attn_got(eng, x, axis, 0), _attn_ref(sd, cfg, x, axis, rounding=False),
                   f"attn ({emb},{groups}) axis {axis}")


# ---------------------------------------------------------------------------------------------------------------------
# attention geometry: (L, head_dim, heads, pos_enc).  L covers no tail / 1 / 2-8 / > 8 tail rows, NQT = 1, 2, >= 3
# (attn_tc2's QG = 1 / 2 / 4), partial head groups (heads % HG != 0) and L > 2304 (RoPE table built per call).
ATTN_CASES = [
    (1, 32, 4, "rope"), (2, 24, 3, "nope"), (3, 16, 6, "rope"), (16, 8, 2, "rope"), (17, 12, 6, "nope"),
    (17, 32, 3, "rope"), (127, 32, 1, "rope"), (128, 16, 8, "nope"), (129, 24, 1, "rope"), (130, 8, 8, "rope"),
    (130, 24, 3, "nope"), (136, 12, 4, "nope"), (137, 32, 2, "rope"), (256, 24, 3, "rope"), (256, 16, 6, "rope"),
    (257, 16, 2, "nope"), (259, 32, 1, "rope"), (259, 8, 6, "nope"), (385, 12, 6, "rope"), (1025, 24, 4, "rope"),
    (2305, 16, 4, "rope"), (2305, 32, 2, "nope"),
]


@pytest.mark.parametrize("L,hd,heads,pos", ATTN_CASES)
def test_attention_geometry(pkg, L, hd, heads, pos):
    cfg = _cfg(64, 4, heads=heads, hd=hd, hidden=64, pos=pos)
    eng, sd = _model(pkg, cfg)
    nseq = 2 if L <= 1025 else 1
    tail = L > 128 and 2 <= L % 128 <= 8
    for axis in (0, 1):
        x = _x((1, nseq, L) if axis == 0 else (1, L, nseq), 64, seed=L)
        want = _attn_ref(sd, cfg, x, axis)
        for opt in (2, 1):
            for tail_opt in ((2, 1) if tail else (2,)):
                with option(OPT_ATTN, opt), option(OPT_TAIL, tail_opt):
                    _gate(_attn_got(eng, x, axis), want, f"attn L {L} hd {hd} x{heads} {pos} kernel {opt} "
                                                         f"tail {tail_opt} axis {axis}")


def test_unsupported_attention_shape_raises(pkg):
    """16 heads x head_dim 16 = 256 projection columns exceed the tcgen05 attention (<= 128): a documented error."""
    from mss_tf_locoformer_b200._lib import TflError
    cfg = _cfg(256, 8, heads=16, hd=16, hidden=64)
    eng, _ = _model(pkg, cfg)
    with pytest.raises(TflError, match="bf16 tcgen05 attention needs"):
        eng.attn_(0, 0, _x((1, 2, 16), 256).cuda(), 1)


# ---------------------------------------------------------------------------------------------------------------------
# FFN geometry: conv kernel K, hidden width, sequence lengths around the tile period TS = 128 - (K - 1)
@pytest.mark.parametrize("k,hidden", [(1, 64), (2, 192), (4, 384), (8, 1024), (8, 64), (1, 1024)])
def test_ffn_geometry(pkg, k, hidden):
    cfg = _cfg(64, 4, hidden=hidden, k=k)
    eng, sd = _model(pkg, cfg)
    ts = 128 - (k - 1)
    for s in sorted({1, k - 1, ts - 1, ts, ts + 1, 2 * ts + 1} - {0}):
        x = _x((1, 3, s), 64, seed=s)
        want = _ffn_ref(sd, cfg, x, 0)
        for opt in (1, 2):
            with option(OPT_FFN, opt):
                _gate(_ffn_got(eng, x, 0), want, f"ffn K {k} H {hidden} S {s} kernel {opt}")


def test_ffn_persistent_loop(pkg):
    """700 sequences of TS + 1 rows: ~720 tiles, more than two per CTA of either kernel, so every CTA loops and reuses
    its A slots and accumulators."""
    cfg = _cfg(64, 4, hidden=64, k=4)
    eng, sd = _model(pkg, cfg)
    x = _x((1, 700, 126), 64, seed=700)
    want = _ffn_ref(sd, cfg, x, 0)
    for opt in (1, 2):
        with option(OPT_FFN, opt):
            _gate(_ffn_got(eng, x, 0), want, f"ffn persistent kernel {opt}")


# ---------------------------------------------------------------------------------------------------------------------
# encoder / decoder in bf16 mode (tf32 mma.sync).  Products of tf32 operands are exact in fp32; the encoder sums 18
# of them (decoder: 9 * C) in fp32, ~2^-24 * sqrt(terms) of the output scale, and the gLN statistics are double sums:
# 1e-5 relative (1e-4 max / RMS) leaves > 10x margin and is 100x below the tf32 rounding the reference models (2^-11).
TF32_REL, TF32_MAX = 1e-5, 1e-4


@pytest.mark.parametrize("emb,groups", [(40, 2), (64, 4), (128, 4)])
@pytest.mark.parametrize("nf", [15, 16, 17, 129, 1025])
def test_encoder_bf16_mode(pkg, emb, groups, nf):
    """enc_conv_mma_kernel against the tf32-rounded encoder, per sample (the gLN statistics are per sample)."""
    cfg = _cfg(emb, groups, heads=2, hidden=64)
    eng, sd = _model(pkg, cfg)
    for tf in (1, 2, 259):
        if nf * tf * emb > 2 ** 24:
            continue                                              # keeps the float64 reference under ~1 GB
        spec = _x((3, tf, nf), 2, seed=nf + tf)
        spec[1] *= 30.0                                           # samples of different loudness
        want = bf16_ref.encoder(spec, sd["conv.0.weight"], sd["conv.0.bias"], sd["conv.1.weight"], sd["conv.1.bias"],
                                cfg["eps"])
        got = eng.enc_conv_gln(spec.cuda(), 1).cpu().double()
        rel, mx, worst = bf16_ref.per_sequence_errors(got, want)
        print(f"encoder emb {emb} F {nf} Tf {tf}: rel {rel:.2e} max/RMS {mx:.2e}")
        assert rel <= TF32_REL and mx <= TF32_MAX, (tf, rel, mx, worst)
        loose, _, _ = bf16_ref.per_sequence_errors(got, bf16_ref.encoder(
            spec, sd["conv.0.weight"], sd["conv.0.bias"], sd["conv.1.weight"], sd["conv.1.bias"], cfg["eps"], False))
        assert loose > 10 * rel                                   # the tf32 rounding is what the reference models


@pytest.mark.parametrize("emb,shape", [(128, (2, 7, 129)), (96, (1, 9, 33)), (48, (3, 2, 17))])
def test_decoder_bf16_mode_tf32_reference(pkg, emb, shape):
    """Both tf32 decoders (TFL_OPT_DEC_KERNEL 2: scatter form where C % 32 == 0 and C <= 128, else and with 1: the 9-tap
    gather) against the tf32-rounded decoder."""
    cfg = _cfg(emb, 4, heads=2, hidden=64)
    eng, sd = _model(pkg, cfg)
    x = _x(shape, emb, seed=emb)
    want = bf16_ref.decoder(x, sd["deconv.weight"], sd["deconv.bias"])                  # [B, Tf, F, 2S]
    b, tf, nf, _ = want.shape
    want = want.reshape(b, tf, nf, -1, 2).permute(0, 3, 1, 2, 4)
    for opt in (2, 1):
        with option(6, opt):
            got = eng.dec_conv(x.cuda(), 1).cpu().double()
        rel, mx, _ = bf16_ref.per_sequence_errors(got, want)
        print(f"decoder emb {emb} kernel {opt}: rel {rel:.2e} max/RMS {mx:.2e}")
        assert rel <= TF32_REL and mx <= TF32_MAX, (opt, rel, mx)


# ---------------------------------------------------------------------------------------------------------------------
# exact properties
@pytest.mark.parametrize("emb,groups", [(128, 1), (128, 4), (96, 2)])
def test_repeated_calls_are_bitwise_identical(pkg, emb, groups):
    """The same call twice, with a call on other data in between, gives the same bits: a kernel that reads shared
    memory it never wrote (stale from the previous launch) fails this."""
    cfg = _cfg(emb, groups)
    eng, sd = _model(pkg, cfg)
    x, other = _x((1, 5, 131), emb).cuda(), _x((1, 5, 131), emb, seed=99, scale=7.0).cuda()
    for axis in (0, 1):
        for opt in (1, 2):
            with option(OPT_FFN, opt):
                a = eng.ffn_(0, axis, 0, x.clone(), 1)
                eng.ffn_(0, axis, 0, other.clone(), 1)
                assert torch.equal(a, eng.ffn_(0, axis, 0, x.clone(), 1)), ("ffn", opt, axis)
        a = eng.attn_(0, axis, x.clone(), 1)
        eng.attn_(0, axis, other.clone(), 1)
        assert torch.equal(a, eng.attn_(0, axis, x.clone(), 1)), ("attn", axis)


@pytest.mark.parametrize("emb,groups", [(128, 1), (128, 4)])
def test_sequence_result_does_not_depend_on_its_place(pkg, emb, groups):
    """A sequence gives the same bits whether it is first in the batch or after others (FFN kernels and attention,
    both axes): tile boundaries, CTA assignment and the stream's zero rows must not change a row's arithmetic."""
    cfg = _cfg(emb, groups)
    eng, _ = _model(pkg, cfg)
    perm = torch.tensor([8, 3, 0, 5, 1, 7, 2, 6, 4]).cuda()
    for axis in (0, 1):
        # nine sequences of 131 rows: axis 0 runs along F (sequences indexed by Tf), axis 1 along Tf (indexed by F)
        dim = 1 if axis == 0 else 2
        x = _x((1, 9, 131) if axis == 0 else (1, 131, 9), emb).cuda()
        calls = [lambda t: eng.attn_(0, axis, t, 1)] + [(lambda t, o=o: _with_ffn(eng, axis, t, o)) for o in (1, 2)]
        for n, call in enumerate(calls):
            full = call(x.clone())
            assert torch.equal(call(x.index_select(dim, perm)), full.index_select(dim, perm)), (axis, n)
            one = x.index_select(dim, perm[:1]).contiguous()
            assert torch.equal(call(one), full.index_select(dim, perm[:1])), (axis, n)


def _with_ffn(eng, axis, t, opt):
    with option(OPT_FFN, opt):
        return eng.ffn_(0, axis, 0, t, 1)


def test_pdl_does_not_change_bits(pkg):
    """Programmatic dependent launch changes when kernels start, never what they compute."""
    cfg = dict(_cfg(128, 1), n_layers=2)
    model = _random_model(pkg, cfg).cuda().eval()
    model.precision = "bf16"
    mix = _mixture(30000, 2).cuda()
    out = {}
    for pdl in (0, 1):
        with option(OPT_PDL, pdl), torch.no_grad():
            out[pdl] = model(mix)
    for k in out[0]:
        assert torch.equal(out[0][k], out[1][k]), k


# ---------------------------------------------------------------------------------------------------------------------
# end to end
@pytest.mark.parametrize("n_samples", [129, 130, 255, 256, 257, 1000, 1024, 4097])
def test_ragged_lengths_bf16(pkg, n_samples):
    """test_ragged_lengths_fp32's lengths (frames 2 ... 33, bins 129) in bf16: >= 40 dB against the oracle, and the rows
    of a batch bitwise equal to the same segments run alone."""
    cfg, sd, arr = load_golden("mss_hop2_macaron")
    model = pkg.TFLocoformerMSS(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    model.precision = "bf16"
    mix = _mixture(n_samples, 1, seed=n_samples)
    batch = torch.cat([mix, 0.5 * mix.flip(-1)], 0)
    want = oracle.mss_forward(sd, cfg, batch)
    with torch.no_grad():
        got = model(batch.cuda())
        alone = [model(batch[b:b + 1].cuda()) for b in range(2)]
    for k in want:
        for b in range(2):
            sdr = oracle.si_sdr_db(got[k][b].cpu(), want[k][b])
            assert sdr >= 40.0, (k, b, sdr)
            assert torch.equal(got[k][b], alone[b][k][0]), (k, b)


def test_separator_nope_k1_bf16(pkg):
    """sep_nope_k1's shape (one group of 32, one head, no RoPE, conv kernel 1) in bf16.  Its FFN hidden width 32 is not a
    multiple of the 64-channel chunk of the tcgen05 FFN: the golden model raises the documented error; with hidden 64
    (random weights) the bf16 forward is >= 40 dB from the oracle."""
    from mss_tf_locoformer_b200._lib import TflError
    cfg, sd, arr = load_golden("sep_nope_k1")
    model = pkg.TFLocoformerSeparator(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    model.precision = "bf16"
    with pytest.raises(TflError, match="bf16 tcgen05 FFN needs"), torch.no_grad():
        model(arr["spec_in"].cuda())
    cfg = dict(cfg, ffn_hidden_dim=[64, 64])
    torch.manual_seed(0)
    model = pkg.TFLocoformerSeparator(**cfg).eval()
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.ndim == 1:
                p.add_(0.1 * torch.randn(p.shape))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    want = oracle.separator_forward(sd, cfg, arr["spec_in"])
    model = model.cuda()
    model.precision = "bf16"
    with torch.no_grad():
        out = model(arr["spec_in"].cuda()).cpu()
    sdr = oracle.si_sdr_db(torch.view_as_real(out), torch.view_as_real(want))
    print(f"sep_nope_k1 shape, hidden 64, bf16: {sdr:.1f} dB")
    assert sdr >= 40.0, sdr


def test_mixed_training_step_one_group(pkg):
    """One mixed-mode training step (bf16 tcgen05 forward of the sub-blocks) at emb 64 with one norm group of 64
    channels -- wider than the 2-CTA FFN's A producers take -- against the float64 reference step."""
    from mss_tf_locoformer_b200.training import Trainer
    from test_gpu_training import SMALL, TOL, _rel, _reference_step
    cfg = dict(SMALL, n_layers=1, emb_dim=64, attention_dim=64, num_groups=1, ffn_hidden_dim=[64, 128])
    weights = (1.0, 0.1, 0.1)
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(5000, 2)
    g = torch.Generator().manual_seed(9)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(cfg["n_sources"], 2, 5000, generator=g)
    want_loss, want_grads, _ = _reference_step(cfg, sd, mix, tgt, weights)
    with option(5, 2):
        tr = Trainer(model.cuda(), si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
        loss, _ = tr.forward_backward(mix.cuda(), tgt.cuda(), want_audio=True)
    tol = TOL["mixed"]
    assert abs(float(loss[0]) - want_loss) <= tol["loss"] * max(1.0, abs(want_loss)), (float(loss[0]), want_loss)
    errs = {k: _rel(tr.grad_of(k), want_grads[k]) for k in want_grads}
    worst = max(errs, key=errs.get)
    print(f"mixed step, one group of 64: worst gradient error {errs[worst]:.2e} ({worst})")
    assert errs[worst] < tol["step"], (worst, errs[worst])


# ---------------------------------------------------------------------------------------------------------------------
# gate sensitivity: the kernel output must fail the gates against each deliberately wrong reference by >= 2x
@pytest.mark.parametrize("kind", ["rope_shift", "gamma_last_group", "conv_last_tap", "softmax_last_key", "b2_dropped",
                                  "eps_x10"])
def test_gates_reject_wrong_references(pkg, kind):
    cfg = _cfg(128, 4)
    eng, sd = _model(pkg, cfg)
    scale = 1e-3 if kind == "eps_x10" else 1.0                    # eps matters where the group RMS is near it
    x = _x((1, 4, 130), 128, scale=scale)
    p = "blocks.0.freq_path"
    what = ("attn " if kind in ("rope_shift", "softmax_last_key", "gamma_last_group") else "ffn ") + kind
    if what.startswith("attn"):
        got, right = _attn_got(eng, x, 0), _attn_ref(sd, cfg, x, 0)
        if kind == "rope_shift":
            pos = torch.arange(130)
            pos[128:] += 1
            wrong = _attn_ref(sd, cfg, x, 0, positions=pos)
        elif kind == "softmax_last_key":
            wrong = _attn_ref(sd, cfg, x, 0, drop_last_key=True)
        else:
            gamma = sd[f"{p}.attn_norm.gamma"].clone()
            gamma[-32:] = 1.0
            wrong = _attn_ref(sd, cfg, x, 0, gamma=gamma)
    else:
        got, right = _ffn_got(eng, x, 0), _ffn_ref(sd, cfg, x, 0)
        if kind == "conv_last_tap":
            w1 = sd[f"{p}.ffn.0.conv1d.weight"].clone()
            w1[:, :, -1] = 0.0
            wrong = _ffn_ref(sd, cfg, x, 0, w1=w1)
        elif kind == "b2_dropped":
            wrong = _ffn_ref(sd, cfg, x, 0, b2=torch.zeros(128))
        else:
            wrong = _ffn_ref(sd, cfg, x, 0, eps=10 * cfg["eps"])
    _gate(got, right, f"{what}: right reference")
    rel, mx, _ = bf16_ref.per_sequence_errors(got, wrong)
    g_rel, g_max = _gates(what)
    print(f"{what}: wrong reference rel L2 {rel:.2e} ({rel / g_rel:.0f}x gate), max/RMS {mx:.2e} ({mx / g_max:.0f}x gate)")
    assert rel >= 2 * g_rel and mx >= 2 * g_max, (kind, rel, mx)
