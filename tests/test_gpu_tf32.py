"""The tf32 precision mode (TFL_PRECISION_TF32): the tcgen05 kind::tf32 tap-GEMM of the ConvSwiGLU FFN against a float64
reference that rounds to tf32 exactly where the kernel does, the encoder / decoder it shares with the bf16 mode, end-to-end
accuracy against the fp32 mode, and bitwise properties.

FFN gates.  The reference rounds the normalised input, both weights and the SwiGLU hidden to tf32 (cvt.rna) and sums
in float64.  It cannot reproduce the rounding of the hidden exactly: the kernel rounds an fp32 hidden whose K*C-term
sum the tensor core accumulated in its own order (the mode-3 self-test measures up to ~1e-6 of sum |products|, i.e.
~1e-5 of |h| after cancellation), so a few percent of the hidden values land on the other side of a tf32 rounding
boundary and move by one tf32 ulp (2^-10 .. 2^-11 relative).  That is noise the reference cannot model: computing the
hidden in float32 on the CPU instead of float64 (another valid fp32 summation order) moves the branch by up to 1e-4
(relative L2) and 2e-4 (max / RMS) on a sequence of length 2, where only a few hundred outputs average the flips.
  * per sequence (as in test_gpu_bf16_sweep.py): REL_L2_TF32 = 5e-4, MAX_OVER_RMS_TF32 = 2e-3 -- about twice the worst
    seen on a B200 over the sweep below (2.7e-4 on length-2 sequences, 8.9e-4);
  * per call, over all sequences, wherever a call has >= CALL_MIN_OUTPUTS outputs (the flips average out):
    REL_L2_CALL = 8e-5 at K*C = 512 (Variant D's conv1d), against ~5e-5 measured there.  The flip rate grows with the
    relative fp32 error of the hidden, i.e. with the cancellation sqrt(K*C), and the branch error with the square root
    of the flip rate, so the gate scales as (K*C / 512)^(1/4) above 512 (x1.41 at K*C = 8 * 256).
A reference without tf32 rounding is off by ~5e-4 (2^-11 / sqrt(3) per rounded operand), one with the hidden left
unrounded by ~2e-4.  The per-sequence gates are too wide to tell those apart on short sequences; the per-call gate is
not: test_gates_discriminate checks that both wrong references fail it by at least 2x, and the sweep applies it.
"""
import os

import pytest
import torch

import bf16_ref
from bf16_ref import tf32
from conftest import load_golden
from test_gpu_bf16_sweep import _cfg, _model, _seqs
from test_gpu_parity import VARIANT_D, _mixture, _random_model

pytestmark = pytest.mark.gpu

FP32, BF16, TF32 = 0, 1, 2
REL_L2_TF32 = 5e-4
MAX_OVER_RMS_TF32 = 2e-3
REL_L2_CALL = 8e-5
CALL_MIN_OUTPUTS = 32768
SISDR_TF32 = 40.0
PATHS = ("freq_path", "frame_path")
F64 = torch.float64


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available()
    return m


# ---- self-test mode 3 -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("taps", [1, 4, 8])
@pytest.mark.parametrize("N", [16, 64, 256])
@pytest.mark.parametrize("Kd", [8, 64, 512])
def test_selftest_mode3(pkg, taps, N, Kd):
    """D[128, N] = sum_tap A[m + tap, :] . B[tap][n, :] on the tf32 tap-GEMM, against float64 on tf32-rounded operands;
    what is left is fp32 accumulation of n = taps * Kd products, bounded by n * 2^-23 * sum |products| (truncating
    additions included).  At small n that bound is far below the 2^-12 relative error of an unrounded operand."""
    from mss_tf_locoformer_b200.engine import tc_selftest
    g = torch.Generator().manual_seed(taps * 100000 + N * 1000 + Kd)
    A = torch.randn(128 + taps - 1, Kd, generator=g)
    B = torch.randn(taps, N, Kd, generator=g)
    D = tc_selftest(A.cuda(), B.cuda(), taps, 3).cpu().double()
    At, Bt = tf32(A), tf32(B)
    want = sum(At[t:t + 128] @ Bt[t].T for t in range(taps))
    bound = sum(At[t:t + 128].abs() @ Bt[t].abs().T for t in range(taps))
    err = (D - want).abs()
    print(f"taps {taps} N {N} Kd {Kd}: max |err| / sum|products| {float((err / bound).max()):.2e}")
    assert bool((err <= taps * Kd * 2.0 ** -23 * bound).all())


# ---- FFN sub-block ----------------------------------------------------------------------------------------------------
def ffn_tf32_ref(sd, cfg, x, axis, j=0, round_ops=True, round_hidden=True):
    """ConvSwiGLU(RMSGroupNorm(x)) of the sequences of x along `axis` in float64, rounded to tf32 where the tf32 mode
    rounds: the normalised input, conv1d.weight, deconv1d.weight and the SwiGLU hidden."""
    p = f"blocks.0.{PATHS[axis]}"
    gamma, w1, b1 = sd[f"{p}.ffn_norm.{j}.gamma"], sd[f"{p}.ffn.{j}.conv1d.weight"], sd[f"{p}.ffn.{j}.conv1d.bias"]
    w2, b2 = sd[f"{p}.ffn.{j}.deconv1d.weight"], sd[f"{p}.ffn.{j}.deconv1d.bias"]
    xs = _seqs(x, axis).to(F64)
    nseq, s, c = xs.shape
    two_h, _, k = w1.shape
    hid = two_h // 2
    a = tf32(xs * bf16_ref._inv_rms(xs, cfg["num_groups"], cfg["eps"]) * gamma.to(F64), round_ops)
    w1, w2 = tf32(w1, round_ops), tf32(w2, round_ops)
    xp = torch.zeros(nseq, s + 2 * (k - 1), c, dtype=F64)
    xp[:, k - 1:k - 1 + s] = a
    hlen = s + k - 1
    h = b1.to(F64).expand(nseq, hlen, -1).clone()
    for kk in range(k):
        h = h + xp[:, kk:kk + hlen] @ w1[:, :, kk].t()
    gate = h[..., hid:]
    g = tf32(h[..., :hid] * (gate * torch.sigmoid(gate)), round_ops and round_hidden)
    out = b2.to(F64).expand(nseq, s, -1).clone()
    for kk in range(k):
        out = out + g[:, (k - 1) - kk:(k - 1) - kk + s] @ w2[:, :, kk]
    return out


def _ffn_got(eng, x, axis, j):
    return _seqs(eng.ffn_(0, axis, j, x.cuda().clone(), TF32).cpu().double() - x.double(), axis)


def _rel_call(got, want):
    return float((got - want).norm() / want.norm())


def _call_gate(k, c):
    return REL_L2_CALL * max(1.0, k * c / 512.0) ** 0.25


def _gate(got, want, what, k, c):
    rel, mx, worst = bf16_ref.per_sequence_errors(got, want)
    call = _rel_call(got, want)
    print(f"{what}: rel L2 {rel:.2e}, max/RMS {mx:.2e} (sequence {worst}); per call {call:.2e}")
    assert rel <= REL_L2_TF32 and mx <= MAX_OVER_RMS_TF32, (what, rel, mx, worst)
    if got.numel() >= CALL_MIN_OUTPUTS:
        assert call <= _call_gate(k, c), (what, call)


# (emb, groups, K, hidden, [B, Tf, F]): norm groups of 4 .. 128 channels, K 1 / 2 / 4 / 8, hidden 64 .. 1024; both axes
# see the lengths Tf and F: 1, 2, 125 .. 131, 259, 1025, 2049, with at least two sequences per call
FFN_CASES = [
    (32, 8, 4, 64, (2, 1, 2)),
    (48, 4, 8, 192, (2, 2, 1)),
    (64, 1, 2, 384, (2, 3, 125)),
    (96, 2, 1, 384, (2, 2, 126)),
    (128, 4, 4, 384, (2, 2, 127)),
    (128, 1, 4, 384, (2, 2, 128)),
    (256, 8, 8, 1024, (2, 2, 129)),
    (256, 2, 4, 1024, (2, 2, 130)),
    (64, 4, 8, 192, (2, 131, 2)),
    (128, 32, 2, 64, (1, 259, 3)),
    (128, 4, 4, 384, (2, 2, 1025)),
    (96, 24, 8, 1024, (1, 2049, 2)),
]


@pytest.mark.parametrize("emb,groups,k,hidden,shape", FFN_CASES)
def test_ffn_against_tf32_reference(pkg, emb, groups, k, hidden, shape):
    cfg = _cfg(emb, groups, heads=8 if emb == 256 else 4, hidden=hidden, k=k)
    eng, sd = _model(pkg, cfg)
    x = torch.randn(*shape, emb, generator=torch.Generator().manual_seed(emb + k + hidden))
    for axis in (0, 1):
        for j in (0, 1):
            _gate(_ffn_got(eng, x, axis, j), ffn_tf32_ref(sd, cfg, x, axis, j),
                  f"ffn emb {emb} groups {groups} K {k} hidden {hidden} {shape} axis {axis} j {j}", k, emb)


def test_ffn_out_of_place_matches_in_place(pkg):
    cfg = _cfg(128, 4)
    eng, _ = _model(pkg, cfg)
    x = torch.randn(2, 3, 129, 128, generator=torch.Generator().manual_seed(5)).cuda()
    y = torch.empty_like(x)
    assert torch.equal(eng.ffn_out(0, 1, 0, x, y, TF32), eng.ffn_(0, 1, 0, x.clone(), TF32))


def test_gates_discriminate(pkg):
    """The per-call gate passes the kernel against the tf32 reference and rejects, by >= 2x, a reference without tf32
    rounding and one that leaves the hidden unrounded."""
    cfg = _cfg(128, 4)
    eng, sd = _model(pkg, cfg)
    x = torch.randn(2, 67, 131, 128, generator=torch.Generator().manual_seed(9))
    for axis in (0, 1):
        got = _ffn_got(eng, x, axis, 0)
        rel = _rel_call(got, ffn_tf32_ref(sd, cfg, x, axis, 0))
        print(f"axis {axis} vs the tf32 reference: per-call rel L2 {rel:.2e}")
        assert rel <= REL_L2_CALL, (axis, rel)
        for name, kw in (("no rounding", dict(round_ops=False)), ("hidden unrounded", dict(round_hidden=False))):
            rel = _rel_call(got, ffn_tf32_ref(sd, cfg, x, axis, 0, **kw))
            print(f"axis {axis} vs reference with {name}: per-call rel L2 {rel:.2e}")
            assert rel >= 2 * REL_L2_CALL, (name, axis, rel)


# ---- encoder / decoder ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("emb,shape", [(128, (2, 7, 1025)), (96, (1, 5, 129)), (48, (2, 3, 65))])
def test_encoder_decoder_equal_bf16_mode(pkg, emb, shape):
    cfg = dict(VARIANT_D, emb_dim=emb, attention_dim=emb)
    eng = _random_model(pkg, cfg).cuda().eval()._ready()
    g = torch.Generator().manual_seed(emb)
    spec = torch.randn(*shape, 2, generator=g).cuda()
    assert torch.equal(eng.enc_conv_gln(spec, TF32), eng.enc_conv_gln(spec, BF16))
    x = torch.randn(*shape, emb, generator=g).cuda()
    assert torch.equal(eng.dec_conv(x, TF32), eng.dec_conv(x, BF16))


# ---- end to end -------------------------------------------------------------------------------------------------------
def _sisdr_worst(est, ref):
    """Worst SI-SDR (dB) over the leading rows of est / ref (complex tensors are compared as (re, im) pairs)."""
    if est.is_complex():
        est, ref = torch.view_as_real(est), torch.view_as_real(ref)
    e = est.reshape(est.shape[0], -1).double().cpu()
    r = ref.reshape(ref.shape[0], -1).double().cpu()
    a = (e * r).sum(1, keepdim=True) / (r * r).sum(1, keepdim=True)
    t = a * r
    return float((10 * torch.log10((t * t).sum(1) / ((e - t) ** 2).sum(1))).min())


def _compare(run, what, bf16_runs=True):
    ref = run("fp32")
    db_tf32 = _sisdr_worst(run("tf32"), ref)
    line = f"{what}: tf32 vs fp32 {db_tf32:.1f} dB"
    if bf16_runs:
        db_bf16 = _sisdr_worst(run("bf16"), ref)
        line += f", bf16 vs fp32 {db_bf16:.1f} dB"
    print(line)
    assert db_tf32 >= SISDR_TF32, (what, db_tf32)
    if bf16_runs:
        assert db_tf32 > db_bf16, (what, db_tf32, db_bf16)


def _mss_runner(model, mix):
    def run(prec):
        model.precision = prec
        with torch.no_grad():
            out = model(mix)
        return torch.stack([out[k] for k in out]).transpose(0, 1)     # [B, S, T]: one row per sample
    return run


XLARGE = dict(VARIANT_D, n_fft=4096, hop_length=1024, emb_dim=256, num_groups=8, n_heads=16, attention_dim=256,
              ffn_hidden_dim=[1024, 1024], conv1d_kernel=4)


@pytest.mark.parametrize("name,cfg,n_samples,bf16_runs", [
    ("variant_d", dict(VARIANT_D, n_layers=2), 44100, True),
    ("xlarge_1layer", dict(XLARGE, n_layers=1), 44100, False),
    ("xlarge_2layers", dict(XLARGE, n_layers=2), 30000, False),
])
def test_mss_end_to_end(pkg, name, cfg, n_samples, bf16_runs):
    """TFLocoformerMSS; the xlarge widths (16 heads x 16) have no bf16 attention, so only the 40 dB gate applies."""
    model = _random_model(pkg, cfg).cuda().eval()
    mix = _mixture(n_samples, 2).cuda()
    _compare(_mss_runner(model, mix), name, bf16_runs)
    if not bf16_runs:
        model.precision = "bf16"
        with pytest.raises(Exception):
            with torch.no_grad():
                model(mix)


SEP = dict(num_spk=2, n_layers=2, emb_dim=48, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           attention_dim=48, pos_enc="rope", ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[192, 192],
           conv1d_kernel=8)


def _perturbed(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.ndim == 1 and not n.endswith("rope.freqs"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    return model


def _spec(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.complex(torch.randn(*shape, generator=g), torch.randn(*shape, generator=g))


def test_separator_end_to_end(pkg):
    model = _perturbed(pkg.TFLocoformerSeparator(**SEP), 1).cuda().eval()
    spec = _spec((2, 40, 129), 2).cuda()

    def run(prec):
        model.precision = prec
        with torch.no_grad():
            return model(spec).transpose(0, 1).reshape(2 * 2, -1)
    _compare(run, "TFLocoformerSeparator")


@pytest.mark.parametrize("n_freq", [65, 129])
def test_espnet_adapter_end_to_end(pkg, n_freq):
    from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as Esp
    model = _perturbed(Esp(n_freq, **SEP), 3).cuda().eval()
    spec = _spec((2, 30, n_freq), 4).cuda()
    ilens = torch.tensor([30, 30])

    def run(prec):
        model.precision = prec
        with torch.no_grad():
            outs, _, _ = model(spec, ilens)
        return torch.stack(outs)
    _compare(run, f"ESPnet adapter F={n_freq}")


def test_bs_locoformer_end_to_end(pkg):
    cfg = dict(SEP, conv1d_kernel=4, sample_rate=44100, stft_size=256)
    model = _perturbed(pkg.BSLocoformerSeparator(**cfg), 5).cuda().eval()
    spec = _spec((2, 24, 129), 6).cuda()

    def run(prec):
        model.precision = prec
        with torch.no_grad():
            return model(spec).transpose(0, 1).reshape(2 * 2, -1)
    _compare(run, "BSLocoformerSeparator")


def test_cli_tf32(pkg, tmp_path):
    """separate.py --precision tf32 writes every source; each is within 40 dB SI-SDR of the fp32 run's."""
    import yaml
    from mss_tf_locoformer_b200 import separate as cli
    cfg, sd, _ = load_golden("mss_hop2_macaron")
    ckpt = os.path.join(tmp_path, "model.pt")
    torch.save({"model_state_dict": sd, "epoch": 3}, ckpt)
    ycfg = os.path.join(tmp_path, "cfg.yaml")
    with open(ycfg, "w") as f:
        yaml.safe_dump({"model": cfg}, f)
    sr = 8000
    wav = os.path.join(tmp_path, "song.wav")
    cli.save_audio(torch.stack([_mixture(9000, 1, seed=1)[0], _mixture(9000, 1, seed=2)[0]]), wav, sample_rate=sr,
                   normalize=False)
    outs = {}
    for prec in ("fp32", "tf32"):
        out_dir = os.path.join(tmp_path, prec)
        cli.main(["--input", wav, "--checkpoint", ckpt, "--config", ycfg, "--output_dir", out_dir,
                  "--sample_rate", str(sr), "--segment", str(1024 / sr), "--batch", "3", "--precision", prec])
        outs[prec] = {f: cli.load_audio(os.path.join(out_dir, f), sample_rate=sr)[0]
                      for f in sorted(os.listdir(out_dir))}
    assert list(outs["tf32"]) == list(outs["fp32"]) and len(outs["tf32"]) >= 2
    for f in outs["fp32"]:
        db = _sisdr_worst(outs["tf32"][f], outs["fp32"][f])
        print(f"cli {f}: tf32 vs fp32 {db:.1f} dB")
        assert db >= SISDR_TF32, (f, db)


# ---- bitwise properties -----------------------------------------------------------------------------------------------
def test_bitwise_repeat_and_batch_position(pkg):
    model = _random_model(pkg, dict(VARIANT_D, n_layers=2)).cuda().eval()
    model.precision = "tf32"
    mix = _mixture(30000, 3).cuda()
    with torch.no_grad():
        a = torch.stack(list(model(mix).values()))
        b = torch.stack(list(model(mix).values()))
        alone = torch.stack(list(model(mix[1:2]).values()))
    assert torch.equal(a, b)
    assert torch.equal(a[:, 1:2], alone)


def test_no_state_leaks_between_modes(pkg):
    model = _random_model(pkg, dict(VARIANT_D, n_layers=1)).cuda().eval()
    mix = _mixture(30000, 2).cuda()

    def run(prec):
        model.precision = prec
        with torch.no_grad():
            return torch.stack(list(model(mix).values()))
    before = {p: run(p) for p in ("fp32", "bf16")}
    run("tf32")
    for p in ("fp32", "bf16"):
        assert torch.equal(run(p), before[p]), p
