"""Training of TFLocoformerMSS through torch autograd, with gradients to the mixture and to the separator's input
spectrogram (``differentiable = True``; DESIGN.md section 8b).

Checker: float64 torch autograd on the CPU -- of the reference model when oracle/_ref is staged, else of
``oracle.mss_forward`` / ``oracle.separator_forward`` -- with ``loss = sum_s <audio_s, G_s>`` (or ``Re<est, G>``) for a
seeded G.  Every trainable parameter's ``.grad`` and the input gradient are compared by relative L2 error against the
whole-step gates of test_gpu_training.py (TOL[mode]["step"]) in the fp32, tf32 and mixed arithmetic of
TFL_OPT_TRAIN_MODE.  The mixture gradient is gated separately on its first n_fft/2 samples, its last n_fft/2 samples and
the rest: the reflect-padding fold only touches the two edges, and an error there must not hide in the global norm.
"""
import pytest
import torch

import oracle
from oracle import build_ref
from test_gpu_parity import VARIANT_D, _mixture, _random_model
from test_gpu_training import SMALL, TOL, _ref_loss, _rel

pytestmark = pytest.mark.gpu

MODES = {"fp32": 0, "tf32": 1, "mixed": 2}
NAMES = oracle.locoformer_oracle.SOURCE_NAMES


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available()
    return m


def _set_mode(mode):
    from mss_tf_locoformer_b200 import _lib
    assert _lib.load().tfl_debug_set_option(5, MODES[mode]) == 0


@pytest.fixture(params=["fp32", "tf32", "mixed"])
def train_mode(request, pkg):
    _set_mode(request.param)
    yield request.param
    _set_mode("mixed")


@pytest.fixture
def fp32_mode(pkg):
    _set_mode("fp32")
    yield "fp32"
    _set_mode("mixed")


def _seeded(shape, seed, complex_=False):
    g = torch.Generator().manual_seed(seed)
    if complex_:
        return torch.complex(torch.randn(*shape, generator=g), torch.randn(*shape, generator=g))
    return torch.randn(*shape, generator=g)


def _inner(out: dict, G: dict):
    """sum_s <out_s, G_s>; Re<., .> for complex outputs."""
    total = 0.0
    for k, v in out.items():
        g = G[k].to(v.device)
        total = total + ((v.real * g.real).sum() + (v.imag * g.imag).sum() if v.is_complex() else (v * g).sum())
    return total


def _cotangents(cfg, B, T, rtd, seed):
    S = cfg["n_sources"]
    if rtd:
        return {n: _seeded((B, T), seed + i) for i, n in enumerate(NAMES[:S])}
    Tf, F = 1 + T // cfg["hop_length"], cfg["n_fft"] // 2 + 1
    return {n: _seeded((B, F, Tf), seed + i, complex_=True) for i, n in enumerate(NAMES[:S])}


def _oracle_mss(cfg, sd, mix, G, rtd):
    """-> (outputs, {key: grad}, d mixture) of float64 CPU autograd."""
    mix64 = mix.double().clone().requires_grad_(True)
    G64 = {k: v.to(torch.complex128 if v.is_complex() else torch.float64) for k, v in G.items()}
    if build_ref.available():
        model = build_ref.load()["TFLocoformerMSS"](**cfg)
        model.load_state_dict(sd, strict=True)
        model = model.double().eval()
        out = model(mix64, return_time_domain=rtd)
        params = dict(model.state_dict(keep_vars=True))
    else:
        params = {k: v.detach().double().clone().requires_grad_(not k.endswith("rope.freqs")) for k, v in sd.items()}
        out = oracle.mss_forward(params, dict(cfg), mix64, return_time_domain=rtd, dtype=torch.float64)
    out = {k: v for k, v in out.items() if k in G64}
    _inner(out, G64).backward()
    return ({k: v.detach() for k, v in out.items()}, {k: p.grad for k, p in params.items() if p.grad is not None},
            mix64.grad)


def _check_forward(got, want, mode, what):
    got = torch.view_as_real(got.detach().cpu()) if got.is_complex() else got.detach().cpu()
    want = torch.view_as_real(want) if want.is_complex() else want
    got, want = got.double(), want.double()
    if mode == "fp32":
        err = float((got - want).abs().max())
        assert err <= 1e-4, (what, err)
    else:
        sd = oracle.si_sdr_db(got.reshape(1, -1), want.reshape(1, -1))
        assert sd >= 40.0, (what, sd)


def _check_grads(model, want, mode, what):
    """Relative L2 error per tensor.  A gradient that vanishes in exact arithmetic (deconv.bias under the iSTFT when T is a
    multiple of hop: every frame's bias term lands on a zero of the periodic Hann window) is measured against the largest
    gradient norm instead, since its float64 value is rounding noise."""
    got = dict(model.named_parameters())
    assert set(want) == {k for k, p in got.items() if p.requires_grad}, what
    scale = max(float(w.double().norm()) for w in want.values())
    errs = {k: _rel(got[k].grad, want[k]) if float(want[k].double().norm()) > 1e-9 * scale
            else float((got[k].grad.detach().double().cpu() - want[k].double()).norm()) / scale for k in want}
    worst = max(errs, key=errs.get)
    print(f"[{mode}] {what}: worst relative gradient error {errs[worst]:.2e} ({worst}) over {len(errs)} tensors")
    assert errs[worst] < TOL[mode]["step"], (what, worst, errs[worst])
    return errs[worst]


def _check_mixture_grad(got, want, pad, mode, what):
    """Relative L2 error on the left edge, the interior and the right edge (the interior is empty when T <= 2 pad)."""
    T = want.shape[-1]
    regions = {"left": slice(0, pad), "right": slice(T - pad, T)}
    if T > 2 * pad:
        regions["interior"] = slice(pad, T - pad)
    errs = {r: _rel(got[:, s], want[:, s]) for r, s in regions.items()}
    print(f"[{mode}] {what}: mixture gradient errors " + ", ".join(f"{r} {e:.2e}" for r, e in errs.items()))
    for r, e in errs.items():
        assert e < TOL[mode]["step"], (what, r, e)


MSS_CASES = [
    (dict(SMALL, n_sources=2), 2560, 2, True),                                                        # T = 20 hops
    (dict(SMALL, n_sources=1, pos_enc="nope", tf_order="tf", ffn_type="swiglu_conv1d", ffn_hidden_dim=64,
          conv1d_kernel=1), 2000, 2, True),                                                          # T % hop != 0
    (dict(SMALL, tf_order="tf", conv1d_kernel=8), 129, 2, False),                                    # T = n_fft/2 + 1
    (dict(VARIANT_D, flash_attention=False), 24000, 1, True),                                        # Variant-D widths
]


@pytest.mark.parametrize("cfg,T,B,rtd", MSS_CASES, ids=["macaron_rope_ft_k4_s2", "single_nope_tf_k1_s1_ragged",
                                                       "macaron_rope_tf_k8_s4_spectral_min_len", "variant_d_widths"])
def test_mss_gradients_vs_oracle_autograd(pkg, train_mode, cfg, T, B, rtd):
    """TFLocoformerMSS: forward output (inference gates), every parameter's .grad and the mixture gradient."""
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(T, B)
    G = _cotangents(cfg, B, T, rtd, 71)
    want_out, want, want_dmix = _oracle_mss(cfg, sd, mix, G, rtd)
    model = model.cuda().train()
    model.differentiable = True
    x = mix.cuda().requires_grad_(True)
    out = model(x, return_time_domain=rtd)
    assert list(out) == list(G) and all(v.requires_grad for v in out.values())
    for k in out:
        assert out[k].shape == want_out[k].shape, k
        _check_forward(out[k], want_out[k], train_mode, f"mss forward {k}")
    _inner(out, G).backward()
    _check_grads(model, want, train_mode, "mss")
    _check_mixture_grad(x.grad, want_dmix, cfg["n_fft"] // 2, train_mode, "mss")
    assert model.blocks[0].freq_path.attn.rope is None or model.blocks[0].freq_path.attn.rope.freqs.grad is None


def test_spectral_output_needs_four_sources(pkg):
    """return_time_domain=False names four sources, as the reference does: n_sources < 4 raises IndexError."""
    model = _random_model(pkg, dict(SMALL, n_sources=2)).cuda().train()
    model.differentiable = True
    with pytest.raises(IndexError):
        model(_mixture(2560, 1).cuda(), return_time_domain=False)


SEP = dict(num_spk=2, n_layers=2, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           flash_attention=False, attention_dim=32, pos_enc="rope", ffn_type=["swiglu_conv1d", "swiglu_conv1d"],
           ffn_hidden_dim=[48, 64], conv1d_kernel=4, conv1d_shift=1, dropout=0.0, eps=1e-5)


def _oracle_sep_input(sd, spec, G, wrt_params=True):
    """-> ({key: grad}, complex d spec) of float64 autograd of oracle.separator_forward, loss Re<est, G>."""
    sd64 = {k: v.detach().double().clone().requires_grad_(wrt_params and not k.endswith("rope.freqs"))
            for k, v in sd.items()}
    spec64 = spec.to(torch.complex128).requires_grad_(True)
    est = oracle.separator_forward(sd64, SEP, spec64, dtype=torch.float64)
    G64 = G.to(torch.complex128)
    ((est.real * G64.real).sum() + (est.imag * G64.imag).sum()).backward()
    return {k: v.grad for k, v in sd64.items() if v.grad is not None}, spec64.grad


def _perturbed_sep(pkg, cls=None, **kw):
    model = (cls or pkg.TFLocoformerSeparator)(**kw)
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.ndim == 1 and not n.endswith("rope.freqs"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    return model


def test_separator_input_gradient_vs_oracle_autograd(pkg, train_mode):
    """TFLocoformerSeparator with a complex input that requires grad: d spec (torch's convention, through
    view_as_real) and every parameter gradient."""
    model = _perturbed_sep(pkg, **SEP)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    spec = _seeded((2, 9, 21), 11, complex_=True)
    G = _seeded((2, 2, 9, 21), 12, complex_=True)
    want, want_dspec = _oracle_sep_input(sd, spec, G)
    model = model.cuda().train()
    model.differentiable = True
    x = spec.cuda().requires_grad_(True)
    est = model(x)
    Gc = G.cuda()
    ((est.real * Gc.real).sum() + (est.imag * Gc.imag).sum()).backward()
    _check_grads(model, want, train_mode, "separator")
    assert x.grad is not None and x.grad.dtype == torch.complex64
    err = _rel(torch.view_as_real(x.grad), torch.view_as_real(want_dspec))
    print(f"[{train_mode}] separator input gradient error {err:.2e}")
    assert err < TOL[train_mode]["step"], err


def test_espnet_adapter_and_frozen_separator_input_gradient(pkg):
    """The ESPnet adapter with a requires-grad [B, T, 1, F] input; and a separator whose parameters are all frozen (a
    separator used inside a larger trained model): the input gets its gradient, no parameter gets one."""
    from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as Esp
    spec = _seeded((2, 9, 17), 21, complex_=True)
    G = _seeded((2, 2, 9, 17), 22, complex_=True)
    model = _perturbed_sep(pkg, Esp, input_dim=17, **SEP, differentiable=True)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    want, want_dspec = _oracle_sep_input(sd, spec, G)
    model = model.cuda().train()
    x = spec.cuda().unsqueeze(2).requires_grad_(True)
    outs, _, _ = model(x, torch.tensor([9, 9]))
    sum((o.real * G[:, i].cuda().real).sum() + (o.imag * G[:, i].cuda().imag).sum() for i, o in enumerate(outs)).backward()
    _check_grads(model, want, "mixed", "espnet adapter")
    assert _rel(torch.view_as_real(x.grad[:, :, 0]), torch.view_as_real(want_dspec)) < TOL["mixed"]["step"]

    frozen = pkg.TFLocoformerSeparator(**SEP)
    frozen.load_state_dict(sd)
    frozen = frozen.cuda().train().requires_grad_(False)
    frozen.differentiable = True
    x = spec.cuda().requires_grad_(True)
    est = frozen(x)
    assert est.requires_grad
    Gc = G.cuda()
    ((est.real * Gc.real).sum() + (est.imag * Gc.imag).sum()).backward()
    assert all(p.grad is None for p in frozen.parameters())
    _, want_dspec = _oracle_sep_input(sd, spec, G, wrt_params=False)
    assert _rel(torch.view_as_real(x.grad), torch.view_as_real(want_dspec)) < TOL["mixed"]["step"]


def test_autograd_matches_trainer(pkg, train_mode):
    """Two copies of one model: Trainer.forward_backward (the CUDA MSSLoss) against autograd of the model's output with
    the loss restated in torch (test_gpu_training._ref_loss, on .cpu().double() of the outputs)."""
    from mss_tf_locoformer_b200.training import Trainer
    cfg, B, T, weights = SMALL, 2, 6000, (1.0, 0.1, 0.1)
    mix = _mixture(T, B)
    g = torch.Generator().manual_seed(9)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(cfg["n_sources"], B, T, generator=g)
    tr = Trainer(_random_model(pkg, cfg).cuda(), si_sdr_weight=weights[0], l1_weight=weights[1],
                 spectral_weight=weights[2])
    tr.forward_backward(mix.cuda(), tgt.cuda())
    model = _random_model(pkg, cfg).cuda().train()
    model.differentiable = True
    out = model(mix.cuda())
    pred = {k: v.cpu().double() for k, v in out.items()}
    loss, _ = _ref_loss(pred, {n: tgt[i].double() for i, n in enumerate(NAMES[:cfg["n_sources"]])}, *weights)
    loss.backward()
    errs = {k: _rel(p.grad, tr.grad_of(k)) for k, p in model.named_parameters() if p.requires_grad}
    worst = max(errs, key=errs.get)
    print(f"[{train_mode}] autograd vs Trainer: worst relative gradient difference {errs[worst]:.2e} ({worst})")
    assert errs[worst] < TOL[train_mode]["step"], (worst, errs[worst])


def test_two_forwards_one_backward_and_accumulation(pkg, fp32_mode):
    """Each forward keeps its own workspace: two forwards and one backward of the summed loss give the sum of the single
    gradients (parameters and mixtures), and so do two backward calls into the same .grad."""
    cfg = dict(SMALL, n_sources=2)
    model = _random_model(pkg, cfg).cuda().train()
    model.differentiable = True
    m1, m2 = _mixture(2560, 2, seed=1).cuda(), _mixture(2560, 2, seed=2).cuda()
    G1, G2 = _cotangents(cfg, 2, 2560, True, 81), _cotangents(cfg, 2, 2560, True, 91)
    params = [p for p in model.parameters() if p.requires_grad]

    def grads_of(fn):
        model.zero_grad(set_to_none=True)
        x1, x2 = m1.clone().requires_grad_(True), m2.clone().requires_grad_(True)
        fn(x1, x2)
        return [p.grad.detach().clone() for p in params] + [x1.grad, x2.grad]

    g1 = grads_of(lambda a, b: _inner(model(a), G1).backward())
    g2 = grads_of(lambda a, b: _inner(model(b), G2).backward())
    both = grads_of(lambda a, b: (_inner(model(a), G1) + _inner(model(b), G2)).backward())
    acc = grads_of(lambda a, b: (_inner(model(a), G1).backward(), _inner(model(b), G2).backward()))
    n = len(params)
    for i, (s, c) in enumerate(zip(both, acc)):
        want = g1[i] + g2[i] if i < n else (g1[i] if i == n else g2[i])
        assert _rel(s, want) < 1e-5 and _rel(c, want) < 1e-5, i


def test_defaults_unchanged_and_workspace_released(pkg):
    """differentiable False: no graph, and a requires-grad mixture is refused; eval mode with differentiable True builds
    no graph; BS-Locoformer still refuses a requires-grad input.  The memory of a forward + backward returns to its
    pre-forward value."""
    cfg = dict(SMALL, n_sources=2)
    model = _random_model(pkg, cfg).cuda().train()
    mix = _mixture(2560, 2).cuda()
    G = _cotangents(cfg, 2, 2560, True, 101)
    assert model.differentiable is False
    assert not any(v.requires_grad for v in model(mix).values())
    with pytest.raises(NotImplementedError, match="forward-only"):
        model(mix.clone().requires_grad_(True))
    model.differentiable = True
    model.eval()
    assert not any(v.requires_grad for v in model(mix).values())
    with pytest.raises(NotImplementedError, match="forward-only"):
        model(mix.clone().requires_grad_(True))
    bs = pkg.BSLocoformerSeparator(**dict(SEP, n_layers=1, sample_rate=44100, stft_size=256)).cuda().train()
    bs.differentiable = True
    with pytest.raises(NotImplementedError, match="forward-only"):
        bs(_seeded((1, 5, 129), 5, complex_=True).cuda().requires_grad_(True))
    model.train()
    x = mix.clone().requires_grad_(True)
    _inner(model(x), G).backward()                        # allocates the .grad tensors
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    loss = _inner(model(x), G)
    assert torch.cuda.memory_allocated() > before         # the saved workspace is alive until backward
    loss.backward()
    del loss
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before


# The MSS training step at SMALL, B 2 x 6000 samples, loss weights (1, 0.1, 0.1): launches per step in modes 0 / 1 / 2,
# and the total loss and gradient norm the step returned before the autograd entry points existed (NVIDIA B200).
STEP_LAUNCHES = {0: 189, 1: 189, 2: 179}
STEP_VALUES = {0: (96.02157592773438, 872.88032), 1: (96.0213394165039, 872.78007), 2: (96.0221939086914, 873.85910)}
SEP_BWD_LAUNCHES = 132      # tfl_sep_train_backward at SEP, batch 2 x 9 frames x 21 bins


def test_launch_counts_of_existing_entry_points_unchanged(pkg):
    from mss_tf_locoformer_b200 import _lib
    from mss_tf_locoformer_b200.training import Trainer
    lib = _lib.load()
    mix = _mixture(6000, 2)
    g = torch.Generator().manual_seed(9)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(4, 2, 6000, generator=g)
    try:
        for mode, want in STEP_LAUNCHES.items():
            assert lib.tfl_debug_set_option(5, mode) == 0
            tr = Trainer(_random_model(pkg, SMALL).cuda(), si_sdr_weight=1.0, l1_weight=0.1, spectral_weight=0.1)
            tr.forward_backward(mix.cuda(), tgt.cuda())         # packs the weights
            torch.cuda.synchronize()
            n0 = lib.tfl_launch_count()
            loss, _ = tr.forward_backward(mix.cuda(), tgt.cuda())
            torch.cuda.synchronize()
            launches = lib.tfl_launch_count() - n0
            got = (float(loss[0]), float(tr.grads.double().norm()))
            print(f"mode {mode}: {launches} launches, loss {got[0]!r}, gradient norm {got[1]!r}")
            assert launches == want, (mode, launches)
            for a, b in zip(got, STEP_VALUES[mode]):             # atomics order moves the last bits only
                assert abs(a - b) <= 1e-5 * abs(b), (mode, got, STEP_VALUES[mode])
        assert lib.tfl_debug_set_option(5, 2) == 0
        sep = _perturbed_sep(pkg, **SEP).cuda().train()
        sep.differentiable = True
        x = _seeded((2, 9, 21), 11, complex_=True).cuda()
        counts = []
        for req in (False, True):
            est = sep(x.clone().requires_grad_(req))
            torch.cuda.synchronize()
            n0 = lib.tfl_launch_count()
            est.abs().sum().backward()
            torch.cuda.synchronize()
            counts.append(lib.tfl_launch_count() - n0)
        print(f"separator backward launches: {counts[0]} (parameters), {counts[1]} (with the input gradient)")
        assert counts[0] == SEP_BWD_LAUNCHES
        assert counts[1] == counts[0] + 1                         # + enc_input_grad_kernel
    finally:
        lib.tfl_debug_set_option(5, 2)
