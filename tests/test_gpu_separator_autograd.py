"""Training of TFLocoformerSeparator, its ESPnet adapter and BSLocoformerSeparator through torch autograd
(``differentiable = True``; DESIGN.md section 8b).

Checker: float64 torch autograd of ``oracle.separator_forward`` / ``oracle.bs_forward`` on the CPU with
``loss = Re<est, G>`` for a seeded complex G.  Every trainable parameter's ``.grad`` is compared by relative L2 error
against the whole-step gates of test_gpu_training.py (TOL[mode]["step"]) in the fp32, tf32 and mixed arithmetic of
TFL_OPT_TRAIN_MODE.
"""
import pytest
import torch

import oracle
from test_gpu_training import TOL, _rel, _sd64

pytestmark = pytest.mark.gpu

MODES = {"fp32": 0, "tf32": 1, "mixed": 2}


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


SEP = dict(num_spk=2, n_layers=2, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           flash_attention=False, attention_dim=32, pos_enc="rope", ffn_type=["swiglu_conv1d", "swiglu_conv1d"],
           ffn_hidden_dim=[48, 64], conv1d_kernel=4, conv1d_shift=1, dropout=0.0, eps=1e-5)
SEP_D = dict(SEP, n_layers=1, emb_dim=128, attention_dim=128, ffn_hidden_dim=[384, 384])      # Variant-D widths


def _perturb(model, seed):
    """Random 1-D parameters (the default init makes every norm gain 1 and every bias ~0: too symmetric a test)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.ndim == 1 and not n.endswith("rope.freqs"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    return model


def _spec(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.complex(torch.randn(*shape, generator=g), torch.randn(*shape, generator=g))


def _inner(est, G):
    """Re<est, G> = sum(est.real * G.real + est.imag * G.imag)."""
    return (est.real * G.real).sum() + (est.imag * G.imag).sum()


def _oracle_sep(cfg, sd, spec, G):
    sd64 = {k: v.detach().double().clone().requires_grad_(not k.endswith("rope.freqs")) for k, v in sd.items()}
    est = oracle.separator_forward(sd64, cfg, spec.to(torch.complex128), dtype=torch.float64)
    _inner(est, G.to(torch.complex128)).backward()
    return est.detach(), {k: v.grad for k, v in sd64.items() if v.grad is not None}


def _check_grads(model, want, mode, what):
    got = dict(model.named_parameters())
    assert set(want) == {k for k, p in got.items() if p.requires_grad}, what
    errs = {k: _rel(got[k].grad, want[k]) for k in want}
    worst = max(errs, key=errs.get)
    print(f"[{mode}] {what}: worst relative gradient error {errs[worst]:.2e} ({worst}) over {len(errs)} tensors")
    assert errs[worst] < TOL[mode]["step"], (what, worst, errs[worst])


def _check_forward(est, want, mode, what):
    got = torch.view_as_real(est.detach().cpu().contiguous()).double()
    ref = torch.view_as_real(want.contiguous())
    if mode == "fp32":
        err = float((got - ref).abs().max())
        assert err <= 1e-4, (what, err)
    else:
        sd = oracle.si_sdr_db(got, ref)
        assert sd >= 40.0, (what, sd)


@pytest.mark.parametrize("cfg,shape", [
    (SEP, (2, 9, 21)),
    (dict(SEP, pos_enc="nope", tf_order="tf", ffn_type="swiglu_conv1d", ffn_hidden_dim=64, conv1d_kernel=1), (2, 7, 17)),
    (dict(SEP, tf_order="tf", conv1d_kernel=8), (2, 11, 13)),
    (SEP_D, (2, 6, 129)),
], ids=["macaron_rope_ft_k4", "single_nope_tf_k1", "macaron_rope_tf_k8", "variant_d_widths"])
def test_separator_gradients_vs_oracle_autograd(pkg, train_mode, cfg, shape):
    """TFLocoformerSeparator: forward output (inference gates) and every parameter's .grad against float64 autograd."""
    model = _perturb(pkg.TFLocoformerSeparator(**cfg), 3)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    spec = _spec(shape, 11)
    G = _spec((shape[0], cfg["num_spk"]) + shape[1:], 12)
    want_est, want = _oracle_sep(cfg, sd, spec, G)
    model = model.cuda().train()
    model.differentiable = True
    est = model(spec.cuda())
    assert est.requires_grad and est.shape == want_est.shape
    _check_forward(est, want_est, train_mode, "separator forward")
    _inner(est, G.cuda()).backward()
    _check_grads(model, want, train_mode, "separator")
    assert model.blocks[0].freq_path.attn.rope is None or model.blocks[0].freq_path.attn.rope.freqs.grad is None


def test_espnet_adapter_trains_through_list_output(pkg):
    """ESPnet interface ([B, T, 1, F] input, list of num_spk outputs): the loss built from the list reaches every
    trainable parameter (default mixed arithmetic), and attn.rope.freqs gets no gradient."""
    from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as Esp
    kw = {k: v for k, v in SEP.items()}
    model = _perturb(Esp(17, **kw, differentiable=True), 5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    spec = _spec((2, 9, 17), 21)
    G = _spec((2, 2, 9, 17), 22)
    _, want = _oracle_sep(SEP, sd, spec, G)
    model = model.cuda().train()
    outs, ilens, extra = model(spec.cuda().unsqueeze(2), torch.tensor([9, 9]))
    assert isinstance(outs, list) and len(outs) == 2 and all(o.requires_grad for o in outs)
    loss = sum(_inner(o, G[:, i].cuda()) for i, o in enumerate(outs))
    loss.backward()
    for n, p in model.named_parameters():
        if n.endswith("rope.freqs"):
            assert p.grad is None, n
        else:
            assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0, n
    _check_grads(model, want, "mixed", "espnet adapter")


BS = dict(num_spk=2, n_layers=1, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
          flash_attention=False, attention_dim=32, pos_enc="rope", ffn_type=["swiglu_conv1d", "swiglu_conv1d"],
          ffn_hidden_dim=[48, 48], conv1d_kernel=4, conv1d_shift=1, dropout=0.0, sample_rate=44100, stft_size=256,
          eps=1e-5, masking=True, stereo=False)
BS_CFG4 = dict(BS, num_spk=4, emb_dim=128, attention_dim=128, ffn_hidden_dim=[384, 384], stft_size=2048, stereo=True)


def _bs_case(pkg, cfg, B, T, mode):
    model = _perturb(pkg.BSLocoformerSeparator(**cfg), 7)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    M, F = (2 if cfg["stereo"] else 1), cfg["stft_size"] // 2 + 1
    shape = (B, M, T, F) if cfg["stereo"] else (B, T, F)
    spec = _spec(shape, 31)
    G = _spec((B, cfg["num_spk"]) + shape[1:], 32)
    sd64 = {k: v.detach().double().clone().requires_grad_(not k.endswith("rope.freqs")) for k, v in sd.items()}
    want_est = oracle.bs_forward(sd64, cfg, spec.to(torch.complex128), dtype=torch.float64)
    _inner(want_est, G.to(torch.complex128)).backward()
    want = {k: v.grad for k, v in sd64.items() if v.grad is not None}
    model = model.cuda().train()
    model.differentiable = True
    est = model(spec.cuda())
    assert est.requires_grad and est.shape == want_est.shape
    _check_forward(est, want_est.detach(), mode, "bs forward")
    _inner(est, G.cuda()).backward()
    _check_grads(model, want, mode, f"bs {cfg['sample_rate']} stereo={cfg['stereo']} masking={cfg['masking']}")


@pytest.mark.parametrize("masking,stereo,sample_rate", [(True, False, 44100), (False, True, 44100), (True, True, 48000),
                                                        (False, False, 48000)])
def test_bs_separator_gradients_vs_oracle_autograd(pkg, train_mode, masking, stereo, sample_rate):
    """BSLocoformerSeparator: band-split / band-wise decoding backward kernels (20 frames: a partial 16-frame tile) and
    the blocks-only backward, every parameter against float64 autograd; 48 kHz includes the four-way rest split."""
    _bs_case(pkg, dict(BS, masking=masking, stereo=stereo, sample_rate=sample_rate), 2, 20, train_mode)


def test_bs_separator_config4_shape_mixed(pkg):
    """BASELINE config 4 widths (stereo, 4 sources, 62 bands, emb 128; one layer, 6 frames) in the default mixed mode."""
    _bs_case(pkg, BS_CFG4, 1, 6, "mixed")


def test_adamw_steps_match_oracle(pkg, fp32_mode):
    """Three torch.optim.AdamW steps on a differentiable separator == the same steps on the float64 oracle: the packed
    weight image follows optimizer.step()."""
    cfg = dict(SEP, n_layers=1)
    model = _perturb(pkg.TFLocoformerSeparator(**cfg), 13)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    spec = _spec((2, 8, 19), 41)
    G = _spec((2, 2, 8, 19), 42)
    sd64 = _sd64(model)
    params64 = [v for v in sd64.values() if v.requires_grad]
    opt64 = torch.optim.AdamW(params64, lr=1e-3, weight_decay=0.01)
    for _ in range(3):
        opt64.zero_grad(set_to_none=True)
        _inner(oracle.separator_forward(sd64, cfg, spec.to(torch.complex128), dtype=torch.float64),
               G.to(torch.complex128)).backward()
        opt64.step()
    model = model.cuda().train()
    model.differentiable = True
    opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-3, weight_decay=0.01)
    for _ in range(3):
        opt.zero_grad(set_to_none=True)
        _inner(model(spec.cuda()), G.cuda()).backward()
        opt.step()
    num = den = 0.0
    for k, p in model.state_dict().items():
        if k.endswith("rope.freqs"):
            continue
        upd_ref = sd64[k].detach() - sd[k].double()
        upd_got = p.detach().double().cpu() - sd[k].double()
        num += float((upd_got - upd_ref).pow(2).sum())
        den += float(upd_ref.pow(2).sum())
    assert (num / den) ** 0.5 < 0.02, (num / den) ** 0.5


def test_two_forwards_one_backward_and_accumulation(pkg, fp32_mode):
    """Each forward keeps its own activations: two forwards on different inputs and one backward of the summed loss give
    the sum of the single gradients, and so do two backward calls into the same .grad."""
    model = _perturb(pkg.TFLocoformerSeparator(**SEP), 17).cuda().train()
    model.differentiable = True
    x1, x2 = _spec((2, 9, 21), 51).cuda(), _spec((2, 9, 21), 52).cuda()
    G1, G2 = _spec((2, 2, 9, 21), 53).cuda(), _spec((2, 2, 9, 21), 54).cuda()
    params = [p for p in model.parameters() if p.requires_grad]

    def grads_of(fn):
        model.zero_grad(set_to_none=True)
        fn()
        return [p.grad.detach().clone() for p in params]

    g1 = grads_of(lambda: _inner(model(x1), G1).backward())
    g2 = grads_of(lambda: _inner(model(x2), G2).backward())
    both = grads_of(lambda: (_inner(model(x1), G1) + _inner(model(x2), G2)).backward())
    acc = grads_of(lambda: (_inner(model(x1), G1).backward(), _inner(model(x2), G2).backward()))
    for a, b, s, c in zip(g1, g2, both, acc):
        assert _rel(s, a + b) < 1e-5 and _rel(c, a + b) < 1e-5


def test_defaults_unchanged_and_workspace_released(pkg):
    """differentiable False: a grad-enabled forward builds no graph and a requires-grad input is still refused.  With
    differentiable True, the memory of a forward + backward returns to its pre-forward value (the saved workspace goes
    with the graph)."""
    model = _perturb(pkg.TFLocoformerSeparator(**SEP), 19).cuda().train()
    x = _spec((2, 9, 21), 61).cuda()
    G = _spec((2, 2, 9, 21), 62).cuda()
    assert model.differentiable is False
    assert model(x).requires_grad is False
    with pytest.raises(NotImplementedError, match="forward-only"):
        model(x.clone().requires_grad_(True))
    bs = pkg.BSLocoformerSeparator(**BS).cuda().train()
    assert bs(_spec((1, 5, 129), 63).cuda()).requires_grad is False
    model.differentiable = True
    with torch.no_grad():
        assert model(x).requires_grad is False
    model.eval()
    assert model(x).requires_grad is False
    model.train()
    _inner(model(x), G).backward()                       # allocates the .grad tensors
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    loss = _inner(model(x), G)
    assert torch.cuda.memory_allocated() > before        # the saved workspace is alive until backward
    loss.backward()
    del loss
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before
