"""Bitwise-reproducible training under ``torch.use_deterministic_algorithms(True)`` (TFL_OPT_DETERMINISTIC).

Every case turns the torch flag on and restores it afterwards, in the fp32, tf32 and mixed arithmetic of
TFL_OPT_TRAIN_MODE, at the SMALL shape of test_gpu_training.py and at one layer of Variant-D widths (many row splits per
weight-gradient GEMM).  Two runs of the same work must agree with ``torch.equal``; the deterministic gradients must agree
with the default (atomics) path to summation-order noise and with the float64 oracle at the whole-step gates; and after
the flag is turned off again the step launches the same kernels and computes what a run that never turned it on does.
"""
import pytest
import torch

from test_gpu_parity import VARIANT_D, _mixture, _random_model
from test_gpu_separator_autograd import BS, SEP, SEP_D, _perturb, _spec
from test_gpu_training import SMALL, TOL, _reference_step, _rel

pytestmark = pytest.mark.gpu

MODES = {"fp32": 0, "tf32": 1, "mixed": 2}
VD1 = dict(VARIANT_D, flash_attention=False)          # one layer at Variant-D widths
SHAPES = {"small": (dict(SMALL, n_layers=1), 4000, 2), "variant_d": (VD1, 24000, 1)}
# deterministic vs default gradients, relative to each tensor's norm (floored at 1e-3 of the largest, for gradients that
# vanish in exact arithmetic): the default path differs from run to run in the last bits of its atomics
ORDER_NOISE = {"fp32": 1e-5, "tf32": 1e-4, "mixed": 1e-4}


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available()
    return m


def _set_mode(m):
    from mss_tf_locoformer_b200 import _lib
    assert _lib.load().tfl_debug_set_option(5, m) == 0


@pytest.fixture(params=list(MODES))
def train_mode(request, pkg):
    _set_mode(MODES[request.param])
    yield request.param
    _set_mode(2)


@pytest.fixture
def deterministic(pkg):
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev)


def _data(cfg, T, B, seed=4):
    mix = _mixture(T, B)
    g = torch.Generator().manual_seed(seed)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(cfg["n_sources"], B, T, generator=g)
    return mix.cuda(), tgt.cuda()


def _trainer(pkg, cfg, sd, **kw):
    from mss_tf_locoformer_b200.training import Trainer
    model = pkg.TFLocoformerMSS(**cfg)
    model.load_state_dict(sd)
    return Trainer(model.cuda(), lr=1e-3, **kw)


def _state(tr):
    return [t.clone() for t in (tr.grads, tr.params, tr.exp_avg, tr.exp_avg_sq)]


def _assert_equal(a, b, what):
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), (what, i, float((x.double() - y.double()).abs().max()))


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("accum", [1, 2])
def test_two_trainers_three_steps_bitwise(pkg, train_mode, deterministic, shape, accum):
    """Two Trainers from the same seed, three steps each: loss, grads, params, exp_avg and exp_avg_sq torch.equal."""
    cfg, T, B = SHAPES[shape]
    sd = {k: v.detach().clone() for k, v in _random_model(pkg, cfg).state_dict().items()}
    mix, tgt = _data(cfg, T, B)
    runs = []
    for _ in range(2):
        tr = _trainer(pkg, cfg, sd, gradient_accumulation_steps=accum)
        losses = [tr.step(mix, tgt).clone() for _ in range(3 * accum)]
        torch.cuda.synchronize()
        runs.append((losses, _state(tr)))
    _assert_equal(runs[0][0], runs[1][0], "loss")
    _assert_equal(runs[0][1], runs[1][1], "grads / params / exp_avg / exp_avg_sq")
    assert bool(torch.isfinite(runs[0][1][1]).all())


def test_resume_continues_bitwise(pkg, train_mode, deterministic):
    """A Trainer restored from state_dict() after step 1 takes steps 2 and 3 exactly as the uninterrupted run."""
    cfg, T, B = SHAPES["small"]
    sd = {k: v.detach().clone() for k, v in _random_model(pkg, cfg).state_dict().items()}
    mix, tgt = _data(cfg, T, B)
    tr_a = _trainer(pkg, cfg, sd)
    tr_a.step(mix, tgt)
    tr_c = _trainer(pkg, cfg, {k: v.detach().clone() for k, v in tr_a.model.state_dict().items()})
    tr_c.load_state_dict(tr_a.state_dict())
    for _ in range(2):
        la, lc = tr_a.step(mix, tgt), tr_c.step(mix, tgt)
        assert torch.equal(la, lc)
    _assert_equal(_state(tr_a), _state(tr_c), "resumed")


@pytest.mark.parametrize("shape", list(SHAPES))
def test_deterministic_matches_default_path(pkg, train_mode, shape):
    """Same inputs, flag on vs off: every parameter gradient within summation-order noise, the loss too."""
    cfg, T, B = SHAPES[shape]
    sd = {k: v.detach().clone() for k, v in _random_model(pkg, cfg).state_dict().items()}
    mix, tgt = _data(cfg, T, B)
    tr = _trainer(pkg, cfg, sd)
    out = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        try:
            loss, _ = tr.forward_backward(mix, tgt)
            out[det] = (loss.clone(), tr.grads.clone())
        finally:
            torch.use_deterministic_algorithms(False)
    floor = 1e-3 * max(float(tr.grad_of(k).norm()) for k in tr.engine.keys if not k.endswith("rope.freqs"))
    worst = 0.0
    for i, k in enumerate(tr.engine.keys):
        o, n = tr.offsets[i], tr.sizes[i]
        if o < 0:
            continue
        a, b = out[True][1][o:o + n].double(), out[False][1][o:o + n].double()
        worst = max(worst, float((a - b).norm()) / max(float(b.norm()), floor))
    print(f"[{train_mode}] {shape}: deterministic vs default, worst relative gradient difference {worst:.2e}")
    assert worst <= ORDER_NOISE[train_mode], worst
    assert abs(float(out[True][0][0]) - float(out[False][0][0])) <= 1e-5 * abs(float(out[False][0][0]))


def test_deterministic_step_vs_float64_oracle(pkg, train_mode, deterministic):
    """The deterministic step against float64 autograd of the reference at the whole-step gates, on the shape, data and
    loss weights at which test_gpu_training.py gates the default step (SMALL, 2 x 6000 samples)."""
    cfg = SMALL
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix, tgt = _data(cfg, 6000, 2, seed=9)
    weights = (1.0, 0.1, 0.1)
    want_loss, want_grads, _ = _reference_step(cfg, sd, mix.cpu(), tgt.cpu(), weights)
    from mss_tf_locoformer_b200.training import Trainer
    tr = Trainer(model.cuda(), si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
    loss, _ = tr.forward_backward(mix, tgt)
    tol = TOL[train_mode]
    assert abs(float(loss[0]) - want_loss) <= tol["loss"] * max(1.0, abs(want_loss)), (float(loss[0]), want_loss)
    errs = {k: _rel(tr.grad_of(k), want_grads[k]) for k in want_grads}
    worst = max(errs, key=errs.get)
    print(f"[{train_mode}] deterministic step vs float64: worst relative gradient error {errs[worst]:.2e} ({worst})")
    assert errs[worst] < tol["step"], (worst, errs[worst])


def test_flag_off_after_on_is_the_default_path(pkg, train_mode):
    """After a deterministic step, turning the flag off gives the default step: its launch count, loss and gradients
    equal those of a Trainer that never saw the flag (loss and gradients to atomics-order noise)."""
    from mss_tf_locoformer_b200 import _lib
    lib = _lib.load()
    cfg, T, B = SHAPES["small"]
    sd = {k: v.detach().clone() for k, v in _random_model(pkg, cfg).state_dict().items()}
    mix, tgt = _data(cfg, T, B)

    def counted(tr):
        torch.cuda.synchronize()
        n0 = lib.tfl_launch_count()
        loss, _ = tr.forward_backward(mix, tgt)
        torch.cuda.synchronize()
        return lib.tfl_launch_count() - n0, loss.clone(), tr.grads.clone()

    never = _trainer(pkg, cfg, sd)
    counted(never)                                             # packs the weights
    want = counted(never)
    tr = _trainer(pkg, cfg, sd)
    torch.use_deterministic_algorithms(True)
    try:
        on = counted(tr)
    finally:
        torch.use_deterministic_algorithms(False)
    got = counted(tr)
    print(f"[{train_mode}] launches per forward_backward: {want[0]} default, {on[0]} deterministic")
    assert on[0] > want[0]
    assert got[0] == want[0]
    assert abs(float(got[1][0]) - float(want[1][0])) <= 1e-5 * abs(float(want[1][0]))
    assert _rel(got[2], want[2]) <= 1e-5


def _twice(fn):
    """Two identical forward + backward passes -> the two lists of gradients (after zeroing)."""
    out = []
    for _ in range(2):
        out.append(fn())
        torch.cuda.synchronize()
    return out


def _grads(model, *extra):
    return [p.grad.clone() for p in model.parameters() if p.grad is not None] + [e.grad.clone() for e in extra]


def test_mss_autograd_bitwise(pkg, train_mode, deterministic):
    """TFLocoformerMSS through autograd: every .grad and mixture.grad, twice, torch.equal (SMALL and Variant-D widths)."""
    for cfg, T, B in SHAPES.values():
        model = _random_model(pkg, cfg).cuda().train()
        model.differentiable = True
        mix, _ = _data(cfg, T, B)
        G = [torch.randn(B, T, generator=torch.Generator().manual_seed(i)).cuda() for i in range(cfg["n_sources"])]

        def run():
            model.zero_grad(set_to_none=True)
            x = mix.clone().requires_grad_(True)
            out = model(x)
            sum((v * G[i]).sum() for i, v in enumerate(out.values())).backward()
            return _grads(model, x)

        a, b = _twice(run)
        assert len(a) == len(b) and len(a) > 1
        _assert_equal(a, b, "mss autograd")


def test_separator_autograd_bitwise(pkg, train_mode, deterministic):
    """TFLocoformerSeparator with an input gradient, at SEP and Variant-D widths, and the ESPnet adapter."""
    from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as Esp
    for cfg, shape in ((SEP, (2, 9, 21)), (SEP_D, (2, 6, 129))):
        model = _perturb(pkg.TFLocoformerSeparator(**cfg), 3).cuda().train()
        model.differentiable = True
        spec = _spec(shape, 11).cuda()
        G = _spec((shape[0], cfg["num_spk"]) + shape[1:], 12).cuda()

        def run():
            model.zero_grad(set_to_none=True)
            x = spec.clone().requires_grad_(True)
            est = model(x)
            ((est.real * G.real).sum() + (est.imag * G.imag).sum()).backward()
            return _grads(model, x)

        _assert_equal(*_twice(run), "separator autograd")
    esp = _perturb(Esp(17, **SEP, differentiable=True), 5).cuda().train()
    spec = _spec((2, 9, 17), 21).cuda()
    G = _spec((2, 2, 9, 17), 22).cuda()

    def run_esp():
        esp.zero_grad(set_to_none=True)
        outs, _, _ = esp(spec.unsqueeze(2), torch.tensor([9, 9]))
        sum((o.real * G[:, i].real).sum() + (o.imag * G[:, i].imag).sum() for i, o in enumerate(outs)).backward()
        return _grads(esp)

    _assert_equal(*_twice(run_esp), "espnet adapter")


def test_bs_separator_autograd_bitwise(pkg, train_mode, deterministic):
    """BSLocoformerSeparator (the blocks-only backward between the band stages): every .grad twice, torch.equal."""
    model = _perturb(pkg.BSLocoformerSeparator(**dict(BS, stereo=True)), 7).cuda().train()
    model.differentiable = True
    F = BS["stft_size"] // 2 + 1
    spec = _spec((2, 2, 20, F), 31).cuda()
    G = _spec((2, BS["num_spk"], 2, 20, F), 32).cuda()

    def run():
        model.zero_grad(set_to_none=True)
        est = model(spec)
        ((est.real * G.real).sum() + (est.imag * G.imag).sum()).backward()
        return _grads(model)

    _assert_equal(*_twice(run), "bs separator autograd")


def _rank_worker(rank, world, port, cfg, sd, mix, tgt, ret):
    import os
    import torch.distributed as dist
    import mss_tf_locoformer_b200 as m
    from mss_tf_locoformer_b200.training import Trainer, allreduce_mean_
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        torch.use_deterministic_algorithms(True)
        model = m.TFLocoformerMSS(**cfg)
        model.load_state_dict(sd, strict=True)
        tr = Trainer(model.cuda(), lr=1e-3)
        tr.forward_backward(mix[rank:rank + 1].cuda(), tgt[:, rank:rank + 1].cuda())
        local = tr.grads.cpu().clone()
        allreduce_mean_(tr.grads)
        torch.cuda.synchronize()
        ret[rank] = local
    finally:
        dist.destroy_process_group()


def test_each_rank_local_gradient_equals_one_gpu(pkg, deterministic):
    """Two ranks, one sample each: every rank's gradient before the all-reduce is torch.equal to one GPU's gradient on
    that rank's sample (the all-reduce itself is NCCL's)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    cfg, T, _ = SHAPES["small"]
    sd = {k: v.detach().clone() for k, v in _random_model(pkg, cfg).state_dict().items()}
    mix, tgt = _data(cfg, T, 2)
    mix, tgt = mix.cpu(), tgt.cpu()
    want = []
    for r in range(2):
        tr = _trainer(pkg, cfg, sd)
        tr.forward_backward(mix[r:r + 1].cuda(), tgt[:, r:r + 1].cuda())
        want.append(tr.grads.cpu().clone())
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_rank_worker, args=(2, port, cfg, sd, mix, tgt, ret), nprocs=2, join=True)
        res = dict(ret)
    for r in range(2):
        assert torch.equal(res[r], want[r]), r
