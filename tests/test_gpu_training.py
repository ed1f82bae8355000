"""GPU parity of the training step (SURVEY.md section 8(f) N1): gradients of the CUDA backward kernels against torch
autograd of the reference (the unmodified modules staged in oracle/_ref when present, else the oracle restatement),
computed on the CPU in float64.  Tolerances: relative L2 error per tensor (the weight gradients accumulate ~10^4-10^6
fp32 products through atomics, order-dependent in the last bits).

Without oracle/_ref the whole-step checker is the oracle forward (pinned to the reference's forward by
tests/golden/*.npz) with `_ref_loss`, a restatement of the reference's MSSLoss.  No stored vector ties that
restatement to the reference's own loss: the reference is not part of this repository, so its training outputs
could not be stored.
"""
import math

import pytest
import torch

import oracle
from oracle import build_ref
from test_gpu_parity import _mixture, _random_model

pytestmark = pytest.mark.gpu

SMALL = dict(n_fft=256, hop_length=128, n_sources=4, n_layers=2, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4,
             tf_order="ft", n_heads=4, flash_attention=False, attention_dim=32, pos_enc="rope",
             ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[48, 64], conv1d_kernel=4, conv1d_shift=1,
             dropout=0.0, eps=1e-5)
WIDE = dict(SMALL, n_layers=1, emb_dim=128, attention_dim=128, ffn_hidden_dim=[384, 384])   # Variant D widths


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available()
    return m


MODES = {"fp32": 0, "tf32": 1, "mixed": 2}


@pytest.fixture(params=["fp32", "tf32", "mixed"])
def gemm_mode(request, pkg):
    """TFL_OPT_TRAIN_MODE of the sub-block tests: exact fp32 on CUDA cores (parity mode, tight tolerances), mma.sync tf32
    GEMMs / attention with fp32 accumulation (2^-11 per operand, tolerances ~20x wider), or the bf16 mma.sync forms of the
    mixed mode (2^-9 per operand; the sub-block entry points have no forward of their own, so "mixed" here = bf16 backward)."""
    from mss_tf_locoformer_b200 import _lib
    lib = _lib.load()
    assert lib.tfl_debug_set_option(5, MODES[request.param]) == 0
    yield request.param
    lib.tfl_debug_set_option(5, 2)


@pytest.fixture(params=["fp32", "tf32", "mixed"])
def train_mode(request, pkg):
    """TFL_OPT_TRAIN_MODE of the whole-step tests; "mixed" (the default) adds the bf16 tcgen05 forward of the sub-blocks:
    the gradient is then taken at activations that carry bf16 rounding (~46 dB), as under the reference's autocast."""
    from mss_tf_locoformer_b200 import _lib
    lib = _lib.load()
    assert lib.tfl_debug_set_option(5, MODES[request.param]) == 0
    yield request.param
    lib.tfl_debug_set_option(5, 2)


# (step: deconv.bias is a sum of terms that largely cancel -- 2.5e-3 against float64 in fp32 mode, everything else < 2e-5)
TOL = {"fp32": dict(dx=1e-4, grad=1e-3, step=5e-3, loss=2e-4), "tf32": dict(dx=5e-3, grad=2e-2, step=3e-2, loss=3e-3),
       "mixed": dict(dx=2e-2, grad=3e-2, step=3e-2, loss=3e-3)}


def _rel(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / (want.norm() + 1e-30))


def _sd64(model):
    return {k: v.detach().double().cpu().clone().requires_grad_(v.dtype.is_floating_point and not k.endswith("rope.freqs"))
            for k, v in model.state_dict().items()}


@pytest.mark.parametrize("cfg,shape", [(SMALL, (2, 9, 21)), (WIDE, (1, 5, 140))])
def test_ffn_backward_vs_autograd(pkg, gemm_mode, cfg, shape):
    """tfl_conv_swiglu_ffn_bwd: dx and the five parameter gradients of x + ConvSwiGLU(norm(x)), both axes, both FFNs."""
    from mss_tf_locoformer_b200 import training
    model = _random_model(pkg, cfg).cuda()
    sd = _sd64(model)
    g = torch.Generator().manual_seed(5)
    xin = torch.randn(*shape, cfg["emb_dim"], generator=g)
    dy = torch.randn(*shape, cfg["emb_dim"], generator=g)
    for axis, path in ((0, "freq_path"), (1, "frame_path")):
        for j in (0, 1):
            p = f"blocks.0.{path}"
            keys = [f"{p}.ffn_norm.{j}.gamma", f"{p}.ffn.{j}.conv1d.weight", f"{p}.ffn.{j}.conv1d.bias",
                    f"{p}.ffn.{j}.deconv1d.weight", f"{p}.ffn.{j}.deconv1d.bias"]
            x64 = xin.double().requires_grad_(True)
            xa = x64 if axis == 0 else x64.transpose(1, 2)
            b, s1, s2, c = xa.shape
            xn = oracle.rms_group_norm(xa, sd[keys[0]], cfg["num_groups"], cfg["eps"])
            y = oracle.swiglu_conv_deconv(xn.reshape(b * s1, s2, c), sd[keys[1]], sd[keys[2]], sd[keys[3]], sd[keys[4]])
            y = y.reshape(xa.shape)
            out = x64 + (y if axis == 0 else y.transpose(1, 2))
            grads = torch.autograd.grad(out, [x64] + [sd[k] for k in keys], grad_outputs=dy.double())
            dx, grad_of = training.ffn_backward(model, 0, axis, j, xin.cuda(), dy.cuda())
            tol = TOL[gemm_mode]
            assert _rel(dx, grads[0]) < tol["dx"], ("dx", axis, j, _rel(dx, grads[0]))
            for k, want in zip(keys, grads[1:]):
                assert _rel(grad_of(k), want) < tol["grad"], (k, _rel(grad_of(k), want))


HD16 = dict(SMALL, n_layers=1, emb_dim=64, attention_dim=64, ffn_hidden_dim=[64, 64])   # head_dim 16 (the xlarge config's)


@pytest.mark.parametrize("cfg,shape", [(SMALL, (2, 9, 21)), (WIDE, (1, 3, 150)), (dict(SMALL, pos_enc="nope"), (1, 4, 33)),
                                       (HD16, (1, 70, 131)), (WIDE, (2, 67, 9))])
def test_attention_backward_vs_autograd(pkg, gemm_mode, cfg, shape):
    """tfl_rope_attn_bwd: dx, d gamma, d qkv.weight, d aggregate_heads.weight of x + Wo MHSA(RoPE(qkv(norm(x))))."""
    from mss_tf_locoformer_b200 import training
    model = _random_model(pkg, cfg).cuda()
    sd = _sd64(model)
    g = torch.Generator().manual_seed(6)
    xin = torch.randn(*shape, cfg["emb_dim"], generator=g)
    dy = torch.randn(*shape, cfg["emb_dim"], generator=g)
    for axis, path in ((0, "freq_path"), (1, "frame_path")):
        p = f"blocks.0.{path}"
        keys = [f"{p}.attn_norm.gamma", f"{p}.attn.qkv.weight", f"{p}.attn.aggregate_heads.0.weight"]
        x64 = xin.double().requires_grad_(True)
        xa = x64 if axis == 0 else x64.transpose(1, 2)
        b, s1, s2, c = xa.shape
        xn = oracle.rms_group_norm(xa, sd[keys[0]], cfg["num_groups"], cfg["eps"])
        freqs = sd.get(f"{p}.attn.rope.freqs")
        y = oracle.attention(xn.reshape(b * s1, s2, c), sd[keys[1]], sd[keys[2]], cfg["n_heads"],
                             None if freqs is None else freqs.detach()).reshape(xa.shape)
        out = x64 + (y if axis == 0 else y.transpose(1, 2))
        grads = torch.autograd.grad(out, [x64] + [sd[k] for k in keys], grad_outputs=dy.double())
        dx, grad_of = training.attn_backward(model, 0, axis, xin.cuda(), dy.cuda())
        tol = TOL[gemm_mode]
        assert _rel(dx, grads[0]) < tol["dx"], ("dx", axis, _rel(dx, grads[0]))
        for k, want in zip(keys, grads[1:]):
            assert _rel(grad_of(k), want) < tol["grad"], (k, _rel(grad_of(k), want))


def _ref_loss(pred, tgt, w_sisdr, w_l1, w_spec, eps=1e-8, n_fft=2048, hop=1024):
    """Restatement of MSSLoss(loss_type='combined') (models/mss_loss.py:57-109) for when oracle/_ref is not staged.
    -> (total loss, {"<source>_si_sdr" | "_l1" | "_spectral": unweighted per-source term}); the spectral term only
    when its weight is non-zero."""
    total, parts = 0.0, {}
    for k in pred:
        e, t = pred[k], tgt[k]
        ez, tz = e - e.mean(-1, keepdim=True), t - t.mean(-1, keepdim=True)
        scale = (ez * tz).sum(-1, keepdim=True) / ((tz ** 2).sum(-1, keepdim=True) + eps)
        st = scale * tz
        sisdr = 10 * torch.log10(((st ** 2).sum(-1) + eps) / (((ez - st) ** 2).sum(-1) + eps))
        parts[f"{k}_si_sdr"], parts[f"{k}_l1"] = -sisdr.mean(), (e - t).abs().mean()
        total = total + w_sisdr * parts[f"{k}_si_sdr"] + w_l1 * parts[f"{k}_l1"]
        if w_spec:
            win = torch.hann_window(n_fft, dtype=e.dtype)
            me = torch.log1p(torch.stft(e, n_fft, hop, window=win, return_complex=True).abs())
            mt = torch.log1p(torch.stft(t, n_fft, hop, window=win, return_complex=True).abs())
            parts[f"{k}_spectral"] = (me - mt).abs().mean()
            total = total + w_spec * parts[f"{k}_spectral"]
    return total, parts


def _reference_step(cfg, sd, mix, tgt, weights):
    """-> (total loss, {state_dict key: gradient}) from torch autograd in float64 on the CPU."""
    names = oracle.locoformer_oracle.SOURCE_NAMES[: cfg["n_sources"]]
    targets = {n: tgt[i].double() for i, n in enumerate(names)}
    if build_ref.available():
        classes = build_ref.load()
        from models.mss_loss import MSSLoss            # the reference's own loss (oracle/_ref)
        model = classes["TFLocoformerMSS"](**cfg)
        model.load_state_dict(sd, strict=True)
        model = model.double().eval()                   # eval: dropout is 0 anyway; keeps the flash flag path simple
        pred = model(mix.double())
        crit = MSSLoss(loss_type="combined", si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
        out = crit(pred, targets)
        loss = out["total_loss"]
        loss.backward()
        grads = {k: p.grad for k, p in dict(model.state_dict(keep_vars=True)).items() if p.grad is not None}
        return float(loss), grads, {k: float(v) for k, v in out.items() if k != "total_loss"}
    sd64 = {k: v.detach().double().clone().requires_grad_(not k.endswith("rope.freqs")) for k, v in sd.items()}
    pred = oracle.mss_forward(sd64, dict(cfg), mix.double(), dtype=torch.float64)
    loss, parts = _ref_loss(pred, targets, *weights)
    loss.backward()
    return (float(loss.detach()), {k: v.grad for k, v in sd64.items() if v.grad is not None},
            {k: float(v.detach()) for k, v in parts.items()})


@pytest.mark.parametrize("cfg,n_samples,batch,weights", [
    (SMALL, 6000, 2, (1.0, 0.1, 0.1)),
    (dict(SMALL, tf_order="tf", ffn_type="swiglu_conv1d", ffn_hidden_dim=64), 5000, 1, (1.0, 0.1, 0.15)),
    (SMALL, 3000, 1, (1.0, 0.5, 0.0)),
])
def test_train_step_gradients_vs_reference_autograd(pkg, train_mode, cfg, n_samples, batch, weights):
    gemm_mode = train_mode
    """tfl_train_forward_backward: total loss, per-source components and EVERY parameter gradient of
    TFLocoformerMSS + MSSLoss against the reference's autograd."""
    from mss_tf_locoformer_b200.training import Trainer
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(n_samples, batch)
    g = torch.Generator().manual_seed(9)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(cfg["n_sources"], batch, n_samples, generator=g)
    want_loss, want_grads, parts = _reference_step(cfg, sd, mix, tgt, weights)
    model = model.cuda()
    tr = Trainer(model, si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
    loss, audio = tr.forward_backward(mix.cuda(), tgt.cuda(), want_audio=True)
    loss = loss.cpu()
    tol = TOL[gemm_mode]
    assert abs(float(loss[0]) - want_loss) <= tol["loss"] * max(1.0, abs(want_loss)), (float(loss[0]), want_loss)
    names = oracle.locoformer_oracle.SOURCE_NAMES[: cfg["n_sources"]]
    for i, n in enumerate(names):
        for j, part in enumerate(("si_sdr", "l1", "spectral")):
            if f"{n}_{part}" in parts:
                assert abs(float(loss[1 + 3 * i + j]) - parts[f"{n}_{part}"]) <= tol["loss"] * max(1.0, abs(parts[f"{n}_{part}"])), (n, part)
    worst, worst_key = 0.0, None
    trainable = [k for k in tr.engine.keys if not k.endswith("rope.freqs")]
    assert set(trainable) == set(want_grads), set(trainable) ^ set(want_grads)
    errs = {k: _rel(tr.grad_of(k), want_grads[k]) for k in trainable}
    worst_key = max(errs, key=errs.get)
    worst = errs[worst_key]
    print(f"[{gemm_mode}] worst relative gradient error {worst:.2e} ({worst_key}) over {len(trainable)} tensors; "
          f"loss {float(loss[0]):.5f} vs {want_loss:.5f}")
    assert worst < tol["step"], (worst_key, worst)
    print(f"worst relative gradient error {worst:.2e} over {len(trainable)} tensors; loss {float(loss[0]):.5f} vs {want_loss:.5f}")


def test_clip_and_adamw_match_torch(pkg):
    """tfl_grad_clip_norm + tfl_adamw_step against torch.nn.utils.clip_grad_norm_ + torch.optim.AdamW, three steps."""
    import ctypes as C
    from mss_tf_locoformer_b200 import _lib
    from mss_tf_locoformer_b200.engine import _stream
    lib = _lib.load()
    g = torch.Generator().manual_seed(2)
    n = 100_003
    p0 = torch.randn(n, generator=g)
    ref = torch.nn.Parameter(p0.clone().cuda())
    opt = torch.optim.AdamW([ref], lr=3e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    p = p0.clone().cuda()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    norm = torch.zeros(2, device="cuda")
    scratch = torch.zeros(592, dtype=torch.float64, device="cuda")
    for step in range(1, 4):
        grad = (torch.randn(n, generator=g) * (0.5 if step == 2 else 0.001)).cuda()   # step 2 is clipped, 1 and 3 are not
        ref.grad = grad.clone()
        total = torch.nn.utils.clip_grad_norm_([ref], max_norm=5.0)
        opt.step()
        assert lib.tfl_grad_clip_norm(grad.data_ptr(), n, 5.0, norm.data_ptr(), scratch.data_ptr(), scratch.numel() * 8, _stream()) == 0
        assert lib.tfl_adamw_step(p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), n, norm.data_ptr(), 3e-3, 0.9,
                                  0.999, 1e-8, 0.01, step, _stream()) == 0
        torch.cuda.synchronize()
        assert abs(float(norm[0]) - float(total)) <= 1e-5 * float(total)
        assert float((p - ref.detach()).abs().max()) <= 2e-6, step


def test_trainer_steps_follow_reference_optimiser(pkg):
    """Three Trainer.step calls on a fixed batch against the same steps of the reference model under torch AdamW
    (float64, CPU): the parameter updates agree and the loss goes down."""
    from mss_tf_locoformer_b200.training import Trainer
    cfg = dict(SMALL, n_layers=1)
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(4000, 1)
    g = torch.Generator().manual_seed(4)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(cfg["n_sources"], 1, 4000, generator=g)
    weights = (1.0, 0.1, 0.1)
    names = oracle.locoformer_oracle.SOURCE_NAMES[: cfg["n_sources"]]
    # reference loop
    if build_ref.available():
        classes = build_ref.load()
        from models.mss_loss import MSSLoss
        ref = classes["TFLocoformerMSS"](**cfg)
        ref.load_state_dict(sd, strict=True)
        ref = ref.double().eval()
        crit = MSSLoss(loss_type="combined", si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
        params = [p for p in ref.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=0.01, eps=1e-8)
        ref_losses = []
        for _ in range(3):
            opt.zero_grad(set_to_none=True)
            loss = crit(ref(mix.double()), {n: tgt[i].double() for i, n in enumerate(names)})["total_loss"]
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, max_norm=5.0)
            opt.step()
            ref_losses.append(float(loss))
        ref_sd = {k: v.detach() for k, v in ref.state_dict().items()}
    else:                                                # the oracle forward + the MSSLoss restatement, same loop
        sd64 = {k: v.detach().double().clone().requires_grad_(not k.endswith("rope.freqs")) for k, v in sd.items()}
        params = [v for v in sd64.values() if v.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=0.01, eps=1e-8)
        ref_losses = []
        for _ in range(3):
            opt.zero_grad(set_to_none=True)
            pred = oracle.mss_forward(sd64, dict(cfg), mix.double(), dtype=torch.float64)
            loss, _ = _ref_loss(pred, {n: tgt[i].double() for i, n in enumerate(names)}, *weights)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, max_norm=5.0)
            opt.step()
            ref_losses.append(float(loss.detach()))
        ref_sd = {k: v.detach() for k, v in sd64.items()}
    model = model.cuda()
    tr = Trainer(model, lr=1e-3, weight_decay=0.01, si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
    losses = [float(tr.step(mix.cuda(), tgt.cuda())[0]) for _ in range(3)]      # default mode: mixed
    assert losses[2] < losses[0], losses
    got_sd = model.state_dict()
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 1e-2 * max(1.0, abs(b)), (losses, ref_losses)
    num = den = 0.0
    for k in tr.engine.keys:
        if k.endswith("rope.freqs"):
            continue
        upd_ref = ref_sd[k].double() - sd[k].double()
        upd_got = got_sd[k].detach().double().cpu() - sd[k].double()
        num += float((upd_got - upd_ref).pow(2).sum())
        den += float(upd_ref.pow(2).sum())
    assert math.sqrt(num / den) < 0.10, math.sqrt(num / den)   # Adam normalises: the update error ~ the gradient's direction error
    # the forward path sees the updated weights (packed image refreshed after the optimiser kernels)
    with torch.no_grad():
        out = model(mix.cuda())
    assert all(torch.isfinite(v).all() for v in out.values())


def _dp_worker(rank, world, port, cfg, sd, mix, tgt, ret):
    import os
    import torch.distributed as dist
    import mss_tf_locoformer_b200 as m
    from mss_tf_locoformer_b200 import _lib
    from mss_tf_locoformer_b200.training import Trainer, allreduce_mean_
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        _lib.load().tfl_debug_set_option(5, 0)          # exact fp32 GEMMs: the comparison below is tight
        model = m.TFLocoformerMSS(**cfg)
        model.load_state_dict(sd, strict=True)
        tr = Trainer(model.cuda(), lr=1e-3)
        loss, _ = tr.forward_backward(mix[rank:rank + 1].cuda(), tgt[:, rank:rank + 1].cuda())
        allreduce_mean_(tr.grads)
        tr.optimizer_step()
        torch.cuda.synchronize()
        ret[rank] = (tr.grads.cpu(), tr.params.cpu(), loss.cpu())
    finally:
        dist.destroy_process_group()


def test_data_parallel_two_gpus_matches_one_gpu_batch_of_two(pkg):
    """One sample per rank + NCCL gradient average == one GPU on the batch of two (every loss term is a batch mean):
    gradients, the clipped AdamW update and the replicas' parameters agree."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    from mss_tf_locoformer_b200 import _lib
    from mss_tf_locoformer_b200.training import Trainer
    cfg = dict(SMALL, n_layers=1)
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(4000, 2)
    g = torch.Generator().manual_seed(4)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(cfg["n_sources"], 2, 4000, generator=g)
    lib = _lib.load()
    lib.tfl_debug_set_option(5, 0)
    try:
        tr = Trainer(model.cuda(), lr=1e-3)
        loss, _ = tr.forward_backward(mix.cuda(), tgt.cuda())
        grads_one = tr.grads.cpu().clone()
        tr.optimizer_step()
        torch.cuda.synchronize()
        params_one = tr.params.cpu().clone()
    finally:
        lib.tfl_debug_set_option(5, 2)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_dp_worker, args=(2, port, cfg, sd, mix, tgt, ret), nprocs=2, join=True)
        res = dict(ret)
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])      # replicas stay identical
    assert _rel(res[0][0], grads_one) < 1e-4, _rel(res[0][0], grads_one)
    assert float((res[0][1] - params_one).abs().max()) <= 2e-4                           # lr 1e-3: a flipped sign would be 2e-3
    assert abs(float(0.5 * (res[0][2][0] + res[1][2][0])) - float(loss[0])) <= 1e-4 * abs(float(loss[0]))


def test_train_step_variant_d_widths_one_layer(pkg, train_mode):
    """The whole step at production widths (n_fft 2048, emb 128, hidden 384, head_dim 32; one layer, 0.55 s of audio):
    every tcgen05 forward kernel of the mixed mode and the 128-wide GEMM tiles of the backward pass."""
    from mss_tf_locoformer_b200.training import Trainer
    from test_gpu_parity import VARIANT_D
    cfg = dict(VARIANT_D, flash_attention=False)
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(24000, 1)
    g = torch.Generator().manual_seed(21)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(4, 1, 24000, generator=g)
    weights = (1.0, 0.1, 0.15)
    want_loss, want_grads, _ = _reference_step(cfg, sd, mix, tgt, weights)
    tr = Trainer(model.cuda(), si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
    loss, _ = tr.forward_backward(mix.cuda(), tgt.cuda())
    tol = TOL[train_mode]
    assert abs(float(loss[0]) - want_loss) <= tol["loss"] * max(1.0, abs(want_loss)), (float(loss[0]), want_loss)
    errs = {k: _rel(tr.grad_of(k), want_grads[k]) for k in want_grads}
    worst_key = max(errs, key=errs.get)
    print(f"[{train_mode}] Variant-D widths: worst relative gradient error {errs[worst_key]:.2e} ({worst_key})")
    assert errs[worst_key] < tol["step"], (worst_key, errs[worst_key])


def test_train_step_xlarge_widths_one_layer(pkg, train_mode):
    """musdb18_rtx5090_xlarge.yaml widths (emb 256, 16 heads x 16, 8 groups, hidden 1024) at a small n_fft, one layer: two
    128-wide tiles along every GEMM dimension, head_dim 16, and -- in mixed mode -- the tcgen05 FFN forward at emb 256 with
    the attention (outside the tcgen05 kernel's shapes) on the tf32 path."""
    from mss_tf_locoformer_b200.training import Trainer
    cfg = dict(SMALL, n_layers=1, emb_dim=256, attention_dim=256, n_heads=16, num_groups=8, ffn_hidden_dim=[1024, 1024])
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(3000, 1)
    g = torch.Generator().manual_seed(31)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(4, 1, 3000, generator=g)
    weights = (1.0, 0.1, 0.15)
    want_loss, want_grads, _ = _reference_step(cfg, sd, mix, tgt, weights)
    tr = Trainer(model.cuda(), si_sdr_weight=weights[0], l1_weight=weights[1], spectral_weight=weights[2])
    loss, _ = tr.forward_backward(mix.cuda(), tgt.cuda())
    tol = TOL[train_mode]
    assert abs(float(loss[0]) - want_loss) <= tol["loss"] * max(1.0, abs(want_loss)), (float(loss[0]), want_loss)
    errs = {k: _rel(tr.grad_of(k), want_grads[k]) for k in want_grads}
    worst_key = max(errs, key=errs.get)
    print(f"[{train_mode}] xlarge widths: worst relative gradient error {errs[worst_key]:.2e} ({worst_key})")
    assert errs[worst_key] < tol["step"], (worst_key, errs[worst_key])


def test_gradient_accumulation_and_resume(pkg):
    """train.py:117-146 with gradient_accumulation_steps = 2: two micro-batches of one sample == one step on the batch of
    two (every loss term is a batch mean); and a Trainer restored from state_dict() continues bit-identically."""
    from mss_tf_locoformer_b200 import _lib
    from mss_tf_locoformer_b200.training import Trainer
    cfg = dict(SMALL, n_layers=1)
    model_a = _random_model(pkg, cfg).cuda()
    sd = {k: v.detach().clone() for k, v in model_a.state_dict().items()}
    mix = _mixture(4000, 2).cuda()
    g = torch.Generator().manual_seed(4)
    tgt = (0.25 * mix.cpu()[None] + 0.05 * torch.randn(4, 2, 4000, generator=g)).cuda()
    lib = _lib.load()
    lib.tfl_debug_set_option(5, 0)                       # exact fp32: the two orders of summation agree to rounding
    try:
        tr_a = Trainer(model_a, lr=1e-3)
        tr_a.step(mix, tgt)
        model_b = pkg.TFLocoformerMSS(**cfg)
        model_b.load_state_dict(sd)
        tr_b = Trainer(model_b.cuda(), lr=1e-3, gradient_accumulation_steps=2)
        tr_b.step(mix[0:1], tgt[:, 0:1])
        assert tr_b.step_count == 0                      # first micro-batch: no optimiser step yet
        tr_b.step(mix[1:2], tgt[:, 1:2])
        assert tr_b.step_count == 1
        assert float((tr_a.params - tr_b.params).abs().max()) <= 2e-4     # lr 1e-3: a flipped update would be 2e-3
        # resume: a fresh Trainer on the saved model + optimiser state takes the same second step
        opt_state = tr_a.state_dict()
        model_c = pkg.TFLocoformerMSS(**cfg)
        model_c.load_state_dict({k: v.detach().clone() for k, v in model_a.state_dict().items()})
        tr_c = Trainer(model_c.cuda(), lr=5e-4)
        tr_c.load_state_dict(opt_state)
        assert tr_c.lr == tr_a.lr and tr_c.step_count == 1
        tr_a.step(mix, tgt)
        tr_c.step(mix, tgt)
        assert float((tr_a.params - tr_c.params).abs().max()) <= 2e-5     # same inputs; atomics order only
        assert set(opt_state["exp_avg"]) == {k for k in sd if not k.endswith("rope.freqs")}
    finally:
        lib.tfl_debug_set_option(5, 2)
