"""Training-step time of TFLocoformerMSS through torch autograd (``differentiable = True``) against training.Trainer.

Variant D (bench.py: 6 layers, emb 128, n_fft 2048, hop 1024), one 6-s sample, mixed arithmetic (TFL_OPT_TRAIN_MODE 2).
CUDA events per step, median of --steps after --warmup, and the peak device memory of the timed steps:

- ``trainer``: ``Trainer.step`` -- the CUDA MSSLoss, clip_grad_norm_(5) and AdamW as kernels;
- ``autograd``: forward, the same MSSLoss restated in torch (SI-SDR + 0.1 L1 + 0.1 log-magnitude L1 at n_fft 2048,
  hop 1024), ``loss.backward()`` and ``torch.optim.AdamW.step()``;
- ``autograd_mixture_grad``: the same with a mixture that requires grad (adds the encoder input gradient, the adjoint
  STFT frames and the reflect-padding fold).

Then a torch.profiler pass over --steps backward calls of the last case gives the device time of the two input-gradient
kernels; ``floor_us`` is the bytes each must move at the 6 550 GB/s copy bandwidth of DESIGN.md section 5 (derived, not
measured here).

    python profiles/time_mss_autograd.py [--steps 10] [--warmup 3] [--out profiles/mss_autograd_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mss_tf_locoformer_b200 as pkg  # noqa: E402
from mss_tf_locoformer_b200.modules import SOURCE_NAMES  # noqa: E402
from mss_tf_locoformer_b200.training import Trainer  # noqa: E402

VARIANT_D = dict(n_fft=2048, hop_length=1024, n_sources=4, n_layers=6, emb_dim=128, norm_type="rmsgroupnorm",
                 num_groups=4, tf_order="ft", n_heads=4, flash_attention=True, attention_dim=128, pos_enc="rope",
                 ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[384, 384], conv1d_kernel=4,
                 conv1d_shift=1, dropout=0.0, eps=1e-5)
T = 264600                       # 6 s at 44.1 kHz
COPY_GBS = 6550.0                # DESIGN.md section 5: device-to-device copy bandwidth


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = line.partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def mss_loss(pred, tgt, w=(1.0, 0.1, 0.1), eps=1e-8, n_fft=2048, hop=1024):
    """MSSLoss(loss_type='combined') in torch, the loss Trainer computes with kernels."""
    total = 0.0
    win = torch.hann_window(n_fft, device=tgt.device)
    for i, k in enumerate(pred):
        e, t = pred[k], tgt[i]
        ez, tz = e - e.mean(-1, keepdim=True), t - t.mean(-1, keepdim=True)
        scale = (ez * tz).sum(-1, keepdim=True) / ((tz ** 2).sum(-1, keepdim=True) + eps)
        st = scale * tz
        sisdr = 10 * torch.log10(((st ** 2).sum(-1) + eps) / (((ez - st) ** 2).sum(-1) + eps))
        me = torch.log1p(torch.stft(e, n_fft, hop, window=win, return_complex=True).abs())
        mt = torch.log1p(torch.stft(t, n_fft, hop, window=win, return_complex=True).abs())
        total = total + w[0] * -sisdr.mean() + w[1] * (e - t).abs().mean() + w[2] * (me - mt).abs().mean()
    return total


def _time(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    times = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return {"median_ms": times[len(times) // 2], "min_ms": times[0], "max_ms": times[-1], "steps": steps,
            "warmup": warmup, "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30,
            "resident_mem_gib": base / 2 ** 30}


def _model(dev):
    torch.manual_seed(0)
    return pkg.TFLocoformerMSS(**VARIANT_D).to(dev).train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: there is no CPU timing")
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    mix = 0.1 * torch.randn(1, T, device=dev, generator=g)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(4, 1, T, device=dev, generator=g)
    res = {"gpu": _gpu(), "arithmetic": "mixed (TFL_OPT_TRAIN_MODE 2)",
           "shape": "TFLocoformerMSS Variant D (6 layers, emb 128, n_fft 2048, hop 1024), batch 1 x 264600 samples",
           "timing": "CUDA events per step after warm-up", "cases": {}}

    model = _model(dev)
    tr = Trainer(model, lr=1e-4)
    r = _time(lambda: tr.step(mix, tgt), args.steps, args.warmup)
    r["step"] = "Trainer.step: CUDA MSSLoss + backward + clip_grad_norm_(5) + AdamW kernels"
    res["cases"]["trainer"] = r
    del tr, model
    torch.cuda.empty_cache()

    for name, x in (("autograd", mix), ("autograd_mixture_grad", mix.clone().requires_grad_(True))):
        model = _model(dev)
        model.differentiable = True
        opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-4)

        def step():
            opt.zero_grad(set_to_none=False)
            if x.requires_grad:
                x.grad = None
            mss_loss(model(x), tgt).backward()
            opt.step()

        r = _time(step, args.steps, args.warmup)
        r["step"] = "forward + MSSLoss in torch + backward() + torch.optim.AdamW.step()" + \
            (" with a mixture that requires grad" if x.requires_grad else "")
        res["cases"][name] = r
        if x.requires_grad:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    step()
                torch.cuda.synchronize()
            kt = {}
            for ev in prof.key_averages():
                for k in ("enc_input_grad_kernel", "stft_fold_kernel", "stft_adj_frames_kernel"):
                    if k in ev.key:
                        kt[k] = {"calls": ev.count, "mean_us": ev.device_time_total / max(ev.count, 1)}
            Tf, F, C = 1 + T // 1024, 1025, 128
            n = Tf * F
            floors = {"enc_input_grad_kernel": (2 * n * C * 4 + 2 * n * 4, "v and dy read once, d spec written"),
                      "stft_fold_kernel": (Tf * 2048 * 4 + T * 4, "adjoint frames read once, d mixture written")}
            for k, (nbytes, what) in floors.items():
                if k in kt:
                    kt[k]["floor_bytes"] = nbytes
                    kt[k]["floor_us"] = nbytes / (COPY_GBS * 1e3)
                    kt[k]["floor_is"] = what
                    kt[k]["fraction_of_floor"] = kt[k]["floor_us"] / kt[k]["mean_us"]
            res["input_gradient_kernels"] = kt
        del model, opt
        torch.cuda.empty_cache()
    res["autograd_over_trainer"] = res["cases"]["autograd"]["median_ms"] / res["cases"]["trainer"]["median_ms"]
    res["mixture_grad_extra_ms"] = (res["cases"]["autograd_mixture_grad"]["median_ms"]
                                    - res["cases"]["autograd"]["median_ms"])
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
