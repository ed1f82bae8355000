"""The tf32 precision mode against the fp32 and bf16 modes, in one process, with the card's name and power limit.

- ``variant_d``: TFLocoformerMSS at Variant D (6 layers, emb 128, n_fft 2048, hop 1024), batch 8 x 6 s: ms per forward
  and audio-s/s in the fp32, tf32 and bf16 modes, timed in alternation (CUDA events, median of --steps after --warmup
  forwards of every mode).
- ``ffn``: one frequency-axis ConvSwiGLU FFN call (tfl_conv_swiglu_ffn) at the same shape, tf32 vs fp32 (CUDA events,
  median over --ffn-reps calls).  Algorithmic FLOP = 6 K C hid B Tf (F + K - 1); the rate is given as a share of the
  1,125 TFLOP/s dense TF32 data-sheet figure of one B200 at 1,000 W, and the tf32 time as a share of the fp32 time.
- ``xlarge``: the musdb18_rtx5090_xlarge widths (12 layers, emb 256, 16 heads x 16, hidden 1024, n_fft 4096), batch
  1 x 15 s: fp32 vs tf32 ms per forward (this model has no bf16 mode: its attention shape is outside the bf16 kernels).

    python profiles/time_tf32.py [--steps 3] [--warmup 1] [--out profiles/tf32_b200.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import mss_tf_locoformer_b200 as pkg  # noqa: E402
from time_mss_autograd import T, VARIANT_D, _gpu  # noqa: E402

XLARGE = dict(VARIANT_D, n_fft=4096, n_layers=12, emb_dim=256, num_groups=8, n_heads=16, attention_dim=256,
              ffn_hidden_dim=[1024, 1024])
T_XL = 661500                      # 15 s at 44.1 kHz
TF32_PEAK = 1125.0                 # TFLOP/s, dense TF32, HGX B200 data sheet per GPU


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _mixture(batch, n, seed):
    g = torch.Generator().manual_seed(seed)
    return (0.1 * torch.randn(batch, n, generator=g)).cuda()


def _model(cfg):
    torch.manual_seed(0)
    return pkg.TFLocoformerMSS(**cfg).cuda().eval()


def _alternate(model, mix, modes, steps, warmup):
    def fwd(mode):
        model.precision = mode
        with torch.no_grad():
            model(mix)
    for mode in modes:
        for _ in range(warmup):
            fwd(mode)
    times = {m: [] for m in modes}
    for _ in range(steps):
        for mode in modes:
            times[mode].append(_timed(lambda: fwd(mode)))
    return {m: statistics.median(v) for m, v in times.items()}, times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--ffn-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"gpu": _gpu(), "steps": args.steps, "warmup": args.warmup}

    B, secs = 8, T / 44100.0
    model = _model(VARIANT_D)
    mix = _mixture(B, T, 1)
    med, raw = _alternate(model, mix, ("fp32", "tf32", "bf16"), args.steps, args.warmup)
    res["variant_d"] = {"batch": B, "seconds": secs, "ms_per_step": med, "raw_ms": raw,
                        "audio_s_per_s": {m: B * secs / (v / 1000.0) for m, v in med.items()}}
    print(json.dumps({"variant_d": res["variant_d"]}), flush=True)

    eng = model._ready()
    Tf, F, C, K, H = 1 + T // VARIANT_D["hop_length"], VARIANT_D["n_fft"] // 2 + 1, 128, 4, 384
    x = torch.randn(B, Tf, F, C, generator=torch.Generator().manual_seed(2)).cuda()
    ffn = {}
    for prec, name in ((2, "tf32"), (0, "fp32")):
        eng.ffn_(0, 0, 0, x, prec)                           # warm-up (and workspace) of this shape
        ffn[name] = statistics.median(_timed(lambda: eng.ffn_(0, 0, 0, x, prec)) for _ in range(args.ffn_reps))
    flop = 6.0 * K * C * H * B * Tf * (F + K - 1)
    tflops = flop / (ffn["tf32"] / 1000.0) / 1e12
    res["ffn"] = {"shape": [B, Tf, F, C], "axis": "freq", "hidden": H, "kernel": K, "flop": flop, "ms": ffn,
                  "tf32_tflops": tflops, "tf32_share_of_datasheet": tflops / TF32_PEAK,
                  "fp32_tflops": flop / (ffn["fp32"] / 1000.0) / 1e12, "tf32_time_share_of_fp32": ffn["tf32"] / ffn["fp32"]}
    print(json.dumps({"ffn": res["ffn"]}), flush=True)
    del model, eng, x, mix
    torch.cuda.empty_cache()

    xl = _model(XLARGE)
    mix = _mixture(1, T_XL, 3)
    med, raw = _alternate(xl, mix, ("fp32", "tf32"), args.steps, args.warmup)
    res["xlarge"] = {"batch": 1, "seconds": T_XL / 44100.0, "ms_per_step": med, "raw_ms": raw,
                     "speedup_tf32": med["fp32"] / med["tf32"]}
    print(json.dumps({"xlarge": res["xlarge"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
