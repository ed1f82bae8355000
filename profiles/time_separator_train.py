"""Training-step time of the spectrogram separators through torch autograd (``differentiable = True``).

Times forward + backward + ``torch.optim.AdamW.step()`` with CUDA events after warm-up, in the default mixed arithmetic
(TFL_OPT_TRAIN_MODE 2), and records the peak device memory of a step.  Two shapes:

- ``whamr``: TFLocoformerSeparator at the WHAMR! recipe's widths as SURVEY.md section 8 cites them (emb 128, 6 layers,
  4 heads, K = 8, hidden [192, 192], n_fft 256 -> F = 129), batch 4 x 501 frames.  501 frames = a 4-s segment at 8 kHz
  with hop 64; the recipe file itself is not in this repository, so the segment length is an assumption.
- ``bs_config4``: BSLocoformerSeparator at BASELINE config 4 (stereo, 4 sources, 62 bands, emb 128, 6 layers, masking),
  batch 1 x 259 frames (6 s at 44.1 kHz, hop 1024).

    python profiles/time_separator_train.py [--steps 10] [--warmup 3] [--out profiles/separator_train_b200.json]

Prints one JSON object (and writes it to --out) with the GPU name and power limit beside every number.
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

WHAMR = dict(num_spk=2, n_layers=6, emb_dim=128, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
             attention_dim=128, pos_enc="rope", ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[192, 192],
             conv1d_kernel=8, conv1d_shift=1, dropout=0.0, eps=1e-5)
BS4 = dict(num_spk=4, n_layers=6, emb_dim=128, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           attention_dim=128, pos_enc="rope", ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[384, 384],
           conv1d_kernel=4, conv1d_shift=1, dropout=0.0, sample_rate=44100, stft_size=2048, eps=1e-5, masking=True,
           stereo=True)


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = line.partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def _time(model, spec, steps, warmup):
    g = torch.Generator(device=spec.device).manual_seed(1)
    opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-4)
    with torch.no_grad():
        est = model(spec)
    G = torch.randn(est.shape, dtype=est.dtype, device=spec.device, generator=g)
    del est

    def step():
        opt.zero_grad(set_to_none=False)
        est = model(spec)
        loss = (est.real * G.real).sum() + (est.imag * G.imag).sum()
        loss.backward()
        opt.step()

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: there is no CPU timing")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    res = {"gpu": _gpu(), "arithmetic": "mixed (TFL_OPT_TRAIN_MODE 2)", "step": "forward + backward + AdamW.step()",
           "timing": "CUDA events per step after warm-up", "shapes": {}}
    sep = pkg.TFLocoformerSeparator(**WHAMR).to(dev).train()
    sep.differentiable = True
    spec = torch.randn(4, 501, 129, dtype=torch.complex64, device=dev)
    r = _time(sep, spec, args.steps, args.warmup)
    r["shape"] = "TFLocoformerSeparator, WHAMR! widths (emb 128, 6 layers, K 8, hidden [192, 192]), batch 4 x 501 frames x 129 bins"
    res["shapes"]["whamr"] = r
    del sep, spec
    torch.cuda.empty_cache()
    bs = pkg.BSLocoformerSeparator(**BS4).to(dev).train()
    bs.differentiable = True
    spec = torch.randn(1, 2, 259, 1025, dtype=torch.complex64, device=dev)
    r = _time(bs, spec, args.steps, args.warmup)
    r["shape"] = "BSLocoformerSeparator, BASELINE config 4 (stereo, 4 sources, 62 bands, emb 128, 6 layers), batch 1 x 259 frames"
    res["shapes"]["bs_config4"] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
