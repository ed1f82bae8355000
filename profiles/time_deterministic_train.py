"""Cost of the deterministic training mode (``torch.use_deterministic_algorithms(True)`` -> TFL_OPT_DETERMINISTIC).

Two training steps, each timed in one process with the flag off and on in alternation (CUDA events per step, median of
--steps after --warmup steps of each), with the kernel launches of one step and the training workspace of each mode:

- ``trainer``: ``Trainer.step`` at Variant D (bench.py: 6 layers, emb 128, n_fft 2048, hop 1024), one 6-s sample, mixed
  arithmetic (TFL_OPT_TRAIN_MODE 2).  Two Trainers over two copies of the same model, one per mode, so neither
  reallocates its workspace when the flag changes.
- ``separator``: forward + backward + ``torch.optim.AdamW.step()`` of TFLocoformerSeparator at the WHAMR! widths of
  profiles/time_separator_train.py (batch 4 x 501 frames x 129 bins), mixed arithmetic.

torch fills uninitialised memory with NaN under the deterministic flag; that fill is switched off here
(``torch.utils.deterministic.fill_uninitialized_memory = False``) so the numbers are the library's cost alone.

    python profiles/time_deterministic_train.py [--steps 10] [--warmup 3] [--out profiles/deterministic_train_b200.json]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import mss_tf_locoformer_b200 as pkg  # noqa: E402
from mss_tf_locoformer_b200 import _lib  # noqa: E402
from mss_tf_locoformer_b200.training import Trainer  # noqa: E402
from time_mss_autograd import T, VARIANT_D, _gpu  # noqa: E402
from time_separator_train import WHAMR  # noqa: E402


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _launches(fn):
    lib = _lib.load()
    torch.cuda.synchronize()
    n0 = lib.tfl_launch_count()
    fn()
    torch.cuda.synchronize()
    return int(lib.tfl_launch_count() - n0)


def _compare(steps_by_mode, steps, warmup):
    """steps_by_mode: {False: fn, True: fn}; each fn runs one step with the flag already set."""
    res = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        for _ in range(warmup):
            steps_by_mode[det]()
        res[det] = {"launches_per_step": _launches(steps_by_mode[det]), "times": []}
    for _ in range(steps):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            res[det]["times"].append(_timed(steps_by_mode[det]))
    torch.use_deterministic_algorithms(False)
    out = {}
    for det, r in res.items():
        t = sorted(r["times"])
        out["deterministic" if det else "default"] = {"median_ms": t[len(t) // 2], "min_ms": t[0], "max_ms": t[-1],
                                                      "launches_per_step": r["launches_per_step"]}
    d, o = out["default"], out["deterministic"]
    out["overhead_pct"] = 100.0 * (o["median_ms"] - d["median_ms"]) / d["median_ms"]
    out["extra_launches_per_step"] = o["launches_per_step"] - d["launches_per_step"]
    out["steps"], out["warmup"] = steps, warmup
    return out


def _trainer_case(dev, steps, warmup):
    lib = _lib.load()
    torch.manual_seed(0)
    src = pkg.TFLocoformerMSS(**VARIANT_D)
    sd = src.state_dict()
    mix = 0.1 * torch.randn(1, T, device=dev)
    tgt = 0.25 * mix[None] + 0.05 * torch.randn(VARIANT_D["n_sources"], 1, T, device=dev)
    trainers = {}
    for det in (False, True):
        m = pkg.TFLocoformerMSS(**VARIANT_D)
        m.load_state_dict(sd)
        trainers[det] = Trainer(m.to(dev).train())
    ws = {}
    for det in (False, True):
        with _lib.deterministic_option(det):
            ws[det] = lib.tfl_train_workspace_bytes(trainers[det].engine.plan, 1, T, 2048, 1024)
    r = _compare({det: (lambda tr=tr: tr.step(mix, tgt)) for det, tr in trainers.items()}, steps, warmup)
    r["workspace_gib"] = {"default": ws[False] / 2 ** 30, "deterministic": ws[True] / 2 ** 30}
    r["shape"] = "Trainer.step, Variant D (6 layers, emb 128, n_fft 2048, hop 1024), 1 x 6 s at 44.1 kHz, mixed mode"
    return r


def _separator_case(dev, steps, warmup):
    torch.manual_seed(0)
    sep = pkg.TFLocoformerSeparator(**WHAMR).to(dev).train()
    sep.differentiable = True
    spec = torch.randn(4, 501, 129, dtype=torch.complex64, device=dev)
    opt = torch.optim.AdamW([p for p in sep.parameters() if p.requires_grad], lr=1e-4)
    g = torch.Generator(device=dev).manual_seed(1)
    G = torch.randn((4, WHAMR["num_spk"], 501, 129), dtype=torch.complex64, device=dev, generator=g)

    def step():
        opt.zero_grad(set_to_none=False)
        est = sep(spec)
        ((est.real * G.real).sum() + (est.imag * G.imag).sum()).backward()
        opt.step()

    lib = _lib.load()
    eng = sep._ready()
    ws = {}
    for det in (False, True):
        with _lib.deterministic_option(det):
            ws[det] = lib.tfl_sep_train_workspace_bytes(eng.plan, 4, 501, 129)
    r = _compare({False: step, True: step}, steps, warmup)
    r["workspace_gib"] = {"default": ws[False] / 2 ** 30, "deterministic": ws[True] / 2 ** 30}
    r["shape"] = ("TFLocoformerSeparator forward + backward + AdamW.step(), WHAMR! widths (emb 128, 6 layers, K 8, "
                  "hidden [192, 192]), batch 4 x 501 frames x 129 bins, mixed mode")
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: there is no CPU timing")
    dev = torch.device("cuda:0")
    torch.utils.deterministic.fill_uninitialized_memory = False
    res = {"gpu": _gpu(), "arithmetic": "mixed (TFL_OPT_TRAIN_MODE 2)",
           "timing": "CUDA events per step, flag off / on alternating, median after warm-up", "cases": {}}
    res["cases"]["trainer"] = _trainer_case(dev, args.steps, args.warmup)
    torch.cuda.empty_cache()
    res["cases"]["separator"] = _separator_case(dev, args.steps, args.warmup)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
