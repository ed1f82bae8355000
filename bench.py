#!/usr/bin/env python
"""Headline benchmark: separated audio-seconds per second of TFLocoformerMSS on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-gpu]
                    [--precision bf16|fp32] [--variant D|Y] [--batch B] [--track SECONDS] [--model mss|bs]
                    [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float32): the separated sources of the
forward and --track runs, the complex estimate of --model bs as `est` (real and imaginary parts in a last axis of 2).
Weights and inputs are seeded, so two builds run with the same arguments can be compared output for output.

Workload (BASELINE.json configs[1], "Variant D" of SURVEY.md F4): n_fft 2048, hop 1024, 6 layers,
emb_dim 128, 4 heads, macaron ConvSwiGLU [384, 384], 4 sources; one step = one batch of 6-s 44.1 kHz
mono segments (stereo mixture averaged to mono, as every reference caller does) through
forward(mixture) -> dict of sources.  Random-init weights, synthetic mixtures.  N > 1: one process
per GPU (torchrun), each rank separates its own batch every step (segment sharding, no data-path
collective), time = max over ranks.

Multi-rank discipline: the process group is torn down right after the last timed collective; every
rank-0-only leg (kernel micro-timing, CPU baseline) runs after that, so no peer ever sits in an NCCL
kernel behind host work.  The CPU baseline runs at N = 1 only.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
import warnings

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 44100
SEG = 264600  # 6 s
MAC = ["swiglu_conv1d", "swiglu_conv1d"]
VARIANTS = {
    # BASELINE.json's parenthetical = class defaults (models/mss_tflocoformer.py:104-129) + macaron [384, 384]
    "D": dict(n_fft=2048, hop_length=1024, n_sources=4, n_layers=6, emb_dim=128, norm_type="rmsgroupnorm",
              num_groups=4, tf_order="ft", n_heads=4, flash_attention=True, attention_dim=128, pos_enc="rope",
              ffn_type=MAC, ffn_hidden_dim=[384, 384], conv1d_kernel=4, conv1d_shift=1, dropout=0.0, eps=1e-5),
    # configs/musdb18.yaml:22-43 as committed (dropout forced to 0: inference)
    "Y": dict(n_fft=2048, hop_length=512, n_sources=4, n_layers=4, emb_dim=96, norm_type="rmsgroupnorm",
              num_groups=4, tf_order="ft", n_heads=4, flash_attention=True, attention_dim=96, pos_enc="rope",
              ffn_type=MAC, ffn_hidden_dim=[384, 384], conv1d_kernel=4, conv1d_shift=1, dropout=0.0, eps=1e-5),
}
VARIANT_D = VARIANTS["D"]
WORKLOADS = {
    "D": "musdb18 Variant D (n_fft 2048, hop 1024, 6 layers, emb 128, macaron 384) 6-s segments",
    "Y": "musdb18.yaml as committed, Variant Y (n_fft 2048, hop 512, 4 layers, emb 96, macaron 384) 6-s segments",
}
METRIC = "separated audio-sec/sec"
WORKLOAD = WORKLOADS["D"]
# BASELINE config 4: standalone/bslocoformer_separator.py defaults at emb 128, stereo, 4 sources, masking
BS_CFG = dict(num_spk=4, n_layers=6, emb_dim=128, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
              flash_attention=True, attention_dim=128, pos_enc="rope", ffn_type=MAC, ffn_hidden_dim=[384, 384],
              conv1d_kernel=4, conv1d_shift=1, dropout=0.0, eps=1e-5, sample_rate=44100, stft_size=2048,
              masking=True, stereo=True)


def algorithmic_flops(cfg, batch, n_samples):
    """SURVEY.md section 8d."""
    L, C, A, K = cfg["n_layers"], cfg["emb_dim"], cfg["attention_dim"], cfg["conv1d_kernel"]
    hid = cfg["ffn_hidden_dim"]
    hids = hid if isinstance(hid, list) else [hid]
    Tf, F = 1 + n_samples // cfg["hop_length"], cfg["n_fft"] // 2 + 1
    N = batch * Tf * F
    rows = batch * Tf * (F + K - 1) + batch * F * (Tf + K - 1)
    ffn = sum(L * 6 * K * C * h * rows for h in hids)
    sdpa = L * 4 * A * N * (F + Tf)
    proj = L * 2 * 8 * C * A * N
    return dict(ffn=ffn, sdpa=sdpa, proj=proj, total=ffn + sdpa + proj + 36 * C * N * (1 + cfg["n_sources"]))


def ffn_call_flops(cfg, batch, n_samples, axis, hidden):
    C, K = cfg["emb_dim"], cfg["conv1d_kernel"]
    Tf, F = 1 + n_samples // cfg["hop_length"], cfg["n_fft"] // 2 + 1
    rows = batch * Tf * (F + K - 1) if axis == 0 else batch * F * (Tf + K - 1)
    return 6 * K * C * hidden * rows


def workload_config(variant, batch):
    """The `config` object of the forward bench line: a static description of the workload, identical for the b200 arm
    and the --impl reference arm (whose bounded sample of it is stated in `cpu_baseline.sample`); measured figures go
    under `derived`, never here."""
    return {"workload": WORKLOADS[variant], "batch_per_gpu": batch, "segment_samples": SEG,
            "l2": "activations per step (>= 1 GB) exceed the 126 MB L2; no explicit flush"}


def make_mixture(batch, n_samples, seed=1234):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n_samples) / SR
    x = 0.1 * torch.randn(batch, 2, n_samples, generator=g)
    for f0 in (55.0, 220.0, 880.0, 3520.0, 7040.0):
        x = x + 0.05 * torch.sin(2 * math.pi * f0 * t)
    return x.clamp(-1, 1).mean(1)  # stereo -> mono, inference/separate.py:135-139


def make_state_dict(cfg, seed=0):
    """Random-init weights of the named architecture (same init order as the reference constructor)."""
    import mss_tf_locoformer_b200 as pkg
    torch.manual_seed(seed)
    model = pkg.TFLocoformerMSS(**cfg).eval()
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.ndim == 1 and not n.endswith("rope.freqs"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    return model


DUMP_BYTES = 64_000_000      # all files of one dump, .npy headers included
NPY_HEADER = 128             # bytes of a .npy v1 header for the shapes dumped here


def dump_outputs(out, directory, budget=DUMP_BYTES):
    """Write each tensor of `out` (name -> tensor) as directory/<name>.npy in float32.  When the files would exceed
    `budget` bytes together, every tensor is cut to the same fixed, seeded sample of its flattened elements (indices
    in ascending order), so that dumps of two builds at the same arguments still compare element for element."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    total = sum(v.numel() for v in out.values())
    keep = min(1.0, (budget - NPY_HEADER * len(out)) / (4 * total))
    for name, v in out.items():
        a = v.detach().to("cpu", torch.float32)
        if keep < 1.0:
            g = torch.Generator().manual_seed(0)
            idx = torch.randperm(a.numel(), generator=g)[: int(a.numel() * keep)].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(directory, name + ".npy"), a.numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- the reference's own implementation (oracle/_ref = the unmodified files, staged by oracle/build_ref.py) ----
def reference_model(cfg, state_dict, device="cpu"):
    """-> (model, kind).  kind "reference": the unmodified reference TFLocoformerMSS from oracle/_ref;
    kind "port": the oracle restatement (when oracle/_ref has not been staged)."""
    warnings.filterwarnings("ignore", category=FutureWarning)
    from oracle import build_ref
    if build_ref.available():
        cls = build_ref.load()["TFLocoformerMSS"]
        m = cls(**cfg).eval()
        m.load_state_dict(state_dict, strict=True)
        return m.to(device), "reference"
    import oracle

    class Port:
        def __call__(self, mix):
            return oracle.mss_forward(state_dict, cfg, mix)
    return Port(), "port"


def cpu_forward(model, mix, threads):
    torch.set_num_threads(threads)
    t0 = time.perf_counter()
    with torch.no_grad():
        out = model(mix)
    return out, time.perf_counter() - t0


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation (models/mss_tflocoformer.py:184-258, unmodified, from
    oracle/_ref) on all host cores; one step = one mono segment of the same workload (6 s when the run fits ~7 minutes,
    else a shorter cut, stated in `sample`).  Rank 0 only."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    cfg = dict(VARIANTS[args.variant])
    model = make_state_dict(cfg)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    ref, kind = reference_model(cfg, sd)
    est_rate = (0.22 if kind == "reference" else 0.1) * min(2.0, cores / 8.0)   # x real time, BASELINE.md section 2
    audio_s = min(6.0, max(1.0, 420.0 / max(1, args.steps) * est_rate))
    if audio_s >= 4.5:
        audio_s = 6.0
    n = int(round(audio_s * SR))
    mix = make_mixture(1, n)
    warm = make_mixture(1, SR)                 # warm-up steps only page the code in and spin the thread pool up
    for _ in range(args.warmup):
        cpu_forward(ref, warm, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_forward(ref, mix, cores)
    dt = time.perf_counter() - t0
    value = args.steps * n / SR / dt
    sample = (f"{n / SR:.2f}-s mono segment, batch 1, fp32, {args.steps} steps, "
              f"{'unmodified reference TFLocoformerMSS (oracle/_ref)' if kind == 'reference' else 'oracle port'}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.variant, args.batch),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def time_reference_gpu(cfg, sd, dev, batch, steps, mode):
    """The unmodified reference model, eager, on the GPU: `mode` "bf16" = torch.autocast(bfloat16) with
    flash_attention=True (the reference's validation setting, training/train.py:214-215), "fp32" = TF32 off and
    flash_attention=False (SURVEY F10).  -> audio-s/s, ms per step."""
    c = dict(cfg)
    c["flash_attention"] = mode == "bf16"
    ref, kind = reference_model(c, sd, dev)
    if kind != "reference":
        return None
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    mix = make_mixture(batch, SEG).to(dev)
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if mode == "bf16" else torch.autocast("cuda", enabled=False)
    with torch.no_grad(), ctx:
        for _ in range(2):
            ref(mix)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ref(mix)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del ref
    torch.cuda.empty_cache()
    return {"value": batch * SEG / SR / (ms / 1e3), "unit": "audio-s/s", "ms_per_step": ms, "batch": batch, "mode": mode,
            "what": "unmodified reference TFLocoformerMSS, PyTorch eager on this GPU (cuDNN / cuBLAS / SDPA kernels)"}


def run_reference_gpu(args, rank):
    """--impl reference-gpu: the vendor-library bar (SURVEY 8d last row).  Rank 0 only, one GPU."""
    if rank != 0:
        return
    dev = torch.device("cuda", 0)
    cfg = dict(VARIANTS[args.variant])
    model = make_state_dict(cfg)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    bf = time_reference_gpu(cfg, sd, dev, args.batch, args.steps, "bf16")
    if bf is None:
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref not staged (python -m oracle.build_ref)"}))
        return
    fp = time_reference_gpu(cfg, sd, dev, min(args.batch, 2), max(1, args.steps // 4), "fp32")
    print(json.dumps({
        "impl": "reference-gpu", "metric": METRIC, "value": bf["value"], "unit": "audio-s/s", "n_gpus": 1,
        "steps": args.steps, "warmup": 2, "ms_per_step": bf["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.variant], "batch_per_gpu": args.batch}, "bf16_autocast": bf, "fp32_tf32_off": fp}))


def run_bs(args, dev):
    """BASELINE config 4: BSLocoformerSeparator (stereo, 4 sources, masking) on spec [B, 2, 259, 1025] complex64."""
    import mss_tf_locoformer_b200 as pkg
    from mss_tf_locoformer_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(0)
    model = pkg.BSLocoformerSeparator(**BS_CFG).eval().to(dev)
    model.precision = args.precision
    B = args.batch
    mix = make_mixture(2 * B, SEG).reshape(B, 2, SEG)
    win = torch.hann_window(2048)
    spec = torch.stft(mix.reshape(2 * B, SEG), 2048, 1024, window=win, return_complex=True)      # [2B, F, Tf]
    spec = spec.transpose(1, 2).reshape(B, 2, spec.shape[2], spec.shape[1]).contiguous().to(dev)  # [B, 2, Tf, F]
    with torch.no_grad():
        for _ in range(max(3, args.warmup)):
            model(spec)
        torch.cuda.synchronize()
        n0 = lib.tfl_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            est = model(spec)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_outputs({"est": torch.view_as_real(est)}, args.dump_outputs)
    print(json.dumps({
        "metric": METRIC, "value": B * SEG / SR / (ms / 1e3), "unit": "audio-s/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": "BS-Locoformer (62 bands, stereo, 4 sources, masking, 6 layers, emb 128) on 6-s stereo "
                               "spectrograms [B, 2, 259, 1025]", "batch_per_gpu": B, "precision": args.precision},
        "gpu_launches": int(lib.tfl_launch_count() - n0)}))


# BASELINE config 5: configs/musdb18_rtx5090_xlarge.yaml:22-44 (dropout forced to 0: SURVEY 8d), 15-s samples, batch 1 per GPU
TRAIN_CFGS = {
    "xlarge": (dict(n_fft=4096, hop_length=1024, n_sources=4, n_layers=12, emb_dim=256, norm_type="rmsgroupnorm",
                    num_groups=8, tf_order="ft", n_heads=16, flash_attention=True, attention_dim=256, pos_enc="rope",
                    ffn_type=MAC, ffn_hidden_dim=[1024, 1024], conv1d_kernel=4, conv1d_shift=1, dropout=0.0, eps=1e-5),
               661500, "musdb18_rtx5090_xlarge.yaml training step (12 layers, emb 256, n_fft 4096, 15-s samples)"),
    "D": (VARIANT_D, SEG, "musdb18 Variant D training step (6 layers, emb 128, n_fft 2048, 6-s samples)"),
}


def time_reference_gpu_train(cfg, sd, dev, mix, tgt, steps, loss_w):
    """The unmodified reference model + MSSLoss + clip + torch AdamW, eager on this GPU under bf16 autocast
    (training/train.py:115-146 with amp_dtype bfloat16).  -> dict or a reason string."""
    from oracle import build_ref
    if not build_ref.available():
        return "oracle/_ref not staged"
    try:
        ref, _ = reference_model(dict(cfg, flash_attention=True), sd, dev)
        from models.mss_loss import MSSLoss
        ref.train()
        crit = MSSLoss(loss_type="combined", si_sdr_weight=loss_w[0], l1_weight=loss_w[1], spectral_weight=loss_w[2])
        opt = torch.optim.AdamW([p for p in ref.parameters() if p.requires_grad], lr=3e-4, weight_decay=0.01, eps=1e-8)
        names = ["vocals", "drums", "bass", "other"]
        targets = {n: tgt[i] for i, n in enumerate(names)}

        def one():
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss = crit(ref(mix), targets)["total_loss"]
            loss.backward()
            torch.nn.utils.clip_grad_norm_(ref.parameters(), max_norm=5.0)
            opt.step()
            return loss
        for _ in range(3):                      # cuDNN / cuBLAS algorithm selection and the allocator settle in the first steps
            one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        peak = torch.cuda.max_memory_allocated() / 2 ** 30
        del ref, opt
        torch.cuda.empty_cache()
        return {"ms_per_step": ms, "value": mix.shape[0] * mix.shape[1] / SR / (ms / 1e3), "unit": "audio-s/s",
                "peak_gib": round(peak, 1), "mode": "bf16 autocast, flash attention, eager autograd, torch AdamW",
                "what": "unmodified reference TFLocoformerMSS + MSSLoss training step, PyTorch eager on this GPU"}
    except RuntimeError as e:   # out of memory at this size is a finding, not a failure of the bench
        torch.cuda.empty_cache()
        return "failed: " + str(e).splitlines()[0][:160]


def train_dtype(cfg):
    """Operand type of the training step's GEMMs in the default TFL_OPT_TRAIN_MODE 2 (accumulation is fp32 everywhere):
    bf16 where the tcgen05 attention path takes the shape (csrc/kernels_attn.cuh attn_tc_supported), else tf32."""
    hd = cfg["attention_dim"] // cfg["n_heads"]
    npart = cfg["n_heads"] * ((hd + 15) // 16 * 16)
    ok = hd % 2 == 0 and hd <= 32 and npart % 32 == 0 and npart <= 128 and cfg["emb_dim"] % 16 == 0
    return "bf16" if ok else "tf32"


def run_train(args, dev, rank, world):
    """BASELINE config 5: one data-parallel training step per `step` (forward, MSSLoss, backward, NCCL gradient average,
    clip, AdamW) through mss_tf_locoformer_b200.training.Trainer; every rank trains on its own sample(s)."""
    import torch.distributed as dist
    import mss_tf_locoformer_b200 as pkg
    from mss_tf_locoformer_b200 import _lib
    from mss_tf_locoformer_b200.training import Trainer
    cfg, n_samples, what = TRAIN_CFGS[args.train]
    if args.train_seconds > 0:
        n_samples = int(args.train_seconds * SR)
    B = args.train_batch
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    torch.manual_seed(0)
    model = pkg.TFLocoformerMSS(**cfg).to(dev)
    loss_w = (1.0, 0.1, 0.15)                       # musdb18_rtx5090_xlarge.yaml:47-52
    tr = Trainer(model, lr=3e-4, weight_decay=0.01, si_sdr_weight=loss_w[0], l1_weight=loss_w[1], spectral_weight=loss_w[2])
    mix_host = make_mixture(B, n_samples, seed=1234 + rank).pin_memory()
    g = torch.Generator().manual_seed(77 + rank)
    tgt_host = (0.25 * mix_host[None] + 0.05 * torch.randn(4, B, n_samples, generator=g)).pin_memory()
    mix, tgt = mix_host.to(dev), tgt_host.to(dev)
    losses = []
    for _ in range(args.warmup):
        losses.append(tr.step(mix, tgt)[0:1].clone())
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = lib.tfl_launch_count()
    sampler = ClockSampler(dev.index or 0)
    with sampler:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            losses.append(tr.step(mix, tgt)[0:1].clone())
        e1.record()
        torch.cuda.synchronize()
    launches = int(lib.tfl_launch_count() - n0)
    ms = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
    # e2e: the step from pinned host memory, loss read back
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(max(1, args.steps // 2)):
        loss = tr.step(mix_host.to(dev, non_blocking=True), tgt_host.to(dev, non_blocking=True))
        loss_host = loss.cpu()
    e3.record()
    torch.cuda.synchronize()
    ms_e2e = torch.tensor([e2.elapsed_time(e3) / max(1, args.steps // 2)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(ms_e2e, op=dist.ReduceOp.MAX)
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    if rank != 0:
        return
    ms, ms_e2e = float(ms), float(ms_e2e)
    secs = B * n_samples / SR
    fl = algorithmic_flops(cfg, B, n_samples)
    ref = None
    if args.reference_gpu:
        sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
        ref = time_reference_gpu_train(cfg, sd, dev, mix, tgt, max(3, args.steps), loss_w)
    ls = [float(x) for x in torch.cat(losses).cpu()]
    print(json.dumps({
        "metric": "trained audio-sec/sec (forward + loss + backward + gradient all-reduce + clip + AdamW)",
        "value": world * secs / (ms / 1e3), "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": train_dtype(cfg), "data": "synthetic",
        "config": {"workload": what, "batch_per_gpu": B, "seconds_per_sample": n_samples / SR, "parallelism": f"dp{world}",
                   "loss": "MSSLoss combined (si_sdr 1.0, l1 0.1, spectral 0.15)", "optimizer": "AdamW lr 3e-4 wd 0.01, clip 5.0",
                   "params": int(sum(p.numel() for p in model.parameters() if p.requires_grad)),
                   "grad_allreduce_bytes": int(tr.total * 4) if world > 1 else 0},
        "e2e": {"value": world * secs / (ms_e2e / 1e3), "unit": "audio-s/s",
                "h2d_bytes_per_step": int(mix_host.numel() * 4 + tgt_host.numel() * 4), "d2h_bytes_per_step": int(loss_host.numel() * 4)},
        "algorithmic_tflops_per_step": 3 * fl["total"] / 1e12,
        "achieved_tflops": 3 * fl["total"] / 1e12 / (ms / 1e3),
        "loss_first_last": [ls[0], ls[-1]], "gpu_launches": launches, "clocks": sampler.summary(),
        "workspace_gib": round(tr._ws.numel() / 2 ** 30, 1), "reference_gpu_train": ref}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--variant", default="D", choices=sorted(VARIANTS))
    ap.add_argument("--model", default="mss", choices=["mss", "bs"])
    ap.add_argument("--batch", type=int, default=8, help="6-s segments per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--reference-gpu", action="store_true",
                    help="also time the unmodified reference model eager on this GPU and add `reference_gpu` to the line")
    ap.add_argument("--track", type=float, default=0.0,
                    help="BASELINE config 3: separate ONE synthetic track of this many seconds, 6-s segments at 50 %% overlap "
                         "sharded over the ranks (strong scaling); prints its own JSON line")
    ap.add_argument("--train", default=None, choices=sorted(TRAIN_CFGS),
                    help="BASELINE config 5: time data-parallel TRAINING steps of this configuration instead of inference")
    ap.add_argument("--train-seconds", type=float, default=0.0, help="seconds of audio per training sample (0 = the configuration's own)")
    ap.add_argument("--train-batch", type=int, default=1, help="training samples per GPU per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed separation step returned (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.train):
        ap.error("--dump-outputs applies to the separation benchmarks of --impl b200 (not --train)")
    args.warmup = max(args.warmup, 3) if (args.impl == "b200" and args.train is None) else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.impl == "reference-gpu":
        run_reference_gpu(args, rank)
        return

    import torch.distributed as dist
    import mss_tf_locoformer_b200 as pkg
    from mss_tf_locoformer_b200 import _lib

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.model == "bs":
        if rank == 0:
            run_bs(args, dev)
        return
    if args.train is not None:
        run_train(args, dev, rank, world)
        return
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    cfg = dict(VARIANTS[args.variant])
    model = make_state_dict(cfg).to(dev)
    model.precision = args.precision
    B = args.batch
    mix_host = make_mixture(B, SEG, seed=1234 + rank).pin_memory()
    mix_dev = mix_host.to(dev)
    names = ["vocals", "drums", "bass", "other"]
    out_host = torch.empty((4, B, SEG), dtype=torch.float32).pin_memory()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def finish_group():
        """Last collective of the run: nothing rank-local may follow while a peer still waits on NCCL."""
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            dist.destroy_process_group()

    def timed(fn, steps):
        """-> (ms over `steps` calls of fn, what the last call returned)."""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    def step_resident():
        with torch.no_grad():
            return model(mix_dev)

    # End to end through the public API, as a caller separating a stream of batches runs it: every step copies its
    # mixtures from pinned host memory, calls forward() and reads the four sources back to pinned host memory; the
    # read-back of step i runs on a second stream under the compute of step i + 1 (two output buffers), and the caller
    # takes delivery of step i - 1 (waits for its copy) before it submits step i + 1.
    copy_stream = torch.cuda.Stream(device=dev)
    out_hosts = [out_host, torch.empty_like(out_host).pin_memory()]
    pending = []                                  # (event of the finished read-back, tensors kept alive until then)
    e2e_count = [0]

    def step_e2e():
        i = e2e_count[0]
        e2e_count[0] += 1
        with torch.no_grad():
            x = mix_host.to(dev, non_blocking=True)
            out = model(x)
            stacked = torch.stack([out[k] for k in names])
        done = torch.cuda.Event()
        done.record()
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done)
            out_hosts[i & 1].copy_(stacked, non_blocking=True)
            copied = torch.cuda.Event()
            copied.record()
        pending.append((copied, stacked, x))
        while len(pending) > 1:                   # delivery of the previous step's result
            pending.pop(0)[0].synchronize()

    def drain_e2e():
        while pending:
            pending.pop(0)[0].synchronize()

    if args.track > 0:
        from mss_tf_locoformer_b200.segments import separate_track, segment_starts
        n_track = int(args.track * SR)
        track = make_mixture(1, n_track, seed=99)[0].to(dev)

        def step_track():
            with torch.no_grad():
                return separate_track(model, track, seg_len=SEG, batch=B)

        for _ in range(max(1, args.warmup // 3)):
            step_track()
        ms, out = timed(step_track, args.steps)
        finish_group()
        if rank == 0 and args.dump_outputs:
            dump_outputs(out, args.dump_outputs)
        if rank == 0:
            print(json.dumps({
                "metric": METRIC, "value": args.track * args.steps / (ms / 1e3), "unit": "audio-s/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
                "data": "synthetic",
                "config": {"workload": f"full-track {args.track:.0f}-s mono, {len(segment_starts(n_track, SEG))} segments of 6 s at "
                                       f"50 % overlap, sharded over {world} rank(s), halo exchange + all-gather stitch",
                           "batch_per_gpu": B, "precision": args.precision}}))
        return

    for _ in range(args.warmup):
        step_resident()
    n0 = lib.tfl_launch_count()
    with ClockSampler(local) as clocks:
        ms, last = timed(step_resident, args.steps)
    launches = lib.tfl_launch_count() - n0
    # host copy before the end-to-end steps run the model again; nothing of it is timed
    last = {k: v.cpu() for k, v in last.items()} if args.dump_outputs else None
    for _ in range(2):
        step_e2e()
    drain_e2e()

    def e2e_steps():
        step_e2e()

    sync_all()
    t_e0, t_e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_e0.record()
    for _ in range(args.steps):
        e2e_steps()
    drain_e2e()                                    # the last read-back is inside the timed region
    t_e1.record()
    sync_all()
    ms_e2e_t = torch.tensor([t_e0.elapsed_time(t_e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_e2e_t, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_e2e_t.item())
    finish_group()          # ---- no collective below this line ----
    if rank != 0:
        return
    if last is not None:
        dump_outputs(last, args.dump_outputs)

    audio_s = world * B * SEG / SR
    value = audio_s * args.steps / (ms / 1e3)
    e2e_value = audio_s * args.steps / (ms_e2e / 1e3)
    line = {
        "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": workload_config(args.variant, B),
        "derived": {"x_realtime_per_gpu": value / world},
        "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": world * mix_host.numel() * 4,
                "d2h_bytes_per_step": world * out_host.numel() * 4},
        "gpu_launches": int(launches) * world,
        "clocks": clocks.summary(),
    }
    fl = algorithmic_flops(cfg, B, SEG)
    line["derived"]["tflops_total_algorithmic"] = fl["total"] * world * args.steps / (ms / 1e3) / 1e12
    # ---- roofline of the dominant kernel: the ConvSwiGLU FFN (83 % of FLOPs), frequency axis ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    # the kernel below is timed alone (10 back-to-back launches): the burst cuBLAS figure is its denominator; the
    # whole-step fraction uses the sustained one (B200_PROFILING.md)
    peak = peaks.get("bf16_tflops", peaks.get("bf16_tflops_sustained", 1400.0))
    peak_sustained = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops (burst; kernel timed alone)" if peaks else "fallback 1.4 PF"
    line["derived"]["step_frac_of_sustained_bf16_peak"] = line["derived"]["tflops_total_algorithmic"] / peak_sustained
    eng = model._ready()
    prec = 1 if args.precision == "bf16" else 0
    Tf, F = 1 + SEG // cfg["hop_length"], cfg["n_fft"] // 2 + 1
    hid_last = cfg["ffn_hidden_dim"][-1]
    x = torch.randn(B, Tf, F, cfg["emb_dim"], device=dev)
    y = torch.empty_like(x)
    for _ in range(3):
        eng.ffn_out(0, 0, 0, x, y, prec)
    reps = 10
    l0 = lib.tfl_launch_count()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.ffn_out(0, 0, 0, x, y, prec)
    e1.record()
    torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1) / reps
    k_launches = (lib.tfl_launch_count() - l0) // reps
    k_flops = ffn_call_flops(cfg, B, SEG, 0, hid_last)
    achieved = k_flops / (k_ms / 1e3) / 1e12
    traffic = None   # DRAM bytes per launch from the committed ncu --set full capture of this very launch shape
    for cap_name in ("r02_ffn2_ncu_b8.json", "r01_ffn2_ncu_b8.json"):
        try:
            cap = json.load(open(os.path.join(ROOT, "profiles", cap_name)))
            if B == 8 and args.precision == "bf16" and args.variant == "D":
                traffic = cap["traffic_bytes_per_launch"]
            break
        except (OSError, KeyError, ValueError):
            continue
    line["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                        "frac": achieved / peak, "frac_of_sustained": achieved / peak_sustained, "traffic": traffic,
                        "kernel": "conv_swiglu_ffn (freq axis), out-of-place kernel launch alone",
                        "launches_per_call": int(k_launches), "ms_per_call": k_ms, "peak_source": peak_src,
                        "flops_per_call": k_flops}
    del x, y
    if world == 1 and args.reference_gpu:
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        line["reference_gpu"] = {"bf16_autocast": time_reference_gpu(cfg, sd, dev, B, 3, "bf16"),
                                 "fp32_tf32_off": time_reference_gpu(cfg, sd, dev, min(B, 2), 2, "fp32")}
    if world == 1 and not args.no_cpu_baseline:
        # ---- CPU baseline: the unmodified reference forward on the host cores, ONE 6-s segment (~20-30 s of CPU);
        # the same forward doubles as a full-size parity check of the GPU path ----
        cores = os.cpu_count() or 1
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        ref, kind = reference_model(cfg, sd)
        n = SEG if kind == "reference" else SEG // 4
        mix = make_mixture(1, n)
        cpu_forward(ref, make_mixture(1, SR // 2), cores)      # spin the thread pool up
        want, dt = cpu_forward(ref, mix, cores)
        with torch.no_grad():
            got = model(mix.to(dev))
        import oracle
        worst = min(oracle.si_sdr_db(got[k].cpu(), want[k]) for k in want)
        err = max(float((got[k].cpu() - want[k]).abs().max()) for k in want)
        line["cpu_baseline"] = {"value": n / SR / dt, "unit": "audio-s/s", "cores": cores, "kind": kind,
                                "sample": f"one {n / SR:.2f}-s mono segment, batch 1, fp32, {dt:.1f} s"}
        line["parity"] = {"vs": f"cpu {kind}, same weights and input, {n / SR:.2f}-s segment",
                          "worst_si_sdr_db": worst, "max_abs": err}
    elif world > 1:
        line["cpu_baseline"] = None   # N = 1 only (see the module docstring)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
