"""Cost of stereo separation and of a higher segment overlap, with the card's name and power limit.

- ``track``: segments.separate_track on a 240-s track at 44.1 kHz, TFLocoformerMSS Variant D in bf16, 6-s segments,
  8 segments per forward, one GPU: mono at 0.5 overlap (the default path, tfl_segment_ola), stereo at 0.5 and stereo
  at 0.75 (tfl_segment_ola_hop).  Seconds per track (host clock around work that ends in a device synchronise; modes
  alternate, median of --steps after --warmup runs of every mode), forwards and rows per forward.
- ``kernel``: one tfl_segment_ola_hop call at the shapes of those runs (4 sources, 8 segments, C channels), CUDA
  events over --reps calls, against its HBM floor computed from shapes: the segment outputs read once
  (4 * S * 8C * L bytes) and the touched span of the track read and written once (8 * S * C * ((8 - 1) * hop + L)),
  over 7.7 TB/s (HGX B200 data sheet, one GPU).  The segment buffers rotate over more than the 126 MB of L2.  The
  mono 0.5 row also times tfl_segment_ola at the same shape.  ``stitch_share`` = kernel time x calls / track time.

    python profiles/time_stereo_overlap.py [--steps 3] [--warmup 1] [--out profiles/stereo_overlap_b200.json]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import mss_tf_locoformer_b200 as pkg  # noqa: E402
from mss_tf_locoformer_b200.segments import SEGMENT_SAMPLES, overlap_hop, segment_starts, separate_track  # noqa: E402

SR = 44100
T = 240 * SR
BATCH = 8
HBM_BYTES_PER_S = 7.7e12
RUNS = {"mono_0.5": (1, 0.5), "stereo_0.5": (2, 0.5), "stereo_0.75": (2, 0.75)}


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = line.partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def _separate(model, track, overlap):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.no_grad():
        out = separate_track(model, track, seg_len=SEGMENT_SAMPLES, batch=BATCH, overlap=overlap)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def _kernel(channels, overlap, reps, S=4):
    L, hop = SEGMENT_SAMPLES, overlap_hop(SEGMENT_SAMPLES, overlap)
    n_seg = len(segment_starts(T, L, hop))
    span = (BATCH - 1) * hop + L
    seg_bytes = 4 * S * BATCH * channels * L
    n_buf = max(2, math.ceil(2 * 126e6 / seg_bytes))
    segs = [torch.randn(S, BATCH * channels, L, device="cuda") for _ in range(n_buf)]
    track = torch.zeros(S, channels, span, device="cuda")
    floor_us = (seg_bytes + 8 * S * channels * span) / HBM_BYTES_PER_S * 1e6

    def timed(fn):
        for i in range(3):
            fn(segs[i % n_buf])
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(segs[i % n_buf])
        b.record()
        b.synchronize()
        return a.elapsed_time(b) * 1e3 / reps

    us = timed(lambda s: pkg.segment_ola_hop(s, channels, hop, 0, n_seg, track))
    res = {"shape": {"sources": S, "segments": BATCH, "channels": channels, "seg_len": L, "hop": hop, "span": span},
           "segment_ola_hop_us": round(us, 2), "hbm_floor_us": round(floor_us, 2),
           "floor_over_time": round(floor_us / us, 3), "calls_per_track": math.ceil(n_seg / BATCH)}
    if channels == 1 and 2 * hop == L:
        mono = torch.zeros(S, span, device="cuda")
        res["segment_ola_us"] = round(timed(lambda s: pkg.segment_ola(s, 0, n_seg, mono)), 2)
    del segs
    torch.cuda.empty_cache()
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--reps", type=int, default=50)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "stereo_overlap_b200.json"))
    args = p.parse_args()
    gpu = _gpu()
    model = bench.make_state_dict(dict(bench.VARIANT_D)).cuda()
    model.precision = "bf16"
    mix = bench.make_mixture(2, T).cuda()                                  # two different channels
    tracks = {name: (mix[0] if c == 1 else mix) for name, (c, _) in RUNS.items()}
    outs = {}
    for _ in range(args.warmup):
        for name, (_, overlap) in RUNS.items():
            _, outs[name] = _separate(model, tracks[name], overlap)
    times = {name: [] for name in RUNS}
    for _ in range(args.steps):
        for name, (_, overlap) in RUNS.items():
            s, _ = _separate(model, tracks[name], overlap)
            times[name].append(s)
    kernels = {name: _kernel(c, overlap, args.reps) for name, (c, overlap) in RUNS.items()}
    result = {"gpu": gpu, "workload": {"model": "TFLocoformerMSS Variant D", "precision": "bf16", "track_s": T / SR,
                                       "seg_len": SEGMENT_SAMPLES, "segments_per_forward": BATCH},
              "track": {}, "kernel": kernels}
    for name, (c, overlap) in RUNS.items():
        hop = overlap_hop(SEGMENT_SAMPLES, overlap)
        n_seg = len(segment_starts(T, SEGMENT_SAMPLES, hop))
        med = statistics.median(times[name])
        k = kernels[name]
        result["track"][name] = {
            "channels": c, "overlap": overlap, "hop": hop, "segments": n_seg, "forwards": math.ceil(n_seg / BATCH),
            "rows_per_forward": BATCH * c, "seconds": round(med, 3), "all_seconds": [round(s, 3) for s in times[name]],
            "track_s_per_s": round(T / SR / med, 1),
            "stitch_share": round(k["segment_ola_hop_us"] * 1e-6 * k["calls_per_track"] / med, 5)}
    # the stereo 0.5 run's left channel against the mono run of that channel (tfl_segment_ola_hop vs tfl_segment_ola)
    result["stereo_0.5_left_vs_mono_max_abs"] = max(
        float((outs["stereo_0.5"][k][0] - outs["mono_0.5"][k]).abs().max()) for k in outs["mono_0.5"])
    print(json.dumps(result, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
