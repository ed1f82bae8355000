"""Host logic of the full-track separation at any overlap and over channels, without a GPU: the general stitch against
oracle.stitch_segments, segments.separate_track (with a CPU stand-in of tfl_segment_ola_hop) on gloo worlds 1-5, the
ownership of the track, the CLI's --overlap / --stereo arguments and the instructions of segment_ola_hop_kernel."""
import os
import re
import shutil
import socket
import subprocess

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
import stitch_hop_ref as ref
from mss_tf_locoformer_b200 import _lib, segments, separate

OVERLAPS = (0.25, 0.5, 0.75, 0.875)


@pytest.mark.parametrize("n,seg", [(40, 64), (1000, 64), (997, 128), (1700, 512), (5, 2)])
def test_general_stitch_at_half_overlap_is_the_oracle(n, seg):
    starts = oracle.segment_starts(n, seg)
    assert ref.segment_starts(n, seg, seg // 2) == starts
    x = torch.randn(len(starts), 3, seg, dtype=torch.float64, generator=torch.Generator().manual_seed(n))
    want = oracle.stitch_segments(x, n)
    got = ref.stitch_segments(x, n, seg // 2)
    assert float((got - want).abs().max()) <= 1e-12


def test_general_stitch_reproduces_a_constant():
    """With f_i = 1 every sample is sum w / E = 1: the normalisation covers every hop, odd ones included."""
    for seg in (7, 8, 64):
        for hop in range(1, seg):
            n = 3 * seg + 5
            k = len(ref.segment_starts(n, seg, hop))
            y = ref.stitch_segments(torch.ones(k, 1, seg, dtype=torch.float64), n, hop)
            assert float((y - 1).abs().max()) <= 1e-12, (seg, hop)


def _cpu_ola(seg_out, i0, n_seg, acc, origin=0):
    """CPU stand-in for tfl_segment_ola (the 50 % path of a 1-D track)."""
    s, b, length = seg_out.shape
    for k in range(b):
        gi = i0 + k
        w = oracle.segment_window(length, gi == 0, gi == n_seg - 1, seg_out.dtype)
        start = gi * (length // 2) - origin
        acc[:, start:start + length] += seg_out[:, k] * w


def _cpu_ola_hop(seg_out, channels, hop, i0, n_seg, acc, origin=0):
    """CPU stand-in for tfl_segment_ola_hop: this call's segments, windowed and divided by the window sum E of every
    segment of the grid covering a sample of the local buffer acc[S, C, n]."""
    _, rows, length = seg_out.shape
    n = acc.shape[-1]
    e = torch.zeros(n, dtype=torch.float64)
    for i in range(n_seg):
        a, b = max(i * hop - origin, 0), min(i * hop + length - origin, n)
        if b > a:
            w = oracle.segment_window(length, i == 0, i == n_seg - 1, torch.float64)
            e[a:b] += w[a - (i * hop - origin):b - (i * hop - origin)]
    for k in range(rows // channels):
        gi = i0 + k
        w = oracle.segment_window(length, gi == 0, gi == n_seg - 1, torch.float64)
        start = gi * hop - origin
        a, b = max(start, 0), min(start + length, n)
        for c in range(channels):
            part = seg_out[:, k * channels + c].double() * w
            acc[:, c, a:b] += (part[:, a - start:b - start] / e[a:b]).to(acc.dtype)


def _fake_model(x):
    """Rows independent, output depends on the position inside the segment (so a misplaced window shows)."""
    ramp = torch.arange(x.shape[-1], dtype=x.dtype) / x.shape[-1]
    return {"a": x * 2.0 + 1.0, "b": -x * x + ramp}


# (n_samples, seg_len): 1 segment, a few, many, an odd segment length, and 4 segments of 64 at 0.75 overlap
# (n = 112), where rank 0's buffer past its own range reaches ranks 1, 2 and 3 on 4 ranks.
CASES = [(40, 64), (112, 64), (300, 64), (1000, 64), (997, 63)]


def _tracks(n):
    g = torch.Generator().manual_seed(n)
    stereo = torch.randn(2, n, generator=g)
    return {"mono1d": stereo[0], "mono": stereo[:1], "stereo": stereo}


def _check_case(n, seg, overlap, kind, track):
    hop = segments.overlap_hop(seg, overlap)
    out = segments.separate_track(_fake_model, track, seg_len=seg, batch=3, ola=_cpu_ola, overlap=overlap,
                                  ola_hop=_cpu_ola_hop)
    want = ref.separate_track(_fake_model, track.double(), seg, hop, batch=2)
    return list(out) == list(want) and all(
        out[k].shape == want[k].shape and float((out[k].double() - want[k]).abs().max()) <= 1e-5 for k in want)


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        failed = []
        for n, seg in CASES:
            for overlap in OVERLAPS:
                for kind, track in _tracks(n).items():
                    if not _check_case(n, seg, overlap, kind, track):
                        failed.append((n, seg, overlap, kind))
        ret[rank] = failed
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_single_process_matches_reference():
    for n, seg in CASES:
        for overlap in OVERLAPS:
            for kind, track in _tracks(n).items():
                assert _check_case(n, seg, overlap, kind, track), (n, seg, overlap, kind)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5])
def test_multi_rank_gloo_matches_reference(world):
    assert len(segments.segment_starts(112, 64, segments.overlap_hop(64, 0.75))) == 4
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
        assert dict(ret) == {r: [] for r in range(world)}


def test_owned_ranges_tile_the_track_for_every_hop():
    seg = 64
    for hop in range(1, seg):
        for n_seg in (1, 2, 3, 4, 7, 79):
            for world in range(1, 9):
                own = segments.owned_ranges(n_seg, seg, world, hop)
                spans = [(a, b) for a, b in own if b > a]
                assert spans[0][0] == 0 and spans[-1][1] == (n_seg - 1) * hop + seg
                assert all(spans[i][1] == spans[i + 1][0] for i in range(len(spans) - 1))
    assert segments.owned_ranges(79, 264_600, 8) == segments.owned_ranges(79, 264_600, 8, 132_300)


def test_overlap_hop():
    assert segments.overlap_hop(264_600, 0.5) == 132_300
    assert segments.overlap_hop(264_600, 0.75) == 66_150
    assert segments.overlap_hop(64, 0.875) == 8
    assert segments.overlap_hop(64, 0.999) == 1                   # at least one sample
    assert segments.overlap_hop(2, 0.01) == 1                     # below the segment length
    for bad in (0.0, 1.0, -0.5, 1.5):
        with pytest.raises(ValueError):
            segments.overlap_hop(64, bad)


def test_separate_track_rejects_bad_input():
    with pytest.raises(ValueError):
        segments.separate_track(_fake_model, torch.zeros(1, 2, 100), seg_len=64, ola_hop=_cpu_ola_hop)
    with pytest.raises(ValueError):
        segments.separate_track(_fake_model, torch.zeros(2, 100), seg_len=64, overlap=1.0, ola_hop=_cpu_ola_hop)


def test_cli_overlap_and_stereo_arguments():
    base = ["--input", "a.wav", "--checkpoint", "m.pt"]
    a = separate.parse_args(base)
    assert (a.overlap, a.stereo) == (0.5, False)
    a = separate.parse_args(base + ["--overlap", "0.75", "--stereo"])
    assert (a.overlap, a.stereo) == (0.75, True)
    for bad in ("0", "1", "-0.25", "1.5", "0.0", "1.0"):
        with pytest.raises(SystemExit):
            separate.parse_args(base + ["--overlap", bad])


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump (CUDA toolkit) not on PATH")
def test_segment_ola_hop_kernel_has_no_atomics():
    _lib.load()
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s*Function : (\S+)\n", sass)
    bodies = {name: body for name, body in zip(parts[1::2], parts[2::2]) if "segment_ola_hop_kernel" in name}
    assert len(bodies) == 1, list(bodies)
    for name, body in bodies.items():
        assert re.search(r"\bSTG\b|\bSTG\.", body), name
        assert not re.search(r"\b(ATOM|ATOMG|ATOMS|RED|REDG)\b|\b(ATOM|ATOMG|ATOMS|RED|REDG)\.", body), name
