"""Full-track separation at any overlap and over channels on the GPU: tfl_segment_ola_hop against the float64 stitch of
tests/stitch_hop_ref.py, its repeatability and its agreement with tfl_segment_ola at 50 %, TFLocoformerMSS on a
stereo track against the oracle model + stitch, channel / mono bit-equality, NCCL on two GPUs and the CLI's --stereo /
--overlap.  Gates as tests/test_gpu_parity.py: fp32 SI-SDR >= 70 dB, bf16 >= 40 dB."""
import math
import os
import socket

import pytest
import torch

import oracle
import stitch_hop_ref as ref
from conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return m


def _mixture(n, batch, seed=1234):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n) / 44100.0
    x = 0.1 * torch.randn(batch, n, generator=g)
    for f0 in (55.0, 220.0, 880.0, 3520.0, 7040.0):
        x = x + 0.05 * torch.sin(2 * math.pi * f0 * t)[None]
    return x.clamp(-1, 1)


def _model(pkg, precision):
    cfg, sd, arr = load_golden("mss_hop2_macaron")
    model = pkg.TFLocoformerMSS(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    model.precision = precision
    return cfg, sd, model


def _stitch(pkg, seg, hop, batch, channels, lo=0, hi=None, origin=0, n_track=None):
    """seg [n_seg, C, S, L] -> track [S, C, n_track] through tfl_segment_ola_hop, segments lo..hi in calls of `batch`."""
    n_seg, C, S, L = seg.shape
    hi = n_seg if hi is None else hi
    n_track = (n_seg - 1) * hop + L - origin if n_track is None else n_track
    track = torch.zeros(S, C, n_track, device="cuda")
    for i0 in range(lo, hi, batch):
        chunk = seg[i0:min(i0 + batch, hi)]                               # [b, C, S, L] -> [S, b * C, L]
        pkg.segment_ola_hop(chunk.permute(2, 0, 1, 3).reshape(S, -1, L).cuda(), channels, hop, i0, n_seg, track, origin)
    return track


def _want(seg, hop, lo, hi, origin, n_track):
    """float64: sum over segments lo..hi-1 of w_i f_i / E on samples [origin, origin + n_track), E over all segments."""
    n_seg, C, S, L = seg.shape
    total = (n_seg - 1) * hop + L
    y = torch.zeros(S, C, total, dtype=torch.float64)
    e = torch.zeros(total, dtype=torch.float64)
    for i in range(n_seg):
        w = oracle.segment_window(L, i == 0, i == n_seg - 1, torch.float64)
        e[i * hop:i * hop + L] += w
        if lo <= i < hi:
            y[:, :, i * hop:i * hop + L] += seg[i].permute(1, 0, 2).double() * w
    return (y / e)[:, :, origin:origin + n_track]


def _rel(got, want):
    return float((got.double().cpu() - want).abs().max()) / float(want.abs().max())


# (seg_len, hop, n_samples, batch, channels, n_src): odd hops, seg_len not a multiple of the hop, overlaps from 0.2 to
# 0.99, one segment, several batches, stereo rows
KERNEL_CASES = [(512, 77, 3000, 3, 1, 4), (500, 128, 2100, 2, 2, 3), (512, 384, 4000, 4, 2, 4), (1024, 1023, 9000, 3, 1, 2),
                (257, 3, 700, 8, 2, 2), (2048, 512, 2048, 1, 2, 4), (4096, 1111, 40000, 5, 2, 4), (64, 1, 200, 16, 3, 1)]


@pytest.mark.parametrize("L,hop,n,batch,C,S", KERNEL_CASES)
def test_kernel_matches_float64_stitch(pkg, L, hop, n, batch, C, S):
    n_seg = len(ref.segment_starts(n, L, hop))
    seg = torch.randn(n_seg, C, S, L, generator=torch.Generator().manual_seed(L + hop))
    got = _stitch(pkg, seg, hop, batch, C)
    total = (n_seg - 1) * hop + L
    assert _rel(got, _want(seg, hop, 0, n_seg, 0, total)) <= 1e-6
    for c in range(C):                                                    # the definition's own stitch, channel c
        want = ref.stitch_segments(seg[:, c].double(), n, hop)
        assert _rel(got[:, c, :n], want) <= 1e-6, c


@pytest.mark.parametrize("L,hop,n,batch,C,S", KERNEL_CASES[:4])
def test_kernel_local_buffer_with_origin(pkg, L, hop, n, batch, C, S):
    """A rank's buffer: segments [lo, hi), samples lo * hop .. (hi - 1) * hop + L, E still over the whole grid."""
    n_seg = len(ref.segment_starts(n, L, hop))
    seg = torch.randn(n_seg, C, S, L, generator=torch.Generator().manual_seed(7))
    lo, hi = n_seg // 3, max(n_seg // 3 + 1, 2 * n_seg // 3)
    origin = lo * hop
    n_track = (hi - 1) * hop + L - origin
    got = _stitch(pkg, seg, hop, batch, C, lo, hi, origin, n_track)
    assert _rel(got, _want(seg, hop, lo, hi, origin, n_track)) <= 1e-6
    # a buffer shorter than the call's span: the kernel clips to it
    got = _stitch(pkg, seg, hop, batch, C, lo, hi, origin, n_track // 2)
    assert _rel(got, _want(seg, hop, lo, hi, origin, n_track // 2)) <= 1e-6


def test_kernel_bitwise_repeatable(pkg):
    L, hop, n, C, S = 4096, 1024 + 7, 60000, 2, 4
    n_seg = len(ref.segment_starts(n, L, hop))
    seg = torch.randn(n_seg, C, S, L, generator=torch.Generator().manual_seed(1))
    a = _stitch(pkg, seg, hop, 5, C)
    b = _stitch(pkg, seg, hop, 5, C)
    assert torch.equal(a, b)


def test_kernel_at_half_overlap_agrees_with_segment_ola(pkg):
    L, n, S = 512, 1700, 3
    n_seg = len(oracle.segment_starts(n, L))
    seg = torch.randn(n_seg, 1, S, L, generator=torch.Generator().manual_seed(5))
    got = _stitch(pkg, seg, L // 2, 2, 1)[:, 0, :n]
    old = torch.zeros(S, n, device="cuda")
    for i0 in range(0, n_seg, 2):
        pkg.segment_ola(seg[i0:i0 + 2, 0].permute(1, 0, 2).contiguous().cuda(), i0, n_seg, old)
    assert _rel(got, old.double().cpu()) <= 1e-6


def test_kernel_rejects_bad_arguments(pkg):
    seg = torch.zeros(2, 4, 64, device="cuda")
    track = torch.zeros(2, 2, 200, device="cuda")
    for hop in (0, 64, 100):
        with pytest.raises(RuntimeError):
            pkg.segment_ola_hop(seg, 2, hop, 0, 5, track)
    with pytest.raises(RuntimeError):
        pkg.segment_ola_hop(seg, 2, 16, 4, 5, track)                      # segments 4, 5 of 5
    with pytest.raises(ValueError):
        pkg.segment_ola_hop(seg, 3, 16, 0, 5, track)                      # 4 rows are not whole channels


@pytest.mark.parametrize("precision,gate", [("fp32", 70.0), ("bf16", 40.0)])
def test_stereo_track_at_075_matches_oracle(pkg, precision, gate):
    from mss_tf_locoformer_b200.segments import overlap_hop, separate_track
    cfg, sd, model = _model(pkg, precision)
    track = _mixture(5000, 2)
    seg = 1024
    hop = overlap_hop(seg, 0.75)
    want = ref.separate_track(lambda x: oracle.mss_forward(sd, cfg, x), track, seg, hop, batch=4)
    with torch.no_grad():
        got = separate_track(model, track.cuda(), seg_len=seg, batch=3, overlap=0.75)
    assert list(got) == list(want)
    for k in want:
        assert got[k].shape == (2, 5000)
        for c in range(2):
            sd_db = oracle.si_sdr_db(got[k][c].cpu(), want[k][c])
            assert sd_db >= gate, (k, c, sd_db)
            if precision == "fp32":
                assert float((got[k][c].cpu() - want[k][c]).abs().max()) <= 1e-4, (k, c)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stereo_channels_equal_mono_separation(pkg, precision):
    """The forward is batch-invariant and the stitch gathers in a fixed order, so each channel of a stereo
    separation is bit for bit the separation of that channel alone, at the same overlap."""
    from mss_tf_locoformer_b200.segments import separate_track
    _, _, model = _model(pkg, precision)
    track = _mixture(7000, 2, seed=3).cuda()
    with torch.no_grad():
        both = separate_track(model, track, seg_len=1024, batch=3, overlap=0.75)
        again = separate_track(model, track, seg_len=1024, batch=3, overlap=0.75)
        for c in range(2):
            one = separate_track(model, track[c], seg_len=1024, batch=3, overlap=0.75)
            for k in both:
                assert torch.equal(both[k][c], one[k]), (k, c)
                assert torch.equal(both[k], again[k]), k


def _track_worker(rank, world, port, ret):
    import torch.distributed as dist
    import mss_tf_locoformer_b200 as m
    from mss_tf_locoformer_b200.segments import separate_track
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        _, _, model = _model(m, "fp32")
        with torch.no_grad():
            out = separate_track(model, _mixture(9000, 2).cuda(), seg_len=1024, batch=3, overlap=0.75)
        ret[rank] = {k: v.cpu() for k, v in out.items()}
    finally:
        dist.destroy_process_group()


def test_two_gpus_nccl_at_075_matches_one_gpu(pkg):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from mss_tf_locoformer_b200.segments import separate_track
    _, _, model = _model(pkg, "fp32")
    with torch.no_grad():
        one = separate_track(model, _mixture(9000, 2).cuda(), seg_len=1024, batch=3, overlap=0.75)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_track_worker, args=(2, port, ret), nprocs=2, join=True)
        res = dict(ret)
    for r in (0, 1):
        for k in one:
            assert torch.allclose(res[r][k], one[k].cpu(), atol=1e-5, rtol=0), (r, k)
    for k in one:
        assert torch.equal(res[0][k], res[1][k])


def _cli_setup(tmp_path):
    import yaml
    cfg, sd, _ = load_golden("mss_hop2_macaron")
    ckpt = os.path.join(tmp_path, "model.pt")
    torch.save({"model_state_dict": sd, "epoch": 3}, ckpt)
    ycfg = os.path.join(tmp_path, "cfg.yaml")
    with open(ycfg, "w") as f:
        yaml.safe_dump({"model": cfg}, f)
    return cfg, sd, ckpt, ycfg


def _run_cli(cli, wav, ckpt, ycfg, out_dir, sr, *extra):
    cli.main(["--input", wav, "--checkpoint", ckpt, "--config", ycfg, "--output_dir", out_dir, "--sample_rate", str(sr),
              "--segment", str(1024 / sr), "--batch", "3", "--precision", "fp32", *extra])
    return {f: open(os.path.join(out_dir, f), "rb").read() for f in sorted(os.listdir(out_dir))}


def test_cli_stereo_and_overlap(pkg, tmp_path):
    from mss_tf_locoformer_b200 import separate as cli
    from mss_tf_locoformer_b200.segments import overlap_hop, separate_track
    cfg, sd, ckpt, ycfg = _cli_setup(tmp_path)
    sr = 8000
    stereo = torch.stack([_mixture(9000, 1, seed=1)[0], 0.5 * _mixture(9000, 1, seed=2)[0]])   # channels differ
    wav = os.path.join(tmp_path, "song.wav")
    cli.save_audio(stereo, wav, sample_rate=sr, normalize=False)
    audio, _ = cli.load_audio(wav, sample_rate=sr)

    # without --stereo: byte for byte the 50 % mono pipeline (down-mix, tfl_segment_ola, duplicated channel)
    default = _run_cli(cli, wav, ckpt, ycfg, os.path.join(tmp_path, "default"), sr)
    explicit = _run_cli(cli, wav, ckpt, ycfg, os.path.join(tmp_path, "explicit"), sr, "--overlap", "0.5")
    model = cli.load_model(ckpt, ycfg)
    model.precision = "fp32"
    with torch.no_grad():
        mono = separate_track(model, cli.downmix(audio).cuda(), seg_len=1024, batch=3)
    legacy = os.path.join(tmp_path, "legacy")
    os.makedirs(legacy)
    for k, v in mono.items():
        cli.save_audio(cli.to_stereo(v.cpu()), os.path.join(legacy, f"song_{k}.wav"), sample_rate=sr)
    want_bytes = {f: open(os.path.join(legacy, f), "rb").read() for f in sorted(os.listdir(legacy))}
    assert default == want_bytes and explicit == want_bytes

    # --stereo --overlap 0.75: two distinct channels, each the oracle's, one peak per stem file
    out_dir = os.path.join(tmp_path, "stereo")
    _run_cli(cli, wav, ckpt, ycfg, out_dir, sr, "--stereo", "--overlap", "0.75")
    want = ref.separate_track(lambda x: oracle.mss_forward(sd, cfg, x), audio, 1024, overlap_hop(1024, 0.75), batch=4)
    for k in want:
        got, got_sr = cli.load_audio(os.path.join(out_dir, f"song_{k}.wav"), sample_rate=sr)
        assert got_sr == sr and got.shape == (2, 9000) and not torch.equal(got[0], got[1])
        peak = want[k].abs().max()
        for c in range(2):
            assert oracle.si_sdr_db(got[c], want[k][c] / peak) >= 70.0, (k, c)
            assert float((got[c] - want[k][c] / peak).abs().max()) <= 2e-4, (k, c)


def test_cli_stereo_flag_keeps_mono_input(pkg, tmp_path):
    from mss_tf_locoformer_b200 import separate as cli
    _, _, ckpt, ycfg = _cli_setup(tmp_path)
    sr = 8000
    wav = os.path.join(tmp_path, "mono.wav")
    cli.save_audio(_mixture(9000, 1, seed=4), wav, sample_rate=sr, normalize=False)
    plain = _run_cli(cli, wav, ckpt, ycfg, os.path.join(tmp_path, "a"), sr)
    flagged = _run_cli(cli, wav, ckpt, ycfg, os.path.join(tmp_path, "b"), sr, "--stereo")
    assert plain and plain == flagged
