"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the committed
reference vectors.  fp32 mode: max-abs <= 1e-4 and SI-SDR >= 70 dB; bf16 mode: SI-SDR >= 40 dB
(BASELINE.json north_star).  Run on the B200 box with ``pytest -m gpu``.
"""
import math

import pytest
import torch

import oracle
from conftest import load_golden

pytestmark = pytest.mark.gpu

FP32_MAXABS = 1e-4
FP32_SISDR = 70.0
BF16_SISDR = 40.0


@pytest.fixture(scope="module")
def pkg():
    import mss_tf_locoformer_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return m


def _check(got, ref, maxabs=FP32_MAXABS, sisdr=FP32_SISDR, what=""):
    got, ref = got.detach().cpu(), ref.detach().cpu()
    if got.is_complex():
        got, ref = torch.view_as_real(got.contiguous()), torch.view_as_real(ref.contiguous())
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = float((got - ref).abs().max())
    sd = oracle.si_sdr_db(got, ref)
    assert err <= maxabs, f"{what}: max-abs {err:.3e} > {maxabs}"
    assert sd >= sisdr, f"{what}: SI-SDR {sd:.1f} dB < {sisdr}"
    return err, sd


def _mss(pkg, name, precision="fp32"):
    cfg, sd, arr = load_golden(name)
    model = pkg.TFLocoformerMSS(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    model.precision = precision
    return cfg, sd, arr, model


@pytest.mark.parametrize("name", ["mss_hop2_macaron", "mss_hop4_single_tf"])
def test_mss_forward_golden_fp32(pkg, name):
    cfg, sd, arr, model = _mss(pkg, name)
    with torch.no_grad():
        out = model(arr["mixture"].cuda())
    assert list(out.keys()) == oracle.locoformer_oracle.SOURCE_NAMES[: cfg["n_sources"]]
    for k, v in out.items():
        _check(v, arr["out/" + k], what=f"{name}/{k}")
    if cfg["n_sources"] >= 4:
        with torch.no_grad():
            sp = model(arr["mixture"].cuda(), return_time_domain=False)
        for k, v in sp.items():
            assert v.shape == arr["spec/" + k].shape
            _check(v, arr["spec/" + k], maxabs=5e-4, what=f"{name}/spec/{k}")


@pytest.mark.parametrize("name", ["sep_rope_k4", "sep_nope_k1", "sep_rope_k8"])
def test_separator_golden_fp32(pkg, name):
    cfg, sd, arr = load_golden(name)
    model = pkg.TFLocoformerSeparator(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    with torch.no_grad():
        out = model(arr["spec_in"].cuda())
        out4 = model(arr["spec_in"].cuda().unsqueeze(1))
    _check(out, arr["spec_out"], maxabs=2e-4, what=name)
    assert torch.equal(out, out4)


def test_stage_kernels_fp32(pkg):
    """Each stage entry point of include/tfl.h against the reference's own stage outputs."""
    cfg, sd, arr, model = _mss(pkg, "mss_hop2_macaron")
    eng = model._ready()
    mix = arr["mixture"].cuda()
    # K1 stft: [B, Tf, F, 2] vs torch.stft of the reference [B, F, Tf]
    spec = eng.stft(mix)
    ref = torch.view_as_real(arr["stft"].transpose(1, 2).contiguous())
    _check(spec, ref, maxabs=2e-4, sisdr=100.0, what="stft")
    got_c = model.transform.stft(mix)
    assert got_c.shape == arr["stft"].shape
    # K7 istft: round trip of the reference STFT back to the mixture
    est = ref.cuda().unsqueeze(1).expand(-1, cfg["n_sources"], -1, -1, -1).contiguous()
    aud = eng.istft(est, mix.shape[-1])
    want = oracle.istft(arr["stft"].transpose(1, 2), cfg["n_fft"], cfg["hop_length"], mix.shape[-1])
    for s in range(cfg["n_sources"]):
        _check(aud[s], want, maxabs=2e-5, sisdr=100.0, what="istft")
    # K2 encoder + gLN
    x = eng.enc_conv_gln(ref.cuda())
    enc_ref = arr["stage/conv:out"].permute(0, 2, 3, 1)
    _check(x, enc_ref, maxabs=5e-5, what="enc_conv_gln")
    # K3 rms group norm (layer 0, freq path, attn_norm)
    nin, nout = arr["stage/blocks.0.freq_path.attn_norm:in"], arr["stage/blocks.0.freq_path.attn_norm:out"]
    _check(eng.rms_group_norm(0, 0, 2, nin.cuda()), nout, maxabs=2e-5, what="rms_group_norm")
    _check(model.blocks[0].freq_path.attn_norm(nin.cuda()), nout, maxabs=2e-5, what="RMSGroupNorm.forward")
    # K5 attention (+norm +residual): x + attn(norm(x))
    want = nin + arr["stage/blocks.0.freq_path.attn:out"].reshape(nin.shape)
    _check(eng.attn_(0, 0, nin.cuda().clone(), 0), want, maxabs=5e-5, what="rope_attn")
    # K4 FFN on both axes vs the oracle
    xin = enc_ref.contiguous()
    for axis, path in ((0, "freq_path"), (1, "frame_path")):
        for j in (0, 1):
            p = f"blocks.0.{path}"
            xa = xin if axis == 0 else xin.transpose(1, 2).contiguous()
            b, s1, s2, c = xa.shape
            xn = oracle.rms_group_norm(xa, sd[f"{p}.ffn_norm.{j}.gamma"], cfg["num_groups"], cfg["eps"])
            y = oracle.swiglu_conv_deconv(xn.reshape(b * s1, s2, c), sd[f"{p}.ffn.{j}.conv1d.weight"],
                                          sd[f"{p}.ffn.{j}.conv1d.bias"], sd[f"{p}.ffn.{j}.deconv1d.weight"],
                                          sd[f"{p}.ffn.{j}.deconv1d.bias"]).reshape(xa.shape) + xa
            want = y if axis == 0 else y.transpose(1, 2)
            _check(eng.ffn_(0, axis, j, xin.cuda().clone(), 0), want, maxabs=5e-5, what=f"ffn axis{axis} j{j}")
    # whole block through the module surface: [B, C, T, F] in / out
    blk = model.blocks[0](arr["stage/conv:out"].cuda())
    _check(blk, arr["stage/blocks.0:out"], maxabs=1e-4, what="TFLocoformerBlock.forward")
    # K6 decoder
    xfin = oracle.blocks_forward(enc_ref.contiguous(), sd, cfg)
    dec = eng.dec_conv(xfin.cuda())                                  # [B, S, Tf, F, 2]
    want = arr["stage/deconv:out"].permute(0, 2, 3, 1)               # [B, Tf, F, 2S]
    b, tf, f, _ = want.shape
    want = want.reshape(b, tf, f, -1, 2).permute(0, 3, 1, 2, 4)
    _check(dec, want, maxabs=1e-4, what="dec_conv")


def _random_model(pkg, cfg, seed=0):
    torch.manual_seed(seed)
    model = pkg.TFLocoformerMSS(**cfg).eval()
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.ndim == 1 and not n.endswith("rope.freqs"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    return model


def _mixture(n, batch, seed=1234):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n) / 44100.0
    x = 0.1 * torch.randn(batch, n, generator=g)
    for f0 in (55.0, 220.0, 880.0, 3520.0, 7040.0):
        x = x + 0.05 * torch.sin(2 * math.pi * f0 * t)[None]
    return x.clamp(-1, 1)


VARIANT_D = dict(n_fft=2048, hop_length=1024, n_sources=4, n_layers=1, emb_dim=128, norm_type="rmsgroupnorm",
                 num_groups=4, tf_order="ft", n_heads=4, flash_attention=True, attention_dim=128, pos_enc="rope",
                 ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[384, 384], conv1d_kernel=4,
                 conv1d_shift=1, dropout=0.0, eps=1e-5)
VARIANT_Y = dict(VARIANT_D, hop_length=512, emb_dim=96, attention_dim=96)
VARIANT_SMALL = dict(VARIANT_D, n_fft=1024, hop_length=256, emb_dim=48, attention_dim=48, ffn_hidden_dim=[192, 192])


@pytest.mark.parametrize("name,cfg,n_samples", [("D", VARIANT_D, 30000), ("Y", VARIANT_Y, 20000),
                                                 ("small", VARIANT_SMALL, 12000)])
def test_real_width_one_layer_fp32(pkg, name, cfg, n_samples):
    """Production channel widths (one layer, ~0.5 s audio) against the live oracle."""
    model = _random_model(pkg, cfg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    mix = _mixture(n_samples, 1)
    ocfg = dict(cfg)
    want = oracle.mss_forward(sd, ocfg, mix)
    model = model.cuda()
    model.precision = "fp32"
    with torch.no_grad():
        got = model(mix.cuda())
    for k in want:
        _check(got[k], want[k], what=f"{name}/{k}")


def test_batch_rows_are_independent(pkg):
    """Size-independent property: a batch of segments equals the segments run one by one, bit for bit."""
    cfg, sd, arr, model = _mss(pkg, "mss_hop2_macaron")
    mix = torch.cat([arr["mixture"], arr["mixture"].flip(0) * 0.5], 0).cuda()
    with torch.no_grad():
        full = model(mix)
        for b in range(mix.shape[0]):
            one = model(mix[b:b + 1])
            for k in full:
                assert torch.equal(full[k][b], one[k][0]), (k, b)


def test_errors(pkg):
    cfg, sd, arr, model = _mss(pkg, "mss_hop2_macaron")
    with pytest.raises(RuntimeError):
        model(torch.zeros(1, cfg["n_fft"] // 2, device="cuda"))          # reflect pad too large, as torch.stft
    with pytest.raises(RuntimeError):
        model(arr["mixture"])                                             # CPU tensor: no CPU path
    model.precision = "fp16"
    with pytest.raises(ValueError):
        model(arr["mixture"].cuda())


def test_segment_ola_matches_oracle(pkg):
    seg_len, n_src, n = 512, 3, 1700
    starts = oracle.segment_starts(n, seg_len)
    g = torch.Generator().manual_seed(5)
    seg = torch.randn(len(starts), n_src, seg_len, generator=g)
    want = oracle.stitch_segments(seg, n)
    track = torch.zeros(n_src, n, device="cuda")
    for i0 in range(0, len(starts), 2):                                  # batches of 2 segments, [S, B, L]
        chunk = seg[i0:i0 + 2].permute(1, 0, 2).contiguous().cuda()
        pkg.segment_ola(chunk, i0, len(starts), track)
    _check(track, want, maxabs=1e-5, sisdr=100.0, what="segment_ola")


def test_full_track_segments_match_oracle_stitch(pkg):
    """BASELINE config 3 in miniature: chunked inference with 50 % overlap == oracle forward per segment + oracle stitch."""
    from mss_tf_locoformer_b200.segments import separate_track
    cfg, sd, arr, model = _mss(pkg, "mss_hop2_macaron")
    track = _mixture(5000, 1)[0]
    seg = 1024
    want = oracle.separate_track(lambda x: oracle.mss_forward(sd, cfg, x), track, seg, batch=2)
    with torch.no_grad():
        got = separate_track(model, track.cuda(), seg_len=seg, batch=3)
    assert list(got) == list(want)
    for k in want:
        _check(got[k], want[k], what=f"track/{k}")


@pytest.mark.parametrize("name", ["bs_stereo_mask", "bs_mono_map"])
def test_bs_separator_golden_fp32(pkg, name):
    """BS-Locoformer (band-split encoder, Locoformer blocks over the band axis, band-wise decoder, complex mask)."""
    cfg, sd, arr = load_golden(name)
    model = pkg.BSLocoformerSeparator(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    with torch.no_grad():
        out = model(arr["spec_in"].cuda())
    assert out.shape == arr["spec_out"].shape
    _check(out, arr["spec_out"], maxabs=2e-4, what=name)


def test_full_size_properties_bf16(pkg):
    """BASELINE configs[1] at full size (Variant D, 6 layers, 6-s segments): properties that need no oracle run."""
    import bench
    model = bench.make_state_dict(dict(bench.VARIANT_D)).cuda()
    model.precision = "bf16"
    mix = bench.make_mixture(3, bench.SEG).cuda()
    with torch.no_grad():
        full = model(mix)
        again = model(mix)
        one = model(mix[1:2])
    for k in full:
        assert full[k].shape == (3, bench.SEG) and torch.isfinite(full[k]).all()
        assert torch.equal(full[k], again[k]), k                      # run-to-run deterministic
        assert torch.equal(full[k][1], one[k][0]), k                  # batch rows independent, bit for bit
    # STFT -> iSTFT round trip (NOLA) through the same kernels at full size
    eng = model._ready()
    spec = eng.stft(mix)
    est = spec.unsqueeze(1).expand(-1, 4, -1, -1, -1).contiguous()
    back = eng.istft(est, bench.SEG)
    n_ok = (bench.SEG // 1024) * 1024 - 2048
    assert float((back[0][:, :n_ok] - mix[:, :n_ok]).abs().max()) < 2e-5


def test_bench_dump_outputs_are_the_timed_forward(pkg, tmp_path):
    """bench.py --dump-outputs, run as a program: the dumped sources are bit for bit the forward of bench's seeded
    weights and mixture (so two runs, or two builds, with the same arguments get the same inputs)."""
    import os
    import subprocess
    import sys
    import numpy as np
    import bench
    dump = tmp_path / "dump"
    proc = subprocess.run([sys.executable, bench.__file__, "--batch", "2", "--steps", "2", "--warmup", "1",
                           "--no-cpu-baseline", "--dump-outputs", str(dump)], cwd=tmp_path, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr[-2000:]
    model = bench.make_state_dict(dict(bench.VARIANT_D)).cuda()
    model.precision = "bf16"
    with torch.no_grad():
        want = model(bench.make_mixture(2, bench.SEG, seed=1234).cuda())
    assert sorted(os.listdir(dump)) == sorted(f"{k}.npy" for k in want)
    for k, v in want.items():
        got = np.load(dump / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, v.cpu().numpy()), k


@pytest.mark.parametrize("n_samples", [129, 130, 255, 256, 257, 1000, 1024, 4097])
def test_ragged_lengths_fp32(pkg, n_samples):
    """Edge lengths around the reflect-pad minimum (n_fft/2 + 1) and hop multiples; workspace re-planned per shape."""
    cfg, sd, arr, model = _mss(pkg, "mss_hop2_macaron")
    mix = _mixture(n_samples, 1, seed=n_samples)
    want = oracle.mss_forward(sd, cfg, mix)
    with torch.no_grad():
        got = model(mix.cuda())
    for k in want:
        assert got[k].shape == (1, n_samples)
        _check(got[k], want[k], what=f"T={n_samples}/{k}")


def _track_worker(rank, world, port, ret):
    import os
    import torch.distributed as dist
    import mss_tf_locoformer_b200 as m
    from mss_tf_locoformer_b200.segments import separate_track
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        cfg, sd, arr = load_golden("mss_hop2_macaron")
        model = m.TFLocoformerMSS(**cfg)
        model.load_state_dict(sd, strict=True)
        model = model.cuda().eval()
        track = _mixture(9000, 1)[0].cuda()
        with torch.no_grad():
            out = separate_track(model, track, seg_len=1024, batch=3)
        ret[rank] = {k: v.cpu() for k, v in out.items()}
    finally:
        dist.destroy_process_group()


def test_full_track_two_gpus_nccl_matches_one_gpu(pkg):
    """Halo exchange (NCCL send/recv) + all-gather of the own ranges on 2 GPUs == the single-GPU stitch: bit-exact
    outside the halo between the two ranks, <= 1 ulp-level inside it (two addends summed in another order)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    from mss_tf_locoformer_b200.segments import separate_track
    cfg, sd, arr, model = _mss(pkg, "mss_hop2_macaron")
    track = _mixture(9000, 1)[0].cuda()
    with torch.no_grad():
        one = separate_track(model, track, seg_len=1024, batch=3)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_track_worker, args=(2, port, ret), nprocs=2, join=True)
        res = dict(ret)
    for r in (0, 1):
        for k in one:
            assert torch.allclose(res[r][k], one[k].cpu(), atol=1e-6, rtol=0), (r, k)
    for k in one:
        assert torch.equal(res[0][k], res[1][k])


def test_device_metrics_match_reference_numpy(pkg):
    """SURVEY N4: evaluation/metrics.py on the device (tfl_pair_stats) against the reference's numpy arithmetic."""
    import numpy as np
    from mss_tf_locoformer_b200 import metrics
    g = torch.Generator().manual_seed(3)
    t = torch.randn(2, 100001, generator=g)
    e = 0.7 * t + 0.2 * torch.randn(2, 100001, generator=g) + 0.01
    en, tn, eps = e.double().numpy().ravel(), t.double().numpy().ravel(), 1e-8
    e0, t0 = en - en.mean(), tn - tn.mean()
    sc = np.dot(e0, t0) / (np.dot(t0, t0) + eps)
    want_si = 10 * np.log10((np.dot(sc * t0, sc * t0) + eps) / (np.dot(e0 - sc * t0, e0 - sc * t0) + eps))
    want_sdr = 10 * np.log10((np.dot(tn, tn) + eps) / (np.dot(en - tn, en - tn) + eps))
    sc2 = np.dot(en, tn) / (np.dot(tn, tn) + eps)
    want_sar = 10 * np.log10((np.dot(sc2 * tn, sc2 * tn) + eps) / (np.dot(en - sc2 * tn, en - sc2 * tn) + eps))
    got = metrics.compute_all_metrics(e.cuda(), t.cuda())
    assert abs(got["si_sdr"] - want_si) < 1e-4 and abs(got["sdr"] - want_sdr) < 1e-4
    assert abs(got["sar"] - want_sar) < 1e-4 and got["sir"] == got["sar"]
    res = metrics.evaluate_source_separation({"vocals": e[0].cuda(), "bass": e[1].cuda()}, {"vocals": t[0].cuda(), "bass": t[1].cuda()})
    assert set(res) == {"vocals", "bass", "average"} and "avg_si_sdr" in res["average"]


def test_cli_end_to_end(pkg, tmp_path):
    """SURVEY N2: the inference CLI (checkpoint + YAML -> wav files) against the oracle run through the same stitch."""
    import os
    import yaml
    from mss_tf_locoformer_b200 import separate as cli
    cfg, sd, arr = load_golden("mss_hop2_macaron")
    ckpt = os.path.join(tmp_path, "model.pt")
    torch.save({"model_state_dict": sd, "epoch": 3}, ckpt)           # utils/common.py:46-74 wrapper
    ycfg = os.path.join(tmp_path, "cfg.yaml")
    with open(ycfg, "w") as f:
        yaml.safe_dump({"model": cfg, "training": {"lr": 1e-3}}, f)
    sr = 8000
    stereo = torch.stack([_mixture(9000, 1, seed=1)[0], _mixture(9000, 1, seed=2)[0]])
    wav = os.path.join(tmp_path, "song.wav")
    cli.save_audio(stereo, wav, sample_rate=sr, normalize=False)
    out_dir = os.path.join(tmp_path, "out")
    cli.main(["--input", wav, "--checkpoint", ckpt, "--config", ycfg, "--output_dir", out_dir, "--sample_rate", str(sr),
              "--segment", str(1024 / sr), "--batch", "3", "--precision", "fp32"])
    mono = stereo.mean(0)
    want = oracle.separate_track(lambda x: oracle.mss_forward(sd, cfg, x), mono, 1024, batch=2)
    for k in want:
        got, got_sr = cli.load_audio(os.path.join(out_dir, f"song_{k}.wav"), sample_rate=sr)
        assert got_sr == sr and got.shape == (2, 9000) and torch.equal(got[0], got[1])
        ref = want[k] / want[k].abs().max()                          # save_audio(normalize=True)
        _check(got[0], ref, maxabs=2e-4, what=f"cli/{k}")


def test_espnet_adapter_forward(pkg):
    """SURVEY N3: the ESPnet AbsSeparator surface (list of num_spk complex [B, T, F], ilens passthrough, OrderedDict)."""
    from collections import OrderedDict
    from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as EspnetSeparator
    cfg, sd, arr = load_golden("sep_rope_k8")
    model = EspnetSeparator(arr["spec_in"].shape[-1], **cfg)
    model.load_state_dict(pkg.strip_prefix({"separator." + k: v for k, v in sd.items()}), strict=True)
    model = model.cuda().eval()
    ilens = torch.tensor([arr["spec_in"].shape[1]] * arr["spec_in"].shape[0])
    with torch.no_grad():
        outs, ol, extra = model(arr["spec_in"].cuda(), ilens)
        outs4, _, _ = model(arr["spec_in"].cuda().unsqueeze(2), ilens)          # ESPnet's [B, T, C = 1, F]
    assert isinstance(extra, OrderedDict) and len(extra) == 0 and ol is ilens and len(outs) == model.num_spk
    for s, o in enumerate(outs):
        _check(o, arr["spec_out"][:, s], maxabs=2e-4, what=f"espnet/spk{s}")
        assert torch.equal(o, outs4[s])


@pytest.mark.parametrize("emb,n_src,batch,n_frames,n_freq", [
    (128, 4, 2, 7, 1025),     # BASELINE width, nine strips (eight full + 17 bins)
    (128, 4, 1, 1, 129),      # a single frame: every output flushed by the last-frame clause
    (128, 4, 3, 2, 126),      # exactly one full strip
    (128, 4, 40, 3, 127),     # more (sample, strip, run) items than resident blocks: accumulators reused across items
    (96, 4, 2, 9, 513),       # Variant Y width (three 32-channel chunks)
    (64, 2, 2, 5, 65),        # two sources (outputs 4..7 unused), F < 126
    (32, 4, 1, 300, 33),      # long frame axis split into runs with halo frames
])
def test_decoder_bf16_mode_kernels(pkg, emb, n_src, batch, n_frames, n_freq):
    """K6 in bf16 mode (tf32 mma.sync): the scatter-form kernel (default) and the 9-tap gather kernel against the
    oracle's ConvTranspose2d restatement (models/mss_tflocoformer.py:182) in float64.  tf32 operands: 2^-11 relative
    per product, so the gate is 2e-3 of the output scale; the two kernels share operands and differ only in summation
    order.  The scatter kernel's summation order does not depend on the batch index or on the strip / run split:
    a sample computed alone is bit-identical to the same sample inside a batch."""
    from mss_tf_locoformer_b200 import _lib
    lib = _lib.load()
    cfg = dict(VARIANT_D, emb_dim=emb, attention_dim=emb, n_sources=n_src, ffn_hidden_dim=[64, 64])
    model = _random_model(pkg, cfg).cuda()
    eng = model._ready()
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    g = torch.Generator().manual_seed(7)
    x = torch.randn(batch, n_frames, n_freq, emb, generator=g)
    want = oracle.decoder(x.double(), sd["deconv.weight"].double(), sd["deconv.bias"].double())
    want = want.reshape(batch, n_frames, n_freq, n_src, 2).permute(0, 3, 1, 2, 4)
    scale = float(want.abs().max())
    got = {}
    try:
        for opt in (2, 1):
            assert lib.tfl_debug_set_option(6, opt) == 0
            got[opt] = eng.dec_conv(x.cuda(), 1).cpu()
            err = float((got[opt].double() - want).abs().max())
            assert err <= 2e-3 * scale, (opt, err, scale)
        assert float((got[1] - got[2]).abs().max()) <= 1e-4 * scale
        lib.tfl_debug_set_option(6, 2)
        b = batch - 1
        alone = eng.dec_conv(x[b:b + 1].cuda(), 1).cpu()
        assert torch.equal(alone[0], got[2][b])
    finally:
        lib.tfl_debug_set_option(6, 2)
