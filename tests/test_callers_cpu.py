"""Host logic of the callers either side of the hot path (SURVEY 8f rows N2-N4) that needs no GPU:
audio I/O helpers of the CLI, the ESPnet adapter's surface, the metric closed forms."""
import math
import os

import numpy as np
import pytest
import torch

from mss_tf_locoformer_b200 import separate as cli
from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as EspnetSeparator
from mss_tf_locoformer_b200.models import TFLocoformerSeparator, strip_prefix

MAC = ["swiglu_conv1d", "swiglu_conv1d"]


def test_wav_round_trip_and_downmix(tmp_path):
    sr = 44100
    g = torch.Generator().manual_seed(0)
    x = 0.5 * torch.randn(2, 5000, generator=g)
    path = os.path.join(tmp_path, "a.wav")
    cli.save_audio(x, path, sample_rate=sr, normalize=False)
    y, got_sr = cli.load_audio(path, sample_rate=sr)
    assert got_sr == sr and y.shape == x.shape and torch.allclose(x, y, atol=1e-7)
    # peak normalisation as utils/audio.py:58-62
    cli.save_audio(x, path, sample_rate=sr, normalize=True)
    z, _ = cli.load_audio(path, sample_rate=sr)
    assert abs(float(z.abs().max()) - 1.0) < 1e-6
    # mono down-mix = channel mean (inference/separate.py:135-139); stereo duplication (:158-162)
    assert torch.allclose(cli.downmix(x), x.mean(0))
    assert cli.downmix(x[:1]).shape == (5000,)
    st = cli.to_stereo(x[0])
    assert st.shape == (2, 5000) and torch.equal(st[0], st[1])
    assert cli.to_stereo(x[:1]).shape == (2, 5000)


def test_int16_and_resample(tmp_path):
    from scipy.io import wavfile
    sr = 22050
    t = np.arange(sr) / sr
    sig = (0.5 * np.sin(2 * math.pi * 440 * t) * 32767).astype(np.int16)
    path = os.path.join(tmp_path, "b.wav")
    wavfile.write(path, sr, sig)
    y, got_sr = cli.load_audio(path, sample_rate=44100)
    assert got_sr == 44100 and y.shape == (1, 44100)
    assert abs(float(y.abs().max()) - 0.5) < 0.02


def test_cli_flags_match_reference():
    a = cli.parse_args(["--input", "x.wav", "--checkpoint", "m.pt"])
    # the reference's flags and defaults (inference/separate.py:28-76)
    assert (a.output_dir, a.config, a.sample_rate, a.seed) == ("./separated", None, 44100, 42)
    assert (a.segment, a.batch, a.precision) == (6.0, 8, "bf16")
    with pytest.raises(SystemExit):
        cli.parse_args(["--input", "x.wav"])                       # --checkpoint is required, as in the reference


def test_espnet_adapter_surface():
    cfg = dict(num_spk=2, n_layers=1, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
               attention_dim=32, pos_enc="rope", ffn_type=MAC, ffn_hidden_dim=[32, 32], conv1d_kernel=8)
    torch.manual_seed(0)
    a = EspnetSeparator(65, **cfg)
    torch.manual_seed(0)
    b = TFLocoformerSeparator(**cfg)
    assert a.num_spk == 2
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)      # same keys, same seeded init
    # ESPnet checkpoints carry "separator." (tests/test_tflocoformer_load_pretrained_weights.py:68-73)
    ck = {"separator." + k: v for k, v in sb.items()}
    ck["encoder.something"] = torch.zeros(1)
    a.load_state_dict(strip_prefix(ck), strict=True)
    with pytest.raises(RuntimeError):
        a(torch.zeros(1, 10, 65, dtype=torch.complex64), torch.tensor([10]))        # CPU tensor: no CPU path


def test_metric_closed_forms_match_reference_formulas():
    """The five-sum closed forms of metrics.py against the reference's numpy code restated literally."""
    g = np.random.default_rng(0)
    t = g.standard_normal(4000)
    e = 0.8 * t + 0.1 * g.standard_normal(4000) + 0.05
    s = [e.sum(), t.sum(), (e * e).sum(), (t * t).sum(), (e * t).sum()]
    n, eps = len(e), 1e-8
    # reference compute_si_sdr (evaluation/metrics.py:35-56)
    e0, t0 = e - e.mean(), t - t.mean()
    scale = np.dot(e0, t0) / (np.dot(t0, t0) + eps)
    st = scale * t0
    want = 10 * np.log10((np.dot(st, st) + eps) / (np.dot(e0 - st, e0 - st) + eps))
    dot = s[4] - s[0] * s[1] / n
    te = s[3] - s[1] * s[1] / n
    ee = s[2] - s[0] * s[0] / n
    sc = dot / (te + eps)
    got = 10 * math.log10((sc * sc * te + eps) / (ee - 2 * sc * dot + sc * sc * te + eps))
    assert abs(got - want) < 1e-8
    # reference compute_sdr (:78-84)
    want = 10 * np.log10((np.dot(t, t) + eps) / (np.dot(e - t, e - t) + eps))
    got = 10 * math.log10((s[3] + eps) / (s[2] - 2 * s[4] + s[3] + eps))
    assert abs(got - want) < 1e-8


def test_bench_reference_arm_line(monkeypatch, capsys):
    """bench.py --impl reference: rank 0 alone prints ONE JSON line whose metric / unit / config are the b200 arm's (the
    bounded sample is named in cpu_baseline.sample), with the reference-arm keys of the measurement contract; other
    ranks print nothing.  The CPU forward itself is stubbed here (it takes a minute per 6-s segment)."""
    import argparse
    import json
    import bench

    class Stub:
        def __call__(self, mix):
            return {"vocals": mix}

    monkeypatch.setattr(bench, "reference_model", lambda cfg, sd, device="cpu": (Stub(), "reference"))
    monkeypatch.setattr(bench, "make_state_dict", lambda cfg, seed=0: torch.nn.Linear(1, 1))
    args = argparse.Namespace(variant="D", steps=2, warmup=1, gpus=2, batch=8)
    bench.run_reference(args, rank=1)
    assert capsys.readouterr().out == ""
    bench.run_reference(args, rank=0)
    lines = [l for l in capsys.readouterr().out.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["unit"] == "audio-s/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 2 and line["steps"] == 2 and line["warmup"] == 1
    assert line["config"] == bench.workload_config("D", 8)
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["value"] == line["value"]
    assert "6.00-s mono segment" in line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_dump_outputs_full_and_sampled(tmp_path):
    """bench.py --dump-outputs: float32 .npy per source, whole when the arrays fit the budget, else the same seeded
    sample of every array (identical from call to call) within it."""
    import bench
    g = torch.Generator().manual_seed(3)
    out = {"vocals": torch.randn(2, 1000, generator=g, dtype=torch.float64), "drums": torch.randn(2, 1000, generator=g)}
    bench.dump_outputs(out, str(tmp_path / "full"))
    for k, v in out.items():
        a = np.load(tmp_path / "full" / f"{k}.npy")
        assert a.dtype == np.float32 and a.shape == (2, 1000)
        assert np.array_equal(a, v.float().numpy())
    budget = 4 * 1000 + 2 * bench.NPY_HEADER              # files of a quarter of the 4000 elements
    for run in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / run), budget=budget)
    sizes = 0
    for k, v in out.items():
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert a.dtype == np.float32 and a.shape == (500,) and np.array_equal(a, b)
        assert np.isin(a, v.float().numpy().reshape(-1)).all()
        sizes += os.path.getsize(tmp_path / "a" / f"{k}.npy")
    assert sizes <= budget


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--dump-outputs", "d", "--train", "D"],
                                  ["--dump-outputs", "d", "--impl", "reference"],
                                  ["--dump-outputs", "d", "--impl", "reference-gpu"]])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    """No timed step, or a dump requested from a path that does not write one: an argument error before any work."""
    import bench
    monkeypatch.setattr("sys.argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2


def test_bench_train_dtype_names_the_operand_type():
    import bench
    assert bench.train_dtype(bench.TRAIN_CFGS["D"][0]) == "bf16"          # tcgen05 forward + bf16 mma.sync backward
    assert bench.train_dtype(bench.TRAIN_CFGS["xlarge"][0]) == "tf32"     # 16 heads x 16 at emb 256: tf32 mma.sync
