"""Host side of the deterministic training mode (TFL_OPT_DETERMINISTIC), without a GPU: the workspace queries with the
option on and off, and the option set from torch's flag around a training call."""
import pytest
import torch

import mss_tf_locoformer_b200 as pkg
from mss_tf_locoformer_b200 import _lib
from mss_tf_locoformer_b200.engine import Engine

MSS = dict(n_fft=256, hop_length=128, n_sources=2, n_layers=1, emb_dim=32, num_groups=4, n_heads=4, attention_dim=32,
           ffn_hidden_dim=64)
VD = dict(n_fft=2048, hop_length=1024, n_sources=4, n_layers=1, emb_dim=128, num_groups=4, n_heads=4, attention_dim=128,
          ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[384, 384])
SEP = dict(num_spk=2, n_layers=1, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           attention_dim=32, pos_enc="rope", ffn_type="swiglu_conv1d", ffn_hidden_dim=64, conv1d_kernel=4)
BS = dict(SEP, sample_rate=44100, stft_size=256)


def _queries(engines):
    """(name, zero-argument query) for every training workspace query, on MSS, separator and blocks-only plans (the
    engines that own the plans are kept in ``engines``)."""
    lib = _lib.load()

    def plan_of(model):
        engines.append(Engine(model._engine_cfg))
        return engines[-1].plan

    out = []
    for name, cfg in (("mss", MSS), ("variant_d", VD)):
        plan = plan_of(pkg.TFLocoformerMSS(**cfg))
        out += [(f"{name} train", lambda p=plan: lib.tfl_train_workspace_bytes(p, 2, 24000, 2048, 1024)),
                (f"{name} mss_train", lambda p=plan: lib.tfl_mss_train_workspace_bytes(p, 2, 24000)),
                (f"{name} stage", lambda p=plan: lib.tfl_train_stage_workspace_bytes(p, 2, 24, 129))]
    sep = plan_of(pkg.TFLocoformerSeparator(**SEP))
    out.append(("sep_train", lambda: lib.tfl_sep_train_workspace_bytes(sep, 2, 9, 21)))
    blocks = plan_of(pkg.BSLocoformerSeparator(**BS))
    out.append(("blocks-only sep_train", lambda: lib.tfl_sep_train_workspace_bytes(blocks, 2, 20, 30)))
    return out


def test_workspace_grows_with_the_option_and_off_is_unchanged():
    lib = _lib.load()
    engines = []
    for name, query in _queries(engines):
        off = query()
        assert off > 0, name
        assert lib.tfl_debug_set_option(_lib.OPT_DETERMINISTIC, 1) == 0
        try:
            on = query()
        finally:
            assert lib.tfl_debug_set_option(_lib.OPT_DETERMINISTIC, 0) == 0
        assert on > off, (name, on, off)
        assert query() == off, name


def test_deterministic_option_follows_the_torch_flag_and_resets():
    """The scope the training entry points run in: the option equals the value given (the callers pass
    torch.are_deterministic_algorithms_enabled()), and is back to 0 afterwards, also when the call raises."""
    lib = _lib.load()
    eng = Engine(pkg.TFLocoformerMSS(**MSS)._engine_cfg)
    plan = eng.plan
    off = lib.tfl_mss_train_workspace_bytes(plan, 2, 6000)
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        for flag in (False, True):
            torch.use_deterministic_algorithms(flag)
            with _lib.deterministic_option(torch.are_deterministic_algorithms_enabled()):
                inside = lib.tfl_mss_train_workspace_bytes(plan, 2, 6000)
            assert (inside > off) == flag
            assert lib.tfl_mss_train_workspace_bytes(plan, 2, 6000) == off
        with pytest.raises(ValueError):
            with _lib.deterministic_option(True):
                raise ValueError("training call failed")
        assert lib.tfl_mss_train_workspace_bytes(plan, 2, 6000) == off
    finally:
        torch.use_deterministic_algorithms(prev)
