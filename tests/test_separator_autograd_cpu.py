"""Host side of the autograd path of the separators, without a GPU: the opt-in flag, the saved-forward workspace query
and the refusal of CPU tensors."""
import pytest
import torch

import mss_tf_locoformer_b200 as pkg
from mss_tf_locoformer_b200 import _lib
from mss_tf_locoformer_b200.engine import Engine
from mss_tf_locoformer_b200.espnet_separator import TFLocoformerSeparator as EspnetSeparator

SEP = dict(num_spk=2, n_layers=1, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           attention_dim=32, pos_enc="rope", ffn_type="swiglu_conv1d", ffn_hidden_dim=64, conv1d_kernel=4)
MSS = dict(n_fft=256, hop_length=128, n_sources=2, n_layers=1, emb_dim=32, num_groups=4, n_heads=4, attention_dim=32,
           ffn_hidden_dim=64)
BS = dict(SEP, sample_rate=44100, stft_size=256)


def test_differentiable_defaults_to_false():
    models = [pkg.TFLocoformerMSS(**MSS), pkg.TFLocoformerSeparator(**SEP), EspnetSeparator(129, **SEP),
              pkg.BSLocoformerSeparator(**BS)]
    assert all(m.differentiable is False for m in models)
    assert EspnetSeparator(129, **SEP, differentiable=True).differentiable is True


def test_saved_forward_workspace_query_is_host_only_and_grows_with_frames():
    lib = _lib.load()
    for model in (pkg.TFLocoformerSeparator(**SEP), pkg.BSLocoformerSeparator(**BS)):
        eng = Engine(model._engine_cfg)
        small = lib.tfl_sep_train_workspace_bytes(eng.plan, 2, 50, 129)
        large = lib.tfl_sep_train_workspace_bytes(eng.plan, 2, 100, 129)
        assert 0 < small < large
        # the saved forward keeps every sub-block input: more than the stage-level backward needs
        assert small > lib.tfl_train_stage_workspace_bytes(eng.plan, 2, 50, 129)
    assert 0 < lib.tfl_bs_band_bwd_workspace_bytes(1, 2, 10, 129, 32, 9, 2, 16) < \
        lib.tfl_bs_band_bwd_workspace_bytes(1, 2, 20, 129, 32, 9, 2, 16)


def test_differentiable_cpu_tensors_have_no_cpu_path():
    sep = pkg.TFLocoformerSeparator(**SEP).train()
    sep.differentiable = True
    x = torch.randn(1, 5, 17, dtype=torch.complex64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        sep(x)
    bs = pkg.BSLocoformerSeparator(**BS).train()
    bs.differentiable = True
    with pytest.raises(RuntimeError, match="no CPU path"):
        bs(torch.randn(1, 5, 129, dtype=torch.complex64))
