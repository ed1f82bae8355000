"""Host side of the autograd path of TFLocoformerMSS and of the separators' input gradient, without a GPU: the
workspace query, the refusal of CPU tensors and the C ABI entries."""
import pytest
import torch

import mss_tf_locoformer_b200 as pkg
from mss_tf_locoformer_b200 import _lib
from mss_tf_locoformer_b200.engine import Engine

MSS = dict(n_fft=256, hop_length=128, n_sources=2, n_layers=1, emb_dim=32, num_groups=4, n_heads=4, attention_dim=32,
           ffn_hidden_dim=64)
SEP = dict(num_spk=2, n_layers=1, emb_dim=32, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           attention_dim=32, pos_enc="rope", ffn_type="swiglu_conv1d", ffn_hidden_dim=64, conv1d_kernel=4)


def test_mss_workspace_query_is_host_only_and_grows_with_samples():
    lib = _lib.load()
    eng = Engine(pkg.TFLocoformerMSS(**MSS)._engine_cfg)
    small = lib.tfl_mss_train_workspace_bytes(eng.plan, 2, 6000)
    large = lib.tfl_mss_train_workspace_bytes(eng.plan, 2, 12000)
    assert 0 < small < large
    assert lib.tfl_mss_train_workspace_bytes(eng.plan, 2, 0) == 0
    assert lib.tfl_mss_train_workspace_bytes(None, 2, 6000) == 0
    # a separator plan has no STFT
    assert lib.tfl_mss_train_workspace_bytes(Engine(pkg.TFLocoformerSeparator(**SEP)._engine_cfg).plan, 2, 6000) == 0


def test_mss_workspace_exceeds_the_separator_workspace_at_the_same_frames():
    """Same network and frame count: the MSS workspace adds the mixture-gradient buffers (d spec, adjoint frames)."""
    lib = _lib.load()
    eng = Engine(pkg.TFLocoformerMSS(**MSS)._engine_cfg)
    T = 6000
    Tf, F = 1 + T // MSS["hop_length"], MSS["n_fft"] // 2 + 1
    assert lib.tfl_mss_train_workspace_bytes(eng.plan, 2, T) > lib.tfl_sep_train_workspace_bytes(eng.plan, 2, Tf, F)


def test_differentiable_cpu_tensors_have_no_cpu_path():
    mss = pkg.TFLocoformerMSS(**MSS).train()
    mss.differentiable = True
    with pytest.raises(RuntimeError, match="no CPU path"):
        mss(torch.randn(1, 1000))
    mss.requires_grad_(False)                        # a frozen model with a requires-grad input takes the same branch
    with pytest.raises(RuntimeError, match="no CPU path"):
        mss(torch.randn(1, 1000, requires_grad=True))
    sep = pkg.TFLocoformerSeparator(**SEP).train().requires_grad_(False)
    sep.differentiable = True
    with pytest.raises(RuntimeError, match="no CPU path"):
        sep(torch.randn(1, 5, 17, dtype=torch.complex64, requires_grad=True))


def test_requires_grad_input_is_refused_without_differentiable():
    """The input gradient is opt-in: without ``differentiable`` (or in eval mode) the forward-only refusal stands."""
    mss = pkg.TFLocoformerMSS(**MSS).train()
    with pytest.raises(NotImplementedError, match="forward-only"):
        mss(torch.randn(1, 1000, requires_grad=True))
    mss.differentiable = True
    mss.eval()
    with pytest.raises(NotImplementedError, match="forward-only"):
        mss(torch.randn(1, 1000, requires_grad=True))
    bs = pkg.BSLocoformerSeparator(**dict(SEP, sample_rate=44100, stft_size=256)).train()
    bs.differentiable = True
    with pytest.raises(NotImplementedError, match="forward-only"):
        bs(torch.randn(1, 5, 129, dtype=torch.complex64, requires_grad=True))


def test_dropout_refusal_comes_first():
    mss = pkg.TFLocoformerMSS(**MSS, dropout=0.1).train()
    mss.differentiable = True
    with pytest.raises(NotImplementedError, match="dropout"):
        mss(torch.randn(1, 1000, requires_grad=True))
