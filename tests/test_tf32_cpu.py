"""Host side of the tf32 precision mode (TFL_PRECISION_TF32), without a GPU: how the mode is selected, its workspace,
the C ABI's precision check, the CLI's arguments, and the instructions the tf32 tap-GEMM kernel is compiled to."""
import ctypes
import re
import shutil
import subprocess
import types

import pytest
import torch

import mss_tf_locoformer_b200 as pkg
from mss_tf_locoformer_b200 import _lib, separate
from mss_tf_locoformer_b200.engine import PRECISIONS, Engine
from mss_tf_locoformer_b200.modules import _resolve_precision

VD = dict(n_fft=2048, hop_length=1024, n_sources=4, n_layers=1, emb_dim=128, num_groups=4, n_heads=4, attention_dim=128,
          ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[384, 384])
XL = dict(n_fft=4096, hop_length=1024, n_sources=4, n_layers=2, emb_dim=256, num_groups=8, n_heads=16, attention_dim=256,
          ffn_type=["swiglu_conv1d", "swiglu_conv1d"], ffn_hidden_dim=[1024, 1024], conv1d_kernel=8)
SEP = dict(num_spk=2, n_layers=1, emb_dim=48, norm_type="rmsgroupnorm", num_groups=4, tf_order="ft", n_heads=4,
           attention_dim=48, pos_enc="rope", ffn_type="swiglu_conv1d", ffn_hidden_dim=192, conv1d_kernel=8)
# tfl_packed_bytes of these configurations: the tf32 mode reads the fp32 images and adds nothing to the pack
PACKED = {"variant_d": 20345088, "xlarge": 306465024, "separator": 3098624}


def _engines():
    return {"variant_d": Engine(pkg.TFLocoformerMSS(**VD)._engine_cfg),
            "xlarge": Engine(pkg.TFLocoformerMSS(**XL)._engine_cfg),
            "separator": Engine(pkg.TFLocoformerSeparator(**SEP)._engine_cfg)}


def test_precision_resolution():
    assert PRECISIONS["tf32"] == 2
    assert _resolve_precision(types.SimpleNamespace(precision="tf32")) == 2
    assert _resolve_precision(types.SimpleNamespace(precision="fp32")) == 0
    assert _resolve_precision(types.SimpleNamespace(precision="bf16")) == 1
    auto = types.SimpleNamespace(precision=None)
    assert _resolve_precision(auto) == 0
    # the default cuDNN flag (True) must not select the tf32 mode
    assert torch.backends.cudnn.allow_tf32
    assert _resolve_precision(auto) == 0
    with pytest.raises(ValueError):
        _resolve_precision(types.SimpleNamespace(precision="tf16"))


def test_precision_resolution_under_autocast(monkeypatch):
    """None follows torch.autocast(cuda): bf16 inside a bfloat16 region, fp32 inside a float16 region and outside."""
    state = {"on": False, "dtype": torch.bfloat16}
    monkeypatch.setattr(torch, "is_autocast_enabled", lambda device_type=None: state["on"])
    monkeypatch.setattr(torch, "get_autocast_dtype", lambda device_type=None: state["dtype"])
    auto = types.SimpleNamespace(precision=None)
    state.update(on=True, dtype=torch.bfloat16)
    assert _resolve_precision(auto) == 1
    state.update(on=True, dtype=torch.float16)
    assert _resolve_precision(auto) == 0
    state.update(on=False, dtype=torch.bfloat16)
    assert _resolve_precision(auto) == 0
    state.update(on=True, dtype=torch.bfloat16)
    assert _resolve_precision(types.SimpleNamespace(precision="tf32")) == 2


def test_workspace_is_the_fp32_layout_and_the_pack_is_unchanged():
    engines = _engines()
    for name, eng in engines.items():
        assert eng.lib.tfl_packed_bytes(eng.plan) == PACKED[name], name
        for shape in ((2, 50, 65), (1, 259, 1025), (8, 7, 2049)):
            assert eng.lib.tfl_workspace_bytes(eng.plan, *shape, 2) == eng.lib.tfl_workspace_bytes(eng.plan, *shape, 0)


def test_c_abi_rejects_unknown_precision():
    eng = _engines()["separator"]
    lib = eng.lib
    fake = ctypes.c_void_p(256)   # never dereferenced: every call below fails a host-side check before any launch
    assert lib.tfl_blocks(eng.plan, fake, fake, 1, 4, 5, fake, 1 << 20, 3, None) != 0
    assert "unknown precision 3" in lib.tfl_last_error().decode()
    assert lib.tfl_enc_conv_gln_mode(eng.plan, fake, fake, 1, 4, 5, fake, fake, 1 << 20, 3, None) != 0
    assert "unknown precision 3" in lib.tfl_last_error().decode()
    assert lib.tfl_conv_swiglu_ffn(eng.plan, fake, 0, 0, 0, fake, 1, 4, 5, fake, 1 << 20, 3, None) != 0
    assert "unknown precision 3" in lib.tfl_last_error().decode()
    # precision 2 passes the precision check and is stopped by a later host-side check before anything is launched: the
    # workspace size (with a device) or the device set-up (without one)
    assert lib.tfl_blocks(eng.plan, fake, fake, 1, 4, 5, fake, 1, 2, None) != 0
    msg = lib.tfl_last_error().decode()
    assert "unknown precision" not in msg
    if torch.cuda.is_available():
        assert "workspace too small" in msg, msg


def test_separate_cli_accepts_tf32():
    args = separate.parse_args(["--input", "a.wav", "--output_dir", "out", "--checkpoint", "m.pt", "--precision", "tf32"])
    assert args.precision == "tf32"
    assert separate.parse_args(["--input", "a.wav", "--output_dir", "out", "--checkpoint", "m.pt"]).precision == "bf16"
    with pytest.raises(SystemExit):
        separate.parse_args(["--input", "a.wav", "--output_dir", "out", "--checkpoint", "m.pt", "--precision", "fp16"])


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump (CUDA toolkit) not on PATH")
def test_tf32_tap_gemm_is_tcgen05():
    """Every instantiation of the tf32 tap-GEMM issues tcgen05 MMAs (UTC*MMA) and no mma.sync (HMMA)."""
    _lib.load()
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s*Function : (\S+)\n", sass)
    bodies = {name: body for name, body in zip(parts[1::2], parts[2::2]) if "tap_gemm_tf32_kernel" in name}
    assert len(bodies) >= 2, list(bodies)
    for name, body in bodies.items():
        assert re.search(r"\bUTC\w*MMA\b", body), name
        assert not re.search(r"\bHMMA\b", body), name
