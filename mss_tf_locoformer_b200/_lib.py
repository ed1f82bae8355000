"""ctypes binding of include/tfl.h.  There is NO fallback: a missing library is an error."""
import contextlib
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TFL_LIB") or os.path.join(HERE, "csrc", "libtfl_b200.so")  # TFL_LIB: A/B builds in profiles/


class TflConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_fft", "hop", "n_src", "n_layers", "emb_dim", "num_groups", "tf_order", "n_heads", "attention_dim",
        "rope", "macaron", "ffn_hidden0", "ffn_hidden1", "conv_kernel", "enc_in_ch")] + [("eps", C.c_float)]


class TflError(RuntimeError):
    pass


_lib = None

class TflLossConfig(C.Structure):
    _fields_ = [("si_sdr_weight", C.c_float), ("l1_weight", C.c_float), ("spectral_weight", C.c_float), ("eps", C.c_float),
                ("spec_n_fft", C.c_int32), ("spec_hop", C.c_int32)]


_P, _I, _Z, _L, _F = C.c_void_p, C.c_int, C.c_size_t, C.c_int64, C.c_float
SIGNATURES = {  # name -> (restype, argtypes); must list every symbol of include/tfl.h
    "tfl_version": (_I, []),
    "tfl_last_error": (C.c_char_p, []),
    "tfl_launch_count": (C.c_uint64, []),
    "tfl_plan_create": (_I, [C.POINTER(TflConfig), C.POINTER(_P)]),
    "tfl_plan_destroy": (None, [_P]),
    "tfl_num_weight_tensors": (_I, [_P]),
    "tfl_packed_bytes": (_Z, [_P]),
    "tfl_pack_weights": (_I, [_P, C.POINTER(_P), _I, _P, _Z, _P]),
    "tfl_workspace_bytes": (_Z, [_P, _I, _I, _I, _I]),
    "tfl_stft": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "tfl_enc_conv_gln": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _Z, _P]),
    "tfl_enc_conv_gln_mode": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _Z, _I, _P]),
    "tfl_rms_group_norm": (_I, [_P, _P, _I, _I, _I, _P, _P, _L, _P]),
    "tfl_conv_swiglu_ffn": (_I, [_P, _P, _I, _I, _I, _P, _I, _I, _I, _P, _Z, _I, _P]),
    "tfl_conv_swiglu_ffn_out": (_I, [_P, _P, _I, _I, _I, _P, _P, _I, _I, _I, _P, _Z, _I, _P]),
    "tfl_rope_attn": (_I, [_P, _P, _I, _I, _P, _I, _I, _I, _P, _Z, _I, _P]),
    "tfl_dec_conv": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "tfl_dec_conv_mode": (_I, [_P, _P, _P, _I, _I, _I, _P, _I, _P]),
    "tfl_istft_ola": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "tfl_blocks": (_I, [_P, _P, _P, _I, _I, _I, _P, _Z, _I, _P]),
    "tfl_forward": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _Z, _I, _P]),
    "tfl_separator_forward": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _Z, _I, _P]),
    "tfl_segment_ola": (_I, [_P, _I, _I, _I, _I, _I, _P, _L, _L, _P]),
    "tfl_segment_ola_hop": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _L, _L, _P]),
    "tfl_pair_stats": (_I, [_P, _P, _I, _L, _P, _P, _Z, _P]),
    "tfl_bs_band_split": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "tfl_bs_band_decode": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P]),
    "tfl_bs_band_bwd_workspace_bytes": (_Z, [_I, _I, _I, _I, _I, _I, _I, _I]),
    "tfl_bs_band_decode_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P, _Z, _P]),
    "tfl_bs_band_split_bwd": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "tfl_train_grad_layout":(_L, [_P, C.POINTER(_L), C.POINTER(_L), _I]),
    "tfl_train_workspace_bytes": (_Z, [_P, _I, _I, _I, _I]),
    "tfl_train_stage_workspace_bytes": (_Z, [_P, _I, _I, _I]),
    "tfl_train_forward_backward": (_I, [_P, _P, C.POINTER(_P), _I, _P, _P, _I, _I, C.POINTER(TflLossConfig), _P, _P, _P, _P, _Z, _P]),
    "tfl_conv_swiglu_ffn_bwd": (_I, [_P, _P, C.POINTER(_P), _I, _I, _I, _I, _P, _P, _I, _I, _I, _P, _P, _Z, _P]),
    "tfl_rope_attn_bwd": (_I, [_P, _P, C.POINTER(_P), _I, _I, _I, _P, _P, _I, _I, _I, _P, _P, _Z, _P]),
    "tfl_sep_train_workspace_bytes": (_Z, [_P, _I, _I, _I]),
    "tfl_sep_train_forward": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _Z, _P]),
    "tfl_sep_train_backward": (_I, [_P, _P, C.POINTER(_P), _I, _P, _P, _I, _I, _I, _P, _P, _Z, _P]),
    "tfl_sep_train_backward_input": (_I, [_P, _P, C.POINTER(_P), _I, _P, _P, _I, _I, _I, _P, _P, _Z, _P, _P]),
    "tfl_mss_train_workspace_bytes": (_Z, [_P, _I, _I]),
    "tfl_mss_train_forward": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _Z, _P]),
    "tfl_mss_train_backward": (_I, [_P, _P, C.POINTER(_P), _I, _P, _P, _I, _I, _P, _P, _P, _Z, _P]),
    "tfl_blocks_train_forward": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _Z, _P]),
    "tfl_blocks_train_backward": (_I, [_P, _P, C.POINTER(_P), _I, _P, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "tfl_grad_clip_norm":(_I, [_P, _L, _F, _P, _P, _Z, _P]),
    "tfl_grad_accumulate": (_I, [_P, _P, _L, _F, _I, _P]),
    "tfl_adamw_step": (_I, [_P, _P, _P, _P, _L, _P, _F, _F, _F, _F, _F, _I, _P]),
    "tfl_debug_set_option": (_I, [_I, _I]),
    "tfl_debug_set_trace": (_I, [_P]),
    "tfl_debug_timeout": (_I, [C.POINTER(C.c_uint32), _I]),
    "tfl_tc_selftest": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
}


def load():
    """Load libtfl_b200.so (built by ``python -m mss_tf_locoformer_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the sm_100a CUDA library has not been built. Run "
            "`python -m mss_tf_locoformer_b200.build` (or __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if os.environ.get("TFL_PDL"):             # A/B: programmatic dependent launch of the bf16 kernels (default off)
        lib.tfl_debug_set_option(4, 1)
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        raise TflError(load().tfl_last_error().decode(errors="replace") or f"tfl error {status}")


OPT_DETERMINISTIC = 7   # include/tfl.h TFL_OPT_DETERMINISTIC


@contextlib.contextmanager
def deterministic_option(on: bool):
    """TFL_OPT_DETERMINISTIC = ``on`` for the duration of one training call, then back to the default 0.  The training
    entry points read it when called, and a workspace query, the saved forward sized by it and that forward's backward
    must all see the same value: callers pass ``torch.are_deterministic_algorithms_enabled()`` as read at the forward."""
    lib = load()
    check(lib.tfl_debug_set_option(OPT_DETERMINISTIC, 1 if on else 0))
    try:
        yield
    finally:
        lib.tfl_debug_set_option(OPT_DETERMINISTIC, 0)
