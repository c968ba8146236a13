"""ctypes binding of `libsnrse_b200.so` (the C ABI in include/snrse_b200.h).

Fails loudly: a missing library raises ImportError-like RuntimeError at load time, and any
non-zero status from the library raises RuntimeError with the library's message.  There is no
fallback implementation behind these calls.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsnrse_b200.so")

_lib = None

vp, i32, i64, u64, f32, f64 = c_void_p, c_int, c_int64, c_uint64, c_float, c_double

# name -> (restype, argtypes); every symbol declared in include/snrse_b200.h
PROTOTYPES = {
    "snrse_version": (i32, []),
    "snrse_last_error": (c_char_p, []),
    "snrse_device_check": (i32, []),
    "snrse_launch_count": (ctypes.c_longlong, []),
    "snrse_set_pdl": (i32, [i32]),
    "snrse_stft": (i32, [vp, vp, vp, i32, vp, i32, i32, i32, i32, f32, f32, i32, vp]),
    "snrse_istft_workspace_bytes": (i64, [i32, i32]),
    "snrse_istft": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, f32, vp]),
    "snrse_spec_transform": (i32, [vp, vp, i64, i32, i32, f32, f32, vp]),
    "snrse_si_sdr": (i32, [vp, vp, vp, i32, i32, vp, vp]),
    "snrse_absmax": (i32, [vp, vp, i32, i32, vp, vp]),
    "snrse_v3_scalars": (i32, [vp, vp, f64, f32, vp, vp, vp, vp, i32, vp]),
    "snrse_snr_ratio": (i32, [vp, vp, i32, vp]),
    "snrse_lincomb": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, vp]),
    "snrse_lincomb_keyed": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, u64, vp, i32, vp, vp, vp, i32, i64, vp]),
    "snrse_rk_combine": (i32, [vp, vp, i32, i64, f32, vp, vp, vp]),
    "snrse_rk_partials": (i32, [i64]),
    "snrse_rk_scaled_sqnorm": (i32, [vp, i32, i64, f32, vp, vp, vp, f32, f32, vp, vp]),
    "snrse_ncsnpp_create": (i32, [POINTER(vp), i32, POINTER(i32), i32, i32, POINTER(i32), i32, i32]),
    "snrse_ncsnpp_destroy": (None, [vp]),
    "snrse_ncsnpp_num_modules": (i32, [vp]),
    "snrse_ncsnpp_num_params": (i32, [vp]),
    "snrse_ncsnpp_weight_bytes": (i64, [vp]),
    "snrse_ncsnpp_param_info": (i32, [vp, i32, c_char_p, i32, POINTER(i32), POINTER(i64), POINTER(i64), POINTER(i64), POINTER(i32)]),
    "snrse_ncsnpp_param_shape": (i32, [vp, i32, POINTER(i64), POINTER(i32)]),
    "snrse_ncsnpp_set_weights": (i32, [vp, vp]),
    "snrse_ncsnpp_plan_bytes": (i64, [vp, i32, i32, i32, i32]),
    "snrse_ncsnpp_plan_bind": (i32, [vp, i32, i32, i32, vp, i64]),
    "snrse_ncsnpp_forward": (i32, [vp, i32, i32, i32, vp, vp, vp, vp, i32, vp]),
    "snrse_ncsnpp_num_launch_groups": (i32, [vp, i32, i32, i32]),
    "snrse_ncsnpp_profile_forward": (i32, [vp, i32, i32, i32, vp, vp, vp, vp, i32, vp, i32, POINTER(i32), POINTER(f64), POINTER(f64), POINTER(f32), POINTER(i32)]),
    "snrse_ncsnpp_read_tap": (i32, [vp, i32, i32, i32, i32, vp, i64, POINTER(i64), vp]),
    "snrse_conv_nhwc": (i32, [vp, i32, i32, vp, i32, vp, i32, vp, vp, i32, vp, f32, vp, i32, i32, i32, i32, vp]),
    "snrse_conv_halo_set_debug": (None, [vp]),
    "snrse_gn_silu_conv3x3_nhwc": (i32, [vp, i32, vp, vp, f32, vp, i32, vp, i32, vp, vp, i32, vp, f32, vp, i32, i32, i32, vp, vp]),
    "snrse_conv3x3_nhwc_stats": (i32, [vp, i32, vp, i32, vp, i32, vp, vp, i32, vp, f32, vp, i32, i32, i32, vp, vp]),
    "snrse_groupnorm_workspace_bytes": (i64, [i32]),
    "snrse_groupnorm_nhwc": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, vp, vp]),
    "snrse_fir_nhwc": (i32, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "snrse_fir_f4": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "snrse_upfirdn2d": (i32, [vp, vp, vp, i64] + [i32] * 12 + [vp]),
    "snrse_attention_workspace_bytes": (i64, [i32, i32, i32]),
    "snrse_attention_nhwc": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    "snrse_snrnet_num_params": (i32, []),
    "snrse_snrnet_param_info": (i32, [i32, c_char_p, i32, POINTER(i64), POINTER(i64), POINTER(i32)]),
    "snrse_snrnet_param_shape": (i32, [i32, POINTER(i64), POINTER(i32)]),
    "snrse_snrnet_weight_bytes": (i64, []),
    "snrse_snrnet_workspace_bytes": (i64, [i32, i32]),
    "snrse_snrnet_forward": (i32, [vp, vp, vp, i32, i32, vp, vp]),
    "snrse_snrnet_forward_varlen": (i32, [vp, vp, vp, vp, i32, i32, vp, vp]),
}

# every symbol declared in include/snrse_b200_layers.h (the executor's launchers, for the layer tests); snrse_view
# arguments are passed by reference (ctypes.byref of a structure mirroring snrse_view)
LAYER_PROTOTYPES = {
    "snrse_dbg_conv": (i32, [vp, i32, vp, vp, i32, vp, vp, i32, vp, f32, vp, vp, vp, i32, vp]),
    "snrse_dbg_gn_stats": (i32, [vp, vp, vp]),
    "snrse_dbg_gn_finalize": (i32, [vp, i32, vp, i32, i32, i64, vp, vp, f32, vp, vp]),
    "snrse_dbg_gn_apply": (i32, [vp, vp, i32, vp, vp]),
    "snrse_dbg_fir": (i32, [vp, vp, i32, vp]),
    "snrse_dbg_fir_dual": (i32, [vp, vp, vp, i32, vp, vp]),
    "snrse_dbg_conv_out4": (i32, [vp, vp, vp, vp, vp, vp, i32, vp]),
    "snrse_dbg_pack_input": (i32, [vp, vp, vp, vp, i32, i64, vp]),
    "snrse_dbg_conv_in4": (i32, [vp, vp, vp, vp, vp]),
    "snrse_dbg_combine4": (i32, [vp, vp, vp, vp, vp, vp]),
    "snrse_dbg_temb": (i32, [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]),
    "snrse_dbg_final": (i32, [vp, vp, vp, vp, vp, vp, i32, i64, i32, vp]),
    "snrse_dbg_attention": (i32, [vp, vp, vp, vp, vp, i32, vp]),
}

# every symbol declared in include/snrse_b200_plans.h (the executor's convolution plans, for the plan tests)
PLAN_PROTOTYPES = {
    "snrse_ncsnpp_dbg_convs": (i32, [vp, i32, i32, i32, i32, i32, vp, i32, POINTER(i32)]),
    "snrse_dbg_conv_plan": (i32, [vp, i32, vp, vp, i32, vp, vp, vp, i32, vp]),
}


def load():
    """Load the shared library (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m snr_aligned_diffse_b200.build` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in {**PROTOTYPES, **LAYER_PROTOTYPES, **PLAN_PROTOTYPES}.items():
        # one flag per parameter makes a call with more arguments than the prototype a TypeError; a plain ctypes
        # function would pass the extra ones on, e.g. a stale argument list's pointer in place of the stream.
        # AttributeError if the ABI and the header drifted apart.
        proto = ctypes.CFUNCTYPE(res, *args)
        setattr(lib, name, proto((name, lib), tuple((1,) for _ in args)) if args else proto((name, lib)))
    _lib = lib
    return lib


def check(status, what=""):
    if status != 0:
        msg = load().snrse_last_error().decode(errors="replace")
        raise RuntimeError(f"libsnrse_b200 {what} failed (status {status}): {msg}")


_device_ok = False


def require_device():
    """Raise unless the current CUDA device is a B200-class (sm_100) GPU (checked once per process)."""
    global _device_ok
    if not _device_ok:
        check(load().snrse_device_check(), "device check")
        _device_ok = True


def ptr(t):
    """Device (or host) address of a torch tensor / None."""
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
