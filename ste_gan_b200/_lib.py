"""ctypes binding of libstegan_b200.so (include/stegan_b200.h).

The product path has NO fallback: if the shared library is missing or a call fails the
caller gets an exception.  `load()` builds the library in-tree when it is absent and nvcc
is available (the authoring container / `__graft_entry__.build()`); on a GPU box the
prebuilt .so travels with the repo snapshot.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libstegan_b200.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_TANH = 0, 1, 2, 3
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05 = 0, 1, 2
PACK_UNFOLD = 1
MAX_TAPS = 48


class StgConv(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "dtype", "engine", "n_samples", "phases", "t_src", "t_dst", "c_src", "c_dst", "groups", "k", "dilation",
        "stride", "pad", "transposed", "pair_sum", "post_shift", "mask_mode", "act", "dup_rows", "out_f32", "w_fwd_pack")] + [
        (n, C.c_void_p) for n in ("src", "w", "bias", "add_pre", "mask", "add_post", "y_raw", "y_act")]


class StgWgrad(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "dtype", "engine", "n_samples", "phases", "t_in", "t_out", "c_in", "c_out", "groups", "k", "dilation",
        "stride", "pad")] + [(n, C.c_void_p) for n in ("x", "dy", "dw", "dbias")]


class StgFoldItem(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("v", "g", "wf", "wd", "scale", "dw", "dv", "dg")] + [
        (n, C.c_int32) for n in ("c_out", "cin_g", "k", "groups", "pg", "flags", "dw_ld", "dw_span", "row0", "tile0")]


class StgL1Item(C.Structure):
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("da", C.c_void_p), ("n", C.c_int64)]


class StgMseItem(C.Structure):
    _fields_ = [("x", C.c_void_p), ("dx", C.c_void_p), ("n", C.c_int64), ("target", C.c_float), ("slot", C.c_int32)]


MAX_LOSS_ITEMS = 32
_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float
_SIGS = {
    "stg_conv": [C.POINTER(StgConv), _P],
    "stg_conv_masked": [C.POINTER(StgConv), _P, C.c_int32, _P],
    "stg_conv_wgrad": [C.POINTER(StgWgrad), _P],
    "stg_conv_tc_supported": [C.POINTER(StgConv)],
    "stg_conv_route": [C.POINTER(StgConv)],
    "stg_wgrad_route": [C.POINTER(StgWgrad)],
    "stg_wgrad_tc_supported": [C.POINTER(StgWgrad)],
    "stg_weightnorm_fold": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P],
    "stg_weightnorm_fold_bwd": [_P, _I, _I, _P, _P, _I, _I, _I, _I, _P, _P, _I, _P],
    "stg_wgrad_layout": [C.POINTER(StgWgrad), C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "stg_spectralnorm_fold": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "stg_spectralnorm_fold_bwd": [_P, _I, _I, _P, _P, _P, _P, _I, _I, _I, _I, _P, _I, _P, _P],
    "stg_tc_pack_groups": [_I, _I, _I],
    "stg_l1_mean_multi": [_P, _I, _I, _P, _F, _P],
    "stg_mse_const_multi": [_P, _I, _I, _I, _P, _F, _P],
    "stg_weightnorm_fold_multi": [_P, _I, _I, _I, _I, _P],
    "stg_weightnorm_fold_bwd_multi": [_P, _I, _I, _I, _P],
    "stg_weightnorm_fold_bwd_range": [_P, _I, _I, _I, _I, _P],
    "stg_debug_set_trace": [_P],
    "stg_debug_rowshift": [_P, _P, _I, _I, _I, _P, _P],
    "stg_debug_row_classes": [_I, _P],
    "stg_debug_group_mma": [_P, _P, _I, _I, _P, _P],
    "stg_debug_conv_plan": [_P, _P],
    "stg_debug_tma_bw": [_P, C.c_longlong, _I, _I, _I, _I, _I, _P, _P],
    "stg_unfold": [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "stg_unfold_bwd": [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "stg_period_first_layer": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, C.c_float, _P, _P],
    "stg_embed_concat": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "stg_embed_concat_bwd": [_P, _P, _I, _I, _I, _I, _I, _P, _P],
    "stg_reflect_pad_right": [_P, _I, _I, _I, _I, _I, _P, _P],
    "stg_reflect_pad_right_bwd": [_P, _I, _I, _I, _I, _I, _P, _P],
    "stg_avgpool4": [_P, _I, _I, _I, _P, _P],
    "stg_avgpool4_bwd": [_P, _I, _I, _I, _P, _P],
    "stg_cast": [_P, _I, _P, _I, _L, _P],
    "stg_act_bwd": [_P, _P, _I, _L, _I, _P, _P],
    "stg_pair_sum_rows": [_P, _L, _I, _I, _P, _P],
    "stg_relu_rows": [_P, _I, _L, _I, _I, _P, _P],
    "stg_axpy_f32": [_P, _P, _I, _F, _L, _P],
    "stg_td_loss": [_P, _P, _I, _I, _I, _P, C.POINTER(C.c_float), _P, _P, _P],
    "stg_td_loss_ex": [_P, _P, _I, _I, _I, _I, C.POINTER(C.c_int), C.POINTER(C.c_int), _I, _I, _P, C.POINTER(C.c_float), _P, _P, _P, _P],
    "stg_td_scores": [_P, _P, _I, _I, _I, _P, C.c_int32, _I, C.POINTER(C.c_int), C.POINTER(C.c_int), _I, _I, _P, _P, _P],
    "stg_td_features": [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P],
    "stg_frame_stats": [_P, _I, _I, _I, _I, _I, _I, _P, _P, _P],
    "stg_window_signal": [_P, _I, _I, _I, _I, _I, _I, _P, _P],
    "stg_average_filter": [_P, _L, _I, _I, _I, _P, _P],
    "stg_mse_const": [_P, _I, _L, _F, _P, _F, _P, _I, _P],
    "stg_l1_mean": [_P, _P, _I, _L, _P, _F, _P, _P],
    "stg_layernorm_fwd": [_P, _I, _P, _P, _I, _I, _F, _P, _P, _P],
    "stg_layernorm_bwd": [_P, _P, _I, _P, _P, _I, _I, _P, _P],
    "stg_relattn_fwd": [_P, _I, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P],
    "stg_relattn_bwd": [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P, _P],
    "stg_relattn_dense_supported": [_I, _I, _I],
    "stg_relattn_band_fwd": [_P, _I, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P],
    "stg_relattn_band_bwd": [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P],
    "stg_relattn_fwd_masked": [_P, _I, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P],
    "stg_relattn_band_fwd_masked": [_P, _I, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P],
    "stg_encoder_losses": [_P, _P, _P, _P, _I, _I, _I, _P, _F, _F, _P, _P, _I, _P],
    "stg_encoder_scores": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P],
    "stg_adamw": [_P, _P, _P, _P, _L, _F, _P, _F, _F, _F, _F, _P, _F, _P, _I, _P],
}
EXPORTS = sorted(list(_SIGS) + ["stg_strerror", "stg_last_cuda_error", "stg_version", "stg_launch_count", "stg_set_sm_limit",
                                   "stg_debug_ingest_bytes"])

_lib = None


class StgError(RuntimeError):
    pass


def load(build_if_missing: bool = True):
    """Load (once) and return the ctypes library object.  Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise StgError(f"{LIB_PATH} is missing; run `python -m ste_gan_b200.build`")
        from . import build as _b
        _b.build()
    import torch  # noqa: F401  (loads libcudart.so.12 so the library binds to the same runtime)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, argtypes in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.stg_strerror.argtypes = [C.c_int]
    lib.stg_strerror.restype = C.c_char_p
    lib.stg_last_cuda_error.argtypes = []
    lib.stg_last_cuda_error.restype = C.c_char_p
    lib.stg_version.argtypes = []
    lib.stg_version.restype = C.c_int
    lib.stg_set_sm_limit.argtypes = [C.c_int]
    lib.stg_set_sm_limit.restype = None
    lib.stg_debug_ingest_bytes.argtypes = [C.c_int]
    lib.stg_debug_ingest_bytes.restype = C.c_double
    lib.stg_launch_count.argtypes = []
    lib.stg_launch_count.restype = C.c_ulonglong
    _lib = lib
    return lib


def check(code: int, what: str = "") -> None:
    if code != 0:
        lib = load()
        msg = lib.stg_strerror(code).decode()
        if code == -2:
            msg += ": " + lib.stg_last_cuda_error().decode()
        raise StgError(f"{what}: {msg} (code {code})")
