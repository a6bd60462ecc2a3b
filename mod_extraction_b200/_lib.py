"""ctypes binding of libmodfx.so (the C ABI declared in include/modfx.h).

The library is the product: there is no CPU or eager-PyTorch fallback.  If it has not been
built (``python -m mod_extraction_b200._build``) or no CUDA device is present, every op raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

from ._build import LIB_PATH as _DEFAULT_LIB_PATH

# MODFX_LIB points the loader at an alternative build of the same ABI (kernel experiments)
LIB_PATH = os.environ.get("MODFX_LIB", _DEFAULT_LIB_PATH)

c_f32p = ctypes.POINTER(ctypes.c_float)
c_i32p = ctypes.POINTER(ctypes.c_int32)


class ModfxParam(ctypes.Structure):
    """modfx_param: (B,) float32 device array or python-float scalar (fx.py:75-79)."""
    _fields_ = [("dev", ctypes.c_void_p), ("value", ctypes.c_double)]


class ModfxModSource(ctypes.Structure):
    _fields_ = [
        ("kind", ctypes.c_int32),
        ("mod", ctypes.c_void_p),
        ("mod_has_ch", ctypes.c_int32),
        ("n_lo", ctypes.c_int64),
        ("sr_lo", ctypes.c_float),
        ("lfo_freq", ctypes.c_void_p),
        ("lfo_phase", ctypes.c_void_p),
        ("lfo_shape", ctypes.c_void_p),
        ("lfo_exp", ctypes.c_void_p),
    ]


MOD_AUDIO_RATE, MOD_CONTROL_RATE, MOD_LFO = 0, 1, 2
CNN_FP32, CNN_TF32 = 0, 1      # modfx_cnn_precision
CNN_FP16 = 3                   # python-side tag only: modfx_cnn_conv_pool_prelu_f16_f32
CNN_TF32X3 = 2                 # python-side tag only: the split entry point modfx_cnn_conv_pool_prelu_tf32x3_f32

SHAPES = ["cos", "rect_cos", "inv_rect_cos", "tri", "saw", "rsaw", "sqr"]   # modfx_shape order
SHAPE_ID = {s: i for i, s in enumerate(SHAPES)}

_lib: Optional[ctypes.CDLL] = None

_vp = ctypes.c_void_p
_i32 = ctypes.c_int32
_i64 = ctypes.c_int64

_SIGNATURES = {
    "modfx_abi_version": ([], ctypes.c_int),
    "modfx_last_error": ([], ctypes.c_char_p),
    "modfx_device_count": ([], ctypes.c_int),
    "modfx_flanger_chorus_f32": ([_vp, _vp, _i32, _i32, _i64, _i32, _i32, ctypes.POINTER(ModfxModSource),
                                  ModfxParam, ModfxParam, ModfxParam, ModfxParam, ModfxParam, _vp, _i32, _vp],
                                 ctypes.c_int),
    "modfx_flanger_chorus_allpass_f32": ([_vp, _vp, _i32, _i32, _i64, _i32, _i32, ctypes.POINTER(ModfxModSource),
                                          ModfxParam, ModfxParam, ModfxParam, ModfxParam, ModfxParam, _vp, _i32, _vp],
                                         ctypes.c_int),
    "modfx_tremolo_f32": ([_vp, _vp, _i32, _i32, _i64, ctypes.POINTER(ModfxModSource), ModfxParam, _vp], ctypes.c_int),
    "modfx_lfo_f32": ([_vp, _i32, _i64, ctypes.c_float, _vp, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_lfo_window_f32": ([_vp, _i32, _i64, _i64, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_interp_linear_f32": ([_vp, _vp, _i64, _i64, _i64, _i32, _vp], ctypes.c_int),
    "modfx_find_corners_f32": ([_vp, _vp, _vp, _i64, _i64, _vp], ctypes.c_int),
    "modfx_lfo_sections_f32": ([_vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_stretch_sections_f32": ([_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_combined_lfo_workspace_bytes": ([_i32, _i64, _i32], _i64),
    "modfx_combined_lfo_f32": ([_vp, _i32, _i64, ctypes.c_float, _vp, _vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_smoothen_f32": ([_vp, _vp, _i64, _i64, _i32, _vp], ctypes.c_int),
    "modfx_stretch_corners_f32": ([_vp, _vp, _i64, _i64, _i32, _vp], ctypes.c_int),
    "modfx_check_mod_sig_f32": ([_vp, _vp, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _vp], ctypes.c_int),
    "modfx_logmel_f32": ([_vp, _vp, _i64, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, ctypes.c_float, _i32,
                          _i64, _i64, _vp, _i32, _vp],
                         ctypes.c_int),
    "modfx_specaugment_fill_f32": ([_vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, ctypes.c_float, _i32, _vp],
                                   ctypes.c_int),
    "modfx_cnn_layernorm_workspace_bytes": ([_i32, _i32, _i32, _i32], _i64),
    "modfx_cnn_layernorm_f32": ([_vp, _vp, _i32, _i32, _i32, _i32, _i32, ctypes.c_float, _i32, _vp, _vp], ctypes.c_int),
    "modfx_cnn_conv_pool_prelu_f32": ([_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp],
                                      ctypes.c_int),
    "modfx_cnn_conv_pool_prelu_tf32x3_f32": ([_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_cnn_conv_pool_prelu_f16_f32": ([_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_cnn_head_f32": ([_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp], ctypes.c_int),
    "modfx_cnn_train_workspace_bytes": ([_i32, _i32, _i32, _i32], _i64),
    "modfx_cnn_conv_pool_prelu_train_f32": ([_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp], ctypes.c_int),
    "modfx_cnn_conv_dgrad_tf32_f32": ([_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp], ctypes.c_int),
    "modfx_cnn_conv_wgrad_tf32_f32": ([_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp], ctypes.c_int),
    "modfx_cnn_pool_prelu_bwd_f32": ([_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp], ctypes.c_int),
    "modfx_cnn_layernorm_bwd_f32": ([_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, ctypes.c_float, _vp, _vp], ctypes.c_int),
    "modfx_cnn_head_bwd_f32": ([_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp], ctypes.c_int),
    "modfx_phaser_workspace_bytes": ([_i32, _i64], _i64),
    "modfx_phaser_f32": ([_vp, _vp, _i32, _i64, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp],
                         ctypes.c_int),
    "modfx_phaser_crop_f32": ([_vp, _i32, _vp, _vp, _i32, _i64, _i64, _vp, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32,
                               _vp, _vp], ctypes.c_int),
    "modfx_phaser_crop_packed_f32": ([_vp, _vp, _vp, _vp, _i32, _i64, _i64, _vp, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _vp,
                                      _i32, _vp, _vp], ctypes.c_int),
}


def exported_symbols():
    """Names every build of libmodfx.so must export (mirrors include/modfx.h)."""
    return sorted(_SIGNATURES)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if LIB_PATH == _DEFAULT_LIB_PATH and os.path.exists(LIB_PATH):
            from . import _build
            if not _build.is_current():     # built from other sources than the ones in this tree: never load it silently
                try:
                    _build.build()
                except Exception as exc:
                    raise RuntimeError(f"{LIB_PATH} was not built from the sources in this tree (content hash mismatch) "
                                       f"and could not be rebuilt: {exc}") from exc
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m mod_extraction_b200._build` "
                "(there is no CPU fallback for the modfx ops)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (argtypes, restype) in _SIGNATURES.items():
            fn = getattr(L, name)       # AttributeError here == header/library mismatch
            fn.argtypes = argtypes
            fn.restype = restype
        if L.modfx_abi_version() != 1:
            raise RuntimeError("libmodfx.so ABI version mismatch")
        _lib = L
    return _lib


def check(status: int) -> None:
    if status != 0:
        msg = lib().modfx_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"modfx error {status}: {msg}")
