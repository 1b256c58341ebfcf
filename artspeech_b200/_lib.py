"""ctypes binding of ``libartspeech_b200.so`` (the C ABI in ``include/artspeech_b200.h``).

There is deliberately no fallback: if the library is missing or an entry point fails the call
raises.  The oracle under ``oracle/`` is test infrastructure and is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

AS_F16, AS_BF16, AS_F32, AS_PCM16 = 0, 1, 2, 3
ACT_NONE, ACT_LRELU, ACT_RELU, ACT_TANH, ACT_SWISH, ACT_ABS = 0, 1, 2, 3, 4, 5

c_i32_p = C.POINTER(C.c_int32)
c_f32_p = C.POINTER(C.c_float)


class ConvParams(C.Structure):
    """Mirror of ``struct as_conv_params``."""
    _fields_ = [
        ("x", C.c_void_p), ("x_dtype", C.c_int32),
        ("B", C.c_int32), ("T", C.c_int32), ("F", C.c_int32), ("Cin", C.c_int32),
        ("x_ld", C.c_int64),
        ("w", C.c_void_p),
        ("ntaps", C.c_int32), ("CinP", C.c_int32), ("CoutP", C.c_int32), ("Cout", C.c_int32),
        ("tap_dt", c_i32_p), ("tap_df", c_i32_p),
        ("To", C.c_int32), ("Fo", C.c_int32),
        ("bias", C.c_void_p),
        ("res1", C.c_void_p), ("res1_dtype", C.c_int32), ("res1_ld", C.c_int64),
        ("res2", C.c_void_p), ("res2_dtype", C.c_int32), ("res2_ld", C.c_int64),
        ("out_scale", C.c_float),
        ("y_raw", C.c_void_p), ("y_raw_dtype", C.c_int32), ("y_raw_ld", C.c_int64),
        ("y_act", C.c_void_p), ("y_act_dtype", C.c_int32), ("y_act_ld", C.c_int64),
        ("act", C.c_int32), ("slope", C.c_float),
        ("lens", C.c_void_p),
        ("stats", C.c_void_p),
    ]


class ResblockPairParams(C.Structure):
    """Mirror of ``struct as_resblock_pair_params``."""
    _fields_ = [
        ("x", C.c_void_p), ("x_ld", C.c_int64), ("dtype", C.c_int32),
        ("B", C.c_int32), ("L", C.c_int32), ("C", C.c_int32), ("k", C.c_int32), ("dil", C.c_int32),
        ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
        ("slope", C.c_float),
        ("res2", C.c_void_p), ("res2_ld", C.c_int64), ("res3", C.c_void_p), ("res3_ld", C.c_int64),
        ("out_scale", C.c_float), ("out_act", C.c_int32), ("out_slope", C.c_float),
        ("y", C.c_void_p), ("y_ld", C.c_int64),
        ("lens", C.c_void_p),
    ]


class AsError(RuntimeError):
    pass


_lib = None

# name -> (restype, argtypes); every symbol declared in include/artspeech_b200.h
SIGNATURES = {
    "as_version": (C.c_int, []),
    "as_last_error": (C.c_char_p, []),
    "as_set_sm_limit": (C.c_int, [C.c_int32]),
    "as_mas_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "as_mas_maximum_path": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                      C.c_void_p]),
    "as_conv_tile_n": (C.c_int32, [C.c_int32]),
    "as_conv_igemm": (C.c_int, [C.POINTER(ConvParams), C.c_void_p]),
    "as_hifigan_resblock_pair": (C.c_int, [C.POINTER(ResblockPairParams), C.c_void_p]),
}


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Load (building in-tree first when needed) and return the ctypes handle."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path) or not _build.is_current():
        if not build_if_missing:
            raise AsError(f"{path} missing or stale; run `python -m artspeech_b200.build`")
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().as_last_error()
        raise AsError(f"{what} failed with status {rc}: {msg.decode() if msg else ''}")

# ---- memory-bound / small kernels -----------------------------------------------------------
_V, _I, _L, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float
SIGNATURES.update({
    "as_embed": (C.c_int, [_V, _V, _I, _I, _I, _I, _F, _V, _V, _V, _I, _V]),
    "as_layernorm": (C.c_int, [_V, _I, _L, _I, _I, _I, _V, _V, _F, _I, _F, _V, _V, _I, _L, _V, _I, _L, _V]),
    "as_relpos_attention": (C.c_int, [_V, _L, _V, _V, _I, _I, _I, _I, _I, _V, _V, _I, _L, _V]),
    "as_conformer_attention": (C.c_int, [_V, _V, _V, _L, _V, _V, _V, _I, _I, _I, _I, _V, _V, _I, _L, _V]),
    "as_instnorm_stats": (C.c_int, [_V, _I, _L, _I, _I, _I, _V, _F, _V, _V]),
    "as_adain_apply": (C.c_int, [_V, _I, _L, _I, _I, _I, _V, _V, _L, _F, _V, _V, _V, _V, _I, _L, _V]),
    "as_adain_norm_apply": (C.c_int, [_V, _I, _L, _I, _I, _I, _V, _L, _F, _F, _V, _V, _V, _V, _I, _L, _V, _V]),
    "as_repeat_rows": (C.c_int, [_V, _I, _L, _I, _I, _I, _I, _V, _V, _I, _L, _V]),
    "as_length_regulate": (C.c_int, [_V, _I, _L, _I, _I, _I, _V, _V, _I, _I, _V, _I, _L, _V, _V]),
    "as_round_durations": (C.c_int, [_V, _L, _I, _I, _V, _V, _V, _V]),
    "as_round_durations_scaled": (C.c_int, [_V, _L, _I, _I, _V, _V, _L, _V, _V, _V]),
    "as_prosody_apply": (C.c_int, [_V, _L, _V, _L, _V, _L, _I, _I, _V, _V, C.c_double, C.c_double, C.c_double,
                                   _V]),
    "as_conv_small": (C.c_int, [_V, _I, _L, _I, _I, _I, _I, _V, _V, _I, c_i32_p, c_i32_p, _I, _V,
                                _V, _I, _L, _V, _I, _L, _I, _F, _V]),
    "as_dwconv": (C.c_int, [_V, _I, _L, _I, _I, _I, _I, _I, _V, _V, _I, _I, _I, _I, _I, _I, _I, _I,
                            _V, _V, _I, _F, _V, _I, _L, _V]),
    "as_avgpool": (C.c_int, [_V, _I, _L, _I, _I, _I, _I, _I, _I, _V, _I, _L, _V]),
    "as_affine_act_maxpool": (C.c_int, [_V, _I, _L, _I, _I, _I, _I, _V, _V, _F, _I, _V, _I, _L, _V]),
    "as_global_avgpool": (C.c_int, [_V, _I, _L, _I, _I, _I, _I, _I, _F, _V, _I, _L, _V]),
    "as_bilstm": (C.c_int, [_V, _L, _V, _I, _I, _I, _V, _V, _I, _L, _V]),
    "as_lstm_onestep": (C.c_int, [_V, _L, _L, _I, _V, _I, _L, _V]),
    "as_log_norm": (C.c_int, [_V, _I, _I, _I, _V, _V]),
    "as_log_mel": (C.c_int, [_V, _L, _V, _I, _I, _V, _V, _V, _V, _I, _I, _I, _F, _F, _F, _V, _I, _V]),
    "as_transpose_cast": (C.c_int, [_V, _I, _V, _I, _I, _I, _I, _L, _I, _V, _V, _V, _V]),
    "as_mas_align": (C.c_int, [_V, _V, _V, _V, _V, _V, _I, _I, _I, _I, _V, C.c_size_t, _V]),
    "as_expand_tokens": (C.c_int, [_V, _V, _V, _I, _I, _I, _I, _V]),
    "as_resample_smem_bytes": (C.c_size_t, [_I, _I, _I, _I]),
    "as_resample_encode": (C.c_int, [_V, _L, _I, _I, _V, _V, _I, _I, _I, _I, _I, _I, _I, _V, _L, _I, _V, _V]),
    "as_resample_encode_gain": (C.c_int, [_V, _L, _I, _I, _V, _V, _I, _I, _I, _I, _I, _I, _I, _V, _L, _I, _V, _V,
                                          _V]),
    "as_loudness_workspace_bytes": (C.c_size_t, [_I, _L, _I]),
    "as_loudness_measure": (C.c_int, [_V, _L, _I, _L, _V, _I, C.POINTER(C.c_double), c_f32_p, C.c_double,
                                      C.c_double, _V, C.c_size_t, _V, _V, _V, _V, _V]),
})
SIGNATURES.update({
    "as_watermark_embed": (C.c_int, [_V, _L, _I, _I, _V, _V, _F, _V, _L, _V]),
    "as_audio_decode": (C.c_int, [_V, _L, _I, _I, _I, _V, _L, _V]),
    "as_audio_to_mono": (C.c_int, [_V, _L, _I, _I, _I, _I, _V, _V, _L, _V]),
    "as_trim_workspace_bytes": (C.c_size_t, [_I, _I]),
    "as_trim_bounds": (C.c_int, [_V, _L, _I, _I, _V, C.c_double, _V, C.c_size_t, _V, _V]),
    "as_log_mel_span": (C.c_int, [_V, _L, _V, _V, _I, _I, _V, _V, _V, _V, _I, _I, _I, _F, _F, _F, _V, _I, _V]),
    "as_watermark_workspace_bytes": (C.c_size_t, [_I, _I]),
    "as_watermark_detect": (C.c_int, [_V, _L, _I, _I, _V, _V, _V, _F, _V, C.c_size_t, _V, _V, _V, _V, _V]),
    "as_denoise_workspace_bytes": (C.c_size_t, [_I, _I]),
    "as_denoise": (C.c_int, [_V, _L, _I, _I, _V, C.c_double, _V, _V, _V, C.c_double, C.c_double, C.c_double,
                             C.c_double, _V, C.c_size_t, _V, _L, _V]),
})
