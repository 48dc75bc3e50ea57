"""ctypes binding of liblbic_b200.so (the C ABI in include/lbic.h).

The product path has no fallback: if the shared library is missing (run `python
__graft_entry__.py build` or `build.py`) or no sm_100 GPU is present, calls raise."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "liblbic_b200.so")
_lib = None


class LbicConfig(ctypes.Structure):
    _fields_ = [("block_size", ctypes.c_int), ("ks", ctypes.c_int * 4), ("n", ctypes.c_int), ("m", ctypes.c_int)]


class LbicTensorDesc(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.c_void_p), ("ndim", ctypes.c_int),
                ("shape", ctypes.c_int64 * 4)]


class LbicDebugLayerArgs(ctypes.Structure):
    _fields_ = [("mode", ctypes.c_int), ("core", ctypes.c_int), ("force_bn", ctypes.c_int), ("R", ctypes.c_int),
                ("cout", ctypes.c_int), ("nseg", ctypes.c_int), ("K", ctypes.c_int * 2), ("A", ctypes.c_void_p * 2),
                ("W", ctypes.c_void_p * 2), ("bias", ctypes.c_void_p), ("aux", ctypes.c_void_p), ("ld_aux", ctypes.c_int),
                ("acc_scale", ctypes.c_float), ("M", ctypes.c_int), ("scale_table", ctypes.c_void_p),
                ("no_clamp", ctypes.c_int), ("out_f32", ctypes.c_void_p), ("out_hi", ctypes.c_void_p),
                ("out_lo", ctypes.c_void_p), ("out_idx", ctypes.c_void_p)]


LBIC_OPT_GEMM_CORE = 1
LBIC_OPT_FORCE_BN = 3
LBIC_OPT_WS = 6
LBIC_OPT_PAIR = 8
LBIC_OPT_DEC_THREAD_ROWS = 9
LBIC_OPT_ENC_THREAD_STREAMS = 10
LBIC_OPT_FLOW = 11
LBIC_OPT_FLOW_MIN_ROWS = 12
LBIC_OPT_HOST_BANDS = 14
LBIC_OPT_WAVE = 15
LBIC_OPT_ENC_BLOCK_STREAMS = 17
LBIC_OPT_WAVE_DEC_MAX_ROWS = 18
LBIC_OPT_WAVE_BN = 19
LBIC_OPT_DEC_SMEM_WARP = 20
LBIC_OPT_CHECK_SATURATION = 26
LBIC_OPT_FLOW_PAIR_MIN_ROWS = 25
LBIC_OPT_WAVE_MAX_ROWS = 16
LBIC_OPT_PDL = 7

# every symbol include/lbic.h declares: (restype, argtypes)
_vp, _i, _sz, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t, ctypes.c_int64
PROTOTYPES = {
    "lbic_last_error": (ctypes.c_char_p, []),
    "lbic_version": (ctypes.c_char_p, []),
    "lbic_create": (_i, [ctypes.POINTER(LbicConfig), _i, ctypes.POINTER(_vp)]),
    "lbic_destroy": (None, [_vp]),
    "lbic_set_option": (_i, [_vp, _i, _i]),
    "lbic_load_weights": (_i, [_vp, ctypes.POINTER(LbicTensorDesc), _i, _vp]),
    "lbic_build_tables": (_i, [_vp, _vp, _i, ctypes.c_double, _vp]),
    "lbic_set_tables": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "lbic_get_tables": (_i, [_vp, ctypes.POINTER(_i), ctypes.POINTER(_i), _vp, _vp, _vp]),
    "lbic_encode": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp, _i, _vp]),
    "lbic_decode": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _vp, _vp, _i, _vp]),
    "lbic_encode_mixed": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _i, _vp]),
    "lbic_decode_mixed": (_i, [_vp, _vp, _vp, _sz, _i, _vp, _vp, _vp, _vp, _i, _vp]),
    "lbic_validate": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "lbic_encode_host": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp, _i]),
    "lbic_decode_host": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _vp, _i]),
    "lbic_check_errors": (_i, [_vp, _vp]),
    "lbic_encode_images_u8_host": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp, _i]),
    "lbic_decode_images_u8_host": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _vp, _i]),
    "lbic_encode_images_u8_host_mixed": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp, _i]),
    "lbic_decode_images_u8_host_mixed": (_i, [_vp, _vp, _vp, _sz, _i, _vp, _vp, _vp, _i]),
    "lbic_image_metrics": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp]),
    "lbic_load_postpm_weights": (_i, [_vp, ctypes.POINTER(LbicTensorDesc), _i, _vp]),
    "lbic_postprocess": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "lbic_band_begin": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "lbic_band_zhat": (_vp, [_vp]),
    "lbic_band_step": (_i, [_vp, _i, _i, _i, _vp]),
    "lbic_band_end": (_i, [_vp, _i, _i, _vp, _vp, _sz, _vp, _vp]),
    "lbic_stream_bound": (_sz, [_vp, _i, _i, _i]),
    "lbic_space_to_depth": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "lbic_depth_to_space": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "lbic_rans_encode": (_i, [_vp, _vp, _vp, _i, _i64, _vp, _sz, _vp, _vp]),
    "lbic_rans_decode": (_i, [_vp, _vp, _vp, _sz, _vp, _i, _i64, _vp, _vp]),
    "lbic_debug_gemm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "lbic_debug_layer": (_i, [_vp, ctypes.POINTER(LbicDebugLayerArgs), _vp]),
    "lbic_debug_selfinfo": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _vp]),
    "lbic_debug_scale_index": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "lbic_debug_rans_encode": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _sz, _vp, _vp]),
    "lbic_debug_rans_decode_steps": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "lbic_debug_compact_tables": (_i, [_vp, ctypes.POINTER(_i), _vp, _vp, _vp]),
    "lbic_debug_gemm_bench": (_i, [_vp, _i, _i, _i, _i, _i, ctypes.POINTER(ctypes.c_double)]),
    "lbic_saturation_count": (_i, [_vp, _vp, ctypes.POINTER(ctypes.c_int64), _i]),
    "lbic_launch_count": (_i64, [_vp]),
    "lbic_set_profiling": (_i, [_vp, _i]),
    "lbic_get_profile": (_i, [_vp, ctypes.POINTER(_i64), ctypes.POINTER(ctypes.c_double),
                              ctypes.POINTER(ctypes.c_double)]),
    "lbic_forward": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "lbic_get_layer_profile": (_i, [_vp, _i, ctypes.POINTER(_i64), ctypes.POINTER(ctypes.c_double),
                                    ctypes.POINTER(ctypes.c_double)]),
}


def lib():
    """Loads liblbic_b200.so; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} not found: build the CUDA extension first (python __graft_entry__.py build). "
                "lbic_b200 has no CPU fallback.")
        L = ctypes.CDLL(SO_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc: int):
    """Maps a negative lbic_status to a Python exception (STATE -> ValueError like the reference's
    _check_cdf_size, entropy_layers_cai.py:185-204; everything else RuntimeError)."""
    if rc == 0:
        return
    msg = lib().lbic_last_error().decode(errors="replace")
    if rc == -3:
        raise ValueError(msg)
    raise RuntimeError(f"lbic error {rc}: {msg}")
