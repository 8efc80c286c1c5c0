"""ctypes binding of libmogstn.so (include/mogstn.h).  No fallback: if the library is missing or a call
fails, this raises."""
from __future__ import annotations

import ctypes
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
# MOG_SO: load another build of the library, e.g. to compare two builds in one session (tools/kbench.py, tools/dbg_bwd.py)
SO_PATH = os.environ.get("MOG_SO") or os.path.join(_PKG, "libmogstn.so")

MOG_ASR_MAX_STEPS = 16
MOG_ASR_MAX_COUNTS = 8
MOG_ASR_NUM_COMPONENTS = 6
ABI_VERSION = 1

_c_float_p = ctypes.c_void_p  # device pointers travel as integers
_i64, _int, _f32, _vp = ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_void_p
_f64 = ctypes.c_double


class AsrConfig(ctypes.Structure):
    """mirror of mog_asr_config"""
    _fields_ = [("canvas_size", _f32), ("max_steps", _int), ("num_counts", _int),
                ("counts", _int * MOG_ASR_MAX_COUNTS),
                ("gamma_num", _f32), ("gamma_margin", _f32), ("gamma_elem", _f32), ("gamma_bbox", _f32),
                ("gamma_size", _f32), ("gamma_area", _f32), ("size_min", _f32), ("size_max", _f32)]


# symbol -> argtypes; every symbol include/mogstn.h declares
SIGNATURES = {
    "mog_version": [],
    "mog_last_error_string": [ctypes.c_char_p, ctypes.c_size_t],
    "mog_stn_forward": [_vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _vp],
    "mog_stn_corners": [_vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_backward": [_vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _vp],
    "mog_stn_fwd_bwd_host": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _i64, _vp, ctypes.c_size_t,
                             ctypes.POINTER(ctypes.c_void_p), _int],
    "mog_stn_host_workspace_bytes": [_i64, _int, _int, _int, _int, _int, _int],
    "mog_stn_batch_fwd_bwd_host": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _i64, _vp, ctypes.c_size_t,
                                   ctypes.POINTER(ctypes.c_void_p), _int],
    "mog_stn_batch_host_workspace_bytes": [_i64, _int, _int, _int, _int, _int, _int, _int],
    "mog_stn_write_composite_forward": [_vp, _vp, _vp, _vp, _f32, _vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_write_composite_backward": [_vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_read_sxy_forward": [_vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_read_sxy_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_write_composite_sxy_forward": [_vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_write_composite_sxy_backward": [_vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _vp],
    "mog_stn_write_composite_host": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _i64, _vp, ctypes.c_size_t,
                                     ctypes.POINTER(ctypes.c_void_p), _int],
    "mog_stn_write_composite_host_workspace_bytes": [_i64, _int, _int, _int, _int, _int, _int],
    "mog_bce_recon_forward": [_vp, _vp, _vp, _vp, _i64, _int, _vp],
    "mog_bce_recon_backward": [_vp, _vp, _vp, _vp, _i64, _int, _vp],
    "mog_air_gauss_sample_forward": [_vp, _vp, _vp, _vp, _vp, _i64, _int, _vp],
    "mog_air_gauss_sample_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp],
    "mog_air_thetas_forward": [_vp, _vp, _vp, _vp, _i64, _vp],
    "mog_air_thetas_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "mog_air_zpres_forward": [_vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "mog_air_zpres_backward": [_vp, _vp, _vp, _f32, _vp, _i64, _vp],
    "mog_air_lstm_pointwise_forward": [_vp, _vp, _vp, _vp, _vp, _i64, _int, _vp],
    "mog_air_lstm_pointwise_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp],
    "mog_air_kl_forward": [_vp] * 13 + [_i64, _int, _int, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp],
    "mog_air_kl_backward": [_vp] * 13 + [_i64, _int, _int, _f32, _f32, _f32, _f32, _f32] + [_vp] * 12 + [_vp],
    "mog_detection_eval": [_vp] * 6 + [_i64, _int, _int, _f64] + [_vp] * 5 + [_vp],
    "mog_air_head_forward": [_vp] * 11 + [_i64, _int, _int, _int, _int, _int] + [_vp] * 4 + [_vp],
    "mog_air_head_backward": [_vp] * 15 + [_i64, _int, _int, _int, _int, _int] + [_vp] * 6 + [_vp],
    "mog_air_bias_act_forward": [_vp, _vp, _vp, _i64, _int, _int, _vp],
    "mog_air_bias_act_backward": [_vp, _vp, _vp, _i64, _int, _vp],
    "mog_air_bias_gauss_forward": [_vp] * 7 + [_i64, _int, _vp],
    "mog_air_bias_gauss_backward": [_vp] * 6 + [_i64, _int, _vp],
    "mog_synth_place": [ctypes.c_uint64, _i64, _i64, _int, _int, _vp, _int, _int, _int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _vp],
    "mog_synth_place_pixels": [ctypes.c_uint64, _i64, _i64, _int, _int, _vp, _int, _int, _int, _int, _int, _int,
                               _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "mog_synth_place_rotated": [ctypes.c_uint64, _i64, _i64, _int, _int, _vp, _int, _int, _int, _int, _int, _int, _int,
                                _vp, _int, _int, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp],
    "mog_asr_reg_colsum": [_vp, _vp, _i64, _int, _vp],
    "mog_asr_reg_forward": [_vp, _vp, _vp, _vp, _f32, _i64, _int, ctypes.POINTER(AsrConfig), _vp, _vp, _vp, _vp],
    "mog_asr_reg_backward": [_vp, _vp, _vp, _vp, _f32, _vp, _vp, _i64, _int, ctypes.POINTER(AsrConfig), _vp, _vp, _vp, _vp],
}

_lib = None
_lock = threading.Lock()


def load() -> ctypes.CDLL:
    """Load libmogstn.so from the package directory (built by mog_asr_b200.build).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(SO_PATH):
                raise RuntimeError(
                    f"{SO_PATH} is missing: build it with `python -m mog_asr_b200.build` "
                    "(there is no CPU or PyTorch fallback for this path)")
            L = ctypes.CDLL(SO_PATH)
            for name, argtypes in SIGNATURES.items():
                fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
                fn.argtypes = argtypes
                fn.restype = ctypes.c_size_t if name.endswith("host_workspace_bytes") else ctypes.c_int
            v = L.mog_version()
            if v != ABI_VERSION:
                raise RuntimeError(f"libmogstn ABI version {v} != expected {ABI_VERSION}")
            _lib = L
    return _lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(512)
    load().mog_last_error_string(buf, 512)
    return buf.value.decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        kind = "bad argument" if rc < 0 else "CUDA error"
        raise RuntimeError(f"{what} failed ({kind} {rc}): {last_error()}")
