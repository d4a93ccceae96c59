"""ctypes binding of libfear_b200.so (the C ABI declared in include/fear_b200.h).

There is no fallback: if the shared object is missing or a call fails, a RuntimeError carrying
``fear_last_error()`` is raised.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

import numpy as np

from .build import LIB_PATH


class FearBox(ctypes.Structure):
    _fields_ = [
        ("x", c_double), ("y", c_double), ("w", c_double), ("h", c_double),
        ("score", c_float), ("row", c_int32), ("col", c_int32), ("flat", c_int32),
    ]


BOX_DTYPE = np.dtype(
    [("x", "<f8"), ("y", "<f8"), ("w", "<f8"), ("h", "<f8"), ("score", "<f4"), ("row", "<i4"), ("col", "<i4"),
     ("flat", "<i4")]
)
assert BOX_DTYPE.itemsize == ctypes.sizeof(FearBox) == 48


class FearFrame(ctypes.Structure):
    _fields_ = [("data", c_uint64), ("h", c_int32), ("w", c_int32)]


FRAME_DTYPE = np.dtype([("data", "<u8"), ("h", "<i4"), ("w", "<i4")])
assert FRAME_DTYPE.itemsize == ctypes.sizeof(FearFrame) == 16


class FearTrack(ctypes.Structure):
    _fields_ = [(name, c_int32) for name in ("x", "y", "w", "h", "cx", "cy", "cw", "ch", "pad_r", "pad_g", "pad_b",
                                             "reserved")]


TRACK_DTYPE = np.dtype([(name, "<i4") for name, _ in FearTrack._fields_])
assert TRACK_DTYPE.itemsize == ctypes.sizeof(FearTrack) == 48

_SIGNATURES = {
    # name: (restype, argtypes)
    "fear_init": (c_int, [c_int]),
    "fear_abi_version": (c_int, []),
    "fear_last_error": (c_char_p, []),
    "fear_weight_count": (c_int, []),
    "fear_weight_name": (c_char_p, [c_int]),
    "fear_weight_numel": (c_int64, [c_int]),
    "fear_pack_weights": (c_int, [c_void_p, POINTER(c_uint64), c_int, POINTER(c_void_p)]),
    "fear_reserve": (c_int, [c_void_p, c_int]),
    "fear_free": (None, [c_void_p]),
    "fear_get_features": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "fear_backbone": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "fear_head": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "fear_head_update": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "fear_track": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "fear_track_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "fear_get_features_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "fear_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "fear_crop_resize_u8": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "fear_track_crops_u8": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_void_p]),
    "fear_track_advance": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "fear_decode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "fear_corr_concat_f32": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "fear_corr_concat_workspace_bytes": (c_size_t, [c_int, c_int]),
    "fear_corr_concat_ws_f32": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "fear_corr_nhwc_f32": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "fear_debug_backbone_prefix": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "fear_debug_head_tensor": (c_int, [c_void_p, c_char_p, c_int, c_void_p, c_void_p]),
    "fear_set_option": (c_int, [c_void_p, c_char_p, c_char_p]),
    "fear_launch_count": (c_int64, [c_void_p]),
    "fear_generation": (c_int64, [c_void_p]),
    "fear_profile": (c_int, [c_void_p, c_int]),
    "fear_stage_count": (c_int, []),
    "fear_stage_name": (c_char_p, [c_int]),
    "fear_stage_ms": (c_int, [c_void_p, c_int, POINTER(c_float), POINTER(c_int64)]),
}

_lib = None
_inited_devices = set()


def exported_symbols():
    return sorted(_SIGNATURES)


def load() -> ctypes.CDLL:
    """dlopen the library (no device needed) and attach signatures."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m feartracker_b200.build` "
                "(there is no CPU / PyTorch fallback for the FEAR hot path)"
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export it
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def last_error() -> str:
    return load().fear_last_error().decode()


def check(code: int, what: str) -> None:
    if code != 0:
        raise RuntimeError(f"{what} failed ({code}): {last_error()}")


def init(device: int = 0) -> ctypes.CDLL:
    """Initialise the library's per-device state (once per device; several devices per process are fine).
    ``fear_init`` makes ``device`` current while a handle is packed; the caller's device is restored here."""
    lib = load()
    if device not in _inited_devices:
        check(lib.fear_init(device), "fear_init")
        _inited_devices.add(device)
    return lib


def weight_table():
    lib = load()
    return [(lib.fear_weight_name(i).decode(), int(lib.fear_weight_numel(i))) for i in range(lib.fear_weight_count())]


def stage_names():
    lib = load()
    return [lib.fear_stage_name(i).decode() for i in range(lib.fear_stage_count())]
