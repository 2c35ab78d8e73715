"""ctypes binding of libvittrack_b200.so (the C ABI declared in include/vittrack_b200.h).

There is no fallback: if the library is missing it is built with nvcc; if that fails, or no CUDA
device is present when a handle is created, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

VT_OK = 0
VT_BLOCKS_SIMT_FP32 = 0
VT_BLOCKS_TCGEN05 = 1
VT_BLOCKS_TCGEN05_3TERM = 2
VT_TRACK_OK, VT_TRACK_TOO_SMALL, VT_TRACK_OUT_OF_DOMAIN, VT_TRACK_NUMERIC_RANGE = 0, 1, 2, 3

STATUS_NAMES = {0: "VT_OK", -1: "VT_ERR_INVALID_ARG", -2: "VT_ERR_CUDA", -3: "VT_ERR_WEIGHTS", -4: "VT_ERR_STATE",
                -5: "VT_ERR_UNSUPPORTED", -6: "VT_ERR_NO_DEVICE"}


class VtConfig(C.Structure):
    _fields_ = [("embed_dim", C.c_int32), ("num_heads", C.c_int32), ("depth", C.c_int32), ("mlp_ratio", C.c_int32),
                ("head_channels", C.c_int32), ("stride", C.c_int32), ("template_size", C.c_int32),
                ("search_size", C.c_int32), ("template_factor", C.c_double), ("search_factor", C.c_double),
                ("max_tracks", C.c_int32), ("chunk_tracks", C.c_int32), ("device", C.c_int32),
                ("blocks_impl", C.c_int32)]


class VtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{STATUS_NAMES.get(code, code)}: {msg}")
        self.code = code


_P = C.c_void_p
# name -> (restype, argtypes); mirrors include/vittrack_b200.h one to one
SIGNATURES = {
    "vt_abi_version": (C.c_int, []),
    "vt_last_error": (C.c_char_p, [_P]),
    "vt_create": (C.c_int, [C.POINTER(VtConfig), C.POINTER(_P)]),
    "vt_destroy": (C.c_int, [_P]),
    "vt_set_tensor": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int32]),
    "vt_finalize_weights": (C.c_int, [_P, _P]),
    "vt_crop_normalize": (C.c_int, [_P, _P, _P, _P, _P, C.c_double, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "vt_forward": (C.c_int, [_P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "vt_cal_bbox": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P]),
    "vt_tracks_init": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P]),
    "vt_tracks_step": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, C.c_int32, _P]),
    "vt_tracks_get_state": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P]),
    "vt_tracks_set_state": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P]),
    "vt_tracks_last_maps": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "vt_launch_count": (C.c_int64, [_P]),
    "vt_profile_enable": (C.c_int, [_P, C.c_int32]),
    "vt_profile_read": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "vt_upload_frame_rect": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "vt_debug_pending": (C.c_int, [_P, C.POINTER(C.c_int32), C.c_int32]),
    "vt_yuv420_to_rgb": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, C.c_int32, _P]),
    "vt_upload_yuv420_rect": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        _P, _P, _P, _P]),
}

_lib = None
_lock = threading.Lock()


def lib_path() -> str:
    return _build.LIB_PATH


def load():
    """Load (building first if needed) the shared library and bind every exported symbol."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        # always go through build(): a no-op when the stamp matches the sources and flags, a rebuild when the library is stale
        # (an old .so after edits to csrc/ would otherwise be measured silently).  Without nvcc an existing library is used as is.
        try:
            path = _build.build()
        except _build.NvccMissing:
            path = _build.LIB_PATH
            if not os.path.isfile(path):
                raise
            if not _build.is_fresh():
                import warnings
                warnings.warn(f"{path} is older than its sources and nvcc is unavailable: loading the stale library")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)        # AttributeError if the .so does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        if lib.vt_abi_version() != 1:
            raise RuntimeError(f"{path}: ABI version {lib.vt_abi_version()} != 1 (stale build? run python -m vittracker_b200.build --force)")
        _lib = lib
        return lib


def check(handle, rc: int) -> None:
    if rc != VT_OK:
        msg = load().vt_last_error(handle)
        raise VtError(rc, msg.decode() if msg else "")
