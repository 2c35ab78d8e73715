"""Several targets per YUV surface without a GPU: the C ABI's declaration of vt_yuv420_crops_to_surface_rgb against its binding, the
exported symbol and the refusal of a null handle.  The device side is tests/test_gpu_shared_surfaces.py."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = "vt_yuv420_crops_to_surface_rgb"


def test_header_declaration_matches_the_binding():
    from vittracker_b200 import _lib
    header = open(os.path.join(ROOT, "include", "vittrack_b200.h")).read()
    decl = re.search(r"\bint\s+" + NAME + r"\s*\(([^)]*)\)\s*;", header)
    assert decl is not None
    params = [p.strip() for p in decl.group(1).split(",")]
    res, args = _lib.SIGNATURES[NAME]
    assert res is C.c_int and len(args) == len(params) == 15
    for p, a in zip(params, args):                         # pointers are void*, scalars keep their width
        if "*" in p or p.startswith("VtHandle"):
            assert a is C.c_void_p, p
        elif p.startswith("int32_t"):
            assert a is C.c_int32, p
        elif p.startswith("double"):
            assert a is C.c_double, p
        else:
            raise AssertionError(p)


def test_the_symbol_is_exported():
    from vittracker_b200 import _lib
    assert hasattr(_lib.load(), NAME)


def test_a_null_handle_is_refused():
    from vittracker_b200 import _lib
    lib = _lib.load()
    planes = (C.c_uint64 * 3)()
    pitch = (C.c_int32 * 2)(2, 2)
    hw = (C.c_int32 * 2)(2, 2)
    surf = (C.c_int32 * 1)(0)
    box = (C.c_double * 4)(0, 0, 1, 1)
    buf = (C.c_uint8 * 64)()
    off = (C.c_int64 * 1)()
    assert getattr(lib, NAME)(None, 1, planes, pitch, hw, 1, surf, box, None, 2.0, 0, 1, buf, off, None) == -1
    assert getattr(lib, NAME)(None, 1, planes, pitch, hw, 1, surf, None, None, 4.0, 0, 1, buf, off, None) == -1
