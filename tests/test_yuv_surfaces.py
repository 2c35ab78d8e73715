"""Device-resident YUV surfaces without a GPU: what ``YuvSurfaces`` refuses before it touches the device, and the C ABI's
refusal of a null handle.  The device side is tests/test_gpu_yuv_surfaces.py."""
import ctypes as C

import pytest
import torch

from vittracker_b200.batched import YuvSurfaces


def planes(H, W, fmt, dtype=torch.uint8):
    y = torch.zeros((H, W), dtype=dtype)
    if fmt == "nv12":
        return y, torch.zeros((H // 2, W), dtype=dtype)
    return y, torch.zeros((H // 2, W // 2), dtype=dtype), torch.zeros((H // 2, W // 2), dtype=dtype)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("hw", [(7, 8), (8, 7), (0, 8), (1, 8)])
def test_odd_or_tiny_sizes_are_refused(fmt, hw):
    H, W = hw
    y = torch.zeros((H, W), dtype=torch.uint8)
    c = torch.zeros((max(H // 2, 1), W), dtype=torch.uint8)
    rest = (c,) if fmt == "nv12" else (c[:, : W // 2], c[:, : W // 2])
    with pytest.raises(ValueError):
        YuvSurfaces(fmt, y, *rest)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_a_pitch_below_the_row_width_is_refused(fmt):
    p = list(planes(8, 8, fmt))
    buf = torch.zeros(256, dtype=torch.uint8)
    p[0] = buf.as_strided((8, 8), (6, 1))                     # rows overlap
    with pytest.raises(ValueError, match="pitch"):
        YuvSurfaces(fmt, *p)
    p = list(planes(8, 8, fmt))
    p[1] = buf.as_strided(tuple(p[1].shape), (p[1].shape[1] - 1, 1))
    with pytest.raises(ValueError, match="pitch"):
        YuvSurfaces(fmt, *p)
    p = list(planes(8, 8, fmt))
    p[0] = buf.as_strided((8, 8), (1, 8))                      # columns not adjacent
    with pytest.raises(ValueError):
        YuvSurfaces(fmt, *p)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_a_wrong_dtype_is_refused(fmt):
    for k in range(3 if fmt == "i420" else 2):
        p = list(planes(8, 8, fmt))
        p[k] = p[k].to(torch.int16)
        with pytest.raises(ValueError, match="uint8"):
            YuvSurfaces(fmt, *p)


def test_chroma_shapes_that_do_not_match_are_refused():
    y = torch.zeros((8, 8), dtype=torch.uint8)
    for c in (torch.zeros((4, 4), dtype=torch.uint8), torch.zeros((8, 8), dtype=torch.uint8), torch.zeros((3, 8), dtype=torch.uint8)):
        with pytest.raises(ValueError):
            YuvSurfaces("nv12", y, c)
    q = torch.zeros((4, 4), dtype=torch.uint8)
    for u, v in ((torch.zeros((4, 8), dtype=torch.uint8), q), (q, torch.zeros((4, 3), dtype=torch.uint8)), (q, torch.zeros((2, 4), dtype=torch.uint8))):
        with pytest.raises(ValueError):
            YuvSurfaces("i420", y, u, v)
    with pytest.raises(ValueError):                            # I420 without V, NV12 with a V plane
        YuvSurfaces("i420", y, q)
    with pytest.raises(ValueError):
        YuvSurfaces("nv12", y, torch.zeros((4, 8), dtype=torch.uint8), q)
    buf = torch.zeros(64, dtype=torch.uint8)
    with pytest.raises(ValueError, match="share one pitch"):
        YuvSurfaces("i420", y, buf.as_strided((4, 4), (4, 1)), buf.as_strided((4, 4), (6, 1)))
    with pytest.raises(ValueError):                            # as many chroma planes as luma planes
        YuvSurfaces("nv12", torch.zeros((2, 8, 8), dtype=torch.uint8), torch.zeros((3, 4, 8), dtype=torch.uint8))
    with pytest.raises(ValueError):
        YuvSurfaces("yuyv", y, torch.zeros((4, 8), dtype=torch.uint8))


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_well_formed_host_planes_are_refused_for_not_being_on_the_device(fmt):
    with pytest.raises(ValueError, match="CUDA"):
        YuvSurfaces(fmt, *planes(8, 8, fmt))


def test_from_frames_checks_the_surface_layout():
    with pytest.raises(ValueError):                            # 13 rows is no (H*3/2) x W frame
        YuvSurfaces.from_frames(torch.zeros((2, 13, 8), dtype=torch.uint8), "nv12")
    with pytest.raises(ValueError):                            # chroma beyond the surface
        YuvSurfaces.from_frames(torch.zeros((2, 12, 8), dtype=torch.uint8), "nv12", height=8, surface_rows=10)
    with pytest.raises(ValueError):                            # surface rows below the picture height
        YuvSurfaces.from_frames(torch.zeros((2, 12, 8), dtype=torch.uint8), "i420", height=8, surface_rows=6)
    with pytest.raises(ValueError):
        YuvSurfaces.from_frames(torch.zeros((2, 12, 8), dtype=torch.float32), "nv12")
    with pytest.raises(ValueError, match="CUDA"):              # a well-formed layout gets as far as the device check
        YuvSurfaces.from_frames(torch.zeros((2, 12, 8), dtype=torch.uint8), "i420")


def test_crop_entry_point_refuses_a_null_handle():
    from vittracker_b200 import _lib
    lib = _lib.load()
    planes_ = (C.c_uint64 * 3)()
    pitch = (C.c_int32 * 2)(2, 2)
    hw = (C.c_int32 * 2)(2, 2)
    box = (C.c_double * 4)(0, 0, 1, 1)
    buf = (C.c_uint8 * 64)()
    off = (C.c_int64 * 1)()
    assert lib.vt_yuv420_crop_to_rgb(None, 1, planes_, pitch, hw, box, 2.0, 0, 1, buf, off, None) == -1
    assert lib.vt_yuv420_crop_to_rgb(None, 1, planes_, pitch, hw, None, 4.0, 0, 1, buf, off, None) == -1
