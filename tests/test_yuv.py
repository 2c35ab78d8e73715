"""YUV 4:2:0 frame ingest without a GPU: the oracle's restatement of cv2.cvtColor(COLOR_YUV2RGB_NV12 / _I420), the even
rectangle the batch-1 tracker uploads, and the C ABI's refusal of a null handle.  The device side is tests/test_gpu_yuv.py."""
import ctypes as C

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from oracle import vt_oracle as O
from oracle import yuv420 as Y
from test_tracking_edges import CASES, FRAMES, _case_boxes

CV = {"nv12": cv2.COLOR_YUV2RGB_NV12, "i420": cv2.COLOR_YUV2RGB_I420}


def exhaustive_yuv420(format):
    """A 4096 x 4096 frame holding every (Y, U, V) triple once: each of the 2^16 (U, V) pairs owns 64 2x2 blocks, which
    carry its 256 Y values."""
    H = W = 4096
    bw, bh = W // 2, H // 2
    nb = bw * bh                                                      # 2^22 blocks
    u = np.repeat(np.arange(256, dtype=np.uint8), 256 * 64)           # per block
    v = np.tile(np.repeat(np.arange(256, dtype=np.uint8), 64), 256)
    yb = np.tile(np.arange(256, dtype=np.uint8).reshape(64, 4), (nb // 64, 1))            # [nb, 4]: the block's 2x2 Y values
    Y = yb.reshape(bh, bw, 2, 2).transpose(0, 2, 1, 3).reshape(H, W)
    if format == "nv12":
        chroma = np.stack([u, v], -1).reshape(bh, W)
    else:
        chroma = np.concatenate([u, v]).reshape(bh, W)
    return np.ascontiguousarray(np.concatenate([Y, chroma], 0))


def random_yuv420(H, W, format, seed):
    return Y.synth_yuv420(1, H, W, seed=seed, format=format)[0]


@pytest.mark.parametrize("format", ["nv12", "i420"])
def test_exhaustive_frame_covers_every_triple(format):
    f = exhaustive_yuv420(format)
    H = 4096
    Y = f[:H].astype(np.int64)
    if format == "nv12":
        U, V = f[H:, 0::2], f[H:, 1::2]
    else:
        U, V = f[H:].reshape(-1)[: H * H // 4].reshape(H // 2, H // 2), f[H:].reshape(-1)[H * H // 4:].reshape(H // 2, H // 2)
    up = lambda a: np.repeat(np.repeat(a.astype(np.int64), 2, 0), 2, 1)
    key = (Y << 16) | (up(U) << 8) | up(V)
    assert np.unique(key).size == 1 << 24


@pytest.mark.parametrize("format", ["nv12", "i420"])
def test_oracle_matches_opencv_on_every_triple(format):
    f = exhaustive_yuv420(format)
    got = Y.yuv420_to_rgb(f, format)
    want = cv2.cvtColor(f, CV[format])
    assert got.shape == want.shape == (4096, 4096, 3)
    assert np.array_equal(got, want), int((got != want).any(-1).sum())


@pytest.mark.parametrize("format", ["nv12", "i420"])
@pytest.mark.parametrize("hw", [(2, 2), (2, 1282), (720, 1280), (1080, 1920)])
def test_oracle_matches_opencv_on_random_frames(format, hw):
    f = random_yuv420(*hw, format, seed=hw[0] + hw[1])
    assert f.shape == (hw[0] * 3 // 2, hw[1])
    assert np.array_equal(Y.yuv420_to_rgb(f, format), cv2.cvtColor(f, CV[format]))


EVEN_CASES = [nm for nm in CASES if CASES[nm][0] in ("hd", "small", "uhd")]


@pytest.mark.parametrize("name", EVEN_CASES)
def test_even_rect_is_aligned_inside_and_covers_crop_rect(name):
    from vittracker_b200.sequences import crop_rect
    from vittracker_b200.tracker import even_rect
    fr, tbox, sbox = _case_boxes(name)
    H, W = FRAMES[fr]
    assert H % 2 == 0 and W % 2 == 0
    for box, factor in ((tbox, O.TEMPLATE_FACTOR), (sbox, O.SEARCH_FACTOR)):
        rect = crop_rect(box, factor, H, W)
        assert rect is not None, name
        ya, yb, xa, xb = even_rect(rect, H, W)
        assert all(v % 2 == 0 for v in (ya, yb, xa, xb)), (name, rect)
        assert 0 <= ya < yb <= H and 0 <= xa < xb <= W, (name, rect)
        assert ya <= rect[0] and yb >= rect[1] and xa <= rect[2] and xb >= rect[3], (name, rect)
        assert ya >= rect[0] - 1 and yb <= rect[1] + 1 and xa >= rect[2] - 1 and xb <= rect[3] + 1, (name, rect)


def test_yuv_entry_points_refuse_a_null_handle():
    from vittracker_b200 import _lib
    lib = _lib.load()
    buf = (C.c_uint8 * 64)()
    off = (C.c_int64 * 1)()
    hw = (C.c_int32 * 2)(2, 2)
    assert lib.vt_yuv420_to_rgb(None, 1, buf, off, hw, buf, off, 1, None) == -1
    assert lib.vt_upload_yuv420_rect(None, 1, buf, 2, 2, 0, 2, 0, 2, buf, buf, buf, None) == -1


def test_frame_format_names_and_shapes_are_checked():
    from vittracker_b200.engine import yuv420_frame_hw, yuv_format
    assert yuv_format("nv12") == 1 and yuv_format("i420") == 2
    with pytest.raises(ValueError):
        yuv_format("yuyv")
    assert yuv420_frame_hw(np.zeros((1080, 1280), np.uint8)) == (720, 1280)
    for shape in [(1081, 1280), (1080, 1279), (10, 4), (0, 4)]:
        with pytest.raises(ValueError):
            yuv420_frame_hw(np.zeros(shape, np.uint8))
    with pytest.raises(ValueError):
        yuv420_frame_hw(np.zeros((1080, 1280, 3), np.uint8))
    with pytest.raises(ValueError):
        yuv420_frame_hw(np.zeros((1080, 1280), np.float32))
