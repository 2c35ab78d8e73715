"""CPU oracle for YUV 4:2:0 frame ingest (NV12 / I420).  TEST INFRASTRUCTURE ONLY, like ``vt_oracle``: nothing under
``vittracker_b200/`` imports it.

``yuv420_to_rgb`` restates cv2.cvtColor(COLOR_YUV2RGB_NV12 / COLOR_YUV2RGB_I420); ``synth_yuv420`` generates seeded YUV
frames for the tests and tools/e2e_yuv.py."""
from __future__ import annotations

import numpy as np

from .vt_oracle import synth_frames


def synth_yuv420(n: int, H: int = 720, W: int = 1280, seed: int = 0, format: str = "nv12", smooth: bool = False) -> np.ndarray:
    """uint8 YUV 4:2:0 frames (n, H*3/2, W) as cv2.cvtColor takes them: Y from channel 0 of ``synth_frames``, U / V from
    channels 1 / 2 at every second row and column."""
    rgb = synth_frames(n, H, W, seed=seed, smooth=smooth)
    U, V = rgb[:, ::2, ::2, 1], rgb[:, ::2, ::2, 2]
    if format == "nv12":
        chroma = np.stack([U, V], -1).reshape(n, H // 2, W)
    elif format == "i420":
        chroma = np.concatenate([U.reshape(n, -1), V.reshape(n, -1)], 1).reshape(n, H // 2, W)
    else:
        raise ValueError(format)
    return np.ascontiguousarray(np.concatenate([rgb[..., 0], chroma], 1))


def yuv420_to_rgb(frame: np.ndarray, format: str) -> np.ndarray:
    """cv2.cvtColor(frame, COLOR_YUV2RGB_NV12 / COLOR_YUV2RGB_I420), restated: OpenCV's integer arithmetic with 20 fractional
    bits (modules/imgproc/src/color_yuv.simd.hpp, OpenCV 4.13.0), one (U, V) sample per 2x2 luma block.  ``frame``: uint8
    (H*3/2, W), H and W even.  Returns uint8 (H, W, 3)."""
    rows, W = frame.shape
    H = rows * 2 // 3
    assert rows == H * 3 // 2 and H % 2 == 0 and W % 2 == 0, frame.shape
    Y = frame[:H].astype(np.int64)
    c = frame[H:]
    if format == "nv12":
        U, V = c[:, 0::2], c[:, 1::2]
    elif format == "i420":
        flat = c.reshape(-1)
        U, V = flat[: H * W // 4].reshape(H // 2, W // 2), flat[H * W // 4:].reshape(H // 2, W // 2)
    else:
        raise ValueError(format)
    up = lambda a: np.repeat(np.repeat(a.astype(np.int64) - 128, 2, 0), 2, 1)
    u, v = up(U), up(V)
    y = np.maximum(0, Y - 16) * 1220542
    sat = lambda a: np.clip(a >> 20, 0, 255).astype(np.uint8)
    return np.stack([sat(y + (1 << 19) + 1673527 * v), sat(y + (1 << 19) - 852492 * v - 409993 * u),
                     sat(y + (1 << 19) + 2116026 * u)], -1)
