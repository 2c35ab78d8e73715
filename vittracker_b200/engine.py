"""Engine: one libvittrack_b200 handle bound to one GPU.  PyTorch is used only for device memory
and streams; every computation is a C-ABI call into hand-written sm_100a kernels."""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib

TEMPLATE_TOKENS, SEARCH_TOKENS = 64, 256


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


YUV_FORMATS = {"nv12": 1, "i420": 2}          # VT_FRAME_NV12, VT_FRAME_I420


def yuv_format(name: str) -> int:
    if name not in YUV_FORMATS:
        raise ValueError(f"unknown YUV format {name!r}: expected one of {sorted(YUV_FORMATS)}")
    return YUV_FORMATS[name]


def yuv420_frame_hw(frame) -> Tuple[int, int]:
    """(H, W) of a YUV 4:2:0 frame laid out as cv2.cvtColor takes it: uint8 (H*3/2) x W with H and W even."""
    if frame.dtype not in (np.uint8, torch.uint8) or frame.ndim != 2:
        raise ValueError("a YUV 4:2:0 frame must be a 2-D uint8 array of shape (H*3/2, W)")
    rows, W = int(frame.shape[0]), int(frame.shape[1])
    if rows % 3 or (rows * 2 // 3) % 2 or W % 2 or rows == 0 or W == 0:
        raise ValueError(f"YUV 4:2:0 frame of shape {tuple(frame.shape)}: expected (H*3/2, W) with H and W even and positive")
    return rows * 2 // 3, W


def hann2d_window(sz: int = 16) -> torch.Tensor:
    """Cosine window the reference builds once per tracker (lib/test/utils/hann.py:6-16,
    centered=True): w[k] = 0.5 (1 - cos(2 pi k / (sz + 1))), k = 1..sz, outer product -> (1,1,sz,sz)."""
    w = 0.5 * (1 - torch.cos((2 * math.pi / (sz + 1)) * torch.arange(1, sz + 1).float()))
    return w.reshape(1, 1, -1, 1) * w.reshape(1, 1, 1, -1)


class Engine:
    def __init__(self, cfg, max_tracks: int = 1, chunk_tracks: int = 0, device: Optional[int] = None,
                 blocks_impl: str = "tcgen05", depth: int = 3):
        if not torch.cuda.is_available():
            raise RuntimeError("vittracker_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.cfg = cfg
        impl = {"simt": _lib.VT_BLOCKS_SIMT_FP32, "tcgen05": _lib.VT_BLOCKS_TCGEN05, "tcgen05_3term": _lib.VT_BLOCKS_TCGEN05_3TERM}[blocks_impl]
        c = _lib.VtConfig(
            embed_dim=int(cfg.MODEL.BACKBONE.CHANNELS), num_heads=int(cfg.MODEL.BACKBONE.HEADS), depth=int(depth),
            mlp_ratio=4, head_channels=int(cfg.MODEL.HEAD.NUM_CHANNELS), stride=int(cfg.MODEL.BACKBONE.STRIDE),
            template_size=int(cfg.TEST.TEMPLATE_SIZE), search_size=int(cfg.TEST.SEARCH_SIZE),
            template_factor=float(cfg.TEST.TEMPLATE_FACTOR), search_factor=float(cfg.TEST.SEARCH_FACTOR),
            max_tracks=int(max_tracks), chunk_tracks=int(chunk_tracks), device=self.device_index, blocks_impl=impl)
        if str(cfg.MODEL.HEAD.TYPE) != "CENTER":
            raise NotImplementedError("only the CENTER head is implemented (the shipped experiment uses it)")
        self.handle = C.c_void_p()
        _lib.check(None, self.lib.vt_create(C.byref(c), C.byref(self.handle)))
        self.max_tracks = int(max_tracks)
        self.template_size, self.search_size = c.template_size, c.search_size
        self.depth, self.C = int(depth), c.embed_dim
        self.weights_loaded = False

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.vt_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        _lib.check(self.handle, rc)

    @property
    def launch_count(self) -> int:
        return int(self.lib.vt_launch_count(self.handle))

    def profile(self, enable: bool) -> None:
        self._check(self.lib.vt_profile_enable(self.handle, 1 if enable else 0))

    def profile_read(self) -> dict:
        """Per-stage device time (ms), launches and items since the last read (syncs on the events)."""
        ms = (C.c_double * 4)()
        nl = (C.c_int64 * 4)()
        ni = (C.c_int64 * 4)()
        self._check(self.lib.vt_profile_read(self.handle, ms, nl, ni))
        return {name: {"ms": ms[i], "launches": int(nl[i]), "items": int(ni[i])}
                for i, name in enumerate(("crop", "stem", "blocks", "head"))}

    # ------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict: Dict[str, torch.Tensor], strict: bool = False) -> Tuple[list, list]:
        """Hand every tensor to the library under its reference key; unknown keys are skipped as
        ``load_state_dict(strict=False)`` does (lib/test/tracker/vit_dist.py:25)."""
        unexpected = []
        for name, t in state_dict.items():
            if not torch.is_tensor(t):
                continue
            if not t.is_floating_point():
                if name.endswith("num_batches_tracked"):
                    continue
                unexpected.append(name)
                continue
            a = t.detach().to("cpu", torch.float32).contiguous()
            shape = (C.c_int64 * max(1, a.dim()))(*a.shape)
            rc = self.lib.vt_set_tensor(self.handle, name.encode(), C.c_void_p(a.data_ptr()), shape, a.dim())
            if rc == -3:
                msg = self.lib.vt_last_error(self.handle).decode()
                if "unknown tensor" in msg:
                    unexpected.append(name)
                    continue
            self._check(rc)
        win = hann2d_window(self.search_size // 16).contiguous()
        shape = (C.c_int64 * 4)(*win.shape)
        self._check(self.lib.vt_set_tensor(self.handle, b"tracker.output_window", C.c_void_p(win.data_ptr()), shape, 4))
        if strict and unexpected:
            raise RuntimeError(f"unexpected keys: {unexpected}")
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_finalize_weights(self.handle, self._stream()))
        self.weights_loaded = True
        return [], unexpected

    # ------------------------------------------------------------------------------------------
    def crop_normalize(self, frames: torch.Tensor, frame_offsets: torch.Tensor, frame_hw: torch.Tensor,
                       boxes: torch.Tensor, factor: float, out_size: int, want_u8: bool = False,
                       want_mask: bool = False):
        """sample_target + Preprocessor for n (frame, box) pairs.  frames: uint8 device buffer;
        frame_offsets int64 [n]; frame_hw int32 [n,2]; boxes float64 [n,4].  Returns a dict."""
        n = boxes.shape[0]
        dev = self.device
        assert frames.dtype == torch.uint8 and frame_offsets.dtype == torch.int64 and frame_hw.dtype == torch.int32
        assert boxes.dtype == torch.float64 and boxes.is_contiguous()
        out = torch.empty((n, 3, out_size, out_size), dtype=torch.float32, device=dev)
        u8 = torch.empty((n, out_size, out_size, 3), dtype=torch.uint8, device=dev) if want_u8 else None
        mask = torch.empty((n, out_size, out_size), dtype=torch.uint8, device=dev) if want_mask else None
        rf = torch.empty((n,), dtype=torch.float64, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            self._check(self.lib.vt_crop_normalize(self.handle, _ptr(frames), _ptr(frame_offsets), _ptr(frame_hw), _ptr(boxes),
                                                   float(factor), int(out_size), int(n), _ptr(out), _ptr(u8), _ptr(mask),
                                                   _ptr(rf), _ptr(status), self._stream()))
        return {"tensors": out, "u8": u8, "mask": mask, "resize_factor": rf, "status": status}

    def forward(self, z: torch.Tensor, x: torch.Tensor, taps: bool = False):
        """OstrackDist.forward(z, x): returns the reference's output dict (+ 'taps' when asked)."""
        n = z.shape[0]
        dev = self.device
        assert z.shape[1:] == (3, self.template_size, self.template_size) and x.shape == (n, 3, self.search_size, self.search_size)
        z = z.to(dev, torch.float32).contiguous()
        x = x.to(dev, torch.float32).contiguous()
        F = self.search_size // 16
        pred = torch.empty((n, 1, 4), dtype=torch.float32, device=dev)
        score = torch.empty((n, 1, F, F), dtype=torch.float32, device=dev)
        size = torch.empty((n, 2, F, F), dtype=torch.float32, device=dev)
        off = torch.empty((n, 2, F, F), dtype=torch.float32, device=dev)
        tp = torch.zeros((self.depth + 2, n, TEMPLATE_TOKENS + SEARCH_TOKENS, self.C), dtype=torch.float32, device=dev) if taps else None
        with torch.cuda.device(dev):
            self._check(self.lib.vt_forward(self.handle, _ptr(z), _ptr(x), int(n), _ptr(pred), _ptr(score), _ptr(size),
                                            _ptr(off), _ptr(tp), self._stream()))
        out = {"pred_boxes": pred, "score_map": score, "size_map": size, "offset_map": off}
        if taps:
            out["taps"] = tp
        return out

    def cal_bbox(self, score: torch.Tensor, size_map: torch.Tensor, offset_map: torch.Tensor) -> torch.Tensor:
        n = score.shape[0]
        dev = self.device
        score = score.to(dev, torch.float32).contiguous()
        size_map = size_map.to(dev, torch.float32).contiguous()
        offset_map = offset_map.to(dev, torch.float32).contiguous()
        boxes = torch.empty((n, 4), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            self._check(self.lib.vt_cal_bbox(self.handle, _ptr(score), _ptr(size_map), _ptr(offset_map), int(n), _ptr(boxes), self._stream()))
        return boxes

    # ------------------------------------------------------------------------------------------
    def yuv420_to_rgb(self, src: torch.Tensor, src_offsets: torch.Tensor, frame_hw: torch.Tensor, dst: torch.Tensor,
                      dst_offsets: torch.Tensor, format: str) -> torch.Tensor:
        """cv2.cvtColor(COLOR_YUV2RGB_NV12 / _I420) of n frames, bit for bit, device -> device: the (H*3/2) x W YUV frame at byte
        ``src_offsets[i]`` of ``src`` becomes the H x W x 3 frame at byte ``dst_offsets[i]`` of ``dst``.  uint8 buffers, int64
        offsets [n], int32 frame_hw [n, 2] (even), all on this engine's device.  Returns ``dst``."""
        fmt = yuv_format(format)
        for t, dt in ((src, torch.uint8), (dst, torch.uint8), (src_offsets, torch.int64), (dst_offsets, torch.int64), (frame_hw, torch.int32)):
            if t.dtype != dt or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"yuv420_to_rgb: expected a contiguous {dt} tensor on {self.device}")
        n = int(src_offsets.shape[0])
        if dst_offsets.shape != (n,) or frame_hw.shape != (n, 2):
            raise ValueError("yuv420_to_rgb: src_offsets [n], dst_offsets [n] and frame_hw [n, 2] required")
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_yuv420_to_rgb(self.handle, fmt, _ptr(src), _ptr(src_offsets), _ptr(frame_hw), _ptr(dst),
                                                  _ptr(dst_offsets), n, self._stream()))
        return dst

    def upload_yuv420_rect(self, format: str, image: np.ndarray, y0: int, y1: int, x0: int, x1: int, staging: torch.Tensor,
                           staging_dev: torch.Tensor, frame_rgb: torch.Tensor) -> None:
        """Rows [y0, y1) x columns [x0, x1) of the host YUV frame ``image`` ((H*3/2) x W uint8), widened to even bounds, into the
        H x W x 3 device frame ``frame_rgb`` through ``staging`` (pinned) and ``staging_dev`` (vt_upload_yuv420_rect)."""
        fmt = yuv_format(format)
        H, W = yuv420_frame_hw(image)
        image = np.ascontiguousarray(image)
        need = H * W * 3 // 2
        if staging.numel() < need or staging_dev.numel() < need or frame_rgb.numel() < H * W * 3:
            raise ValueError("upload_yuv420_rect: staging buffers need (H*3/2) x W bytes and frame_rgb H x W x 3")
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_upload_yuv420_rect(self.handle, fmt, image.ctypes.data, H, W, int(y0), int(y1), int(x0), int(x1),
                                                       _ptr(staging), _ptr(staging_dev), _ptr(frame_rgb), self._stream()))

    # ------------------------------------------------------------------------------------------
    def tracks_init(self, frames, frame_offsets, frame_hw, boxes, first: int = 0) -> torch.Tensor:
        n = boxes.shape[0]
        assert boxes.dtype == torch.float64 and boxes.is_contiguous() and boxes.device == self.device
        status = torch.empty((n,), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_tracks_init(self.handle, _ptr(frames), _ptr(frame_offsets), _ptr(frame_hw), _ptr(boxes),
                                                int(first), int(n), _ptr(status), self._stream()))
        return status

    def tracks_step(self, frames, frame_offsets, frame_hw, first: int = 0, n: Optional[int] = None,
                    out_boxes: Optional[torch.Tensor] = None, out_detail: Optional[torch.Tensor] = None,
                    update_state: bool = True, detail: bool = False):
        n = frame_offsets.shape[0] if n is None else n
        if out_boxes is None:
            out_boxes = torch.empty((n, 5), dtype=torch.float64, device=self.device)
        if detail and out_detail is None:
            out_detail = torch.empty((n, 8), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_tracks_step(self.handle, _ptr(frames), _ptr(frame_offsets), _ptr(frame_hw), int(first), int(n),
                                                _ptr(out_boxes), _ptr(out_detail), 1 if update_state else 0, self._stream()))
        return (out_boxes, out_detail) if detail else out_boxes

    def tracks_get_state(self, first: int = 0, n: Optional[int] = None) -> torch.Tensor:
        n = self.max_tracks - first if n is None else n
        out = torch.empty((n, 4), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_tracks_get_state(self.handle, _ptr(out), int(first), int(n), self._stream()))
        return out

    def tracks_set_state(self, boxes: torch.Tensor, first: int = 0) -> None:
        assert boxes.dtype == torch.float64 and boxes.is_contiguous() and boxes.device == self.device
        with torch.cuda.device(self.device):
            self._check(self.lib.vt_tracks_set_state(self.handle, _ptr(boxes), int(first), int(boxes.shape[0]), self._stream()))

    def tracks_last_maps(self, first: int, n: int):
        dev = self.device
        score = torch.empty((n, 1, 16, 16), dtype=torch.float32, device=dev)
        size = torch.empty((n, 2, 16, 16), dtype=torch.float32, device=dev)
        off = torch.empty((n, 2, 16, 16), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            self._check(self.lib.vt_tracks_last_maps(self.handle, int(first), int(n), _ptr(score), _ptr(size), _ptr(off), self._stream()))
        return {"score_map": score, "size_map": size, "offset_map": off}
