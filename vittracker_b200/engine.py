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


def tensor_ptr(t: Optional[torch.Tensor], name: str, dtype: torch.dtype, device: torch.device, shape: Optional[tuple] = None,
               align: int = 1, optional: bool = False) -> C.c_void_p:
    """The address a C-ABI call takes for ``t``, once ``t`` is what the call reads there: a contiguous ``dtype`` tensor on ``device``,
    of exactly ``shape`` when one is given (a per-item array is [n, ...]), at an address that is a multiple of ``align`` bytes.
    ``None`` passes NULL where the call takes it (``optional``).  Anything else raises ValueError, before the call."""
    if t is None and optional:
        return C.c_void_p(0)
    if (not torch.is_tensor(t) or t.dtype != dtype or t.device != device or not t.is_contiguous()
            or (shape is not None and t.shape != shape) or t.data_ptr() % align):
        got = f"{t.dtype} {tuple(t.shape)} on {t.device}" if torch.is_tensor(t) else type(t).__name__
        raise ValueError(f"{name}: expected a contiguous {dtype} tensor{'' if shape is None else f' of shape {tuple(shape)}'} on {device}"
                         f"{f', {align}-byte aligned' if align > 1 else ''}; got {got}")
    return C.c_void_p(t.data_ptr())


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

    def _call(self, name: str, *args) -> None:
        """``name``(handle, *args, stream) on this engine's device and its current stream; VtError for a failed status."""
        with torch.cuda.device(self.device):
            self._check(getattr(self.lib, name)(self.handle, *args, self._stream()))

    def _frames(self, frames, frame_offsets, frame_hw, n: int) -> tuple:
        """The frame arguments of a crop: uint8 frames, int64 frame_offsets [n] (bytes), int32 frame_hw [n, 2]."""
        dev = self.device
        return (tensor_ptr(frames, "frames", torch.uint8, dev), tensor_ptr(frame_offsets, "frame_offsets", torch.int64, dev, (n,)),
                tensor_ptr(frame_hw, "frame_hw", torch.int32, dev, (n, 2)))

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
        self._call("vt_finalize_weights")
        self.weights_loaded = True
        return [], unexpected

    # ------------------------------------------------------------------------------------------
    def crop_normalize(self, frames: torch.Tensor, frame_offsets: torch.Tensor, frame_hw: torch.Tensor,
                       boxes: torch.Tensor, factor: float, out_size: int, want_u8: bool = False,
                       want_mask: bool = False):
        """sample_target + Preprocessor for n (frame, box) pairs.  frames: uint8 device buffer;
        frame_offsets int64 [n]; frame_hw int32 [n,2]; boxes float64 [n,4].  Returns a dict."""
        n = int(boxes.shape[0])
        dev = self.device
        out = torch.empty((n, 3, out_size, out_size), dtype=torch.float32, device=dev)
        u8 = torch.empty((n, out_size, out_size, 3), dtype=torch.uint8, device=dev) if want_u8 else None
        mask = torch.empty((n, out_size, out_size), dtype=torch.uint8, device=dev) if want_mask else None
        rf = torch.empty((n,), dtype=torch.float64, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)
        self._call("vt_crop_normalize", *self._frames(frames, frame_offsets, frame_hw, n),
                   tensor_ptr(boxes, "boxes", torch.float64, dev, (n, 4)), float(factor), int(out_size), n, _ptr(out), _ptr(u8), _ptr(mask),
                   _ptr(rf), _ptr(status))
        return {"tensors": out, "u8": u8, "mask": mask, "resize_factor": rf, "status": status}

    def forward(self, z: torch.Tensor, x: torch.Tensor, taps: bool = False):
        """OstrackDist.forward(z, x): returns the reference's output dict (+ 'taps' when asked)."""
        n = int(z.shape[0])
        dev = self.device
        z = z.to(dev, torch.float32).contiguous()
        x = x.to(dev, torch.float32).contiguous()
        T, S = self.template_size, self.search_size
        F = S // 16
        pred = torch.empty((n, 1, 4), dtype=torch.float32, device=dev)
        score = torch.empty((n, 1, F, F), dtype=torch.float32, device=dev)
        size = torch.empty((n, 2, F, F), dtype=torch.float32, device=dev)
        off = torch.empty((n, 2, F, F), dtype=torch.float32, device=dev)
        tp = torch.zeros((self.depth + 2, n, TEMPLATE_TOKENS + SEARCH_TOKENS, self.C), dtype=torch.float32, device=dev) if taps else None
        self._call("vt_forward", tensor_ptr(z, "z", torch.float32, dev, (n, 3, T, T)), tensor_ptr(x, "x", torch.float32, dev, (n, 3, S, S)), n,
                   _ptr(pred), _ptr(score), _ptr(size), _ptr(off), _ptr(tp))
        out = {"pred_boxes": pred, "score_map": score, "size_map": size, "offset_map": off}
        if taps:
            out["taps"] = tp
        return out

    def cal_bbox(self, score: torch.Tensor, size_map: torch.Tensor, offset_map: torch.Tensor) -> torch.Tensor:
        n = int(score.shape[0])
        dev = self.device
        F = self.search_size // 16
        score, size_map, offset_map = (t.to(dev, torch.float32).contiguous() for t in (score, size_map, offset_map))
        boxes = torch.empty((n, 4), dtype=torch.float32, device=dev)
        self._call("vt_cal_bbox", tensor_ptr(score, "score", torch.float32, dev, (n, 1, F, F)),
                   tensor_ptr(size_map, "size_map", torch.float32, dev, (n, 2, F, F)),
                   tensor_ptr(offset_map, "offset_map", torch.float32, dev, (n, 2, F, F)), n, _ptr(boxes))
        return boxes

    # ------------------------------------------------------------------------------------------
    def yuv420_to_rgb(self, src: torch.Tensor, src_offsets: torch.Tensor, frame_hw: torch.Tensor, dst: torch.Tensor,
                      dst_offsets: torch.Tensor, format: str) -> torch.Tensor:
        """cv2.cvtColor(COLOR_YUV2RGB_NV12 / _I420) of n frames, bit for bit, device -> device: the (H*3/2) x W YUV frame at byte
        ``src_offsets[i]`` of ``src`` becomes the H x W x 3 frame at byte ``dst_offsets[i]`` of ``dst``.  uint8 buffers, int64
        offsets [n], int32 frame_hw [n, 2] (even), all on this engine's device.  Returns ``dst``."""
        fmt = yuv_format(format)
        n = int(src_offsets.shape[0])
        dev = self.device
        self._call("vt_yuv420_to_rgb", fmt, tensor_ptr(src, "src", torch.uint8, dev),
                   tensor_ptr(src_offsets, "src_offsets", torch.int64, dev, (n,)), tensor_ptr(frame_hw, "frame_hw", torch.int32, dev, (n, 2)),
                   tensor_ptr(dst, "dst", torch.uint8, dev), tensor_ptr(dst_offsets, "dst_offsets", torch.int64, dev, (n,)), n)
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
        host, dev = torch.device("cpu"), self.device
        self._call("vt_upload_yuv420_rect", fmt, image.ctypes.data, H, W, int(y0), int(y1), int(x0), int(x1),
                   tensor_ptr(staging, "staging", torch.uint8, host), tensor_ptr(staging_dev, "staging_dev", torch.uint8, dev),
                   tensor_ptr(frame_rgb, "frame_rgb", torch.uint8, dev))

    def yuv420_crop_to_rgb(self, format: str, planes: torch.Tensor, pitches: torch.Tensor, frame_hw: torch.Tensor, dst: torch.Tensor,
                           dst_offsets: torch.Tensor, factor: float, boxes: Optional[torch.Tensor] = None, first: int = 0) -> torch.Tensor:
        """vt_yuv420_crop_to_rgb: per item, only the even-widened rectangle the crop of its box (``boxes`` float64 [n, 4], or None: the
        state of tracks [first, first + n)) reads, from pitched planes (``planes`` int64 [n, 3] device addresses Y, U or UV, V;
        ``pitches`` int32 [n, 2]) into the H x W x 3 frame at byte ``dst_offsets[i]`` of ``dst``, bit for bit cv2.cvtColor.  No
        allocation and no synchronisation (capturable in a CUDA graph).  Returns ``dst``."""
        fmt = yuv_format(format)
        n = int(planes.shape[0])
        dev = self.device
        self._call("vt_yuv420_crop_to_rgb", fmt, tensor_ptr(planes, "planes", torch.int64, dev, (n, 3)),
                   tensor_ptr(pitches, "pitches", torch.int32, dev, (n, 2)), tensor_ptr(frame_hw, "frame_hw", torch.int32, dev, (n, 2)),
                   tensor_ptr(boxes, "boxes", torch.float64, dev, (n, 4), optional=True), float(factor), int(first), n,
                   tensor_ptr(dst, "dst", torch.uint8, dev), tensor_ptr(dst_offsets, "dst_offsets", torch.int64, dev, (n,)))
        return dst

    def yuv420_crops_to_surface_rgb(self, format: str, planes: torch.Tensor, pitches: torch.Tensor, frame_hw: torch.Tensor,
                                    dst: torch.Tensor, dst_offsets: torch.Tensor, item_surface: torch.Tensor, factor: float,
                                    boxes: Optional[torch.Tensor] = None, slots: Optional[torch.Tensor] = None,
                                    first: int = 0) -> torch.Tensor:
        """vt_yuv420_crops_to_surface_rgb: n items on m surfaces (``planes`` int64 [m, 3], ``pitches`` / ``frame_hw`` int32 [m, 2],
        ``dst_offsets`` int64 [m]: one RGB frame per surface); item i lies on surface ``item_surface[i]`` (int32 [n]).  Each surface's
        frame gets, bit for bit cv2.cvtColor, the bounding rectangle of the crops of its items, whose boxes are ``boxes`` (float64
        [n, 4]) or the state of tracks ``slots[i]`` (int32 [n]) or [first, first + n).  Items with a surface outside [0, m), a bad slot or
        a degenerate crop are skipped.  No allocation and no synchronisation (capturable in a CUDA graph).  Returns ``dst``."""
        fmt = yuv_format(format)
        m, n = int(planes.shape[0]), int(item_surface.shape[0])
        dev = self.device
        self._call("vt_yuv420_crops_to_surface_rgb", fmt, tensor_ptr(planes, "planes", torch.int64, dev, (m, 3)),
                   tensor_ptr(pitches, "pitches", torch.int32, dev, (m, 2)), tensor_ptr(frame_hw, "frame_hw", torch.int32, dev, (m, 2)), m,
                   tensor_ptr(item_surface, "item_surface", torch.int32, dev, (n,)),
                   tensor_ptr(boxes, "boxes", torch.float64, dev, (n, 4), optional=True),
                   tensor_ptr(slots, "slots", torch.int32, dev, (n,), optional=True), float(factor), int(first), n,
                   tensor_ptr(dst, "dst", torch.uint8, dev), tensor_ptr(dst_offsets, "dst_offsets", torch.int64, dev, (m,)))
        return dst

    # ------------------------------------------------------------------------------------------
    def tracks_init(self, frames, frame_offsets, frame_hw, boxes, first: int = 0) -> torch.Tensor:
        n = int(boxes.shape[0])
        status = torch.empty((n,), dtype=torch.int32, device=self.device)
        self._call("vt_tracks_init", *self._frames(frames, frame_offsets, frame_hw, n),
                   tensor_ptr(boxes, "boxes", torch.float64, self.device, (n, 4)), int(first), n, _ptr(status))
        return status

    def tracks_step(self, frames, frame_offsets, frame_hw, first: int = 0, n: Optional[int] = None,
                    out_boxes: Optional[torch.Tensor] = None, out_detail: Optional[torch.Tensor] = None,
                    update_state: bool = True, detail: bool = False):
        n = int(frame_offsets.shape[0] if n is None else n)
        dev = self.device
        if out_boxes is None:
            out_boxes = torch.empty((n, 5), dtype=torch.float64, device=dev)
        if detail and out_detail is None:
            out_detail = torch.empty((n, 8), dtype=torch.float64, device=dev)
        self._call("vt_tracks_step", *self._frames(frames, frame_offsets, frame_hw, n), int(first), n,
                   tensor_ptr(out_boxes, "out_boxes", torch.float64, dev, (n, 5)),
                   tensor_ptr(out_detail, "out_detail", torch.float64, dev, (n, 8), optional=True), 1 if update_state else 0)
        return (out_boxes, out_detail) if detail else out_boxes

    def tracks_init_slots(self, frames, frame_offsets, frame_hw, boxes, slots: torch.Tensor) -> torch.Tensor:
        """vt_tracks_init_slots: item i initialises track ``slots[i]`` (int32 device tensor [n]).  Returns the status per item
        (VT_TRACK_BAD_SLOT for an entry outside [0, max_tracks) or repeating an earlier one)."""
        n = int(boxes.shape[0])
        dev = self.device
        status = torch.empty((n,), dtype=torch.int32, device=dev)
        self._call("vt_tracks_init_slots", *self._frames(frames, frame_offsets, frame_hw, n),
                   tensor_ptr(boxes, "boxes", torch.float64, dev, (n, 4)), tensor_ptr(slots, "slots", torch.int32, dev, (n,)), n, _ptr(status))
        return status

    def tracks_step_slots(self, frames, frame_offsets, frame_hw, slots: torch.Tensor, out_boxes: Optional[torch.Tensor] = None,
                          out_detail: Optional[torch.Tensor] = None, update_state: bool = True, detail: bool = False):
        """vt_tracks_step_slots: item i steps track ``slots[i]`` (int32 device tensor [n]); outputs are in item order."""
        n = int(slots.shape[0])
        dev = self.device
        if out_boxes is None:
            out_boxes = torch.empty((n, 5), dtype=torch.float64, device=dev)
        if detail and out_detail is None:
            out_detail = torch.empty((n, 8), dtype=torch.float64, device=dev)
        self._call("vt_tracks_step_slots", *self._frames(frames, frame_offsets, frame_hw, n),
                   tensor_ptr(slots, "slots", torch.int32, dev, (n,)), n, tensor_ptr(out_boxes, "out_boxes", torch.float64, dev, (n, 5)),
                   tensor_ptr(out_detail, "out_detail", torch.float64, dev, (n, 8), optional=True), 1 if update_state else 0)
        return (out_boxes, out_detail) if detail else out_boxes

    def set_range_fallback(self, enable: bool, counter: Optional[torch.Tensor] = None) -> None:
        """vt_set_range_fallback: with ``enable``, every item of a tracking step that the tensor-core kernels flag
        VT_TRACK_NUMERIC_RANGE is recomputed on the fp32 kernels within the same call, bit for bit what a ``simt`` engine gives.
        ``counter`` (optional int64 device tensor of one element) has the number of recomputed items added to it by every step."""
        ptr = tensor_ptr(counter, "counter", torch.int64, self.device, (1,), optional=True)
        self._check(self.lib.vt_set_range_fallback(self.handle, 1 if enable else 0, ptr))
        # a CUDA graph captured while a counter was set keeps adding to its address on every replay, whatever the fallback's setting
        # since: every counter handed over lives as long as this engine
        if counter is not None:
            self._fallback_counters = getattr(self, "_fallback_counters", []) + [counter]

    # ------------------------------------------------------------------------------------------
    @property
    def weights_fingerprint(self) -> int:
        """vt_weights_fingerprint: the hash of the configuration, template route and tensors this engine's weights were finalised from
        (records.weights_fingerprint restates it).  Equal fingerprints: a track record moves between the two engines bit for bit."""
        out = C.c_uint64()
        self._check(self.lib.vt_weights_fingerprint(self.handle, C.byref(out)))
        return int(out.value)

    @property
    def track_record_bytes(self) -> int:
        """R, the size of one track record of this engine (64 + 256 C bytes)."""
        out = C.c_int64()
        self._check(self.lib.vt_track_record_bytes(self.handle, C.byref(out)))
        return int(out.value)

    def _records(self, records: torch.Tensor, n: int) -> C.c_void_p:
        return tensor_ptr(records, "records", torch.uint8, self.device, (n, self.track_record_bytes), align=16)

    def tracks_export(self, first: int = 0, n: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """vt_tracks_export: the records of tracks [first, first + n) as uint8 [n, R] (into ``out`` when given)."""
        n = self.max_tracks - first if n is None else int(n)
        out = torch.empty((n, self.track_record_bytes), dtype=torch.uint8, device=self.device) if out is None else out
        self._call("vt_tracks_export", int(first), n, self._records(out, n))
        return out

    def tracks_export_slots(self, slots: torch.Tensor, out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """vt_tracks_export_slots: record i of track ``slots[i]``; returns (records [n, R], status [n]: VT_TRACK_OK or
        VT_TRACK_BAD_SLOT, whose record is all zeros)."""
        n = int(slots.shape[0])
        out = torch.empty((n, self.track_record_bytes), dtype=torch.uint8, device=self.device) if out is None else out
        status = torch.empty((n,), dtype=torch.int32, device=self.device)
        self._call("vt_tracks_export_slots", tensor_ptr(slots, "slots", torch.int32, self.device, (n,)), n, self._records(out, n),
                   _ptr(status))
        return out, status

    def tracks_import(self, records: torch.Tensor, first: int = 0) -> torch.Tensor:
        """vt_tracks_import: record i into track first + i, checked on the device.  Returns the status per item: VT_TRACK_OK, or
        VT_TRACK_BAD_RECORD (header, fingerprint, checksum or box rejected; the track is left as it was)."""
        n = int(records.shape[0])
        status = torch.empty((n,), dtype=torch.int32, device=self.device)
        self._call("vt_tracks_import", self._records(records, n), int(first), n, _ptr(status))
        return status

    def tracks_import_slots(self, records: torch.Tensor, slots: torch.Tensor) -> torch.Tensor:
        """vt_tracks_import_slots: record i into track ``slots[i]``; status per item as tracks_import's, or VT_TRACK_BAD_SLOT."""
        n = int(slots.shape[0])
        status = torch.empty((n,), dtype=torch.int32, device=self.device)
        self._call("vt_tracks_import_slots", self._records(records, n), tensor_ptr(slots, "slots", torch.int32, self.device, (n,)), n,
                   _ptr(status))
        return status

    def tracks_get_state(self, first: int = 0, n: Optional[int] = None) -> torch.Tensor:
        n = self.max_tracks - first if n is None else int(n)
        out = torch.empty((n, 4), dtype=torch.float64, device=self.device)
        self._call("vt_tracks_get_state", _ptr(out), int(first), n)
        return out

    def tracks_set_state(self, boxes: torch.Tensor, first: int = 0) -> None:
        n = int(boxes.shape[0])
        self._call("vt_tracks_set_state", tensor_ptr(boxes, "boxes", torch.float64, self.device, (n, 4)), int(first), n)

    def tracks_last_maps(self, first: int, n: int):
        dev = self.device
        score = torch.empty((n, 1, 16, 16), dtype=torch.float32, device=dev)
        size = torch.empty((n, 2, 16, 16), dtype=torch.float32, device=dev)
        off = torch.empty((n, 2, 16, 16), dtype=torch.float32, device=dev)
        self._call("vt_tracks_last_maps", int(first), int(n), _ptr(score), _ptr(size), _ptr(off))
        return {"score_map": score, "size_map": size, "offset_map": off}
