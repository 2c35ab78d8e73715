"""Batched form of the tracker: B independent tracks advanced per step on one GPU, and the sharded
form that spreads tracks over the ranks of a ``torch.distributed`` job.

The reference runs one process per sequence and binds it to ``worker_id % num_gpu``
(lib/test/evaluation/running.py:105-113,167-186); here a single process per GPU owns a contiguous
slice of tracks whose state (previous box, cached template tokens) stays on the device, and the
only inter-GPU traffic is one gather of ``(x, y, w, h, confidence)`` per step."""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from .engine import YUV_FORMATS, Engine, yuv420_frame_hw, yuv_format
from .records import TrackRecords


class FramePool:
    """uint8 HWC frames resident in HBM, addressed by byte offset (what vt_* entry points take)."""

    def __init__(self, frames, device: torch.device):
        if isinstance(frames, np.ndarray):
            frames = torch.from_numpy(np.ascontiguousarray(frames))
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError("frames must be uint8 [F, H, W, 3]")
        self.F, self.H, self.W = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
        if frames.device.type == "cpu":
            frames = frames.pin_memory() if torch.cuda.is_available() else frames
        self.data = frames.to(device, non_blocking=True).contiguous()
        self.frame_bytes = self.H * self.W * 3

    @classmethod
    def from_yuv420(cls, engine: Engine, frames, format: str) -> "FramePool":
        """RGB pool converted on the device from YUV 4:2:0 frames [F, H*3/2, W] uint8 ("nv12" or "i420", each frame laid out as
        cv2.cvtColor takes it), on the host or already on the device (decoder output): the pool holds, bit for bit,
        cv2.cvtColor(frame, COLOR_YUV2RGB_NV12 / _I420) of every frame."""
        yuv_format(format)
        if isinstance(frames, np.ndarray):
            frames = torch.from_numpy(np.ascontiguousarray(frames))
        if frames.dim() != 3:
            raise ValueError("frames must be uint8 [F, H*3/2, W]")
        H, W = yuv420_frame_hw(frames[0] if frames.shape[0] else frames.new_zeros((0, 0)))
        F, dev = int(frames.shape[0]), engine.device
        if frames.device.type == "cpu":
            frames = frames.pin_memory() if torch.cuda.is_available() else frames
        src = frames.to(dev, non_blocking=True).contiguous()
        pool = cls(torch.empty((F, H, W, 3), dtype=torch.uint8, device=dev), dev)
        conv = _YuvBatch(F, H, W, dev)
        engine.yuv420_to_rgb(src, conv.src_off, conv.hw, pool.data, conv.dst_off, format)
        return pool

    def offsets(self, index: torch.Tensor) -> torch.Tensor:
        return index.to(torch.int64) * self.frame_bytes

    def hw(self, n: int) -> torch.Tensor:
        return torch.tensor([[self.H, self.W]], dtype=torch.int32, device=self.data.device).expand(n, 2).contiguous()


class _YuvBatch:
    """Offsets and sizes of F contiguous (H*3/2) x W YUV frames and of their H x W x 3 RGB counterparts, on the device."""

    def __init__(self, F: int, H: int, W: int, device: torch.device):
        idx = torch.arange(F, dtype=torch.int64)
        self.src_off = (idx * (H * W * 3 // 2)).to(device)
        self.dst_off = (idx * (H * W * 3)).to(device)
        self.hw = torch.tensor([[H, W]], dtype=torch.int32).expand(F, 2).contiguous().to(device)


def _planes(x, what: str) -> list:
    """2-D uint8 planes from a 3-D tensor [n, rows, cols] (one plane per item), a 2-D tensor (one item) or a sequence of 2-D tensors;
    objects with ``__cuda_array_interface__`` (CuPy, Numba, decoder bindings) go through ``torch.as_tensor``, which shares their memory."""
    def tensor(a):
        return a if torch.is_tensor(a) else torch.as_tensor(a)
    if torch.is_tensor(x) or hasattr(x, "__cuda_array_interface__"):
        x = tensor(x)
        if x.dim() == 2:
            return [x]
        if x.dim() != 3:
            raise ValueError(f"{what}: expected a 2-D plane or a 3-D batch of planes, got shape {tuple(x.shape)}")
        return list(x.unbind(0))
    return [tensor(a) for a in x]


class YuvSurfaces:
    """n device-resident YUV 4:2:0 surfaces ("nv12" or "i420") of one picture size H x W, as a hardware decoder hands them out:
    every plane is a strided 2-D uint8 CUDA tensor whose rows are ``stride(0)`` bytes apart (the surface pitch, >= the row width) and
    whose columns are adjacent.  ``luma`` [H, W]; ``chroma`` NV12: the interleaved U V plane [H/2, W]; I420: the U plane [H/2, W/2],
    with ``v`` the V plane [H/2, W/2] at the same pitch.  Each argument is a 3-D tensor [n, rows, cols], a sequence of 2-D planes or
    one 2-D plane; planes may sit anywhere (padding bytes and padding surface rows are never read).

    ``planes`` (int64 [n, 3] device addresses Y, U or UV, V), ``pitches`` (int32 [n, 2] luma, chroma) and ``hw`` (int32 [n, 2]) live on
    the device; the object keeps the plane tensors alive.  The surfaces' contents may change between calls (a decoder reusing them):
    what is read is what they hold when the conversion runs on the stream."""

    def __init__(self, format: str, luma, chroma, v=None):
        i420 = yuv_format(format) == YUV_FORMATS["i420"]
        ys, us = _planes(luma, "luma"), _planes(chroma, "chroma")
        if i420 and v is None:
            raise ValueError("I420 surfaces need the V planes")
        if not i420 and v is not None:
            raise ValueError("NV12 surfaces have no separate V plane (the chroma plane interleaves U and V)")
        vs = _planes(v, "v") if i420 else None
        n = len(ys)
        if n == 0 or len(us) != n or (vs is not None and len(vs) != n):
            raise ValueError(f"{n} luma planes, {len(us)} chroma planes{'' if vs is None else f', {len(vs)} V planes'}: expected as many of each, at least one")
        for p in ys + us + (vs or []):
            if p.dtype != torch.uint8 or p.dim() != 2:
                raise ValueError(f"YUV planes must be 2-D uint8 tensors (got {p.dtype}, shape {tuple(p.shape)})")
        H, W = int(ys[0].shape[0]), int(ys[0].shape[1])
        if H < 2 or W < 2 or H % 2 or W % 2:
            raise ValueError(f"YUV 4:2:0 surfaces need an even H and W of at least 2 (got {H} x {W})")
        cshape = (H // 2, W // 2) if i420 else (H // 2, W)

        def check(p, shape, name):
            if tuple(p.shape) != shape:
                raise ValueError(f"{name} plane of shape {tuple(p.shape)}: expected {shape} for {format} surfaces of {H} x {W}")
            if p.stride(1) != 1 or not shape[1] <= p.stride(0) < 2 ** 31:
                raise ValueError(f"{name} plane with strides {p.stride()}: expected (pitch, 1) with {shape[1]} <= pitch < 2^31")

        for k in range(n):
            check(ys[k], (H, W), "luma")
            check(us[k], cshape, "U" if i420 else "chroma")
            if i420:
                check(vs[k], cshape, "V")
                if vs[k].stride(0) != us[k].stride(0):
                    raise ValueError(f"I420 U and V planes must share one pitch (got {us[k].stride(0)} and {vs[k].stride(0)})")
        devices = {p.device for p in ys + us + (vs or [])}
        if len(devices) != 1 or next(iter(devices)).type != "cuda":
            raise ValueError(f"YUV surfaces must be CUDA tensors on one device (got {sorted(map(str, devices))})")
        self.format, self.n, self.H, self.W = format, n, H, W
        self.device = next(iter(devices))
        addr = [[ys[k].data_ptr(), us[k].data_ptr(), vs[k].data_ptr() if i420 else 0] for k in range(n)]
        self.planes = torch.tensor(addr, dtype=torch.int64).to(self.device)
        self.pitches = torch.tensor([[ys[k].stride(0), us[k].stride(0)] for k in range(n)], dtype=torch.int32).to(self.device)
        self.hw = torch.tensor([[H, W]], dtype=torch.int32).expand(n, 2).contiguous().to(self.device)
        self._keep = (ys, us, vs)

    @classmethod
    def from_frames(cls, frames, format: str, height: Optional[int] = None, surface_rows: Optional[int] = None) -> "YuvSurfaces":
        """Surfaces from one uint8 CUDA tensor [n, rows, W] (or [rows, W] for one) whose rows are ``stride(-2)`` bytes apart (the pitch):
        per frame the luma plane is rows [0, H), and the chroma starts at row ``surface_rows`` (default H; a decoder's padded surface
        height, e.g. 1088 for 1080p).  NV12: chroma rows [S, S + H/2).  I420: the U plane at byte S * pitch with rows pitch/2 apart,
        the V plane (S/2) * (pitch/2) bytes after it.  With the defaults and pitch W, a frame is laid out as cv2.cvtColor takes it,
        (H*3/2) x W.  ``height`` defaults to rows * 2/3."""
        yuv_format(format)
        f = frames if torch.is_tensor(frames) else torch.as_tensor(frames)
        if f.dim() == 2:
            f = f.unsqueeze(0)
        if f.dim() != 3 or f.dtype != torch.uint8 or f.stride(2) != 1:
            raise ValueError("frames must be a uint8 tensor [n, rows, W] with adjacent columns")
        n, R, W = (int(v) for v in f.shape)
        H = R * 2 // 3 if height is None else int(height)
        if height is None and R != H * 3 // 2:
            raise ValueError(f"frames of {R} rows: give the picture height, or use the (H*3/2) x W layout")
        S = H if surface_rows is None else int(surface_rows)
        P = f.stride(1)
        if H < 2 or H % 2 or S < H or S % 2:
            raise ValueError(f"picture height {H} / surface rows {S}: expected even values with surface rows >= height")
        if format == "nv12":
            if S + H // 2 > R:
                raise ValueError(f"NV12 frames of {R} rows cannot hold {S} surface rows + {H // 2} chroma rows")
            return cls(format, f[:, :H], f[:, S:S + H // 2])
        if P % 2 or S * P + (S // 2) * (P // 2) + (H // 2) * (P // 2) > R * P:
            raise ValueError(f"I420 frames of {R} rows x pitch {P} cannot hold {S} surface rows and two chroma planes (pitch must be even)")
        base = f.storage_offset() + S * P
        u = f.as_strided((n, H // 2, W // 2), (f.stride(0), P // 2, 1), base)
        v = f.as_strided((n, H // 2, W // 2), (f.stride(0), P // 2, 1), base + (S // 2) * (P // 2))
        return cls(format, f[:, :H], u, v)


def check_slots(slots, max_tracks: int) -> list:
    """A host sequence of track slots as a list of ints; ValueError for an entry outside [0, max_tracks) or named twice."""
    out = [int(v) for v in slots]
    seen = set()
    for v in out:
        if not 0 <= v < max_tracks:
            raise ValueError(f"slot {v} outside [0, {max_tracks})")
        if v in seen:
            raise ValueError(f"slot {v} listed twice")
        seen.add(v)
    return out


class BatchedTracker:
    """``initialize(pool, frame_index, boxes)`` / ``track(pool, frame_index)`` for n tracks at once:
    the batched counterpart of ``Vit_dist.initialize`` / ``Vit_dist.track``.

    Without ``slots`` these calls work on tracks 0..n-1.  With ``slots`` (a host sequence of ints, checked here, or a CUDA integer
    tensor, passed through: the device gives a bad entry status VT_TRACK_BAD_SLOT), item i works on track ``slots[i]`` and results come
    back in slot-list order, so targets can be added to free slots, retired, and the live set stepped in one call.

    ``range_fallback=True`` recomputes, within the same step, every track the tensor-core kernels flag as out of fp16 range
    (VT_TRACK_NUMERIC_RANGE) on the fp32 kernels: such a track gets the result a ``blocks_impl="simt"`` tracker would give instead of
    confidence -1.  ``fallback_items`` counts the recomputed items."""

    def __init__(self, cfg, state_dict, max_tracks: int, device: Optional[int] = None, chunk_tracks: int = 0,
                 blocks_impl: str = "tcgen05", depth: Optional[int] = None, range_fallback: bool = False):
        depth = int(getattr(cfg.MODEL.BACKBONE, "DEPTH", 3)) if depth is None else int(depth)
        self.engine = Engine(cfg, max_tracks=max_tracks, chunk_tracks=chunk_tracks, device=device, blocks_impl=blocks_impl, depth=depth)
        self.engine.load_state_dict(state_dict)
        self.device = self.engine.device
        self._fallback_count = None
        if range_fallback:
            self._fallback_count = torch.zeros((1,), dtype=torch.int64, device=self.device)
            self.engine.set_range_fallback(True, self._fallback_count)
        self.max_tracks = max_tracks
        self.n = 0
        self._hw = None
        self.out_boxes = torch.zeros((max_tracks, 5), dtype=torch.float64, device=self.device)
        self.template_factor, self.search_factor = float(cfg.TEST.TEMPLATE_FACTOR), float(cfg.TEST.SEARCH_FACTOR)
        self._yuv_rgb: Optional[torch.Tensor] = None             # initialize_yuv / track_yuv: one RGB frame per track
        self._yuv_off: Optional[torch.Tensor] = None
        self._surf_rgb: Optional[torch.Tensor] = None            # ... with surface=: one RGB frame per surface, plus one for bad entries
        self._surf_off: Optional[torch.Tensor] = None
        # (H, W) of every slot's frames, for steps by slot list; row max_tracks takes the writes of bad entries
        self._slot_hw = torch.zeros((max_tracks + 1, 2), dtype=torch.int32, device=self.device)

    @property
    def fallback_items(self) -> int:
        """Items recomputed on the fp32 kernels so far (0 without ``range_fallback``).  Reading it synchronises with the device."""
        return 0 if self._fallback_count is None else int(self._fallback_count.item())

    def _slots(self, slots) -> torch.Tensor:
        """The slot list as the contiguous int32 device tensor the engine takes."""
        if torch.is_tensor(slots) and slots.is_cuda:
            if slots.dtype not in (torch.int32, torch.int64) or slots.dim() != 1 or slots.device != self.device:
                raise ValueError(f"slots: expected a 1-D integer tensor on {self.device}")
            return slots.to(torch.int32).contiguous()
        return torch.tensor(check_slots(slots.tolist() if torch.is_tensor(slots) else slots, self.max_tracks), dtype=torch.int32,
                            device=self.device)

    def _rows(self, slots: torch.Tensor) -> torch.Tensor:
        """Per item the slot it works on, as the device resolves the list (first occurrence of an in-range slot), or max_tracks for a bad
        entry: indexes per-slot tensors that have a spare last row, without a host synchronisation."""
        mt, n = self.max_tracks, slots.shape[0]
        s = slots.to(torch.int64)
        item = torch.arange(n, dtype=torch.int64, device=self.device)
        s = torch.where((s >= 0) & (s < mt), s, mt)
        first = torch.full((mt + 1,), n, dtype=torch.int64, device=self.device).scatter_reduce_(0, s, item, "amin")
        return torch.where(first[s] == item, s, mt)

    def initialize(self, pool: FramePool, frame_index: torch.Tensor, boxes, slots=None) -> torch.Tensor:
        boxes = torch.as_tensor(boxes, dtype=torch.float64).reshape(-1, 4).to(self.device).contiguous()
        n = boxes.shape[0]
        if n > self.max_tracks:
            raise ValueError(f"{n} tracks > max_tracks {self.max_tracks}")
        offs = pool.offsets(frame_index.to(self.device))
        if slots is not None:
            return self._init_slots(pool.data, offs, pool.hw(n), boxes, self._slots(slots))
        self.n = n
        self._hw = pool.hw(n)
        self._slot_hw[:n] = self._hw
        status = self.engine.tracks_init(pool.data, offs, self._hw, boxes, first=0)
        return status

    def _init_slots(self, frames, offsets, hw, boxes, slots: torch.Tensor) -> torch.Tensor:
        if slots.shape[0] != boxes.shape[0]:
            raise ValueError(f"{slots.shape[0]} slots for {boxes.shape[0]} boxes")
        self._slot_hw[self._rows(slots)] = hw
        return self.engine.tracks_init_slots(frames, offsets, hw, boxes, slots)

    def set_state(self, boxes, slots=None) -> None:
        """Overwrite the boxes of tracks 0..n-1, or of the listed slots (a bad entry of a CUDA slot tensor is skipped)."""
        boxes = torch.as_tensor(boxes, dtype=torch.float64).reshape(-1, 4).to(self.device).contiguous()
        if slots is None:
            self.engine.tracks_set_state(boxes, first=0)
            return
        slots = self._slots(slots)
        state = torch.cat([self.engine.tracks_get_state(0, self.max_tracks), boxes.new_zeros((1, 4))])
        state[self._rows(slots)] = boxes
        self.engine.tracks_set_state(state[: self.max_tracks].contiguous(), first=0)

    def get_state(self, slots=None) -> torch.Tensor:
        """Boxes [n, 4] of tracks 0..n-1, or of the listed slots in list order (NaN for a bad entry of a CUDA slot tensor)."""
        if slots is None:
            return self.engine.tracks_get_state(0, self.n)
        slots = self._slots(slots)
        state = torch.cat([self.engine.tracks_get_state(0, self.max_tracks), torch.full((1, 4), float("nan"), dtype=torch.float64,
                                                                                          device=self.device)])
        return state[self._rows(slots)]

    def track(self, pool: FramePool, frame_index: torch.Tensor, update_state: bool = True, detail: bool = False, slots=None):
        """One step for all tracks (or for the listed slots, frame_index[i] for slots[i]); returns the device tensor [n,5] (x, y, w, h,
        confidence)."""
        offs = pool.offsets(frame_index.to(self.device))
        return self.track_offsets(pool.data, offs, update_state=update_state, detail=detail, slots=slots)

    def track_offsets(self, frames: torch.Tensor, offsets: torch.Tensor, update_state: bool = True, detail: bool = False, slots=None):
        if slots is not None:
            slots = self._slots(slots)
            return self._step_slots(frames, offsets, self._slot_hw[self._rows(slots)], slots, update_state, detail)
        out = self.out_boxes[: self.n]
        r = self.engine.tracks_step(frames, offsets, self._hw, first=0, n=self.n, out_boxes=out,
                                    update_state=update_state, detail=detail)
        return r

    def _step_slots(self, frames, offsets, hw, slots: torch.Tensor, update_state: bool, detail: bool):
        if offsets.shape[0] != slots.shape[0]:
            raise ValueError(f"{offsets.shape[0]} frames for {slots.shape[0]} slots")
        return self.engine.tracks_step_slots(frames, offsets, hw, slots, out_boxes=self.out_boxes[: slots.shape[0]],
                                             update_state=update_state, detail=detail)

    def export_tracks(self, slots=None) -> TrackRecords:
        """Track records of tracks 0..n-1, or of the listed slots in list order, with each track's frame size: save them, or import them
        into this or another tracker (``records.to("cuda:1")`` moves them to another GPU).  A bad entry of a CUDA slot tensor gets an
        all-zero record, which every import rejects."""
        if slots is None:
            return TrackRecords(self.engine.tracks_export(0, self.n), self._slot_hw[: self.n].clone())
        slots = self._slots(slots)
        records, _ = self.engine.tracks_export_slots(slots)
        return TrackRecords(records, self._slot_hw[self._rows(slots)])

    def import_tracks(self, records: TrackRecords, slots=None) -> torch.Tensor:
        """Continue exported tracks here, bit for bit: without ``slots`` as tracks 0..n-1 (as ``initialize`` sets them up), else into the
        listed slots.  The device checks every record; returns the status per item: VT_TRACK_OK, VT_TRACK_BAD_RECORD (5: other weights,
        another embed dim, or an altered record; the track is left as it was, records.describe_rejection says why) or, by slot,
        VT_TRACK_BAD_SLOT.  Frame sizes are taken for the accepted items only, without a host synchronisation."""
        if not isinstance(records, TrackRecords):
            raise ValueError("records: expected a TrackRecords (BatchedTracker.export_tracks / TrackRecords.load)")
        rec, hw = records.records, records.frame_hw
        R, n = self.engine.track_record_bytes, len(records)
        if rec.dtype != torch.uint8 or rec.dim() != 2 or rec.shape[1] != R:
            raise ValueError(f"records of {tuple(rec.shape)} {rec.dtype}: this tracker's records are uint8 [n, {R}]")
        if not (rec.is_contiguous() and hw.is_contiguous()) or rec.data_ptr() % 16:
            raise ValueError("records: expected contiguous, 16-byte aligned tensors")
        if rec.device != self.device or hw.device != self.device:
            raise ValueError(f"records on {rec.device}, tracker on {self.device}: move them with records.to(...)")
        if n > self.max_tracks:
            raise ValueError(f"{n} records > max_tracks {self.max_tracks}")
        if slots is None:
            status = self.engine.tracks_import(rec, first=0)
            self._slot_hw[:n] = torch.where((status == 0)[:, None], hw, self._slot_hw[:n])
            self.n = n
            self._hw = self._slot_hw[:n].clone()
            return status
        slots = self._slots(slots)
        if slots.shape[0] != n:
            raise ValueError(f"{slots.shape[0]} slots for {n} records")
        rows = self._rows(slots)
        status = self.engine.tracks_import_slots(rec, slots)
        self._slot_hw[rows] = torch.where((status == 0)[:, None], hw, self._slot_hw[rows])
        return status

    def _yuv_frames(self, surfaces: YuvSurfaces) -> Tuple[torch.Tensor, torch.Tensor]:
        if surfaces.n > self.max_tracks:
            raise ValueError(f"{surfaces.n} surfaces > max_tracks {self.max_tracks}")
        if surfaces.device != self.device:
            raise ValueError(f"surfaces on {surfaces.device}, tracker on {self.device}")
        if self._yuv_rgb is None or tuple(self._yuv_rgb.shape[1:3]) != (surfaces.H, surfaces.W):
            self._yuv_rgb = None
            # zero-filled once: the crop kernels read the first pixels of a row with weight 0 for taps in the padding.  The frame
            # after the last track's takes the conversions of bad slot-list entries.
            self._yuv_rgb = torch.zeros((self.max_tracks + 1, surfaces.H, surfaces.W, 3), dtype=torch.uint8, device=self.device)
            self._yuv_off = torch.arange(self.max_tracks + 1, dtype=torch.int64, device=self.device) * (surfaces.H * surfaces.W * 3)
        return self._yuv_rgb, self._yuv_off[: surfaces.n]

    def _surface_frames(self, surfaces: YuvSurfaces) -> Tuple[torch.Tensor, torch.Tensor]:
        if surfaces.n > self.max_tracks:
            raise ValueError(f"{surfaces.n} surfaces > max_tracks {self.max_tracks}")
        if surfaces.device != self.device:
            raise ValueError(f"surfaces on {surfaces.device}, tracker on {self.device}")
        shape = (surfaces.n + 1, surfaces.H, surfaces.W, 3)
        if self._surf_rgb is None or tuple(self._surf_rgb.shape) != shape:
            self._surf_rgb = None
            # zero-filled once, as the per-track frames; the last frame is the one bad entries of a CUDA surface tensor crop from
            self._surf_rgb = torch.zeros(shape, dtype=torch.uint8, device=self.device)
            self._surf_off = torch.arange(surfaces.n + 1, dtype=torch.int64, device=self.device) * (surfaces.H * surfaces.W * 3)
        return self._surf_rgb, self._surf_off

    def _surface_items(self, surfaces: YuvSurfaces, surface, n: int, slots: Optional[torch.Tensor]):
        """Per item its surface (int32 device tensor [n]), frame offset and size, gathered on the device, and the slot list the step takes:
        ``slots`` as given, or None for a range call; with a CUDA surface tensor, a list in which every entry whose surface lies outside
        [0, m) is bad (-1), so that the device steps it as a bad slot-list entry."""
        m = surfaces.n
        frames, soff = self._surface_frames(surfaces)
        if torch.is_tensor(surface) and surface.is_cuda:
            if surface.dtype not in (torch.int32, torch.int64) or surface.dim() != 1 or surface.device != self.device:
                raise ValueError(f"surface: expected a 1-D integer tensor on {self.device}")
            if surface.shape[0] != n:
                raise ValueError(f"{surface.shape[0]} surface entries for {n} items")
            surf, checked = surface.to(torch.int32).contiguous(), False
        else:
            vals = [int(v) for v in (surface.tolist() if torch.is_tensor(surface) else surface)]
            if len(vals) != n:
                raise ValueError(f"{len(vals)} surface entries for {n} items")
            for v in vals:
                if not 0 <= v < m:
                    raise ValueError(f"surface {v} outside [0, {m})")
            surf, checked = torch.tensor(vals, dtype=torch.int32, device=self.device), True
        s = surf.to(torch.int64)
        ok = (s >= 0) & (s < m)
        row = torch.where(ok, s, m)
        offs, hw = soff[row], surfaces.hw[row.clamp(max=m - 1)]
        if not checked:
            base = slots if slots is not None else torch.arange(n, dtype=torch.int32, device=self.device)
            slots = torch.where(ok, base, -1).to(torch.int32)
        return frames, soff[:m], offs, hw, surf, slots

    def _init_surfaces(self, surfaces: YuvSurfaces, boxes: torch.Tensor, slots, surface) -> torch.Tensor:
        n = boxes.shape[0]
        if n > self.max_tracks:
            raise ValueError(f"{n} tracks > max_tracks {self.max_tracks}")
        listed = None if slots is None else self._slots(slots)
        if listed is not None and listed.shape[0] != n:
            raise ValueError(f"{listed.shape[0]} slots for {n} boxes")
        frames, soff, offs, hw, surf, eff = self._surface_items(surfaces, surface, n, listed)
        self.engine.yuv420_crops_to_surface_rgb(surfaces.format, surfaces.planes, surfaces.pitches, surfaces.hw, frames, soff, surf,
                                                self.template_factor, boxes=boxes, slots=eff)
        if listed is None:
            self.n = n
            self._hw = hw
            if eff is None:
                self._slot_hw[:n] = hw
                return self.engine.tracks_init(frames, offs, hw, boxes, first=0)
        return self._init_slots(frames, offs, hw, boxes, eff)

    def initialize_yuv(self, surfaces: YuvSurfaces, boxes, slots=None, surface=None) -> torch.Tensor:
        """``initialize`` for tracks 0..n-1 from device-resident YUV surfaces (``YuvSurfaces``, track i on surface i): only the rectangle
        each template crop reads is converted (vt_yuv420_crop_to_rgb, bit for bit cv2.cvtColor), into an RGB frame per track that
        this tracker owns, then vt_tracks_init runs on it on the same stream.  Those frames cost max_tracks x H x W x 3 bytes of
        device memory (2.76 MB per track at 720p, 6.2 MB at 1080p), allocated at the first call for a picture size.  With ``slots``,
        surface i belongs to track slots[i], whose RGB frame it is converted into.

        ``surface`` (several targets per surface): item i - box i, and track i or slots[i] - lies on ``surfaces`` entry ``surface[i]``,
        a host sequence of ints (checked here: ValueError outside [0, surfaces.n)) or a CUDA integer tensor (passed through: an entry
        outside [0, surfaces.n) makes the item a bad slot-list entry, VT_TRACK_BAD_SLOT, which touches no track state).  Each surface
        is converted once, over the bounding rectangle of its items' crops (vt_yuv420_crops_to_surface_rgb), into one RGB frame per
        surface: (surfaces.n + 1) x H x W x 3 bytes instead of (max_tracks + 1) x H x W x 3.  Results are bit for bit those of the
        per-track path."""
        boxes = torch.as_tensor(boxes, dtype=torch.float64).reshape(-1, 4).to(self.device).contiguous()
        if surface is not None:
            return self._init_surfaces(surfaces, boxes, slots, surface)
        if boxes.shape[0] != surfaces.n:
            raise ValueError(f"{boxes.shape[0]} boxes for {surfaces.n} surfaces")
        frames, offs = self._yuv_frames(surfaces)
        if slots is not None:
            slots = self._slots(slots)
            offs = self._yuv_off[self._rows(slots)]
            self.engine.yuv420_crop_to_rgb(surfaces.format, surfaces.planes, surfaces.pitches, surfaces.hw, frames, offs,
                                           self.template_factor, boxes=boxes)
            return self._init_slots(frames, offs, surfaces.hw, boxes, slots)
        self.engine.yuv420_crop_to_rgb(surfaces.format, surfaces.planes, surfaces.pitches, surfaces.hw, frames, offs,
                                       self.template_factor, boxes=boxes)
        self.n = surfaces.n
        self._hw = surfaces.hw
        self._slot_hw[: self.n] = self._hw
        return self.engine.tracks_init(frames, offs, self._hw, boxes, first=0)

    def track_yuv(self, surfaces: YuvSurfaces, update_state: bool = True, detail: bool = False, slots=None, surface=None):
        """``track`` from device-resident YUV surfaces (surface i for track i): the rectangle each search crop reads is computed on the
        device from the track's current state - the host never waits for it - and converted; then vt_tracks_step runs on the same
        stream.  No allocation after the first call for a picture size, so a step can be captured in a CUDA graph.  With ``slots``,
        surface i belongs to track slots[i]: its state is gathered on the device and the surface is converted into that track's frame.

        ``surface`` as for ``initialize_yuv``: item i (track i, or slots[i]) is on surface ``surface[i]``; each surface is converted once,
        over the bounding rectangle of its items' search crops, computed on the device from the tracks' states.  With a CUDA surface
        tensor (needed for CUDA-graph capture) the step runs as a slot list, so that an entry outside [0, surfaces.n) gets
        VT_TRACK_BAD_SLOT and leaves its track as it was."""
        if surface is not None:
            listed = None if slots is None else self._slots(slots)
            n = self.n if listed is None else listed.shape[0]
            frames, soff, offs, hw, surf, eff = self._surface_items(surfaces, surface, n, listed)
            self.engine.yuv420_crops_to_surface_rgb(surfaces.format, surfaces.planes, surfaces.pitches, surfaces.hw, frames, soff, surf,
                                                    self.search_factor, boxes=None, slots=eff, first=0)
            if eff is None:
                self._hw = hw
                return self.track_offsets(frames, offs, update_state=update_state, detail=detail)
            return self._step_slots(frames, offs, hw, eff, update_state, detail)
        if slots is not None:
            slots = self._slots(slots)
            if slots.shape[0] != surfaces.n:
                raise ValueError(f"{surfaces.n} surfaces for {slots.shape[0]} slots")
            frames, _ = self._yuv_frames(surfaces)
            rows = self._rows(slots)
            boxes = self.engine.tracks_get_state(0, self.max_tracks)[rows.clamp(max=self.max_tracks - 1)]
            offs = self._yuv_off[rows]
            self.engine.yuv420_crop_to_rgb(surfaces.format, surfaces.planes, surfaces.pitches, surfaces.hw, frames, offs,
                                           self.search_factor, boxes=boxes)
            return self._step_slots(frames, offs, surfaces.hw, slots, update_state, detail)
        if surfaces.n != self.n:
            raise ValueError(f"{surfaces.n} surfaces for {self.n} tracks")
        frames, offs = self._yuv_frames(surfaces)
        self.engine.yuv420_crop_to_rgb(surfaces.format, surfaces.planes, surfaces.pitches, surfaces.hw, frames, offs,
                                       self.search_factor, boxes=None, first=0)
        self._hw = surfaces.hw
        return self.track_offsets(frames, offs, update_state=update_state, detail=detail)


class PipelinedFrameFeeder:
    """Host -> HBM frame ingest overlapped with tracking: two device frame pools and a copy stream.

    ``upload(host_frames, host_boxes)`` starts the asynchronous copy of the next step's frames (pinned uint8
    [F, H, W, 3]) - and optionally of that step's per-track boxes (pinned float64 [n, 4]) - into the idle pool;
    ``acquire()`` makes the compute stream wait for the oldest pending upload and returns that pool (its boxes, if
    any, are ``pool.boxes``); ``release(pool)`` marks the pool reusable once the work queued so far on the compute
    stream (the step that read it) has finished.

    Every host-to-device copy of a step goes through the copy stream, small ones first: a copy engine serves its
    queue in submission order, so a small upload issued on the compute stream would wait behind the next step's
    frames and stall the step that needs it.

    ``frame_format="nv12"`` or ``"i420"`` (``engine`` required): host frames are YUV 4:2:0 [F, H*3/2, W], half the bytes of
    RGB on the link.  They land in one of two YUV upload pools; ``acquire()`` converts that pool on the compute stream
    (vt_yuv420_to_rgb, bit for bit cv2.cvtColor) into its paired RGB pool and returns the RGB pool; ``release()``
    covers both."""

    def __init__(self, F: int, H: int, W: int, device: torch.device, max_tracks: int = 0, frame_format: str = "rgb",
                 engine: Optional[Engine] = None):
        self.device = device
        self.frame_format = frame_format
        self.yuv = None
        if frame_format != "rgb":
            yuv_format(frame_format)
            if engine is None:
                raise ValueError("a YUV frame_format needs the engine that converts the frames")
            if H < 2 or W < 2 or H % 2 or W % 2:
                raise ValueError(f"YUV 4:2:0 frames need an even H and W (got {H} x {W})")
            self.engine = engine
            self.yuv = [torch.zeros((F, H * 3 // 2, W), dtype=torch.uint8, device=device) for _ in range(2)]
            self._conv = _YuvBatch(F, H, W, device)
        self.pools = [FramePool(torch.zeros((F, H, W, 3), dtype=torch.uint8), device) for _ in range(2)]
        for p in self.pools:
            p.boxes = torch.zeros((max_tracks, 4), dtype=torch.float64, device=device) if max_tracks > 0 else None
        self.copy_stream = torch.cuda.Stream(device=device)
        self._ready = [torch.cuda.Event(), torch.cuda.Event()]
        self._free = [None, None]
        self._pending = []
        self._next = 0

    def upload(self, host_frames: torch.Tensor, host_boxes: Optional[torch.Tensor] = None) -> None:
        i = self._next
        self._next ^= 1
        with torch.cuda.stream(self.copy_stream):
            if self._free[i] is not None:
                self.copy_stream.wait_event(self._free[i])
            if host_boxes is not None:
                self.pools[i].boxes[: host_boxes.shape[0]].copy_(host_boxes, non_blocking=True)
            (self.pools[i].data if self.yuv is None else self.yuv[i]).copy_(host_frames, non_blocking=True)
            self._ready[i].record(self.copy_stream)
        self._pending.append(i)

    def acquire(self) -> FramePool:
        i = self._pending.pop(0)
        torch.cuda.current_stream(self.device).wait_event(self._ready[i])
        if self.yuv is not None:
            c = self._conv
            self.engine.yuv420_to_rgb(self.yuv[i], c.src_off, c.hw, self.pools[i].data, c.dst_off, self.frame_format)
        return self.pools[i]

    def release(self, pool: FramePool) -> None:
        i = 0 if pool is self.pools[0] else 1
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._free[i] = ev


class _CompactingWork:
    """``wait()`` of an asynchronous all-gather over ragged shards: waits, then gathers the valid rows into ``out``."""

    def __init__(self, work, flat, index, out):
        self.work, self.flat, self.index, self.out = work, flat, index, out

    def wait(self):
        r = self.work.wait()
        torch.index_select(self.flat, 0, self.index, out=self.out)
        return r


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous slice [lo, hi) of ``total`` tracks owned by ``rank`` (sizes differ by at most one)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class ShardedTracker:
    """Tracks sharded over the ranks of the default process group; ``gather`` all-gathers the boxes.

    The data path has no collective: each rank crops, runs the model and updates the state of its
    own slice.  ``gather`` is the single exchange step (NCCL all-gather over NVLink on GPUs, gloo on
    CPU for the host-logic tests); ragged slices are padded to the largest slice."""

    def __init__(self, total_tracks: int, local: Optional[BatchedTracker] = None, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.total = total_tracks
        self.lo, self.hi = shard_range(total_tracks, self.rank, self.world)
        self.local = local
        self.max_local = max(shard_range(total_tracks, r, self.world)[1] - shard_range(total_tracks, r, self.world)[0]
                             for r in range(self.world))
        self._gather_buf = None

    @property
    def n_local(self) -> int:
        return self.hi - self.lo

    def _buffers(self, k: int, dev, dt):
        if self._gather_buf is None or self._gather_buf[0].device != dev or self._gather_buf[0].dtype != dt:
            self._gather_buf = [torch.zeros((self.world, self.max_local, 5), dtype=dt, device=dev) for _ in range(2)]
            self._send_buf = [torch.zeros((self.max_local, 5), dtype=dt, device=dev) for _ in range(2)]
        return self._gather_buf[k], self._send_buf[k]

    def _ordered(self, buf: torch.Tensor) -> torch.Tensor:
        if self.total % self.world == 0:
            return buf.view(-1, 5)
        parts = []
        for r in range(self.world):
            lo, hi = shard_range(self.total, r, self.world)
            parts.append(buf[r, : hi - lo])
        return torch.cat(parts, 0)

    def gather(self, local_boxes: torch.Tensor) -> torch.Tensor:
        """[n_local, 5] per rank -> [total, 5] on every rank, ordered by global track id."""
        if self.world == 1:
            return local_boxes
        buf, send = self._buffers(0, local_boxes.device, local_boxes.dtype)
        send[: self.n_local].copy_(local_boxes)
        self.dist.all_gather_into_tensor(buf.view(-1, 5), send, group=self.group)
        return self._ordered(buf)

    def gather_async(self, local_boxes: torch.Tensor):
        """Start the gather of this step's boxes and return ``(work, result)``: the collective runs on NCCL's stream, so the
        next step's kernels are not ordered behind it (nor behind the slowest rank); call ``work.wait()`` before reading
        ``result`` ([total, 5] ordered by global track id, valid for two calls - the buffers alternate).  At most one gather
        may be outstanding.  With ragged shards (total % world != 0) ``work.wait()`` also drops the padding rows."""
        if self.world == 1:
            return None, local_boxes
        self._flip = getattr(self, "_flip", 0) ^ 1
        buf, send = self._buffers(self._flip, local_boxes.device, local_boxes.dtype)
        send[: self.n_local].copy_(local_boxes)
        work = self.dist.all_gather_into_tensor(buf.view(-1, 5), send, group=self.group, async_op=True)
        if self.total % self.world == 0:
            return work, buf.view(-1, 5)
        # ragged: rows of the padded [world, max_local, 5] buffer in global-track order, compacted once the gather has landed
        if getattr(self, "_order_idx", None) is None or self._order_idx.device != buf.device:
            idx = [r * self.max_local + k for r in range(self.world) for k in range(shard_range(self.total, r, self.world)[1] - shard_range(self.total, r, self.world)[0])]
            self._order_idx = torch.tensor(idx, dtype=torch.int64, device=buf.device)
            self._ordered_out = [torch.zeros((self.total, 5), dtype=buf.dtype, device=buf.device) for _ in range(2)]
        res = self._ordered_out[self._flip]
        return _CompactingWork(work, buf.view(-1, 5), self._order_idx, res), res
