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

from .engine import Engine, yuv420_frame_hw, yuv_format


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


class BatchedTracker:
    """``initialize(pool, frame_index, boxes)`` / ``track(pool, frame_index)`` for n tracks at once:
    the batched counterpart of ``Vit_dist.initialize`` / ``Vit_dist.track``."""

    def __init__(self, cfg, state_dict, max_tracks: int, device: Optional[int] = None, chunk_tracks: int = 0,
                 blocks_impl: str = "tcgen05", depth: Optional[int] = None):
        depth = int(getattr(cfg.MODEL.BACKBONE, "DEPTH", 3)) if depth is None else int(depth)
        self.engine = Engine(cfg, max_tracks=max_tracks, chunk_tracks=chunk_tracks, device=device, blocks_impl=blocks_impl, depth=depth)
        self.engine.load_state_dict(state_dict)
        self.device = self.engine.device
        self.max_tracks = max_tracks
        self.n = 0
        self._hw = None
        self.out_boxes = torch.zeros((max_tracks, 5), dtype=torch.float64, device=self.device)

    def initialize(self, pool: FramePool, frame_index: torch.Tensor, boxes) -> torch.Tensor:
        boxes = torch.as_tensor(boxes, dtype=torch.float64).reshape(-1, 4).to(self.device).contiguous()
        n = boxes.shape[0]
        if n > self.max_tracks:
            raise ValueError(f"{n} tracks > max_tracks {self.max_tracks}")
        self.n = n
        self._hw = pool.hw(n)
        status = self.engine.tracks_init(pool.data, pool.offsets(frame_index.to(self.device)), self._hw, boxes, first=0)
        return status

    def set_state(self, boxes) -> None:
        boxes = torch.as_tensor(boxes, dtype=torch.float64).reshape(-1, 4).to(self.device).contiguous()
        self.engine.tracks_set_state(boxes, first=0)

    def get_state(self) -> torch.Tensor:
        return self.engine.tracks_get_state(0, self.n)

    def track(self, pool: FramePool, frame_index: torch.Tensor, update_state: bool = True, detail: bool = False):
        """One step for all tracks; returns the device tensor [n,5] (x, y, w, h, confidence)."""
        offs = pool.offsets(frame_index.to(self.device))
        return self.track_offsets(pool.data, offs, update_state=update_state, detail=detail)

    def track_offsets(self, frames: torch.Tensor, offsets: torch.Tensor, update_state: bool = True, detail: bool = False):
        out = self.out_boxes[: self.n]
        r = self.engine.tracks_step(frames, offsets, self._hw, first=0, n=self.n, out_boxes=out,
                                    update_state=update_state, detail=detail)
        return r


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
