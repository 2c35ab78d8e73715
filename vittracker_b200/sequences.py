"""Batched multi-sequence driver: many ``Sequence``s advanced concurrently on one GPU (SURVEY 8f, rank 1).

The reference evaluates a dataset with ``multiprocessing.Pool`` - one process, one tracker, one sequence at a time per
worker, ``worker_id % num_gpu`` picks the GPU (lib/test/evaluation/running.py:105-113,159-187) - and
``Tracker._track_sequence`` (lib/test/evaluation/tracker.py:90-152) walks the frames.  Here ``slots`` sequences share one
``BatchedTracker``: every step uploads the next frame of each running sequence, advances all of them with one
``vt_tracks_step_slots`` over the running slots, and a slot whose sequence ended is re-initialised with the next pending one
(ragged lengths, mixed frame sizes).  Outputs keep the reference's shape - per sequence ``{'target_bbox': [[x, y, w, h], ...], 'time': [...]}``
with the init box as entry 0 - and ``save_tracker_output`` writes the same ``<seq>.txt`` / ``<seq>_time.txt`` files
(running.py:14-102), so the analysis tooling reads them unchanged."""
from __future__ import annotations

import math
import os
import time
from concurrent.futures import Future, ThreadPoolExecutor
from typing import Callable, Dict, List, Optional, Sequence as Seq, Tuple, Union

import numpy as np

from .batched import check_slots

Frame = Union[np.ndarray, str, bytes, list, Callable[[], np.ndarray]]


class Sequence:
    """What the driver needs of lib/test/evaluation/data.py:Sequence: a name, the frames (arrays, image paths or
    zero-argument loaders) and the initial box [x, y, w, h]."""

    def __init__(self, name: str, frames: Seq[Frame], init_bbox, dataset: str = ""):
        self.name = name
        self.frames = list(frames)
        self.init_bbox = [float(v) for v in init_bbox]
        self.dataset = dataset

    def init_info(self) -> dict:
        return {"init_bbox": list(self.init_bbox)}


_LMDB_HANDLES: Dict[str, object] = {}


def decode_image(buf) -> np.ndarray:
    """Encoded image bytes -> HxWx3 uint8 RGB: the decode step of lib/utils/lmdb_utils.py:23-30 (cv.imdecode + BGR2RGB)."""
    import cv2 as cv
    im = cv.imdecode(np.frombuffer(buf, np.uint8), cv.IMREAD_COLOR)
    if im is None:
        raise ValueError("image bytes could not be decoded")
    return cv.cvtColor(im, cv.COLOR_BGR2RGB)


def read_image(frame: Frame) -> np.ndarray:
    """HxWx3 uint8 RGB, as Tracker._read_image delivers it (lib/test/evaluation/tracker.py:282-289): a path goes through cv.imread +
    BGR2RGB; a two-element list [lmdb_file, key] through the LMDB lookup + cv.imdecode of lib/utils/lmdb_utils.py:11-30.  Also accepted:
    an array (used as is), a zero-argument loader, and encoded image bytes (the LMDB value itself)."""
    if isinstance(frame, np.ndarray):
        return frame
    if callable(frame):
        return frame()
    if isinstance(frame, (bytes, bytearray, memoryview)):
        return decode_image(frame)
    if isinstance(frame, (list, tuple)) and len(frame) == 2:
        import lmdb                                                     # the reference's dependency for this branch; not bundled
        name, key = frame
        handle = _LMDB_HANDLES.get(name)
        if handle is None:
            env = lmdb.open(name, readonly=True, lock=False, readahead=False, meminit=False)
            handle = _LMDB_HANDLES[name] = env.begin(write=False)
        buf = handle.get(key.encode())
        if buf is None:
            raise FileNotFoundError(f"{name}: no LMDB entry {key!r}")
        return decode_image(buf)
    if not isinstance(frame, str):
        raise ValueError("type of image_file should be str or list")        # tracker.py:289
    import cv2 as cv
    im = cv.imread(frame)
    if im is None:
        raise FileNotFoundError(frame)
    return cv.cvtColor(im, cv.COLOR_BGR2RGB)


def results_path(results_dir: str, seq: Sequence) -> str:
    """running.py:20-27: trackingnet / got10k results go into a folder named after the dataset."""
    if seq.dataset in ("trackingnet", "got10k"):
        return os.path.join(results_dir, seq.dataset, seq.name)
    return os.path.join(results_dir, seq.name)


def save_tracker_output(results_dir: str, seq: Sequence, output: dict) -> None:
    """Same files as running.py:_save_tracker_output: boxes truncated to int, tab separated, '%d'; times '%f'."""
    base = results_path(results_dir, seq)
    os.makedirs(os.path.dirname(base), exist_ok=True)
    if output.get("target_bbox"):
        np.savetxt(base + ".txt", np.array(output["target_bbox"]).astype(int), delimiter="\t", fmt="%d")
    if output.get("time"):
        np.savetxt(base + "_time.txt", np.array(output["time"]).astype(float), delimiter="\t", fmt="%f")


class _Slot:
    __slots__ = ("seq", "next_frame", "output", "prefetch", "prefetch_idx")

    def __init__(self):
        self.seq: Optional[Sequence] = None
        self.next_frame = 0
        self.output: Optional[dict] = None
        self.prefetch: Optional[Future] = None          # decode of frame `prefetch_idx`, started while the previous step ran
        self.prefetch_idx = -1


def crop_rows(box, factor: float, H: int) -> Optional[tuple]:
    """Rows [ya, yb) of an H-row frame that sample_target(im, box, factor, .) can read (processing_utils.py:30-48: crop_sz =
    ceil(sqrt(w h) factor), y1 = round(y + h/2 - crop_sz/2) with Python's round); None when the crop is degenerate."""
    x, y, w, h = [float(v) for v in box]
    if not (w * h >= 0):
        return None
    crop_sz = math.ceil(math.sqrt(w * h) * factor)
    if crop_sz < 1:
        return None
    y1 = round(y + 0.5 * h - crop_sz * 0.5)
    ya, yb = max(0, y1), min(H, y1 + crop_sz)
    return (ya, yb) if yb > ya else None


def crop_rect(box, factor: float, H: int, W: int) -> Optional[tuple]:
    """Rows [ya, yb) x columns [xa, xb) of an H x W frame that sample_target(im, box, factor, .) can read: crop_rows for the rows, and
    x1 = round(x + w/2 - crop_sz/2) .. x1 + crop_sz for the columns (processing_utils.py:34-48), widened by one spare column on either
    side so that a boundary pixel never depends on the host's and the device's rounding of x1 agreeing; None when the crop is degenerate
    or misses the frame."""
    rows = crop_rows(box, factor, H)
    if rows is None:
        return None
    x, y, w, h = [float(v) for v in box]
    crop_sz = math.ceil(math.sqrt(w * h) * factor)
    x1 = round(x + 0.5 * w - crop_sz * 0.5)
    xa, xb = max(0, x1 - 1), min(W, x1 + crop_sz + 1)
    return (rows[0], rows[1], xa, xb) if xb > xa else None


class BatchedBackend:
    """The device side of the driver: one initialisation for any set of free slots, one step for the running slots.  Split from the
    scheduler so that the scheduling logic is testable without a GPU.

    Uploads are ROW-STAGED like the batch-1 tracker's (tracker.py `_upload`): a step sends, per slot, only the frame rows its search
    crop can read (the state is known on the host: it is what the previous step returned), packed back to back in one pinned buffer
    and moved with one copy.  The kernels address a frame by a byte offset, so a slot's offset simply points `ya` rows BEFORE its
    packed rows - rows outside [ya, yb) are never read.  Packing runs on a small thread pool (NumPy copies release the GIL)."""

    _PAD = 256           # bytes between packed regions: the gather reads aligned words around a tap (< 16 bytes past a row's end)

    def __init__(self, cfg, state_dict, slots: int, device: Optional[int] = None, blocks_impl: str = "tcgen05", stage_workers: int = 8,
                 row_staging: bool = True, range_fallback: bool = False):
        import torch
        from .batched import BatchedTracker
        self.torch = torch
        # range_fallback: a step recomputes the tracks flagged as out of fp16 range on the fp32 kernels, so they are not dropped
        self.bt = BatchedTracker(cfg, state_dict, max_tracks=slots, device=device, blocks_impl=blocks_impl, range_fallback=range_fallback)
        self.dev = self.bt.device
        self.slots = slots
        self.search_factor = float(cfg.TEST.SEARCH_FACTOR)
        self.template_factor = float(cfg.TEST.TEMPLATE_FACTOR)
        self.row_staging = row_staging
        self._cap = 0
        self._pin = None
        self._devbuf = None
        self._hw = torch.zeros((slots, 2), dtype=torch.int32).pin_memory()
        self._off = torch.zeros((slots,), dtype=torch.int64).pin_memory()
        self._hw_np, self._off_np = self._hw.numpy(), self._off.numpy()        # the same memory, written without tensor indexing
        self._out_pin = torch.zeros((slots, 5), dtype=torch.float64).pin_memory()
        self._state: List[Optional[list]] = [None] * slots          # host copy of every slot's box (what the device holds)
        self._pool = ThreadPoolExecutor(max_workers=stage_workers, thread_name_prefix="vt-stage") if stage_workers > 0 else None
        self._workers = max(1, stage_workers)
        self.bytes_uploaded = 0
        self._slot_ids = torch.zeros((slots,), dtype=torch.int32).pin_memory()
        self._slot_ids_np = self._slot_ids.numpy()

    def _stage(self, frames: List[np.ndarray], rois: Optional[List[Optional[tuple]]] = None):
        """Pack the frames (or, with `rois`, the rows [ya, yb) of each) into one pinned buffer, upload with one copy; returns per-frame
        byte offsets of the (virtual) frame starts inside the device buffer."""
        torch = self.torch
        spans = []
        o = self._PAD
        for i, f in enumerate(frames):
            H, W = f.shape[0], f.shape[1]
            ya, yb = (0, H) if rois is None or rois[i] is None else rois[i]
            nbytes = (yb - ya) * W * 3
            spans.append((o, ya, yb, nbytes))
            o += (nbytes + self._PAD + 15) // 16 * 16
        total = o
        if total > self._cap:
            # sized for every slot holding a whole frame of the largest size seen: pinned allocations cost ~0.4 ms per MB, so the buffers
            # should be allocated once, not grown step by step as more slots fill up
            largest = max(f.shape[0] * f.shape[1] * 3 for f in frames)
            self._cap = max(int(total * 1.25), self.slots * (largest + 2 * self._PAD)) + 1024
            self._pin = torch.empty((self._cap,), dtype=torch.uint8).pin_memory()
            self._devbuf = torch.empty((self._cap,), dtype=torch.uint8, device=self.dev)
            self._devbuf.zero_()
        pin = self._pin.numpy()

        def pack(lo, hi):
            for i in range(lo, hi):
                o, ya, yb, nbytes = spans[i]
                pin[o:o + nbytes] = np.ascontiguousarray(frames[i][ya:yb]).reshape(-1)

        n = len(frames)
        workers = self._workers if self._pool is not None else 1
        # Up to four groups of frames, >= 8 MB each: a group is packed by all workers (one task per worker - a task per frame costs more in
        # hand-over than the copy of a small ROI; NumPy's copy releases the GIL) and its bytes cross the link while the next group is packed.
        groups = max(1, min(4, total // (8 << 20), n))
        g0 = 0
        for g in range(groups):
            g1 = n if g == groups - 1 else max(g0 + 1, (n * (g + 1)) // groups)
            if workers > 1 and g1 - g0 > 1:
                per = (g1 - g0 + workers - 1) // workers
                list(self._pool.map(lambda lo: pack(lo, min(g1, lo + per)), range(g0, g1, per)))
            else:
                pack(g0, g1)
            b0 = 0 if g == 0 else spans[g0][0]
            b1 = total if g == groups - 1 else spans[g1][0]
            self._devbuf[b0:b1].copy_(self._pin[b0:b1], non_blocking=True)
            g0 = g1
        self.bytes_uploaded += total
        # virtual frame start: `ya` rows before the packed rows (never dereferenced outside [ya, yb)); may be negative
        return [o - ya * frames[i].shape[1] * 3 for i, (o, ya, yb, _) in enumerate(spans)]

    def close(self) -> None:
        if self._pool is not None:
            self._pool.shutdown(wait=False)
            self._pool = None

    @staticmethod
    def _check_image(image) -> None:
        if image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != 3:
            raise ValueError("image must be HxWx3 uint8")

    def initialize_many(self, items) -> List[Optional[Exception]]:
        """items = [(slot, image, box), ...] -> per item None or the exception the reference's initialize() would have raised.  One staging
        pass + upload for all of them (only the rows the template crop reads, like a step) and one vt_tracks_init_slots, instead of a
        staging pass, a launch and a blocking status read per sequence."""
        torch = self.torch
        errors: List[Optional[Exception]] = [None] * len(items)
        ok = []
        for k, (slot, image, box) in enumerate(items):
            try:
                self._check_image(image)
                ok.append(k)
            except Exception as e:
                errors[k] = e
        if not ok:
            return errors
        frames = [items[k][1] for k in ok]
        rois = None
        if self.row_staging:
            rois = [crop_rows(items[k][2], self.template_factor, items[k][1].shape[0]) for k in ok]
        offs = self._stage(frames, rois)
        m = len(ok)
        meta = np.zeros((m, 8), dtype=np.float64)               # H, W, offset (exact in fp64: < 2^53), box, slot
        for j, k in enumerate(ok):
            f = frames[j]
            meta[j, 0], meta[j, 1], meta[j, 2] = f.shape[0], f.shape[1], offs[j]
            meta[j, 3:7] = [float(v) for v in items[k][2]]
            meta[j, 7] = items[k][0]
        hw = torch.from_numpy(meta[:, 0:2].astype(np.int32)).to(self.dev)
        off = torch.from_numpy(meta[:, 2].astype(np.int64)).to(self.dev)
        bx = torch.from_numpy(np.ascontiguousarray(meta[:, 3:7])).to(self.dev)
        slots = self.bt._slots(meta[:, 7].astype(np.int64))
        status = self.bt._init_slots(self._devbuf, off, hw, bx, slots)
        codes = status.cpu().numpy()
        for j, k in enumerate(ok):
            code = int(codes[j])
            if code == 1:
                errors[k] = Exception("Too small bounding box.")            # processing_utils.py:32-33
            elif code != 0:
                errors[k] = ValueError("crop lies outside the image (undefined in the reference)")
            else:
                self._state[items[k][0]] = [float(v) for v in items[k][2]]
        return errors

    def step_active(self, slots: List[int], images: List[np.ndarray]) -> np.ndarray:
        """images[j] = next frame of slot slots[j]; stages and steps only those slots.  Returns [len(slots), 5] boxes + confidence, in the
        order of `slots`."""
        torch = self.torch
        ids = check_slots(slots, self.slots)
        n = len(images)
        if n == 0:
            return np.zeros((0, 5))
        rois = None
        if self.row_staging:
            rois = [crop_rows(self._state[t], self.search_factor, f.shape[0]) if self._state[t] is not None else None for t, f in zip(ids, images)]
        offs = self._stage(images, rois)
        hw_np, off_np = self._hw_np, self._off_np
        for i, f in enumerate(images):
            hw_np[i, 0], hw_np[i, 1] = f.shape[0], f.shape[1]
        off_np[:n] = offs
        hw = self._hw[:n].to(self.dev, non_blocking=True)
        off = self._off[:n].to(self.dev, non_blocking=True)
        self._slot_ids_np[:n] = ids
        out = self.bt._step_slots(self._devbuf, off, hw, self._slot_ids[:n].to(self.dev, non_blocking=True), True, False)
        self._out_pin[:n].copy_(out, non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()
        res = self._out_pin[:n].numpy().copy()
        boxes = res[:, :4].tolist()
        good = (res[:, 4] >= 0).tolist()
        for i, t in enumerate(ids):
            if good[i]:                                                # a flagged track keeps its state on the device too
                self._state[t] = boxes[i]
        return res


class MultiSequenceRunner:
    """``run(sequences)``: the batched counterpart of run_dataset + Tracker.run_sequence for one GPU."""

    def __init__(self, backend, slots: int, results_dir: Optional[str] = None, skip_existing: bool = True, verbose: bool = False,
                 read_workers: int = 8):
        """backend: ``initialize_many([(slot, image, box), ...]) -> [None or exception, ...]`` and ``step_active(slots, images) ->
        [len(slots), 5]`` boxes + confidence, as BatchedBackend offers them.
        read_workers: threads that decode frames (SURVEY 8f rank 2, frame ingest: cv.imread + BGR2RGB release the GIL).  The frames of a
        step are decoded in parallel, and the frames of step t + 1 while the device runs step t; 0 = decode on the calling thread."""
        self.backend = backend
        self.slots = [_Slot() for _ in range(slots)]
        self.results_dir = results_dir
        self.skip_existing = skip_existing
        self.verbose = verbose
        self._readers = ThreadPoolExecutor(max_workers=read_workers, thread_name_prefix="vt-read") if read_workers > 0 else None

    def close(self) -> None:
        if self._readers is not None:
            self._readers.shutdown(wait=False, cancel_futures=True)
            self._readers = None

    def _drop(self, slot: _Slot) -> None:
        if slot.prefetch is not None:
            slot.prefetch.cancel()
        slot.seq, slot.output, slot.prefetch, slot.prefetch_idx = None, None, None, -1

    def _step_images(self, active: List[int]) -> Tuple[List[int], List[np.ndarray]]:
        """(slots, images): the running slots of `active` and the next frame of each.  A sequence whose frame cannot be read is reported,
        dropped and left out, like a sequence that raises inside the reference's run_sequence (running.py:135-142)."""
        futs: List[Optional[Future]] = []
        for i in active:
            s = self.slots[i]
            if s.prefetch is not None and s.prefetch_idx == s.next_frame:
                futs.append(s.prefetch)
            elif self._readers is not None:
                futs.append(self._readers.submit(read_image, s.seq.frames[s.next_frame]))
            else:
                futs.append(None)
            s.prefetch, s.prefetch_idx = None, -1
        slots, images = [], []
        for i, fut in zip(active, futs):
            s = self.slots[i]
            try:
                images.append(fut.result() if fut is not None else read_image(s.seq.frames[s.next_frame]))
                slots.append(i)
            except Exception as e:
                print(e)
                self._drop(s)
        return slots, images

    def _prefetch_next(self, active: List[int]) -> None:
        if self._readers is None:
            return
        for i in active:
            s = self.slots[i]
            if s.seq is not None and s.next_frame + 1 < len(s.seq.frames):
                s.prefetch_idx = s.next_frame + 1
                s.prefetch = self._readers.submit(read_image, s.seq.frames[s.prefetch_idx])

    def _finish(self, slot: _Slot, results: Dict[str, dict]) -> None:
        seq, out = slot.seq, slot.output
        if len(out["target_bbox"]) <= 1:                               # tracker.py:148-150
            out.pop("target_bbox")
        results[seq.name] = out
        if self.results_dir is not None:
            save_tracker_output(self.results_dir, seq, out)
        if self.verbose:
            t = float(np.sum(out["time"]))
            print("FPS: {}".format(len(out["time"]) / t if t > 0 else float("inf")))          # running.py:146-150
        self._drop(slot)

    def run(self, sequences: Seq[Sequence]) -> Dict[str, dict]:
        pending = []
        for s in sequences:
            if self.results_dir is not None and self.skip_existing and os.path.isfile(results_path(self.results_dir, s) + ".txt"):
                if self.verbose:
                    print("FPS: {}".format(-1))                        # running.py:116-131: results exist, skip
                continue
            pending.append(s)
        pending.reverse()
        results: Dict[str, dict] = {}
        while True:
            # (re)fill free slots; a sequence whose initialisation fails is reported and skipped (running.py:135-142).  The slots that
            # are free at this point are initialised together (one staging pass, one upload).
            while pending:
                free = [i for i, slot in enumerate(self.slots) if slot.seq is None]
                if not free:
                    break
                batch = []
                t0 = time.time()
                for i in free:
                    if not pending:
                        break
                    seq = pending.pop()
                    try:
                        batch.append((i, seq, read_image(seq.frames[0])))
                    except Exception as e:
                        print(e)
                if not batch:
                    continue
                errors = self.backend.initialize_many([(i, im, seq.init_bbox) for (i, seq, im) in batch])
                dt = (time.time() - t0) / len(batch)
                for (i, seq, im), err in zip(batch, errors):
                    if err is not None:
                        print(err)
                        continue
                    slot = self.slots[i]
                    slot.seq, slot.next_frame = seq, 1
                    slot.output = {"target_bbox": [list(seq.init_bbox)], "time": [dt]}
                    if len(seq.frames) == 1:
                        self._finish(slot, results)
            active = [i for i, s in enumerate(self.slots) if s.seq is not None]
            if not active:
                break
            t0 = time.time()
            active, images = self._step_images(active)                         # minus the sequences whose frame could not be read
            self._prefetch_next(active)                                        # decode step t + 1 while the device runs step t
            boxes = self.backend.step_active(active, images) if active else np.zeros((0, 5))
            # `time`: the reference records the wall time of one sequence's track() call (tracker.py:139-146); a batched step
            # advances every running sequence at once, so each is charged its share of the step - sum(time) over all sequences
            # is the wall time spent tracking, and the printed FPS is this sequence's share of the batched throughput
            dt = (time.time() - t0) / max(1, len(active))
            for j, i in enumerate(active):
                slot = self.slots[i]
                if boxes[j, 4] < 0:
                    # per-track failure flagged by vt_tracks_step (confidence -1, state kept: crop too small / outside the image /
                    # numeric range): the reference's track() would have raised and run_sequence dropped the sequence (running.py:135-142)
                    print(f"{slot.seq.name}: tracking failed at frame {slot.next_frame} (track status != 0), sequence dropped")
                    self._drop(slot)
                    continue
                slot.output["target_bbox"].append([float(v) for v in boxes[j, :4]])
                slot.output["time"].append(dt)
                slot.next_frame += 1
                if slot.next_frame >= len(slot.seq.frames):
                    self._finish(slot, results)
        return results


def run_sequences(sequences: Seq[Sequence], cfg, state_dict, slots: int = 64, results_dir: Optional[str] = None,
                  device: Optional[int] = None, blocks_impl: str = "tcgen05", row_staging: bool = True, range_fallback: bool = False,
                  **kw) -> Dict[str, dict]:
    """Track every sequence; ``slots`` run concurrently on one GPU.  ``range_fallback``: see BatchedTracker."""
    slots = max(1, min(slots, len(sequences)))
    backend = BatchedBackend(cfg, state_dict, slots, device=device, blocks_impl=blocks_impl, row_staging=row_staging,
                             range_fallback=range_fallback)
    runner = MultiSequenceRunner(backend, slots, results_dir=results_dir, **kw)
    try:
        return runner.run(sequences)
    finally:
        runner.close()
        backend.close()
