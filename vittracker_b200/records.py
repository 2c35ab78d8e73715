"""Track records: a whole track state (box + cached template tokens) as the fixed-size, self-checking byte image of
include/vittrack_b200.h (vt_tracks_export / vt_tracks_import), so that a track can be saved, restored, forked, or moved to another
slot, tracker or GPU and continue bit for bit.

The constants mirror the header; ``checksum`` and ``weights_fingerprint`` restate the header's two functions in numpy, so that a
record can be checked and a handle's fingerprint predicted on the host."""
from __future__ import annotations

import struct
from typing import Mapping, Optional

import numpy as np
import torch

VT_TRACK_RECORD_MAGIC = 0x52545456            # "VTTR" as little-endian bytes
VT_TRACK_RECORD_VERSION = 1
VT_TRACK_RECORD_HEADER_BYTES = 64             # header fields and the box, before the template tokens
VT_TRACK_BAD_RECORD = 5
TEMPLATE_ROWS = 64
FINGERPRINT_VERSION = b"vittrack_b200 weights v1"

_GOLDEN = np.uint64(0x9E3779B97F4A7C15)
_FNV_BASIS, _FNV_PRIME, _M64 = 0xCBF29CE484222325, 0x100000001B3, (1 << 64) - 1
_HEADER = struct.Struct("<IIQiiQ")            # magic, version, fingerprint, C, rows, checksum (32 bytes)


def record_bytes(C: int) -> int:
    """R, the size of one record at embed dim C."""
    return VT_TRACK_RECORD_HEADER_BYTES + 256 * int(C)


def _splitmix64(z: np.ndarray) -> np.ndarray:
    z = z + _GOLDEN
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def checksum(payload: np.ndarray) -> int:
    """The header's payload checksum: sum mod 2^64 of splitmix64(w_k + k * 0x9E3779B97F4A7C15) over the payload's little-endian uint64
    words (``payload`` is bytes [32, R) of a record: box, then tokens, as uint8)."""
    w = np.ascontiguousarray(payload, dtype=np.uint8).view("<u8").astype(np.uint64)
    with np.errstate(over="ignore"):
        k = np.arange(w.size, dtype=np.uint64)
        return int(_splitmix64(w + k * _GOLDEN).sum(dtype=np.uint64))


def _fnv_words(stream: bytes) -> int:
    stream += b"\0" * (-len(stream) % 8)
    h = _FNV_BASIS
    for w in np.frombuffer(stream, dtype="<u8").tolist():
        h = ((h ^ w) * _FNV_PRIME) & _M64
    return h


def template_route(cfg, depth: int, blocks_impl: str) -> int:
    """The header's template route id: 0 for vit_48_h32 (every blocks_impl), else 1 simt, 2 tensor-core GEMMs, 3 split-image GEMMs."""
    C, heads, hc = int(cfg.MODEL.BACKBONE.CHANNELS), int(cfg.MODEL.BACKBONE.HEADS), int(cfg.MODEL.HEAD.NUM_CHANNELS)
    if (C, heads, int(depth), hc) == (48, 1, 3, 32):
        return 0
    if blocks_impl == "simt":
        return 1
    return 3 if C % 128 == 0 else 2


def weights_fingerprint(cfg, state_dict: Mapping[str, torch.Tensor], depth: int = 3, blocks_impl: str = "tcgen05") -> int:
    """The fingerprint ``Engine(cfg, depth=depth, blocks_impl=blocks_impl).load_state_dict(state_dict)`` gives its handle: the tensors
    the handle keeps (known floating-point keys; ``*.num_batches_tracked`` and unknown keys dropped), plus the Hann window
    ``tracker.output_window`` that Engine.load_state_dict always sets, hashed as the header specifies."""
    from .engine import hann2d_window
    from .weights import param_shapes
    known = {k for k in param_shapes(cfg, depth) if not k.endswith("num_batches_tracked")} | {"tracker.output_window"}
    held = {}
    for name, t in state_dict.items():
        if torch.is_tensor(t) and t.is_floating_point() and name in known:
            held[name] = t.detach().to("cpu", torch.float32).contiguous()
    held["tracker.output_window"] = hann2d_window(int(cfg.TEST.SEARCH_SIZE) // 16).contiguous()
    parts = [FINGERPRINT_VERSION,
             struct.pack("<8i", int(cfg.MODEL.BACKBONE.CHANNELS), int(cfg.MODEL.BACKBONE.HEADS), int(depth), 4,
                         int(cfg.MODEL.HEAD.NUM_CHANNELS), int(cfg.MODEL.BACKBONE.STRIDE), int(cfg.TEST.TEMPLATE_SIZE),
                         int(cfg.TEST.SEARCH_SIZE)),
             struct.pack("<2d", float(cfg.TEST.TEMPLATE_FACTOR), float(cfg.TEST.SEARCH_FACTOR)),
             struct.pack("<i", template_route(cfg, depth, blocks_impl))]
    for name in sorted(held, key=lambda s: s.encode()):
        t = held[name]
        parts += [name.encode() + b"\0", struct.pack(f"<i{t.dim()}q", t.dim(), *t.shape), t.numpy().astype("<f4").tobytes()]
    return _fnv_words(b"".join(parts))


def describe_rejection(record, fingerprint: int, C: int) -> Optional[str]:
    """Why a handle with this fingerprint and embed dim C rejects ``record`` (one record, uint8), or None if it accepts it."""
    r = np.asarray(record.cpu() if torch.is_tensor(record) else record, dtype=np.uint8).reshape(-1)
    if r.size < VT_TRACK_RECORD_HEADER_BYTES:
        return f"record of {r.size} bytes is shorter than its header"
    magic, version, fp, rc, rows, cs = _HEADER.unpack(r[:32].tobytes())
    if magic != VT_TRACK_RECORD_MAGIC:
        return f"bad magic 0x{magic:08x} (not a track record, or exported from a bad slot)"
    if version != VT_TRACK_RECORD_VERSION:
        return f"record version {version}, this library reads version {VT_TRACK_RECORD_VERSION}"
    if rc != C or r.size < record_bytes(C):
        return f"record embed dim C = {rc} ({r.size} bytes), this handle has C = {C}"
    if rows != TEMPLATE_ROWS:
        return f"record holds {rows} template rows, expected {TEMPLATE_ROWS}"
    if fp != fingerprint:
        return f"weights fingerprint 0x{fp:016x} of the exporting handle differs from this handle's 0x{fingerprint:016x}"
    if checksum(r[32:record_bytes(C)]) != cs:
        return "payload checksum mismatch (the record was altered)"
    if not np.isfinite(r[32:64].view("<f8")).all():
        return "non-finite box"
    return None


class TrackRecords:
    """n exported tracks: ``records`` uint8 [n, R] (device or host) and ``frame_hw`` int32 [n, 2], the frame size each track was
    stepped on (BatchedTracker keeps it per slot)."""

    def __init__(self, records: torch.Tensor, frame_hw: torch.Tensor):
        if records.dtype != torch.uint8 or records.dim() != 2 or (records.shape[1] - VT_TRACK_RECORD_HEADER_BYTES) % 256:
            raise ValueError(f"records: expected uint8 [n, 64 + 256 C], got {records.dtype} {tuple(records.shape)}")
        if frame_hw.dtype != torch.int32 or tuple(frame_hw.shape) != (records.shape[0], 2):
            raise ValueError(f"frame_hw: expected int32 [{records.shape[0]}, 2]")
        self.records, self.frame_hw = records, frame_hw

    def __len__(self) -> int:
        return int(self.records.shape[0])

    @property
    def C(self) -> int:
        return (int(self.records.shape[1]) - VT_TRACK_RECORD_HEADER_BYTES) // 256

    @property
    def device(self) -> torch.device:
        return self.records.device

    def to(self, device) -> "TrackRecords":
        return TrackRecords(self.records.to(device).contiguous(), self.frame_hw.to(device).contiguous())

    def cpu(self) -> "TrackRecords":
        return self.to("cpu")

    @property
    def fingerprint(self) -> Optional[int]:
        """The weights fingerprint in the headers of the records with a valid magic (None if there are none)."""
        head = self.records[:, :16].cpu().numpy()
        magic, fp = head[:, :4].copy().view("<u4")[:, 0], head[:, 8:16].copy().view("<u8")[:, 0]
        fps = {int(v) for v in fp[magic == VT_TRACK_RECORD_MAGIC]}
        if len(fps) > 1:
            raise ValueError(f"records from {len(fps)} different weights fingerprints")
        return fps.pop() if fps else None

    def save(self, path) -> None:
        with open(path, "wb") as f:                 # a file object: numpy adds no ".npz" to the name
            np.savez(f, records=self.records.cpu().numpy(), frame_hw=self.frame_hw.cpu().numpy())

    @classmethod
    def load(cls, path, device="cpu") -> "TrackRecords":
        with np.load(path) as z:
            return cls(torch.from_numpy(z["records"]), torch.from_numpy(z["frame_hw"])).to(device)
