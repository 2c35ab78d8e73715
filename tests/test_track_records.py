"""Track records without a device: the header's declarations and constants against the binding and records.py, the exports and
host argument checks of the C ABI, the numpy fingerprint and checksum restatements, TrackRecords files, and the argument checks of
BatchedTracker.import_tracks / Vit_dist.restore on a fake engine."""
import ctypes as C
import os
import re
import types

import numpy as np
import pytest
import torch

from vittracker_b200 import _lib, load_cfg
from vittracker_b200 import records as REC
from vittracker_b200.weights import random_init_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALLS = ("vt_weights_fingerprint", "vt_track_record_bytes", "vt_tracks_export", "vt_tracks_export_slots", "vt_tracks_import",
         "vt_tracks_import_slots")


def _header():
    with open(os.path.join(ROOT, "include", "vittrack_b200.h")) as f:
        return f.read()


def test_header_declares_the_calls_as_bound():
    h = _header()
    for name in CALLS:
        m = re.search(r"\bint " + name + r"\(([^;]*)\);", h)
        assert m, name
        assert len(m.group(1).split(",")) == len(_lib.SIGNATURES[name][1]), name
        assert _lib.SIGNATURES[name][0] is C.c_int


def test_header_constants_match_records_py():
    h = _header()
    define = lambda k: int(re.search(r"#define " + k + r"\s+(0x[0-9a-fA-F]+|\d+)", h).group(1), 0)
    assert define("VT_TRACK_RECORD_MAGIC") == REC.VT_TRACK_RECORD_MAGIC == int.from_bytes(b"VTTR", "little")
    assert define("VT_TRACK_RECORD_VERSION") == REC.VT_TRACK_RECORD_VERSION
    assert define("VT_TRACK_RECORD_HEADER_BYTES") == REC.VT_TRACK_RECORD_HEADER_BYTES
    assert define("VT_TRACK_BAD_RECORD") == REC.VT_TRACK_BAD_RECORD == _lib.VT_TRACK_BAD_RECORD
    assert h.index("#define VT_TRACK_BAD_RECORD") > h.index("#define VT_TRACK_BAD_SLOT")
    assert REC.FINGERPRINT_VERSION.decode() in h
    assert REC.record_bytes(48) == 12352 and REC.record_bytes(768) == 196672


def test_entry_points_are_exported_and_refuse_bad_arguments():
    lib = _lib.load()
    for name in CALLS:
        assert hasattr(lib, name)
    z, one = C.c_void_p(0), C.c_void_p(16)                         # never dereferenced: the handle check fails first
    fp, rb = C.c_uint64(), C.c_int64()
    assert lib.vt_weights_fingerprint(z, C.byref(fp)) == -1
    assert lib.vt_track_record_bytes(z, C.byref(rb)) == -1
    assert lib.vt_tracks_export(z, 0, 1, one, z) == -1
    assert lib.vt_tracks_export_slots(z, one, 1, one, z, z) == -1
    assert lib.vt_tracks_import(z, one, 0, 1, z, z) == -1
    assert lib.vt_tracks_import_slots(z, one, one, 1, z, z) == -1


def _splitmix_ref(z):
    m = (1 << 64) - 1
    z = (z + 0x9E3779B97F4A7C15) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return z ^ (z >> 31)


def test_checksum_known_answer_and_position_sensitivity():
    # splitmix64(0) is the first output of the reference generator seeded with 0
    assert _splitmix_ref(0) == 0xE220A8397B1DCDAF
    payload = np.arange(4 * 8 + 48 * 4, dtype=np.uint8)
    words = payload.view("<u8").tolist()
    ref = sum(_splitmix_ref((w + k * 0x9E3779B97F4A7C15) & ((1 << 64) - 1)) for k, w in enumerate(words)) & ((1 << 64) - 1)
    assert REC.checksum(payload) == ref
    assert REC.checksum(np.zeros(16, np.uint8)) == (_splitmix_ref(0) + _splitmix_ref(0x9E3779B97F4A7C15)) & ((1 << 64) - 1)
    swapped = payload.view("<u8").copy()
    swapped[[3, 7]] = swapped[[7, 3]]                               # the same words at other positions
    assert REC.checksum(swapped.view(np.uint8)) != REC.checksum(payload)
    flipped = payload.copy()
    flipped[100] ^= 1
    assert REC.checksum(flipped) != REC.checksum(payload)


def _cfg(C=48, heads=1, hc=32):
    cfg = load_cfg()
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.HEAD.NUM_CHANNELS = C, heads, hc
    return cfg


def test_fingerprint_restatement_properties():
    cfg = _cfg()
    sd = random_init_state_dict(cfg, 3, torch.Generator().manual_seed(4))
    base = REC.weights_fingerprint(cfg, sd)
    assert REC.weights_fingerprint(cfg, dict(reversed(list(sd.items())))) == base              # insertion order
    no_nbt = {k: v for k, v in sd.items() if not k.endswith("num_batches_tracked")}
    assert REC.weights_fingerprint(cfg, no_nbt) == base
    nbt = dict(sd)
    nbt["patch_embed.net.0.bn.num_batches_tracked"] = torch.tensor(12345)
    assert REC.weights_fingerprint(cfg, nbt) == base
    assert REC.weights_fingerprint(cfg, {**sd, "unknown.weight": torch.ones(3)}) == base         # unknown keys are not held
    for impl in ("simt", "tcgen05_3term"):                                                       # one template route on vit_48_h32
        assert REC.weights_fingerprint(cfg, sd, blocks_impl=impl) == base
    # one ulp of one value
    for key in ("blocks.1.mlp.fc2.weight", "pos_embed_z", "box_head.conv5_size.bias"):
        t = sd[key].clone().reshape(-1)
        t[1] = torch.nextafter(t[1], torch.tensor(np.inf))
        assert REC.weights_fingerprint(cfg, {**sd, key: t.reshape(sd[key].shape)}) != base, key
    # a renamed tensor (a different name of the same shape)
    a, b = "blocks.0.norm1.weight", "blocks.0.norm2.weight"
    swapped = {**sd, a: sd[b] * 0.5, b: sd[a]}
    assert REC.weights_fingerprint(cfg, swapped) != base
    # result-relevant configuration fields; max_tracks / chunk_tracks are not part of the configuration it reads
    for field, value in (("TEST.SEARCH_FACTOR", 4.5), ("TEST.TEMPLATE_FACTOR", 2.5), ("MODEL.BACKBONE.STRIDE", 8)):
        c2 = load_cfg()
        node, leaf = c2, field.split(".")
        for k in leaf[:-1]:
            node = node[k]
        node[leaf[-1]] = value
        assert REC.weights_fingerprint(c2, sd) != base, field
    assert REC.weights_fingerprint(cfg, sd, depth=2) != base
    # shape: the same values under another shape need another configuration; the routes of the generic path differ
    g = _cfg(128, 2, 64)
    sdg = random_init_state_dict(g, 1, torch.Generator().manual_seed(5))
    fps = {impl: REC.weights_fingerprint(g, sdg, depth=1, blocks_impl=impl) for impl in ("simt", "tcgen05", "tcgen05_3term")}
    assert fps["simt"] != fps["tcgen05"] == fps["tcgen05_3term"]
    assert REC.template_route(g, 1, "tcgen05") == 3 and REC.template_route(_cfg(96, 3, 64), 2, "tcgen05") == 2
    assert REC.template_route(cfg, 3, "simt") == 0


def test_fingerprint_hashes_shape():
    cfg = _cfg()
    sd = random_init_state_dict(cfg, 3, torch.Generator().manual_seed(4))
    h0 = REC.weights_fingerprint(cfg, sd)
    # the hashed stream of a tensor is name, ndim, shape, data: the same bytes under another shape change the fingerprint.  Such a
    # tensor never reaches a handle (vt_set_tensor checks shapes), so the restatement is probed below its filter.
    held = {"x": torch.ones(2, 3)}
    s1 = REC._fnv_words(b"x\0" + np.array([2], "<i4").tobytes() + np.array([2, 3], "<i8").tobytes() + held["x"].numpy().tobytes())
    s2 = REC._fnv_words(b"x\0" + np.array([2], "<i4").tobytes() + np.array([3, 2], "<i8").tobytes() + held["x"].numpy().tobytes())
    assert s1 != s2 and h0 != 0


def test_describe_rejection_and_track_records_file(tmp_path):
    C_ = 48
    R = REC.record_bytes(C_)
    rng = np.random.default_rng(3)
    rec = np.zeros(R, np.uint8)
    rec[32:64] = np.array([10.0, 20.0, 30.0, 40.0], "<f8").view(np.uint8)
    rec[64:] = rng.standard_normal(64 * C_).astype("<f4").view(np.uint8)
    fp = 0x0123456789ABCDEF
    rec[:32] = np.frombuffer(REC._HEADER.pack(REC.VT_TRACK_RECORD_MAGIC, 1, fp, C_, 64, REC.checksum(rec[32:])), np.uint8)
    assert REC.describe_rejection(rec, fp, C_) is None
    assert "fingerprint" in REC.describe_rejection(rec, fp + 1, C_)
    assert "embed dim" in REC.describe_rejection(rec, fp, 96)
    for off, word in ((0, "magic"), (4, "version"), (20, "rows"), (24, "checksum"), (40, "checksum"), (5000, "checksum")):
        bad = rec.copy()
        bad[off] ^= 0x10
        assert word in REC.describe_rejection(bad, fp, C_), off
    recs = np.stack([rec, np.zeros(R, np.uint8)])
    tr = REC.TrackRecords(torch.from_numpy(recs), torch.tensor([[720, 1280], [0, 0]], dtype=torch.int32))
    assert tr.fingerprint == fp and len(tr) == 2 and tr.C == C_
    path = tmp_path / "tracks.rec"
    tr.save(path)
    back = REC.TrackRecords.load(path)
    assert torch.equal(back.records, tr.records) and torch.equal(back.frame_hw, tr.frame_hw)
    with pytest.raises(ValueError):
        REC.TrackRecords(torch.zeros((2, 100), dtype=torch.uint8), torch.zeros((2, 2), dtype=torch.int32))


class FakeEngine:
    """Records every call; the argument checks must raise before any."""

    def __init__(self, C=48):
        self.C, self.calls, self.device = C, [], torch.device("cpu")
        self.track_record_bytes = REC.record_bytes(C)
        self.weights_fingerprint = 7

    def __getattr__(self, name):
        if name.startswith("tracks_"):
            def call(*a, **k):
                self.calls.append(name)
                raise AssertionError(f"{name} called")
            return call
        raise AttributeError(name)


def _batched(engine):
    from vittracker_b200.batched import BatchedTracker
    bt = object.__new__(BatchedTracker)
    bt.engine, bt.device, bt.max_tracks, bt.n = engine, engine.device, 4, 0
    bt._slot_hw = torch.zeros((5, 2), dtype=torch.int32)
    return bt


def test_import_tracks_argument_errors_before_any_engine_call():
    eng = FakeEngine()
    bt = _batched(eng)
    R = eng.track_record_bytes
    hw = torch.zeros((2, 2), dtype=torch.int32)
    cases = [
        ("not records", torch.zeros((2, R), dtype=torch.uint8)),
        ("width", REC.TrackRecords(torch.zeros((2, REC.record_bytes(96)), dtype=torch.uint8), hw)),
        ("non-contiguous", REC.TrackRecords(torch.zeros((R, 2), dtype=torch.uint8).t(), hw)),
        ("device", REC.TrackRecords(torch.zeros((2, R), dtype=torch.uint8, device="meta"), hw)),
        ("too many", REC.TrackRecords(torch.zeros((5, R), dtype=torch.uint8), torch.zeros((5, 2), dtype=torch.int32))),
    ]
    for what, arg in cases:
        with pytest.raises(ValueError):
            bt.import_tracks(arg)
    with pytest.raises(ValueError):
        REC.TrackRecords(torch.zeros((2, R), dtype=torch.int8), hw)                          # dtype
    ok = REC.TrackRecords(torch.zeros((2, R), dtype=torch.uint8), hw)
    with pytest.raises(ValueError):
        bt.import_tracks(ok, slots=[0, 0])                                                    # slot listed twice (host list)
    with pytest.raises(ValueError):
        bt.import_tracks(ok, slots=[0, 1, 2])                                                 # slots for 2 records
    assert eng.calls == []


def test_vit_dist_restore_argument_errors():
    from vittracker_b200.tracker import Vit_dist
    eng = FakeEngine()
    t = object.__new__(Vit_dist)
    t.engine, t._dev = eng, torch.device("cpu")
    with pytest.raises(ValueError, match="bytes"):
        t.restore({"record": b"\0" * 100, "state": [1, 2, 3, 4], "frame_id": 3, "z_patch_arr": np.zeros((1,))})
    assert eng.calls == []
    t.state = None
    with pytest.raises(RuntimeError):
        t.snapshot()
