"""Range fallback without a GPU: the exported symbol and its binding, and the Python arguments that switch it on, from Vit_dist and
run_sequences down to the engine."""
import ctypes as C
import inspect
import os
import re

import numpy as np

from vittracker_b200 import _lib
from vittracker_b200.sequences import Sequence

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_declares_the_call_as_bound():
    header = open(os.path.join(ROOT, "include", "vittrack_b200.h")).read()
    assert re.search(r"int vt_set_range_fallback\(VtHandle h, int32_t enable, int64_t\* counter_dev\);", header)
    assert _lib.SIGNATURES["vt_set_range_fallback"] == (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p])
    assert "vt_set_range_fallback" in header[header.index("#define VT_TRACK_NUMERIC_RANGE"):header.index("#define VT_TRACK_BAD_SLOT")]


def test_library_exports_the_symbol():
    path = _lib.lib_path()
    if not os.path.isfile(path):
        import pytest
        pytest.skip("library not built")
    lib = C.CDLL(path)
    assert hasattr(lib, "vt_set_range_fallback")


def test_python_arguments_default_off():
    from vittracker_b200.batched import BatchedTracker
    from vittracker_b200.engine import Engine
    from vittracker_b200.model import OstrackDistB200
    from vittracker_b200.sequences import BatchedBackend, run_sequences
    for fn in (BatchedTracker.__init__, OstrackDistB200.__init__, BatchedBackend.__init__, run_sequences):
        assert inspect.signature(fn).parameters["range_fallback"].default is False, fn
    assert list(inspect.signature(Engine.set_range_fallback).parameters) == ["self", "enable", "counter"]
    assert isinstance(inspect.getattr_static(BatchedTracker, "fallback_items"), property)


def test_tracker_plumbs_params_range_fallback(monkeypatch):
    import vittracker_b200.tracker as T
    seen = {}

    class Stop(Exception):
        pass

    def fake_build(cfg, **kw):
        seen.update(kw)
        raise Stop

    monkeypatch.setattr(T, "build_ostrack_dist", fake_build)

    class P:
        cfg = type("cfg", (), {})()
    for value, want in ((None, False), (True, True)):
        p = P()
        if value is not None:
            p.range_fallback = value
        p.cfg.MODEL = type("m", (), {"BACKBONE": type("b", (), {"DEPTH": 3})()})()
        seen.clear()
        try:
            T.Vit_dist(p)
        except Stop:
            pass
        assert seen["range_fallback"] is want


def test_driver_hands_the_option_to_the_tracker(monkeypatch):
    """run_sequences -> BatchedBackend -> BatchedTracker: the option reaches the tracker that switches the engine's fallback on (the fake
    tracker stops the backend's construction there)."""
    import vittracker_b200.batched as B
    from vittracker_b200.sequences import run_sequences
    seen = []

    class Stop(Exception):
        pass

    class Tracker:
        def __init__(self, cfg, state_dict, max_tracks, device=None, blocks_impl="tcgen05", range_fallback=False):
            seen.append((max_tracks, blocks_impl, range_fallback))
            raise Stop

    monkeypatch.setattr(B, "BatchedTracker", Tracker)
    seqs = [Sequence(f"s{i}", [np.zeros((8, 8, 3), np.uint8)] * 2, [1.0, 2.0, 3.0, 4.0]) for i in range(3)]
    for kw in ({}, {"range_fallback": True}, {"range_fallback": False, "blocks_impl": "tcgen05_3term"}):
        try:
            run_sequences(seqs, None, {}, slots=2, **kw)
        except Stop:
            pass
    assert seen == [(2, "tcgen05", False), (2, "tcgen05", True), (2, "tcgen05_3term", False)]
