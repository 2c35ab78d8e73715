"""Slot lists without a device: the C ABI's exports and host-side argument checks, the host validation of a slot sequence, and the
sequence runner's use of a backend's step_active (only the running slots, no parking, the same results)."""
import ctypes as C

import numpy as np
import pytest

from test_sequences import FakeBackend, _frames
from vittracker_b200.batched import check_slots
from vittracker_b200.sequences import MultiSequenceRunner, Sequence


def test_slot_entry_points_are_exported_and_refuse_bad_arguments():
    from vittracker_b200 import _lib
    lib = _lib.load()
    for name in ("vt_tracks_init_slots", "vt_tracks_step_slots"):
        assert hasattr(lib, name)
    z = C.c_void_p(0)
    one = C.c_void_p(8)                                            # never dereferenced: the checks fail first
    # null handle
    assert lib.vt_tracks_init_slots(z, one, one, one, one, one, 1, z, z) == -1
    assert lib.vt_tracks_step_slots(z, one, one, one, one, 1, one, z, 1, z) == -1
    # n < 0, null slots (the handle check comes first, and without a device there is no handle)
    assert lib.vt_tracks_init_slots(z, one, one, one, one, one, -1, z, z) == -1
    assert lib.vt_tracks_step_slots(z, one, one, one, z, 1, one, z, 1, z) == -1


def test_host_slot_validation():
    assert check_slots([3, 0, 2], 4) == [3, 0, 2]
    assert check_slots(np.array([1, 0], dtype=np.int64), 2) == [1, 0]
    assert check_slots([], 1) == []
    for bad in ([-1], [4], [0, 5, 1]):
        with pytest.raises(ValueError, match="outside"):
            check_slots(bad, 4)
    with pytest.raises(ValueError, match="twice"):
        check_slots([1, 2, 1], 4)


class ActiveBackend(FakeBackend):
    """FakeBackend with step_active: steps only the listed slots and checks that they are exactly the running ones."""

    def __init__(self, slots):
        super().__init__(slots)
        self.runner = None
        self.calls = []

    def park(self, slot):
        raise AssertionError("park called on a backend with step_active")

    def step_active(self, slots, images):
        running = [i for i, s in enumerate(self.runner.slots) if s.seq is not None]
        assert list(slots) == running and len(images) == len(slots)
        self.calls.append(list(slots))
        out = np.zeros((len(slots), 5))
        for j, (i, im) in enumerate(zip(slots, images)):
            self.state[i][0] += 1.0
            self.log.append((i, int(im[0, 0, 0])))
            out[j, :4] = self.state[i]
            out[j, 4] = 0.5
        return out


def test_runner_with_step_active_matches_the_range_step(tmp_path):
    lengths = [5, 1, 3, 7, 2, 4, 6]
    seqs = [Sequence(f"s{i}", _frames(n, i), [10.0 * i + 0.7, 5.9, 20.5, 30.2]) for i, n in enumerate(lengths)]
    seqs.append(Sequence("bad", _frames(3, 9), [1.0, 1.0, 0.0, 5.0]))
    ref = MultiSequenceRunner(FakeBackend(3), 3).run(seqs)
    be = ActiveBackend(3)
    runner = MultiSequenceRunner(be, 3)
    be.runner = runner
    got = runner.run(seqs)
    assert set(got) == set(ref)
    for name in ref:                                               # "time" is wall clock
        assert got[name].get("target_bbox") == ref[name].get("target_bbox") and len(got[name]["time"]) == len(ref[name]["time"])
    assert sum(len(c) for c in be.calls) == sum(n - 1 for n in lengths)
    assert any(len(c) < 3 for c in be.calls)
