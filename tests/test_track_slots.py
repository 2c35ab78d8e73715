"""Slot lists without a device: the C ABI's exports and host-side argument checks, and the host validation of a slot sequence.  The
sequence runner's steps over exactly the running slots are checked by the fake backend of test_sequences.py."""
import ctypes as C

import numpy as np
import pytest

from vittracker_b200.batched import check_slots


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
