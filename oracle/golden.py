"""Format of tests/golden/*.npz: arrays recorded from the reference, and seeded inputs the oracle regenerates bit for bit.

A seeded input (synthetic weights, synthetic frames) is stored as one entry ``seeded::<key>`` instead of its arrays: a JSON string
{"fn", "kw", "sha256"}.  ``fn`` is ``make_state_dict`` (the entry stands for the arrays ``<key><name>``, one per parameter) or
``synth_frames`` (the array ``<key>``), ``kw`` its keyword arguments and ``sha256`` the digest of the arrays the reference was run on.
load() regenerates them and fails if the digest differs, so the tests see exactly the recorded inputs while every file stays small.
"""
from __future__ import annotations

import hashlib
import json
from typing import Dict

import numpy as np

from oracle import vt_oracle as O

PREFIX = "seeded::"


def _generate(fn: str, kw: dict, key: str) -> Dict[str, np.ndarray]:
    if fn == "make_state_dict":
        return {key + k: v.numpy() for k, v in O.make_state_dict(**kw).items()}
    if fn == "synth_frames":
        return {key: O.synth_frames(**kw)}
    raise ValueError(f"unknown generator {fn!r}")


def digest(arrays: Dict[str, np.ndarray]) -> str:
    h = hashlib.sha256()
    for k in sorted(arrays):
        a = np.ascontiguousarray(arrays[k])
        h.update(f"{k} {a.dtype.str} {a.shape}\n".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def seeded(fn: str, key: str, **kw) -> Dict[str, np.ndarray]:
    """The entry that stands for O.<fn>(**kw) in a golden file (pass it to np.savez_compressed with the recorded arrays)."""
    return {PREFIX + key: np.array(json.dumps({"fn": fn, "kw": kw, "sha256": digest(_generate(fn, kw, key))}))}


def load(path: str) -> Dict[str, np.ndarray]:
    """Every array of a golden file, seeded inputs regenerated and checked against their recorded digest."""
    out = {}
    with np.load(path) as z:
        for name in z.files:
            if not name.startswith(PREFIX):
                out[name] = z[name]
                continue
            spec = json.loads(str(z[name]))
            arrays = _generate(spec["fn"], spec["kw"], name[len(PREFIX):])
            if digest(arrays) != spec["sha256"]:
                raise AssertionError(f"{path}: {spec['fn']}(**{spec['kw']}) no longer reproduces the recorded input {name}")
            out.update(arrays)
    return out
