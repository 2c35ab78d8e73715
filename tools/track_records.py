#!/usr/bin/env python
"""Cost of moving whole track states as records (vt_tracks_export* / vt_tracks_import*) on one GPU; writes one JSON document.

    python tools/track_records.py --out profiles/track_records_b200.json

device       export + import of n tracks: vit_48_h32 at 1024 tracks, the widest configuration (C 768, 12 heads, depth 12, head 256) at
             256 and 4096.  Range and slot-list calls (a shuffled list), ms per call from CUDA events over `--iters` calls after a
             warm-up, and the record bytes moved (an export writes n R bytes, an import reads them).  The tracks need no
             initialisation: a never-initialised slot exports the zero box and whatever its template rows hold, and imports back.
host         the records of 1024 vit_48_h32 tracks and 256 widest tracks to pinned host memory and back (host clock around work ending
             in a device synchronisation).
fingerprint  vt_finalize_weights of the widest configuration (381 MB of fp32 weights), host clock: it packs, uploads and hashes the
             weights (the fingerprint is the word-wise FNV-1a pass over the caller's tensors).
The card's name and power limit are read in the same process as the measurements."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = (v.strip() for v in q.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def engine(widest: bool, max_tracks: int):
    from oracle import vt_oracle as O
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    from vittracker_b200.weights import random_init_state_dict
    cfg = load_cfg()
    depth = 3
    if widest:
        cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.HEAD.NUM_CHANNELS, depth = 768, 12, 256, 12
        sd = random_init_state_dict(cfg, depth, torch.Generator().manual_seed(3))
    else:
        sd = O.make_state_dict(seed=21, stress=True)
    e = Engine(cfg, max_tracks=max_tracks, depth=depth)
    t0 = time.perf_counter()
    e.load_state_dict(sd)
    load_s = time.perf_counter() - t0
    return e, sd, load_s


def timed(fn, iters: int) -> float:
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def device_costs(e, n: int, iters: int) -> dict:
    dev, R = e.device, e.track_record_bytes
    rec = torch.empty((n, R), dtype=torch.uint8, device=dev)
    slots = torch.randperm(e.max_tracks, device=dev)[:n].to(torch.int32)
    e.tracks_export(0, n, out=rec)
    out = {"tracks": n, "record_bytes": R, "bytes_per_call": n * R}
    out["export_ms"] = timed(lambda: e.tracks_export(0, n, out=rec), iters)
    out["import_ms"] = timed(lambda: e.tracks_import(rec, first=0), iters)
    out["export_slots_ms"] = timed(lambda: e.tracks_export_slots(slots, out=rec), iters)
    out["import_slots_ms"] = timed(lambda: e.tracks_import_slots(rec, slots), iters)
    st = e.tracks_import_slots(rec, slots)
    out["all_accepted"] = bool((st == 0).all().item())
    for k in ("export", "import"):
        out[f"{k}_GBps"] = n * R / (out[f"{k}_ms"] * 1e6)
    return out


def host_round_trip(e, n: int, iters: int) -> dict:
    rec = e.tracks_export(0, n)
    pinned = torch.empty(rec.shape, dtype=torch.uint8).pin_memory()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        t0 = time.perf_counter()
        pinned.copy_(rec)
        rec.copy_(pinned)
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    return {"tracks": n, "bytes": int(rec.numel()), "round_trip_ms_median": float(np.median(times)),
            "round_trip_ms_min": float(np.min(times))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    doc = {"card": card(), "device": [], "host": []}
    e, _, _ = engine(False, 1024)
    doc["device"].append({"config": "vit_48_h32", **device_costs(e, 1024, args.iters)})
    doc["host"].append({"config": "vit_48_h32", **host_round_trip(e, 1024, 20)})
    del e
    e, sd, load_s = engine(True, 4096)
    for n in (256, 4096):
        doc["device"].append({"config": "widest", **device_costs(e, n, args.iters)})
    doc["host"].append({"config": "widest", **host_round_trip(e, 256, 10)})
    finals = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e._check(e.lib.vt_finalize_weights(e.handle, e._stream()))
        finals.append((time.perf_counter() - t0) * 1e3)
    weight_bytes = sum(t.numel() * 4 for t in sd.values() if t.is_floating_point())
    doc["fingerprint"] = {"config": "widest", "weight_bytes": weight_bytes, "finalize_ms": finals, "load_state_dict_s": load_s}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc, indent=1))


if __name__ == "__main__":
    main()
