#!/usr/bin/env python
"""Cost of the range fallback (vt_set_range_fallback) on one GPU; writes one JSON document.

    python tools/range_fallback.py --out profiles/range_fallback_b200.json

zero      1024 tracks on 720p frames with weights that flag nothing, open loop (update_state=0), one tcgen05 engine with the fallback
          switched on and off between rounds, alternated; ms per step from CUDA events over `--steps` steps per round, the spread
          over rounds, and whether the outputs and maps are the same bits.
flagged   1024 tracks, stem conv1 weights x 3e4 (tests/test_gpu_range_fallback.py): a track on a noise frame overflows the fp16
          operand range, a track on a flat frame at the normalisation mean does not.  k = 0, 1, 16, 128 and 1024 tracks on the noise
          frame; ms per step with the fallback on, and the number of items it recomputed per step.
track     batch-1 Vit_dist.track() wall time (host clock, the call ends in a synchronisation) on 720p frames, p50 / p99 over
          `--frames` frames with params.range_fallback on and off, alternated in blocks of 50 frames; nothing is flagged.
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

H, W, F = 720, 1280, 8


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = (v.strip() for v in q.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, steps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def zero(n: int, steps: int, rounds: int) -> dict:
    from oracle import vt_oracle as O
    from vittracker_b200 import FramePool, load_cfg
    from vittracker_b200.engine import Engine
    e = Engine(load_cfg(), max_tracks=n)
    e.load_state_dict(O.make_state_dict(seed=21, stress=True))
    dev = e.device
    pool = FramePool(O.synth_frames(F, H, W, seed=31, smooth=True), dev)
    hw, off = pool.hw(n), pool.offsets(torch.arange(n, device=dev) % F)
    e.tracks_init(pool.data, off, hw, torch.from_numpy(O.synth_boxes(n, H, W, seed=32)).to(dev), 0)
    e.tracks_set_state(torch.from_numpy(O.synth_boxes(n, H, W, seed=33)).to(dev), 0)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    out = {k: torch.empty((n, 5), dtype=torch.float64, device=dev) for k in ("off", "on")}
    det = {k: torch.empty((n, 8), dtype=torch.float64, device=dev) for k in ("off", "on")}

    def run(k):
        e.set_range_fallback(k == "on", counter)
        return lambda: e.tracks_step(pool.data, off, hw, 0, n, out[k], det[k], update_state=False)
    maps = {}
    for k in ("off", "on"):
        f = run(k)
        for _ in range(3):
            f()
        maps[k] = e.tracks_last_maps(0, n)
    torch.cuda.synchronize()
    same = torch.equal(out["off"], out["on"]) and torch.equal(det["off"], det["on"]) and all(
        torch.equal(torch.nan_to_num(maps["off"][q]), torch.nan_to_num(maps["on"][q])) for q in maps["off"])
    ms = {"off": [], "on": []}
    for r in range(rounds):
        for k in (("off", "on") if r % 2 == 0 else ("on", "off")):
            ms[k].append(timed(run(k), steps))
    res = {k: {"ms_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v)), "rounds": v} for k, v in ms.items()}
    res["overhead_pct"] = 100.0 * (res["on"]["ms_mean"] / res["off"]["ms_mean"] - 1.0)
    res["spread_pct_off"] = 100.0 * (res["off"]["ms_max"] - res["off"]["ms_min"]) / res["off"]["ms_mean"]
    res["same_bits"] = bool(same)
    res["flagged_items"] = int(counter.item())
    res.update(tracks=n, steps_per_round=steps)
    return res


def flagged(n: int, steps: int, counts) -> dict:
    from oracle import vt_oracle as O
    from vittracker_b200 import FramePool, load_cfg
    from vittracker_b200.engine import Engine
    sd = O.make_state_dict(seed=5, stress=True)
    sd["patch_embed.net.0.c.weight"] = sd["patch_embed.net.0.c.weight"] * 3e4
    e = Engine(load_cfg(), max_tracks=n)
    e.load_state_dict(sd)
    dev = e.device
    h, w = 480, 640
    flat = np.empty((h, w, 3), np.uint8)
    flat[...] = (124, 116, 104)
    noise = np.random.default_rng(7).integers(0, 256, (h, w, 3), dtype=np.uint8)
    pool = FramePool(np.stack([flat, noise]), dev)
    rng = np.random.default_rng(11)
    boxes = np.stack([rng.uniform(230, 380, n), rng.uniform(150, 260, n), rng.uniform(30, 50, n), rng.uniform(30, 50, n)], 1)
    hw = pool.hw(n)
    e.tracks_init(pool.data, pool.offsets(torch.zeros(n, dtype=torch.int64, device=dev)), hw, torch.from_numpy(boxes).to(dev), 0)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    res = []
    for k in counts:
        idx = torch.zeros(n, dtype=torch.int64, device=dev)
        idx[torch.from_numpy(np.random.default_rng(k).permutation(n)[:k]).to(dev)] = 1
        off = pool.offsets(idx)
        row = {"noise_tracks": int(k)}
        for mode in ("off", "on"):
            e.set_range_fallback(mode == "on", counter)
            f = lambda: e.tracks_step(pool.data, off, hw, 0, n, update_state=False)       # noqa: E731
            for _ in range(3):
                f()
            torch.cuda.synchronize()
            c0 = int(counter.item())
            row[f"ms_{mode}"] = timed(f, steps)
            if mode == "on":
                row["recomputed_per_step"] = (int(counter.item()) - c0) / steps
        res.append(row)
    return {"tracks": n, "steps": steps, "rows": res}


def track_latency(frames: int) -> dict:
    from oracle import vt_oracle as O
    from vittracker_b200 import get_tracker_class, parameters
    sd = O.make_state_dict(seed=21, stress=True)
    seq = O.synth_frames(16, H, W, seed=41, smooth=True)
    box = [float(v) for v in O.synth_boxes(1, H, W, seed=42)[0]]
    trk = {}
    for mode in ("off", "on"):
        p = parameters("vit_48_h32_noKD")
        p.state_dict = sd
        p.range_fallback = mode == "on"
        trk[mode] = get_tracker_class()(p, "synthetic")
        trk[mode].initialize(seq[0], {"init_bbox": box})
    times = {"off": [], "on": []}
    block = 50
    for b in range(-(-frames // block) + 1):
        for mode in (("off", "on") if b % 2 == 0 else ("on", "off")):
            for i in range(block):
                im = seq[1 + (b * block + i) % 15]
                trk[mode].state = box                           # open loop: the same search region every frame
                t0 = time.perf_counter()
                trk[mode].track(im)
                dt = (time.perf_counter() - t0) * 1e3
                if b > 0:                                       # the first block warms up (and captures the CUDA graph)
                    times[mode].append(dt)
    return {k: {"p50_ms": float(np.percentile(v, 50)), "p99_ms": float(np.percentile(v, 99)), "frames": len(v)} for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--frames", type=int, default=500)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("range_fallback.py measures on the GPU; no CUDA device is present")
    doc = {"card": card(), "zero_flagged": zero(1024, a.steps, a.rounds), "flagged": flagged(1024, a.steps, (0, 1, 16, 128, 1024)),
           "track_b1": track_latency(a.frames)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({"zero_flagged": {k: doc["zero_flagged"][k] for k in ("overhead_pct", "spread_pct_off", "same_bits")},
                      "flagged": doc["flagged"]["rows"], "track_b1": doc["track_b1"], "card": doc["card"]}))


if __name__ == "__main__":
    main()
