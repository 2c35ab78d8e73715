#!/usr/bin/env python
"""Cost of stepping tracks by slot list (vt_tracks_*_slots) on one GPU; writes one JSON document.

    python tools/track_slots.py --out profiles/track_slots_b200.json [--bench BEFORE.jsonl AFTER.jsonl]

overhead  1024 tracks on 720p frames, open loop (update_state=0: every step sees the same state), vt_tracks_step_slots with the
          identity slot list against vt_tracks_step over [0, 1024), alternated in one process; ms per step from CUDA events over
          `--steps` steps per round, and whether the outputs, detail rows and maps are the same bits.
churn     4096 slots with 100 %, 50 % and 25 % of them live.  Each step about 2 % of the live tracks end and as many start in
          random free slots (closed loop).  slot path: one vt_tracks_init_slots for the new tracks, one vt_tracks_step_slots over
          the live slots.  range path (what a caller of the range calls does): one vt_tracks_init per run of consecutive new
          slots, the ended slots parked on a dummy frame the same way, one vt_tracks_step over [0, highest live slot].  Live
          frames per second = live tracks stepped / wall time, each step ending in a device synchronisation (the host's bookkeeping
          is part of the cost).
bench     bench.py result lines recorded before and after the change (alternated by the caller), embedded as given.
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


def setup(max_tracks: int):
    from oracle import vt_oracle as O
    from vittracker_b200 import FramePool, load_cfg
    from vittracker_b200.engine import Engine
    e = Engine(load_cfg(), max_tracks=max_tracks)
    e.load_state_dict(O.make_state_dict(seed=21, stress=True))
    pool = FramePool(O.synth_frames(F, H, W, seed=31, smooth=True), e.device)
    return e, pool, O


def overhead(n: int, steps: int, rounds: int) -> dict:
    e, pool, O = setup(n)
    dev = e.device
    hw = pool.hw(n)
    off = pool.offsets(torch.arange(n, device=dev) % F)
    e.tracks_init(pool.data, off, hw, torch.from_numpy(O.synth_boxes(n, H, W, seed=32)).to(dev), 0)
    e.tracks_set_state(torch.from_numpy(O.synth_boxes(n, H, W, seed=33)).to(dev), 0)
    ident = torch.arange(n, dtype=torch.int32, device=dev)
    out = {k: torch.empty((n, 5), dtype=torch.float64, device=dev) for k in ("range", "slots")}
    det = {k: torch.empty((n, 8), dtype=torch.float64, device=dev) for k in ("range", "slots")}
    run = {"range": lambda: e.tracks_step(pool.data, off, hw, 0, n, out["range"], det["range"], update_state=False),
           "slots": lambda: e.tracks_step_slots(pool.data, off, hw, ident, out["slots"], det["slots"], update_state=False)}
    maps = {}
    for k in run:                                               # warm-up, and the bits of each path
        for _ in range(3):
            run[k]()
        maps[k] = e.tracks_last_maps(0, n)
    torch.cuda.synchronize()
    same = torch.equal(out["range"], out["slots"]) and torch.equal(det["range"], det["slots"]) and all(
        torch.equal(torch.nan_to_num(maps["range"][q]), torch.nan_to_num(maps["slots"][q])) for q in maps["range"])
    ms = {k: [] for k in run}
    for r in range(rounds):
        for k in (("range", "slots") if r % 2 == 0 else ("slots", "range")):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                run[k]()
            b.record()
            b.synchronize()
            ms[k].append(a.elapsed_time(b) / steps)
    e.close()
    med = {k: float(np.median(v)) for k, v in ms.items()}
    return {"tracks": n, "steps_per_round": steps, "rounds": rounds, "ms_per_step_median": med,
            "ms_per_step_rounds": ms, "slots_over_range": med["slots"] / med["range"], "bit_identical": bool(same)}


def runs(ids):
    ids = sorted(ids)
    out, s = [], 0
    for k in range(1, len(ids) + 1):
        if k == len(ids) or ids[k] != ids[k - 1] + 1:
            out.append((ids[s], k - s))
            s = k
    return out


def churn(slots: int, frac: float, steps: int, warmup: int, seed: int) -> dict:
    e, pool, O = setup(slots)
    dev = e.device
    rng = np.random.default_rng(seed)
    live_n = int(round(slots * frac))
    dummy = pool.offsets(torch.zeros(1, dtype=torch.int64, device=dev))          # parked slots: frame 0 with a small box
    dummy_box = [24.0, 24.0, 16.0, 16.0]
    boxes_of = lambda k: O.synth_boxes(k, H, W, seed=int(rng.integers(1 << 30)))
    res = {}
    for method in ("range", "slots"):
        e.tracks_init(pool.data, pool.offsets(torch.zeros(slots, dtype=torch.int64, device=dev)), pool.hw(slots),
                      torch.tensor([dummy_box] * slots, dtype=torch.float64, device=dev), 0)
        live = sorted(rng.permutation(slots)[:live_n].tolist())
        st = torch.from_numpy(boxes_of(live_n)).to(dev)
        e.tracks_init_slots(pool.data, pool.offsets(torch.zeros(live_n, dtype=torch.int64, device=dev)), pool.hw(live_n), st,
                            torch.tensor(live, dtype=torch.int32, device=dev))
        stepped, t0 = 0, None
        for t in range(warmup + steps):
            if t == warmup:
                torch.cuda.synchronize()
                t0, stepped = time.perf_counter(), 0
            k = max(1, int(round(0.02 * len(live))))
            ended = set(rng.choice(live, size=k, replace=False).tolist())
            free = sorted(set(range(slots)) - set(live) | ended)
            new = sorted(rng.choice(free, size=k, replace=False).tolist())
            live = sorted((set(live) - ended) | set(new))
            nb = torch.from_numpy(boxes_of(k)).to(dev)
            fi = t % F
            if method == "slots":
                e.tracks_init_slots(pool.data, pool.offsets(torch.full((k,), fi, dtype=torch.int64, device=dev)), pool.hw(k), nb,
                                    torch.tensor(new, dtype=torch.int32, device=dev))
                n = len(live)
                off = pool.offsets(torch.full((n,), (fi + 1) % F, dtype=torch.int64, device=dev))
                e.tracks_step_slots(pool.data, off, pool.hw(n), torch.tensor(live, dtype=torch.int32, device=dev))
            else:
                parked = sorted(ended - set(new))
                for first, m in runs(parked):
                    e.tracks_init(pool.data, dummy.expand(m).contiguous(), pool.hw(m),
                                  torch.tensor([dummy_box] * m, dtype=torch.float64, device=dev), first)
                pos = {s: j for j, s in enumerate(new)}
                for first, m in runs(new):
                    j = pos[first]
                    e.tracks_init(pool.data, pool.offsets(torch.full((m,), fi, dtype=torch.int64, device=dev)), pool.hw(m),
                                  nb[j:j + m].contiguous(), first)
                high = live[-1] + 1
                is_live = np.zeros(high, bool)
                is_live[live] = True
                off = torch.where(torch.from_numpy(is_live).to(dev), pool.offsets(torch.full((high,), (fi + 1) % F, dtype=torch.int64,
                                                                                          device=dev)), dummy)
                e.tracks_step(pool.data, off.contiguous(), pool.hw(high), 0, high)
            torch.cuda.synchronize()
            stepped += len(live)
        el = time.perf_counter() - t0
        res[method] = {"live_frames_per_s": stepped / el, "ms_per_step": 1e3 * el / steps, "live_tracks_mean": stepped / steps}
    e.close()
    return {"slots": slots, "live_fraction": frac, "steps": steps, "warmup": warmup, **res,
            "slots_over_range": res["slots"]["live_frames_per_s"] / res["range"]["live_frames_per_s"]}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--churn-steps", type=int, default=30)
    ap.add_argument("--bench", nargs=2, metavar=("BEFORE", "AFTER"), help="files of bench.py result lines, before and after")
    a = ap.parse_args()
    doc = {"card": card(), "overhead": overhead(1024, a.steps, a.rounds),
           "churn": [churn(4096, f, a.churn_steps, 5, seed=40 + i) for i, f in enumerate((1.0, 0.5, 0.25))]}
    if a.bench:
        doc["bench"] = {tag: [json.loads(line) for line in open(p) if line.strip().startswith("{")] for tag, p in zip(("before", "after"), a.bench)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps({"overhead": doc["overhead"]["ms_per_step_median"], "bit_identical": doc["overhead"]["bit_identical"],
                      "churn": [(c["live_fraction"], c["slots_over_range"]) for c in doc["churn"]]}))
