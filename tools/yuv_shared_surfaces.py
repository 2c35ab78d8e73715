"""Several targets per decoder surface: one conversion per surface (the bounding rectangle of its crops) against one conversion per
track.

    python tools/yuv_shared_surfaces.py [--out profiles/yuv_shared_surfaces_b200.json] [--reps 3] [--steps 10]

1024 tracks on 64 pitched NV12 1080p surfaces (1088 surface rows, pitch 2048), 16 targets per surface, with two box sets: bench.py's
open-loop distribution (w, h ~ U(16, 400)) and small targets (w, h ~ U(16, 120)).  Open loop: every step starts from a seeded state.
Two arms alternate in one process, on one BatchedTracker:
  (a) per_track: the per-track path fed each track's surface (the same 64 surfaces, each listed 16 times): vt_yuv420_crop_to_rgb
      converts every track's rectangle into that track's own RGB frame (max_tracks + 1 frames), then the tracking step;
  (b) shared: vt_yuv420_crops_to_surface_rgb converts each surface's bounding rectangle once into one RGB frame per surface
      (64 + 1 frames), then the tracking step (BatchedTracker.track_yuv(surface=...)).
Both arms' boxes are asserted equal before any time is taken.  Per arm: the conversion and the step from CUDA events around every
step, frames/s over the timed steps, and the bytes of RGB frames the arm keeps (computed from the frame count).  The GPU's name and
power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from yuv_surfaces import gpu_info  # noqa: E402

N, M = 1024, 64
H, W, P, S = 1080, 1920, 2048, 1088


def box_sets(nsets):
    from oracle import vt_oracle as O
    rng = np.random.default_rng(78)
    small = []
    for _ in range(nsets):
        wh = rng.uniform(16, 120, (N, 2))
        xy = rng.uniform(0, 1, (N, 2)) * (np.array([W, H]) - wh)
        small.append(np.concatenate([xy, wh], 1))
    return {"bench": [O.synth_boxes(N, H, W, seed=4000 + s) for s in range(nsets)], "small": small}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "yuv_shared_surfaces_b200.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("yuv_shared_surfaces.py measures on a CUDA device; there is none")
    from oracle import vt_oracle as O
    from oracle import yuv420 as Y
    from vittracker_b200 import BatchedTracker, YuvSurfaces, load_cfg

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    bt = BatchedTracker(load_cfg(), O.make_state_dict(seed=1, stress=True), max_tracks=N, chunk_tracks=N)
    eng = bt.engine
    nsets = 8
    # 64 surfaces with 16 distinct pictures among them; the padding bytes are left as allocated
    pics = torch.from_numpy(Y.synth_yuv420(16, H, W, seed=12, format="nv12", smooth=True)).to(dev)
    idx = torch.arange(M, device=dev) % 16
    buf = torch.empty((M, S * 3 // 2, P), dtype=torch.uint8, device=dev)
    buf[:, :H, :W] = pics[idx, :H]
    buf[:, S:S + H // 2, :W] = pics[idx, H:]
    del pics
    shared = YuvSurfaces.from_frames(buf[:, :, :W], "nv12", height=H, surface_rows=S)
    surface = (np.arange(N) // (N // M)).tolist()                            # 16 consecutive tracks per surface
    ys, us, _ = shared._keep
    per_track = YuvSurfaces("nv12", [ys[s] for s in surface], [us[s] for s in surface])     # the same memory, listed per track
    frame_bytes = H * W * 3

    frames_p, offs_p = bt._yuv_frames(per_track)
    frames_s, soff, offs_s, hw_s, surf_t, _ = bt._surface_items(shared, surface, N, None)

    def convert(arm):
        if arm == "per_track":
            eng.yuv420_crop_to_rgb("nv12", per_track.planes, per_track.pitches, per_track.hw, frames_p, offs_p, bt.search_factor,
                                   boxes=None)
        else:
            eng.yuv420_crops_to_surface_rgb("nv12", shared.planes, shared.pitches, shared.hw, frames_s, soff, surf_t, bt.search_factor)

    def step(arm):
        if arm == "per_track":
            return bt.track_offsets(frames_p, offs_p, update_state=False)
        return bt.track_offsets(frames_s, offs_s, update_state=False)

    results = {}
    for set_name, sets in box_sets(nsets).items():
        dev_sets = [torch.from_numpy(b).to(dev) for b in sets]
        assert int(bt.initialize_yuv(per_track, sets[0]).abs().sum()) == 0
        # the two arms track identically before any time is taken, through the public calls too
        outs = {}
        for arm in ("per_track", "shared"):
            eng.tracks_set_state(dev_sets[1], first=0)
            convert(arm)
            outs[arm] = step(arm).cpu().numpy().copy()
        eng.tracks_set_state(dev_sets[1], first=0)
        api = bt.track_yuv(shared, update_state=False, surface=surface).cpu().numpy()
        assert np.array_equal(outs["per_track"], outs["shared"]) and np.array_equal(api, outs["shared"]), set_name

        timing = {"per_track": [], "shared": []}
        for rep in range(args.reps):
            for arm in (("per_track", "shared") if rep % 2 == 0 else ("shared", "per_track")):
                for t in range(2):                                      # warm-up
                    eng.tracks_set_state(dev_sets[t % nsets], first=0)
                    convert(arm)
                    step(arm)
                ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
                torch.cuda.synchronize(dev)
                for t in range(args.steps):
                    eng.tracks_set_state(dev_sets[t % nsets], first=0)
                    ev[t][0].record()
                    convert(arm)
                    ev[t][1].record()
                    step(arm)
                    ev[t][2].record()
                torch.cuda.synchronize(dev)
                conv = sum(e[0].elapsed_time(e[1]) for e in ev) / args.steps
                stp = sum(e[1].elapsed_time(e[2]) for e in ev) / args.steps
                total = ev[0][0].elapsed_time(ev[-1][2])
                timing[arm].append({"convert_ms": conv, "step_ms": stp, "frames_per_s": N * args.steps / (total * 1e-3)})
        med = lambda arm, k: float(np.median([x[k] for x in timing[arm]]))
        results[set_name] = {
            arm: {"convert_ms": med(arm, "convert_ms"), "step_ms": med(arm, "step_ms"), "frames_per_s": med(arm, "frames_per_s"),
                  "rgb_frames": (N if arm == "per_track" else M) + 1,
                  "rgb_frame_bytes": ((N if arm == "per_track" else M) + 1) * frame_bytes, "runs": timing[arm]}
            for arm in ("per_track", "shared")}
        results[set_name]["boxes_identical"] = True
        print(set_name, json.dumps({arm: {k: results[set_name][arm][k] for k in ("convert_ms", "step_ms", "frames_per_s")}
                                    for arm in ("per_track", "shared")}))
    out = {
        "gpu": gpu_info(),
        "workload": f"{N} tracks on {M} pitched NV12 {H}p surfaces ({S} surface rows, pitch {P}; 16 distinct pictures among them), "
                    f"{N // M} consecutive tracks per surface, stress-init weights, open-loop seeded states; {args.steps} timed steps "
                    f"after 2 warm-up steps, {args.reps} alternating repeats per arm; convert_ms is the conversion alone, step_ms the "
                    f"tracking step alone; rgb_frame_bytes are the RGB frames each arm keeps ({H} x {W} x 3 bytes each, one spare "
                    f"frame for bad entries included)",
        "results": results,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": out["gpu"]}))


if __name__ == "__main__":
    main()
