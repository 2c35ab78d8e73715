"""Tracking from device-resident, pitched NV12 surfaces (decoder output): whole-frame conversion against conversion of only the
rectangle each crop reads.

    python tools/yuv_surfaces.py [--out profiles/yuv_surfaces_b200.json] [--reps 3] [--steps 10]

1024 tracks, each on its own pitched NV12 surface (the run_sequences shape: a distinct frame per track per step), at 720p (pitch
1280 + 256) and at 1080p (1088 surface rows, pitch 2048), with two box sets: bench.py's open-loop distribution (w, h ~ U(16, 400))
and small targets (w, h ~ U(16, 120)).  Open loop: every step starts from a seeded state.  Two arms alternate in one process:
  (a) repack: every surface is copied into the contiguous (H*3/2) x W layout, vt_yuv420_to_rgb converts the whole frames, then the
      tracking step;
  (b) rect: vt_yuv420_crop_to_rgb converts the rectangle each search crop reads, computed on the device from the state
      (BatchedTracker.track_yuv), then the tracking step.
Both arms' boxes are asserted equal before any time is taken.  Per arm: the conversion (for (a) including the repack copies) and
the step from CUDA events around every step, frames/s over the timed steps, and the bytes the conversion reads and writes, computed
from the frame sizes and, for (b), from the rectangles of the step's states.  The GPU's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, F = 1024, 16
SURFACES = {"720p": (720, 1280, 1280 + 256, 720), "1080p": (1080, 1920, 2048, 1088)}       # H, W, pitch, surface rows


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except Exception as e:                                              # the numbers stand without it, but say so
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def box_sets(H, W, nsets):
    from oracle import vt_oracle as O
    rng = np.random.default_rng(77)
    small = []
    for s in range(nsets):
        wh = rng.uniform(16, 120, (N, 2))
        xy = rng.uniform(0, 1, (N, 2)) * (np.array([W, H]) - wh)
        small.append(np.concatenate([xy, wh], 1))
    return {"bench": [O.synth_boxes(N, H, W, seed=3000 + s) for s in range(nsets)], "small": small}


def rect_bytes(boxes, factor, H, W):
    """Bytes the rectangle conversion reads (Y + interleaved UV) and writes (RGB) for these states."""
    from vittracker_b200.sequences import crop_rect
    from vittracker_b200.tracker import even_rect
    rd = wr = 0
    for b in boxes:
        r = crop_rect(b, factor, H, W)
        if r is None:
            continue
        ya, yb, xa, xb = even_rect(r, H, W)
        px = (yb - ya) * (xb - xa)
        rd += px * 3 // 2
        wr += px * 3
    return rd, wr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "yuv_surfaces_b200.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("yuv_surfaces.py measures on a CUDA device; there is none")
    from oracle import vt_oracle as O
    from oracle import yuv420 as Y
    from vittracker_b200 import BatchedTracker, YuvSurfaces, load_cfg

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = load_cfg()
    bt = BatchedTracker(cfg, O.make_state_dict(seed=1, stress=True), max_tracks=N, chunk_tracks=N)
    eng = bt.engine
    nsets = 8
    results = {}
    for res_name, (H, W, P, S) in SURFACES.items():
        # 1024 surfaces, F distinct pictures among them; the padding bytes are left as allocated
        pics = torch.from_numpy(Y.synth_yuv420(F, H, W, seed=11, format="nv12", smooth=True)).to(dev)
        idx = torch.arange(N, device=dev) % F
        surf_buf = torch.empty((N, S * 3 // 2, P), dtype=torch.uint8, device=dev)
        surf_buf[:, :H, :W] = pics[idx, :H]
        surf_buf[:, S:S + H // 2, :W] = pics[idx, H:]
        del pics
        surfaces = YuvSurfaces.from_frames(surf_buf[:, :, :W], "nv12", height=H, surface_rows=S)
        repack = torch.empty((N, H * 3 // 2, W), dtype=torch.uint8, device=dev)
        rgb = torch.zeros((N, H, W, 3), dtype=torch.uint8, device=dev)
        ar = torch.arange(N, dtype=torch.int64, device=dev)
        src_off, dst_off = ar * (H * W * 3 // 2), ar * (H * W * 3)
        hw = surfaces.hw

        def convert(arm):
            if arm == "repack":
                repack[:, :H] = surf_buf[:, :H, :W]
                repack[:, H:] = surf_buf[:, S:S + H // 2, :W]
                eng.yuv420_to_rgb(repack, src_off, hw, rgb, dst_off, "nv12")
            else:
                frames, offs = bt._yuv_frames(surfaces)
                eng.yuv420_crop_to_rgb("nv12", surfaces.planes, surfaces.pitches, hw, frames, offs, bt.search_factor, boxes=None)

        def step(arm):
            if arm == "repack":
                return bt.track_offsets(rgb, dst_off, update_state=False)
            frames, offs = bt._yuv_frames(surfaces)
            return bt.track_offsets(frames, offs, update_state=False)

        for set_name, sets in box_sets(H, W, nsets).items():
            dev_sets = [torch.from_numpy(b).to(dev) for b in sets]
            assert int(bt.initialize_yuv(surfaces, sets[0]).abs().sum()) == 0
            # the two arms track identically before any time is taken
            outs = {}
            for arm in ("repack", "rect"):
                eng.tracks_set_state(dev_sets[1], first=0)
                convert(arm)
                outs[arm] = step(arm).cpu().numpy().copy()
            assert np.array_equal(outs["repack"], outs["rect"]), (res_name, set_name)

            timing = {"repack": [], "rect": []}
            for rep in range(args.reps):
                for arm in (("repack", "rect") if rep % 2 == 0 else ("rect", "repack")):
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
            rd = wr = 0
            for t in range(args.steps):
                r, w = rect_bytes(sets[t % nsets], bt.search_factor, H, W)
                rd += r
                wr += w
            med = lambda arm, k: float(np.median([x[k] for x in timing[arm]]))
            results[f"{res_name}/{set_name}"] = {
                "surface": {"H": H, "W": W, "pitch": P, "surface_rows": S},
                "repack": {"convert_ms": med("repack", "convert_ms"), "step_ms": med("repack", "step_ms"),
                           "frames_per_s": med("repack", "frames_per_s"),
                           "bytes_read_per_step": N * (H * W * 3 // 2) * 2, "bytes_written_per_step": N * (H * W * 3 // 2 + H * W * 3),
                           "runs": timing["repack"]},
                "rect": {"convert_ms": med("rect", "convert_ms"), "step_ms": med("rect", "step_ms"),
                         "frames_per_s": med("rect", "frames_per_s"),
                         "bytes_read_per_step": rd // args.steps, "bytes_written_per_step": wr // args.steps,
                         "runs": timing["rect"]},
                "boxes_identical": True,
            }
            print(res_name, set_name, json.dumps({k: {kk: v[kk] for kk in ("convert_ms", "step_ms", "frames_per_s")}
                                                  for k, v in results[f"{res_name}/{set_name}"].items() if k in ("repack", "rect")}))
        del surf_buf, repack, rgb, surfaces
        torch.cuda.empty_cache()
    out = {
        "gpu": gpu_info(),
        "workload": f"{N} tracks, each on its own pitched NV12 surface ({F} distinct pictures among them), stress-init weights, "
                    f"open-loop seeded states; {args.steps} timed steps after 2 warm-up steps, {args.reps} alternating repeats per arm; "
                    f"convert_ms of 'repack' includes the two copies into the contiguous layout; bytes are what the conversion needs "
                    f"(repack copies included), not DRAM sectors",
        "results": results,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": out["gpu"]}))


if __name__ == "__main__":
    main()
