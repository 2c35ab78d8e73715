"""End-to-end tracking rate with NV12 frames against RGB frames, and what the YUV path costs on the device.

    python tools/e2e_yuv.py [--out profiles/e2e_yuv_b200.json] [--reps 3] [--steps 10] [--latency-frames 2000]

Restates bench.py's e2e leg on its seeded inputs (1024 tracks, 64 distinct 720p frames per step, stress-init weights,
open-loop boxes re-seeded every step, PipelinedFrameFeeder double-buffering the upload on a copy stream) once with RGB
host frames and once with NV12 host frames - the RGB frames are cv2.cvtColor of the NV12 ones, so both runs must return
identical boxes, which is asserted before any rate is printed.  The two formats alternate in one process, each repeated
--reps times.  Also reported, from the same run: bytes uploaded per step, the pinned host -> HBM bandwidth, the
vt_yuv420_to_rgb kernel over the 64-frame batch as bytes/s (1.5 read + 3 written per pixel; the 265 MB working set is
twice the 126 MB L2) and its share of the 7.7 TB/s data-sheet HBM bandwidth, the batch-1 Vit_dist.track() latency for
RGB and NV12 frames, and the GPU's name and power limit."""
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
sys.path.insert(0, ROOT)

N, F, H, W = 1024, 64, 720, 1280
HBM_TBPS = 7.7


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except Exception as e:                                              # the numbers stand without it, but say so
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "e2e_yuv_b200.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--latency-frames", type=int, default=2000)
    args = ap.parse_args()
    assert args.steps >= 10 and args.reps >= 3
    if not torch.cuda.is_available():
        raise SystemExit("e2e_yuv.py measures on a CUDA device; there is none")
    import cv2
    from oracle import vt_oracle as O
    from oracle import yuv420 as Y
    from vittracker_b200 import BatchedTracker, FramePool, PipelinedFrameFeeder, get_tracker_class, load_cfg, parameters

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    sd = O.make_state_dict(seed=1, stress=True)
    bt = BatchedTracker(load_cfg(), sd, max_tracks=N, chunk_tracks=N)
    assert int(bt.initialize(FramePool(O.synth_frames(F, H, W, seed=1000), dev), torch.arange(N, device=dev) % F,
                             O.synth_boxes(N, H, W, seed=2000)).abs().sum()) == 0
    nsets = 8
    host_boxes = torch.stack([torch.tensor(O.synth_boxes(N, H, W, seed=3000 + s)) for s in range(nsets)]).pin_memory()
    step_offsets = [torch.from_numpy(((np.arange(N) + t) % F) * H * W * 3).to(dev) for t in range(F)]
    nv12 = [Y.synth_yuv420(F, H, W, seed=5000 + k, format="nv12") for k in range(2)]
    host = {"nv12": [torch.from_numpy(a).pin_memory() for a in nv12],
            "rgb": [torch.from_numpy(np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2RGB_NV12) for f in a])).pin_memory() for a in nv12]}
    feeders = {"rgb": PipelinedFrameFeeder(F, H, W, dev, max_tracks=N),
               "nv12": PipelinedFrameFeeder(F, H, W, dev, max_tracks=N, frame_format="nv12", engine=bt.engine)}
    host_out = torch.empty((N, 5), dtype=torch.float64).pin_memory()

    def e2e_run(fmt, steps, keep=None):
        feeder, pools = feeders[fmt], host[fmt]
        feeder.upload(pools[0], host_boxes[0])
        for t in range(steps):
            fp = feeder.acquire()
            if t + 1 < steps:
                feeder.upload(pools[(t + 1) % 2], host_boxes[(t + 1) % nsets])
            bt.engine.tracks_set_state(fp.boxes, first=0)
            out = bt.track_offsets(fp.data, step_offsets[t % F], update_state=True)
            feeder.release(fp)
            host_out.copy_(out, non_blocking=True)
            if keep is not None:
                torch.cuda.synchronize(dev)
                keep.append(host_out.numpy().copy())

    # the two formats must track identically before any rate means anything
    got = {}
    for fmt in ("rgb", "nv12"):
        got[fmt] = []
        e2e_run(fmt, 4, got[fmt])
    same = all(np.array_equal(a, b) for a, b in zip(got["rgb"], got["nv12"]))
    assert same, "NV12 and RGB boxes differ"

    rates = {"rgb": [], "nv12": []}
    for rep in range(args.reps):
        for fmt in (("rgb", "nv12") if rep % 2 == 0 else ("nv12", "rgb")):
            e2e_run(fmt, 3)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            e2e_run(fmt, args.steps)
            e1.record()
            torch.cuda.synchronize(dev)
            rates[fmt].append(N * args.steps / (e0.elapsed_time(e1) * 1e-3))

    # pinned host -> HBM bandwidth, as bench.py measures it (one of the pinned RGB pools)
    h = host["rgb"][0].reshape(-1)
    d = torch.empty(h.numel(), dtype=torch.uint8, device=dev)
    for _ in range(2):
        d.copy_(h, non_blocking=True)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(8):
        d.copy_(h, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    h2d_gbps = h.numel() * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del d

    # the conversion kernel alone over the 64-frame batch
    fy = feeders["nv12"]
    conv, src, dst = fy._conv, fy.yuv[0], fy.pools[0].data
    fy.yuv[0].copy_(host["nv12"][0])
    reps = 200
    for _ in range(10):
        bt.engine.yuv420_to_rgb(src, conv.src_off, conv.hw, dst, conv.dst_off, "nv12")
    torch.cuda.synchronize(dev)
    launches0 = bt.engine.launch_count
    e0.record()
    for _ in range(reps):
        bt.engine.yuv420_to_rgb(src, conv.src_off, conv.hw, dst, conv.dst_off, "nv12")
    e1.record()
    torch.cuda.synchronize(dev)
    assert bt.engine.launch_count - launches0 == reps
    kern_ms = e0.elapsed_time(e1) / reps
    kern_bytes = F * H * W * 4.5
    assert torch.equal(dst.cpu(), host["rgb"][0])

    # batch-1 latency: Vit_dist.track() on a host 720p frame, open loop, RGB and NV12 in alternating blocks
    params = {}
    trk = {}
    for fmt in ("rgb", "nv12"):
        params[fmt] = parameters("vit_48_h32_noKD")
        params[fmt].state_dict = sd
        if fmt != "rgb":
            params[fmt].frame_format = fmt
        trk[fmt] = get_tracker_class()(params[fmt], "synthetic")
    fr_y = Y.synth_yuv420(8, H, W, seed=77, format="nv12")
    fr = {"nv12": list(fr_y), "rgb": [cv2.cvtColor(f, cv2.COLOR_YUV2RGB_NV12) for f in fr_y]}
    boxes = O.synth_boxes(args.latency_frames + 40, H, W, seed=78)
    lat = {"rgb": [], "nv12": []}
    for fmt in ("rgb", "nv12"):
        trk[fmt].initialize(fr[fmt][0], {"init_bbox": list(boxes[0])})
    block = 250
    for b0 in range(0, args.latency_frames + 40, block):
        for fmt in ("rgb", "nv12") if (b0 // block) % 2 == 0 else ("nv12", "rgb"):
            for i in range(b0, min(b0 + block, args.latency_frames + 40)):
                trk[fmt].state = list(boxes[i])
                t0 = time.perf_counter()
                r = trk[fmt].track(fr[fmt][i % 8], {})
                lat[fmt].append((time.perf_counter() - t0, r["target_bbox"]))
    for i in range(len(lat["rgb"])):
        assert lat["rgb"][i][1] == lat["nv12"][i][1], ("batch-1 boxes differ", i)
    lat_ms = {fmt: np.array([x[0] for x in v[40:]]) * 1e3 for fmt, v in lat.items()}

    spread = lambda v: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": [float(x) for x in v]}
    res = {
        "gpu": gpu_info(),
        "workload": f"{N} tracks, {F} distinct {H}x{W} frames per step, open-loop seeded boxes, stress-init weights, "
                    f"PipelinedFrameFeeder; {args.steps} timed steps after 3 warm-up steps, {args.reps} alternating repeats",
        "boxes_identical_rgb_vs_nv12": same,
        "e2e_frames_per_s": {fmt: spread(v) for fmt, v in rates.items()},
        "e2e_nv12_over_rgb": float(np.median(rates["nv12"]) / np.median(rates["rgb"])),
        "upload_bytes_per_step": {"rgb": F * H * W * 3 + N * 32, "nv12": F * H * W * 3 // 2 + N * 32},
        "pinned_h2d_GBps": h2d_gbps,
        "copy_floor_ms_per_step": {fmt: (F * H * W * (3 if fmt == "rgb" else 1.5)) / (h2d_gbps * 1e9) * 1e3 for fmt in ("rgb", "nv12")},
        "yuv420_to_rgb_kernel": {"frames": F, "ms_per_launch": kern_ms, "unique_bytes": kern_bytes,
                                 "TBps": kern_bytes / (kern_ms * 1e-3) / 1e12,
                                 "share_of_7.7TBps_datasheet": kern_bytes / (kern_ms * 1e-3) / 1e12 / HBM_TBPS,
                                 "launches_timed": reps},
        "batch1_track_ms": {fmt: {"p50": float(np.percentile(v, 50)), "p99": float(np.percentile(v, 99)), "frames": int(v.size)}
                            for fmt, v in lat_ms.items()},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
