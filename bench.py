#!/usr/bin/env python
"""Benchmark of the VitTracker per-frame hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this implementation (N>1: under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port), rank 0 only
    python bench.py --gpus N --total-tracks 8192             # BASELINE configs[3] as named: 8192 tracks STRONG-sharded over N GPUs
    python bench.py --gpus 8 --config vit_768_h256_d12 --tracks 512     # BASELINE configs[4]: widest config, 4096 tracks on 8 GPUs
    python bench.py --gpus 1 --steps K --dump-outputs DIR                # also write the last timed step's boxes as DIR/boxes.npy

A "step" advances every track by one frame: crop + normalise + stem + 3 ViT blocks + head + Hann /
arg-max / box decode (+ for N>1 one NCCL all-gather of the boxes).  Default workload per GPU (BASELINE.json
configs[2]): 1024 concurrent synthetic tracks over 64 distinct 720x1280 uint8 frames resident in HBM
(177 MB > L2), open-loop seeded boxes re-seeded every step, stress-init weights; with N > 1 the line also
carries `strong_8192` = configs[3] (8192 tracks / N per GPU) measured in the same run.  Prints ONE JSON line
(see README / DESIGN.md for the keys).

Every input is generated from fixed seeds, so a run with the same arguments sees the same inputs.  --dump-outputs DIR writes
what the timed path returned in its last timed step as DIR/boxes.npy: x y w h confidence of every track in float64 (rank 0;
--impl reference: its 256-track sample), at most 64 MB (beyond that a fixed, seeded sample of the tracks), so that two builds
of the project can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_JSON_OUT = sys.stdout
METRIC = "tracked frames/sec over B concurrent tracks"
UNIT = "frames/s"
FLOP_BLOCKS = 112.07e6        # algorithmic FLOP per tracked frame in the 3 ViT blocks (SURVEY 8d)
FLOP_STEM = 21.23e6
FLOP_HEAD = 30.53e6
# widest configuration (C 768 / 12 heads / depth 12 / head 256, SURVEY 8d): MAC counts per tracked frame, template tokens cached
WIDEST = {"name": "vit_768_h256_d12", "C": 768, "depth": 12, "head_ch": 256,
          "flop_blocks_head": 2.0 * (12 * 2422210560 + 1656266752), "flop_stem": 2.0 * 2080899072, "flop_frame": 66.65e9}
FRAME_H, FRAME_W = 720, 1280


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(blocks, items_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the block kernel, from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json, bytes per track), scaled to this launch size."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            per_track = json.load(f)[blocks]["dram_bytes_per_track"]
        return per_track * items_per_launch
    except Exception:
        return None


def hbm_rooflines(boxes_xywh, stages, peaks, S=256, factor=4.0):
    """The stem and the head against the measured copy bandwidth (north star: achieved HBM GB/s for the crop and the head), on
    ALGORITHMIC bytes (SURVEY 8d).  Stem (crop + resize + normalise fused into conv1, conv2-4): read = the unique source bytes the
    crops touch, 3 * min(crop_sz^2, 4 S^2) per track clipped to the image, write = the 256 x 48 fp32 search tokens.  Head + decode:
    read = the tokens, write = (x, y, w, h, conf) - 49 KB per track for 30.5 MFLOP: the head is NOT HBM-bound (a serial five-layer
    chain per track; the ncu profile shows it latency-bound), so its entry is labelled `tensor` and carries its algorithmic TFLOP/s
    against the tensor peak, with the HBM figure beside it."""
    b = np.asarray(boxes_xywh, dtype=np.float64)
    crop_sz = np.ceil(np.sqrt(b[:, 2] * b[:, 3]) * factor)
    x1 = np.rint(b[:, 0] + 0.5 * b[:, 2] - 0.5 * crop_sz)
    y1 = np.rint(b[:, 1] + 0.5 * b[:, 3] - 0.5 * crop_sz)
    wx = np.clip(np.minimum(x1 + crop_sz, FRAME_W - 1) - np.maximum(x1, 0), 0, None)       # columns / rows 0 .. W-2 / H-2 are readable
    wy = np.clip(np.minimum(y1 + crop_sz, FRAME_H - 1) - np.maximum(y1, 0), 0, None)
    frac_in = np.where(crop_sz > 0, (wx * wy) / np.maximum(crop_sz * crop_sz, 1), 0.0)
    src = 3.0 * np.minimum(crop_sz * crop_sz, 4.0 * S * S) * frac_in
    tokens = 256 * 48 * 4
    per_track = {"stem": float(src.mean()) + tokens, "head": tokens + 5 * 4}
    out = {}
    for k, bytes_per_track in per_track.items():
        st = stages[k]
        launches = max(1, st["launches"])
        ms, items = st["ms"] / launches, st["items"] / launches
        achieved = bytes_per_track * items / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                traffic = json.load(f)[k]["dram_bytes_per_track"] * items
        except Exception:
            pass
        out[k] = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                  "traffic": traffic, "algorithmic_bytes_per_launch": bytes_per_track * items, "avg_launch_ms": ms}
        if k == "head":
            tf = FLOP_HEAD * items / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
            out[k].update({"bound": "tensor", "note": "latency-bound (serial layer chain per track): neither HBM nor the tensor pipe limits it",
                           "hbm_gbs": achieved, "hbm_frac": achieved / peaks["hbm_gbs"],
                           "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"]})
    return out


DUMP_LIMIT = 64 << 20         # bytes --dump-outputs may write


def dump_outputs(out_dir, boxes):
    """--dump-outputs: `boxes` as <out_dir>/boxes.npy in float64.  Beyond DUMP_LIMIT a fixed, seeded sample of its rows is kept and
    their indices are written as <out_dir>/rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    boxes = np.asarray(boxes, dtype=np.float64)
    if boxes.nbytes > DUMP_LIMIT:
        keep = DUMP_LIMIT // (boxes[0].nbytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(len(boxes), keep, replace=False))
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
        boxes = boxes[rows]
    np.save(os.path.join(out_dir, "boxes.npy"), boxes)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def count(self) -> int:
        """Samples written so far."""
        try:
            self.fh.flush()
            with open(self.path) as f:
                return sum(1 for line in f if line.count(",") >= 8)
        except Exception:
            return 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# --------------------------------------------------------------------------------------------------
# CPU path (the reference's algorithm; oracle port) - used for cpu_baseline and --impl reference
# --------------------------------------------------------------------------------------------------
class CpuPath:
    """Reference per-frame path on the host: cv2 crop + normalise + PyTorch fp32 forward (template
    stem re-run every frame, as the reference does) + Hann / arg-max / decode / clip.  Tracks are
    processed in groups of `group` so that the forward is batched (best CPU throughput, BASELINE.md 3)."""

    def __init__(self, sd, frames, group=16):
        from oracle import vt_oracle as O
        self.O = O
        self.model = O.OracleModel(sd)
        self.win = O.hann2d(16, 16)
        self.frames = frames
        self.group = group

    def prepare(self, init_boxes):
        O = self.O
        self.z = torch.cat([O.preprocess(O.sample_target_cv(self.frames[i % len(self.frames)], list(b), 2.0, 128)[0])
                            for i, b in enumerate(init_boxes)])

    def step(self, boxes, t):
        """One frame for every track; returns [x, y, w, h, confidence] per track, as the reference's track() does."""
        O = self.O
        n = len(boxes)
        out_states = []
        for g0 in range(0, n, self.group):
            idx = range(g0, min(n, g0 + self.group))
            crops, rfs = [], []
            for i in idx:
                p, rf, _ = O.sample_target_cv(self.frames[(i + t) % len(self.frames)], list(boxes[i]), 4.0, 256)
                crops.append(O.preprocess(p)); rfs.append(rf)
            out = self.model.forward(self.z[g0:g0 + len(crops)], torch.cat(crops))
            resp = self.win * out["score_map"]
            pb = self.model.cal_bbox(resp, out["size_map"], out["offset_map"])
            conf = out["score_map"].flatten(1).max(1).values.tolist()
            for k, i in enumerate(idx):
                pred = (pb[k] * 256 / rfs[k]).tolist()
                out_states.append(O.clip_box(O.map_box_back(list(boxes[i]), pred, rfs[k]), FRAME_H, FRAME_W, margin=10) + [conf[k]])
        return out_states


def cpu_sample(sd, budget_s=12.0, tracks=64, frames_n=4):
    """Bounded sample of the same workload on the host cores: `tracks` tracks over 720p frames,
    repeated until ~budget_s seconds have passed.  Returns (frames/s, cores, description)."""
    from oracle import vt_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    frames = O.synth_frames(frames_n, FRAME_H, FRAME_W, seed=100)
    cp = CpuPath(sd, frames)
    cp.prepare(O.synth_boxes(tracks, FRAME_H, FRAME_W, seed=101))
    cp.step(O.synth_boxes(tracks, FRAME_H, FRAME_W, seed=102), 0)          # warm-up
    done, t0, step = 0, time.perf_counter(), 0
    while True:
        cp.step(O.synth_boxes(tracks, FRAME_H, FRAME_W, seed=103 + step), step)
        done += tracks; step += 1
        el = time.perf_counter() - t0
        if el >= budget_s:
            break
    return done / el, torch.get_num_threads(), f"{done} tracked frames ({step} steps x {tracks} tracks, forward batched by 16) in {el:.1f} s"


def cpu_model_name() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_b1_sample(sd, threads, budget_s=2.0):
    """The reference's own shape of the path - one sequence, batch 1 (SURVEY 8d: B = 1, all threads and one thread) - on the host:
    frames/s of crop + forward + decode for a single track."""
    from oracle import vt_oracle as O
    torch.set_num_threads(threads)
    frames = O.synth_frames(2, FRAME_H, FRAME_W, seed=110)
    cp = CpuPath(sd, frames, group=1)
    cp.prepare(O.synth_boxes(1, FRAME_H, FRAME_W, seed=111))
    boxes = O.synth_boxes(64, FRAME_H, FRAME_W, seed=112)
    cp.step(boxes[:1], 0)
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        cp.step(boxes[done % 64:done % 64 + 1], done)
        done += 1
    return done / (time.perf_counter() - t0)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on this box's host cores (all of them), on the same
    workload: each step is a bounded sample of 256 tracks (of the 1024 per GPU) over 720p frames."""
    if rank != 0:
        return
    from oracle import vt_oracle as O
    sd = O.make_state_dict(seed=1, stress=True)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    tracks = 256                                       # bounded sample per step (>= 0.3 s of CPU work per step)
    frames = O.synth_frames(8, FRAME_H, FRAME_W, seed=100)
    cp = CpuPath(sd, frames)
    cp.prepare(O.synth_boxes(tracks, FRAME_H, FRAME_W, seed=101))
    for w in range(args.warmup):
        cp.step(O.synth_boxes(tracks, FRAME_H, FRAME_W, seed=200 + w), w)
    per_step = []
    t0 = time.perf_counter()
    for s in range(args.steps):
        boxes = O.synth_boxes(tracks, FRAME_H, FRAME_W, seed=300 + s)
        ts = time.perf_counter()
        last = cp.step(boxes, s)
        per_step.append(tracks / (time.perf_counter() - ts))
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    v = tracks * args.steps / el
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world, note=f"CPU sample: {tracks} tracks per step"),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{tracks} tracks x {args.steps} steps ({el:.1f} s), cv2 crop + torch fp32 forward batched by 16 + decode",
                             "per_step_spread": {"min": float(min(per_step)), "median": float(np.median(per_step)), "max": float(max(per_step))},
                             "cpu_model": cpu_model_name(), "os_cpu_count": os.cpu_count()},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def workload_config(args, world, note=None):
    n = per_gpu_tracks(args, world)
    strong = args.total_tracks > 0
    which = "BASELINE configs[4]" if args.config != "vit_48_h32_noKD" else ("BASELINE configs[3]" if strong else "BASELINE configs[2]")
    c = {"workload": f"{args.config}, {n} concurrent synthetic tracks per GPU ({which}; {n * world} total"
                     f"{', strong-sharded' if strong else ''}), {args.frames} distinct {FRAME_H}x{FRAME_W} uint8 frames per GPU in HBM, "
                     f"open-loop seeded boxes, stress-init weights",
         "tracks_per_gpu": n, "total_tracks": n * world, "frames_per_gpu": args.frames,
         "frame_hw": [FRAME_H, FRAME_W], "chunk_tracks": args.chunk, "blocks_impl": args.blocks,
         "parallelism": f"tracks sharded x{world}, all-gather of boxes" if world > 1 else "single GPU",
         "l2": "inputs larger than L2 (frame pool %.0f MB + per-chunk intermediates)" % (args.frames * FRAME_H * FRAME_W * 3 / 1e6)}
    if note:
        c["note"] = note
    return c


def per_gpu_tracks(args, world):
    if args.total_tracks > 0:
        if args.total_tracks % world:
            raise SystemExit(f"--total-tracks {args.total_tracks} is not divisible by {world} GPUs")
        return args.total_tracks // world
    return args.tracks


def bind_rank(local_rank, world):
    """Pin this rank's host threads to the CPUs the driver reports as local to its GPU (nvmlDeviceGetCpuAffinity) - split evenly
    between the ranks that share them - and prefer that NUMA node for the pinned staging pools allocated afterwards.  Returns a
    description for the bench line.  Best effort: every failure leaves the process as it was."""
    info = {"cpus": None, "numa_node": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        local = [c for c in range(ncpu) if (words[c // 64] >> (c % 64)) & 1]
        allowed = sorted(set(local) & os.sched_getaffinity(0)) or sorted(os.sched_getaffinity(0))
        # ranks whose GPUs report the same CPU set share it evenly
        same = []
        for r in range(world):
            try:
                w = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(r), (ncpu + 63) // 64)
                if list(w) == list(words):
                    same.append(r)
            except Exception:
                pass
        if len(same) > 1 and len(allowed) >= 2 * len(same):
            k = same.index(local_rank)
            per = len(allowed) // len(same)
            allowed = allowed[k * per:(k + 1) * per]
        os.sched_setaffinity(0, allowed)
        info["cpus"] = f"{allowed[0]}-{allowed[-1]} ({len(allowed)})"
        try:
            pci = pynvml.nvmlDeviceGetPciInfo(h).busId
            pci = pci.decode() if isinstance(pci, bytes) else pci
            with open(f"/sys/bus/pci/devices/{pci[-12:].lower()}/numa_node") as f:
                node = int(f.read().strip())
            info["numa_node"] = node
            if node >= 0:
                import ctypes
                libc = ctypes.CDLL(None, use_errno=True)
                mask = ctypes.c_ulong(1 << node)
                MPOL_PREFERRED = 1
                if libc.syscall(238, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(64)) != 0:     # set_mempolicy (x86_64)
                    info["numa_node"] = f"{node} (set_mempolicy failed)"
        except Exception as e:
            info["numa_node"] = f"unknown ({type(e).__name__})"
    except Exception as e:
        info["error"] = f"{type(e).__name__}: {e}"
    return info


def h2d_cap(dev, world, host_buf, reps=8):
    """Pinned host -> HBM copy bandwidth of this rank with EVERY rank copying at once (the e2e leg's limiter): per-rank GB/s.
    `host_buf`: one of the pinned frame pools the e2e leg itself uploads (same pages, same placement)."""
    import torch.distributed as dist
    h = host_buf.reshape(-1)
    n = h.numel()
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    for _ in range(2):
        d.copy_(h, non_blocking=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        d.copy_(h, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    return n * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


class Workload:
    """One tracker + its resident frames + pre-generated open-loop states; step(t) is what the timed loops call."""

    def __init__(self, args, cfg, sd, n, rank, world, dev, frames_host, depth=None):
        import torch.distributed as dist
        from oracle import vt_oracle as O
        from vittracker_b200 import BatchedTracker, FramePool, ShardedTracker
        self.O, self.dist = O, dist
        self.n, self.F, self.rank, self.world, self.dev = n, args.frames, rank, world, dev
        self.bt = BatchedTracker(cfg, sd, max_tracks=n, chunk_tracks=min(args.chunk, n), blocks_impl=args.blocks, depth=depth)
        self.pool = FramePool(frames_host, dev)
        self.sharded = ShardedTracker(n * world, self.bt) if world > 1 else None
        F = self.F
        init_boxes = O.synth_boxes(n, FRAME_H, FRAME_W, seed=2000 + rank)
        status = self.bt.initialize(self.pool, torch.arange(n, device=dev) % F, init_boxes)
        assert int(status.abs().sum()) == 0
        # open-loop: a fresh seeded state per step (SURVEY 7.2 item 4), generated up front on the device
        self.nsets = 8
        self.step_boxes_host = [O.synth_boxes(n, FRAME_H, FRAME_W, seed=3000 + 97 * rank + s) for s in range(self.nsets)]
        self.step_boxes = torch.stack([torch.tensor(b) for b in self.step_boxes_host]).to(dev)
        # per-step frame offsets prepared up front: the timed loop launches only this library's kernels
        self.fidx_host = np.arange(n, dtype=np.int64) % F
        self.step_offsets = [torch.from_numpy(((self.fidx_host + t) % F) * self.pool.frame_bytes).to(dev) for t in range(F)]
        self.pending = None

    def finish_gather(self):
        if self.pending is not None:
            self.pending.wait()               # current stream waits for the gather of the previous step
            self.pending = None

    def step(self, t, detail=False):
        self.bt.engine.tracks_set_state(self.step_boxes[t % self.nsets], first=0)
        out = self.bt.track_offsets(self.pool.data, self.step_offsets[t % self.F], update_state=True, detail=detail)
        if self.sharded is not None and not detail:
            # the only exchange step: all-gather of (x, y, w, h, conf); it overlaps the next step's kernels
            self.finish_gather()
            self.pending, out = self.sharded.gather_async(out)
        return out

    def local_step(self, t):
        """The step without its exchange (the clock sampler's load on rank 0 alone: no collective may be issued there)."""
        self.bt.engine.tracks_set_state(self.step_boxes[t % self.nsets], first=0)
        self.bt.track_offsets(self.pool.data, self.step_offsets[t % self.F], update_state=True)

    def barrier(self):
        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
            torch.cuda.synchronize(self.dev)

    def timed(self, W, K, sampler=None):
        """W warm-up steps, then exactly K steps between barrier + synchronize; returns (ms max over ranks, stages, launches)."""
        for t in range(W):
            self.step(t)
        self.finish_gather()
        if sampler is not None:
            # The timed region is tens of milliseconds and nvidia-smi needs longer than that to deliver its first sample: the sampler is
            # started here and the SAME steps keep running (untimed) until it has reported once, so that its 50 ms samples bracket the
            # timed region under the load that is being timed; the load is kept up for three more sampling periods after the region.
            sampler.start()
            t_end = time.time() + 3.0
            while sampler.proc is not None and sampler.count() < 1 and time.time() < t_end:
                for t in range(8):
                    self.local_step(t % max(1, W))
                torch.cuda.synchronize()
        self.barrier()
        eng = self.bt.engine
        launches0 = eng.launch_count
        eng.profile(True)
        eng.profile_read()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for t in range(K):
            out = self.step(W + t)
        self.finish_gather()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        self.step_out = out.cpu().numpy().copy()            # what the last timed step returned (all tracks by global id when sharded)
        stages = eng.profile_read()
        eng.profile(False)
        launches = eng.launch_count - launches0 + (K if self.world > 1 else 0)
        clocks = None
        if sampler is not None:
            n0, t_end = sampler.count(), time.time() + 1.0
            while sampler.proc is not None and sampler.count() < n0 + 3 and time.time() < t_end:
                for t in range(8):
                    self.local_step(t % max(1, W))
                torch.cuda.synchronize()
            clocks = sampler.stop()
        tms = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(tms, op=self.dist.ReduceOp.MAX)
        return float(tms.item()), stages, launches, clocks

    def parity_spot(self, t_last, last_out, k=32):
        """Compare `k` tracks of the LAST TIMED step with the CPU oracle (the checker): re-run that step with the detail rows
        (open-loop states make it idempotent - the boxes must be bit-identical to the timed step's), then arg-max index, box and
        confidence of the first k tracks against cv2 crop + torch fp32 forward + decode."""
        O = self.O
        out, det = self.step(t_last, detail=True)
        out_h, det_h = out.cpu().numpy(), det.cpu().numpy()
        same = bool(np.array_equal(out_h, last_out))
        boxes = self.step_boxes_host[t_last % self.nsets][:k]
        frames = self.pool.data.view(self.F, FRAME_H, FRAME_W, 3)
        model = O.OracleModel(self.sd_ref, depth=getattr(self, "oracle_depth", 3), num_heads=getattr(self, "oracle_heads", 1))
        win = O.hann2d(16, 16)
        init = O.synth_boxes(self.n, FRAME_H, FRAME_W, seed=2000 + self.rank)[:k]
        need = sorted({int(self.fidx_host[i]) for i in range(k)} | {int((self.fidx_host[i] + t_last) % self.F) for i in range(k)})
        fr = {j: frames[j].cpu().numpy() for j in need}
        zs, xs, rfs = [], [], []
        for i in range(k):
            zs.append(O.preprocess(O.sample_target_cv(fr[int(self.fidx_host[i])], list(init[i]), 2.0, 128)[0]))
            xp, rf, _ = O.sample_target_cv(fr[int((self.fidx_host[i] + t_last) % self.F)], list(boxes[i]), 4.0, 256)
            xs.append(O.preprocess(xp)); rfs.append(rf)
        o = model.forward(torch.cat(zs), torch.cat(xs))
        resp = (win * o["score_map"]).flatten(1)
        top = torch.topk(resp, 2, dim=1).values
        pb = model.cal_bbox(resp.view(-1, 1, 16, 16), o["size_map"], o["offset_map"])
        flips = ties = 0
        box_err = conf_err = 0.0
        for i in range(k):
            if float(top[i, 0] - top[i, 1]) < 1e-5:
                ties += 1
                continue
            if int(det_h[i, 5]) != int(resp[i].argmax()):
                flips += 1
                continue
            pred = (pb[i] * 256 / rfs[i]).tolist()
            want = O.clip_box(O.map_box_back(list(boxes[i]), pred, rfs[i]), FRAME_H, FRAME_W, margin=10)
            box_err = max(box_err, float(np.abs(out_h[i, :4] - np.array(want, dtype=np.float64)).max()))
            conf_err = max(conf_err, abs(float(out_h[i, 4]) - float(o["score_map"][i].max())))
        return {"tracks": k, "flips": flips, "ties_excluded": ties, "max_box_err": box_err, "max_conf_err": conf_err,
                "status_nonzero": int((det_h[:, 6] != 0).sum()), "rerun_bit_identical_to_timed_step": same,
                "checker": "CPU oracle: cv2 crop + torch fp32 forward + Hann / arg-max / decode / clip on the timed step's inputs"}


def gpu_eager_leg(sd, dev, depth, num_heads, batches=(1024, 1)):
    """The comparison line 'stock PyTorch eager on this B200' (SURVEY 2.3, BASELINE.md 4): the reference's module graph
    (oracle restatement, op for op the reference's torch calls) in fp32 with TF32 off on the GPU - forward(z, x) + Hann window +
    cal_bbox, inputs (normalised crops) already resident: the reference itself crops on the CPU with OpenCV.  A baseline leg,
    timed with CUDA events; nothing of the product runs in it."""
    from oracle import vt_oracle as O
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    model = O.OracleModel(sd, depth=depth, num_heads=num_heads).to(dev)
    win = O.hann2d(16, 16).to(dev)
    out = {"scope": "forward(z, x) + Hann window + cal_bbox in fp32 (TF32 off), normalised crops resident in HBM; no crop, no clip / state update",
           "torch": torch.__version__}
    g = torch.Generator(device="cpu").manual_seed(5)
    for B in batches:
        try:
            z = torch.randn((B, 3, 128, 128), generator=g).to(dev)
            x = torch.randn((B, 3, 256, 256), generator=g).to(dev)

            def run():
                o = model.forward(z, x)
                return model.cal_bbox(win * o["score_map"], o["size_map"], o["offset_map"])
            iters = 5 if B > 1 else 200
            for _ in range(3 if B > 1 else 20):
                run()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                run()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / iters
            out[f"batch{B}"] = {"ms_per_forward": ms, "frames_per_s": B / (ms * 1e-3)}
            del z, x
        except Exception as e:
            out[f"batch{B}"] = {"error": f"{type(e).__name__}: {e}"}
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tracks", type=int, default=0, help="concurrent tracks per GPU (default 1024; 512 for the widest config)")
    ap.add_argument("--total-tracks", type=int, default=0, help="strong sharding: this many tracks split over the GPUs (BASELINE configs[3]: 8192)")
    ap.add_argument("--config", default="vit_48_h32_noKD", choices=["vit_48_h32_noKD", WIDEST["name"]])
    ap.add_argument("--frames", type=int, default=64, help="distinct frames resident per GPU")
    ap.add_argument("--chunk", type=int, default=0, help="tracks per internal pass (default 1024; 128 for the widest config)")
    ap.add_argument("--blocks", default="tcgen05", choices=["simt", "tcgen05", "tcgen05_3term"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--no-strong-leg", action="store_true", help="skip the configs[3] leg a multi-GPU default run adds")
    ap.add_argument("--no-bind", action="store_true", help="do not pin the rank to its GPU's CPUs / NUMA node")
    ap.add_argument("--latency-frames", type=int, default=10000, help="open-loop frames of the batch-1 latency leg (SURVEY C2: 10000)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/boxes.npy (float64: x, y, w, h, confidence per track)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    widest = args.config == WIDEST["name"]
    if args.tracks <= 0:
        args.tracks = 512 if widest else 1024
    if args.chunk <= 0:
        args.chunk = 128 if widest else 1024

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries the one JSON line and nothing else: library chatter (e.g. NCCL's version banner) goes to stderr
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from oracle import vt_oracle as O          # synthetic workload generators + the checker / baseline legs only
    from vittracker_b200 import load_cfg, parameters

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the CUDA path has no CPU fallback")
    binding = None if args.no_bind else bind_rank(local_rank, world)      # before any pinned allocation
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    if widest:
        cfg = parameters(WIDEST["name"]).cfg
        sd = O.make_state_dict(seed=1, stress=True, C=WIDEST["C"], depth=WIDEST["depth"], head_ch=WIDEST["head_ch"])
        depth, heads = WIDEST["depth"], 12
    else:
        cfg = load_cfg()
        sd = O.make_state_dict(seed=1, stress=True)
        depth, heads = 3, 1
    n, F, K, W = per_gpu_tracks(args, world), args.frames, args.steps, args.warmup
    frames = O.synth_frames(F, FRAME_H, FRAME_W, seed=1000 + rank)
    wl = Workload(args, cfg, sd, n, rank, world, dev, frames, depth=depth if widest else None)
    wl.sd_ref, wl.oracle_depth, wl.oracle_heads = sd, depth, heads
    bt, pool, sharded = wl.bt, wl.pool, wl.sharded
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms, stages, launches, clocks = wl.timed(W, K, sampler)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl.step_out)
    value = n * world * K / (ms / 1e3)
    last_out = wl.step_out[:n]                                      # rank 0's boxes of the last timed step, as dumped
    try:
        parity = wl.parity_spot(W + K - 1, last_out, k=8 if widest else 32) if rank == 0 else None
    except Exception as e:                                         # secondary: never at the expense of the line
        parity = {"error": f"{type(e).__name__}: {e}"}
    wl.barrier()

    # ---- end to end through the public API with HOST buffers: every step uploads its 64 frames (pinned host
    # memory -> HBM on a copy stream, double-buffered so that the upload of step t+1 overlaps the compute of
    # step t), uploads the boxes, runs the step and reads the boxes back
    from vittracker_b200 import PipelinedFrameFeeder
    nsets, step_offsets, step_boxes = wl.nsets, wl.step_offsets, wl.step_boxes
    host_pools = [torch.from_numpy(O.synth_frames(F, FRAME_H, FRAME_W, seed=5000 + rank + k)).pin_memory() for k in range(2)]
    host_boxes = step_boxes.cpu().pin_memory()
    host_out = torch.empty((n * world if world > 1 else n, 5), dtype=torch.float64).pin_memory()
    feeder = PipelinedFrameFeeder(F, FRAME_H, FRAME_W, dev, max_tracks=n)
    prev = [None]

    def e2e_run(steps):
        feeder.upload(host_pools[0], host_boxes[0])
        for t in range(steps):
            fp = feeder.acquire()
            if t + 1 < steps:
                feeder.upload(host_pools[(t + 1) % 2], host_boxes[(t + 1) % nsets])
            bt.engine.tracks_set_state(fp.boxes, first=0)
            out = bt.track_offsets(fp.data, step_offsets[t % F], update_state=True)
            feeder.release(fp)
            if sharded is not None:
                # read back the PREVIOUS step's gathered boxes (its gather overlapped this step), then start this step's
                if wl.pending is not None:
                    wl.finish_gather()
                    host_out.copy_(prev[0], non_blocking=True)
                wl.pending, prev[0] = sharded.gather_async(out)
            else:
                host_out.copy_(out, non_blocking=True)
        if sharded is not None:
            wl.finish_gather()
            host_out.copy_(prev[0], non_blocking=True)

    e2e_run(3)
    wl.barrier()
    Ke = max(3, min(K, 10))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(Ke)
    e1.record()
    wl.barrier()
    tms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    e2e_value = n * world * Ke / (float(tms.item()) / 1e3)
    h2d = F * FRAME_H * FRAME_W * 3 + n * 32
    d2h = host_out.numel() * 8
    # the limiter of that leg, measured: pinned host -> HBM bandwidth with every rank copying at once
    cap = torch.tensor([h2d_cap(dev, world, host_pools[0])], device=dev, dtype=torch.float64)
    cap_all = [torch.zeros_like(cap) for _ in range(world)]
    if world > 1:
        dist.all_gather(cap_all, cap)
    else:
        cap_all = [cap]
    cap_ranks = [float(c.item()) for c in cap_all]
    del host_pools, feeder
    torch.cuda.empty_cache()

    # ---- BASELINE configs[3] as named: 8192 tracks strong-sharded over the GPUs, in the same run (default multi-GPU runs only)
    strong = None
    if world > 1 and not widest and args.total_tracks == 0 and not args.no_strong_leg and 8192 % world == 0:
        try:
            ns = 8192 // world
            if ns == n:
                strong = {"total_tracks": 8192, "tracks_per_gpu": ns, "value": value, "ms_per_step": ms / K, "note": "identical to the main workload at this N"}
            else:
                del wl, bt, pool, sharded
                torch.cuda.empty_cache()
                wl2 = Workload(args, cfg, sd, ns, rank, world, dev, frames)
                ms2, _, _, _ = wl2.timed(W, max(3, K // 2))
                strong = {"total_tracks": 8192, "tracks_per_gpu": ns, "value": 8192 * max(3, K // 2) / (ms2 / 1e3),
                          "ms_per_step": ms2 / max(3, K // 2), "scaling": "strong", "steps": max(3, K // 2)}
                del wl2
                torch.cuda.empty_cache()
        except Exception as e:
            strong = {"error": f"{type(e).__name__}: {e}"}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    blk = stages["blocks"]
    blk_ms = blk["ms"] / max(1, blk["launches"])
    blk_items = blk["items"] / max(1, blk["launches"])
    flop_blk = WIDEST["flop_blocks_head"] if widest else FLOP_BLOCKS
    achieved = flop_blk * blk_items / (blk_ms * 1e-3) / 1e12 if blk_ms > 0 else 0.0
    total_stage_ms = sum(s["ms"] for s in stages.values()) or 1.0
    crop = stages["crop"]
    # a kernel timed alone in a sub-second region runs at burst clocks: the burst cuBLAS figure is the honest denominator; a
    # seconds-long power-capped region (the widest config) takes the sustained one
    timed_s = ms / 1e3
    burst = timed_s < 1.0
    peak_tf = peaks["bf16_tflops"] if burst else peaks["bf16_tflops_sustained"]
    kernel = "gemm_tc_kernel (blocks + head stage of the generic path)" if widest else {"simt": "blocks_simt_kernel", "tcgen05": "blocks_tc_kernel<1>", "tcgen05_3term": "blocks_tc_kernel<3>"}[args.blocks]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if args.total_tracks > 0 else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
        "roofline": {"kernel": kernel, "bound": "tensor",
                     "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": achieved / peak_tf, "traffic": None if widest else ncu_traffic(args.blocks, blk_items),
                     "peak_source": peaks["source"] + (", bf16 dense burst (timed region %.0f ms < 1 s)" % (timed_s * 1e3) if burst
                                                      else ", bf16 dense sustained (timed region %.1f s)" % timed_s),
                     "frac_of_sustained_peak": achieved / peaks["bf16_tflops_sustained"],
                     "algorithmic_flop_per_launch": flop_blk * blk_items, "avg_launch_ms": blk_ms,
                     "share_of_step": blk["ms"] / total_stage_ms},
        "stages": {k: {"ms_per_step": v["ms"] / K, "share": v["ms"] / total_stage_ms, "launches_per_step": v["launches"] / K}
                   for k, v in stages.items()},
        "clocks": clocks,
        "parity_spot": parity,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "h2d_cap_gbs": float(sum(cap_ranks)), "h2d_cap_gbs_per_rank": cap_ranks,
                "h2d_cap_frames_per_s": float(sum(cap_ranks)) * 1e9 / (h2d / n),
                "frac_of_h2d_cap": e2e_value / (float(sum(cap_ranks)) * 1e9 / (h2d / n)),
                # every rank moves the same bytes per step and the step time is the max over ranks: the slowest rank's link sets the pace
                "h2d_cap_frames_per_s_at_slowest_rank": world * min(cap_ranks) * 1e9 / (h2d / n),
                "frac_of_slowest_rank_cap": e2e_value / (world * min(cap_ranks) * 1e9 / (h2d / n)),
                "binding": binding,
                "note": "per step: H2D of all %d frames + boxes from pinned host memory (upload of step t+1 overlaps compute "
                        "of step t on a copy stream), step, D2H of the boxes; h2d_cap_gbs = pinned host -> HBM bandwidth measured in this run "
                        "with every rank copying at once (the limiter of this leg: %d bytes per tracked frame)" % (F, h2d // n)},
        "gpu_launches": int(launches),
    }
    if strong is not None:
        line["strong_8192"] = strong
    if crop["ms"] > 0:
        line["stages"]["crop"]["note"] = "HBM-bound gather; see profiles/ for achieved GB/s"
    if not widest:
        try:
            line["roofline_hbm"] = hbm_rooflines(O.synth_boxes(n, FRAME_H, FRAME_W, seed=3000 + 97 * rank), stages, peaks)
        except Exception as e:                             # secondary figures: never at the expense of the line
            line["roofline_hbm"] = {"error": f"{type(e).__name__}: {e}"}

    if world == 1 and not args.no_gpu_eager:
        try:
            line["gpu_eager"] = gpu_eager_leg(sd, dev, depth, heads, batches=(64, 1) if widest else (1024, 1))
        except Exception as e:
            line["gpu_eager"] = {"error": f"{type(e).__name__}: {e}"}
    if world == 1 and not args.no_latency and not widest:
        line["latency_b1"] = latency_b1(cfg, sd, iters=args.latency_frames)
        try:
            line["e2e_sequences"] = e2e_sequences_leg(cfg, dev)
        except Exception as e:
            line["e2e_sequences"] = {"error": f"{type(e).__name__}: {e}"}
    if world == 1 and not args.no_cpu_baseline:
        if widest:
            line["cpu_baseline"] = cpu_widest_sample(sd)
        else:
            v, cores, sample = cpu_sample(sd)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "cpu_model": cpu_model_name(), "os_cpu_count": os.cpu_count()}
            try:                                           # SURVEY 8d: the reference's own batch-1 shape, all threads and one thread
                line["cpu_baseline"]["batch1_frames_per_s"] = {"all_threads": cpu_b1_sample(sd, cores), "one_thread": cpu_b1_sample(sd, 1)}
            except Exception as e:
                line["cpu_baseline"]["batch1_frames_per_s"] = {"error": f"{type(e).__name__}: {e}"}
    print(json.dumps(line, default=float), file=_JSON_OUT, flush=True)     # default: NumPy scalars, should one slip in
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def e2e_sequences_leg(cfg, dev, slots=128, length=9, distinct=16):
    """The reference's own mode through the batched driver: ONE target per sequence (run_sequences / MultiSequenceRunner,
    lib/test/evaluation/running.py + tracker.py), `slots` synthetic 720p sequences of `length` frames advanced concurrently, frames
    handed over as host arrays (no image decode), closed loop with scale-stable weights.  Per step and sequence the backend stages
    only the frame rows the search crop can read, uploads, tracks, reads the boxes back.  Wall clock around runner.run()."""
    from oracle import vt_oracle as O
    from vittracker_b200.sequences import BatchedBackend, MultiSequenceRunner, Sequence
    sd = O.make_state_dict(seed=1, stress=True, stable_size=True)
    pool = O.synth_frames(distinct, FRAME_H, FRAME_W, seed=900, smooth=True)
    rng = np.random.default_rng(901)
    seqs = []
    for i in range(slots):
        w, h = rng.uniform(60, 160), rng.uniform(60, 160)
        box = [float(rng.uniform(100, FRAME_W - 100 - w)), float(rng.uniform(100, FRAME_H - 100 - h)), float(w), float(h)]
        seqs.append(Sequence(f"s{i}", [pool[(i + k) % distinct] for k in range(length)], box))
    backend = BatchedBackend(cfg, sd, slots, device=dev.index)
    runner = MultiSequenceRunner(backend, slots, read_workers=0)
    try:
        runner.run(seqs[:8])                                           # warm-up (allocations, first launches)
        backend.bytes_uploaded = 0
        t0 = time.perf_counter()
        res = runner.run(seqs)
        el = time.perf_counter() - t0
    finally:
        runner.close()
        backend.close()
    tracked = sum(len(r.get("target_bbox", [1])) - 1 for r in res.values())
    return {"value": tracked / el, "unit": UNIT, "sequences": slots, "frames_per_sequence": length, "tracked_frames": tracked,
            "wall_s": el, "h2d_bytes_per_tracked_frame": backend.bytes_uploaded / max(1, tracked + slots),
            "full_frame_bytes": FRAME_H * FRAME_W * 3,
            "note": "one target per sequence (the reference's mode), host numpy frames in, boxes out; row-staged uploads; includes initialize()"}


def cpu_widest_sample(sd, budget_s=15.0):
    """cpu_baseline of the widest configuration: forward(z, x) of the oracle graph at batch 4 on all host cores (crop excluded: ~1 % of it)."""
    from oracle import vt_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = O.OracleModel(sd, depth=WIDEST["depth"], num_heads=12)
    z, x = torch.randn(4, 3, 128, 128), torch.randn(4, 3, 256, 256)
    model.forward(z, x)
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        model.forward(z, x)
        done += 4
    el = time.perf_counter() - t0
    return {"value": done / el, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{done} forwards (batch 4) of the widest config in {el:.1f} s; crop / decode excluded",
            "cpu_model": cpu_model_name(), "os_cpu_count": os.cpu_count()}


def latency_b1(cfg, sd, frames_n=8, iters=10000, burst=8):
    """BASELINE configs[1] (SURVEY 8d, C2): batch-1 initialize() + track() loop through the drop-in tracker (host numpy
    frame in, Python list out), wall clock per call.  `iters` open-loop frames (state re-seeded per frame), then
    closed-loop bursts of `burst` frames after a re-initialisation (iters // 40 bursts), initialize() timed as well."""
    from oracle import vt_oracle as O
    from vittracker_b200 import get_tracker_class, parameters
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    trk = get_tracker_class()(params, "synthetic")
    frames = O.synth_frames(frames_n, FRAME_H, FRAME_W, seed=77)
    boxes = O.synth_boxes(iters + 20, FRAME_H, FRAME_W, seed=78)
    trk.initialize(frames[0], {"init_bbox": list(boxes[0])})
    lat = []
    for i in range(iters + 20):
        trk.state = list(boxes[i])                      # open loop: re-seeded state per frame
        t0 = time.perf_counter()
        trk.track(frames[i % frames_n], {})
        lat.append(time.perf_counter() - t0)
    lat = np.array(lat[20:]) * 1e3
    out = {"p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)), "frames": iters,
           "path": "Vit_dist.track(): host frame rectangle H2D + crop + forward + decode + D2H, blocking",
           "cuda_graph": getattr(trk, "_graph", None) is not None}
    n_bursts = iters // 40
    if n_bursts > 0 and burst > 0:
        try:
            out.update(_latency_bursts(trk, frames, boxes, frames_n, n_bursts, burst))
        except Exception as e:                         # the headline line must not depend on this leg
            out["closed_loop"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def _latency_bursts(trk, frames, boxes, frames_n, n_bursts, burst):
    lat_c, lat_i = [], []
    for b in range(n_bursts):
        t0 = time.perf_counter()
        trk.initialize(frames[b % frames_n], {"init_bbox": list(boxes[b])})
        lat_i.append(time.perf_counter() - t0)
        for k in range(burst):                          # closed loop: the tracker follows its own state
            t0 = time.perf_counter()
            trk.track(frames[(b + 1 + k) % frames_n], {})
            lat_c.append(time.perf_counter() - t0)
    lat_c, lat_i = np.array(lat_c) * 1e3, np.array(lat_i) * 1e3
    return {"closed_loop": {"p50_ms": float(np.percentile(lat_c, 50)), "p99_ms": float(np.percentile(lat_c, 99)),
                            "frames": int(lat_c.size), "bursts": n_bursts, "burst": burst},
            "initialize": {"p50_ms": float(np.percentile(lat_i, 50)), "p99_ms": float(np.percentile(lat_i, 99)), "calls": n_bursts}}


if __name__ == "__main__":
    main()
