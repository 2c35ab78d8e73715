#!/usr/bin/env python
"""A/B bit-identity check between two builds of libvittrack_b200.so (e.g. before / after an instruction-level
rewrite that must not change a single result bit).

    VT_LIB_DIR=<build A> python tools/ab_identity.py --dump gpurun_out/ab_a.npz
    VT_LIB_DIR=<build B> python tools/ab_identity.py --dump gpurun_out/ab_b.npz
    python tools/ab_identity.py --compare gpurun_out/ab_a.npz gpurun_out/ab_b.npz
    python tools/ab_identity.py --ab <build A dir> <build B dir>            # the same in one process
    python tools/ab_identity.py --ab <A> <B> --generic 96,3,2,64 --blocks simt   # a generic configuration: C,heads,depth,hc

The workload is 2048 seeded open-loop tracks on smooth + white-noise 360x640 frames (boxes incl. border-touching and
up-scaling cases, stress-init weights): dumped are the decoded boxes + confidence, the per-track detail row and the
score / size / offset maps of every track, and Engine.forward(z, x, taps=True) on four seeded crops of those frames (boxes,
maps and every tap), compared as raw bits."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def use_library(lib_dir: str) -> None:
    """Point the ctypes binding at another build (both builds can live in one process: dlopen handles are local)."""
    from vittracker_b200 import _lib, build as _build
    _build.LIB_PATH = os.path.join(os.path.abspath(lib_dir), "libvittrack_b200.so")
    _lib._lib = None


def dump(path: str, n: int, blocks: str, generic=None) -> None:
    from oracle import vt_oracle as O          # only the seeded synthetic inputs / weights come from the test infrastructure
    from vittracker_b200 import BatchedTracker, FramePool, load_cfg
    H, W, F = 360, 640, 8
    cfg, depth = load_cfg(), None
    if generic:                                # built as tests/test_generic_edges.py builds its configurations
        C, heads, depth, hc = generic
        cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS = C, heads
        cfg.MODEL.HEAD.NUM_CHANNELS = hc
        sd = O.make_state_dict(seed=21, stress=True, C=C, depth=depth, head_ch=hc)
    else:
        sd = O.make_state_dict(seed=21, stress=True)
    frames = np.concatenate([O.synth_frames(F // 2, H, W, seed=91, smooth=True), O.synth_frames(F - F // 2, H, W, seed=92)])
    init_boxes = O.synth_boxes(n, H, W, seed=93)
    step_boxes = O.synth_boxes(n, H, W, seed=94)
    bt = BatchedTracker(cfg, sd, max_tracks=n, chunk_tracks=0 if generic else min(1024, n), blocks_impl=blocks, depth=depth)
    pool = FramePool(frames, bt.device)
    st = bt.initialize(pool, torch.from_numpy(np.arange(n) % F), init_boxes)
    assert int(st.abs().sum()) == 0
    bt.set_state(step_boxes)
    out, det = bt.track(pool, torch.from_numpy((np.arange(n) * 7 + 3) % F), update_state=True, detail=True)
    maps = bt.engine.tracks_last_maps(0, n)
    fwd_boxes = O.synth_boxes(4, H, W, seed=95)
    z = torch.cat([O.preprocess(O.sample_target_spec(frames[0], b, O.TEMPLATE_FACTOR, O.TEMPLATE_SIZE)[0]) for b in fwd_boxes])
    x = torch.cat([O.preprocess(O.sample_target_spec(frames[1], b, O.SEARCH_FACTOR, O.SEARCH_SIZE)[0]) for b in fwd_boxes])
    fwd = bt.engine.forward(z, x, taps=True)
    torch.cuda.synchronize()
    np.savez(path, boxes=out.cpu().numpy(), detail=det.cpu().numpy(), score=maps["score_map"].cpu().numpy(),
             size=maps["size_map"].cpu().numpy(), offset=maps["offset_map"].cpu().numpy(),
             **{"fwd_" + k: v.cpu().numpy() for k, v in fwd.items()})
    print(f"dumped {n} tracks ({blocks}{', generic ' + str(generic) if generic else ''}) from {os.environ.get('VT_LIB_DIR', 'the in-tree build')} to {path}")


def compare(a: str, b: str) -> int:
    A, B = np.load(a), np.load(b)
    res = {}
    for k in A.files:
        x, y = np.ascontiguousarray(A[k]), np.ascontiguousarray(B[k])
        same = x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))
        res[k] = {"identical_bits": bool(same), "elements": int(x.size),
                  "max_abs_diff": 0.0 if same else float(np.nanmax(np.abs(x.astype(np.float64) - y.astype(np.float64))))}
    ok = all(v["identical_bits"] for v in res.values())
    print(json.dumps({"a": a, "b": b, "bit_identical": ok, "arrays": res}))
    return 0 if ok else 1


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump")
    ap.add_argument("--compare", nargs=2)
    ap.add_argument("--n", type=int, default=2048)
    ap.add_argument("--blocks", default="tcgen05")
    ap.add_argument("--generic", type=lambda v: tuple(int(t) for t in v.split(",")), metavar="C,heads,depth,hc",
                    help="a generic configuration instead of vit_48_h32")
    ap.add_argument("--ab", nargs=2, metavar=("LIB_DIR_A", "LIB_DIR_B"), help="dump both builds in this process and compare")
    a = ap.parse_args()
    if a.compare:
        sys.exit(compare(*a.compare))
    if a.ab:
        import tempfile
        tmp = tempfile.mkdtemp()
        paths = []
        for tag, d in zip("ab", a.ab):
            use_library(d)
            paths.append(os.path.join(tmp, f"{tag}.npz"))
            dump(paths[-1], a.n, a.blocks, a.generic)
        sys.exit(compare(*paths))
    dump(a.dump, a.n, a.blocks, a.generic)
