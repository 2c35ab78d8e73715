#!/usr/bin/env python
"""Small workload for compute-sanitizer (tools/sanitize.sh): every hand-written kernel once, at sizes a 10 - 100x slowdown can afford.
Fast path (vit_48_h32): tracks_init + two closed-loop steps of 5 tracks, then track records out and back in, then two targets per NV12 surface (surface union + surface conversion kernels), on tcgen05 (crop_taps, crop_conv1, conv_s2_tc x3, blocks_tc,
head_tc), the same on the fp32 CUDA-core kernels, vt_forward, vt_crop_normalize, vt_cal_bbox.  Generic path (C 96 / 3 heads / depth 2 /
head 64): tracks + forward (im2col, gemm_tc_kernel NT / NN, sgemm, layernorm, softmax, decode)."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import vt_oracle as O
from oracle import yuv420 as Y
from vittracker_b200 import BatchedTracker, FramePool, YuvSurfaces, load_cfg

which = sys.argv[1] if len(sys.argv) > 1 else "all"
frames = O.synth_frames(2, 360, 640, seed=7, smooth=True)
boxes = O.synth_boxes(5, 360, 640, seed=8)
if which in ("all", "fast"):
    for blocks in ("tcgen05", "simt"):
        bt = BatchedTracker(load_cfg(), O.make_state_dict(seed=3, stress=True), max_tracks=5, chunk_tracks=3, blocks_impl=blocks)
        pool = FramePool(frames, bt.device)
        assert int(bt.initialize(pool, torch.zeros(5, dtype=torch.int64), boxes).abs().sum()) == 0
        for t in range(2):
            out = bt.track(pool, torch.full((5,), (t + 1) % 2, dtype=torch.int64), update_state=True)
        recs = bt.export_tracks(slots=[4, 0, 2])                   # track records: export and import kernels, by range and by slot
        assert int(bt.import_tracks(recs, slots=[1, 3, 0]).abs().sum()) == 0
        assert int(bt.import_tracks(bt.export_tracks()).abs().sum()) == 0
        surf = YuvSurfaces.from_frames(torch.from_numpy(Y.synth_yuv420(2, 360, 640, seed=9)).to(bt.device), "nv12")
        assert int(bt.initialize_yuv(surf, boxes, surface=[0, 1, 0, 1, 0]).abs().sum()) == 0
        bt.track_yuv(surf, surface=torch.tensor([1, 0, 1, 0, 1], device=bt.device), slots=[4, 3, 2, 1, 0])
        z = torch.randn(3, 3, 128, 128)
        x = torch.randn(3, 3, 256, 256)
        fw = bt.engine.forward(z, x, taps=True)
        bt.engine.cal_bbox(fw["score_map"], fw["size_map"], fw["offset_map"])
        bt.engine.crop_normalize(pool.data, pool.offsets(torch.zeros(5, dtype=torch.int64, device=bt.device)), pool.hw(5),
                                 torch.tensor(boxes, device=bt.device), 4.0, 256, want_u8=True, want_mask=True)
        torch.cuda.synchronize()
        assert torch.isfinite(out).all()
        print("fast path", blocks, "OK", out[0].tolist())
        del bt
if which in ("all", "generic"):
    # C = 96: converting GEMM (gemm_tc_kernel) + CUDA-core GEMM;  C = 128: split-image GEMM (gemm_img_kernel, layernorm_img, im2col_img)
    for C, heads in ((96, 3), (128, 2)):
        cfg = load_cfg()
        cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.BACKBONE.DEPTH, cfg.MODEL.HEAD.NUM_CHANNELS = C, heads, 2, 64
        sd = O.make_state_dict(seed=21, stress=True, C=C, depth=2, head_ch=64)
        bt = BatchedTracker(cfg, sd, max_tracks=3, chunk_tracks=2, depth=2)
        pool = FramePool(frames, bt.device)
        assert int(bt.initialize(pool, torch.zeros(3, dtype=torch.int64), boxes[:3]).abs().sum()) == 0
        out = bt.track(pool, torch.ones(3, dtype=torch.int64), update_state=True)
        torch.cuda.synchronize()
        assert torch.isfinite(out).all()
        print("generic path C =", C, "OK", out[0].tolist())
        del bt
