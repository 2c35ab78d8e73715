"""Stage-by-stage diagnosis on the GPU box: per-tap max error against the oracle, then stage timings.
Development aid (not part of the product or the test-suite); prints to stdout."""
import os
import sys
import time
import traceback

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import golden, vt_oracle as O  # noqa: E402
from vittracker_b200 import BatchedTracker, FramePool, load_cfg  # noqa: E402
from vittracker_b200.engine import Engine  # noqa: E402

blocks = sys.argv[1] if len(sys.argv) > 1 else "tcgen05"
cfg = load_cfg()
print("device", torch.cuda.get_device_name(0), "blocks_impl", blocks)


def section(name, fn):
    print(f"--- {name}")
    try:
        fn()
    except Exception:
        traceback.print_exc()
    sys.stdout.flush()


g = golden.load(os.path.join(ROOT, "tests", "golden", "model.npz"))
sd = {k[3:]: torch.from_numpy(np.array(g[k])) for k in g if k.startswith("w::")}
eng = Engine(cfg, max_tracks=512, chunk_tracks=128, blocks_impl=blocks)
eng.load_state_dict(sd)


def crop():
    frame = O.synth_frames(1, 360, 480, seed=1, smooth=True)[0]
    boxes = O.synth_boxes(16, 360, 480, seed=2)
    dev = eng.device
    f = torch.from_numpy(frame).to(dev).reshape(-1)
    out = eng.crop_normalize(f, torch.zeros(16, dtype=torch.int64, device=dev), torch.tensor([[360, 480]] * 16, dtype=torch.int32, device=dev),
                             torch.tensor(boxes, device=dev), 4.0, 256, want_u8=True, want_mask=True)
    u8 = out["u8"].cpu().numpy()
    for i, b in enumerate(boxes):
        p, rf, m = O.sample_target_spec(frame, list(b), 4.0, 256)
        d = np.abs(u8[i].astype(int) - p)
        print(i, "status", int(out["status"][i]), "maxdiff", d.max(), "ndiff", int((d > 0).sum()), "rf_equal", float(out["resize_factor"][i]) == rf,
              "mask_ndiff", int((out["mask"][i].cpu().numpy().astype(bool) != m).sum()))


def forward():
    z = torch.cat([O.preprocess(p) for p in g["z_patch"]])
    x = torch.cat([O.preprocess(p) for p in g["x_patch"]])
    out = eng.forward(z, x, taps=True)
    taps = out["taps"].cpu().numpy()
    for i, n in enumerate(["tokens0", "tokens1", "tokens2", "tokens3", "tokens_norm"]):
        d = np.abs(taps[i] - g[f"tap::{n}"])
        print(n, "max abs err", d.max(), "mean", d.mean(), "| z part", d[:, :64].max(), "x part", d[:, 64:].max())
    for k in ("score_map", "size_map", "offset_map", "pred_boxes"):
        print(k, "max abs err", np.abs(out[k].cpu().numpy() - g[k]).max())


def timing():
    n, F = 512, 32
    frames = O.synth_frames(F, 720, 1280, seed=3)
    bt = BatchedTracker(cfg, sd, max_tracks=n, chunk_tracks=256, blocks_impl=blocks)
    pool = FramePool(frames, bt.device)
    boxes = O.synth_boxes(n, 720, 1280, seed=4)
    fidx = torch.arange(n) % F
    bt.initialize(pool, fidx, boxes)
    for _ in range(2):
        bt.track(pool, fidx, update_state=False)
    torch.cuda.synchronize()
    bt.engine.profile(True)
    bt.engine.profile_read()
    t0 = time.perf_counter()
    for _ in range(5):
        bt.track(pool, fidx, update_state=False)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    st = bt.engine.profile_read()
    print(f"{n} tracks: {el / 5 * 1e3:.3f} ms/step -> {n * 5 / el:.0f} frames/s")
    for k, v in st.items():
        print(f"  {k:7s} {v['ms'] / 5:.3f} ms/step ({v['launches'] // 5} launches) -> {v['ms'] / 5 / n * 1e3:.3f} us/track")


section("crop", crop)
section("forward", forward)
section("timing", timing)
