"""Generate tests/golden/*.npz by running the UNMODIFIED reference (through oracle/ref_shim.py) in
this container, and assert while doing so that oracle/vt_oracle.py reproduces it.

    python oracle/make_golden.py          # needs a checkout of the original project at oracle/_ref (or $VT_REFERENCE_ROOT); writes tests/golden/

TEST INFRASTRUCTURE.  The tests compare the oracle and the CUDA path with these recorded reference outputs, so they need
no copy of the reference.  Seeded inputs are stored as digests (oracle/golden.py), which keeps every file under 1 MB.
"""
from __future__ import annotations

import hashlib
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import golden, ref_shim, vt_oracle as O  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def golden_crops(ns):
    """sample_target from the reference on a 240x320 frame: full patches for a few boxes, sha256 for many."""
    H, W = 240, 320
    frame = O.synth_frames(1, H, W, seed=11, smooth=True)[0]
    boxes = O.synth_boxes(160, H, W, seed=12)
    # hand-picked edge cases: integer boxes at .5 rounding, borders, tiny (upscale), huge (all padding around)
    extra = np.array([[10, 10, 9, 9], [0, 0, 30, 20], [W - 25, H - 25, 25, 25], [100, 80, 3, 3], [5, 5, 1, 1],
                      [60, 40, 200, 160], [0, 0, W, H], [150.5, 100.5, 33, 31], [31, 17, 64, 64], [1, 1, 2, 2]],
                     dtype=np.float64)
    boxes = np.concatenate([extra, boxes])
    keep, hashes_x, hashes_z, hashes_mx, rf_x, rf_z, full_x, full_z, full_idx = [], [], [], [], [], [], [], [], []
    for i, b in enumerate(boxes):
        if not (O.crop_in_domain(b, 4.0, H, W) and O.crop_in_domain(b, 2.0, H, W)):
            continue
        px, rx, mx = ns.sample_target(frame, list(b), 4.0, output_sz=256)
        pz, rz, mz = ns.sample_target(frame, list(b), 2.0, output_sz=128)
        ox, orx, omx = O.sample_target_spec(frame, list(b), 4.0, 256)
        oz, orz, omz = O.sample_target_spec(frame, list(b), 2.0, 128)
        assert np.array_equal(px, ox) and np.array_equal(pz, oz), f"oracle crop != reference for box {b}"
        assert np.array_equal(mx, omx) and np.array_equal(mz, omz), f"oracle mask != reference for box {b}"
        assert rx == orx and rz == orz
        keep.append(b); hashes_x.append(sha(px)); hashes_z.append(sha(pz)); hashes_mx.append(sha(mx))
        rf_x.append(rx); rf_z.append(rz)
        if len(full_idx) < 4 or i in (3, 6):
            full_idx.append(len(keep) - 1); full_x.append(px); full_z.append(pz)
    np.savez_compressed(os.path.join(GOLDEN, "crops.npz"), frame=frame, boxes=np.array(keep),
                        sha_search=np.array(hashes_x), sha_template=np.array(hashes_z), sha_mask_search=np.array(hashes_mx),
                        rf_search=np.array(rf_x), rf_template=np.array(rf_z), full_idx=np.array(full_idx),
                        full_search=np.stack(full_x), full_template=np.stack(full_z))
    print(f"crops.npz: {len(keep)} boxes x (search, template), all equal to the oracle")
    return frame


def golden_model(ns, frame):
    """Reference build_ostrack_dist(cfg).forward(z, x) on stress-init weights and real crops."""
    sd_kw = dict(seed=1, stress=True)
    sd = O.make_state_dict(**sd_kw)
    cfg = ref_shim.reference_cfg()
    net = ns.build_ostrack_dist(cfg)
    net.load_state_dict(sd, strict=True)
    net.eval()
    pre = ns.data_utils.Preprocessor()
    H, W = frame.shape[:2]
    boxes = [[120.0, 90.0, 40.0, 30.0], [30.0, 20.0, 90.0, 70.0]]
    zs, xs, zp, xp = [], [], [], []
    for b in boxes:
        pz, _, mz = ns.sample_target(frame, b, 2.0, output_sz=128)
        px, _, mx = ns.sample_target(frame, [b[0] + 7, b[1] - 5, b[2] * 1.1, b[3] * 0.9], 4.0, output_sz=256)
        zs.append(pre.process(pz, mz).tensors); xs.append(pre.process(px, mx).tensors)
        zp.append(pz); xp.append(px)
        assert torch.equal(zs[-1], O.preprocess(pz)) and torch.equal(xs[-1], O.preprocess(px)), "preprocess differs"
    z, x = torch.cat(zs), torch.cat(xs)
    with torch.no_grad():
        ref = net.forward(z=z.clone(), x=x.clone())
    taps = {}
    om = O.OracleModel(sd)
    out = om.forward(z, x, taps)
    for k in ref:
        d = (ref[k] - out[k]).abs().max().item()
        assert d <= 1e-6, f"oracle {k} differs from reference by {d}"
    win = ns.hann.hann2d(torch.tensor([16, 16]).long(), centered=True)
    assert torch.equal(win, O.hann2d(16, 16))
    resp = win * ref["score_map"]
    ref_boxes_win = net.box_head.cal_bbox(resp, ref["size_map"], ref["offset_map"])
    assert torch.equal(ref_boxes_win, om.cal_bbox(resp, out["size_map"], out["offset_map"]))
    arrs = golden.seeded("make_state_dict", "w::", **sd_kw)
    arrs.update(z_patch=np.stack(zp), x_patch=np.stack(xp), hann=win.numpy(),
                pred_boxes=ref["pred_boxes"].numpy(), score_map=ref["score_map"].numpy(),
                size_map=ref["size_map"].numpy(), offset_map=ref["offset_map"].numpy(),
                pred_boxes_windowed=ref_boxes_win.numpy(),
                argmax_windowed=resp.flatten(1).argmax(1).numpy())
    for k in ("tokens0", "tokens1", "tokens2", "tokens3", "tokens_norm"):
        arrs[f"tap::{k}"] = taps[k].numpy()
    np.savez_compressed(os.path.join(GOLDEN, "model.npz"), **arrs)
    print("model.npz: reference forward == oracle forward (<=1e-6), windowed boxes equal")
    return sd


def golden_track(ns, sd):
    """Reference Vit_dist.initialize()/track() closed loop, default and scale-stable weights."""
    H, W = 240, 320
    frames_kw, stable_kw = dict(n=4, H=H, W=W, seed=21, smooth=True), dict(seed=2, stress=True, stable_size=True)
    frames = O.synth_frames(**frames_kw)
    out = golden.seeded("synth_frames", "frames", **frames_kw)
    for tag, sdict in (("stress", sd), ("stable", O.make_state_dict(**stable_kw))):
        with tempfile.TemporaryDirectory() as tmp:
            trk = ref_shim.build_reference_tracker(sdict, tmp)
        otrk = O.OracleTracker(O.OracleModel(sdict))
        otrk_cv = O.OracleTracker(O.OracleModel(sdict), use_cv=True)
        init = [140.0, 100.0, 36.0, 28.0]
        trk.initialize(frames[0], {"init_bbox": list(init)})
        otrk.initialize(frames[0], {"init_bbox": list(init)})
        otrk_cv.initialize(frames[0], {"init_bbox": list(init)})
        assert np.array_equal(trk.z_patch_arr, otrk.z_patch_arr)
        states, confs = [], []
        for t in range(1, 9):
            r = trk.track(frames[t % 4], {})
            o = otrk.track(frames[t % 4], {})
            oc = otrk_cv.track(frames[t % 4], {})
            assert list(r["target_bbox"]) == list(o["target_bbox"]) == list(oc["target_bbox"]), \
                f"{tag} frame {t}: reference {r['target_bbox']} oracle {o['target_bbox']}"
            assert float(r["confidence"]) == float(o["confidence"])
            states.append([float(v) for v in r["target_bbox"]]); confs.append(float(r["confidence"]))
        out[f"{tag}_init"] = np.array(init)
        out[f"{tag}_states"] = np.array(states, dtype=np.float64)
        out[f"{tag}_conf"] = np.array(confs, dtype=np.float64)
        if tag == "stable":
            out.update(golden.seeded("make_state_dict", "w_stable::", **stable_kw))
        print(f"track.npz[{tag}]: 8 closed-loop frames, reference == oracle exactly; last state {states[-1]}")
    np.savez_compressed(os.path.join(GOLDEN, "track.npz"), **out)


def main():
    if not ref_shim.available():
        raise SystemExit(f"no checkout of the original project at {ref_shim.REFERENCE_ROOT}: golden vectors are recorded from it")
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(1)          # deterministic reduction order for the recorded reference outputs
    ns = ref_shim.load_reference()
    frame = golden_crops(ns)
    sd = golden_model(ns, frame)
    golden_track(ns, sd)
    for f in sorted(os.listdir(GOLDEN)):
        print(f, os.path.getsize(os.path.join(GOLDEN, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
