"""CPU: the oracle against the golden vectors recorded from the reference (tests/golden, written by
oracle/make_golden.py) and against OpenCV; re-pins against the reference itself where a checkout of it is present."""
import hashlib
import json

import numpy as np
import pytest
import torch

from conftest import state_dict_from_npz
from oracle import golden, ref_shim, vt_oracle as O


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_crop_spec_matches_reference_golden(golden_crops):
    g = golden_crops
    frame, boxes = g["frame"], g["boxes"]
    for i, b in enumerate(boxes):
        px, rx, mx = O.sample_target_spec(frame, list(b), 4.0, 256)
        pz, rz, _ = O.sample_target_spec(frame, list(b), 2.0, 128)
        assert sha(px) == str(g["sha_search"][i]) and sha(pz) == str(g["sha_template"][i]), f"box {i} {b}"
        assert sha(mx) == str(g["sha_mask_search"][i])
        assert rx == g["rf_search"][i] and rz == g["rf_template"][i]
    for j, i in enumerate(g["full_idx"]):
        px, _, _ = O.sample_target_spec(frame, list(boxes[i]), 4.0, 256)
        assert np.array_equal(px, g["full_search"][j])


def test_crop_spec_matches_opencv_many_sizes():
    rng = np.random.default_rng(5)
    im = O.synth_frames(1, 200, 300, seed=6)[0]
    n = 0
    for side in list(range(1, 40)) + [47, 63, 64, 65, 100, 127, 128, 129, 200, 255, 256, 257, 300, 511, 513, 640, 777]:
        w = side / 4.0                                     # crop_sz == side for factor 4 (w == h)
        x, y = rng.uniform(-20, 250), rng.uniform(-20, 150)
        box = [x, y, w, w]
        for f, S in ((4.0, 256), (2.0, 128)):
            if not O.crop_in_domain(box, f, 200, 300):
                continue
            a, ra, ma = O.sample_target_spec(im, box, f, S)
            b, rb, mb = O.sample_target_cv(im, box, f, S)
            assert np.array_equal(a, b) and ra == rb and np.array_equal(ma, mb), (side, f, S)
            n += 1
    assert n > 60


def test_crop_too_small_raises():
    im = np.zeros((50, 60, 3), np.uint8)
    with pytest.raises(Exception, match="Too small"):
        O.sample_target_spec(im, [5, 5, 0, 0], 4.0, 256)


def test_preprocess_lut_equals_elementwise():
    lut = O.preprocess_lut()
    patch = np.arange(256, dtype=np.uint8).reshape(16, 16, 1).repeat(3, 2)
    t = O.preprocess(patch)[0].numpy()
    for c in range(3):
        assert np.array_equal(t[c].reshape(-1), lut[c])


def test_model_matches_reference_golden(golden_model):
    g = golden_model
    sd = state_dict_from_npz(g)
    torch.set_num_threads(1)
    m = O.OracleModel(sd)
    z = torch.cat([O.preprocess(p) for p in g["z_patch"]])
    x = torch.cat([O.preprocess(p) for p in g["x_patch"]])
    taps = {}
    out = m.forward(z, x, taps)
    for k in ("pred_boxes", "score_map", "size_map", "offset_map"):
        np.testing.assert_allclose(out[k].numpy(), g[k], rtol=0, atol=1e-6, err_msg=k)
    for k in ("tokens0", "tokens1", "tokens2", "tokens3", "tokens_norm"):
        np.testing.assert_allclose(taps[k].numpy(), g[f"tap::{k}"], rtol=1e-5, atol=1e-5, err_msg=k)
    assert np.array_equal(O.hann2d(16, 16).numpy(), g["hann"])
    resp = O.hann2d(16, 16) * out["score_map"]
    assert np.array_equal(resp.flatten(1).argmax(1).numpy(), g["argmax_windowed"])
    np.testing.assert_allclose(m.cal_bbox(resp, out["size_map"], out["offset_map"]).numpy(), g["pred_boxes_windowed"], atol=1e-6)


@pytest.mark.parametrize("tag", ["stress", "stable"])
def test_tracker_matches_reference_golden(golden_track, golden_model, tag):
    g = golden_track
    sd = state_dict_from_npz(golden_model) if tag == "stress" else state_dict_from_npz(g, "w_stable::")
    torch.set_num_threads(1)
    trk = O.OracleTracker(O.OracleModel(sd))
    frames = g["frames"]
    trk.initialize(frames[0], {"init_bbox": [float(v) for v in g[f"{tag}_init"]]})
    for t in range(1, 9):
        out = trk.track(frames[t % 4], {})
        np.testing.assert_allclose(np.array(out["target_bbox"], dtype=np.float64), g[f"{tag}_states"][t - 1], rtol=1e-5, atol=1e-3)
        assert abs(float(out["confidence"]) - g[f"{tag}_conf"][t - 1]) < 1e-5


def test_golden_seeded_inputs_are_regenerated_and_checked(tmp_path):
    entry = golden.seeded("synth_frames", "frames", n=1, H=8, W=12, seed=3)
    np.savez(tmp_path / "ok.npz", **entry, other=np.arange(3))
    g = golden.load(str(tmp_path / "ok.npz"))
    assert set(g) == {"frames", "other"} and np.array_equal(g["frames"], O.synth_frames(1, 8, 12, seed=3))
    spec = json.loads(str(entry["seeded::frames"]))
    spec["kw"]["seed"] = 4                                  # a generator that no longer gives the recorded input
    np.savez(tmp_path / "bad.npz", **{"seeded::frames": np.array(json.dumps(spec))})
    with pytest.raises(AssertionError, match="no longer reproduces"):
        golden.load(str(tmp_path / "bad.npz"))


def test_clip_box_python_semantics():
    assert O.clip_box([-5.0, 3.0, 20.0, 4.0], 100, 200, margin=10) == [0, 3.0, 15.0, 10]
    assert O.clip_box([195.0, 95.0, 20.0, 20.0], 100, 200, margin=10) == [190, 90, 10, 10]


@pytest.mark.skipif(not ref_shim.available(), reason="no checkout of the original project at oracle/_ref or $VT_REFERENCE_ROOT")
def test_oracle_repinned_against_reference_itself():
    ns = ref_shim.load_reference()
    im = O.synth_frames(1, 180, 240, seed=3, smooth=True)[0]
    for b in O.synth_boxes(25, 180, 240, seed=4):
        if not O.crop_in_domain(b, 4.0, 180, 240):
            continue
        p, r, m = ns.sample_target(im, list(b), 4.0, output_sz=256)
        q, s, k = O.sample_target_spec(im, list(b), 4.0, 256)
        assert np.array_equal(p, q) and r == s and np.array_equal(m, k)
    sd = O.make_state_dict(seed=7, stress=True)
    net = ns.build_ostrack_dist(ref_shim.reference_cfg())
    net.load_state_dict(sd, strict=True)
    net.eval()
    torch.manual_seed(1)
    z, x = torch.randn(1, 3, 128, 128), torch.randn(1, 3, 256, 256)
    with torch.no_grad():
        ref = net.forward(z=z.clone(), x=x.clone())
    out = O.OracleModel(sd).forward(z, x)
    for k in ref:
        assert (ref[k] - out[k]).abs().max().item() <= 1e-6


@pytest.mark.skipif(not ref_shim.available(), reason="no checkout of the original project at oracle/_ref or $VT_REFERENCE_ROOT")
@pytest.mark.parametrize("C,heads,depth,hc", [(96, 3, 2, 64), (40, 5, 1, 24)])
def test_oracle_generic_family_against_reference_itself(C, heads, depth, hc):
    """The generic-configuration path (BASELINE configs[4]) is checked on the GPU against the oracle at other widths / head counts /
    depths: pin the oracle there too, against the reference's own build_ostrack_dist(cfg, depth) (vit_dist.py:159-164)."""
    import copy
    ns = ref_shim.load_reference()
    cfg = copy.deepcopy(ref_shim.reference_cfg())
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.HEAD.NUM_CHANNELS = C, heads, hc
    sd = O.make_state_dict(seed=9, stress=True, C=C, depth=depth, head_ch=hc)
    net = ns.build_ostrack_dist(cfg, depth=depth)
    net.load_state_dict(sd, strict=True)
    net.eval()
    torch.manual_seed(2)
    z, x = torch.randn(2, 3, 128, 128), torch.randn(2, 3, 256, 256)
    with torch.no_grad():
        ref = net.forward(z=z.clone(), x=x.clone())
    out = O.OracleModel(sd, depth=depth, num_heads=heads).forward(z, x)
    for k in ref:
        assert ref[k].shape == out[k].shape
        assert (ref[k] - out[k]).abs().max().item() <= 1e-6, k
