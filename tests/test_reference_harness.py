"""The drop-in tracker class under the REFERENCE'S OWN evaluation harness (lib/test/evaluation/tracker.py:66-152 `_track_sequence`,
lib/test/evaluation/running.py:14-102 `_save_tracker_output`), beside the reference's own `Vit_dist` on the same sequence and weights.

The harness test runs where a checkout of the original project is present (oracle/_ref or $VT_REFERENCE_ROOT; imported through
oracle/ref_shim.py and NOT modified); without it, the drop-in class is held to the reference's recorded closed loop (tests/golden).
These tests run on the CPU, so the CUDA engine behind `vittracker_b200.tracker.Vit_dist` is replaced by a stand-in that the engine's calls (tracks_init / tracks_set_state / tracks_step / crop_normalize) with the CPU oracle.  What is under test is
everything of the product that the harness touches: the plugin surface (`__init__(params, dataset_name)`, `params.save_all_boxes`,
`initialize` returning None, `track` returning `target_bbox` / `confidence`), the host-side float64 box arithmetic, the aliasing of
`target_bbox` and `state`, `z_patch_arr`, and the result-file writer.  The kernels themselves are covered by the `-m gpu` tests."""
import os

import numpy as np
import pytest
import torch

from conftest import state_dict_from_npz
from oracle import ref_shim, vt_oracle as O


class OracleEngine:
    """Engine stand-in (CPU): same call surface and buffer conventions as vittracker_b200.engine.Engine for one track."""

    def __init__(self, sd):
        self.device = torch.device("cpu")
        self.model = O.OracleModel(sd)
        self.win = O.hann2d(16, 16)
        self.z = None
        self.box = None

    def _frame(self, frames, hw):
        H, W = int(hw[0, 0]), int(hw[0, 1])
        return frames.numpy().reshape(H, W, 3)

    def tracks_init(self, frames, offs, hw, boxes, first=0):
        im = self._frame(frames, hw)
        box = boxes[0].tolist()
        zp, _, _ = O.sample_target_cv(self._masked(im, box, 2.0), box, 2.0, 128)
        self.z = O.preprocess(zp)
        self.box = box
        return torch.zeros(1, dtype=torch.int32)

    def _masked(self, im, box, factor):
        return im          # the tracker stages only the rows the crop reads; the others are never touched by sample_target

    def tracks_set_state(self, boxes, first=0):
        self.box = boxes[0].tolist()

    def crop_normalize(self, frames, offs, hw, boxes, factor, out_size, want_u8=False, want_mask=False):
        im = self._frame(frames, hw)
        p, rf, _ = O.sample_target_cv(im, boxes[0].tolist(), factor, out_size)
        return {"u8": torch.from_numpy(p.copy())[None], "tensors": O.preprocess(p), "resize_factor": torch.tensor([rf]), "status": torch.zeros(1)}

    def tracks_step(self, frames, offs, hw, first=0, n=1, out_boxes=None, out_detail=None, update_state=False, detail=False):
        im = self._frame(frames, hw)
        xp, rf, _ = O.sample_target_cv(im, self.box, 4.0, 256)
        out = self.model.forward(self.z, O.preprocess(xp))
        resp = self.win * out["score_map"]
        pb = self.model.cal_bbox(resp, out["size_map"], out["offset_map"]).view(-1, 4)
        pred = (pb.mean(dim=0) * 256 / rf).tolist()                 # vit_dist.py:108-109
        out_boxes[0, 4] = float(out["score_map"].max())
        out_detail[0, :4] = torch.tensor(pred, dtype=torch.float64)
        out_detail[0, 4] = rf
        out_detail[0, 5] = float(resp.flatten().argmax())
        out_detail[0, 6] = 0.0
        out_detail[0, 7] = float(resp.max())
        return out_boxes, out_detail


class FakeNetwork:
    def __init__(self, sd):
        self.engine = OracleEngine(sd)

    def load_state_dict(self, sd, strict=False):
        return [], []

    def cuda(self):
        return self

    def eval(self):
        return self


@pytest.fixture()
def sequence(tmp_path):
    cv = pytest.importorskip("cv2")
    frames = O.synth_frames(7, 240, 320, seed=71, smooth=True)
    paths = []
    for k, f in enumerate(frames):
        p = str(tmp_path / f"{k:04d}.png")
        assert cv.imwrite(p, f[..., ::-1])                           # files hold BGR; _read_image converts back
        paths.append(p)
    return frames, paths, [120.5, 80.25, 60.0, 44.0]


@pytest.mark.parametrize("tag", ["stress", "stable"])
def test_dropin_class_reproduces_the_recorded_reference_closed_loop(golden_track, golden_model, tag, monkeypatch):
    """The reference's own Vit_dist.initialize()/track() on 8 frames, recorded by oracle/make_golden.py, against the drop-in class on the same
    frames and weights: the same Python numbers frame by frame (the host-side float64 map-back and clip), `target_bbox` aliasing the state."""
    g = golden_track
    sd = state_dict_from_npz(golden_model) if tag == "stress" else state_dict_from_npz(g, "w_stable::")
    torch.set_num_threads(1)                                    # the reduction order the reference was recorded with
    import vittracker_b200.tracker as vt_tracker
    from vittracker_b200 import parameters
    monkeypatch.setattr(vt_tracker, "build_ostrack_dist", lambda cfg, depth=3, **kw: FakeNetwork(sd))
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    trk = vt_tracker.get_tracker_class()(params, "synthetic")
    frames = g["frames"]
    assert trk.initialize(frames[0], {"init_bbox": [float(v) for v in g[f"{tag}_init"]]}) is None
    for t in range(1, 9):
        out = trk.track(frames[t % 4], {})
        assert out["target_bbox"] is trk.state
        assert [float(v) for v in out["target_bbox"]] == g[f"{tag}_states"][t - 1].tolist(), (tag, t)
        assert float(out["confidence"]) == g[f"{tag}_conf"][t - 1], (tag, t)


@pytest.mark.skipif(not ref_shim.available(), reason="no checkout of the original project at oracle/_ref or $VT_REFERENCE_ROOT")
def test_dropin_class_under_the_reference_harness(tmp_path, sequence, monkeypatch):
    ref = ref_shim.load_reference()
    import importlib
    ev_tracker = importlib.import_module("lib.test.evaluation.tracker")
    ev_running = importlib.import_module("lib.test.evaluation.running")
    ev_data = importlib.import_module("lib.test.evaluation.data")
    frames, paths, init_box = sequence
    sd = O.make_state_dict(seed=9, stress=True, stable_size=True)

    def make_seq(name):
        gt = np.array([init_box] + [[0, 0, 0, 0]] * (len(paths) - 1), dtype=np.float64)
        return ev_data.Sequence(name, list(paths), "synthetic", gt)

    def harness(results_dir):
        t = ev_tracker.Tracker("vit_dist", "vit_48_h32_noKD", "synthetic")
        t.results_dir = results_dir
        return t

    # --- the reference's own tracker through its own harness --------------------------------------------------------
    ref_trk = ref_shim.build_reference_tracker(sd, str(tmp_path))
    h_ref = harness(str(tmp_path / "ref"))
    seq_ref = make_seq("seq")
    out_ref = h_ref._track_sequence(ref_trk, seq_ref, seq_ref.init_info())
    ev_running._save_tracker_output(seq_ref, h_ref, out_ref)

    # --- the drop-in class through the same harness (engine = oracle stand-in) ------------------------------------
    import vittracker_b200.tracker as vt_tracker
    from vittracker_b200 import parameters
    monkeypatch.setattr(vt_tracker, "build_ostrack_dist", lambda cfg, depth=3, **kw: FakeNetwork(sd))
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    h_new = harness(str(tmp_path / "new"))
    h_new.tracker_class = vt_tracker.get_tracker_class()              # what the stub module of INTEGRATION.md hands the harness
    new_trk = h_new.create_tracker(params)
    assert new_trk.params is params and new_trk.params.save_all_boxes is False
    seq_new = make_seq("seq")
    out_new = h_new._track_sequence(new_trk, seq_new, seq_new.init_info())
    ev_running._save_tracker_output(seq_new, h_new, out_new)

    assert set(out_new) == set(out_ref) == {"target_bbox", "time"}
    assert len(out_new["target_bbox"]) == len(out_ref["target_bbox"]) == len(paths)
    for a, b in zip(out_new["target_bbox"], out_ref["target_bbox"]):
        assert [float(v) for v in a] == [float(v) for v in b], (a, b)                 # identical Python numbers, frame by frame
    assert new_trk.state is out_new["target_bbox"][-1]                                # target_bbox aliases the state (vit_dist.py:111,147)
    assert new_trk.frame_id == ref_trk.frame_id == len(paths) - 1
    assert np.array_equal(new_trk.z_patch_arr, ref_trk.z_patch_arr)                   # vit_dist.py:57
    for name in ("seq.txt",):
        assert open(os.path.join(str(tmp_path / "new"), name), "rb").read() == open(os.path.join(str(tmp_path / "ref"), name), "rb").read()

    # --- our result writer against the reference's, byte for byte ---------------------------------------------------
    from vittracker_b200.sequences import Sequence, save_tracker_output
    for dataset in ("synthetic", "got10k"):
        s_new = Sequence("seq", list(paths), init_box, dataset=dataset)
        save_tracker_output(str(tmp_path / "ours"), s_new, out_ref)
        s_ref = ev_data.Sequence("seq", list(paths), dataset, np.array([init_box], dtype=np.float64))
        h = harness(str(tmp_path / "theirs"))
        ev_running._save_tracker_output(s_ref, h, out_ref)
        sub = dataset if dataset == "got10k" else ""
        for leaf in ("seq.txt", "seq_time.txt"):
            ours = open(os.path.join(str(tmp_path / "ours"), sub, leaf), "rb").read()
            theirs = open(os.path.join(str(tmp_path / "theirs"), sub, leaf), "rb").read()
            assert ours == theirs, (dataset, leaf)


def test_track_returns_a_tensor_confidence_and_raises_like_the_reference(sequence, monkeypatch):
    frames, paths, init_box = sequence
    sd = O.make_state_dict(seed=9, stress=True)
    import vittracker_b200.tracker as vt_tracker
    from vittracker_b200 import parameters
    monkeypatch.setattr(vt_tracker, "build_ostrack_dist", lambda cfg, depth=3, **kw: FakeNetwork(sd))
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    trk = vt_tracker.Vit_dist(params, "synthetic")
    assert trk.initialize(frames[0], {"init_bbox": init_box}) is None
    out = trk.track(frames[1], {})
    assert torch.is_tensor(out["confidence"]) and out["confidence"].dim() == 0 and out["confidence"].dtype == torch.float32
    assert isinstance(out["target_bbox"], list) and len(out["target_bbox"]) == 4
    with pytest.raises(Exception, match="Too small bounding box"):
        trk.initialize(frames[0], {"init_bbox": [10.0, 10.0, 0.0, 0.0]})
