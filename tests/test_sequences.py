"""Batched multi-sequence driver (SURVEY 8f rank 1 + rank 4): scheduling over ragged sequences and the reference's result
files, on a fake backend (no GPU); and on the GPU, equality with the drop-in tracker run sequence by sequence."""
import os

import numpy as np
import pytest

from vittracker_b200.sequences import MultiSequenceRunner, Sequence, results_path, run_sequences, save_tracker_output


class FakeBackend:
    """Box of a slot after k steps = init box + k in x; remembers which slot served which frame, the slots of every initialisation
    and every step, and checks that each step lists exactly the slots whose sequence is running (see _runner)."""

    def __init__(self, slots):
        self.state = [None] * slots
        self.log = []
        self.batches = []
        self.calls = []
        self.runner = None

    def initialize_many(self, items):
        self.batches.append([slot for (slot, _, _) in items])
        errors = []
        for slot, image, box in items:
            if box[2] <= 0:
                errors.append(Exception("Too small bounding box."))
                continue
            self.state[slot] = [float(v) for v in box]
            errors.append(None)
        return errors

    def step_active(self, slots, images):
        running = [i for i, s in enumerate(self.runner.slots) if s.seq is not None]
        assert list(slots) == running and len(images) == len(slots)
        self.calls.append(list(slots))
        out = np.zeros((len(slots), 5))
        for j, (i, im) in enumerate(zip(slots, images)):
            assert self.state[i] is not None
            self.state[i][0] += 1.0
            self.log.append((i, int(im[0, 0, 0])))
            out[j, :4] = self.state[i]
            out[j, 4] = 0.5
        return out


def _runner(be, slots, **kw):
    """A runner over the fake backend `be`, which checks every step against this runner's running slots."""
    be.runner = MultiSequenceRunner(be, slots, **kw)
    return be.runner


def _frames(n, tag):
    return [np.full((4, 4, 3), tag, dtype=np.uint8) for _ in range(n)]


def test_scheduler_ragged_sequences_and_result_files(tmp_path):
    lengths = [5, 1, 3, 7, 2, 4]
    seqs = [Sequence(f"s{i}", _frames(n, i), [10.0 * i + 0.7, 5.9, 20.5, 30.2], dataset="got10k" if i == 2 else "") for i, n in enumerate(lengths)]
    seqs.append(Sequence("bad", _frames(3, 9), [1.0, 1.0, 0.0, 5.0]))          # init fails: reported and skipped
    be = FakeBackend(3)
    res = _runner(be, 3, results_dir=str(tmp_path)).run(seqs)
    assert set(res) == {f"s{i}" for i in range(len(lengths))}
    assert sum(len(c) for c in be.calls) == sum(n - 1 for n in lengths)         # every tracked frame stepped once, nothing else
    assert any(len(c) < 3 for c in be.calls)                                    # the run drains: the last steps list fewer slots
    for i, n in enumerate(lengths):
        out = res[f"s{i}"]
        if n == 1:
            assert "target_bbox" not in out and len(out["time"]) == 1       # tracker.py:148-150
            continue
        assert len(out["target_bbox"]) == n and len(out["time"]) == n
        assert out["target_bbox"][0] == seqs[i].init_bbox
        assert [b[0] for b in out["target_bbox"]] == [seqs[i].init_bbox[0] + k for k in range(n)]
        # every frame of the sequence was served by one slot, in order
        assert [t for (_, t) in be.log if t == i] == [i] * (n - 1)
    # the reference's file format: ints, tab separated; got10k goes into its own folder
    got = np.loadtxt(results_path(str(tmp_path), seqs[0]) + ".txt", delimiter="\t")
    assert got.shape == (5, 4) and got[0].tolist() == [0, 5, 20, 30] and got[3].tolist() == [3, 5, 20, 30]
    assert os.path.isfile(os.path.join(str(tmp_path), "got10k", "s2.txt"))
    assert np.loadtxt(results_path(str(tmp_path), seqs[0]) + "_time.txt").shape == (5,)
    # resumable: sequences whose results exist are skipped (running.py:116-131)
    be2 = FakeBackend(3)
    res2 = _runner(be2, 3, results_dir=str(tmp_path)).run(seqs[:5])
    assert set(res2) == {"s1"} and not be2.log            # s1 has a single frame: no box file is ever written for it


def test_free_slots_are_initialised_together_when_the_backend_can(tmp_path):
    """The backend gets every free slot in ONE initialize_many call per refill round; a sequence whose initialisation fails is reported,
    skipped and its slot offered to the next pending sequence (running.py:135-142); every other sequence is tracked to its end."""
    lengths = [4, 2, 6, 3, 5, 1, 4]
    seqs = [Sequence(f"s{i}", _frames(n, i), [10.0 * i + 1, 5.0, 20.0, 30.0]) for i, n in enumerate(lengths)]
    seqs.insert(2, Sequence("bad", _frames(3, 9), [1.0, 1.0, 0.0, 5.0]))                # fails inside the first batch
    be = FakeBackend(3)
    res = _runner(be, 3).run(seqs)
    assert set(res) == {f"s{i}" for i in range(len(lengths))}
    for i, n in enumerate(lengths):
        out = res[f"s{i}"]
        assert len(out["time"]) == n
        if n == 1:
            assert "target_bbox" not in out
            continue
        assert out["target_bbox"] == [[10.0 * i + 1 + k, 5.0, 20.0, 30.0] for k in range(n)]
    assert be.batches[0] == [0, 1, 2]                       # all three slots at once ...
    assert be.batches[1] == [2]                             # ... and the failed one again, with the next pending sequence
    assert all(len(b) >= 1 for b in be.batches)


def test_threaded_frame_ingest_from_image_files(tmp_path):
    """SURVEY 8f rank 2: frames given as image paths are decoded (cv.imread + BGR2RGB, tracker.py:282-289) by reader threads, the next
    step's frames while the current step runs - same frames, same order, same results as decoding on the calling thread; a sequence
    whose frame cannot be read is reported and dropped without disturbing the others."""
    cv = pytest.importorskip("cv2")
    lengths = [6, 3, 9, 4, 5]
    seqs = []
    for i, n in enumerate(lengths):
        paths = []
        for k in range(n):
            rgb = np.zeros((6, 8, 3), dtype=np.uint8)
            rgb[..., 0], rgb[..., 1], rgb[..., 2] = i, k, 200             # R = sequence, G = frame index
            path = str(tmp_path / f"s{i}_{k:03d}.png")
            assert cv.imwrite(path, rgb[..., ::-1])                       # files hold BGR
            paths.append(path)
        seqs.append(Sequence(f"s{i}", paths, [10.0 * i, 5.0, 20.0, 30.0]))

    class Recorder(FakeBackend):
        def step_active(self, slots, images):
            for i, im in zip(slots, images):
                assert im.shape == (6, 8, 3) and int(im[0, 0, 2]) == 200              # RGB order restored
                self.log.append(("frame", i, int(im[0, 0, 0]), int(im[0, 0, 1])))
            return super().step_active(slots, images)

    def run(workers, sequences):
        be = Recorder(2)
        r = _runner(be, 2, read_workers=workers)
        try:
            return r.run(sequences), be
        finally:
            r.close()

    res0, be0 = run(0, seqs)
    res4, be4 = run(4, seqs)
    assert set(res0) == set(res4) == {f"s{i}" for i in range(len(lengths))}
    for name in res0:
        assert res0[name]["target_bbox"] == res4[name]["target_bbox"]
    frames0 = [e for e in be0.log if e[0] == "frame"]
    frames4 = [e for e in be4.log if e[0] == "frame"]
    assert frames0 == frames4
    for i, n in enumerate(lengths):                                       # every sequence saw its frames 1 .. n-1 in order
        assert [k for (_, _, s, k) in frames4 if s == i] == list(range(1, n))

    os.remove(seqs[2].frames[4])                                          # s2 breaks at frame 4
    res, be = run(4, seqs)
    assert set(res) == {"s0", "s1", "s3", "s4"}
    for name in res:
        assert res[name]["target_bbox"] == res0[name]["target_bbox"]
    assert [e[3] for e in be.log if e[0] == "frame" and e[2] == 2] == [1, 2, 3]


def test_read_image_branches_match_the_reference_reader(tmp_path, monkeypatch):
    """read_image = Tracker._read_image (tracker.py:282-289): path -> cv.imread + BGR2RGB; [lmdb_file, key] -> LMDB value ->
    cv.imdecode + BGR2RGB (lmdb_utils.py:23-30).  lmdb is not in this image: the lookup runs against an in-memory stand-in module."""
    cv = pytest.importorskip("cv2")
    import sys
    import types
    from vittracker_b200 import sequences as S
    rng = np.random.default_rng(1)
    rgb = rng.integers(0, 256, size=(12, 20, 3), dtype=np.uint8)
    path = str(tmp_path / "f.png")
    assert cv.imwrite(path, rgb[..., ::-1])
    assert np.array_equal(S.read_image(path), rgb)
    ok, enc = cv.imencode(".png", rgb[..., ::-1])
    assert ok and np.array_equal(S.read_image(enc.tobytes()), rgb)
    store = {"seq/0001.png": enc.tobytes()}
    opened = []

    class _Txn:
        def get(self, key):
            return store.get(key.decode())

    class _Env:
        def begin(self, write=False):
            return _Txn()

    fake = types.ModuleType("lmdb")
    fake.open = lambda name, **kw: (opened.append((name, kw)), _Env())[1]
    monkeypatch.setitem(sys.modules, "lmdb", fake)
    S._LMDB_HANDLES.clear()
    assert np.array_equal(S.read_image(["db.lmdb", "seq/0001.png"]), rgb)
    assert np.array_equal(S.read_image(["db.lmdb", "seq/0001.png"]), rgb) and len(opened) == 1      # the handle is cached (lmdb_utils.py:11-20)
    assert opened[0][1] == dict(readonly=True, lock=False, readahead=False, meminit=False)
    with pytest.raises(FileNotFoundError):
        S.read_image(["db.lmdb", "missing"])
    with pytest.raises(ValueError):
        S.read_image(42)
    S._LMDB_HANDLES.clear()


def test_crop_rows_cover_what_sample_target_reads():
    """Row staging uploads rows [ya, yb) of a frame: exactly the slice sample_target takes (processing_utils.py:34-48)."""
    from oracle import vt_oracle as O
    from vittracker_b200.sequences import crop_rows
    H, W = 240, 320
    rng = np.random.default_rng(3)
    im = rng.integers(1, 255, size=(H, W, 3), dtype=np.uint8)
    for _ in range(300):
        w, h = rng.uniform(2, 200), rng.uniform(2, 200)
        box = [rng.uniform(-20, W), rng.uniform(-40, H + 20), w, h]
        if rng.random() < 0.2:
            box = [float(round(v)) for v in box]                      # .5 rounding cases
        r = crop_rows(box, 4.0, H)
        if not O.crop_in_domain(box, 4.0, H, W):
            continue
        assert r is not None
        ya, yb = r
        masked = np.zeros_like(im)
        masked[ya:yb] = im[ya:yb]                                     # rows outside the ROI never matter
        a = O.sample_target_cv(im, box, 4.0, 256)[0]
        b = O.sample_target_cv(masked, box, 4.0, 256)[0]
        assert np.array_equal(a, b), (box, r)
    assert crop_rows([10, 10, 0, 0], 4.0, H) is None


def test_crop_rect_covers_what_sample_target_reads():
    """The batch-1 tracker uploads rows [ya, yb) x columns [xa, xb) of a frame (vt_upload_frame_rect): everything sample_target reads
    (processing_utils.py:34-48) lies inside, for search and template crops, boxes over every border, up-scaling crops and .5 rounding."""
    from oracle import vt_oracle as O
    from vittracker_b200.sequences import crop_rect
    H, W = 240, 320
    rng = np.random.default_rng(4)
    im = rng.integers(1, 255, size=(H, W, 3), dtype=np.uint8)
    checked = 0
    for k in range(400):
        factor, S = ((4.0, 256), (2.0, 128))[k % 2]
        w, h = rng.uniform(2, 200), rng.uniform(2, 200)
        box = [rng.uniform(-60, W + 20), rng.uniform(-40, H + 20), w, h]
        if rng.random() < 0.2:
            box = [float(round(v)) for v in box]
        if not O.crop_in_domain(box, factor, H, W):
            continue
        r = crop_rect(box, factor, H, W)
        assert r is not None, box
        ya, yb, xa, xb = r
        assert 0 <= ya < yb <= H and 0 <= xa < xb <= W
        masked = np.zeros_like(im)
        masked[ya:yb, xa:xb] = im[ya:yb, xa:xb]
        a = O.sample_target_cv(im, box, factor, S)[0]
        b = O.sample_target_cv(masked, box, factor, S)[0]
        assert np.array_equal(a, b), (box, r)
        checked += 1
    assert checked > 150
    assert crop_rect([10, 10, 0, 0], 4.0, H, W) is None
    assert crop_rect([W + 500.0, 10, 20, 20], 4.0, H, W) is None          # the crop misses the frame horizontally


def test_save_tracker_output_truncates_like_astype_int(tmp_path):
    s = Sequence("q", _frames(2, 0), [1, 2, 3, 4])
    save_tracker_output(str(tmp_path), s, {"target_bbox": [[1.9, 2.1, 3.999, 4.5], [10.2, -0.5, 7.7, 8.0]], "time": [0.25, 0.5]})
    assert open(os.path.join(str(tmp_path), "q.txt")).read() == "1\t2\t3\t4\n10\t0\t7\t8\n"
    assert open(os.path.join(str(tmp_path), "q_time.txt")).read() == "0.250000\n0.500000\n"


@pytest.mark.gpu
def test_batched_sequences_match_the_dropin_tracker(tmp_path):
    from oracle import vt_oracle as O
    from vittracker_b200 import get_tracker_class, load_cfg, parameters
    sd = O.make_state_dict(seed=31, stress=True, stable_size=True)
    rng = np.random.default_rng(5)
    seqs = []
    for i, (n, (H, W)) in enumerate(zip([4, 1, 6, 3, 5], [(360, 640), (240, 320), (360, 640), (300, 500), (240, 320)])):
        frames = O.synth_frames(n, H, W, seed=40 + i, smooth=True)
        box = [float(rng.uniform(40, W - 140)), float(rng.uniform(40, H - 120)), float(rng.uniform(30, 90)), float(rng.uniform(30, 70))]
        seqs.append(Sequence(f"seq{i}", list(frames), box))
    res = run_sequences(seqs, load_cfg(), sd, slots=3, results_dir=str(tmp_path))
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    for s in seqs:
        trk = get_tracker_class()(params, "synthetic")
        trk.initialize(s.frames[0], s.init_info())
        want = [list(s.init_bbox)] + [list(trk.track(f, {})["target_bbox"]) for f in s.frames[1:]]
        if len(s.frames) == 1:
            assert "target_bbox" not in res[s.name]
            continue
        got = res[s.name]["target_bbox"]
        assert len(got) == len(want)
        assert np.allclose(np.array(got), np.array(want, dtype=np.float64), rtol=1e-6, atol=1e-6), (s.name, got, want)
        assert os.path.isfile(os.path.join(str(tmp_path), s.name + ".txt"))
