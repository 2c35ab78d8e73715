"""Tracks initialised and stepped by slot list (vt_tracks_init_slots / vt_tracks_step_slots) against the range calls, bit for bit:
shuffled slots over several chunks and closed-loop steps, bad entries (out of range, repeated) next to valid ones, update_state=0,
never-initialised slots, CUDA-graph replay with new slot contents, YUV surfaces, and the sequence driver's step over running slots."""
import numpy as np
import pytest
import torch

from oracle import vt_oracle as O
from test_generic_edges import CONFIGS, make_cfg
from test_scale_invariance import IMPLS, _weights
from test_tracking_edges import MAPS, Tracks, _frames, _table_specs

pytestmark = pytest.mark.gpu
BAD = 4                     # VT_TRACK_BAD_SLOT
SPARE = 7                   # slots beyond the tracks of the table
CHUNK = 5                   # tracks per internal pass: every call spans several chunks


def _flag_specs():
    """The crop-edge table plus rows the crop flags: a zero box (too small) and a box off the frame (out of domain)."""
    hd = "hd"
    return _table_specs() + [("too_small", hd, 1, (600.0, 300.0, 40.0, 40.0), (600.0, 300.0, 0.0, 0.0)),
                             ("off_frame", hd, 2, (600.0, 300.0, 40.0, 40.0), (5000.0, 4000.0, 30.0, 30.0))]


@pytest.fixture(scope="module")
def table():
    return Tracks(_frames(), _flag_specs())


def _make(impl, n, golden_model):
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    blocks, gen = IMPLS[impl]
    if gen is None:
        e = Engine(load_cfg(), max_tracks=n, blocks_impl=blocks, chunk_tracks=CHUNK)
    else:
        C, heads, depth, hc, _ = CONFIGS[gen]
        e = Engine(make_cfg(C, heads, hc), max_tracks=n, blocks_impl=blocks, depth=depth, chunk_tracks=CHUNK)
    e.load_state_dict(_weights(gen, golden_model))
    return e


def _np(t):
    return t.cpu().numpy()


def _i32(a, dev):
    return torch.tensor(np.asarray(a), dtype=torch.int32, device=dev)


def _runs(ids):
    """Maximal runs of consecutive ids (sorted): [(first, n), ...]."""
    ids = sorted(ids)
    out, s = [], 0
    for k in range(1, len(ids) + 1):
        if k == len(ids) or ids[k] != ids[k - 1] + 1:
            out.append((ids[s], k - s))
            s = k
    return out


def _same(a, b, what):
    assert np.array_equal(a, b, equal_nan=True), what


def _set_slots(e, slots, boxes):
    state = e.tracks_get_state(0, e.max_tracks)
    state[torch.as_tensor(slots, dtype=torch.int64, device=e.device)] = boxes
    e.tracks_set_state(state.contiguous(), 0)


@pytest.mark.parametrize("impl", list(IMPLS))
def test_slot_steps_equal_range_steps_bit_for_bit(table, golden_model, impl):
    n = table.n
    A, B = _make(impl, n, golden_model), _make(impl, n + SPARE, golden_model)
    dev = A.device
    d = table.device(dev)
    rng = np.random.default_rng(11)
    perm = rng.permutation(n + SPARE)[:n]                         # track k lives in B's slot perm[k]
    order = rng.permutation(n)                                     # B initialises its tracks in this order
    st_a = _np(A.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0))
    sel = torch.as_tensor(order, device=dev)
    st_b = _np(B.tracks_init_slots(d.buf, d.off[0][sel].contiguous(), d.hw[sel].contiguous(), d.tbox[sel].contiguous(),
                                   _i32(perm[order], dev)))
    _same(st_b, st_a[order], "init status")
    A.tracks_set_state(d.sbox, 0)
    _set_slots(B, perm, d.sbox)
    flagged = set()
    for step in range(4):
        k = int(rng.integers(n // 2, n + 1))
        sub = rng.permutation(n)[:k]                              # a random subset in random order
        fr = d.off[1 + step % 2]
        ia = {}
        for first, m in _runs(sub):
            o, det = A.tracks_step(d.buf, fr[first:first + m].contiguous(), d.hw[first:first + m].contiguous(), first=first, n=m,
                                   detail=True)
            maps = A.tracks_last_maps(first, m)
            for j in range(m):
                ia[first + j] = (_np(o[j]), _np(det[j]), {q: _np(maps[q][j]) for q in MAPS})
        s = torch.as_tensor(sub, device=dev)
        o, det = B.tracks_step_slots(d.buf, fr[s].contiguous(), d.hw[s].contiguous(), _i32(perm[sub], dev), detail=True)
        maps = B.tracks_last_maps(0, k)
        o, det, maps = _np(o), _np(det), {q: _np(v) for q, v in maps.items()}
        for j, t in enumerate(sub):
            _same(o[j], ia[t][0], (step, t, "boxes"))
            _same(det[j], ia[t][1], (step, t, "detail"))
            for q in MAPS:
                _same(maps[q][j], ia[t][2][q], (step, t, q))
            if det[j][6] != 0:
                flagged.add(int(det[j][6]))
        _same(_np(B.tracks_get_state(0, n + SPARE))[perm], _np(A.tracks_get_state(0, n)), (step, "state"))
    assert {1, 2} <= flagged                                       # too small and out of domain landed on their items


def _bad_list(perm, M, rng):
    """The valid list with -1, M and a repeat of an earlier slot mixed in; returns (list, item -> valid index or -1)."""
    items = [(int(s), k) for k, s in enumerate(perm)]
    for bad in (-1, M, int(perm[2])):
        pos = int(rng.integers(3, len(items) + 1))
        items.insert(pos, (bad, -1))
    return [s for s, _ in items], [k for _, k in items]


@pytest.mark.parametrize("impl", list(IMPLS))
def test_bad_entries_are_flagged_and_touch_nothing(table, golden_model, impl):
    n = table.n
    M = n + SPARE
    R, X = _make(impl, M, golden_model), _make(impl, M, golden_model)
    dev = R.device
    d = table.device(dev)
    rng = np.random.default_rng(12)
    perm = rng.permutation(M)[:n]
    slots, src = _bad_list(perm, M, rng)
    # a bad item takes the frame and boxes of the last track, so that processing it would change what it touched
    take = torch.as_tensor([k if k >= 0 else n - 1 for k in src], device=dev)
    valid = np.array(src) >= 0
    vk = np.array([k for k in src if k >= 0])
    st_r = _np(R.tracks_init_slots(d.buf, d.off[0], d.hw, d.tbox, _i32(perm, dev)))
    st_x = _np(X.tracks_init_slots(d.buf, d.off[0][take].contiguous(), d.hw[take].contiguous(), d.tbox[take].contiguous(),
                                   _i32(slots, dev)))
    _same(st_x[valid], st_r[vk], "init status")
    assert (st_x[~valid] == BAD).all()
    _same(_np(X.tracks_get_state(0, M)), _np(R.tracks_get_state(0, M)), "state after init")
    for e in (R, X):
        _set_slots(e, perm, d.sbox)
    for step in range(2):                                          # the same list again: the claims were released
        fr = d.off[1 + step]
        o_r, d_r = R.tracks_step_slots(d.buf, fr, d.hw, _i32(perm, dev), detail=True)
        m_r = {q: _np(v) for q, v in R.tracks_last_maps(0, n).items()}
        o_x, d_x = X.tracks_step_slots(d.buf, fr[take].contiguous(), d.hw[take].contiguous(), _i32(slots, dev), detail=True)
        m_x = {q: _np(v) for q, v in X.tracks_last_maps(0, len(slots)).items()}
        o_r, d_r, o_x, d_x = _np(o_r), _np(d_r), _np(o_x), _np(d_x)
        _same(o_x[valid], o_r[vk], (step, "boxes"))
        _same(d_x[valid], d_r[vk], (step, "detail"))
        for q in MAPS:
            _same(m_x[q][valid], m_r[q][vk], (step, q))
            assert np.isnan(m_x[q][~valid]).all(), (step, q)
        _same(o_x[~valid], np.tile([0.0, 0.0, 0.0, 0.0, -1.0], (int((~valid).sum()), 1)), (step, "bad boxes"))
        assert (d_x[~valid][:, 6] == BAD).all() and (d_x[~valid][:, 5] == -1).all()
        _same(_np(X.tracks_get_state(0, M)), _np(R.tracks_get_state(0, M)), (step, "state"))


@pytest.mark.parametrize("impl", list(IMPLS))
def test_update_state_zero_and_never_initialised_slots(table, golden_model, impl):
    n = table.n
    M = n + SPARE
    e = _make(impl, M, golden_model)
    dev = e.device
    d = table.device(dev)
    slots = np.arange(SPARE, M)[::-1].copy()
    e.tracks_init_slots(d.buf, d.off[0], d.hw, d.tbox, _i32(slots, dev))
    before = _np(e.tracks_get_state(0, M))
    e.tracks_step_slots(d.buf, d.off[1], d.hw, _i32(slots, dev), update_state=False)
    _same(_np(e.tracks_get_state(0, M)), before, "update_state=0")
    o, det = e.tracks_step_slots(d.buf, d.off[1][:3].contiguous(), d.hw[:3].contiguous(), _i32([0, SPARE - 1, SPARE], dev),
                                 detail=True, update_state=True)
    o, det = _np(o), _np(det)
    assert det[0][6] == 1 and det[1][6] == 1 and o[0][4] == -1 and o[1][4] == -1       # VT_TRACK_TOO_SMALL, no fault
    _same(_np(e.tracks_get_state(0, SPARE)), np.zeros((SPARE, 4)), "zero state kept")


def _bt_setup(blocks, n=12):
    from vittracker_b200 import BatchedTracker, FramePool, load_cfg
    sd = O.make_state_dict(seed=5, stress=True)
    bt = BatchedTracker(load_cfg(), sd, max_tracks=n, blocks_impl=blocks)
    frames = O.synth_frames(3, 360, 640, seed=9, smooth=True)
    pool = FramePool(frames, bt.device)
    boxes = O.synth_boxes(n, 360, 640, seed=4)
    return bt, pool, boxes, frames


@pytest.mark.parametrize("blocks", ["tcgen05", "simt"])
def test_cuda_graph_replays_with_new_slot_contents(blocks):
    bt, pool, boxes, _ = _bt_setup(blocks)
    dev = bt.device
    assert int(bt.initialize(pool, torch.zeros(12, dtype=torch.int64), boxes).abs().sum()) == 0
    k = 5
    t = torch.zeros(k, dtype=torch.int32, device=dev)
    fi = torch.ones(k, dtype=torch.int64, device=dev)
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        t.copy_(torch.arange(k, dtype=torch.int32))
        bt.track(pool, fi, update_state=False, slots=t)
    torch.cuda.current_stream(dev).wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = bt.track(pool, fi, update_state=False, slots=t)
    rng = np.random.default_rng(3)
    for _ in range(4):
        lst = rng.permutation(12)[:k]
        t.copy_(torch.as_tensor(lst, dtype=torch.int32))
        g.replay()
        got = out.clone()
        want = bt.track(pool, fi, update_state=False, slots=torch.as_tensor(lst, dtype=torch.int32, device=dev)).clone()
        assert torch.equal(got, want)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_track_yuv_by_slot_equals_rgb_of_opencv(fmt):
    cv2 = pytest.importorskip("cv2")
    from oracle import yuv420 as Y
    from vittracker_b200 import BatchedTracker, FramePool, load_cfg
    from vittracker_b200.batched import YuvSurfaces
    CV = {"nv12": cv2.COLOR_YUV2RGB_NV12, "i420": cv2.COLOR_YUV2RGB_I420}
    n, M, H, W, F = 8, 13, 360, 640, 4
    sd = O.make_state_dict(seed=5, stress=True)
    bt_y, bt_r = BatchedTracker(load_cfg(), sd, max_tracks=M), BatchedTracker(load_cfg(), sd, max_tracks=M)
    dev = bt_y.device
    frames = Y.synth_yuv420(F, H, W, seed=21, format=fmt, smooth=True)
    pool = FramePool(np.stack([cv2.cvtColor(f, CV[fmt]) for f in frames]), dev)
    rng = np.random.default_rng(8)
    slots = rng.permutation(M)[:n]
    boxes = O.synth_boxes(n, H, W, seed=6)
    for t in range(4):
        idx = (np.arange(n) + t) % F
        surf = YuvSurfaces.from_frames(torch.from_numpy(frames[idx]).to(dev), fmt)
        if t == 0:
            a = bt_y.initialize_yuv(surf, boxes, slots=slots)
            b = bt_r.initialize(pool, torch.from_numpy(idx), boxes, slots=slots)
            assert torch.equal(a, b) and int(a.abs().sum()) == 0
            continue
        sub = rng.permutation(n)[: n - 2]                         # a subset of the tracks, each on its own surface
        surf = YuvSurfaces.from_frames(torch.from_numpy(frames[idx[sub]]).to(dev), fmt)
        oy, dy = bt_y.track_yuv(surf, detail=True, slots=slots[sub])
        oy, dy = oy.clone(), dy.clone()
        my = bt_y.engine.tracks_last_maps(0, len(sub))
        orr, dr = bt_r.track(pool, torch.from_numpy(idx[sub]), detail=True, slots=slots[sub])
        mr = bt_r.engine.tracks_last_maps(0, len(sub))
        assert torch.equal(oy, orr) and torch.equal(dy, dr), t
        for q in MAPS:
            assert torch.equal(torch.nan_to_num(my[q]), torch.nan_to_num(mr[q])), (t, q)
        assert torch.equal(bt_y.get_state(slots=slots), bt_r.get_state(slots=slots))


def test_sequence_driver_steps_only_running_sequences():
    from vittracker_b200 import load_cfg
    from vittracker_b200.sequences import BatchedBackend, MultiSequenceRunner, Sequence
    sd = O.make_state_dict(seed=31, stress=True, stable_size=True)
    rng = np.random.default_rng(5)
    lengths = [4, 1, 6, 3, 9, 2, 7]
    seqs = []
    for i, n in enumerate(lengths):
        H, W = (360, 640) if i % 2 else (240, 320)
        frames = O.synth_frames(n, H, W, seed=60 + i, smooth=True)
        box = [float(rng.uniform(40, W - 140)), float(rng.uniform(40, H - 120)), float(rng.uniform(30, 90)), float(rng.uniform(30, 70))]
        seqs.append(Sequence(f"seq{i}", list(frames), box))
    log = []

    class Profiled(BatchedBackend):
        def step_active(self, slots, images):
            self.bt.engine.profile_read()
            r = super().step_active(slots, images)
            log.append((list(slots), self.bt.engine.profile_read()))
            return r

    be = Profiled(load_cfg(), sd, 3)
    be.bt.engine.profile(True)
    runner = MultiSequenceRunner(be, 3, read_workers=0)
    res = runner.run(seqs)
    runner.close()
    be.close()
    assert sum(len(s) for s, _ in log) == sum(n - 1 for n in lengths)     # every tracked frame stepped once, nothing else
    for slots, prof in log:
        for stage in ("stem", "blocks", "head"):
            assert prof[stage]["items"] == len(slots), (slots, prof)
    assert any(len(s) < 3 for s, _ in log)                         # the run drains: the last steps cover fewer slots
    assert all(len(res[s.name].get("target_bbox", [None])) in (1, len(s.frames)) for s in seqs)
