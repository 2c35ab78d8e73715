"""Track records on the device (vt_tracks_export* / vt_tracks_import*): an imported track continues bit for bit as the exported one
would have - in other slots of the same handle, in another handle (through the host and a file), between handle kinds whose weights
fingerprints are equal, across GPUs, with the range fallback - and a record that fails a check writes nothing."""
import pickle

import numpy as np
import pytest
import torch

from oracle import vt_oracle as O
from test_generic_edges import CONFIGS, make_cfg
from test_gpu_track_slots import _flag_specs, _i32, _make, _np
from test_scale_invariance import IMPLS, _weights
from test_tracking_edges import MAPS, Tracks, _frames

pytestmark = pytest.mark.gpu
BAD_SLOT, BAD_RECORD = 4, 5
CHUNK = 5


@pytest.fixture(scope="module")
def table():
    return Tracks(_frames(), _flag_specs())


def _same(a, b, what):
    assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)), what


def _step(e, d, fr, slots=None, first=0, n=None):
    """One closed-loop step: (boxes, detail, maps) in item order."""
    if slots is None:
        o, det = e.tracks_step(d.buf, fr, d.hw, first=first, n=n, detail=True)
        k = int(fr.shape[0])
    else:
        o, det = e.tracks_step_slots(d.buf, fr, d.hw, _i32(slots, e.device), detail=True)
        k = len(slots)
    maps = e.tracks_last_maps(0, k) if slots is not None else e.tracks_last_maps(first, k)
    return _np(o), _np(det), {q: _np(v) for q, v in maps.items()}


def _compare(a, b, what):
    _same(a[0], b[0], (what, "boxes"))
    _same(a[1], b[1], (what, "detail"))
    for q in MAPS:
        _same(a[2][q], b[2][q], (what, q))


def _check_checksums(records):
    from vittracker_b200 import records as REC
    r = _np(records)
    for row in r:
        if int(row[:4].view("<u4")[0]) == REC.VT_TRACK_RECORD_MAGIC:
            assert REC.checksum(row[32:]) == int(row[24:32].view("<u8")[0])


@pytest.mark.parametrize("impl", list(IMPLS))
def test_same_handle_other_slots(table, golden_model, impl):
    n = table.n
    M = 2 * n + 3
    e = _make(impl, M, golden_model)
    dev = e.device
    d = table.device(dev)
    assert e.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0).shape == (n,)
    e.tracks_set_state(d.sbox, 0)
    _step(e, d, d.off[1], first=0, n=n)                             # the tracks have moved on from their templates
    rng = np.random.default_rng(5)
    src = rng.permutation(n)
    dst = n + 3 + rng.permutation(n)
    before = e.launch_count
    rec, st = e.tracks_export_slots(_i32(src, dev))
    assert e.launch_count - before == 2 and (_np(st) == 0).all()
    _check_checksums(rec)
    st = e.tracks_import_slots(rec, _i32(dst, dev))
    assert (_np(st) == 0).all()
    # the source tracks in item order src, the copies in the same order: first step by range for the source, then both by slot list
    order = torch.as_tensor(src, device=dev)
    for step in range(3):
        fr = d.off[2 if step % 2 == 0 else 1]
        frs = fr[order].contiguous()
        hws = d.hw[order].contiguous()
        if step == 0:
            o, det = e.tracks_step(d.buf, fr, d.hw, first=0, n=n, detail=True)
            maps = e.tracks_last_maps(0, n)
            a = (_np(o)[src], _np(det)[src], {q: _np(v)[src] for q, v in maps.items()})
        else:
            o, det = e.tracks_step_slots(d.buf, frs, hws, _i32(src, dev), detail=True)
            maps = e.tracks_last_maps(0, n)
            a = (_np(o), _np(det), {q: _np(v) for q, v in maps.items()})
        o, det = e.tracks_step_slots(d.buf, frs, hws, _i32(dst, dev), detail=True)
        maps = e.tracks_last_maps(0, n)
        _compare(a, (_np(o), _np(det), {q: _np(v) for q, v in maps.items()}), (impl, step))
        state = _np(e.tracks_get_state(0, M))
        _same(state[dst], state[src], (impl, step, "state"))
    a, _ = e.tracks_export_slots(_i32(src, dev))
    b, _ = e.tracks_export_slots(_i32(dst, dev))
    _same(_np(a), _np(b), (impl, "records after the steps"))


@pytest.mark.parametrize("impl", ["tcgen05", "small"])
def test_other_handle_through_a_file_import_only(table, golden_model, impl, tmp_path):
    from vittracker_b200.records import TrackRecords
    n = table.n
    src = _make(impl, n + 2, golden_model)
    dev = src.device
    d = table.device(dev)
    src.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)
    src.tracks_set_state(d.sbox, 0)
    _step(src, d, d.off[1], first=0, n=n)
    recs = TrackRecords(src.tracks_export(0, n), d.hw.clone())
    recs.cpu().save(tmp_path / "tracks.rec")
    back = TrackRecords.load(tmp_path / "tracks.rec", device=dev)
    _same(_np(back.records), _np(recs.records), "file round trip")
    # a handle with another capacity and chunk whose only tracks come from imports, stepped by slot list
    blocks, gen = IMPLS[impl]
    from vittracker_b200.engine import Engine
    from vittracker_b200 import load_cfg
    if gen is None:
        dst = Engine(load_cfg(), max_tracks=3 * n, blocks_impl=blocks, chunk_tracks=3)
    else:
        C, heads, depth, hc, _ = CONFIGS[gen]
        dst = Engine(make_cfg(C, heads, hc), max_tracks=3 * n, blocks_impl=blocks, depth=depth, chunk_tracks=3)
    dst.load_state_dict(_weights(gen, golden_model))
    slots = list(np.random.default_rng(6).permutation(3 * n)[:n])
    assert (_np(dst.tracks_import_slots(back.records, _i32(slots, dev))) == 0).all()
    for step in range(3):
        fr = d.off[2 - step % 2]
        a = _step(src, d, fr, first=0, n=n)
        b = _step(dst, d, fr, slots=slots)
        _compare(a, b, (impl, step))
    _same(_np(dst.tracks_get_state(0, 3 * n))[slots], _np(src.tracks_get_state(0, n)), "state")


def _kind_engine(cfg_name, impl, max_tracks, sd=None, golden_model=None):
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    if cfg_name is None:
        cfg, depth = load_cfg(), 3
        sd = sd if sd is not None else _weights(None, golden_model)
    else:
        C, heads, depth, hc, _ = CONFIGS[cfg_name]
        cfg = make_cfg(C, heads, hc)
        sd = sd if sd is not None else _weights(cfg_name, golden_model)
    e = Engine(cfg, max_tracks=max_tracks, blocks_impl=impl, depth=depth, chunk_tracks=CHUNK)
    e.load_state_dict(sd)
    return e, cfg, sd, depth


@pytest.mark.parametrize("cfg_name", [None, "small", "img"])
def test_fingerprint_contract_between_handle_kinds(table, golden_model, cfg_name):
    from vittracker_b200 import records as REC
    n = table.n
    kinds = {}
    for impl in ("simt", "tcgen05", "tcgen05_3term"):
        e, cfg, sd, depth = _kind_engine(cfg_name, impl, 2 * n, golden_model=golden_model)
        assert e.weights_fingerprint == REC.weights_fingerprint(cfg, sd, depth, impl), impl
        kinds[impl] = e
    dev = kinds["simt"].device
    d = table.device(dev)
    exported = {}
    for impl, e in kinds.items():
        e.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)
        exported[impl] = e.tracks_export(0, n)
        _check_checksums(exported[impl])
    if cfg_name is None:
        assert len({e.weights_fingerprint for e in kinds.values()}) == 1             # one template route on vit_48_h32
    else:
        assert kinds["simt"].weights_fingerprint != kinds["tcgen05"].weights_fingerprint == kinds["tcgen05_3term"].weights_fingerprint
    for x, ex in kinds.items():
        for y, ey in kinds.items():
            equal = ex.weights_fingerprint == ey.weights_fingerprint
            if equal:                                                # the same template tokens: the payloads are the same bytes
                _same(_np(exported[x]), _np(exported[y]), (x, y, "records"))
            st = _np(ey.tracks_import(exported[x], first=n))
            assert (st == (0 if equal else BAD_RECORD)).all(), (x, y, st)
            if not equal:
                continue
            for step in range(2):
                fr = d.off[1 + step]
                a = _step(ey, d, fr, first=0, n=n)
                b = _step(ey, d, fr, first=n, n=n)
                _compare(a, b, (cfg_name, x, y, step))
            ey.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)     # back to the template state for the next pair


def _flip(rec, off):
    r = rec.clone()
    r[:, off] ^= 0x20
    return r


def test_rejected_records_write_nothing(table, golden_model):
    from vittracker_b200 import records as REC
    n = table.n
    e, cfg, sd, _ = _kind_engine(None, "tcgen05", n + 4, golden_model=golden_model)
    dev = e.device
    d = table.device(dev)
    e.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)
    good = e.tracks_export(1, 1)
    target = n + 1
    before = _np(e.tracks_export(target, 1))
    R = e.track_record_bytes
    # header fields (magic, version, fingerprint, C, rows, checksum), the box and a token
    cases = {off: _flip(good, off) for off in (0, 4, 8, 15, 16, 20, 24, 31, 40, 64 + 1001, R - 1)}
    nan_box = good.clone()
    nan_box[0, 32:40] = torch.tensor(np.array([np.nan], "<f8").view(np.uint8), device=dev)
    cs = REC.checksum(_np(nan_box)[0, 32:])                             # a valid checksum: only the finite-box check rejects it
    nan_box[0, 24:32] = torch.tensor(np.array([cs], "<u8").view(np.uint8), device=dev)
    cases["nan box"] = nan_box
    # weights one ulp away in one tensor
    sd2 = dict(sd)
    t = sd2["blocks.2.attn.proj.weight"].clone()
    t.view(-1)[7] = torch.nextafter(t.view(-1)[7], torch.tensor(np.inf))
    sd2["blocks.2.attn.proj.weight"] = t
    e2, *_ = _kind_engine(None, "tcgen05", n, sd=sd2)
    assert e2.weights_fingerprint != e.weights_fingerprint
    e2.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)
    cases["1 ulp"] = e2.tracks_export(1, 1)
    # another embed dim: a C = 96 record cut to this handle's width
    e3, *_ = _kind_engine("small", "tcgen05", n, golden_model=golden_model)
    e3.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)
    cases["C 96"] = e3.tracks_export(1, 1)[:, :R].contiguous()
    for what, rec in cases.items():
        st = _np(e.tracks_import(rec, first=target))
        assert st.tolist() == [BAD_RECORD], what
        assert REC.describe_rejection(_np(rec)[0], e.weights_fingerprint, 48) is not None, what
        _same(_np(e.tracks_export(target, 1)), before, what)
        st = _np(e.tracks_import_slots(rec, _i32([target], dev)))
        assert st.tolist() == [BAD_RECORD], what
        _same(_np(e.tracks_export(target, 1)), before, what)
    assert _np(e.tracks_import(good, first=target)).tolist() == [0]
    _same(_np(e.tracks_export(target, 1)), _np(good), "accepted")
    # bad slots: negative, >= max_tracks, repeated (the first wins); BAD_SLOT before BAD_RECORD
    M = e.max_tracks
    recs, st = e.tracks_export_slots(_i32([2, -1, M, 3, 2], dev))
    assert _np(st).tolist() == [0, BAD_SLOT, BAD_SLOT, 0, BAD_SLOT]
    r = _np(recs)
    assert (r[[1, 2, 4]] == 0).all() and (r[[0, 3], :4].view("<u4") == REC.VT_TRACK_RECORD_MAGIC).all()
    imp = torch.stack([good[0], recs[3], recs[1], recs[0], _flip(good, 0)[0]]).contiguous()
    st = _np(e.tracks_import_slots(imp, _i32([target, target, -1, M, n + 2], dev)))
    assert st.tolist() == [0, BAD_SLOT, BAD_SLOT, BAD_SLOT, BAD_RECORD]
    _same(_np(e.tracks_export(target, 1)), _np(good), "first occurrence wins")


def test_graph_capture_and_launch_counts(table, golden_model):
    n = table.n
    M = 2 * n
    G, *_ = _kind_engine(None, "tcgen05", M, golden_model=golden_model)
    E, *_ = _kind_engine(None, "tcgen05", M, golden_model=golden_model)
    dev = G.device
    d = table.device(dev)
    for e in (G, E):
        e.tracks_init(d.buf, d.off[0], d.hw, d.tbox, first=0)
        e.tracks_set_state(d.sbox, 0)
    c = G.launch_count
    G.tracks_import(G.tracks_export(0, 2), first=n)
    assert G.launch_count - c == 2                                      # one kernel per range call
    E.tracks_import(E.tracks_export(0, 2), first=n)
    k = 6
    s_exp, s_imp = _i32(np.arange(k), dev), _i32(n + np.arange(k), dev)
    rec = torch.empty((k, G.track_record_bytes), dtype=torch.uint8, device=dev)
    c = G.launch_count
    _, st = G.tracks_export_slots(s_exp, out=rec)
    st2 = G.tracks_import_slots(rec, s_imp)
    assert G.launch_count - c == 4                                      # two kernels per slot-list call
    E.tracks_import_slots(E.tracks_export_slots(s_exp)[0], s_imp)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, st = G.tracks_export_slots(s_exp, out=rec)
        st2 = G.tracks_import_slots(rec, s_imp)
    rng = np.random.default_rng(8)
    for rep in range(3):
        a = rng.permutation(n)[:k]
        b = n + rng.permutation(n)[:k]
        if rep == 2:
            a[1], b[3] = -1, b[0]                                        # a bad export entry and a repeated import slot
        s_exp.copy_(_i32(a, dev))
        s_imp.copy_(_i32(b, dev))
        g.replay()
        er, est = E.tracks_export_slots(_i32(a, dev))
        ist = E.tracks_import_slots(er, _i32(b, dev))
        torch.cuda.synchronize()
        _same(_np(rec), _np(er), (rep, "records"))
        _same(_np(st), _np(est), (rep, "export status"))
        _same(_np(st2), _np(ist), (rep, "import status"))
        _same(_np(G.tracks_export(0, M)), _np(E.tracks_export(0, M)), (rep, "all tracks"))


def test_range_fallback_tracks_move_with_their_flags():
    import test_gpu_range_fallback as RF
    from test_gpu_range_fallback import CHUNK as FCHUNK, N, Run, _engine, _frame_idx
    cfg, sd, frames, boxes = _fallback_setup()
    for impl in RF.TC_IMPLS:
        ca = torch.zeros(1, dtype=torch.int64, device="cuda")
        cb = torch.zeros(1, dtype=torch.int64, device="cuda")
        a = Run(_engine(cfg, sd, impl, True, ca), frames, boxes)
        eb = _engine(cfg, sd, impl, True, cb, max_tracks=N + 9, chunk=FCHUNK + 3)
        assert (_np(eb.tracks_import(a.e.tracks_export(0, N), first=0)) == 0).all()
        b = Run.__new__(Run)
        b.e, b.frames, b.n, b.hw = eb, a.frames, N, a.hw
        for step in range(2):
            idx = _frame_idx() if step == 0 else 1 - _frame_idx()
            x, y = a.step(idx), b.step(idx)
            for k in ("boxes", "detail", "score_map", "size_map", "offset_map", "state"):
                _same(x[k], y[k], (impl, step, k))
        assert int(ca.item()) == int(cb.item()) > 0


def _fallback_setup():
    """The setup of test_gpu_range_fallback: tracks on its noise frame are flagged, tracks on its flat frame are not."""
    import test_gpu_range_fallback as RF
    from vittracker_b200 import load_cfg
    sd = O.make_state_dict(seed=5, stress=True)
    sd[RF.KEY] = sd[RF.KEY] * RF.FACTOR
    flat = np.empty((RF.H, RF.W, 3), np.uint8)
    flat[...] = (124, 116, 104)
    noise = np.random.default_rng(7).integers(0, 256, (RF.H, RF.W, 3), dtype=np.uint8)
    rng = np.random.default_rng(11)
    N = RF.N
    boxes = np.stack([rng.uniform(230, 380, N), rng.uniform(150, 260, N), rng.uniform(30, 50, N), rng.uniform(30, 50, N)], 1)
    return load_cfg(), sd, np.stack([flat, noise]), boxes


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus(table, golden_model):
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    from vittracker_b200.records import TrackRecords
    n = table.n
    sd = _weights(None, golden_model)
    e0 = Engine(load_cfg(), max_tracks=n, device=0)
    e1 = Engine(load_cfg(), max_tracks=n + 5, device=1, chunk_tracks=4)
    e0.load_state_dict(sd)
    e1.load_state_dict(sd)
    d0, d1 = table.device(e0.device), table.device(e1.device)
    e0.tracks_init(d0.buf, d0.off[0], d0.hw, d0.tbox, first=0)
    recs = TrackRecords(e0.tracks_export(0, n), d0.hw.clone()).to("cuda:1")
    assert (_np(e1.tracks_import(recs.records, first=0)) == 0).all()
    for step in range(2):
        a = _step(e0, d0, d0.off[1 + step], first=0, n=n)
        b = _step(e1, d1, d1.off[1 + step], first=0, n=n)
        _compare(a, b, step)


def test_vit_dist_snapshot_restore(golden_track, golden_model):
    from conftest import state_dict_from_npz
    from vittracker_b200 import get_tracker_class, parameters
    sd = state_dict_from_npz(golden_model)

    def tracker(weights):
        p = parameters("vit_48_h32_noKD")
        p.state_dict = weights
        return get_tracker_class()(p, "synthetic")

    frames = golden_track["frames"]
    init = [float(v) for v in golden_track["stress_init"]]
    ref = tracker(sd)
    ref.initialize(frames[0], {"init_bbox": init})
    for t in range(1, 4):
        ref.track(frames[t % 4], {})
    snap = ref.snapshot()
    want = [ref.track(frames[t % 4], {}) for t in range(4, 8)]
    want = [(o["target_bbox"], float(o["confidence"])) for o in want]

    def run(trk):
        return [(o["target_bbox"], float(o["confidence"])) for o in (trk.track(frames[t % 4], {}) for t in range(4, 8))]

    ref.restore(snap)                                                   # rewind
    assert ref.frame_id == 3
    assert run(ref) == want
    fresh = tracker(sd)
    fresh.restore(snap)
    assert run(fresh) == want
    again = tracker(sd)
    again.restore(pickle.loads(pickle.dumps(snap)))
    assert run(again) == want and np.array_equal(again.z_patch_arr, ref.z_patch_arr)
    other = dict(sd)
    other["norm.bias"] = other["norm.bias"] + 1e-3
    with pytest.raises(ValueError, match="fingerprint"):
        tracker(other).restore(snap)


def test_batched_tracker_export_import_by_slot(golden_model):
    from conftest import state_dict_from_npz
    from vittracker_b200 import BatchedTracker, FramePool, load_cfg
    sd = state_dict_from_npz(golden_model)
    fa = O.synth_frames(2, 360, 640, seed=7, smooth=True)
    fb = O.synth_frames(2, 240, 320, seed=9, smooth=True)
    ba = O.synth_boxes(4, 360, 640, seed=8)
    bb = O.synth_boxes(3, 240, 320, seed=10)
    src = BatchedTracker(load_cfg(), sd, max_tracks=8, chunk_tracks=3)
    pa, pb = FramePool(fa, src.device), FramePool(fb, src.device)
    z = lambda k: torch.zeros(k, dtype=torch.int64)
    src.initialize(pa, z(4), ba, slots=[5, 0, 2, 7])
    src.initialize(pb, z(3), bb, slots=[1, 3, 6])
    recs = src.export_tracks(slots=[6, 2, 1])
    assert _np(recs.frame_hw).tolist() == [[240, 320], [360, 640], [240, 320]]
    dst = BatchedTracker(load_cfg(), sd, max_tracks=5, chunk_tracks=2)
    assert (_np(dst.import_tracks(recs, slots=[4, 0, 2])) == 0).all()
    for t in range(3):
        fr = torch.full((3,), (t + 1) % 2, dtype=torch.int64)
        # source slots 6 and 1 live on pool b, slot 2 on pool a: step each tracker per pool, the same items in the same order
        a1 = _np(src.track(pb, fr[:2], slots=[6, 1]))
        a2 = _np(src.track(pa, fr[:1], slots=[2]))
        b1 = _np(dst.track(pb, fr[:2], slots=[4, 2]))
        b2 = _np(dst.track(pa, fr[:1], slots=[0]))
        _same(a1, b1, t)
        _same(a2, b2, t)
    bad = dst.import_tracks(recs, slots=torch.tensor([1, 1, 9], dtype=torch.int32, device=dst.device))
    assert _np(bad).tolist() == [0, BAD_SLOT, BAD_SLOT]
    assert _np(dst._slot_hw[1]).tolist() == [240, 320]
