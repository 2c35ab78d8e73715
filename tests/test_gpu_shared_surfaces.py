"""Several targets on one YUV surface: vt_yuv420_crops_to_surface_rgb converts the bounding rectangle of each surface's crops once,
into one RGB frame per surface.  The bytes against cv2.cvtColor with canary-checked bounds, the tracker on shared surfaces against the
per-track path fed each surface once per track (bit for bit, by range and by shuffled slot list), CUDA-graph capture, bad surface
entries, and the C ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")

from oracle import vt_oracle as O
from oracle import yuv420 as Y
from test_gpu_yuv_surfaces import CANARY, CV, FORMATS, _config, _init_boxes, edge_boxes, expected_rect, pack_surface

pytestmark = pytest.mark.gpu
BAD = 4                                                   # VT_TRACK_BAD_SLOT


@pytest.fixture(scope="module")
def engine():
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    return Engine(load_cfg(), max_tracks=64)


def surfaces_of(frames, fmt, dev, P, S, seed=0):
    """YuvSurfaces over one device tensor [m, S*3/2, P] of pitched, poisoned surfaces; returns (surfaces, buffer)."""
    from vittracker_b200.batched import YuvSurfaces
    rng = np.random.default_rng(seed)
    H, W = frames.shape[1] * 2 // 3, frames.shape[2]
    buf = torch.from_numpy(np.stack([pack_surface(f, fmt, P, S, rng) for f in frames])).to(dev)
    return YuvSurfaces.from_frames(buf[:, :, :W], fmt, height=H, surface_rows=S), buf


def repeated(buf, surface, fmt, H, S, W=1280):
    """The per-track path's input: surface[i]'s contents as item i's own surface (a copy, with the same pitch and padding)."""
    from vittracker_b200.batched import YuvSurfaces
    idx = torch.as_tensor(surface, device=buf.device).to(torch.int64).clamp(0, buf.shape[0] - 1)
    return YuvSurfaces.from_frames(buf[idx][:, :, :W], fmt, height=H, surface_rows=S)


def bounding(rects):
    rects = [r for r in rects if r is not None]
    if not rects:
        return None
    return (min(r[0] for r in rects), max(r[1] for r in rects), min(r[2] for r in rects), max(r[3] for r in rects))


def check_frames(got, want_rgb, rects, dst_off, H, W, tag):
    """Inside each surface's rectangle its frame equals cvtColor; every other byte (other surfaces' rows and columns, the gaps) is
    the canary."""
    written = np.zeros(got.size, bool)
    for s, (rect, o) in enumerate(zip(rects, dst_off)):
        if rect is None:
            continue
        ya, yb, xa, xb = rect
        img = got[o:o + H * W * 3].reshape(H, W, 3)
        assert np.array_equal(img[ya:yb, xa:xb], want_rgb[s][ya:yb, xa:xb]), (tag, s, rect)
        written[o:o + H * W * 3].reshape(H, W, 3)[ya:yb, xa:xb] = True
    assert (got[~written] == CANARY).all(), (tag, int((got[~written] != CANARY).sum()))


# ------------------------------------------------------------------------------------------------
# the bytes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(720, 1280), (6, 10)])
@pytest.mark.parametrize("fmt", FORMATS)
def test_each_surface_gets_the_bounding_rectangle_of_its_crops_and_nothing_else(engine, fmt, hw):
    H, W = hw
    dev, factor = engine.device, 4.0
    m = 4
    frames = Y.synth_yuv420(m, H, W, seed=H + 3, format=fmt)
    surf, _ = surfaces_of(frames, fmt, dev, P=W + 64 + 6, S=H + 10, seed=2)
    want = [cv2.cvtColor(f, CV[fmt]) for f in frames]
    many = edge_boxes(H, W)
    one = np.array([[W * 0.4, H * 0.4, W * 0.1 + 1, H * 0.1 + 1]])
    degenerate = np.array([[50.0, 50.0, 0.0, 20.0], [-500.0, 10.0, 30.0, 30.0], [W + 200.0, H + 200.0, 30.0, 30.0]])
    # surface 0: no item; 1: one; 2: many, at every edge, degenerate ones included; 3: only degenerate ones.  Items with surface -1
    # or m (a box covering everything) are skipped.
    boxes = np.concatenate([one, many, degenerate, [[0.0, 0.0, W, H]] * 2])
    surface = [1] + [2] * len(many) + [3] * len(degenerate) + [-1, m]
    n = len(surface)
    rng = np.random.default_rng(5)
    order = rng.permutation(n)                              # items of one surface interleave with the others'
    boxes, surface = boxes[order], [surface[k] for k in order]
    rects = [expected_rect(b, factor, H, W) if 0 <= s < m else None for b, s in zip(boxes, surface)]
    want_rect = [bounding([r for r, s in zip(rects, surface) if s == k]) for k in range(m)]
    assert want_rect[0] is None and want_rect[3] is None and want_rect[1] is not None
    if H > 6:
        assert want_rect[2] == (0, H, 0, W)                   # the edge boxes reach every border

    dst_off = [k * (H * W * 3 + 7) + 3 for k in range(m)]                  # every alignment mod 4, canary gaps between frames
    offs = torch.tensor(dst_off, dtype=torch.int64, device=dev)
    surf_t = torch.tensor(surface, dtype=torch.int32, device=dev)
    bx = torch.from_numpy(boxes).to(dev)

    def run(**kw):
        dst = torch.full((m * (H * W * 3 + 7) + 8,), CANARY, dtype=torch.uint8, device=dev)
        engine.yuv420_crops_to_surface_rgb(fmt, surf.planes, surf.pitches, surf.hw, dst, offs, surf_t, factor, **kw)
        return dst.cpu().numpy()

    launches = engine.launch_count
    got = run(boxes=bx)
    assert engine.launch_count == launches + 2
    check_frames(got, want, want_rect, dst_off, H, W, (fmt, hw, "boxes"))
    assert np.array_equal(run(boxes=bx), got)                # the scratch was left empty: a second call gives the same bytes

    # the state of tracks [first, first + n)
    first = 64 - n
    engine.tracks_set_state(bx, first=first)
    check_frames(run(boxes=None, first=first), want, want_rect, dst_off, H, W, (fmt, hw, "range"))

    # the state of tracks slots[i], shuffled; bad and repeated slots are skipped whatever their box
    slots = rng.permutation(64)[:n].astype(np.int32)
    state = np.zeros((64, 4))
    state[slots] = boxes
    big = [[0.0, 0.0, float(W), float(H)]]
    slots_x = np.concatenate([slots, [-1, 64, slots[0]]]).astype(np.int32)
    surface_x = surface + [1, 1, 1]
    engine.tracks_set_state(torch.from_numpy(state).to(dev), first=0)
    launches = engine.launch_count
    dst = torch.full((m * (H * W * 3 + 7) + 8,), CANARY, dtype=torch.uint8, device=dev)
    engine.yuv420_crops_to_surface_rgb(fmt, surf.planes, surf.pitches, surf.hw, dst, offs,
                                       torch.tensor(surface_x, dtype=torch.int32, device=dev), factor, boxes=None,
                                       slots=torch.from_numpy(slots_x).to(dev))
    assert engine.launch_count == launches + 3
    check_frames(dst.cpu().numpy(), want, want_rect, dst_off, H, W, (fmt, hw, "slots"))
    # explicit boxes with a slot list: the slots only decide which items are skipped
    bx_x = torch.from_numpy(np.concatenate([boxes, big * 3])).to(dev)
    dst.fill_(CANARY)
    engine.yuv420_crops_to_surface_rgb(fmt, surf.planes, surf.pitches, surf.hw, dst, offs,
                                       torch.tensor(surface_x, dtype=torch.int32, device=dev), factor, boxes=bx_x,
                                       slots=torch.from_numpy(slots_x).to(dev))
    check_frames(dst.cpu().numpy(), want, want_rect, dst_off, H, W, (fmt, hw, "boxes + slots"))


# ------------------------------------------------------------------------------------------------
# the tracker: bit for bit the per-track path
# ------------------------------------------------------------------------------------------------
NB, M, HB, WB, PB, SB, STEPS = 32, 4, 720, 1280, 1280 + 256, 736, 8


def _outputs(bt, o, d, n, slots=None):
    maps = {k: v.cpu().numpy() for k, v in bt.engine.tracks_last_maps(0, n).items()}
    return o.cpu().numpy().copy(), d.cpu().numpy().copy(), maps, bt.get_state(slots).cpu().numpy()


def _same(a, b, tag):
    (oa, da, ma, sa), (ob, db, mb, sb) = a, b
    assert np.array_equal(oa, ob), tag
    assert np.array_equal(da, db), tag
    for k in ma:
        assert np.array_equal(ma[k], mb[k], equal_nan=True), (tag, k)
    assert np.array_equal(sa, sb, equal_nan=True), tag


@pytest.mark.parametrize("kind", ["tcgen05", "simt", "generic"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_shared_surfaces_track_bit_for_bit_like_one_surface_per_track(fmt, kind):
    from vittracker_b200 import BatchedTracker
    cfg, sd, kw = _config(kind)
    bt_s = BatchedTracker(cfg, sd, max_tracks=NB, **kw)
    bt_p = BatchedTracker(cfg, sd, max_tracks=NB, **kw)
    dev = bt_s.device
    pics = Y.synth_yuv420(2 * M, HB, WB, seed=41, format=fmt, smooth=True)
    rng = np.random.default_rng(7)
    boxes = _init_boxes()

    def frame_set(t):
        return surfaces_of(pics[(np.arange(M) + t) % (2 * M)], fmt, dev, P=PB, S=SB, seed=t)

    # range: init, then closed-loop steps; surface given as a host list
    surface = rng.integers(0, M, NB).tolist()
    surf, buf = frame_set(0)
    st_s = bt_s.initialize_yuv(surf, boxes, surface=surface)
    st_p = bt_p.initialize_yuv(repeated(buf, surface, fmt, HB, SB), boxes)
    assert torch.equal(st_s, st_p) and int(st_s.abs().sum()) == 0
    assert bt_s._surf_rgb.shape[0] == M + 1
    assert torch.equal(bt_s.export_tracks().records, bt_p.export_tracks().records)
    for t in range(1, STEPS + 1):
        surf, buf = frame_set(t)
        surface = rng.integers(0, M, NB).tolist()
        upd = t % 3 != 2
        o, d = bt_s.track_yuv(surf, update_state=upd, detail=True, surface=surface)
        a = _outputs(bt_s, o, d, NB)
        o, d = bt_p.track_yuv(repeated(buf, surface, fmt, HB, SB), update_state=upd, detail=True)
        _same(a, _outputs(bt_p, o, d, NB), ("range", t))

    # shuffled slot lists: init a subset, then step other shuffled subsets; surface as a CUDA tensor on odd steps
    n = NB - 8
    slots = rng.permutation(NB)[:n].tolist()
    surface = rng.integers(0, M, n)
    surf, buf = frame_set(STEPS + 1)
    st_s = bt_s.initialize_yuv(surf, boxes[:n], slots=slots, surface=torch.from_numpy(surface).to(dev))
    st_p = bt_p.initialize_yuv(repeated(buf, surface, fmt, HB, SB), boxes[:n], slots=slots)
    assert torch.equal(st_s, st_p) and int(st_s.abs().sum()) == 0
    assert torch.equal(bt_s.export_tracks(slots=slots).records, bt_p.export_tracks(slots=slots).records)
    for t in range(STEPS + 2, 2 * STEPS + 2):
        k = int(rng.integers(n - 6, n + 1))
        step_slots = rng.permutation(slots)[:k].tolist()
        surface = rng.integers(0, M, k)
        surf, buf = frame_set(t)
        upd = t % 3 != 1
        sv = torch.from_numpy(surface).to(dev) if t % 2 else surface.tolist()
        o, d = bt_s.track_yuv(surf, update_state=upd, detail=True, slots=step_slots, surface=sv)
        a = _outputs(bt_s, o, d, k, step_slots)
        o, d = bt_p.track_yuv(repeated(buf, surface, fmt, HB, SB), update_state=upd, detail=True, slots=step_slots)
        _same(a, _outputs(bt_p, o, d, k, step_slots), ("slots", t))
    assert torch.equal(bt_s.engine.tracks_get_state(), bt_p.engine.tracks_get_state())


# ------------------------------------------------------------------------------------------------
# CUDA graph
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", FORMATS)
def test_track_yuv_on_shared_surfaces_in_a_cuda_graph_equals_plain_launches(fmt):
    from vittracker_b200 import BatchedTracker
    cfg, sd, kw = _config("tcgen05")
    n, steps = 16, 6
    pics = Y.synth_yuv420(steps + M, HB, WB, seed=29, format=fmt, smooth=True)
    plain, graphed = BatchedTracker(cfg, sd, max_tracks=n, **kw), BatchedTracker(cfg, sd, max_tracks=n, **kw)
    dev = plain.device
    data = [surfaces_of(pics[t:t + M], fmt, dev, P=PB, S=SB, seed=t)[1] for t in range(steps)]
    surf, buf = surfaces_of(pics[:M], fmt, dev, P=PB, S=SB)                   # fixed surfaces, refilled per step
    rng = np.random.default_rng(3)
    assign = [torch.from_numpy(rng.integers(0, M, n).astype(np.int32)).to(dev) for _ in range(steps)]
    surface = assign[0].clone()                                               # fixed surface tensor, refilled per step
    boxes = _init_boxes()[:n]
    out = {"plain": [], "graph": []}
    for key, bt in (("plain", plain), ("graph", graphed)):
        buf.copy_(data[0])
        surface.copy_(assign[0])
        assert int(bt.initialize_yuv(surf, boxes, surface=surface).abs().sum()) == 0
        buf.copy_(data[1])
        surface.copy_(assign[1])
        out[key].append(bt.track_yuv(surf, surface=surface).cpu().numpy())
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize(dev)
    with torch.cuda.graph(g):
        graphed.track_yuv(surf, surface=surface)
    moved = torch.from_numpy(O.synth_boxes(n, HB, WB, seed=61)).to(dev)
    for t in range(2, steps):
        if t == 4:                                                            # new states as well as new surface contents
            plain.set_state(moved)
            graphed.set_state(moved)
        buf.copy_(data[t])
        surface.copy_(assign[t])
        out["plain"].append(plain.track_yuv(surf, surface=surface).cpu().numpy())
        buf.copy_(data[t])
        surface.copy_(assign[t])
        g.replay()
        out["graph"].append(graphed.out_boxes[:n].cpu().numpy())
        mp, mg = plain.engine.tracks_last_maps(0, n), graphed.engine.tracks_last_maps(0, n)
        for k in mp:
            assert torch.equal(torch.nan_to_num(mp[k]), torch.nan_to_num(mg[k])), (t, k)
    for t, (a, b) in enumerate(zip(out["plain"], out["graph"])):
        assert np.array_equal(a, b), t
    assert torch.equal(plain.get_state(), graphed.get_state())


# ------------------------------------------------------------------------------------------------
# bad entries
# ------------------------------------------------------------------------------------------------
def test_bad_surface_entries_are_bad_slots_on_the_device_and_refused_on_the_host():
    from vittracker_b200 import BatchedTracker
    cfg, sd, kw = _config("tcgen05")
    n, fmt = 16, "nv12"
    bt_s, bt_p = BatchedTracker(cfg, sd, max_tracks=n, **kw), BatchedTracker(cfg, sd, max_tracks=n, **kw)
    dev = bt_s.device
    pics = Y.synth_yuv420(2 * M, HB, WB, seed=53, format=fmt, smooth=True)
    surf, buf = surfaces_of(pics[:M], fmt, dev, P=PB, S=SB)
    rng = np.random.default_rng(11)
    surface = rng.integers(0, M, n)
    boxes = _init_boxes()[:n]
    assert int(bt_s.initialize_yuv(surf, boxes, surface=surface.tolist()).abs().sum()) == 0
    assert int(bt_p.initialize_yuv(repeated(buf, surface, fmt, HB, SB), boxes).abs().sum()) == 0
    bad = np.zeros(n, bool)
    bad[[2, 9]] = True
    surface_x = surface.copy()
    surface_x[2], surface_x[9] = -1, M
    surf, buf = surfaces_of(pics[M:], fmt, dev, P=PB, S=SB, seed=1)
    before = bt_s.get_state().cpu().numpy()
    o, d = bt_s.track_yuv(surf, detail=True, surface=torch.from_numpy(surface_x).to(dev))
    o, d = o.cpu().numpy(), d.cpu().numpy()
    assert (d[bad, 6] == BAD).all() and (d[bad, 5] == -1).all() and (o[bad, 4] == -1).all()
    after = bt_s.get_state().cpu().numpy()
    assert np.array_equal(after[bad], before[bad])
    # the other items: bit for bit the per-track path stepping them alone
    good = [int(i) for i in np.flatnonzero(~bad)]
    op, dp = bt_p.track_yuv(repeated(buf, surface[good], fmt, HB, SB), detail=True, slots=good)
    assert np.array_equal(o[~bad], op.cpu().numpy()) and np.array_equal(d[~bad], dp.cpu().numpy())
    assert np.array_equal(after[~bad], bt_p.get_state().cpu().numpy()[~bad])
    # with a slot list too
    slots = rng.permutation(n).tolist()
    o, d = bt_s.track_yuv(surf, detail=True, slots=slots, surface=torch.from_numpy(surface_x).to(dev))
    assert (d.cpu().numpy()[bad, 6] == BAD).all()
    # host sequences are checked here
    launches = bt_s.engine.launch_count
    for sv in (surface_x.tolist(), list(surface) + [0], list(surface)[:-1]):
        with pytest.raises(ValueError):
            bt_s.track_yuv(surf, surface=sv)
        with pytest.raises(ValueError):
            bt_s.initialize_yuv(surf, boxes, surface=sv)
    with pytest.raises(ValueError):
        bt_s.track_yuv(surf, surface=torch.zeros((n, 1), dtype=torch.int32, device=dev))
    assert bt_s.engine.launch_count == launches


# ------------------------------------------------------------------------------------------------
# argument checks
# ------------------------------------------------------------------------------------------------
def test_invalid_arguments_are_refused_before_any_launch(engine):
    lib, h = engine.lib, engine.handle
    dev = engine.device
    planes = torch.zeros((2, 3), dtype=torch.int64, device=dev)
    pitches = torch.full((2, 2), 8, dtype=torch.int32, device=dev)
    hw = torch.full((2, 2), 8, dtype=torch.int32, device=dev)
    surface = torch.zeros(2, dtype=torch.int32, device=dev)
    boxes = torch.zeros((2, 4), dtype=torch.float64, device=dev)
    slots = torch.zeros(2, dtype=torch.int32, device=dev)
    dst = torch.zeros(512, dtype=torch.uint8, device=dev)
    off = torch.zeros(2, dtype=torch.int64, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    P, Q, W_, S_, B, L, D, O_ = p(planes), p(pitches), p(hw), p(surface), p(boxes), p(slots), p(dst), p(off)
    #          format planes pitches hw  m  surface boxes slots factor first n  dst dst_offsets
    ok = dict(f=1, P=P, Q=Q, W=W_, m=2, S=S_, B=B, L=None, x=2.0, first=0, n=2, D=D, O=O_)
    calls = {
        "format 0": dict(f=0), "format 3": dict(f=3), "factor 0": dict(x=0.0), "factor < 0": dict(x=-4.0), "factor nan": dict(x=float("nan")),
        "negative n": dict(n=-1), "negative m": dict(m=-1), "m > max_tracks": dict(m=65),
        "state past max_tracks": dict(B=None, first=63), "state first < 0": dict(B=None, first=-1),
        "state first = INT_MAX": dict(B=None, first=2 ** 31 - 1),
        "null planes": dict(P=None), "null pitches": dict(Q=None), "null frame_hw": dict(W=None), "null item_surface": dict(S=None),
        "null dst": dict(D=None), "null dst_offsets": dict(O=None),
    }
    before = engine.launch_count
    for name, change in calls.items():
        a = {**ok, **change}
        rc = lib.vt_yuv420_crops_to_surface_rgb(h, a["f"], a["P"], a["Q"], a["W"], a["m"], a["S"], a["B"], a["L"], a["x"], a["first"],
                                                a["n"], a["D"], a["O"], None)
        assert rc == -1, name
        assert lib.vt_last_error(h), name
    assert engine.launch_count == before
    assert lib.vt_yuv420_crops_to_surface_rgb(h, 1, None, None, None, 0, None, None, None, 2.0, 0, 0, None, None, None) == 0   # n == 0
    assert lib.vt_yuv420_crops_to_surface_rgb(h, 1, None, None, None, 5, None, None, None, 4.0, 70, 0, None, None, None) == 0
    assert engine.launch_count == before
    for bad in (dict(format="yuv444"), dict(planes=planes.to(torch.int32)), dict(boxes=boxes[:1]), dict(item_surface=surface.to(torch.int64)),
                dict(slots=slots[:1]), dict(dst_offsets=off[:1])):
        a = dict(format="nv12", planes=planes, pitches=pitches, frame_hw=hw, dst=dst, dst_offsets=off, item_surface=surface, boxes=boxes)
        a.update(bad)
        fmt = a.pop("format")
        with pytest.raises(ValueError):
            engine.yuv420_crops_to_surface_rgb(fmt, a.pop("planes"), a.pop("pitches"), a.pop("frame_hw"), a.pop("dst"), a.pop("dst_offsets"),
                                               a.pop("item_surface"), 2.0, **a)
    assert engine.launch_count == before
