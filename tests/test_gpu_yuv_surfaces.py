"""Device-resident, pitched YUV 4:2:0 surfaces (decoder output) converted only where a crop reads them: the rectangle kernel
against cv2.cvtColor byte for byte with canary-checked bounds, the batched and batch-1 trackers against their RGB paths fed
cv2.cvtColor of the same frames (bit for bit), CUDA-graph capture, and the C ABI's argument checks."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")

from oracle import vt_oracle as O
from oracle import yuv420 as Y

pytestmark = pytest.mark.gpu
FORMATS = ["nv12", "i420"]
CV = {"nv12": cv2.COLOR_YUV2RGB_NV12, "i420": cv2.COLOR_YUV2RGB_I420}
CANARY = 0xA5


@pytest.fixture(scope="module")
def cfg():
    from vittracker_b200 import load_cfg
    return load_cfg()


@pytest.fixture(scope="module")
def engine(cfg):
    from vittracker_b200.engine import Engine
    return Engine(cfg, max_tracks=64)


@pytest.fixture(scope="module")
def sd():
    return O.make_state_dict(seed=5, stress=True)


def pack_surface(frame, fmt, P, S, rng):
    """A (H*3/2) x W cvtColor-layout frame as a decoder surface of S rows (>= H) and pitch P (>= W): luma rows [0, H); NV12 chroma
    rows [S, S + H/2); I420 U at byte S * P with rows P/2 apart, V (S/2) * (P/2) bytes after it.  Every other byte (row padding, the
    surface rows below H, the gap between the planes) holds random poison, so a read of any of them changes the result."""
    H, W = frame.shape[0] * 2 // 3, frame.shape[1]
    out = rng.integers(0, 256, (S * 3 // 2, P), dtype=np.uint8)
    out[:H, :W] = frame[:H]
    if fmt == "nv12":
        out[S:S + H // 2, :W] = frame[H:]
        return out
    c = frame[H:].reshape(-1)
    flat = out.reshape(-1)
    rows, cols = np.arange(H // 2)[:, None] * (P // 2), np.arange(W // 2)[None, :]
    flat[S * P + rows + cols] = c[: H * W // 4].reshape(H // 2, W // 2)
    flat[S * P + (S // 2) * (P // 2) + rows + cols] = c[H * W // 4:].reshape(H // 2, W // 2)
    return out


def surfaces_of(frames, fmt, dev, P, S, seed=0):
    """YuvSurfaces over one device tensor [n, S*3/2, P] holding the frames as pitched, poisoned surfaces; returns (surfaces, buffer)."""
    from vittracker_b200.batched import YuvSurfaces
    rng = np.random.default_rng(seed)
    H, W = frames.shape[1] * 2 // 3, frames.shape[2]
    buf = torch.from_numpy(np.stack([pack_surface(f, fmt, P, S, rng) for f in frames])).to(dev)
    return YuvSurfaces.from_frames(buf[:, :, :W], fmt, height=H, surface_rows=S), buf


def expected_rect(box, factor, H, W):
    """What the device converts for a box: even_rect(crop_rect(...)), or None where it writes nothing (odd / tiny frame, crop status
    VT_TRACK_TOO_SMALL or VT_TRACK_OUT_OF_DOMAIN as vt_geom.cuh's crop_geometry decides it)."""
    from vittracker_b200.sequences import crop_rect
    from vittracker_b200.tracker import even_rect
    if H < 2 or W < 2 or H % 2 or W % 2:
        return None
    x, y, w, h = [float(v) for v in box]
    side = math.ceil(math.sqrt(w * h) * factor) if w * h >= 0 else float("nan")
    if not side >= 1:
        return None
    x1, y1 = round(x + 0.5 * w - side * 0.5), round(y + 0.5 * h - side * 0.5)
    if not (max(0, x1) < min(x1 + side, W - 1) and max(0, y1) < min(y1 + side, H - 1)):
        return None
    rect = crop_rect(box, factor, H, W)
    assert rect is not None
    return even_rect(rect, H, W)


def edge_boxes(H, W):
    """Boxes at all four borders, partly off the frame, with x1 / y1 landing on .5 before rounding, odd and even rectangle edges,
    and degenerate ones (crop_sz < 1, crop off the frame)."""
    b = [
        [0.0, 0.0, 40.0, 30.0], [W - 40.0, H - 30.0, 40.0, 30.0], [W - 12.0, 5.0, 30.0, 20.0], [3.0, H - 9.0, 25.0, 40.0],
        [-30.0, H / 2, 60.0, 50.0], [W / 2, -25.0, 50.0, 60.0], [W - 20.0, H / 2, 70.0, 33.0], [W / 3, H - 11.0, 41.0, 60.0],
        [100.0, 100.0, 25.0, 25.0], [101.0, 101.0, 25.0, 25.0], [100.5, 99.5, 25.0, 25.0], [37.25, 61.75, 17.0, 13.0],
        [W / 2 + 0.5, H / 2 - 0.5, 9.0, 9.0], [11.0, 13.0, 3.0, 5.0], [12.0, 14.0, 3.0, 5.0],
        [50.0, 50.0, 0.0, 20.0], [50.0, 50.0, -4.0, 20.0], [5.0, 4.0, 1e-4, 1e-4],          # crop_sz < 1, NaN side; crop_sz = 1
        [-500.0, 10.0, 30.0, 30.0], [W + 200.0, H + 200.0, 30.0, 30.0], [10.0, -400.0, 20.0, 20.0],   # off the frame
    ]
    rng = np.random.default_rng(H + W)
    for _ in range(20):                                   # anywhere, partly outside included, small to large
        w, h = rng.uniform(2, max(3, W / 3)), rng.uniform(2, max(3, H / 3))
        b.append([rng.uniform(-w, W), rng.uniform(-h, H), w, h])
    return np.array(b, dtype=np.float64)


def _check_items(got, want_rgb, rects, dst_off, H, W, tag):
    written = np.zeros(got.size, bool)
    for i, (rect, o) in enumerate(zip(rects, dst_off)):
        if rect is None:
            continue
        ya, yb, xa, xb = rect
        img = got[o:o + H * W * 3].reshape(H, W, 3)
        assert np.array_equal(img[ya:yb, xa:xb], want_rgb[i][ya:yb, xa:xb]), (tag, i, rect)
        region = written[o:o + H * W * 3].reshape(H, W, 3)
        region[ya:yb, xa:xb] = True
    assert (got[~written] == CANARY).all(), (tag, int((got[~written] != CANARY).sum()))


# ------------------------------------------------------------------------------------------------
# the rectangle kernel
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("factor", [2.0, 4.0])
@pytest.mark.parametrize("hw", [(720, 1280), (6, 10)])
@pytest.mark.parametrize("fmt", FORMATS)
def test_rectangle_equals_opencv_and_nothing_else_is_written(engine, fmt, hw, factor):
    H, W = hw
    dev = engine.device
    boxes = edge_boxes(H, W)
    n = boxes.shape[0]
    frames = Y.synth_yuv420(4, H, W, seed=H + 7, format=fmt)[np.arange(n) % 4]
    surf, _ = surfaces_of(frames, fmt, dev, P=W + 64 + 6, S=H + 10, seed=1)
    want = [cv2.cvtColor(f, CV[fmt]) for f in frames]
    # items n, n+1: odd frame sizes; n+2: a luma pitch below the width; they alias item 0's planes and own canary regions
    extra_hw = [(H + 1, W), (H, W - 1), (H, W)]
    planes = torch.cat([surf.planes, surf.planes[:1].expand(3, 3)]).contiguous()
    pitches = torch.cat([surf.pitches, surf.pitches[:1].expand(3, 2)]).clone()
    pitches[n + 2, 0] = W - 2
    hw_t = torch.cat([surf.hw, torch.tensor(extra_hw, dtype=torch.int32, device=dev)]).contiguous()
    bx = torch.from_numpy(np.concatenate([boxes, np.repeat(boxes[:1], 3, 0)])).to(dev)
    m = n + 3
    dst_off = [k * (H * W * 3 + 7) + 3 for k in range(m)]                  # every alignment mod 4, canary gaps between items
    dst = torch.full((m * (H * W * 3 + 7) + 8,), CANARY, dtype=torch.uint8, device=dev)
    offs = torch.tensor(dst_off, dtype=torch.int64, device=dev)
    launches = engine.launch_count
    engine.yuv420_crop_to_rgb(fmt, planes, pitches, hw_t, dst, offs, factor, boxes=bx)
    assert engine.launch_count == launches + 1
    rects = [expected_rect(b, factor, H, W) for b in boxes] + [None, None, None]
    assert any(r is None for r in rects[:n]) and sum(r is not None for r in rects) >= 10
    _check_items(dst.cpu().numpy(), want + [None] * 3, rects, dst_off, H, W, (fmt, hw, factor))

    # the state of tracks [first, first + k) instead of a box array: the same bytes
    k, first = min(n, 64 - 5), 5
    engine.tracks_set_state(bx[:k].contiguous(), first=first)
    dst2 = torch.full_like(dst, CANARY)
    engine.yuv420_crop_to_rgb(fmt, planes[:k].contiguous(), pitches[:k].contiguous(), hw_t[:k].contiguous(), dst2, offs[:k].contiguous(),
                              factor, boxes=None, first=first)
    _check_items(dst2.cpu().numpy(), want[:k], rects[:k], dst_off[:k], H, W, (fmt, hw, factor, "state"))


@pytest.mark.parametrize("fmt", FORMATS)
def test_mixed_pitches_and_offsets_in_one_call_equal_one_call_per_item(engine, fmt):
    from vittracker_b200.batched import YuvSurfaces
    H, W = 360, 640
    dev = engine.device
    frames = Y.synth_yuv420(6, H, W, seed=31, format=fmt)
    rng = np.random.default_rng(2)
    ys, us, vs = [], [], []
    for k, f in enumerate(frames):
        P, S = W + 2 * k + (0 if k % 2 else 130), H + 2 * k         # pitches and surface heights differ per item
        arr = pack_surface(f, fmt, P, S, rng)
        lead = 1 + 5 * k                                            # the surface starts at an odd byte of its own buffer
        raw = torch.from_numpy(np.concatenate([rng.integers(0, 256, lead, dtype=np.uint8), arr.reshape(-1)])).to(dev)
        t = raw[lead:].view(S * 3 // 2, P)
        ys.append(t[:H, :W])
        if fmt == "nv12":
            us.append(t[S:S + H // 2, :W])
        else:
            u0 = lead + S * P
            us.append(raw.as_strided((H // 2, W // 2), (P // 2, 1), u0))
            vs.append(raw.as_strided((H // 2, W // 2), (P // 2, 1), u0 + (S // 2) * (P // 2)))
    surf = YuvSurfaces(fmt, ys, us, vs if fmt == "i420" else None)
    assert len(set(surf.pitches[:, 0].tolist())) == len(frames)
    boxes = torch.from_numpy(np.array([[20.0 + 90 * k, 30.0 + 40 * k, 50.0 + 7 * k, 40.0 + 5 * k] for k in range(len(frames))])).to(dev)
    offs = torch.arange(len(frames), dtype=torch.int64, device=dev) * (H * W * 3 + 1)
    one = torch.full((len(frames) * (H * W * 3 + 1),), CANARY, dtype=torch.uint8, device=dev)
    each = one.clone()
    engine.yuv420_crop_to_rgb(fmt, surf.planes, surf.pitches, surf.hw, one, offs, 4.0, boxes=boxes)
    for k in range(len(frames)):
        s = YuvSurfaces(fmt, ys[k], us[k], vs[k] if fmt == "i420" else None)
        engine.yuv420_crop_to_rgb(fmt, s.planes, s.pitches, s.hw, each, offs[k:k + 1].contiguous(), 4.0, boxes=boxes[k:k + 1].contiguous())
    assert torch.equal(one, each)
    rects = [expected_rect(b, 4.0, H, W) for b in boxes.cpu().numpy()]
    _check_items(one.cpu().numpy(), [cv2.cvtColor(f, CV[fmt]) for f in frames], rects, offs.tolist(), H, W, fmt)


# ------------------------------------------------------------------------------------------------
# the batched tracker
# ------------------------------------------------------------------------------------------------
NB, FB, HB, WB, STEPS = 32, 8, 720, 1280, 8


def _config(kind):
    from vittracker_b200 import load_cfg
    cfg = load_cfg()
    if kind != "generic":
        return cfg, O.make_state_dict(seed=5, stress=True), {"blocks_impl": kind}
    C_, heads, depth, hc = 96, 3, 2, 64                     # the "small" configuration of test_gpu_generic.py
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.BACKBONE.DEPTH = C_, heads, depth
    cfg.MODEL.HEAD.NUM_CHANNELS = hc
    return cfg, O.make_state_dict(seed=3, C=C_, depth=depth, head_ch=hc), {"depth": depth}


def _init_boxes():
    """The bench's open-loop boxes plus small targets (w, h ~ U(16, 120))."""
    b = O.synth_boxes(NB, HB, WB, seed=90)
    rng = np.random.default_rng(91)
    for i in range(0, NB, 4):
        w, h = rng.uniform(16, 120, 2)
        b[i] = [rng.uniform(0, WB - w), rng.uniform(0, HB - h), w, h]
    return b


@pytest.mark.parametrize("kind", ["tcgen05", "simt", "generic"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_closed_loop_on_surfaces_equals_rgb_of_opencv(fmt, kind):
    from vittracker_b200 import BatchedTracker, FramePool
    cfg, sd, kw = _config(kind)
    bt_y = BatchedTracker(cfg, sd, max_tracks=NB, **kw)
    bt_r = BatchedTracker(cfg, sd, max_tracks=NB, **kw)
    dev = bt_y.device
    frames = Y.synth_yuv420(FB, HB, WB, seed=17, format=fmt, smooth=True)
    pool = FramePool(np.stack([cv2.cvtColor(f, CV[fmt]) for f in frames]), dev)
    boxes = _init_boxes()
    res = {"yuv": [], "rgb": []}
    for t in range(STEPS + 1):
        idx = (np.arange(NB) + t) % FB
        surf, _ = surfaces_of(frames[idx], fmt, dev, P=WB + 256, S=HB + 8, seed=t)
        if t == 0:
            st_y = bt_y.initialize_yuv(surf, boxes)
            st_r = bt_r.initialize(pool, torch.from_numpy(idx).to(dev), boxes)
            assert torch.equal(st_y, st_r) and int(st_y.abs().sum()) == 0
            continue
        for key, bt, run in (("yuv", bt_y, lambda: bt_y.track_yuv(surf, detail=True)),
                             ("rgb", bt_r, lambda: bt_r.track(pool, torch.from_numpy(idx).to(dev), detail=True))):
            o, d = run()
            maps = bt.engine.tracks_last_maps(0, NB)
            res[key].append((o.cpu().numpy(), d.cpu().numpy(), {k: v.cpu().numpy() for k, v in maps.items()}))
    for t, ((oa, da, ma), (ob, db, mb)) in enumerate(zip(res["yuv"], res["rgb"])):
        assert np.array_equal(oa, ob), t
        assert np.array_equal(da, db), t
        for k in ma:
            assert np.array_equal(ma[k], mb[k], equal_nan=True), (t, k)


@pytest.mark.parametrize("fmt", FORMATS)
def test_track_yuv_in_a_cuda_graph_equals_plain_launches(cfg, sd, fmt):
    from vittracker_b200 import BatchedTracker
    n, steps = 16, 5
    frames = Y.synth_yuv420(steps, HB, WB, seed=23, format=fmt, smooth=True)
    plain, graphed = BatchedTracker(cfg, sd, max_tracks=n), BatchedTracker(cfg, sd, max_tracks=n)
    dev = plain.device
    data = [surfaces_of(frames[(np.arange(n) + t) % steps], fmt, dev, P=WB + 128, S=HB + 16, seed=t)[1] for t in range(steps)]
    surf, buf = surfaces_of(frames[np.zeros(n, int)], fmt, dev, P=WB + 128, S=HB + 16)          # fixed surfaces, refilled per step
    boxes = _init_boxes()[:n]
    out = {"plain": [], "graph": []}
    for key, bt in (("plain", plain), ("graph", graphed)):
        buf.copy_(data[0])
        assert int(bt.initialize_yuv(surf, boxes).abs().sum()) == 0
        buf.copy_(data[1])
        out[key].append(bt.track_yuv(surf).cpu().numpy())
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize(dev)
    with torch.cuda.graph(g):
        graphed.track_yuv(surf)
    for t in range(2, steps):
        buf.copy_(data[t])
        out["plain"].append(plain.track_yuv(surf).cpu().numpy())
        buf.copy_(data[t])
        g.replay()
        out["graph"].append(graphed.out_boxes[:n].cpu().numpy())
        mp, mg = plain.engine.tracks_last_maps(0, n), graphed.engine.tracks_last_maps(0, n)
        for k in mp:
            assert torch.equal(torch.nan_to_num(mp[k]), torch.nan_to_num(mg[k])), (t, k)
    for t, (a, b) in enumerate(zip(out["plain"], out["graph"])):
        assert np.array_equal(a, b), t


# ------------------------------------------------------------------------------------------------
# the batch-1 tracker
# ------------------------------------------------------------------------------------------------
def _tracker(sd, fmt, blocks="tcgen05", graph=True):
    from vittracker_b200 import get_tracker_class, parameters
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    params.blocks_impl = blocks
    params.cuda_graph = graph
    params.frame_format = fmt
    return get_tracker_class()(params, "synthetic")


def _device_frame(f, fmt, dev, form, rng):
    """One host frame on the device: "tensor" = a (H*3/2) x W tensor with a padded pitch, "planes" = separate strided planes."""
    H, W = f.shape[0] * 2 // 3, f.shape[1]
    P = W + 96
    arr = torch.from_numpy(pack_surface(f, fmt, P, H, rng)).to(dev)
    if form == "tensor":
        return arr[:, :W]
    if fmt == "nv12":
        return (arr[:H, :W].contiguous(), arr[H:, :W])                       # a luma plane of pitch W, a chroma plane of pitch P
    flat = arr.reshape(-1)
    return (arr[:H, :W], flat.as_strided((H // 2, W // 2), (P // 2, 1), H * P),
            flat.as_strided((H // 2, W // 2), (P // 2, 1), H * P + (H // 2) * (P // 2)))


@pytest.mark.parametrize("blocks", ["tcgen05", "simt"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_batch1_device_frames_equal_host_frames(sd, fmt, blocks):
    from test_gpu_yuv import _same_result, _sequence
    td, th = _tracker(sd, fmt, blocks), _tracker(sd, fmt, blocks)
    dev = td.engine.device
    seq = _sequence(fmt)                                   # 20 frames at 720p, then 15 at 1080 x 1920
    rng = np.random.default_rng(4)
    init = {"init_bbox": [600.0, 300.0, 80.0, 60.0]}
    assert td.initialize(_device_frame(seq[0], fmt, dev, "tensor", rng), dict(init)) is None
    assert th.initialize(seq[0], dict(init)) is None
    assert np.array_equal(td.z_patch_arr, th.z_patch_arr)
    edges = {8: [-20.0, 600.0, 80.0, 90.0], 14: [1230.0, 3.0, 70.0, 50.0], 24: [1880.0, -15.0, 70.0, 60.0], 30: [7.0, 1050.0, 90.0, 41.0]}
    for t in range(1, len(seq)):
        if t in edges:                                      # crops that overhang the frame
            td.state, th.state = list(edges[t]), list(edges[t])
        dframe = _device_frame(seq[t], fmt, dev, "tensor" if t % 2 else "planes", rng)
        _same_result(td.track(dframe, {}), th.track(seq[t], {}), td, th, (fmt, blocks, t))
    assert td._graph is not None


def test_batch1_refuses_host_tensors_and_wrong_planes(sd):
    td = _tracker(sd, "nv12")
    with pytest.raises(ValueError):
        td.initialize(torch.zeros((1080, 1280), dtype=torch.uint8), {"init_bbox": [10.0, 10.0, 20.0, 20.0]})
    dev = td.engine.device
    with pytest.raises(ValueError):
        td.initialize((torch.zeros((720, 1280), dtype=torch.uint8, device=dev), torch.zeros((360, 640), dtype=torch.uint8, device=dev)),
                      {"init_bbox": [10.0, 10.0, 20.0, 20.0]})


# ------------------------------------------------------------------------------------------------
# argument checks
# ------------------------------------------------------------------------------------------------
def test_invalid_arguments_are_refused_before_any_launch(engine):
    lib, h = engine.lib, engine.handle
    dev = engine.device
    planes = torch.zeros((2, 3), dtype=torch.int64, device=dev)
    pitches = torch.full((2, 2), 8, dtype=torch.int32, device=dev)
    hw = torch.full((2, 2), 8, dtype=torch.int32, device=dev)
    boxes = torch.zeros((2, 4), dtype=torch.float64, device=dev)
    dst = torch.zeros(512, dtype=torch.uint8, device=dev)
    off = torch.zeros(2, dtype=torch.int64, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    P, Q, W_, B, D, O_ = p(planes), p(pitches), p(hw), p(boxes), p(dst), p(off)
    before = engine.launch_count
    calls = {
        "format 0": (0, P, Q, W_, B, 2.0, 0, 2, D, O_), "format 3": (3, P, Q, W_, B, 2.0, 0, 2, D, O_),
        "null planes": (1, None, Q, W_, B, 2.0, 0, 2, D, O_), "null pitches": (1, P, None, W_, B, 2.0, 0, 2, D, O_),
        "null frame_hw": (1, P, Q, None, B, 2.0, 0, 2, D, O_), "null dst": (1, P, Q, W_, B, 2.0, 0, 2, None, O_),
        "null dst_offsets": (1, P, Q, W_, B, 2.0, 0, 2, D, None), "negative n": (1, P, Q, W_, B, 2.0, 0, -1, D, O_),
        "factor 0": (1, P, Q, W_, B, 0.0, 0, 2, D, O_), "factor < 0": (2, P, Q, W_, B, -4.0, 0, 2, D, O_),
        "factor nan": (1, P, Q, W_, B, float("nan"), 0, 2, D, O_),
        "state past max_tracks": (1, P, Q, W_, None, 4.0, 63, 2, D, O_), "state first < 0": (2, P, Q, W_, None, 4.0, -1, 2, D, O_),
    }
    for name, args in calls.items():
        assert lib.vt_yuv420_crop_to_rgb(h, *args, None) == -1, name
        assert lib.vt_last_error(h), name
    assert lib.vt_yuv420_crop_to_rgb(h, 1, None, None, None, None, 2.0, 0, 0, None, None, None) == 0        # n == 0: a no-op
    assert lib.vt_yuv420_crop_to_rgb(h, 1, None, None, None, None, 4.0, 70, 0, None, None, None) == 0
    assert engine.launch_count == before
    with pytest.raises(ValueError):
        engine.yuv420_crop_to_rgb("yuv444", planes, pitches, hw, dst, off, 2.0, boxes=boxes)
    with pytest.raises(ValueError):
        engine.yuv420_crop_to_rgb("nv12", planes.to(torch.int32), pitches, hw, dst, off, 2.0, boxes=boxes)
    with pytest.raises(ValueError):
        engine.yuv420_crop_to_rgb("nv12", planes, pitches, hw, dst, off, 2.0, boxes=boxes[:1])
    assert engine.launch_count == before
