"""YUV 4:2:0 (NV12 / I420) frames on the device: the conversion kernel against cv2.cvtColor byte for byte, the rectangle
upload's bounds, the batch-1 tracker and the batched feeder against their RGB paths fed cv2.cvtColor of the same frames
(bit for bit), and the C ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")

from conftest import state_dict_from_npz
from oracle import vt_oracle as O
from oracle import yuv420 as Y
from test_tracking_edges import CASES, FRAMES, _case_boxes
from test_yuv import CV, exhaustive_yuv420

pytestmark = pytest.mark.gpu
FORMATS = ["nv12", "i420"]
CANARY = 0xA5


@pytest.fixture(scope="module")
def cfg():
    from vittracker_b200 import load_cfg
    return load_cfg()


@pytest.fixture(scope="module")
def engine(cfg):
    from vittracker_b200.engine import Engine
    return Engine(cfg, max_tracks=1)


@pytest.fixture(scope="module")
def stress_sd(golden_model):
    return state_dict_from_npz(golden_model)


def rgb_of(frames, fmt):
    return np.stack([cv2.cvtColor(f, CV[fmt]) for f in frames])


def _convert(engine, frames, fmt, src_mis, dst_mis, extra_hw=()):
    """Whole frames at the given byte offsets mod 4 in one call; returns (dst buffer, dst offsets, sizes)."""
    src_parts, src_off, dst_off, hw, pos, dpos = [], [], [], [], 0, 0
    for f, sm, dm in zip(frames, src_mis, dst_mis):
        H, W = f.shape[0] * 2 // 3, f.shape[1]
        pos = (pos + 3) // 4 * 4 + sm
        dpos = (dpos + 3) // 4 * 4 + dm
        src_parts.append((pos, f.reshape(-1)))
        src_off.append(pos); dst_off.append(dpos); hw.append((H, W))
        pos += f.size + 5
        dpos += H * W * 3 + 7
    for (H, W) in extra_hw:                  # items whose size the device must refuse: they point at the same bytes
        src_off.append(0); dst_off.append(0); hw.append((H, W))
    src = np.zeros(pos + 16, np.uint8)
    for p, a in src_parts:
        src[p:p + a.size] = a
    dev = engine.device
    dst = torch.full((dpos + 16,), CANARY, dtype=torch.uint8, device=dev)
    t = lambda a, dt: torch.tensor(np.asarray(a), dtype=dt, device=dev)
    engine.yuv420_to_rgb(torch.from_numpy(src).to(dev), t(src_off, torch.int64), t(hw, torch.int32).reshape(-1, 2), dst,
                         t(dst_off, torch.int64), fmt)
    return dst.cpu().numpy(), dst_off[: len(frames)], hw[: len(frames)]


# ------------------------------------------------------------------------------------------------
# 1 + 2: the kernel
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", FORMATS)
def test_kernel_every_triple_equals_opencv(engine, fmt):
    f = exhaustive_yuv420(fmt)
    dst, off, _ = _convert(engine, [f], fmt, [0], [0])
    got = dst[off[0]:off[0] + 4096 * 4096 * 3].reshape(4096, 4096, 3)
    want = cv2.cvtColor(f, CV[fmt])
    assert np.array_equal(got, want), int((got != want).any(-1).sum())


@pytest.mark.parametrize("fmt", FORMATS)
def test_kernel_geometry_alignment_and_bounds(engine, fmt):
    sizes = [(2, 2), (2, 1282), (6, 10), (2160, 3840)]
    frames, src_mis, dst_mis = [], [], []
    for k, (H, W) in enumerate(sizes):
        for m in range(4):
            if H == 2160 and m % 2:
                continue
            frames.append(Y.synth_yuv420(1, H, W, seed=10 * k + m, format=fmt)[0])
            src_mis.append(m)
            dst_mis.append((m + k + 1) % 4)
    # an odd-sized item is skipped on the device: nothing is written for it (it aliases the first frame's destination)
    dst, off, hw = _convert(engine, frames, fmt, src_mis, dst_mis, extra_hw=[(3, 4), (4, 5)])
    written = np.zeros(dst.size, bool)
    for f, o, (H, W) in zip(frames, off, hw):
        got = dst[o:o + H * W * 3].reshape(H, W, 3)
        assert np.array_equal(got, cv2.cvtColor(f, CV[fmt])), (H, W, o % 4)
        written[o:o + H * W * 3] = True
    assert (dst[~written] == CANARY).all()


RECTS = {"odd": (3, 8, 5, 11), "edge_bottom_right": (-3, None, -7, None), "edge_top_left": (0, 1, 0, 3),
         "one_pixel": (-1, None, 0, 1), "one_pixel_odd": (5, 6, 9, 10), "whole": (0, None, 0, None)}


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("hw", [(720, 1280), (6, 10)])
def test_rect_upload_writes_exactly_the_widened_rectangle(engine, fmt, hw):
    from vittracker_b200.tracker import even_rect
    H, W = hw
    f = Y.synth_yuv420(1, H, W, seed=H, format=fmt)[0]
    want = cv2.cvtColor(f, CV[fmt])
    dev = engine.device
    staging = torch.empty(H * W * 3 // 2, dtype=torch.uint8).pin_memory()
    staging_dev = torch.empty(H * W * 3 // 2, dtype=torch.uint8, device=dev)
    for name, (y0, y1, x0, x1) in RECTS.items():
        y0, x0 = y0 % H if y0 < 0 else y0, x0 % W if x0 < 0 else x0
        y1, x1 = H if y1 is None else min(y1, H), W if x1 is None else min(x1, W)
        frame = torch.full((H * W * 3 + 8,), CANARY, dtype=torch.uint8, device=dev)
        launches = engine.launch_count
        engine.upload_yuv420_rect(fmt, f, y0, y1, x0, x1, staging, staging_dev, frame[4:])
        assert engine.launch_count == launches + 1
        got = frame.cpu().numpy()
        assert (got[:4] == CANARY).all() and (got[-4:] == CANARY).all(), name
        got = got[4:-4].reshape(H, W, 3)
        ya, yb, xa, xb = even_rect((y0, y1, x0, x1), H, W)
        inside = np.zeros((H, W), bool)
        inside[ya:yb, xa:xb] = True
        assert np.array_equal(got[inside], want[inside]), name
        assert (got[~inside] == CANARY).all(), name


# ------------------------------------------------------------------------------------------------
# 3: the batch-1 tracker
# ------------------------------------------------------------------------------------------------
def _tracker(sd, blocks, fmt, graph):
    from vittracker_b200 import get_tracker_class, parameters
    params = parameters("vit_48_h32_noKD")
    params.state_dict = sd
    params.blocks_impl = blocks
    params.cuda_graph = graph
    if fmt != "rgb":
        params.frame_format = fmt
    return get_tracker_class()(params, "synthetic")


def _same_result(a, b, ta, tb, tag):
    assert a["target_bbox"] == b["target_bbox"], (tag, a["target_bbox"], b["target_bbox"])
    assert float(a["confidence"]) == float(b["confidence"]), tag
    assert ta.last_detail == tb.last_detail, tag


def _sequence(fmt):
    """35 frames: 20 at 720p, then 15 at 1080 x 1920 (a frame-size change mid-sequence)."""
    a = Y.synth_yuv420(4, 720, 1280, seed=41, format=fmt, smooth=True)
    b = Y.synth_yuv420(3, 1080, 1920, seed=42, format=fmt, smooth=True)
    return [a[t % 4] for t in range(20)] + [b[t % 3] for t in range(15)]


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("weights", ["default", "stress"])
@pytest.mark.parametrize("blocks", ["tcgen05", "simt"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_tracker_closed_loop_equals_rgb_of_opencv(stress_sd, fmt, blocks, weights, graph):
    sd = stress_sd if weights == "stress" else O.make_state_dict(seed=0)
    ty, tr = _tracker(sd, blocks, fmt, graph), _tracker(sd, blocks, "rgb", graph)
    seq = _sequence(fmt)
    init = {"init_bbox": [600.0, 300.0, 80.0, 60.0]}
    assert ty.initialize(seq[0], dict(init)) is None and tr.initialize(cv2.cvtColor(seq[0], CV[fmt]), dict(init)) is None
    assert np.array_equal(ty.z_patch_arr, tr.z_patch_arr)
    for t in range(1, len(seq)):
        _same_result(ty.track(seq[t], {}), tr.track(cv2.cvtColor(seq[t], CV[fmt]), {}), ty, tr, (fmt, blocks, weights, t))
    if graph:
        assert ty._graph is not None


EVEN_CASES = [nm for nm in CASES if CASES[nm][0] in ("hd", "small", "uhd")]


@pytest.mark.parametrize("blocks", ["tcgen05", "simt"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_tracker_crops_overhanging_every_side(stress_sd, fmt, blocks):
    ty, tr = _tracker(stress_sd, blocks, fmt, True), _tracker(stress_sd, blocks, "rgb", True)
    frames = {k: Y.synth_yuv420(2, *FRAMES[k], seed=500 + i, format=fmt) for i, k in enumerate(("hd", "small", "uhd"))}
    for name in sorted(EVEN_CASES, key=lambda nm: CASES[nm][0]):
        fr, tbox, sbox = _case_boxes(name)
        f0, f1 = frames[fr]
        ty.initialize(f0, {"init_bbox": list(tbox)})
        tr.initialize(cv2.cvtColor(f0, CV[fmt]), {"init_bbox": list(tbox)})
        assert np.array_equal(ty.z_patch_arr, tr.z_patch_arr), name
        ty.state = [float(v) for v in sbox]
        tr.state = [float(v) for v in sbox]
        _same_result(ty.track(f1, {}), tr.track(cv2.cvtColor(f1, CV[fmt]), {}), ty, tr, name)


def test_tracker_short_run_against_oracle_closed_loop(stress_sd):
    from test_gpu_parity import TIE_GAP, close
    seq = _sequence("nv12")[:6]
    ty = _tracker(stress_sd, "simt", "nv12", True)
    ref = O.OracleTracker(O.OracleModel(stress_sd))
    init = {"init_bbox": [600.0, 300.0, 80.0, 60.0]}
    ty.initialize(seq[0], dict(init))
    ref.initialize(Y.yuv420_to_rgb(seq[0], "nv12"), dict(init))
    assert np.array_equal(ty.z_patch_arr, ref.z_patch_arr)
    for t in range(1, len(seq)):
        got = ty.track(seq[t], {})
        want = ref.track(Y.yuv420_to_rgb(seq[t], "nv12"), {})
        top = torch.topk(ref.last["response"].flatten(), 2).values
        if float(top[0] - top[1]) >= TIE_GAP:                  # a near-tie may resolve either way (SURVEY 8d)
            assert close(got["target_bbox"], want["target_bbox"]), (t, got["target_bbox"], want["target_bbox"])
            assert abs(float(got["confidence"]) - float(want["confidence"])) < 1e-4
        ty.state = ref.state = list(want["target_bbox"])        # both loops go on from the oracle's box


def test_tracker_rejects_malformed_yuv_frames(stress_sd):
    ty = _tracker(stress_sd, "tcgen05", "nv12", True)
    for bad in (np.zeros((720, 1280, 3), np.uint8), np.zeros((1081, 1280), np.uint8), np.zeros((1080, 1279), np.uint8)):
        with pytest.raises(ValueError):
            ty.initialize(bad, {"init_bbox": [10.0, 10.0, 20.0, 20.0]})
    with pytest.raises(ValueError):
        _tracker(stress_sd, "tcgen05", "yuyv", True)


# ------------------------------------------------------------------------------------------------
# 4: batched
# ------------------------------------------------------------------------------------------------
N, F, FH, FW = 1024, 64, 720, 1280


@pytest.fixture(scope="module")
def nv12_frames():
    return Y.synth_yuv420(2 * F, FH, FW, seed=7, format="nv12")


def _bt(cfg, sd, **kw):
    from vittracker_b200 import BatchedTracker
    return BatchedTracker(cfg, sd, max_tracks=N, **kw)


def _run_feeder(bt, feeder, host_sets, boxes, steps=5):
    offs = torch.from_numpy((np.arange(N) % F) * FH * FW * 3).to(bt.device)
    out = []
    feeder.upload(host_sets[0], boxes[0])
    for t in range(steps):
        fp = feeder.acquire()
        if t + 1 < steps:
            feeder.upload(host_sets[(t + 1) % 2], boxes[(t + 1) % len(boxes)])
        bt.engine.tracks_set_state(fp.boxes, first=0)
        o, d = bt.track_offsets(fp.data, offs, update_state=True, detail=True)
        feeder.release(fp)
        maps = bt.engine.tracks_last_maps(0, N)
        out.append((o.cpu().numpy(), d.cpu().numpy(), {k: v.cpu().numpy() for k, v in maps.items()}))
    return out


def _assert_same_steps(a, b):
    for t, ((oa, da, ma), (ob, db, mb)) in enumerate(zip(a, b)):
        assert np.array_equal(oa, ob), t
        assert np.array_equal(da, db), t
        for k in ma:
            assert np.array_equal(ma[k], mb[k]), (t, k)


def test_feeder_nv12_equals_rgb_feeder_of_opencv(cfg, stress_sd, nv12_frames):
    from vittracker_b200 import FramePool, PipelinedFrameFeeder
    bt_y, bt_r = _bt(cfg, stress_sd), _bt(cfg, stress_sd)
    dev = bt_y.device
    yuv_sets = [torch.from_numpy(nv12_frames[k * F:(k + 1) * F]).pin_memory() for k in range(2)]
    rgb_sets = [torch.from_numpy(rgb_of(nv12_frames[k * F:(k + 1) * F], "nv12")).pin_memory() for k in range(2)]
    boxes = [torch.from_numpy(O.synth_boxes(N, FH, FW, seed=60 + s)).pin_memory() for s in range(5)]
    init_pool = FramePool(rgb_sets[1], dev)
    for bt in (bt_y, bt_r):
        assert int(bt.initialize(init_pool, torch.arange(N, device=dev) % F, O.synth_boxes(N, FH, FW, seed=59)).abs().sum()) == 0
    fy = PipelinedFrameFeeder(F, FH, FW, dev, max_tracks=N, frame_format="nv12", engine=bt_y.engine)
    fr = PipelinedFrameFeeder(F, FH, FW, dev, max_tracks=N)
    _assert_same_steps(_run_feeder(bt_y, fy, yuv_sets, boxes), _run_feeder(bt_r, fr, rgb_sets, boxes))


@pytest.mark.parametrize("fmt", FORMATS)
def test_framepool_from_device_yuv_equals_rgb_pool(cfg, stress_sd, fmt):
    from vittracker_b200 import FramePool
    frames = Y.synth_yuv420(F, FH, FW, seed=8, format=fmt, smooth=True)
    bt = _bt(cfg, stress_sd)
    p_y = FramePool.from_yuv420(bt.engine, torch.from_numpy(frames).to(bt.device), fmt)
    p_r = FramePool(rgb_of(frames, fmt), bt.device)
    assert torch.equal(p_y.data, p_r.data)
    p_h = FramePool.from_yuv420(bt.engine, frames, fmt)                       # from host memory too
    assert torch.equal(p_h.data, p_r.data)
    with pytest.raises(ValueError):
        FramePool.from_yuv420(bt.engine, frames[:, :-1], fmt)


def test_generic_configuration_steps_on_converted_frames(nv12_frames):
    from vittracker_b200 import FramePool, load_cfg
    C_, heads, depth, hc = 96, 3, 2, 64                  # the "small" configuration of test_gpu_generic.py
    cfg = load_cfg()
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.BACKBONE.DEPTH = C_, heads, depth
    cfg.MODEL.HEAD.NUM_CHANNELS = hc
    sd = O.make_state_dict(seed=3, C=C_, depth=depth, head_ch=hc)
    n = 256
    res = []
    for fmt in ("nv12", "rgb"):
        bt = _bt(cfg, sd, depth=depth)
        frames = nv12_frames[:16]
        pool = FramePool.from_yuv420(bt.engine, frames, "nv12") if fmt == "nv12" else FramePool(rgb_of(frames, "nv12"), bt.device)
        idx = torch.arange(n, device=bt.device) % 16
        assert int(bt.initialize(pool, idx, O.synth_boxes(n, FH, FW, seed=70)).abs().sum()) == 0
        o, d = bt.track(pool, (idx + 1) % 16, detail=True)
        res.append((o.cpu().numpy(), d.cpu().numpy()))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])


# ------------------------------------------------------------------------------------------------
# 5: argument checks
# ------------------------------------------------------------------------------------------------
def test_invalid_arguments_are_refused_before_any_launch(engine):
    lib, h = engine.lib, engine.handle
    dev = engine.device
    buf = torch.zeros(4096, dtype=torch.uint8, device=dev)
    pin = torch.zeros(4096, dtype=torch.uint8).pin_memory()
    img = np.zeros((12, 8), np.uint8)                                  # an 8 x 8 frame
    off = torch.zeros(1, dtype=torch.int64, device=dev)
    hw = torch.tensor([[8, 8]], dtype=torch.int32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    I, b, s = img.ctypes.data, p(buf), None
    before = engine.launch_count
    rect_calls = {
        "odd H": (1, I, 7, 8, 0, 2, 0, 2, p(pin), b, b), "odd W": (1, I, 8, 7, 0, 2, 0, 2, p(pin), b, b),
        "format": (3, I, 8, 8, 0, 2, 0, 2, p(pin), b, b), "format 0": (0, I, 8, 8, 0, 2, 0, 2, p(pin), b, b),
        "empty rows": (1, I, 8, 8, 2, 2, 0, 2, p(pin), b, b), "empty cols": (1, I, 8, 8, 0, 2, 3, 3, p(pin), b, b),
        "below": (1, I, 8, 8, 0, 9, 0, 2, p(pin), b, b), "right": (1, I, 8, 8, 0, 2, 0, 9, p(pin), b, b),
        "negative": (1, I, 8, 8, -1, 2, 0, 2, p(pin), b, b),
        "null image": (1, None, 8, 8, 0, 2, 0, 2, p(pin), b, b), "null staging": (1, I, 8, 8, 0, 2, 0, 2, None, b, b),
        "null staging_dev": (1, I, 8, 8, 0, 2, 0, 2, p(pin), None, b), "null frame": (1, I, 8, 8, 0, 2, 0, 2, p(pin), b, None),
    }
    for name, args in rect_calls.items():
        assert lib.vt_upload_yuv420_rect(h, *args, s) == -1, name
        assert lib.vt_last_error(h), name
    conv_calls = {
        "format": (9, b, p(off), p(hw), b, p(off), 1), "null src": (1, None, p(off), p(hw), b, p(off), 1),
        "null src_offsets": (1, b, None, p(hw), b, p(off), 1), "null frame_hw": (1, b, p(off), None, b, p(off), 1),
        "null dst": (1, b, p(off), p(hw), None, p(off), 1), "null dst_offsets": (1, b, p(off), p(hw), b, None, 1),
        "negative n": (1, b, p(off), p(hw), b, p(off), -1),
    }
    for name, args in conv_calls.items():
        assert lib.vt_yuv420_to_rgb(h, *args, s) == -1, name
    assert lib.vt_yuv420_to_rgb(h, 1, None, None, None, None, None, 0, s) == 0          # n == 0: a no-op
    assert engine.launch_count == before
    with pytest.raises(ValueError):
        engine.yuv420_to_rgb(buf, off, hw, buf, off, "yuv444")
