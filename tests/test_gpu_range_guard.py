"""fp16 operand range of the tensor-core path: never a silent inf.

Every tensor-core contraction takes fp16 hi + lo operands, so an activation with |v| >= 65504 cannot be represented.  A random-init
model stays far inside that range; a trained checkpoint is not guaranteed to.  These tests scale single weight tensors until an operand
overflows and require the per-track status VT_TRACK_NUMERIC_RANGE (state kept, confidence -1, maps NaN) from the tensor-core kernels,
while the fp32 CUDA-core kernels (VT_BLOCKS_SIMT_FP32) keep producing the oracle's answer for the same weights."""
import numpy as np
import pytest
import torch

from oracle import vt_oracle as O

pytestmark = pytest.mark.gpu

VT_TRACK_NUMERIC_RANGE = 3


def _scaled(sd, key, factor, rows=None):
    out = {k: v.clone() for k, v in sd.items()}
    if rows is None:
        out[key] = out[key] * factor
    else:
        out[key][rows[0]:rows[1]] = out[key][rows[0]:rows[1]] * factor
    return out


CASES = [
    ("stem conv1 output", "patch_embed.net.0.c.weight", 1e5, None),
    ("stem conv3 output", "patch_embed.net.4.c.weight", 1e6, None),
    # q and k rows together: scaling k alone (or q alone) only moves scale between them, which weight ingest rebalances away
    ("attention queries and keys", "blocks.0.attn.qkv.weight", 3e5, (0, 96)),
    ("attention values", "blocks.1.attn.qkv.weight", 1e6, (96, 144)),
    ("MLP hidden (GELU output)", "blocks.2.mlp.fc1.weight", 1e6, None),
    ("head conv1 output", "box_head.conv1_ctr.0.weight", 1e7, None),
    ("head conv2 output", "box_head.conv2_size.0.weight", 1e7, None),
]


@pytest.fixture(scope="module")
def setup():
    from vittracker_b200 import load_cfg
    cfg = load_cfg()
    sd = O.make_state_dict(seed=5, stress=True)
    frames = O.synth_frames(2, 360, 640, seed=31, smooth=True)
    boxes = O.synth_boxes(6, 360, 640, seed=32)
    return cfg, sd, frames, boxes


def _run(cfg, sd, frames, boxes, blocks):
    from vittracker_b200 import BatchedTracker, FramePool
    n = len(boxes)
    bt = BatchedTracker(cfg, sd, max_tracks=n, blocks_impl=blocks)
    pool = FramePool(frames, bt.device)
    assert int(bt.initialize(pool, torch.zeros(n, dtype=torch.int64), boxes).abs().sum()) == 0
    before = bt.get_state().cpu().numpy().copy()
    out, det = bt.track(pool, torch.ones(n, dtype=torch.int64), update_state=True, detail=True)
    maps = bt.engine.tracks_last_maps(0, n)
    return out.cpu().numpy(), det.cpu().numpy(), before, bt.get_state().cpu().numpy(), maps


def test_in_range_weights_are_not_flagged(setup):
    cfg, sd, frames, boxes = setup
    out, det, _, _, maps = _run(cfg, sd, frames, boxes, "tcgen05")
    assert (det[:, 6] == 0).all() and (out[:, 4] > 0).all()
    assert torch.isfinite(maps["score_map"]).all()


@pytest.mark.parametrize("what,key,factor,rows", CASES, ids=[c[0] for c in CASES])
def test_overflowing_operand_is_flagged_not_silent(setup, what, key, factor, rows):
    cfg, sd, frames, boxes = setup
    big = _scaled(sd, key, factor, rows)
    out, det, before, after, maps = _run(cfg, big, frames, boxes, "tcgen05")
    assert (det[:, 6] == VT_TRACK_NUMERIC_RANGE).all(), (what, det[:, 6])
    assert (out[:, 4] == -1.0).all(), "confidence of a withheld result is -1"
    assert np.array_equal(out[:, :4], before) and np.array_equal(after, before), "the track state must be kept"
    for m in maps.values():
        assert torch.isnan(m).all(), f"{what}: maps of a flagged track are NaN, never plausible numbers"


@pytest.mark.parametrize("what,key,factor,rows", [CASES[0], CASES[4]], ids=[CASES[0][0], CASES[4][0]])
def test_fp32_kernels_cover_the_same_weights(setup, what, key, factor, rows):
    """The exact mode has no fp16 operands: same weights, finite result, the oracle's arg-max."""
    cfg, sd, frames, boxes = setup
    big = _scaled(sd, key, factor, rows)
    out, det, _, _, maps = _run(cfg, big, frames, boxes, "simt")
    assert (det[:, 6] == 0).all(), det[:, 6]
    assert np.isfinite(out).all() and torch.isfinite(maps["score_map"]).all()
    model = O.OracleModel(big)
    for i in range(2):
        trk = O.OracleTracker(model)
        trk.initialize(frames[0], {"init_bbox": list(boxes[i])})
        trk.track(frames[1], {})
        resp = trk.last["response"].flatten()
        top = torch.topk(resp, 2).values
        if float(top[0] - top[1]) >= 1e-5:
            assert int(det[i, 5]) == int(resp.argmax())


def test_forward_poisons_maps_and_tracker_raises(setup):
    cfg, sd, frames, boxes = setup
    from vittracker_b200 import build_ostrack_dist, get_tracker_class, parameters
    big = _scaled(sd, "blocks.0.mlp.fc1.weight", 1e6)
    net = build_ostrack_dist(cfg)
    net.load_state_dict(big, strict=False)
    net.cuda()
    z = torch.randn(2, 3, 128, 128)
    x = torch.randn(2, 3, 256, 256)
    out = net.forward(z=z, x=x)
    for k in ("score_map", "size_map", "offset_map", "pred_boxes"):
        assert torch.isnan(out[k]).all(), k
    params = parameters("vit_48_h32_noKD")
    params.state_dict = big
    trk = get_tracker_class()(params, "synthetic")
    trk.initialize(frames[0], {"init_bbox": list(boxes[0])})
    with pytest.raises(FloatingPointError):
        trk.track(frames[1], {})
