"""Range fallback (vt_set_range_fallback): tracks the tensor-core kernels flag as out of fp16 range are recomputed on the fp32 kernels
in the same step.

One stem weight is scaled so that tracks on a high-contrast frame overflow the fp16 operand range of the tensor-core path while tracks
on a flat frame at the normalisation mean do not (oracle, on the CPU: the unscaled stem conv1 output of a search crop peaks at 3.7 on
the noise frame and at 0.012 on the flat frame; x 3e4 puts the first past 65504 and keeps the second near 400).  A recomputed item must
be bit-identical to a VT_BLOCKS_SIMT_FP32 engine, every other item to the same engine with the fallback off."""
import numpy as np
import pytest
import torch

from oracle import vt_oracle as O

pytestmark = pytest.mark.gpu

RANGE, BAD = 3, 4
H, W = 480, 640
KEY, FACTOR = "patch_embed.net.0.c.weight", 3e4
N, CHUNK = 40, 8
TC_IMPLS = ["tcgen05", "tcgen05_3term"]


@pytest.fixture(scope="module")
def setup():
    from vittracker_b200 import load_cfg
    sd = O.make_state_dict(seed=5, stress=True)
    sd[KEY] = sd[KEY] * FACTOR
    flat = np.empty((H, W, 3), np.uint8)
    flat[...] = (124, 116, 104)                          # round(255 * mean): normalises to ~0
    noise = np.random.default_rng(7).integers(0, 256, (H, W, 3), dtype=np.uint8)
    rng = np.random.default_rng(11)
    # every search crop (4 x sqrt(w h) <= 200 px) lies inside the frame: no zero padding, whose normalised value is not ~0
    boxes = np.stack([rng.uniform(230, 380, N), rng.uniform(150, 260, N), rng.uniform(30, 50, N), rng.uniform(30, 50, N)], 1)
    return load_cfg(), sd, np.stack([flat, noise]), boxes


def _engine(cfg, sd, impl, fallback=False, counter=None, max_tracks=N + 4, chunk=CHUNK):
    from vittracker_b200.engine import Engine
    e = Engine(cfg, max_tracks=max_tracks, blocks_impl=impl, chunk_tracks=chunk)
    e.load_state_dict(sd)
    if fallback:
        e.set_range_fallback(True, counter)
    return e


def _dev(a, dt, dev):
    return torch.as_tensor(np.asarray(a), dtype=dt).to(dev).contiguous()


class Run:
    """One engine with its frames, initialised on the flat frame."""

    def __init__(self, e, frames, boxes):
        self.e, dev = e, e.device
        self.frames = _dev(frames, torch.uint8, dev)
        n = self.n = len(boxes)
        self.hw = _dev([[H, W]] * n, torch.int32, dev)
        st = e.tracks_init(self.frames, self.offs(np.zeros(n, int)), self.hw, _dev(boxes, torch.float64, dev))
        assert int(st.abs().sum()) == 0

    def offs(self, idx):
        return _dev(np.asarray(idx, np.int64) * H * W * 3, torch.int64, self.e.device)

    def step(self, idx, update_state=True, slots=None):
        n = len(idx)
        hw = _dev([[H, W]] * n, torch.int32, self.e.device)
        if slots is None:
            b, d = self.e.tracks_step(self.frames, self.offs(idx), hw, first=0, n=n, update_state=update_state, detail=True)
        else:
            b, d = self.e.tracks_step_slots(self.frames, self.offs(idx), hw, _dev(slots, torch.int32, self.e.device),
                                            update_state=update_state, detail=True)
        maps = self.e.tracks_last_maps(0, n)
        return {"boxes": b.cpu().numpy(), "detail": d.cpu().numpy(), "state": self.e.tracks_get_state(0, self.n).cpu().numpy(),
                **{k: v.cpu().numpy().reshape(n, -1) for k, v in maps.items()}}


def _same(a, b, rows, what):
    for k in ("boxes", "detail", "score_map", "size_map", "offset_map"):
        x, y = a[k][rows], b[k][rows]
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (what, k)


def _frame_idx():
    return np.array([1 if i % 3 == 0 else 0 for i in range(N)])      # noise frame for items 0, 3, 6, ...: flagged in every chunk


@pytest.mark.parametrize("impl", TC_IMPLS)
def test_mixed_batch_range_steps(setup, impl):
    cfg, sd, frames, boxes = setup
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    off, on, simt = (Run(_engine(cfg, sd, impl), frames, boxes), Run(_engine(cfg, sd, impl, True, counter), frames, boxes),
                     Run(_engine(cfg, sd, "simt"), frames, boxes))
    total = 0
    for step in range(2):                                        # closed loop: the second step starts from the recomputed states
        idx = _frame_idx() if step == 0 else 1 - _frame_idx()
        a, b, c = off.step(idx), on.step(idx), simt.step(idx)
        flagged = a["detail"][:, 6] == RANGE
        assert flagged.any() and not flagged.all(), flagged
        assert len({i // CHUNK for i in np.flatnonzero(flagged)}) > 1
        assert (c["detail"][:, 6] == 0).all()
        _same(b, a, ~flagged, "unflagged vs fallback off")
        _same(b, c, flagged, "recomputed vs simt")
        assert (b["detail"][:, 6] == 0).all()
        assert np.array_equal(b["state"][flagged], c["state"][flagged])       # range step: item i is track i
        assert np.array_equal(b["state"][~flagged], a["state"][~flagged])
        total += int(flagged.sum())
        assert int(counter.item()) == total
        # keep the three engines on the same states for the next step
        off.e.tracks_set_state(torch.as_tensor(b["state"]).cuda(), first=0)
        simt.e.tracks_set_state(torch.as_tensor(b["state"]).cuda(), first=0)


@pytest.mark.parametrize("impl", TC_IMPLS)
def test_mixed_batch_slot_lists(setup, impl):
    cfg, sd, frames, boxes = setup
    off, on, simt = (Run(_engine(cfg, sd, impl), frames, boxes), Run(_engine(cfg, sd, impl, True), frames, boxes),
                     Run(_engine(cfg, sd, "simt"), frames, boxes))
    rng = np.random.default_rng(3)
    slots = list(rng.permutation(N)[:30]) + [-1, N + 100, 4, 7, 30]     # bad: negative, past max_tracks, repeated
    slots = [int(s) for s in rng.permutation(np.array(slots))]
    idx = np.array([1 if s >= 0 and s % 2 == 0 else 0 for s in slots])
    for update in (1, 0):
        a, b, c = off.step(idx, update, slots), on.step(idx, update, slots), simt.step(idx, update, slots)
        flagged = a["detail"][:, 6] == RANGE
        assert flagged.any() and not flagged.all()
        bad = a["detail"][:, 6] == BAD
        want = [k for k, s in enumerate(slots) if not 0 <= s < N + 4 or s in slots[:k]]
        assert np.flatnonzero(bad).tolist() == want and (b["detail"][bad, 6] == BAD).all()
        _same(b, a, ~flagged, "unflagged vs fallback off")
        _same(b, c, flagged, "recomputed vs simt")
        fs = [slots[i] for i in np.flatnonzero(flagged)]
        assert np.array_equal(b["state"][fs], c["state"][fs])
        assert np.array_equal(np.delete(b["state"], fs, 0), np.delete(a["state"], fs, 0))
        off.e.tracks_set_state(torch.as_tensor(b["state"]).cuda(), first=0)
        simt.e.tracks_set_state(torch.as_tensor(b["state"]).cuda(), first=0)


def test_many_flagged_items_take_every_grid_stride_loop_round(setup):
    """The counted fp32 kernels stride over the flagged items with grids of about one wave: at the default 1024-track chunk, 700
    flagged items in the first chunk and 76 in the second give every CTA of every counted kernel several items (blocks and head: one CTA
    per SM; crop + conv1: 37 items per round; conv4 and the scatter: 592)."""
    cfg, sd, frames, _ = setup
    n = 1100
    rng = np.random.default_rng(13)
    boxes = np.stack([rng.uniform(230, 380, n), rng.uniform(150, 260, n), rng.uniform(30, 50, n), rng.uniform(30, 50, n)], 1)
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    off, on, simt = (Run(_engine(cfg, sd, "tcgen05", max_tracks=n, chunk=0), frames, boxes),
                     Run(_engine(cfg, sd, "tcgen05", True, counter, max_tracks=n, chunk=0), frames, boxes),
                     Run(_engine(cfg, sd, "simt", max_tracks=n, chunk=0), frames, boxes))
    idx = np.array([1 if (i < 1024 and i % 3 != 0) or i >= 1024 else 0 for i in range(n)])
    a, b, c = off.step(idx), on.step(idx), simt.step(idx)
    flagged = a["detail"][:, 6] == RANGE
    assert flagged[:1024].sum() > 592 and flagged[1024:].sum() > 37 and not flagged.all(), (flagged[:1024].sum(), flagged[1024:].sum())
    _same(b, a, ~flagged, "unflagged vs fallback off")
    _same(b, c, flagged, "recomputed vs simt")
    assert (b["detail"][:, 6] == 0).all()
    assert np.array_equal(b["state"][flagged], c["state"][flagged]) and np.array_equal(b["state"][~flagged], a["state"][~flagged])
    assert int(counter.item()) == int(flagged.sum())


def test_update_state_zero_and_counter(setup):
    cfg, sd, frames, boxes = setup
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    on = Run(_engine(cfg, sd, "tcgen05", True, counter), frames, boxes)
    before = on.e.tracks_get_state(0, N).cpu().numpy()
    r = on.step(_frame_idx(), update_state=False)
    assert np.array_equal(r["state"], before)
    off = Run(_engine(cfg, sd, "tcgen05"), frames, boxes)
    flagged = off.step(_frame_idx(), update_state=False)["detail"][:, 6] == RANGE
    assert int(counter.item()) == int(flagged.sum()) > 0


def test_cuda_graph_replay_follows_the_frames(setup):
    cfg, sd, frames, boxes = setup
    on = Run(_engine(cfg, sd, "tcgen05", True), frames, boxes)
    off, simt = Run(_engine(cfg, sd, "tcgen05"), frames, boxes), Run(_engine(cfg, sd, "simt"), frames, boxes)
    idx = _frame_idx()
    offs, hw = on.offs(idx), _dev([[H, W]] * N, torch.int32, on.e.device)
    out_b = torch.zeros((N, 5), dtype=torch.float64, device="cuda")
    out_d = torch.zeros((N, 8), dtype=torch.float64, device="cuda")

    def launch():
        on.e.tracks_step(on.frames, offs, hw, first=0, n=N, out_boxes=out_b, out_detail=out_d, update_state=False, detail=True)
    launch()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    seen = []
    for swap in (False, True, False):
        src = frames[::-1] if swap else frames
        for r in (on, off, simt):
            r.frames.copy_(torch.from_numpy(np.ascontiguousarray(src)))
        g.replay()
        torch.cuda.synchronize()
        b = {"boxes": out_b.cpu().numpy(), "detail": out_d.cpu().numpy()}
        m = on.e.tracks_last_maps(0, N)
        b.update({k: v.cpu().numpy().reshape(N, -1) for k, v in m.items()})
        a, c = off.step(idx, False), simt.step(idx, False)
        flagged = a["detail"][:, 6] == RANGE
        assert flagged.any() and not flagged.all()
        _same(b, a, ~flagged, "replay: unflagged")
        _same(b, c, flagged, "replay: recomputed")
        seen.append(tuple(np.flatnonzero(flagged)))
    assert seen[0] != seen[1] and seen[0] == seen[2]


def test_nothing_flagged_same_bits_fixed_launches(setup):
    cfg, sd, frames, boxes = setup
    off, on = Run(_engine(cfg, sd, "tcgen05"), frames, boxes), Run(_engine(cfg, sd, "tcgen05", True), frames, boxes)
    flat = np.zeros(N, int)
    deltas = []
    for idx in (flat, _frame_idx()):
        l0, l1 = off.e.launch_count, on.e.launch_count
        a, b = off.step(idx, False), on.step(idx, False)
        deltas.append((on.e.launch_count - l1) - (off.e.launch_count - l0))
        if idx is flat:
            assert (a["detail"][:, 6] == 0).all()
            _same(b, a, np.ones(N, bool), "nothing flagged")
    chunks = -(-N // CHUNK)
    assert deltas[0] == deltas[1] == 1 + 5 * chunks + 3


def test_handle_kinds(setup):
    cfg, sd, frames, boxes = setup
    from test_generic_edges import CONFIGS, make_cfg
    from vittracker_b200._lib import VtError
    from vittracker_b200.engine import Engine
    C, heads, depth, hc, _ = CONFIGS["small"]
    g = Engine(make_cfg(C, heads, hc), max_tracks=4, blocks_impl="tcgen05", depth=depth)
    with pytest.raises(VtError) as ei:
        g.set_range_fallback(True)
    assert ei.value.code == -5
    plain, fb = Run(_engine(cfg, sd, "simt"), frames, boxes), Run(_engine(cfg, sd, "simt", True), frames, boxes)
    l0, l1 = plain.e.launch_count, fb.e.launch_count
    a, b = plain.step(_frame_idx()), fb.step(_frame_idx())
    _same(b, a, np.ones(N, bool), "simt handle")
    assert plain.e.launch_count - l0 == fb.e.launch_count - l1


def test_tracker_matches_simt_frame_by_frame(setup):
    cfg, sd, frames, boxes = setup
    from vittracker_b200 import get_tracker_class, parameters

    def tracker(**kw):
        p = parameters("vit_48_h32_noKD")
        p.state_dict = sd
        for k, v in kw.items():
            setattr(p, k, v)
        return get_tracker_class()(p, "synthetic")
    on, ref = tracker(range_fallback=True), tracker(blocks_impl="simt")
    box = [float(v) for v in boxes[0]]
    on.initialize(frames[0], {"init_bbox": box})
    ref.initialize(frames[0], {"init_bbox": box})
    rng = np.random.default_rng(9)
    for k in range(6):                                          # every frame is flagged; graph capture starts after two frames
        im = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        a, b = on.track(im), ref.track(im)
        assert a["target_bbox"] == b["target_bbox"], k
        assert float(a["confidence"]) == float(b["confidence"]), k


def test_run_sequences_keeps_flagged_sequences(setup, tmp_path):
    cfg, sd, frames, boxes = setup
    from vittracker_b200.sequences import Sequence, run_sequences
    rng = np.random.default_rng(21)
    seqs = []
    for i in range(4):
        noisy = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(4)]
        fr = [frames[0]] + (noisy if i % 2 == 0 else [frames[0]] * 4)
        seqs.append(Sequence(f"seq{i}", fr, [float(v) for v in boxes[i]]))
    dropped = run_sequences(seqs, cfg, sd, slots=4, results_dir=str(tmp_path / "tc"), read_workers=0)
    assert {s.name for s in seqs} - set(dropped) == {"seq0", "seq2"}      # the noisy sequences are flagged without the fallback
    kept = run_sequences(seqs, cfg, sd, slots=4, results_dir=str(tmp_path / "fb"), range_fallback=True, read_workers=0)
    ref = run_sequences(seqs, cfg, sd, slots=4, results_dir=str(tmp_path / "simt"), blocks_impl="simt", read_workers=0)
    assert set(kept) == set(ref) == {s.name for s in seqs}
    for s in seqs:
        assert (tmp_path / "fb" / f"{s.name}.txt").read_bytes() == (tmp_path / "simt" / f"{s.name}.txt").read_bytes(), s.name
