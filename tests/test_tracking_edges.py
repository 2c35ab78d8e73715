"""The tracking step (``vt_tracks_step``) at crop edges, across batch shapes and through the box decode.

The step's search branch reads the raw frame through per-track tap tables and, on the tensor-core paths, never writes
the crop out (vt_taps.cuh, vt_stem_fused.cu): it can only be observed through the maps and boxes the step returns.  This
file checks those outputs where a tap, a border bias, a byte alignment or a work split can be wrong:

1. Maps against float64.  A table of named geometries - five frame sizes, down to 3 x 5 px, each frame placed at byte
   offsets of 0..3 mod 4; crop sizes 1, 2, 16, 139, 256 (identity), 512 (exact 2x), 716 and 1601; overhang on every
   side and corner, crops larger than the frame, crops that cover column W-1 / row H-1 (which the reference drops),
   a single reachable column or row, x1 / y1 rounded half-to-even from .5 - is stepped once per implementation and
   weight set, and every track's full score, size and offset maps are compared with the oracle run in float64 on the
   oracle's exact crops.  For tcgen05 the float64 reference rounds q and k to fp16 before q k^T, as that kernel does
   by design (single-pass scores); against plain float64 its error is that rounding's, 6.7e-6 / 1.3e-5 / 3.9e-5
   (score / size / offset) on the one-pixel crop c1_last_reachable with default weights, which a CPU emulation of the
   single-pass scores reproduces to 2 %.  Maximum absolute error measured on an NVIDIA B200 (over both weight sets and
   all cases; two runs gave the same maxima) -> tolerance asserted:

       blocks          score              size               offset
       simt            7.6e-7 -> 2.5e-6   1.0e-6 -> 3e-6     3.5e-6 -> 1e-5
       tcgen05         1.5e-6 -> 4.5e-6   1.7e-6 -> 5e-6     4.8e-6 -> 1.5e-5
       tcgen05_3term   1.5e-6 -> 4.5e-6   1.3e-6 -> 4e-6     4.6e-6 -> 1.5e-5

2. The same bits in every batch shape.  1031 tracks (the table at all four alignments plus random boxes) give
   bit-identical maps, boxes and detail rows whatever the chunking (units of four bands, single-band tails), the
   order, a sub-range step or a batch of one; the batch-1 drop-in tracker (rectangle upload, CUDA graph, a frame
   buffer holding a previous frame's pixels) returns the same bits.

3. The decode is exact.  Box, confidence and detail row are recomputed from the device's own maps with the reference's
   post-processing (Hann window, cal_bbox, map_box_back, clip_box) and must match with tolerance 0, including
   all-tied and partly tied scores (first index wins), saturated sizes and frames narrower than the clip margin.
"""
import numpy as np
import pytest
import torch
from types import SimpleNamespace

from conftest import state_dict_from_npz
from oracle import vt_oracle as O

BLOCKS = ["simt", "tcgen05", "tcgen05_3term"]
# max |device - float64 reference| allowed per map; the module docstring gives the measurement behind each value
TOL = {"simt": {"score_map": 2.5e-6, "size_map": 3e-6, "offset_map": 1e-5},
       "tcgen05": {"score_map": 4.5e-6, "size_map": 5e-6, "offset_map": 1.5e-5},
       "tcgen05_3term": {"score_map": 4.5e-6, "size_map": 4e-6, "offset_map": 1.5e-5}}
MAPS = ("score_map", "size_map", "offset_map")
SLACK = 64                 # bytes after every frame in the device buffer: nothing may depend on reads past an allocation
CLAMP_HI = float(np.float32(1 - 1e-4))

FRAMES = {"hd": (720, 1280), "odd": (241, 321), "small": (48, 64), "micro": (3, 5), "uhd": (2160, 3840)}


def _box(c, x1, y1, factor):
    """A square box whose crop at ``factor`` has crop_sz ``c`` and corner (round(x1), round(y1)) (half-to-even)."""
    w = c / factor
    return [x1 + 0.5 * c - 0.5 * w, y1 + 0.5 * c - 0.5 * w, w, w]


# name: (frame, template crop (crop_sz, x1, y1), search crop (crop_sz, x1, y1)); W-1 / H-1 is the last column / row
CASES = {
    "c1_origin": ("hd", (1, 0, 0), (1, 0, 0)),
    "c1_last_reachable": ("hd", (2, 1278, 718), (1, 1278, 718)),
    "c2_bottom_right": ("hd", (1, 1278, 0), (2, 1278, 718)),
    "c16_single_col_left": ("hd", (16, -15, 300), (16, -15, 300)),
    "c16_single_row_top": ("hd", (2, 600, -1), (16, 600, -15)),
    "c139_single_col_right": ("hd", (139, 1278, 201.5), (139, 1278, 200.5)),
    "c139_single_row_bottom": ("hd", (64, 501.5, 718), (139, 500.5, 718)),
    "c256_identity_bottom_right": ("hd", (128, 1152, 592), (256, 1024, 464)),
    "c256_identity_top_left": ("hd", (256, -50, -60), (256, -100.5, -37.5)),
    "c512_exact_2x_top_right": ("hd", (512, 1100, -300), (512, 1000, -200)),
    "c716_bottom_left": ("hd", (358, -100, 500), (716, -300, 300)),
    "c716_bottom_right": ("hd", (716, 1000, 400), (716, 900.5, 200.5)),
    "odd_all_sides": ("odd", (360, -20, -60), (400, -40, -80)),
    "odd_top_left_half": ("odd", (70, -20.5, -10.5), (139, -60.5, -30.5)),
    "odd_bottom_right_half": ("odd", (100, 251.5, 171.5), (139, 250.5, 150.5)),
    "odd_interior_half": ("odd", (33, 101.5, 81.5), (139, 91.5, 51.5)),
    "small_all_sides": ("small", (100, -20, -30), (139, -40, -50)),
    "small_c1_last_col": ("small", (2, 0, 46), (1, 62, 0)),
    "small_c16_top_right": ("small", (16, 60, -10), (16, 55, -7)),
    "micro_all_sides": ("micro", (8, -2, -3), (16, -6, -7)),
    "micro_c2": ("micro", (1, 0, 0), (2, 3, 1)),
    "uhd_c1601_top_right": ("uhd", (801, 3200, -100), (1601, 3000, -400)),
    "uhd_c1601_bottom_left": ("uhd", (800, -300, 1500), (1601, -700.5, 1000.5)),
    "uhd_interior": ("uhd", (358, 1700, 900), (716, 1500, 800)),
}
NAMES = list(CASES)


def _case_boxes(name):
    fr, t, s = CASES[name]
    return fr, _box(*t, O.TEMPLATE_FACTOR), _box(*s, O.SEARCH_FACTOR)


def _frames():
    out = {}
    for i, (k, (H, W)) in enumerate(FRAMES.items()):
        # frame 0: template, 1: search, 2: a different frame of the same size (stale pixels for the drop-in tracker)
        out[k] = O.synth_frames(3, H, W, seed=300 + i, smooth=k in ("hd", "odd"))
    return out


class Tracks:
    """n tracks: frame size, template and search box, and where their frames sit in one device buffer."""

    def __init__(self, frames, specs):
        # specs: list of (label, frame name, byte alignment, template box, search box)
        self.labels = [s[0] for s in specs]
        self.fr = [s[1] for s in specs]
        self.hw = np.array([FRAMES[f] for f in self.fr], dtype=np.int32)
        self.tbox = np.array([s[3] for s in specs], dtype=np.float64)
        self.sbox = np.array([s[4] for s in specs], dtype=np.float64)
        chunks, pos, where = [], 0, {}
        for _, f, mis, _, _ in specs:
            if (f, mis) in where:
                continue
            pos = (pos + 3) // 4 * 4 + mis
            offs = []
            for k in range(3):
                a = frames[f][k].reshape(-1)
                chunks.append((pos, a))
                offs.append(pos)
                pos += a.size + SLACK
            where[(f, mis)] = offs
        buf = np.zeros(pos, dtype=np.uint8)
        for p, a in chunks:
            buf[p:p + a.size] = a
        self.buf = buf
        self.off = np.array([where[(s[1], s[2])] for s in specs], dtype=np.int64)      # [n, 3]
        self.frames = frames
        self.n = len(specs)

    def frame(self, i, k):
        return self.frames[self.fr[i]][k]

    def device(self, dev):
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        return SimpleNamespace(buf=t(self.buf), off=[t(self.off[:, k]) for k in range(3)], hw=t(self.hw),
                               tbox=t(self.tbox), sbox=t(self.sbox))


def _table_specs(rotate=0):
    return [(nm, CASES[nm][0], (i + rotate) % 4, *_case_boxes(nm)[1:]) for i, nm in enumerate(NAMES)]


@pytest.fixture(scope="module")
def frames():
    return _frames()


@pytest.fixture(scope="module")
def table(frames):
    return Tracks(frames, _table_specs())


@pytest.fixture(scope="module")
def stress_sd(golden_model):
    return state_dict_from_npz(golden_model)


def _weights(which, stress_sd):
    return stress_sd if which == "stress" else O.make_state_dict(seed=0)


@pytest.fixture(scope="module")
def cfg():
    from vittracker_b200 import load_cfg
    return load_cfg()


# ------------------------------------------------------------------------------------------------
# float64 reference and the exact decode
# ------------------------------------------------------------------------------------------------
def _crops(tr):
    z = torch.cat([O.preprocess(O.sample_target_spec(tr.frame(i, 0), list(tr.tbox[i]), O.TEMPLATE_FACTOR, O.TEMPLATE_SIZE)[0])
                   for i in range(tr.n)])
    x = torch.cat([O.preprocess(O.sample_target_spec(tr.frame(i, 1), list(tr.sbox[i]), O.SEARCH_FACTOR, O.SEARCH_SIZE)[0])
                   for i in range(tr.n)])
    return z, x


class Model64(O.OracleModel):
    """The oracle in float64.  ``fp16_scores``: q (scaled) and k are rounded to fp16 before q k^T - the one rounding the
    tcgen05 blocks make by design (vt_block_tc.cu: single-pass scores); everything else stays float64."""

    def __init__(self, sd, fp16_scores=False):
        super().__init__(sd)
        self.sd = {k: v.double() if v.is_floating_point() else v for k, v in self.sd.items()}
        self.fp16_scores = fp16_scores

    def block(self, x, b):
        if not self.fp16_scores:
            return super().block(x, b)
        p = f"blocks.{b}"
        C = self.C
        h = torch.nn.functional.layer_norm(x, (C,), self.sd[f"{p}.norm1.weight"], self.sd[f"{p}.norm1.bias"], O.LN_EPS)
        qkv = torch.nn.functional.linear(h, self.sd[f"{p}.attn.qkv.weight"], self.sd[f"{p}.attn.qkv.bias"])
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        f16 = lambda t: t.half().double()
        attn = (f16(q * (C ** -0.5)) @ f16(k).transpose(-2, -1)).softmax(dim=-1)
        x = x + torch.nn.functional.linear(attn @ v, self.sd[f"{p}.attn.proj.weight"], self.sd[f"{p}.attn.proj.bias"])
        h = torch.nn.functional.layer_norm(x, (C,), self.sd[f"{p}.norm2.weight"], self.sd[f"{p}.norm2.bias"], O.LN_EPS)
        h = torch.nn.functional.gelu(torch.nn.functional.linear(h, self.sd[f"{p}.mlp.fc1.weight"], self.sd[f"{p}.mlp.fc1.bias"]))
        return x + torch.nn.functional.linear(h, self.sd[f"{p}.mlp.fc2.weight"], self.sd[f"{p}.mlp.fc2.bias"])


def oracle64(sd, tr, fp16_scores=False):
    """The oracle's maps in float64 on the oracle's exact crops (the reference's fp32 normalised inputs)."""
    z, x = _crops(tr)
    return Model64(sd, fp16_scores).forward(z.double(), x.double())


_FEAT = SimpleNamespace(feat_sz=O.FEAT_SZ)


def exact_decode(score, size, off, state, H, W):
    """Vit_dist.track's post-processing (vit_dist.py:103-111,147-156) on one track's maps and search state:
    returns the (out_boxes row, out_detail row) the step must produce, bit for bit."""
    score = torch.as_tensor(score, dtype=torch.float32).reshape(1, 1, 16, 16)
    size = torch.as_tensor(size, dtype=torch.float32).reshape(1, 2, 16, 16)
    off = torch.as_tensor(off, dtype=torch.float32).reshape(1, 2, 16, 16)
    state = [float(v) for v in state]
    _, _, _, rf = O.crop_geometry(state, O.SEARCH_FACTOR, O.SEARCH_SIZE)
    resp = O.hann2d(O.FEAT_SZ, O.FEAT_SZ) * score
    pred_boxes = O.OracleModel.cal_bbox(_FEAT, resp, size, off).view(-1, 4)
    pred_box = (pred_boxes.mean(dim=0) * O.SEARCH_SIZE / rf).tolist()
    box = O.clip_box(O.map_box_back(state, pred_box, rf), H, W, margin=10)
    win_max, idx = torch.max(resp.flatten(1), dim=1)
    return [*box, float(score.max())], [*pred_box, rf, float(idx), 0.0, float(win_max)]


def assert_decode_exact(maps, out, det, tr, rows=None, tag=""):
    rows = range(tr.n) if rows is None else rows
    for j, i in enumerate(rows):
        H, W = (int(v) for v in tr.hw[i])
        want_b, want_d = exact_decode(maps["score_map"][j], maps["size_map"][j], maps["offset_map"][j], tr.sbox[i], H, W)
        assert np.array_equal(out[j], np.array(want_b)), (tag, tr.labels[i], out[j].tolist(), want_b)
        assert np.array_equal(det[j], np.array(want_d)), (tag, tr.labels[i], det[j].tolist(), want_d)


# ------------------------------------------------------------------------------------------------
# CPU self-checks of the pieces above
# ------------------------------------------------------------------------------------------------
def test_geometry_table_is_in_domain_and_spec_matches_opencv(frames):
    halves = set()
    for nm in NAMES:
        fr, tb, sb = _case_boxes(nm)
        H, W = FRAMES[fr]
        for box, (c, x1, y1), factor, S in ((tb, CASES[nm][1], O.TEMPLATE_FACTOR, O.TEMPLATE_SIZE),
                                            (sb, CASES[nm][2], O.SEARCH_FACTOR, O.SEARCH_SIZE)):
            assert O.crop_in_domain(box, factor, H, W), (nm, factor)
            assert O.crop_geometry(box, factor, S)[:3] == (c, round(x1), round(y1)), (nm, factor)
            for v in (x1, y1):
                if v != int(v):
                    halves.add(int(np.floor(v)) % 2)
            for k in (0, 1):
                p, rf, m = O.sample_target_spec(frames[fr][k], box, factor, S)
                pc, rfc, mc = O.sample_target_cv(frames[fr][k], box, factor, S)
                assert np.array_equal(p, pc) and rf == rfc and np.array_equal(m, mc), (nm, factor, k)
    assert halves == {0, 1}, "x1 / y1 on .5 must round both ways"
    # the table reaches what it is meant to: the dropped last column / row, single reachable columns and rows, all four sides
    s = [CASES[nm][2] for nm in NAMES]
    hw = [FRAMES[CASES[nm][0]] for nm in NAMES]
    assert any(round(x1) + c >= W for (c, x1, _), (_, W) in zip(s, hw))
    assert any(round(y1) + c >= H for (c, _, y1), (H, _) in zip(s, hw))
    assert any(round(x1) + c == 1 for c, x1, _ in s) and any(round(x1) == W - 2 for (c, x1, _), (_, W) in zip(s, hw))
    assert any(round(y1) + c == 1 for c, _, y1 in s) and any(round(y1) == H - 2 for (c, _, y1), (H, _) in zip(s, hw))
    assert any(x1 < 0 and y1 < 0 and x1 + c > W and y1 + c > H for (c, x1, y1), (H, W) in zip(s, hw))
    assert {c for c, _, _ in s} >= {1, 2, 16, 139, 256, 512, 716, 1601}


def test_buffer_places_frames_at_every_alignment_with_slack(table):
    assert sorted({int(o) % 4 for o in table.off.reshape(-1)}) == [0, 1, 2, 3]
    ends = sorted((int(o), int(o) + int(np.prod(table.hw[i])) * 3) for i in range(table.n) for o in table.off[i])
    for (a, e), (b, _) in zip(ends, ends[1:]):
        assert a == b or e + SLACK <= b
    assert ends[-1][1] + SLACK <= table.buf.size
    for i in range(table.n):
        for k in range(3):
            o = int(table.off[i, k])
            assert np.array_equal(table.buf[o:o + table.frame(i, k).size], table.frame(i, k).reshape(-1))


@pytest.mark.parametrize("weights", ["stress", "default"])
def test_exact_decode_reproduces_oracle_tracker(table, stress_sd, weights):
    model = O.OracleModel(_weights(weights, stress_sd))
    for i in range(table.n):
        trk = O.OracleTracker(model)
        trk.initialize(table.frame(i, 0), {"init_bbox": list(table.tbox[i])})
        trk.state = [float(v) for v in table.sbox[i]]
        want = trk.track(table.frame(i, 1), {})
        out = trk.last["out"]
        H, W = (int(v) for v in table.hw[i])
        b, d = exact_decode(out["score_map"], out["size_map"], out["offset_map"], table.sbox[i], H, W)
        assert b[:4] == want["target_bbox"] and b[4] == float(want["confidence"]), table.labels[i]
        assert d[5] == int(trk.last["response"].flatten().argmax()) and d[4] == trk.last["resize_factor"]


def test_float64_oracle_agrees_with_fp32_oracle(table, stress_sd):
    sd = _weights("stress", stress_sd)
    want = oracle64(sd, table)
    z, x = _crops(table)
    got = O.OracleModel(sd).forward(z, x)
    for k in MAPS:
        assert want[k].dtype == torch.float64
        assert float((got[k].double() - want[k]).abs().max()) < 1e-5, k


# ------------------------------------------------------------------------------------------------
# 1. maps against float64 at the edges
# ------------------------------------------------------------------------------------------------
def _step(engine, d, n, first=0, rows=None):
    """tracks_init on frame 0 with the template boxes, state := search boxes, one step on frame 1 (state kept)."""
    sl = slice(None) if rows is None else rows
    off0, off1, hw = d.off[0][sl].contiguous(), d.off[1][sl].contiguous(), d.hw[sl].contiguous()
    st = engine.tracks_init(d.buf, off0, hw, d.tbox[sl].contiguous(), first=first)
    assert st.cpu().tolist() == [0] * n
    engine.tracks_set_state(d.sbox[sl].contiguous(), first=first)
    out, det = engine.tracks_step(d.buf, off1, hw, first=first, n=n, update_state=False, detail=True)
    maps = engine.tracks_last_maps(first, n)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in maps.items()}, out.cpu().numpy(), det.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["stress", "default"])
@pytest.mark.parametrize("blocks", BLOCKS)
def test_maps_against_float64_at_edges(cfg, table, stress_sd, blocks, weights):
    from vittracker_b200.engine import Engine
    sd = _weights(weights, stress_sd)
    e = Engine(cfg, max_tracks=table.n, blocks_impl=blocks)
    e.load_state_dict(sd)
    maps, out, det = _step(e, table.device(e.device), table.n)
    want = oracle64(sd, table, fp16_scores=(blocks == "tcgen05"))
    report = {}
    for k in MAPS:
        err = np.abs(maps[k].astype(np.float64) - want[k].numpy()).reshape(table.n, -1).max(1)
        i = int(err.argmax())
        report[k] = (float(err[i]), table.labels[i])
    print(f"max |err| vs float64 [{blocks}, {weights}]:", report)
    for k in MAPS:
        assert report[k][0] <= TOL[blocks][k], (blocks, weights, k, report[k])
    assert_decode_exact(maps, out, det, table, tag=blocks)
    # W - 10 < 0 and H - 10 < 0: clip_box pins the box to (W - 10, H - 10, 10, 10) whatever the prediction
    i = NAMES.index("micro_all_sides")
    assert out[i, :4].tolist() == [-5.0, -7.0, 10.0, 10.0]


# ------------------------------------------------------------------------------------------------
# 2. the same bits in every batch shape
# ------------------------------------------------------------------------------------------------
N_BATCH = 1031


@pytest.fixture(scope="module")
def batch(frames):
    specs = []
    for r in range(4):                                   # the table at all four byte alignments
        specs += [(f"{nm}@{(i + r) % 4}", fr, mis, tb, sb) for i, (nm, fr, mis, tb, sb) in enumerate(_table_specs(r))]
    m = N_BATCH - len(specs)
    H, W = FRAMES["hd"]
    tb, sb = O.synth_boxes(m, H, W, seed=401), O.synth_boxes(m, H, W, seed=402)
    specs += [(f"synth{i}", "hd", i % 4, list(tb[i]), list(sb[i])) for i in range(m)]
    return Tracks(frames, specs)


_BASE = {}


def _baseline(cfg, batch, sd, blocks):
    """One engine with max_tracks = chunk_tracks = 1031 (units of four bands, a single-band tail)."""
    if blocks not in _BASE:
        from vittracker_b200.engine import Engine
        e = Engine(cfg, max_tracks=N_BATCH, chunk_tracks=N_BATCH, blocks_impl=blocks)
        e.load_state_dict(sd)
        d = batch.device(e.device)
        _BASE[blocks] = (e, d, _step(e, d, N_BATCH))
    return _BASE[blocks]


def _same(got, want, rows, what):
    gm, go, gd = got
    wm, wo, wd = want
    bad = [i for j, i in enumerate(rows)
           if not (all(np.array_equal(gm[k][j], wm[k][i]) for k in MAPS) and np.array_equal(go[j], wo[i]) and np.array_equal(gd[j], wd[i]))]
    assert not bad, f"{what}: {len(bad)} tracks differ from the baseline, first {bad[:5]}"


@pytest.mark.gpu
@pytest.mark.parametrize("blocks,chunks", [("tcgen05", (256, 97)), ("simt", (97,))])
def test_bits_identical_across_batch_shapes(cfg, batch, stress_sd, blocks, chunks):
    from vittracker_b200.engine import Engine
    e, d, base = _baseline(cfg, batch, stress_sd, blocks)
    n = N_BATCH
    assert_decode_exact(*base, batch, tag=blocks)
    # one geometry at four byte alignments: the frame's placement changes no bit
    k = len(NAMES)
    for r in (1, 2, 3):
        got = ({m: v[k * r:k * (r + 1)] for m, v in base[0].items()}, base[1][k * r:k * (r + 1)], base[2][k * r:k * (r + 1)])
        _same(got, base, range(k), f"alignment {r} vs 0")
    for c in chunks:
        ec = Engine(cfg, max_tracks=n, chunk_tracks=c, blocks_impl=blocks)
        ec.load_state_dict(stress_sd)
        _same(_step(ec, d, n), base, range(n), f"chunk {c}")
        del ec
    # the batch reversed
    er = Engine(cfg, max_tracks=n, chunk_tracks=n, blocks_impl=blocks)
    er.load_state_dict(stress_sd)
    perm = torch.arange(n - 1, -1, -1, device=e.device)
    dr = SimpleNamespace(buf=d.buf, off=[o[perm].contiguous() for o in d.off], hw=d.hw[perm].contiguous(),
                         tbox=d.tbox[perm].contiguous(), sbox=d.sbox[perm].contiguous())
    _same(_step(er, dr, n), base, list(range(n - 1, -1, -1)), "reversed")
    del er
    # a sub-range step (first > 0) of the baseline engine, then every table track alone (one track over all its CTAs)
    lo, m = 333, 500
    sub = slice(lo, lo + m)
    out, det = e.tracks_step(d.buf, d.off[1][sub].contiguous(), d.hw[sub].contiguous(), first=lo, n=m, update_state=False, detail=True)
    maps = {k: v.cpu().numpy() for k, v in e.tracks_last_maps(lo, m).items()}
    _same((maps, out.cpu().numpy(), det.cpu().numpy()), base, range(lo, lo + m), "sub-range")
    for i in range(len(NAMES)):
        out, det = e.tracks_step(d.buf, d.off[1][i:i + 1].contiguous(), d.hw[i:i + 1].contiguous(), first=i, n=1,
                                 update_state=False, detail=True)
        maps = {k: v.cpu().numpy() for k, v in e.tracks_last_maps(i, 1).items()}
        _same((maps, out.cpu().numpy(), det.cpu().numpy()), base, [i], f"alone: {NAMES[i]}")


@pytest.mark.gpu
@pytest.mark.parametrize("blocks", ["tcgen05", "simt"])
def test_dropin_tracker_matches_batched_bits(cfg, batch, stress_sd, blocks):
    from vittracker_b200 import get_tracker_class, parameters
    _, _, (bm, bo, bd) = _baseline(cfg, batch, stress_sd, blocks)
    params = parameters("vit_48_h32_noKD")
    params.state_dict = stress_sd
    params.blocks_impl = blocks
    trk = get_tracker_class()(params, "synthetic")
    # cases grouped by frame size, so that the frame buffer is reused (and the step replayed from its CUDA graph)
    order = sorted(range(len(NAMES)), key=lambda i: batch.fr[i])
    for i in order:
        trk.initialize(batch.frame(i, 0), {"init_bbox": list(batch.tbox[i])})
        trk.state = [float(v) for v in batch.sbox[i]]
        trk.track(batch.frame(i, 2), {})                # leaves another frame's pixels in the device buffer
        trk.state = [float(v) for v in batch.sbox[i]]
        got = trk.track(batch.frame(i, 1), {})
        assert got["target_bbox"] == bo[i, :4].tolist(), (NAMES[i], got["target_bbox"], bo[i, :4].tolist())
        assert float(got["confidence"]) == float(np.float32(bo[i, 4])) == bo[i, 4], NAMES[i]
        ld = trk.last_detail
        assert (ld["argmax"], ld["resize_factor"], ld["window_max"]) == (int(bd[i, 5]), bd[i, 4], bd[i, 7]), NAMES[i]
        assert ld["device_box"] == bo[i, :4].tolist(), NAMES[i]
        maps = trk.engine.tracks_last_maps(0, 1)
        for k in MAPS:
            assert np.array_equal(maps[k].cpu().numpy()[0], bm[k][i]), (NAMES[i], k)
    assert trk._graph is not None, "the drop-in tracker never replayed a CUDA graph"


# ------------------------------------------------------------------------------------------------
# 3. exact decode: ties, clamps, margins
# ------------------------------------------------------------------------------------------------
# conv5_ctr.bias for which part of each map saturates at 1 - 1e-4 and part does not (default weights, seed 0)
PARTIAL_CTR_BIAS = 9.0

SATURATIONS = {"ctr+30": {"box_head.conv5_ctr.bias": 30.0}, "ctr_partial": {"box_head.conv5_ctr.bias": PARTIAL_CTR_BIAS},
               "size+30": {"box_head.conv5_size.bias": 30.0}, "size-30": {"box_head.conv5_size.bias": -30.0}}


def _saturated_sd(kind, **shape_kw):
    sd = O.make_state_dict(seed=0, **shape_kw)
    for k, v in SATURATIONS[kind].items():
        sd[k] = torch.full_like(sd[k], v)
    return sd


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(SATURATIONS))
@pytest.mark.parametrize("blocks", ["tcgen05", "simt"])
def test_decode_exact_on_saturated_maps(cfg, table, blocks, kind):
    from vittracker_b200.engine import Engine
    sd = _saturated_sd(kind)
    e = Engine(cfg, max_tracks=table.n, blocks_impl=blocks)
    e.load_state_dict(sd)
    maps, out, det = _step(e, table.device(e.device), table.n)
    assert_decode_exact(maps, out, det, table, tag=f"{blocks} {kind}")
    score = maps["score_map"].reshape(table.n, -1)
    if kind == "ctr+30":
        # every score clamps to fp32(1 - 1e-4): the windowed response ties four ways at the centre and the first index wins
        assert (score == np.float32(CLAMP_HI)).all()
        assert (det[:, 5] == 119).all() and (out[:, 4] == CLAMP_HI).all()
        assert (det[:, 7] == float(O.hann2d(16, 16).flatten()[119] * np.float32(CLAMP_HI))).all()
    elif kind == "ctr_partial":
        clamped = (score == np.float32(CLAMP_HI)).sum(1)
        assert ((clamped > 0) & (clamped < 256)).sum() >= table.n // 2, clamped.tolist()
    elif kind == "size+30":
        assert (maps["size_map"] == np.float32(CLAMP_HI)).all()
    else:
        assert (maps["size_map"] == np.float32(1e-4)).all()
        assert (out[:, 2] == 10.0).all() and (out[:, 3] == 10.0).all()      # clip_box widens to the margin


@pytest.mark.gpu
def test_forward_all_tied_scores_take_index_zero(cfg, table):
    from vittracker_b200.engine import Engine
    e = Engine(cfg, max_tracks=8, blocks_impl="tcgen05")
    e.load_state_dict(_saturated_sd("ctr+30"))
    rows = [NAMES.index(nm) for nm in ("c256_identity_top_left", "odd_all_sides", "micro_all_sides", "uhd_c1601_top_right")]
    z, x = _crops(table)
    got = e.forward(z[rows], x[rows])
    g = {k: v.cpu() for k, v in got.items()}
    assert (g["score_map"] == np.float32(CLAMP_HI)).all()
    want = O.OracleModel.cal_bbox(_FEAT, g["score_map"], g["size_map"], g["offset_map"]).view(-1, 1, 4)
    assert torch.equal(g["pred_boxes"], want)
    at0 = torch.stack([g["offset_map"][:, 0, 0, 0] / 16, g["offset_map"][:, 1, 0, 0] / 16,
                       g["size_map"][:, 0, 0, 0], g["size_map"][:, 1, 0, 0]], 1)
    assert torch.equal(g["pred_boxes"].view(-1, 4), at0)


@pytest.mark.gpu
def test_generic_path_decode_on_saturated_scores(table):
    """The generic-configuration path (vt_generic.cu) decodes through the same arg-max and box code: all-tied scores."""
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    C, heads, depth, hc = 96, 3, 2, 64                   # the "small" configuration of test_gpu_generic.py
    cfg = load_cfg()
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS, cfg.MODEL.BACKBONE.DEPTH = C, heads, depth
    cfg.MODEL.HEAD.NUM_CHANNELS = hc
    e = Engine(cfg, max_tracks=table.n, depth=depth)
    e.load_state_dict(_saturated_sd("ctr+30", C=C, depth=depth, head_ch=hc))
    maps, out, det = _step(e, table.device(e.device), table.n)
    assert (maps["score_map"] == np.float32(CLAMP_HI)).all()
    assert (det[:, 5] == 119).all() and (out[:, 4] == CLAMP_HI).all()
    assert_decode_exact(maps, out, det, table, tag="generic")
