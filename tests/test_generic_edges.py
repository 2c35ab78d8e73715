"""The generic-configuration path (vt_generic.cu) on every GEMM route, against float64.

Every vit_dist member other than vit_48_h32 runs through vt_generic.cu, which picks a kernel per layer from the layer's shape:
``sgemm_kernel`` (fp32, NT or NN), ``gemm_tc_kernel`` (fp16 hi / lo operand splits, fp32 or split-image output),
``gemm_img_kernel`` (pre-split operand images; fp32, image, ``c_group`` rows with the ``rmod`` positional embedding, residual),
three forms of im2col, two LayerNorms and the fp32-rows -> image conversion of P V.  This file checks that path:

1. A route table.  ``routes()`` restates the selection rules of vt_generic.cu in Python (``gemm_tc_ok``, ``use_img``,
   ``fp32_only``, ``ci % 32`` for the convolution images, ``cn % 16`` and ``3 hc % 16`` in the head) and gives, for each
   configuration of CONFIGS, layer -> (kernel, NT / NN or form, activation, output).  A CPU test asserts that CONFIGS reach
   every route and shape edge that any accepted configuration (C up to 1024, every head count, head width up to 512, both
   block implementations) can reach, and lists them.  Two pairs do not exist in the code: ``sgemm`` never takes an ``rmod``
   residual (the stem's last convolution on ``sgemm`` adds the positional embedding per track, batch stride 0) and
   ``gemm_tc_kernel`` writes a split image only for P V, which is NN.

2. Every stage against float64.  ``Engine.forward(z, x, taps=True)`` on three oracle crops (one interior, two with zero
   padding on two sides each) per configuration; each tap (tokens after stem + positional embedding, after every block,
   after the final LayerNorm) is measured as max |err| / RMS of the float64 tap, then the maps and boxes as max |err|.
   Measured on an NVIDIA B200 at a 1000 W power limit (two runs gave the same values) -> asserted (about 3x):

       config        stem tap            block taps          score               size                offset              boxes
       odd           1.5e-6 -> 5e-6      1.6e-6 -> 5e-6      2.4e-7 -> 7.5e-7    5.2e-7 -> 1.5e-6    1.7e-6 -> 5e-6      2.3e-7 -> 7e-7
       small         2.2e-6 -> 7e-6      5.1e-6 -> 1.5e-5    1.2e-6 -> 4e-6      1.2e-6 -> 4e-6      6.7e-6 -> 2e-5      5.2e-7 -> 1.5e-6
       small_hd96    2.2e-6 -> 7e-6      1.0e-5 -> 3e-5      9.5e-7 -> 3e-6      8.5e-7 -> 2.5e-6    3.2e-6 -> 1e-5      2.7e-7 -> 8e-7
       img           4.9e-6 -> 1.5e-5    1.1e-5 -> 3.3e-5    1.4e-6 -> 4.5e-6    2.0e-6 -> 6e-6      9.0e-6 -> 2.7e-5    1.4e-6 -> 4e-6
       img_hd32      4.9e-6 -> 1.5e-5    6.2e-6 -> 2e-5      1.5e-6 -> 4.5e-6    2.0e-6 -> 6e-6      9.7e-6 -> 3e-5      1.3e-6 -> 4e-6
       img_hc24      4.9e-6 -> 1.5e-5    9.1e-6 -> 2.7e-5    1.3e-6 -> 4e-6      1.3e-6 -> 4e-6      4.1e-6 -> 1.2e-5    4.8e-7 -> 1.5e-6
       img_hd192     1.7e-5 -> 5e-5      2.0e-5 -> 6e-5      3.0e-6 -> 9e-6      2.9e-6 -> 9e-6      1.8e-5 -> 5.5e-5    8.3e-7 -> 2.5e-6
       img_hd256     1.0e-5 -> 3e-5      1.6e-5 -> 5e-5      3.1e-6 -> 9.5e-6    1.9e-6 -> 6e-6      1.2e-5 -> 3.6e-5    9.7e-7 -> 3e-6
       widest        3.2e-5 -> 1e-4      4.7e-5 -> 1.4e-4    9.8e-6 -> 3e-5      1.2e-5 -> 3.7e-5    2.8e-5 -> 8.5e-5    7.2e-6 -> 2.2e-5
       small_simt    1.0e-6 -> 3e-6      2.1e-6 -> 6e-6      4.7e-7 -> 1.5e-6    6.8e-7 -> 2e-6      2.3e-6 -> 7e-6      1.1e-7 -> 3.5e-7
       widest_simt   4.8e-6 -> 1.5e-5    6.6e-6 -> 2e-5      1.1e-6 -> 3e-6      1.3e-6 -> 4e-6      3.8e-6 -> 1.2e-5    4.8e-7 -> 1.5e-6

   A dropped hi / lo split term (profiles/experiments/generic_edges_mutants.diff) gives 4e-4 to 1.2e-3 on the taps where
   the Linear layers or the convolutions take the broken kernel, 25 to 100x above these bounds; where only the attention
   products take it (gemm_tc_kernel under ``img``), 6e-5, 2x above.  Under ``widest`` that case stays inside the wider
   bound: the other configurations catch it.  The GPU tests of this file take 10 s on a B200.

3. The tracking step.  The crop-edge table of test_tracking_edges.py is stepped through ``small`` (Linear layers on
   ``gemm_tc_kernel``) and ``img`` (``gemm_img_kernel``): maps against float64, boxes and detail rows decoded exactly.  300
   tracks of ``odd`` give the same bits with chunk_tracks 1, 7, 256 and 300, in reverse order and in a sub-range step (256
   tracks put 65536 row tiles in stem conv1's grid: more than gridDim.y allows in one launch).

4. The range guard.  Weights scaled until an fp16 operand overflows: under tcgen05 every track is flagged
   VT_TRACK_NUMERIC_RANGE with NaN maps; under simt (fp32 on every GEMM) none is, and the maps match float64.
"""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import vt_oracle as O
from test_tracking_edges import FRAMES, NAMES, Tracks, _crops, _frames, _same, _step, _table_specs, assert_decode_exact

KN = 320                        # tokens per track: 64 template + 256 search
N_FWD = 3                       # tracks of the forward test: 960 token rows, 7.5 row tiles of 128

# name: (C, heads, depth, head channels, blocks_impl)
CONFIGS = {
    "odd": (40, 5, 1, 24, "tcgen05"),             # all but head conv1 on sgemm; K = 40 and 27 are not multiples of the 16-wide k-tile
    "small": (96, 3, 2, 64, "tcgen05"),           # Linear layers on gemm_tc, scores and P V on sgemm
    "small_hd96": (96, 1, 1, 64, "tcgen05"),      # scores (NT) and P V (NN) on gemm_tc, fp32 out
    "img": (128, 2, 2, 64, "tcgen05"),            # split-image route; P V on gemm_tc with an image epilogue
    "img_hd32": (128, 4, 1, 64, "tcgen05"),       # split-image route with head dim 32: P V on sgemm, then the image
    "img_hc24": (128, 2, 1, 24, "tcgen05"),       # head conv1 with 72 outputs: not a multiple of gemm_img's 16 columns
    "img_hd192": (384, 2, 1, 32, "tcgen05"),      # ragged N tile (192) on gemm_tc, image epilogue at n0 = 128
    "img_hd256": (256, 1, 1, 32, "tcgen05"),      # image epilogue at n0 = 128, head dim 256
    "widest": (768, 12, 12, 256, "tcgen05"),
    "small_simt": (96, 3, 2, 64, "simt"),
    "widest_simt": (768, 12, 12, 256, "simt"),
}

# measured max (module docstring) x ~3; keys: "stem" / "blocks" taps (relative to the tap's RMS), maps and boxes (absolute)
TOL = {
    "odd": dict(stem=5e-6, blocks=5e-6, score_map=7.5e-7, size_map=1.5e-6, offset_map=5e-6, pred_boxes=7e-7),
    "small": dict(stem=7e-6, blocks=1.5e-5, score_map=4e-6, size_map=4e-6, offset_map=2e-5, pred_boxes=1.5e-6),
    "small_hd96": dict(stem=7e-6, blocks=3e-5, score_map=3e-6, size_map=2.5e-6, offset_map=1e-5, pred_boxes=8e-7),
    "img": dict(stem=1.5e-5, blocks=3.3e-5, score_map=4.5e-6, size_map=6e-6, offset_map=2.7e-5, pred_boxes=4e-6),
    "img_hd32": dict(stem=1.5e-5, blocks=2e-5, score_map=4.5e-6, size_map=6e-6, offset_map=3e-5, pred_boxes=4e-6),
    "img_hc24": dict(stem=1.5e-5, blocks=2.7e-5, score_map=4e-6, size_map=4e-6, offset_map=1.2e-5, pred_boxes=1.5e-6),
    "img_hd192": dict(stem=5e-5, blocks=6e-5, score_map=9e-6, size_map=9e-6, offset_map=5.5e-5, pred_boxes=2.5e-6),
    "img_hd256": dict(stem=3e-5, blocks=5e-5, score_map=9.5e-6, size_map=6e-6, offset_map=3.6e-5, pred_boxes=3e-6),
    "widest": dict(stem=1e-4, blocks=1.4e-4, score_map=3e-5, size_map=3.7e-5, offset_map=8.5e-5, pred_boxes=2.2e-5),
    "small_simt": dict(stem=3e-6, blocks=6e-6, score_map=1.5e-6, size_map=2e-6, offset_map=7e-6, pred_boxes=3.5e-7),
    "widest_simt": dict(stem=1.5e-5, blocks=2e-5, score_map=3e-6, size_map=4e-6, offset_map=1.2e-5, pred_boxes=1.5e-6),
}
MAPS = ("score_map", "size_map", "offset_map")


# ------------------------------------------------------------------------------------------------
# the selection rules of vt_generic.cu, restated
# ------------------------------------------------------------------------------------------------
def tc_ok(M, N, K, lda, strides=(), nn=False, ldb=None, bstrides=()):
    """gemm_tc_ok.  Every operand base is 16-byte aligned: workspace slots are 64-float multiples, weights 16-byte slots."""
    if not (K % 8 == 0 and K >= 64 and N >= 64 and M >= 128 and lda % 4 == 0 and all(s % 4 == 0 for s in strides)):
        return False
    return nn or (ldb % 4 == 0 and all(s % 4 == 0 for s in bstrides))


def routes(C, heads, depth, hc, impl, n=N_FWD):
    """layer -> (kernel, form, activation, output), and the shape edges each GEMM reaches, for one configuration.
    Every block takes the same routes, so block 0 stands for all."""
    fp32_only = impl == "simt"
    use_img = not fp32_only and C % 128 == 0
    hd = C // heads
    table, edges = {}, set()

    def gemm(layer, M, N, K, act, out, nn=False, lda=None, strides=(), ldb=None, bstrides=(), image=False):
        tc = not fp32_only and tc_ok(M, N, K, K if lda is None else lda, strides, nn, K if ldb is None else ldb, bstrides)
        if image and not (tc and hd % 8 == 0):
            table[layer] = ("sgemm", "NN", act, "fp32")
            table[layer + "/image"] = ("rows_img", "-", "none", "image")
            kern = "sgemm"
        else:
            kern = "gemm_tc" if tc else "sgemm"
            table[layer] = (kern, "NN" if nn else "NT", act, "image" if image else out)
        tm, tn, tk = (128, 128, 32) if kern == "gemm_tc" else (64, 64, 16)
        if M % tm:
            edges.add((kern, "ragged M"))
        if N % tn and N > tn:
            edges.add((kern, "ragged N"))
        if K % tk:
            edges.add((kern, "K % k-tile"))
        if kern == "gemm_tc" and image and N > 128:
            edges.add((kern, "image epilogue at n0 > 0"))

    def img_gemm(layer, M, N, K, act, out):
        table[layer] = ("gemm_img", "-", act, out)
        if M % 128:
            edges.add(("gemm_img", "ragged M"))

    ch = [3, C // 8, C // 4, C // 2, C]
    for S, tag in ((128, "z"), (256, "x")):
        H = S
        for l in range(4):
            Ho, K = H // 2, 9 * ch[l]
            name = f"stem{l + 1}_{tag}"
            if l > 0 and use_img and ch[l] % 32 == 0:
                table[name + "/im2col"] = ("im2col", "img", "-", "image")
                if l < 3:
                    img_gemm(name, n * Ho * Ho, ch[l + 1], K, "hardswish", "fp32")
                else:
                    img_gemm(name, n * Ho * Ho, C, K, "none", "c_group+rmod")
            else:
                table[name + "/im2col"] = ("im2col", "nchw" if l == 0 else "nhwc", "-", "fp32")
                if l < 3:
                    gemm(name, n * Ho * Ho, ch[l + 1], K, "hardswish", "fp32")
                else:           # one GEMM per track, the positional embedding as a residual with batch stride 0
                    gemm(name, Ho * Ho, C, K, "none", "residual", strides=(Ho * Ho * K,))
            H = Ho
    rows = n * KN
    qk = dict(lda=3 * C, strides=(KN * 3 * C, hd), ldb=3 * C, bstrides=(KN * 3 * C, hd))
    pv = dict(nn=True, lda=KN, strides=(heads * KN * KN, KN * KN))
    if use_img:
        table["ln1"] = ("layernorm", "img", "-", "image")
        img_gemm("qkv", rows, 3 * C, C, "none", "fp32")
        gemm("scores", KN, KN, hd, "none", "fp32", **qk)
        gemm("pv", KN, hd, KN, "none", "image", image=True, **pv)
        img_gemm("proj", rows, C, C, "none", "residual")
        img_gemm("fc1", rows, 4 * C, C, "gelu", "image")
        img_gemm("fc2", rows, C, 4 * C, "none", "residual")
    else:
        table["ln1"] = ("layernorm", "fp32", "-", "fp32")
        gemm("qkv", rows, 3 * C, C, "none", "fp32")
        gemm("scores", KN, KN, hd, "none", "fp32", **qk)
        gemm("pv", KN, hd, KN, "none", "fp32", **pv)
        gemm("proj", rows, C, C, "none", "residual")
        gemm("fc1", rows, 4 * C, C, "gelu", "fp32")
        gemm("fc2", rows, C, 4 * C, "none", "residual")
    table["norm"] = ("layernorm", "fp32", "-", "fp32")
    co = [C, hc, hc // 2, hc // 4, hc // 8]
    prow = n * 256
    if use_img and (3 * hc) % 16 == 0:
        table["head1/im2col"] = ("im2col", "img", "-", "image")
        img_gemm("head1", prow, 3 * hc, 9 * C, "relu", "fp32")
    else:
        table["head1/im2col"] = ("im2col", "nhwc", "-", "fp32")
        gemm("head1", prow, 3 * hc, 9 * C, "relu", "fp32")
    for l in range(1, 4):
        ci, cn = co[l], co[l + 1]
        if use_img and ci % 32 == 0 and cn % 16 == 0:
            table[f"head{l + 1}/im2col"] = ("im2col", "img", "-", "image")
            img_gemm(f"head{l + 1}", prow, cn, 9 * ci, "relu", "fp32")
        else:
            table[f"head{l + 1}/im2col"] = ("im2col", "nhwc", "-", "fp32")
            gemm(f"head{l + 1}", prow, cn, 9 * ci, "relu", "fp32")
    for t, outs in (("ctr", 1), ("offset", 2), ("size", 2)):
        gemm(f"head5_{t}", prow, outs, co[4], "none", "fp32", lda=3 * co[4])
    return table, edges


ROUTES = {name: routes(*c) for name, c in CONFIGS.items()}


def _accepted_configs():
    """vt_create's generic configurations in a grid wide enough to reach every rule's both sides."""
    for C in range(8, 1025, 8):
        for heads in (h for h in range(1, 33) if C % h == 0):
            for hc in range(8, 513, 8):
                for impl in ("tcgen05", "simt"):
                    yield C, heads, 1, hc, impl


def _union(items):
    r, e = set(), set()
    for t, ed in items:
        r |= set(t.values())
        e |= ed
    return r, e


def test_route_table_reaches_every_route_and_edge():
    got_r, got_e = _union(ROUTES.values())
    all_r, all_e = _union(routes(*c) for c in _accepted_configs())
    assert all_r - got_r == set(), sorted(all_r - got_r)
    assert all_e - got_e == set(), sorted(all_e - got_e)
    # the pairs named in the module docstring, written out
    want = {("sgemm", "NT", a, "fp32") for a in ("none", "hardswish", "relu", "gelu")} | {
        ("sgemm", "NT", "none", "residual"), ("sgemm", "NN", "none", "fp32"),
        *{("gemm_tc", "NT", a, "fp32") for a in ("none", "hardswish", "relu", "gelu")},
        ("gemm_tc", "NT", "none", "residual"), ("gemm_tc", "NN", "none", "fp32"), ("gemm_tc", "NN", "none", "image"),
        ("gemm_img", "-", "hardswish", "fp32"), ("gemm_img", "-", "none", "fp32"), ("gemm_img", "-", "relu", "fp32"),
        ("gemm_img", "-", "gelu", "image"), ("gemm_img", "-", "none", "c_group+rmod"), ("gemm_img", "-", "none", "residual"),
        ("im2col", "nchw", "-", "fp32"), ("im2col", "nhwc", "-", "fp32"), ("im2col", "img", "-", "image"),
        ("layernorm", "fp32", "-", "fp32"), ("layernorm", "img", "-", "image"), ("rows_img", "-", "none", "image")}
    assert want == all_r, (sorted(want - all_r), sorted(all_r - want))
    assert {("gemm_tc", "ragged M"), ("gemm_img", "ragged M"), ("gemm_tc", "ragged N"), ("gemm_tc", "image epilogue at n0 > 0"),
            ("sgemm", "K % k-tile"), ("gemm_tc", "K % k-tile")} <= got_e


def test_route_table_matches_the_named_cases():
    r = {k: v[0] for k, v in ROUTES.items()}
    assert {v[0] for k, v in r["odd"].items() if k != "head1"} == {"sgemm", "im2col", "layernorm"} and r["odd"]["head1"][0] == "gemm_tc"
    assert r["small"]["qkv"][0] == r["small"]["fc1"][0] == "gemm_tc" and r["small"]["scores"][0] == r["small"]["pv"][0] == "sgemm"
    assert r["small_hd96"]["scores"][:2] == ("gemm_tc", "NT") and r["small_hd96"]["pv"] == ("gemm_tc", "NN", "none", "fp32")
    assert r["img"]["pv"] == ("gemm_tc", "NN", "none", "image") and r["img"]["qkv"][0] == "gemm_img"
    assert r["img_hd32"]["pv"] == ("sgemm", "NN", "none", "fp32") and "pv/image" in r["img_hd32"]
    assert r["img_hc24"]["head1"][0] == "gemm_tc"
    for name in ("small_simt", "widest_simt"):        # fp32 everywhere
        assert {v[0] for v in r[name].values()} <= {"sgemm", "im2col", "layernorm"}, name
    assert ("sgemm", "K % k-tile") in ROUTES["odd"][1]


# ------------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------------
def make_cfg(C, heads, hc):
    from vittracker_b200 import load_cfg
    cfg = load_cfg()
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS = C, heads
    cfg.MODEL.HEAD.NUM_CHANNELS = hc
    return cfg


def model64(sd, depth, heads):
    m = O.OracleModel(sd, depth=depth, num_heads=heads)
    m.sd = {k: v.double() if v.is_floating_point() else v for k, v in m.sd.items()}
    return m


def make_sd(name, seed=41):
    C, heads, depth, hc, _ = CONFIGS[name]
    return O.make_state_dict(seed=seed, stress=True, C=C, depth=depth, head_ch=hc)


@pytest.fixture(scope="module")
def fwd_crops():
    """Three (template, search) crops: interior, overhanging top and left, overhanging bottom and right (zero padding)."""
    frames = O.synth_frames(2, 360, 640, seed=43, smooth=True)
    boxes = [[300.0, 150.0, 60.0, 40.0], [5.0, 5.0, 50.0, 50.0], [600.0, 330.0, 30.0, 25.0]]
    z = torch.cat([O.preprocess(O.sample_target_spec(frames[0], b, O.TEMPLATE_FACTOR, O.TEMPLATE_SIZE)[0]) for b in boxes])
    x = torch.cat([O.preprocess(O.sample_target_spec(frames[1], b, O.SEARCH_FACTOR, O.SEARCH_SIZE)[0]) for b in boxes])
    return z, x, boxes


def test_forward_crops_have_padding_on_two_sides(fwd_crops):
    _, _, boxes = fwd_crops
    pads = []
    for b in boxes:
        c, x1, y1, _ = O.crop_geometry(b, O.SEARCH_FACTOR, O.SEARCH_SIZE)
        pads.append((x1 < 0, y1 < 0, x1 + c > 639, y1 + c > 359))
    assert pads[0] == (False,) * 4 and pads[1] == (True, True, False, False) and pads[2] == (False, False, True, True)


def test_float64_oracle_agrees_with_fp32_oracle(fwd_crops):
    z, x, _ = fwd_crops
    for name in ("odd", "img_hd32"):
        C, heads, depth, hc, _ = CONFIGS[name]
        sd = make_sd(name)
        want = model64(sd, depth, heads).forward(z.double(), x.double())
        got = O.OracleModel(sd, depth=depth, num_heads=heads).forward(z, x)
        for k in MAPS:
            assert want[k].dtype == torch.float64
            assert float((got[k].double() - want[k]).abs().max()) < 1e-5, (name, k)


# ------------------------------------------------------------------------------------------------
# 2. every stage against float64
# ------------------------------------------------------------------------------------------------
def _tap_errors(got_taps, want_taps, depth):
    """max |err| / RMS(float64 tap) per tap: 'stem', 'block1'.., 'norm'."""
    keys = ["tokens0"] + [f"tokens{b + 1}" for b in range(depth)] + ["tokens_norm"]
    names = ["stem"] + [f"block{b + 1}" for b in range(depth)] + ["norm"]
    out = {}
    for i, (k, nm) in enumerate(zip(keys, names)):
        w = want_taps[k]
        g = got_taps[i].double().cpu()
        out[nm] = float((g - w).abs().max() / w.pow(2).mean().sqrt())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_forward_taps_and_maps_against_float64(fwd_crops, name):
    from vittracker_b200.engine import Engine
    C, heads, depth, hc, impl = CONFIGS[name]
    torch.set_num_threads(16)
    z, x, _ = fwd_crops
    sd = make_sd(name)
    taps64 = {}
    want = model64(sd, depth, heads).forward(z.double(), x.double(), taps=taps64)
    e = Engine(make_cfg(C, heads, hc), max_tracks=N_FWD, blocks_impl=impl, depth=depth)
    e.load_state_dict(sd)
    got = e.forward(z, x, taps=True)
    torch.cuda.synchronize()
    taps = _tap_errors(got["taps"], taps64, depth)
    maps = {k: float((got[k].double().cpu() - want[k]).abs().max()) for k in (*MAPS, "pred_boxes")}
    print(f"\n[{name}] taps max|err|/rms:", {k: f"{v:.2e}" for k, v in taps.items()}, "maps max|err|:", {k: f"{v:.2e}" for k, v in maps.items()})
    tol = TOL[name]
    for k, v in taps.items():
        assert v <= tol["stem" if k == "stem" else "blocks"], (name, k, v, taps)
    for k, v in maps.items():
        assert v <= tol[k], (name, k, v)


# ------------------------------------------------------------------------------------------------
# 3. the tracking step on the generic path
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def frames():
    return _frames()


@pytest.fixture(scope="module")
def table(frames):
    return Tracks(frames, _table_specs())


def _engine(name, n, chunk=0, sd=None, impl=None):
    from vittracker_b200.engine import Engine
    C, heads, depth, hc, impl0 = CONFIGS[name]
    e = Engine(make_cfg(C, heads, hc), max_tracks=n, chunk_tracks=chunk, blocks_impl=impl or impl0, depth=depth)
    e.load_state_dict(make_sd(name) if sd is None else sd)
    return e


def _maps64(name, tr, sd=None):
    C, heads, depth, hc, _ = CONFIGS[name]
    z, x = _crops(tr)
    return model64(make_sd(name) if sd is None else sd, depth, heads).forward(z.double(), x.double())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small", "img"])
def test_step_maps_against_float64_at_edges(table, name):
    torch.set_num_threads(16)
    e = _engine(name, table.n)
    maps, out, det = _step(e, table.device(e.device), table.n)
    want = _maps64(name, table)
    report = {}
    for k in MAPS:
        err = np.abs(maps[k].astype(np.float64) - want[k].numpy()).reshape(table.n, -1).max(1)
        i = int(err.argmax())
        report[k] = (float(err[i]), table.labels[i])
    print(f"\nstep max |err| vs float64 [{name}]:", report)
    for k in MAPS:
        assert report[k][0] <= TOL[name][k], (name, k, report[k])
    assert_decode_exact(maps, out, det, table, tag=name)


N_BITS = 300


@pytest.fixture(scope="module")
def bits_tracks(frames):
    specs = []
    for r in range(4):
        specs += [(f"{nm}@{(i + r) % 4}", fr, mis, tb, sb) for i, (nm, fr, mis, tb, sb) in enumerate(_table_specs(r))]
    m = N_BITS - len(specs)
    H, W = FRAMES["hd"]
    tb, sb = O.synth_boxes(m, H, W, seed=411), O.synth_boxes(m, H, W, seed=412)
    specs += [(f"synth{i}", "hd", i % 4, list(tb[i]), list(sb[i])) for i in range(m)]
    return Tracks(frames, specs)


@pytest.mark.gpu
def test_step_bits_identical_across_chunks_order_and_subrange(bits_tracks):
    """``odd``: the kernel route does not depend on the number of tracks, so no bit may either.  Chunk 256 and 300 put
    65536 and 76800 row tiles into stem conv1 of the search crop: the launch is split at gridDim.y's 65535."""
    n = N_BITS
    e = _engine("odd", n, chunk=n)
    d = bits_tracks.device(e.device)
    base = _step(e, d, n)
    assert np.isfinite(base[1]).all() and (base[2][:, 6] == 0).all()
    assert_decode_exact(*base, bits_tracks, tag="odd chunk 300")
    for c in (1, 7, 256):
        ec = _engine("odd", n, chunk=c)
        _same(_step(ec, d, n), base, range(n), f"chunk {c}")
        del ec
    perm = torch.arange(n - 1, -1, -1, device=e.device)
    dr = SimpleNamespace(buf=d.buf, off=[o[perm].contiguous() for o in d.off], hw=d.hw[perm].contiguous(),
                         tbox=d.tbox[perm].contiguous(), sbox=d.sbox[perm].contiguous())
    er = _engine("odd", n, chunk=256)
    _same(_step(er, dr, n), base, list(range(n - 1, -1, -1)), "reversed")
    del er
    lo, m = 37, 250
    sub = slice(lo, lo + m)
    out, det = e.tracks_step(d.buf, d.off[1][sub].contiguous(), d.hw[sub].contiguous(), first=lo, n=m, update_state=False, detail=True)
    maps = {k: v.cpu().numpy() for k, v in e.tracks_last_maps(lo, m).items()}
    _same((maps, out.cpu().numpy(), det.cpu().numpy()), base, range(lo, lo + m), "sub-range")


# ------------------------------------------------------------------------------------------------
# 4. range guard: tcgen05 flags what overflows fp16, simt computes it in fp32
# ------------------------------------------------------------------------------------------------
VT_TRACK_NUMERIC_RANGE = 3
GUARD_CASES = {          # key, factor, rows (None: all)
    "stem conv1": ("patch_embed.net.0.c.weight", 1e6, None),
    "attention values": ("blocks.0.attn.qkv.weight", 1e6, (192, 288)),
    "MLP hidden": ("blocks.0.mlp.fc1.weight", 1e6, None),
    "head conv1": ("box_head.conv1_ctr.0.weight", 1e7, None),
}
GUARD_ROWS = ["c256_identity_top_left", "odd_interior_half", "uhd_interior"]


@pytest.mark.gpu
@pytest.mark.parametrize("impl", ["tcgen05", "simt"])
@pytest.mark.parametrize("what", list(GUARD_CASES))
def test_range_guard_flags_tcgen05_and_simt_stays_fp32(frames, what, impl):
    key, factor, rows = GUARD_CASES[what]
    sd = make_sd("small")
    big = {k: v.clone() for k, v in sd.items()}
    lo, hi = rows if rows else (0, big[key].shape[0])
    big[key][lo:hi] = big[key][lo:hi] * factor
    tr = Tracks(frames, [s for s in _table_specs() if s[0] in GUARD_ROWS])
    e = _engine("small", tr.n, sd=big, impl=impl)
    maps, out, det = _step(e, tr.device(e.device), tr.n)
    if impl == "tcgen05":
        assert (det[:, 6] == VT_TRACK_NUMERIC_RANGE).all(), (what, det[:, 6])
        assert (out[:, 4] == -1.0).all()
        for k in MAPS:
            assert np.isnan(maps[k]).all(), (what, k)
        return
    assert (det[:, 6] == 0).all(), (what, "flagged under simt", det[:, 6])
    torch.set_num_threads(16)
    want = _maps64("small", tr, sd=big)
    err = {k: float(np.abs(maps[k].astype(np.float64) - want[k].numpy()).max()) for k in MAPS}
    print(f"\nrange guard simt [{what}]:", err)
    for k in MAPS:
        assert err[k] <= TOL["small_simt"][k], (what, k, err[k])
    assert_decode_exact(maps, out, det, tr, tag=f"simt {what}")
