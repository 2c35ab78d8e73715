"""Every path's bits under exact power-of-two rescalings of the weights.

A checkpoint may split scale freely between a LayerNorm or BatchNorm affine and the next layer's weights, between the q and k rows of
a block's qkv, and between its v rows and the output projection.  LayerNorm's affine, ReLU and BatchNorm's running statistics (they
normalise the product, not each factor) make "LN gain 2^-8 with weights 2^8 times larger" the same model, and the fp32 oracle gives
the same bits for it.  The tensor-core paths split every operand into fp16 hi + lo (vt_tc.cuh), which holds ~22 bits only while both
halves are normal fp16 numbers: the random-init weights of every other test keep each operand near magnitude 1, a trained checkpoint
need not.  At weight ingest vt_api.cu (``rebalance``) moves a power of two across each pair below so that the packed operands do not
depend on how the checkpoint splits the scale.

Rewrite table, s = 2^-k, written for any (C, depth, head channels); "moves" names the tensor-core operands of the tuned path:

    name        rewrite                                                          moves
    norm        norm.{weight,bias} x s, box_head.conv1_*.0.weight x 1/s          head conv1 A (LayerNorm output) and B
    head_bn<i>  per tower conv<i>_t.1.{weight,bias} x s, conv<i+1>_t.0.weight    conv i B (folded weights), conv i+1 A; conv4 is fp32
                x 1/s (conv5_t.weight for i = 4)
    head_bn4                                                                     none: fp32 control
    ln1         blocks.b.norm1.{weight,bias} x s, attn.qkv.weight x 1/s          QKV A and B
    ln2         norm2.{weight,bias} x s, mlp.fc1.weight x 1/s                    fc1 A and B
    qk          qkv.{weight,bias} rows [0, C) x 1/s, rows [C, 2C) x s            q and K of the scores
    vproj       qkv rows [2C, 3C) x s, attn.proj.weight x 1/s                    tuned path none (Wproj Wv is folded in float64):
                                                                                 control; generic path P V and proj

at k in {-12, -6, 6, 12}; ``norm`` also at k = -14, where the LayerNorm output nears fp16's 65504; and one composite case: every rewrite at
once, a seeded k in [-12, 12] per block, per tower and per pair.

1. CPU.  The fp32 oracle's maps, boxes and taps are bit-identical under every rewrite (tokens_norm under ``norm``: exactly
   ldexp(tap, -k)).  The unscaled fp16 hi / lo emulation (tools/precision_budget.py: mm_split) of each contraction a rewrite moves
   differs from rung 0's: a kernel that split the checkpoint's operands as they come could not pass the GPU test by accident.

2. GPU.  simt, tcgen05, tcgen05_3term, and the generic configurations ``small`` (Linear layers on gemm_tc) and ``img`` (gemm_img) of
   test_generic_edges.py: one engine per implementation steps the crop-edge table of test_tracking_edges.py once per rewrite and rung
   (reloading the weights with load_state_dict), and runs Engine.forward(z, x, taps=True) on the table's oracle crops.  Maps, boxes,
   detail rows, pred_boxes and block taps must be bit-identical to rung 0 and decode exactly; tokens_norm is scaled by exactly 2^-k
   under ``norm``.  A failing case prints its max |err| against the float64 oracle of the rewritten weights.

   Measured on an NVIDIA B200 at the parent commit, before the rebalance (max |score_map - float64| over the table, rung 0 of each
   implementation in brackets):

       case                     simt        tcgen05  tcgen05_3term          small            img
       rung 0              (3.5e-07)      (1.8e-06)      (1.5e-06)      (1.2e-06)      (1.4e-06)
       norm@-12                    =        3.1e-04        3.1e-04        5.7e-04        7.6e-04
       norm@-6                     =        9.2e-06        8.6e-06        1.3e-05        2.0e-05
       norm@6                      =        1.8e-06        1.7e-06        1.3e-06        1.5e-06
       norm@12                     =        4.7e-05        4.4e-05        4.2e-05        4.7e-05
       head_bn1@-12                =        2.9e-04        2.9e-04        1.1e-06        4.7e-04
       head_bn1@-6                 =        3.0e-06        2.9e-06        1.1e-06        6.3e-06
       head_bn1@6                  =        9.2e-06        8.7e-06        1.3e-05        1.9e-05
       head_bn1@12                 =        3.0e-04        3.0e-04        5.7e-04        7.6e-04
       head_bn2@-12                =        2.9e-04        2.9e-04              =        3.2e-04
       head_bn2@-6                 =        4.7e-06        4.2e-06              =        5.4e-06
       head_bn2@6                  =        3.1e-06        3.2e-06              =        6.6e-06
       head_bn2@12                 =        3.1e-04        3.1e-04              =        4.9e-04
       head_bn3@-12                =        1.8e-06        1.5e-06              =        1.4e-06
       head_bn3@-6                 =        1.8e-06        1.5e-06              =        1.4e-06
       head_bn3@6                  =        4.8e-06        4.3e-06              =        5.5e-06
       head_bn3@12                 =        2.9e-04        2.9e-04              =        3.2e-04
       head_bn4@-12                =              =              =              =              =
       head_bn4@-6                 =              =              =              =              =
       head_bn4@6                  =              =              =              =              =
       head_bn4@12                 =              =              =              =              =
       ln1@-12                     =        8.2e-04        8.2e-04        6.1e-04        5.2e-04
       ln1@-6                      =        1.4e-05        1.5e-05        1.0e-05        1.4e-05
       ln1@6                       =        1.9e-06        1.7e-06        1.2e-06        1.3e-06
       ln1@12                      =        3.8e-06        3.5e-06        3.1e-06        4.5e-06
       ln2@-12                     =        1.6e-04        1.6e-04        1.7e-04        3.7e-04
       ln2@-6                      =        2.8e-06        2.9e-06        2.3e-06        4.6e-06
       ln2@6                       =        2.0e-06        1.7e-06        1.2e-06        1.6e-06
       ln2@12                      =        2.5e-05        2.4e-05        2.0e-05        2.6e-05
       qk@-12                      =        2.4e-06        2.5e-06        2.6e-06        8.2e-06
       qk@-6                       =        1.7e-06        1.5e-06        1.2e-06        1.4e-06
       qk@6                        =        1.8e-06        1.5e-06        1.2e-06        1.6e-06
       qk@12                       =        1.4e-06        1.1e-06        1.4e-06        3.2e-06
       vproj@-12                   =              =              =        5.3e-04        5.4e-04
       vproj@-6                    =              =              =        6.1e-06        1.2e-05
       vproj@6                     =              =              =        1.1e-05        1.5e-05
       vproj@12                    =              =              =        5.9e-04        5.5e-04
       norm@-14                    =        1.9e-03        1.9e-03        3.3e-03        4.9e-03
       composite                   =        flagged        flagged        1.9e-04        flagged

   "=": bit-identical to rung 0; "flagged": every track withheld as VT_TRACK_NUMERIC_RANGE (an operand past 65504).  simt (fp32 on
   every layer), head_bn4 and the tuned path's vproj were identical already; head_bn2 / head_bn3 under ``small`` too (its head conv2 -
   conv4 run on the fp32 sgemm).  norm at -14 was not flagged on any path, but off by 2e-3 to 5e-3.  With the rebalance every case of
   every implementation is bit-identical to rung 0; the GPU tests of this file take 10 s on a B200.
"""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import vt_oracle as O
from test_generic_edges import CONFIGS, make_cfg, make_sd, model64
from test_tracking_edges import MAPS, Tracks, _crops, _step, _table_specs, assert_decode_exact, oracle64

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from precision_budget import mm_split  # noqa: E402

REWRITES = ("norm", "head_bn1", "head_bn2", "head_bn3", "head_bn4", "ln1", "ln2", "qk", "vproj")
RUNGS = (-12, -6, 6, 12)
CASES = [(r, k) for r in REWRITES for k in RUNGS] + [("norm", -14), ("composite", 0)]
IDS = [f"{r}@{k}" if r != "composite" else r for r, k in CASES]
COMPOSITE_SEED = 1234
VT_TRACK_NUMERIC_RANGE = 3


def _depth(sd):
    return sum(1 for k in sd if k.endswith(".norm1.weight"))


def _scale(t, e, lo=None, hi=None):
    """t[lo:hi] *= 2^e in place (exact in fp32)."""
    if lo is None:
        t.mul_(2.0 ** e)
    else:
        t[lo:hi] *= 2.0 ** e


def apply_rewrite(sd, name, k, block=None, tower=None):
    """One rewrite of the table at rung k (s = 2^-k), in place; ``block`` / ``tower``: only that one (None: all)."""
    C = sd["norm.weight"].numel()
    if name == "norm":
        _scale(sd["norm.weight"], -k)
        _scale(sd["norm.bias"], -k)
        for t in O.TOWERS:
            _scale(sd[f"box_head.conv1_{t}.0.weight"], k)
    elif name.startswith("head_bn"):
        i = int(name[-1])
        for t in O.TOWERS if tower is None else (tower,):
            _scale(sd[f"box_head.conv{i}_{t}.1.weight"], -k)
            _scale(sd[f"box_head.conv{i}_{t}.1.bias"], -k)
            _scale(sd[f"box_head.conv{i + 1}_{t}.0.weight" if i < 4 else f"box_head.conv5_{t}.weight"], k)
    else:
        for b in range(_depth(sd)) if block is None else (block,):
            p = f"blocks.{b}."
            w, bias = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
            if name in ("ln1", "ln2"):
                _scale(sd[p + f"norm{name[-1]}.weight"], -k)
                _scale(sd[p + f"norm{name[-1]}.bias"], -k)
                _scale(w if name == "ln1" else sd[p + "mlp.fc1.weight"], k)
            elif name == "qk":
                for t in (w, bias):
                    _scale(t, k, 0, C)
                    _scale(t, -k, C, 2 * C)
            elif name == "vproj":
                for t in (w, bias):
                    _scale(t, -k, 2 * C, 3 * C)
                _scale(sd[p + "attn.proj.weight"], k)
            else:
                raise ValueError(name)


def rewritten(sd, name, k):
    """(a rewritten copy of sd, the rung of ``norm`` in it)."""
    out = {n: v.clone() for n, v in sd.items()}
    if name != "composite":
        apply_rewrite(out, name, k)
        return out, (k if name == "norm" else 0)
    rng = np.random.default_rng(COMPOSITE_SEED)
    draw = lambda: int(rng.integers(-12, 13))
    k_norm = draw()
    apply_rewrite(out, "norm", k_norm)
    for name in REWRITES[1:]:
        if name.startswith("head_bn"):
            for t in O.TOWERS:
                apply_rewrite(out, name, draw(), tower=t)
        else:
            for b in range(_depth(sd)):
                apply_rewrite(out, name, draw(), block=b)
    return out, k_norm


# ------------------------------------------------------------------------------------------------
# weights, crops, implementations
# ------------------------------------------------------------------------------------------------
# implementation -> (blocks_impl, generic configuration or None)
IMPLS = {"simt": ("simt", None), "tcgen05": ("tcgen05", None), "tcgen05_3term": ("tcgen05_3term", None),
         "small": ("tcgen05", "small"), "img": ("tcgen05", "img")}
CPU_ROWS = ["c256_identity_top_left", "odd_interior_half", "uhd_interior"]


@pytest.fixture(scope="module")
def frames():
    from test_tracking_edges import _frames
    return _frames()


@pytest.fixture(scope="module")
def table(frames):
    return Tracks(frames, _table_specs())


def _weights(gen, golden_model):
    if gen is None:
        from conftest import state_dict_from_npz
        return state_dict_from_npz(golden_model)
    return make_sd(gen)


def _oracle(sd, gen):
    if gen is None:
        return O.OracleModel(sd)
    _, heads, depth, _, _ = CONFIGS[gen]
    return O.OracleModel(sd, depth=depth, num_heads=heads)


# ------------------------------------------------------------------------------------------------
# 1. CPU: the fp32 oracle is invariant, the unscaled split is not
# ------------------------------------------------------------------------------------------------
def test_rewrites_are_exact_and_composite_moves_every_pair(golden_model):
    sd = _weights(None, golden_model)
    for name, k in CASES:
        got, k_norm = rewritten(sd, name, k)
        changed = {n for n in sd if not torch.equal(sd[n], got[n])}
        assert changed, (name, k)
        back = {n: v.clone() for n, v in got.items()}
        if name != "composite":
            apply_rewrite(back, name, -k)
            assert all(torch.equal(back[n], sd[n]) for n in sd), (name, k, "the rewrite at -k must undo the rewrite at k")
    got, _ = rewritten(sd, "composite", 0)
    moved = {n for n in sd if not torch.equal(sd[n], got[n])}
    for name, k in CASES[:-2]:
        one, _ = rewritten(sd, name, k)
        assert {n for n in sd if not torch.equal(sd[n], one[n])} <= moved, name


@pytest.mark.parametrize("gen", [None, "small"], ids=["vit_48_h32", "small"])
def test_oracle_bits_unchanged_by_every_rewrite(frames, golden_model, gen):
    torch.set_num_threads(16)
    tr = Tracks(frames, [s for s in _table_specs() if s[0] in CPU_ROWS])
    z, x = _crops(tr)
    sd = _weights(gen, golden_model)
    taps0 = {}
    want = _oracle(sd, gen).forward(z, x, taps0)
    for name, k in CASES:
        rsd, k_norm = rewritten(sd, name, k)
        taps = {}
        got = _oracle(rsd, gen).forward(z, x, taps)
        for m in (*MAPS, "pred_boxes"):
            assert torch.equal(got[m], want[m]), (gen, name, k, m)
        assert set(taps) == set(taps0)
        for t in taps0:
            w = torch.ldexp(taps0[t], torch.tensor(-k_norm)) if t == "tokens_norm" else taps0[t]
            assert torch.equal(taps[t], w), (gen, name, k, t)


class Operands(O.OracleModel):
    """The fp32 oracle, recording the operands A [.., M, K] and B [.., K, N] of every contraction the tensor-core paths split:
    qkv, scores, pv, proj, fc1, fc2 of each block (unfused), and head conv1 - conv4 of each tower (im2col x BatchNorm-folded weights)."""

    def forward(self, z, x, taps=None):
        self.ops = {}
        return super().forward(z, x, taps)

    def block(self, x, b):
        p = f"blocks.{b}"
        B, N, C = x.shape
        hd = C // self.num_heads
        def lin(a, n):
            key = {"qkv": "attn.qkv", "proj": "attn.proj", "fc1": "mlp.fc1", "fc2": "mlp.fc2"}[n]
            self.ops[f"{n}{b}"] = (a, self.sd[f"{p}.{key}.weight"].t())
            return F.linear(a, self.sd[f"{p}.{key}.weight"], self.sd[f"{p}.{key}.bias"])

        h = F.layer_norm(x, (C,), self.sd[f"{p}.norm1.weight"], self.sd[f"{p}.norm1.bias"], O.LN_EPS)
        qkv = lin(h, "qkv").reshape(B, N, 3, self.num_heads, hd).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0] * (hd ** -0.5), qkv[1], qkv[2]
        self.ops[f"scores{b}"] = (q, k.transpose(-2, -1))
        attn = (q @ k.transpose(-2, -1)).softmax(dim=-1)
        self.ops[f"pv{b}"] = (attn, v)
        x = x + lin((attn @ v).transpose(1, 2).reshape(B, N, C), "proj")
        h = F.layer_norm(x, (C,), self.sd[f"{p}.norm2.weight"], self.sd[f"{p}.norm2.bias"], O.LN_EPS)
        return x + lin(F.gelu(lin(h, "fc1")), "fc2")

    def head(self, feat):
        for t in O.TOWERS:
            y = feat
            for i in range(4):
                p = f"box_head.conv{i + 1}_{t}"
                g, var = self.sd[f"{p}.1.weight"].double(), self.sd[f"{p}.1.running_var"].double()
                wf = (self.sd[f"{p}.0.weight"].double() * (g / torch.sqrt(var + O.BN_EPS))[:, None, None, None]).float()
                self.ops[f"conv{i + 1}_{t}"] = (F.unfold(y, 3, padding=1).transpose(1, 2), wf.reshape(wf.shape[0], -1).t())
                y = F.conv2d(y, self.sd[f"{p}.0.weight"], self.sd[f"{p}.0.bias"], stride=1, padding=1)
                y = F.relu(F.batch_norm(y, self.sd[f"{p}.1.running_mean"], self.sd[f"{p}.1.running_var"], self.sd[f"{p}.1.weight"],
                                        self.sd[f"{p}.1.bias"], False, 0.0, O.BN_EPS))
        return super().head(feat)


def moved(name, depth):
    """The contractions a rewrite moves on some tensor-core path (module docstring)."""
    towers = lambda *layers: [f"conv{i}_{t}" for i in layers for t in O.TOWERS]
    blocks = lambda *ops: [f"{o}{b}" for o in ops for b in range(depth)]
    return {"norm": towers(1), "head_bn1": towers(1, 2), "head_bn2": towers(2, 3), "head_bn3": towers(3), "head_bn4": [],
            "ln1": blocks("qkv"), "ln2": blocks("fc1"), "qk": blocks("scores"), "vproj": blocks("pv", "proj")}[name]


def test_unscaled_split_of_every_moved_contraction_differs(frames, golden_model):
    torch.set_num_threads(16)
    tr = Tracks(frames, [s for s in _table_specs() if s[0] in CPU_ROWS[:2]])
    z, x = _crops(tr)
    sd = _weights(None, golden_model)
    m0 = Operands(sd)
    m0.forward(z, x)
    split0 = {n: mm_split(a, b, None) for n, (a, b) in m0.ops.items()}
    for name, k in CASES[:-1]:
        m = Operands(rewritten(sd, name, k)[0])
        m.forward(z, x)
        for n in moved(name, m.depth):
            a, b = m.ops[n]
            assert not torch.equal(mm_split(a, b, None), split0[n]), (name, k, n)


# ------------------------------------------------------------------------------------------------
# 2. GPU: the same bits on every path
# ------------------------------------------------------------------------------------------------
_F64 = {}


def _err64(gen, name, k, rsd, tr, maps):
    """max |map - float64 oracle of the rewritten weights| (cached per weight set: the tuned implementations share it)."""
    key = (gen, name, k)
    if key not in _F64:
        torch.set_num_threads(16)
        if gen is None:
            _F64[key] = oracle64(rsd, tr)
        else:
            _, heads, depth, _, _ = CONFIGS[gen]
            z, x = _crops(tr)
            _F64[key] = model64(rsd, depth, heads).forward(z.double(), x.double())
    want = _F64[key]
    return {m: float(np.nanmax(np.abs(maps[m].astype(np.float64) - want[m].numpy()))) for m in MAPS}


def _engine(impl, n):
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    blocks, gen = IMPLS[impl]
    if gen is None:
        return Engine(load_cfg(), max_tracks=n, blocks_impl=blocks)
    C, heads, depth, hc, _ = CONFIGS[gen]
    return Engine(make_cfg(C, heads, hc), max_tracks=n, blocks_impl=blocks, depth=depth)


def _forward(e, z, x):
    got = e.forward(z, x, taps=True)
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in got.items()}


def _differences(step, fwd, step0, fwd0, k_norm):
    """What differs from rung 0: '<n> tracks' of the step (maps, boxes or detail rows), forward outputs and taps by name."""
    (gm, go, gd), (wm, wo, wd) = step, step0
    n = go.shape[0]
    bad = [i for i in range(n) if not (all(np.array_equal(gm[m][i], wm[m][i]) for m in MAPS)
                                       and np.array_equal(go[i], wo[i]) and np.array_equal(gd[i], wd[i]))]
    out = [f"step: {len(bad)} of {n} tracks"] if bad else []
    flagged = int((gd[:, 6] == VT_TRACK_NUMERIC_RANGE).sum())
    if flagged:
        out.append(f"{flagged} tracks flagged VT_TRACK_NUMERIC_RANGE")
    for m in (*MAPS, "pred_boxes"):
        if not torch.equal(fwd[m], fwd0[m]):
            out.append(f"forward {m}")
    taps, taps0 = fwd["taps"], fwd0["taps"]
    last = taps.shape[0] - 1
    for i in range(last):
        if not torch.equal(taps[i], taps0[i]):
            out.append("stem tap" if i == 0 else f"block {i} tap")
    if not torch.equal(taps[last], torch.ldexp(taps0[last], torch.tensor(-k_norm))):
        out.append("tokens_norm tap")
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("impl", list(IMPLS))
def test_every_rewrite_gives_rung_0_bits(table, golden_model, impl):
    blocks, gen = IMPLS[impl]
    sd = _weights(gen, golden_model)
    e = _engine(impl, table.n)
    d = table.device(e.device)
    z, x = _crops(table)
    e.load_state_dict(sd)
    step0, fwd0 = _step(e, d, table.n), _forward(e, z, x)
    assert (step0[2][:, 6] == 0).all()
    assert_decode_exact(*step0, table, tag=f"{impl} rung 0")
    failures = []
    for name, k in CASES:
        rsd, k_norm = rewritten(sd, name, k)
        e.load_state_dict(rsd)
        step, fwd = _step(e, d, table.n), _forward(e, z, x)
        diff = _differences(step, fwd, step0, fwd0, k_norm)
        try:
            assert_decode_exact(*step, table, tag=impl)
        except AssertionError:
            diff.append("decode not exact")
        if diff:
            failures.append((name, k, diff, _err64(gen, name, k, rsd, table, step[0])))
    print(f"\n[{impl}] rung 0: max |err| vs float64 {_err64(gen, 'rung0', 0, sd, table, step0[0])}")
    for name, k, diff, err in failures:
        print(f"[{impl}] {name}@{k}: {'; '.join(diff)}; max |err| vs float64 {err}")
    assert not failures, f"{impl}: {len(failures)} of {len(CASES)} rewrites change the bits: {[(f[0], f[1]) for f in failures]}"
