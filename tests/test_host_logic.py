"""CPU: host-side logic - config/params mirrors, the C-ABI library's exports and error behaviour
without a device, track sharding + the box gather over gloo (world_size 2)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_config_overlay_and_unknown_key(tmp_path):
    from vittracker_b200 import config
    c = config.load_cfg()
    assert c.MODEL.BACKBONE.CHANNELS == 48 and c.MODEL.BACKBONE.HEADS == 1 and c.MODEL.HEAD.NUM_CHANNELS == 32
    assert c.TEST.SEARCH_SIZE == 256 and c.TEST.SEARCH_FACTOR == 4.0 and c.TEST.TEMPLATE_SIZE == 128
    assert config.default_cfg().TEST.SEARCH_SIZE == 320            # family default untouched
    bad = tmp_path / "bad.yaml"
    bad.write_text("MODEL:\n  NOT_A_KEY: 1\n")
    with pytest.raises(ValueError, match="NOT_A_KEY not exist in config.py"):
        config.update_config_from_file(str(bad), config.default_cfg())


def test_parameters_bag():
    from vittracker_b200 import parameters
    p = parameters("vit_48_h32_noKD", save_dir="/tmp/vt")
    assert (p.template_factor, p.template_size, p.search_factor, p.search_size) == (2.0, 128, 4.0, 256)
    assert p.checkpoint == "/tmp/vt/checkpoints/train/vit_dist/vit_48_h32_noKD/OstrackDist_ep0300.pth.tar"
    assert p.save_all_boxes is False and p.get("missing", 3) == 3 and p.has("cfg")


def test_state_dict_names_match_oracle():
    from oracle import vt_oracle as O
    from vittracker_b200 import load_cfg
    from vittracker_b200.weights import param_shapes, random_init_state_dict
    a, b = param_shapes(load_cfg()), O.param_shapes()
    assert a == b
    sd = random_init_state_dict(load_cfg())
    n = sum(v.numel() for k, v in sd.items() if v.is_floating_point() and "running" not in k)
    assert n == 174403                                              # SURVEY: 174 403 parameters


def test_library_exports_every_declared_symbol():
    from vittracker_b200 import _lib
    header = open(os.path.join(ROOT, "include", "vittrack_b200.h")).read()
    declared = set(re.findall(r"\b(vt_[a-z_0-9]+)\s*\(", header))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.vt_abi_version() == 1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device failure path")
def test_no_cpu_fallback():
    from vittracker_b200 import _lib, load_cfg
    lib = _lib.load()
    h = C.c_void_p()
    cfg = _lib.VtConfig(48, 1, 3, 4, 32, 16, 128, 256, 2.0, 4.0, 1, 0, 0, 0)
    assert lib.vt_create(C.byref(cfg), C.byref(h)) == -6
    assert b"no CPU fallback" in lib.vt_last_error(None)
    from vittracker_b200.engine import Engine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Engine(load_cfg())


def test_unsupported_config_rejected():
    from vittracker_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    # stride 8, embed dim not a multiple of 8, depth out of range: no kernels -> VT_ERR_UNSUPPORTED before any device work
    for bad in ((48, 1, 3, 4, 32, 8, 128, 256), (50, 1, 3, 4, 32, 16, 128, 256), (768, 12, 64, 4, 256, 16, 128, 256),
                (48, 1, 3, 4, 32, 16, 128, 320)):
        cfg = _lib.VtConfig(*bad, 2.0, 4.0, 1, 0, 0, 0)
        assert lib.vt_create(C.byref(cfg), C.byref(h)) == -5, bad
    assert lib.vt_create(None, C.byref(h)) == -1


def test_tensor_ptr_refuses_what_the_abi_would_misread():
    from vittracker_b200.engine import tensor_ptr
    cpu = torch.device("cpu")
    boxes = torch.zeros((3, 4), dtype=torch.float64)
    assert tensor_ptr(boxes, "boxes", torch.float64, cpu, (3, 4)).value == boxes.data_ptr()
    assert tensor_ptr(None, "out_detail", torch.float64, cpu, (3, 8), optional=True).value is None
    bad = {"None": None, "dtype": boxes.float(), "device": boxes.to("meta"), "non-contiguous": torch.zeros((4, 3), dtype=torch.float64).t(),
           "short": boxes[:2], "numpy": boxes.numpy()}
    for what, t in bad.items():
        with pytest.raises(ValueError, match="boxes"):
            tensor_ptr(t, "boxes", torch.float64, cpu, (3, 4))
    R = 12352
    base = torch.zeros(2 * R + 16, dtype=torch.uint8)
    assert tensor_ptr(base[16:16 + 2 * R].view(2, R), "records", torch.uint8, cpu, (2, R), align=16).value == base.data_ptr() + 16
    with pytest.raises(ValueError, match="16-byte aligned"):
        tensor_ptr(base[1:1 + 2 * R].view(2, R), "records", torch.uint8, cpu, (2, R), align=16)
    assert tensor_ptr(base, "frames", torch.uint8, cpu).value == base.data_ptr()            # no shape: any buffer


def test_shard_range_partitions():
    from vittracker_b200.batched import shard_range
    for total in (0, 1, 7, 8, 1024, 8191, 8192):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_tracker_clip_box_matches_oracle():
    from oracle import vt_oracle as O
    from vittracker_b200.tracker import clip_box
    rng = np.random.default_rng(0)
    for _ in range(200):
        b = list(rng.uniform(-50, 400, size=4))
        assert clip_box(b, 240, 320, margin=10) == O.clip_box(b, 240, 320, margin=10)


_GLOO_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["VT_ROOT"])
from vittracker_b200.batched import ShardedTracker, shard_range
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["VT_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
for total in (8, 7, 3):
    sh = ShardedTracker(total)
    lo, hi = sh.lo, sh.hi
    local = torch.arange(lo, hi, dtype=torch.float64).unsqueeze(1) * torch.tensor([[1., 10., 100., 1000., 0.5]], dtype=torch.float64)
    full = sh.gather(local)
    want = torch.arange(0, total, dtype=torch.float64).unsqueeze(1) * torch.tensor([[1., 10., 100., 1000., 0.5]], dtype=torch.float64)
    assert full.shape == (total, 5) and torch.equal(full, want), (total, full)
    # overlapped form: two gathers one after the other, alternating buffers; ragged shards (7, 3) come back compacted too
    w1, r1 = sh.gather_async(local)
    w1.wait()
    w2, r2 = sh.gather_async(local * 2)
    w2.wait()
    assert r1.shape == (total, 5) and r2.shape == (total, 5), (total, r1.shape)
    assert torch.equal(r1, want) and torch.equal(r2, want * 2), (total, r1, r2)
dist.barrier()
dist.destroy_process_group()
print("OK", os.environ["RANK"])
'''


def test_sharded_gather_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", VT_ROOT=ROOT, VT_PORT=port, MASTER_ADDR="127.0.0.1")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0 and "OK" in out, out


def test_table_free_normalisation_is_exact():
    """The fused crop + conv1 kernel normalises pixels in registers (vt_stem.cu: normalize_px): its two divisions by constants
    must equal the reference's rounded ((v / 255) - mean) / std for all 256 values x 3 channels (exact rational arithmetic)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("norm_exact_check", os.path.join(ROOT, "tools", "norm_exact_check.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.check() == 0


def test_ab_identity_compare_detects_a_single_bit(tmp_path):
    """tools/ab_identity.py --compare is the gate for instruction-level rewrites: equal dumps pass, one flipped mantissa bit fails."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ab_identity", os.path.join(ROOT, "tools", "ab_identity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rng = np.random.default_rng(0)
    a = {"boxes": rng.standard_normal((4, 5)), "score": rng.standard_normal((4, 1, 16, 16)).astype(np.float32)}
    np.savez(tmp_path / "a.npz", **a)
    np.savez(tmp_path / "b.npz", **a)
    assert mod.compare(str(tmp_path / "a.npz"), str(tmp_path / "b.npz")) == 0
    b = {k: v.copy() for k, v in a.items()}
    b["score"].view(np.uint32)[0, 0, 3, 7] ^= 1
    np.savez(tmp_path / "c.npz", **b)
    assert mod.compare(str(tmp_path / "a.npz"), str(tmp_path / "c.npz")) == 1


def test_hardswish_division_algorithm_on_samples():
    """vt_internal.h div6_exact / hardswish_exact_n: q = p r; q' = fma(fma(-6, q, p), r, q), r = fl(1/6), sign of a zero product restored with
    an OR, IEEE division below 1e-36.  The exhaustive check is the GPU tool (tools/div6_check.cu); here the same algorithm is emulated in exact
    rational arithmetic on edge cases + 20 000 random bit patterns and compared with the correctly rounded p / 6."""
    import importlib.util
    from fractions import Fraction as Fr
    spec = importlib.util.spec_from_file_location("norm_exact_check", os.path.join(ROOT, "tools", "norm_exact_check.py"))
    nx = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(nx)
    fl, ex, fma, bits = nx.fl, nx.ex, nx.fma, nx.bits
    r = np.float32(0.16666667163372039794921875)
    assert bits(r) == bits(fl(Fr(1, 6)))
    rng = np.random.default_rng(5)
    pats = rng.integers(0, 2 ** 32, size=20000, dtype=np.uint64).astype(np.uint32)
    edge = np.array([0x00000000, 0x80000000, 0x03aa2425, 0x03aa2424, 0x83aa2425, 0x3f800000, 0x40c00000, 0x7f7fffff, 0xff7fffff,
                     0x00800000, 0x01000000, 0x3e2aaaab, 0x40400000], dtype=np.uint32)
    bad = 0
    for u in np.concatenate([edge, pats]):
        p = np.array([u], dtype=np.uint32).view(np.float32)[0]
        if not np.isfinite(p):
            continue
        want = fl(ex(p) / 6)
        if abs(float(p)) >= 1e-36 or p == 0:
            q = fl(ex(p) * ex(r))
            f = fma(fma(np.float32(-6.0), q, p), r, q)
            got_bits = bits(f) | (int(u) & 0x80000000)          # the OR that keeps -0 (x <= -3 gives p = -0)
        else:
            got_bits = None
        want_bits = bits(want) | ((int(u) & 0x80000000) if want == 0 else 0)     # fl() drops the sign of a zero quotient
        if not (abs(float(p)) >= 1e-36 or p == 0):
            got_bits = want_bits                                 # the out-of-line IEEE division
        bad += got_bits != want_bits
    assert bad == 0
