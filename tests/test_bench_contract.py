"""The contract of bench.py: the reference arm runs without a GPU (it is the CPU path), the last recorded B200 line under
profiles/ must carry every key the contract names, and on a GPU two runs with the same arguments dump identical outputs."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "cpu_baseline", "e2e"}


def test_reference_arm_prints_one_contract_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                       # stdout carries the JSON line and nothing else
    d = json.loads(lines[0])
    assert BASE_KEYS | {"impl"} <= set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["unit"] == "frames/s" and d["value"] > 0 and d["steps"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert "workload" in d["config"] and "model" not in d["config"]
    boxes = np.load(tmp_path / "out" / "boxes.npy")
    assert boxes.dtype == np.float64 and boxes.shape == (256, 5) and np.isfinite(boxes).all()
    assert ((boxes[:, 4] > 0) & (boxes[:, 4] <= 1)).all()                       # confidence: the max of a sigmoid score map


def test_recorded_b200_line_has_every_contract_key():
    recorded = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_bench.json")))
    assert recorded, "no recorded bench line under profiles/"
    with open(recorded[-1]) as f:
        d = json.loads(f.read().strip().splitlines()[-1])
    assert BASE_KEYS | {"roofline", "clocks", "gpu_launches"} <= set(d)
    rf = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(rf) and rf["bound"] in ("hbm", "tensor")
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert d["gpu_launches"] > 0 and d["warmup"] >= 3 and d["n_gpus"] == 1
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_secondary_figures_are_json_safe_and_sane():
    """The pieces bench.py adds after the timed region (HBM rooflines of the stem and head, batch-1 CPU legs) run on the host: check them here,
    so that a mistake in them cannot cost the GPU run its line."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import vt_oracle as O
    stages = {k: {"ms": ms * 20, "launches": 20, "items": 1024 * 20} for k, ms in (("stem", 0.794), ("head", 0.173), ("blocks", 0.58), ("crop", 0.0))}
    r = bench.hbm_rooflines(O.synth_boxes(1024, bench.FRAME_H, bench.FRAME_W, seed=3000), stages, bench.measured_peaks())
    json.dumps(r)
    for k in ("stem", "head"):
        assert 0 < r[k]["frac"] < 1 and abs(r[k]["frac"] - r[k]["achieved"] / r[k]["peak"]) < 1e-12
    assert r["stem"]["bound"] == "hbm" and r["stem"]["unit"] == "GB/s"
    assert r["head"]["bound"] == "tensor" and r["head"]["unit"] == "TFLOP/s" and 0 < r["head"]["hbm_frac"] < 1      # latency-bound: labelled as such
    # a 720p crop reads at most 4 S^2 pixels x 3 bytes, and the tokens are 48 KB
    assert 49152 * 1024 < r["stem"]["algorithmic_bytes_per_launch"] <= (3 * 4 * 256 * 256 + 49152) * 1024
    assert r["stem"]["traffic"] > r["stem"]["algorithmic_bytes_per_launch"]
    assert isinstance(bench.cpu_model_name(), str)
    sd = O.make_state_dict(seed=1, stress=True)
    assert bench.cpu_b1_sample(sd, 1, budget_s=0.5) > 0


def test_dump_outputs_keeps_a_seeded_sample_within_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    boxes = np.random.default_rng(1).standard_normal((1000, 5))
    bench.dump_outputs(str(tmp_path / "all"), boxes)
    assert np.array_equal(np.load(tmp_path / "all" / "boxes.npy"), boxes) and not (tmp_path / "all" / "rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT", 4800)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), boxes)
    rows, got = np.load(tmp_path / "a" / "rows.npy"), np.load(tmp_path / "a" / "boxes.npy")
    assert rows.dtype == got.dtype == np.float64 and rows.nbytes + got.nbytes <= 4800
    idx = rows.astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0) and np.array_equal(got, boxes[idx])
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy")) and np.array_equal(got, np.load(tmp_path / "b" / "boxes.npy"))


@pytest.mark.gpu
def test_bench_dump_outputs_identical_from_run_to_run(tmp_path):
    """Two runs with the same arguments see the same inputs, so the boxes of their last timed step must be identical; the dumped boxes
    are the ones bench.py's parity leg re-runs bit for bit and checks against the CPU oracle."""
    lines = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "3", "--tracks", "256",
                            "--frames", "8", "--no-cpu-baseline", "--no-latency", "--no-gpu-eager", "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert all(d["steps"] == 3 for d in lines)
    for d in lines:
        p = d["parity_spot"]
        assert p["rerun_bit_identical_to_timed_step"] is True and p["flips"] == 0 and p["status_nonzero"] == 0, p
        assert p["max_box_err"] <= 1e-2 + 1e-3 * 1280 and p["max_conf_err"] < 1e-3, p
    a, b = np.load(tmp_path / "a" / "boxes.npy"), np.load(tmp_path / "b" / "boxes.npy")
    assert a.dtype == np.float64 and a.shape == (256, 5) and np.isfinite(a).all()
    assert np.array_equal(a, b)
