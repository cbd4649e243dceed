"""The bench line contract, checked on CPU: the committed final line of the round (profiles/r2j_bench_c2_n1.jsonl,
written by `python bench.py` on a B200) carries every key the driver and the judge read, with consistent values;
bench.py parses and its argument surface is the driver's (`--gpus --steps --warmup --impl`).  No GPU work here."""
import ast
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lines():
    with open(os.path.join(ROOT, "profiles", "r2j_bench_c2_n1.jsonl")) as f:
        return [json.loads(x) for x in f if x.startswith("{")]


def test_committed_bench_line_has_the_contract_keys():
    ours = _lines()[0]
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in ours, k
    assert ours["unit"] == "pairs/s" and ours["higher_is_better"] is True and ours["n_gpus"] == 1
    assert ours["warmup"] >= 3 and ours["data"] == "synthetic" and ours["vs_baseline"] is None
    assert "workload" in ours["config"] and "1000" in ours["config"]["workload"]
    assert isinstance(baseline.get("metric"), str) and baseline["metric"]
    # value really is pairs / device time of the timed steps
    pairs = ours["config"]["pairs"]
    assert abs(ours["value"] - pairs / (ours["ms_per_step"] * 1e-3)) / ours["value"] < 1e-6
    r = ours["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "kernel"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and r["unit"] == "GB/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    # achieved = algorithmic bytes of a step / the kernel's own time, and the kernel fits inside the step
    assert abs(r["achieved"] - r["algorithmic_bytes_per_step"] / (r["ms_per_step"] * 1e-3) / 1e9) / r["achieved"] < 1e-6
    assert r["ms_per_step"] <= ours["ms_per_step"]
    assert "ESTIMATED" in r["traffic_source"]  # the DRAM figure is an estimate and says so
    c = ours["cpu_baseline"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in c, k
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1
    e = ours["e2e"]
    assert e["h2d_bytes_per_step"] == 1000 * 5_000_000 and e["d2h_bytes_per_step"] > 0 and e["value"] > 0
    assert ours["gpu_launches"] > 0
    assert not set(ours["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_committed_reference_arm_line():
    ref = [x for x in _lines() if x.get("impl") == "reference"]
    assert ref, "the --impl reference line of the round is committed next to ours"
    ref = ref[0]
    assert ref["unit"] == "pairs/s" and ref["cpu_baseline"]["value"] == ref["value"]
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["e2e"]["d2h_bytes_per_step"] == 0
    assert ref.get("product_library_loaded") is False  # the arm never touches libgkd.so


def test_bench_argument_surface():
    src = open(os.path.join(ROOT, "bench.py")).read()
    ast.parse(src)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr


def test_dump_outputs_samples_large_results_at_fixed_pairs(tmp_path, monkeypatch):
    """more pairs than DUMP_PAIRS: the same seeded, sorted pair sample every time, values taken at those pairs"""
    import numpy as np

    import bench

    monkeypatch.setattr(bench, "DUMP_PAIRS", 500)
    total = 4950
    inter = (np.arange(total, dtype=np.uint64) * 7919) % 100003
    dist = 1.0 - np.arange(total) / total
    got = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), inter, dist)
        got.append({n: np.load(tmp_path / d / (n + ".npy")) for n in ("pair_index", "intersections", "distances")})
    idx = got[0]["pair_index"]
    assert all(x.dtype == np.float64 and x.shape == (500,) for x in got[0].values())
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < total
    k = idx.astype(np.int64)
    assert np.array_equal(got[0]["intersections"], inter[k].astype(np.float64))
    assert np.array_equal(got[0]["distances"], dist[k])
    for n in got[0]:
        assert np.array_equal(got[0][n], got[1][n])
