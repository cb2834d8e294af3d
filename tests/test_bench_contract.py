"""The committed bench lines (profiles/r1_bench*.json) carry every key of the driver's contract — a guard for
later edits of bench.py (the lines themselves are produced on a B200 by `python bench.py`)."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _line(name):
    with open(os.path.join(ROOT, "profiles", name)) as fp:
        return json.loads(fp.read().strip().splitlines()[-1])


@pytest.mark.parametrize("name", ["r1_bench.json", "r1_bench_2gpu.json", "r1_bench_8gpu.json"])
def test_own_arm_line(name):
    d = _line(name)
    assert BASE <= set(d) and "clocks" in d and "roofline" in d
    assert d["metric"] == "loci genotyped/sec" and d["unit"] == "loci/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["warmup"] >= 3 and d["value"] > 0 and d["gpu_launches"] > 0
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e)
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
    g = d["roofline_grid"]
    assert g["bound"] == "hbm" and abs(g["frac"] - g["achieved"] / g["peak"]) < 1e-9
    c = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c)
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if d["n_gpus"] == 1:
        b = d["cpu_baseline"]
        assert {"value", "unit", "cores", "kind", "sample"} <= set(b) and b["kind"] in ("reference", "port")
        assert b["calls_identical_to_gpu"].split("/")[0] == b["calls_identical_to_gpu"].split("/")[1]
        s = d["roofline_grid_stress"]
        assert s["bound"] == "hbm" and s["points"] == 32032000 and 0 < s["frac"] < 1


def test_dump_outputs_layout_and_seeded_sample(tmp_path, monkeypatch):
    """--dump-outputs: one float64 .npy per call field + problem.npy; above the size limit the same sorted sample of
    rows on every run, within the limit."""
    import numpy as np
    import bench
    from tredparse_b200 import cohort
    calls = np.zeros(1000, cohort.CALL_DTYPE)
    calls["allele1"], calls["pp"] = np.arange(1000), np.linspace(0, 1, 1000)
    calls["ci"] = np.arange(4000).reshape(1000, 4)
    bench.dump_outputs(str(tmp_path / "all"), calls, np.arange(1000) * 30 + 7)
    names = sorted(p.name for p in (tmp_path / "all").iterdir())
    assert names == sorted(n + ".npy" for n in cohort.CALL_DTYPE.names + ("problem",))
    got = {n[:-4]: np.load(str(tmp_path / "all" / n)) for n in names}
    assert all(a.dtype == np.float64 for a in got.values()) and got["ci"].shape == (1000, 4)
    assert np.array_equal(got["pp"], calls["pp"]) and np.array_equal(got["problem"], np.arange(1000) * 30 + 7)
    monkeypatch.setattr(bench, "DUMP_BYTES", 12 * 1024 + 100 * 15 * 8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), calls, np.arange(1000))
    a, b = (np.load(str(tmp_path / d / "problem.npy")) for d in ("a", "b"))
    assert len(a) == 100 and np.array_equal(a, b) and np.all(np.diff(a) > 0)
    assert np.array_equal(np.load(str(tmp_path / "a" / "allele1.npy")), a)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES


def test_reference_arm_line():
    d = _line("r1_bench_reference.json")
    assert d["impl"] == "reference" and BASE - {"gpu_launches"} <= set(d)
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    own = _line("r1_bench.json")
    assert (d["metric"], d["unit"], d["higher_is_better"]) == (own["metric"], own["unit"], own["higher_is_better"])


@pytest.mark.parametrize("name", ["r2_bench.json", "r2_bench_2gpu.json", "r2_bench_4gpu.json", "r2_bench_8gpu.json",
                                  "r2_bench_cohort10000.json"])
def test_round2_lines(name):
    """this round's lines: per-run roofline counters (not literals), distinct batches, the reference's own code as the
    CPU arm with a call-by-call parity check, the from-BAM leg"""
    d = _line(name)
    assert BASE <= set(d) and d["metric"] == "loci genotyped/sec" and d["value"] > 1e6 * d["n_gpus"]
    assert d["scaling"] == ("strong" if "cohort10000" in name else "weak")
    r = d["roofline"]
    assert r["calibration"] == "current" and 0.5 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert 2.0 < r["alu_lane_instr_per_executed_cell"] < 4.0 and r["traffic"] > 1e9
    assert "nothing is replayed" in d["config"]["l2"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 5e7 and 0 < e["value"] < d["value"] and e["transfer"] in ("bytes", "packed4")
    if name == "r2_bench.json":
        b = d["cpu_baseline"]
        same, total = b["identical_to_gpu"].split()[0].split("/")
        assert b["kind"] == "reference" and same == total and int(total) >= 390
        s = d["roofline_grid_stress"]
        assert s["points"] == 32032000 and s["kernel_ms"] < 0.6 and s["traffic"] < 8 * s["points"]
        f = d["from_bam"]
        assert f["gpu_ingest"] is True and f["value"] > 10 * 355 and f["reference"]["identical_to_gpu"].startswith("240/240")
        ref = _line("r2_bench_reference.json")
        assert ref["impl"] == "reference" and abs(ref["value"] / b["value"] - 1) < 0.15      # the arm is repeatable
