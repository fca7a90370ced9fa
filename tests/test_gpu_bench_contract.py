"""bench.py prints ONE JSON line with the keys the driver reads (small --reads so it runs in seconds)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _run(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=280, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().split("\n") if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_bench_line_contract():
    j = _run("--reads", "200000", "--steps", "3", "--warmup", "3", "--recover-paths", "1", "--ref-sample", "4000",
             "--bam-reads", "50000")
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert key in j, key
    assert j["n_gpus"] == 1 and j["steps"] == 3 and j["value"] > 0 and j["gpu_launches"] > 0
    assert j["vs_baseline"] is None and j["data"] == "synthetic" and "workload" in j["config"]
    assert j["e2e"]["value"] > 0 and j["e2e"]["h2d_bytes_per_step"] > 0 and j["e2e"]["d2h_bytes_per_step"] > 0
    assert j["e2e"]["value"] < j["value"]                       # the end-to-end number includes the copies
    r = j["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    c = j["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    assert j["recovery"]["haplotypes"] >= 0
    assert j["parity_probe"]["ok"] is True and j["parity_probe"]["rows_equal"] and j["parity_probe"]["band_sum"] > 0
    b = j["e2e_bam"]
    assert b["reads_per_s"] > 0 and b["same_totals_as_packed_arrays"] and 0 < b["gpu_share"] < 1
    assert set(b["stage_seconds"]) >= {"read", "inflate", "scan", "walk", "gather", "gpu_ingest"}


def _dumped(d):
    names = sorted(os.listdir(d))
    assert names == ["band.npy", "band_rows.npy", "totals.npy"]
    assert sum(os.path.getsize(os.path.join(d, n)) for n in names) <= 64 << 20
    return {n[:-4]: np.load(os.path.join(d, n)) for n in names}


def test_dump_outputs(tmp_path):
    """--dump-outputs writes the last timed step's totals and counts, identical from run to run."""
    args = ("--reads", "200000", "--steps", "2", "--warmup", "1", "--recover-paths", "0", "--no-cpu-baseline",
            "--bam-reads", "0")
    j = _run(*args, "--dump-outputs", str(tmp_path / "a"))
    _run(*args, "--dump-outputs", str(tmp_path / "b"))
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert a["band"].dtype == np.float32 and a["totals"].dtype == np.float64 and a["band_rows"].dtype == np.float64
    assert j["steps"] == 2 and j["e2e"]["steps"] == 2
    assert a["band"].shape == (j["parity_probe"]["rows"], j["band_w"], 7, 7)
    assert np.array_equal(a["band_rows"], np.arange(j["parity_probe"]["rows"]))
    assert a["totals"][1] == j["observations_per_step"] == j["parity_probe"]["n_crumbs"]
    assert a["band"].sum(dtype=np.float64) == j["parity_probe"]["band_sum"]
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_dump_outputs_samples_a_large_band(tmp_path):
    """A band over 64 MB (80 SNPs per read: band_w 110, 206 MB) is cut to a seeded sample of whole rows."""
    j = _run("--workload", "mid", "--reads", "20000", "--steps", "1", "--warmup", "1", "--recover-paths", "0",
             "--no-cpu-baseline", "--bam-reads", "0", "--dump-outputs", str(tmp_path))
    d = _dumped(tmp_path)
    rows = d["band_rows"].astype(np.int64)
    assert 0 < len(rows) < j["parity_probe"]["rows"] and np.all(np.diff(rows) > 0)
    assert d["band"].shape == (len(rows), j["band_w"], 7, 7) and d["band"].sum() > 0
    assert d["totals"][1] == j["observations_per_step"]


def test_reference_arm_contract():
    j = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-sample", "3000")
    assert j["impl"] == "reference" and j["value"] > 0 and j["gpu_launches"] == 0
    assert j["cpu_baseline"]["kind"] == "port" and j["e2e"]["h2d_bytes_per_step"] == 0
