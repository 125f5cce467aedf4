"""bench.py prints ONE JSON line with the keys the driver reads (metric / value / unit / roofline / e2e / cpu_baseline /
clocks / gpu_launches); the reference arm runs without a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    """--impl reference: the reference's own CPU implementation (the unmodified Python modules when baseline/_ref is
    installed, else the C port), same metric / unit / config as the main arm"""
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"], 900)
    assert d["impl"] == "reference" and d["metric"] == "edge_evals_per_s" and d["unit"] == "edges/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_main_arm_line():
    d = _run(["--steps", "3", "--warmup", "3", "--no-extras"], 900)
    assert d["metric"] == "edge_evals_per_s" and d["unit"] == "edges/s" and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3
    assert d["value"] > 1e8 and d["ms_per_step"] > 0 and d["scaling"] == "weak" and d["dtype"] == "f32" and d["vs_baseline"] is None
    r = d["roofline"]
    assert r["bound"] == "fp32" and r["unit"] == "TFLOP/s" and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["value"] < d["value"] * 1.05 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] == 3 and d["clocks"]["sm_mhz"] > 0 and isinstance(d["clocks"]["reasons"], list)
    assert "workload" in d["config"] and d["data"] == "synthetic"


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs writes the last timed step's records and chains as float64 .npy files; two runs with the same
    arguments write the same arrays"""
    import numpy as np
    for run in ("a", "b"):
        d = _run(["--steps", "2", "--warmup", "0", "--no-extras", "--dump-outputs", str(tmp_path / run)], 900)
        assert d["steps"] == 2
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and {"chain.npy", "cost.npy", "status.npy", "query.npy"} <= set(names)
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and len(a) == 4096 and np.array_equal(a, b), n
    assert (np.load(tmp_path / "a" / "status.npy") == 0).mean() > 0.9
