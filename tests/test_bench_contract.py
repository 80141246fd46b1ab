"""bench.py keeps the driver's contract: exactly one JSON line on stdout with the required keys.
The reference arm runs on CPU (here); the GPU arm is exercised on a small workload under -m gpu."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _one_json_line(cmd, timeout):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + cmd, capture_output=True,
                       text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    return json.loads(lines[0])


def test_reference_arm_contract():
    d = _one_json_line(["--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-n", "3000"], 300)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "forceatlas_pair_interactions_per_sec" and d["unit"] == "pair-interactions/s"
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["config"]["workload"].startswith("config4")


def test_dump_outputs_samples_rows_above_the_budget(tmp_path, monkeypatch):
    import bench
    x = np.arange(2000.0).reshape(1000, 2)
    bench.dump_outputs(str(tmp_path / "all"), {"coords": x, "forces": -x})
    assert np.array_equal(np.load(tmp_path / "all" / "coords.npy"), x)
    assert np.array_equal(np.load(tmp_path / "all" / "forces.npy"), -x)
    assert not (tmp_path / "all" / "rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 40)
    bench.dump_outputs(str(tmp_path / "a"), {"coords": x, "forces": -x})
    bench.dump_outputs(str(tmp_path / "b"), {"coords": x, "forces": -x})
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.shape == (100,) and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "coords.npy"), x[rows.astype(np.int64)])
    assert np.array_equal(np.load(tmp_path / "a" / "forces.npy"), -x[rows.astype(np.int64)])


@pytest.mark.gpu
def test_gpu_arm_contract(tmp_path):
    d = _one_json_line(["--steps", "3", "--warmup", "3", "--n", "40000", "--attr-n", "150000", "--galerkin-n", "60000",
                        "--no-refhier", "--heldout-n", "60000", "--heldout-rmat", "14",
                        "--dump-outputs", str(tmp_path)], 600)
    assert BASE_KEYS <= set(d)
    assert {"roofline", "clocks", "gpu_launches", "embed", "fp32"} <= set(d)
    assert d["dtype"] == "f64" and d["scaling"] == "strong" and d["n_gpus"] == 1
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in d["roofline"]
    assert 0 < d["roofline"]["frac"] < 1.2
    assert d["gpu_launches"] >= 3 * d["steps"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["parity_ok"] and d["parity_max_err"] < 1e-10 and d["parity_rows_checked"] >= 32
    x, f = np.load(tmp_path / "coords.npy"), np.load(tmp_path / "forces.npy")
    assert x.dtype == f.dtype == np.float64 and x.shape == f.shape and x.shape[1] == 2
    assert np.isfinite(x).all() and np.isfinite(f).all()
