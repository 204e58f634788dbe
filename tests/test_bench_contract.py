"""The driver-facing contract of `bench.py --impl reference` (the CPU arm), checked without a GPU on a small grid:
one JSON line with the metric / unit / config of the GPU arm, `impl`, `cpu_baseline` {value, unit, cores, kind, sample}
and `e2e` {value, unit, h2d_bytes_per_step, d2h_bytes_per_step}; under torchrun only rank 0 works.  --dump-outputs
writes the vectors the timed path computed, in both arms (the GPU arm against the reference arm on a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from tests.conftest import ROOT


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--nx", "32",
                           "--cpu-nx", "32", "--steps", "2", "--warmup", "1", *args],
                          capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "apply_inverse_per_s" and d["unit"] == "1/s"
    assert d["higher_is_better"] is True and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1e3 / d["value"]) < 1e-9 * d["ms_per_step"]
    assert "workload" in d["config"] and "32^3" in d["config"]["workload"]
    assert d["config"]["same_config"] is True and d["config"]["extrapolated"] is False
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["unit"] == "1/s" and cb["value"] == d["value"]
    assert "F-matrix ordering" in cb["sample"] and "32^3" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "1/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    g = d["gmres"]
    assert g["converged"] and g["iterations"] > 0 and g["explicit_rel_residual"] < 1e-6 and len(g["history_first15"]) > 1


def test_reference_arm_other_ranks_exit_without_work():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2", "--no-solve")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=60)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_reference_arm_dumps_its_outputs(tmp_path):
    r = _run(None, "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["apply_inverse_x.npy", "gmres_x.npy"]
    A, _, _, b, _ = bench.problem(32)
    x, xs = np.load(tmp_path / "apply_inverse_x.npy"), np.load(tmp_path / "gmres_x.npy")
    assert x.dtype == xs.dtype == np.float64 and x.shape == xs.shape == (A.shape[0],)
    assert np.all(np.isfinite(x)) and np.linalg.norm(x) > 0
    assert np.linalg.norm(A @ xs - b) <= 1e-7 * np.linalg.norm(b)


def test_dump_outputs_samples_the_same_rows_of_every_vector(tmp_path):
    n = 10000
    v = {"a": np.arange(n, dtype=np.float64), "b": 2 * np.arange(n, dtype=np.float32)}
    bench.dump_outputs(str(tmp_path / "full"), v)
    assert sorted(os.listdir(tmp_path / "full")) == ["a.npy", "b.npy"]
    assert np.array_equal(np.load(tmp_path / "full" / "a.npy"), v["a"])
    assert np.load(tmp_path / "full" / "b.npy").dtype == np.float64
    limit = 4096 + 3 * 8 * 1000        # room for 1000 rows of a, b and the row indices
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), v, limit=limit)
    s1, s2 = tmp_path / "s1", tmp_path / "s2"
    assert sum(f.stat().st_size for f in s1.iterdir()) <= limit
    rows = np.load(s1 / "rows.npy")
    assert len(rows) == 1000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(s1 / "a.npy"), rows) and np.array_equal(np.load(s1 / "b.npy"), 2 * rows)
    for name in ("rows.npy", "a.npy", "b.npy"):
        assert np.array_equal(np.load(s1 / name), np.load(s2 / name))


@pytest.mark.gpu
def test_gpu_arm_dumps_the_apply_inverse_the_reference_arm_computes(tmp_path):
    """Both arms on the same small workload: the dumped vectors are the ApplyInverse and the GMRES solution of the
    same right-hand side.  (The bound leaves room for the rounding error of the FP64 sparse-LU reference arm; a wrong
    or stale vector is O(1) away.)"""
    args = ["--nx", "32", "--sx", "8", "--cx", "2", "--steps", "3", "--warmup", "1"]
    g = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / "gpu")],
                       capture_output=True, text=True, timeout=900)
    assert g.returncode == 0, g.stderr[-2000:]
    d = json.loads([ln for ln in g.stdout.splitlines() if ln.startswith("{")][0])
    assert d["steps"] == 3
    r = _run(None, "--sx", "8", "--cx", "2", "--steps", "1", "--dump-outputs", str(tmp_path / "ref"))
    assert r.returncode == 0, r.stderr[-2000:]
    A, _, _, b, _ = bench.problem(32)
    xg, xr = np.load(tmp_path / "gpu" / "apply_inverse_x.npy"), np.load(tmp_path / "ref" / "apply_inverse_x.npy")
    assert xg.shape == (A.shape[0],) and np.linalg.norm(xg - xr) <= 1e-9 * np.linalg.norm(xr)
    assert np.linalg.norm(A @ np.load(tmp_path / "gpu" / "gmres_x.npy") - b) <= 1e-7 * np.linalg.norm(b)
