"""bench.py's output contract on the CPU arm (`--impl reference`): one JSON line with the keys the driver reads.

The GPU arm prints the same keys plus `roofline` (checked on the GPU box by the driver's own run); here the reference
arm is run at a toy size so that the line's shape, the exact step count and the rank-0-only rule are covered.
On the GPU arm, `--dump-outputs` is checked for identical outputs from two runs with the same arguments.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "cpu_baseline", "e2e", "gpu_launches", "impl"]


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample", "48",
           "--ntrain", "96", "--pop", "256", "--dim", "6", "--obj", "3", *args]
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1
    assert d["higher_is_better"] is True and d["unit"] == "candidates/s" and d["value"] > 0
    assert d["config"]["workload"].startswith("NSGA2 surrogate generation")
    cb = d["cpu_baseline"]
    has_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "dmosopt"))
    assert cb["kind"] == ("reference" if has_ref else "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_falls_back_to_the_port_without_the_reference_package(tmp_path):
    r = _run({"DMOSOPT_REF": str(tmp_path)})  # an empty directory: no dmosopt package there, and baseline/_ref is not consulted
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["cpu_baseline"]["kind"] == "port"


def test_reference_arm_other_ranks_stay_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, args=("--gpus", "2"))
    assert r.returncode == 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(tmp_path):
    """--dump-outputs: the last timed step's population, ranks and hypervolume as float64 .npy files, identical for two runs
    with the same arguments; --steps is the number of timed steps."""
    args = ["--steps", "3", "--warmup", "1", "--pop", "512", "--dim", "6", "--obj", "3", "--ntrain", "128", "--e2e-steps", "1",
            "--no-cpu-baseline", "--no-sort-hv"]
    dumps = []
    for run in ("a", "b"):
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / run)]
        r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
        assert d["steps"] == 3 and d["warmup"] == 1
        dumps.append({f.stem: np.load(f) for f in sorted((tmp_path / run).iterdir())})
    a, b = dumps
    assert sorted(a) == ["hypervolume", "population_x", "population_y", "rank"]
    assert a["population_x"].shape == (512, 6) and a["population_y"].shape == (512, 3) and a["rank"].shape == (512,)
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["hypervolume"][0] == d["hypervolume"] > 0
    for k in a:
        assert np.array_equal(a[k], b[k]), k
