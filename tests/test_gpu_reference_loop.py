"""The reference's own results against the GPU plugins on hardware, and the plain-C host of include/dmosopt_b200.h executed
on the GPU.

The reference's results come from tests/golden/reference_loop.npz (written by tests/golden/make_golden.py with dmosopt
importable): three generations of its NSGA2 and its controller helpers (MOASMO.get_best, MOEA.get_duplicates /
crowding_distance_metric, hv.AdaptiveHyperVolume) on seeded inputs.
"""

import os
import shutil
import subprocess
import sys
import types

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_and_plugin_nsga2_agree_on_a_generation():
    """Same initial state and the same offspring: the reference's NSGA2.update_strategy (dda_ens + sortMO on the CPU)
    and the GPU plugin keep the same survivors, in the same order, with the same ranks."""
    import dmosopt_b200 as b2

    g = load_golden("reference_loop")
    x0, y0 = g["nsga2_x0"], g["nsga2_y0"]
    pop, d = x0.shape
    M = y0.shape[1]
    bounds = np.column_stack((np.zeros(d), np.ones(d)))

    def f(x):
        return np.column_stack((x[:, 0] + x[:, 3:].sum(1) * 0.1, (1 - x[:, 0]) * (1 + x[:, 1]), x[:, 2] ** 2 + 0.5 * x[:, 1]))

    bo = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=None, distance_metric=None)
    bo.initialize_strategy(x0.astype(np.float32), y0.copy(), bounds, np.random.default_rng(1))
    assert np.array_equal(g["nsga2_init_rank"], bo.state.rank)
    for gi in range(3):
        x_gen = g[f"nsga2_g{gi}_xgen"]  # the reference's own offspring of this generation
        bo.update(x_gen, f(x_gen), {"crossover_indices": g[f"nsga2_g{gi}_cidx"], "mutation_indices": g[f"nsga2_g{gi}_midx"]})
        assert np.array_equal(g[f"nsga2_g{gi}_rank"], np.asarray(bo.state.rank)), gi
        assert np.array_equal(g[f"nsga2_g{gi}_py"], np.asarray(bo.state.population_obj)), gi


def test_plain_c_host_runs_the_resident_step_on_the_gpu(tmp_path):
    """examples/nsga2_step.c: gcc -std=c99 against include/dmosopt_b200.h, linked with the in-tree library, executed."""
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    libdir = os.path.join(ROOT, "dmosopt_b200")
    exe = str(tmp_path / "nsga2_step")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "nsga2_step.c"),
                        "-L", libdir, "-ldmosopt_b200", f"-Wl,-rpath,{libdir}", "-lm", "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout + run.stderr
    lines = [ln for ln in run.stdout.splitlines() if ln.startswith("generation")]
    assert len(lines) == 5
    hv = [float(ln.rsplit(" ", 1)[1]) for ln in lines]
    assert all(b >= a - 1e-12 for a, b in zip(hv, hv[1:])), hv  # elitist survival: the hypervolume never shrinks


def _standin_package(monkeypatch, name):
    """A package shaped like dmosopt's MOEA / indicators / dda / hv modules whose helpers fail when called: whatever
    answers after install() was routed to the GPU library."""

    def unrouted(*args, **kwargs):
        raise AssertionError("stand-in helper called: install() did not route it")

    class AdaptiveHyperVolume:
        def __init__(self, ref_point, dimension_threshold_exact=10):
            self.ref_point = np.asarray(ref_point, dtype=np.float64)
            self.n_objectives = len(ref_point)
            self.dimension_threshold_exact = dimension_threshold_exact

        compute_hypervolume = unrouted

    mods = {}
    for sub, attrs in (("MOEA", ("get_duplicates", "remove_duplicates", "sortMO", "orderMO", "remove_worst", "crowding_distance_metric", "dda_ens")),
                       ("indicators", ("crowding_distance_metric", "euclidean_distance_metric")), ("dda", ("dda_ens",)), ("hv", ())):
        m = types.ModuleType(f"{name}.{sub}")
        for a in attrs:
            setattr(m, a, unrouted)
        mods[sub] = m
    mods["hv"].AdaptiveHyperVolume = AdaptiveHyperVolume
    monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
    for sub, m in mods.items():
        monkeypatch.setitem(sys.modules, f"{name}.{sub}", m)
    return mods


def test_install_routes_controller_helpers_to_the_gpu_with_identical_results(monkeypatch):
    """dmosopt_b200.install(): MOASMO.get_best (duplicates + sortMO, MOASMO.py:581-639), the resample helpers
    (MOASMO.py:441-448) and the termination hypervolume (hv.py:123-189) give the reference's own results once routed
    to the GPU, and uninstall() restores the module attributes."""
    import dmosopt_b200 as b2
    from dmosopt_b200 import _lib

    g = load_golden("reference_loop")
    x, y, x0, ref_pt = g["help_x"], g["help_y"], g["help_x0"], g["help_ref"]
    n = x.shape[0]
    mods = _standin_package(monkeypatch, "dmosopt_standin")
    rMOEA, rhv = mods["MOEA"], mods["hv"]
    originals = {a: getattr(rMOEA, a) for a in ("get_duplicates", "sortMO", "crowding_distance_metric", "dda_ens")}
    launches0 = _lib.launch_count()
    patched = b2.install("dmosopt_standin")
    try:
        assert any(name.endswith("get_duplicates") for name in patched)
        # MOASMO.get_best without constraints or epochs: duplicates of y dropped, then the rank-0 rows of sortMO's order
        dup_y = rMOEA.get_duplicates(y)
        xs, ys, rank, _, perm = rMOEA.sortMO(x[~dup_y], y[~dup_y], return_perm=True)
        dup_gpu = rMOEA.get_duplicates(x, x0)
        y_tf = y[np.r_[0:50, 51:400, 401:n]]  # tie-free columns: with exact ties the reference's own crowding depends on argsort's order
        cd_gpu = rMOEA.crowding_distance_metric(y_tf)
        hv_gpu = rhv.AdaptiveHyperVolume(ref_pt).compute_hypervolume(y[:300])
    finally:
        b2.uninstall()
    assert _lib.launch_count() > launches0
    assert all(getattr(rMOEA, a) is fn for a, fn in originals.items())  # restored
    assert np.array_equal(xs[rank == 0], g["help_best_x"]) and np.array_equal(ys[rank == 0], g["help_best_y"])
    assert np.array_equal(np.asarray(perm), g["help_best_perm"])
    assert np.array_equal(g["help_dup"], dup_gpu) and g["help_dup"].sum() == 40
    assert np.array_equal(g["help_cd"], cd_gpu)  # float64 bit-exact crowding (tie-free columns)
    hv_ref = float(g["help_hv"])
    assert abs(hv_gpu - hv_ref) <= 1e-9 * abs(hv_ref)
