#!/usr/bin/env python
"""Headline benchmark: candidate-evaluations / second of one surrogate generation step.

Workload (BASELINE.json metric): NSGA-II generation at pop = 65 536, dim = 30, 3 objectives, exact-GP surrogate with
N_train = 4096 (fixed initial theta: ConstantKernel(1) * Matern(l=0.5, nu=2.5) + WhiteKernel(1e-6), BASELINE.md
section 3), synthetic DTLZ2-shaped training targets.  One *step* = one generation of MOASMO.optimize's loop
(dmosopt/MOASMO.py:92-122) including the per-generation termination hypervolume (hv_termination.py:1093-1106):

    tournament -> SBX / polynomial mutation (P ~ pop offspring) -> GP posterior mean + variance of the offspring
    -> non-dominated rank of the merged 2*pop set + stable truncation to pop -> exact hypervolume of the population

  value : the step with the population resident in HBM (C-ABI calls on device buffers)
  e2e   : the same step through the reference-facing plugin API (NSGA2.generate / GPR_Matern.predict /
          NSGA2.update / Hypervolume.do) with HOST buffers, host<->device copies inside the timed region

  python bench.py --gpus N --steps K --warmup W            # this build (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference ...                     # CPU arm: the UNMODIFIED reference (baseline/_ref) on the host
                                                           # cores at a bounded population; the oracle port if it is absent
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's population as DIR/<name>.npy

Extra legs printed in the same JSON line (rank 0, N = 1): `hv_contrib` (the second half of BASELINE's metric: expected-HV-
improvement contributions / s, A17) and `sort_hv` (rank + truncation + hypervolume on SURVEY section 8d's three objective
sets: GP-predicted, uniform, near-single-front sphere).
"""

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "candidate-evals/sec (GP+sort+HV) pop=65536 dim=30 obj=3"
UNIT = "candidates/s"
REF_DIR = os.environ.get("DMOSOPT_REF") or os.path.join(ROOT, "baseline", "_ref")

# DRAM bytes of one gp_var launch from the committed `ncu --set full` captures (profiles/), keyed by
# (kernel version, pop, d, M, N); null for anything else -- the number is not re-measured inside the timed run
# (a run under ncu is never a bench value).
NCU_TRAFFIC = {
    ("v3", 65536, 30, 3, 4096): ("profiles/r2_gp_var_tc3_kernel_details.txt", 5.134091e9 + 16.331008e6),
    ("v2", 65536, 30, 3, 4096): ("profiles/r1_gp_var_tc2_kernel_details.txt", 22.553779e9 + 7.566592e6),
}


def workload(pop, d, M, N, seed=20260921 + 2):
    rng = np.random.default_rng(seed)
    xlb, xub = np.zeros(d), np.ones(d)
    Xtr = rng.random((N, d))
    g = ((Xtr[:, M - 1 :] - 0.5) ** 2).sum(axis=1)
    Ytr = np.ones((N, M)) * (1.0 + g)[:, None]
    for i in range(M):  # DTLZ2 (dmosopt/benchmarks/moo_benchmarks.py:59-94), vectorised
        for j in range(M - 1 - i):
            Ytr[:, i] *= np.cos(0.5 * np.pi * Xtr[:, j])
        if i > 0:
            Ytr[:, i] *= np.sin(0.5 * np.pi * Xtr[:, M - 1 - i])
    X0 = rng.random((pop, d))
    return dict(rng=rng, xlb=xlb, xub=xub, Xtr=Xtr, Ytr=Ytr, X0=X0)


def objective_sets(n, M, seed=20260921 + 7):
    """SURVEY section 8d: objective sets for the sort / HV legs besides the GP-predicted one."""
    rng = np.random.default_rng(seed)
    uni = rng.random((n, M))  # many fronts
    v = np.abs(rng.standard_normal((n, M)))
    sph = v / np.linalg.norm(v, axis=1, keepdims=True) * (1.0 + 0.01 * rng.random((n, 1)))  # DTLZ2 sphere x (1 + 0.01 u)
    return {"uniform": uni, "sphere": sph}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md).

    The sampler is started before the warm-up steps (spawning nvidia-smi takes longer than a short timed region) and
    writes time-stamped rows every 50 ms; ``stop`` keeps the rows that fall inside the marked region.  If the region was
    shorter than one sampling period the rows of the warm-up steps just before it (same load) are used and the
    ``window`` field says so.
    """

    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.f = tempfile.TemporaryFile(mode="w+")  # the benchmark writes nothing into the tree (it may be read-only)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.device)],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self._terminate)  # no sampler outlives a run that fails before stop()
        except Exception:
            self.proc = None

    def _terminate(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def mark_begin(self):
        import datetime

        self.t0 = datetime.datetime.now()

    def mark_end(self):
        import datetime

        self.t1 = datetime.datetime.now()

    def stop(self):
        import datetime

        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.06)  # one more sampling period so that a row stamped inside the region is flushed
        self._terminate()
        self.f.seek(0)
        lines = self.f.readlines()
        self.f.close()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f")
                rows.append((ts, float(parts[2]), float(parts[3]), [nm for nm, val in zip(names, parts[6:10]) if val.lower().startswith("active")],
                             float(parts[4])))
            except ValueError:
                continue
        window = "timed region"
        sel = [r for r in rows if self.t0 is not None and self.t1 is not None and self.t0 <= r[0] <= self.t1]
        if not sel and self.t1 is not None:  # region shorter than a sampling period: the last rows taken under the same load
            sel = [r for r in rows if r[0] <= self.t1][-3:]
            window = "steps immediately before the timed region (region shorter than one 50 ms sample)"
        if not sel and rows and self.t1 is not None:  # nvidia-smi came up late: the row nearest to the region
            sel = [min(rows, key=lambda r: abs((r[0] - self.t1).total_seconds()))]
            window = "nearest sample to the timed region (nvidia-smi started late)"
        if sel:
            reasons = sorted({nm for r in sel for nm in r[3]})
            out = {"sm_mhz": float(np.median([r[1] for r in sel])), "sm_max_mhz": float(max(r[2] for r in sel)), "reasons": reasons,
                   "samples": len(sel), "window": window, "power_w_median": float(np.median([r[4] for r in sel]))}
        return out


# ----------------------------------------------------------------------------------------------------------------------
# CPU arms
def use_all_host_threads():
    """BLAS / OpenMP pools to every host core (torchrun exports OMP_NUM_THREADS=1).  Returns the thread count of the BLAS
    pool NumPy / SciPy compute with (the only multi-threaded part of the reference path; the OpenBLAS build in this image
    stops at 64 threads) -- the same number whether or not torch's own pools are loaded in the process."""
    n = os.cpu_count() or 1
    try:
        import threadpoolctl

        threadpoolctl.threadpool_limits(limits=n)
        info = threadpoolctl.threadpool_info()
        blas = [p.get("num_threads", 1) for p in info if p.get("user_api") == "blas" and "numpy" in str(p.get("filepath", "")) + str(p.get("prefix", ""))]
        if not blas:
            blas = [p.get("num_threads", 1) for p in info if p.get("user_api") == "blas"]
        return int(min(blas)) if blas else n
    except Exception:
        return n


def have_reference():
    return os.path.isdir(os.path.join(REF_DIR, "dmosopt"))


def fit_sklearn_fixed(w, M):
    """The three scikit-learn regressors of GPR_Matern at the reference's initial theta, optimizer=None
    (dmosopt/model.py:1224-1251 with the SCE-UA search switched off: it cannot run at N_train = 4096, BASELINE.md section 3)."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import ConstantKernel, Matern, WhiteKernel

    kernel = ConstantKernel(1, (1e-4, 1e3)) * Matern(length_scale=0.5, length_scale_bounds=(1e-3, 100.0), nu=2.5) + WhiteKernel(
        noise_level=1e-6, noise_level_bounds=(1e-9, 1e-2))
    x = (w["Xtr"] - w["xlb"]) / (w["xub"] - w["xlb"])
    return [GaussianProcessRegressor(kernel=kernel, optimizer=None, normalize_y=True).fit(x, w["Ytr"][:, i]) for i in range(M)]


class ReferenceGeneration:
    """One NSGA-II surrogate generation through the UNMODIFIED reference (baseline/_ref): dmosopt.NSGA2.NSGA2
    generate / update (tournament, SBX, mutation, dda_ens, sortMO), dmosopt.model.GPR_Matern.predict (scikit-learn) and
    dmosopt.indicators.Hypervolume -- at a bounded population against the full N_train model.

    Only the construction of GPR_Matern is bypassed: its constructor always runs the SCE-UA hyper-parameter search
    (model.py:1238-1243), which is not part of the per-generation path and does not terminate at N_train = 4096; the
    instance is given the same scikit-learn regressors with the initial theta (``smlist``) and every per-generation
    method then runs as the reference wrote it.
    """

    def __init__(self, w, pop_s, d, M, smlist, seed=1):
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        from dmosopt import NSGA2 as rN
        from dmosopt import indicators as rind
        from dmosopt import model as rmodel

        sm = rmodel.GPR_Matern.__new__(rmodel.GPR_Matern)
        sm.nInput, sm.nOutput, sm.xlb, sm.xub, sm.xrg = d, M, w["xlb"], w["xub"], w["xub"] - w["xlb"]
        sm.logger, sm.return_mean_variance, sm.smlist = None, False, smlist
        self.sm = sm
        x0 = w["X0"][:pop_s]
        y0 = sm.evaluate(x0).astype(np.float32)
        self.opt = rN.NSGA2(popsize=pop_s, nInput=d, nOutput=M, model=rmodel.Model(objective=sm), distance_metric=None)
        self.opt.initialize_strategy(x0, y0, np.column_stack((w["xlb"], w["xub"])), np.random.default_rng(seed))
        ref = y0.max(axis=0).astype(np.float64) + 0.1 * (y0.max(axis=0) - y0.min(axis=0))
        self.hv = rind.Hypervolume(ref_point=ref)
        self.pop_s = pop_s

    def step(self):
        t = [time.perf_counter()]
        x_gen, st = self.opt.generate()  # MOASMO.py:105
        t.append(time.perf_counter())
        y, _ = self.sm.predict(x_gen)  # model.py:1254-1268 (mean and variance)
        t.append(time.perf_counter())
        self.opt.update(x_gen, y, st)  # MOASMO.py:116
        t.append(time.perf_counter())
        _, py = self.opt.population_objectives
        self.hv.do(py.astype(np.float64))  # hv_termination.py:1093-1106
        t.append(time.perf_counter())
        dt = np.diff(t)
        return {"variation": dt[0], "gp": dt[1], "sort": dt[2], "hv": dt[3], "total": t[-1] - t[0], "children": x_gen.shape[0]}


class PortGeneration:
    """The same generation restated on the CPU (oracle/, kind = "port"): used when the reference package is not shipped."""

    def __init__(self, w, pop_s, d, M, N):
        from oracle import gp

        self.w, self.pop_s, self.d = w, pop_s, d
        self.st = gp.fit_fixed(w["Xtr"], w["Ytr"], w["xlb"], w["xub"], 1.0, 0.5, 1e-6)

    def step(self):
        from oracle import dda, gp, hv, moea

        rng = np.random.default_rng(1)
        x_par = rng.random((self.pop_s, self.d))
        y_par = gp.predict(self.st, x_par)[0]
        x_gen = np.clip(x_par + 0.05 * rng.standard_normal((self.pop_s, self.d)), 0, 1)
        t0 = time.perf_counter()
        y_gen, _ = gp.predict(self.st, x_gen)
        t1 = time.perf_counter()
        X, Y = np.vstack((x_gen, x_par)), np.vstack((y_gen, y_par))
        xs, ys, rank, perm = moea.remove_worst(X, Y, self.pop_s, None, rank_fn=dda.rank_canonical)
        t2 = time.perf_counter()
        hv.hypervolume(ys, Y.max(axis=0) + 0.1)
        t3 = time.perf_counter()
        return {"variation": 0.0, "gp": t1 - t0, "sort": t2 - t1, "hv": t3 - t2, "total": t3 - t0, "children": self.pop_s}


def cpu_arm(w, pop_s, d, M, N, smlist=None):
    """(stepper, kind, sample text)."""
    pop = w["X0"].shape[0]
    if have_reference():
        sm = smlist if smlist is not None else fit_sklearn_fixed(w, M)
        return (ReferenceGeneration(w, pop_s, d, M, sm), "reference",
                f"one NSGA-II surrogate generation of the unmodified reference (baseline/_ref: NSGA2.generate/update, GPR_Matern.predict, "
                f"indicators.Hypervolume) at pop={pop_s} (of {pop}) against the full N_train={N} model, fixed theta")
    return (PortGeneration(w, pop_s, d, M, N), "port",
            f"one generation at pop={pop_s} (of {pop}) against the full N_train={N} model; oracle/ NumPy+BLAS port of the reference path "
            f"(reference package not shipped)")


def run_reference(args):
    """--impl reference: the CPU arm, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    pop, d, M, N = args.pop, args.dim, args.obj, args.ntrain
    w = workload(pop, d, M, N)
    cores = use_all_host_threads()
    gen, kind, sample = cpu_arm(w, args.cpu_sample, d, M, N)
    for _ in range(args.warmup):
        gen.step()
    ts = [gen.step() for _ in range(max(1, args.steps))]  # one bounded sample per step
    tot = float(np.mean([t["total"] for t in ts]))
    val = float(np.mean([t["children"] for t in ts])) / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(ts), "warmup": args.warmup,
        "ms_per_step": tot * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"NSGA2 surrogate generation pop={pop} dim={d} obj={M} N_train={N} (CPU arm: bounded sample pop={args.cpu_sample}, full model)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "breakdown_s": {k: float(np.mean([t[k] for t in ts])) for k in ("variation", "gp", "sort", "hv")}},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
class ResidentStep:
    """One NSGA-II surrogate generation with the population resident in HBM (C-ABI on device buffers)."""

    def __init__(self, L, gp_handle, pop, d, M, xlb, xub, x0, y0, rank0, ref, seed, world=1, rank=0, dist=None, torch=None):
        self.L, self.gp, self.pop, self.d, self.M = L, gp_handle, pop, d, M
        self.world, self.rank_id, self.dist, self.torch = world, rank, dist, torch
        self.cap = pop + 1
        DA = L.DeviceArray
        self.pop_x = DA((pop, d)).upload(x0)
        self.pop_y = DA((pop, M)).upload(y0)
        self.rank = DA((pop,), np.int32).upload(rank0.astype(np.int32))
        self.pool = DA((pop // 2,), np.int64)
        self.Xs = DA((self.cap + pop, d))
        self.Ys = DA((self.cap + pop, M))
        self.kind = DA((self.cap,), np.int32)
        self.perm = DA((pop,), np.int64)
        self.xlb, self.xub = DA((d,)).upload(xlb), DA((d,)).upload(xub)
        self.dic, self.dim = DA((d,)).upload(np.full(d, 1.0)), DA((d,)).upload(np.full(d, 20.0))
        self.ref = np.asarray(ref, dtype=np.float64)
        self.seed, self.stream = seed, 0
        self.nch = np.zeros(1, dtype=np.int64)
        self.hv = 0.0
        if world > 1:
            per = -(-self.cap // world)
            self.per = per
            # torch work is issued on the library's own stream (ExternalStream), so the all-gather is stream-ordered
            # with the kernels before and after it: no device-wide synchronisation, no staging copy
            self.ext = torch.cuda.ExternalStream(L.stream_ptr())
            self.t_mean = torch.zeros((per, M), dtype=torch.float64, device="cuda")
            self.t_var = torch.zeros((per, M), dtype=torch.float64, device="cuda")
            self.t_all = torch.empty((world * per, M), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()

    def step(self):
        import ctypes

        L, lib, ctx = self.L, self.L.load_library(), self.L.context()
        pop, d, M = self.pop, self.d, self.M
        chk = L._check
        out = ctypes.c_double(0.0)
        if self.world == 1:
            # one C call per generation: the fused resident step (include/dmosopt_b200.h, dmo_nsga2_step)
            chk(lib.dmo_nsga2_step(ctx, self.gp._h, self.pop_x.ptr, self.pop_y.ptr, self.rank.ptr, pop, d, M, 0.9, 0.1, 1.0 / d, self.dic.ptr,
                                   self.dim.ptr, self.xlb.ptr, self.xub.ptr, self.seed, self.stream + 1, self.precision, self.metric, 1, 1,
                                   self.ref.ctypes.data, self.nch.ctypes.data, ctypes.byref(out)), "nsga2_step")
            self.stream += 2
            self.hv = out.value
            return int(self.nch[0])
        torch = self.torch
        self.stream += 1
        chk(lib.dmo_tournament(ctx, self.rank.ptr, None, pop, pop // 2, self.seed, self.stream, self.pool.ptr, None), "tournament")
        self.stream += 1
        chk(lib.dmo_nsga2_generate(ctx, self.pop_x.ptr, pop, d, self.pool.ptr, pop // 2, pop, 0.9, 0.1, 1.0 / d, self.dic.ptr, self.dim.ptr,
                                   self.xlb.ptr, self.xub.ptr, self.seed, self.stream, self.Xs.ptr, self.kind.ptr, self.nch.ctypes.data, None), "generate")
        P = int(self.nch[0])
        per = self.per
        lo = min(self.rank_id * per, P)
        hi = min(lo + per, P)
        if hi > lo:  # this rank's row block of the offspring: posterior mean and variance
            chk(lib.dmo_gp_predict(ctx, self.gp._h, self.Xs.offset(lo * d), hi - lo, self.t_mean.data_ptr(), self.t_var.data_ptr(), self.precision), "gp_predict")
        with torch.cuda.stream(self.ext):
            self.dist.all_gather_into_tensor(self.t_all, self.t_mean)  # the one exchange step: predicted objectives (NCCL / NVLink)
        # stack the gathered children over the parents (NSGA2.py:205-206), rank + stable truncation, float32 state rounding
        L.memcpy(self.Ys.ptr, self.t_all.data_ptr(), P * M * 8)
        L.memcpy(self.Xs.offset(P * d), self.pop_x.ptr, pop * d * 8)
        L.memcpy(self.Ys.offset(P * M), self.pop_y.ptr, pop * M * 8)
        chk(lib.dmo_remove_worst(ctx, self.Xs.ptr, self.Ys.ptr, P + pop, d, M, self.metric, None, 0, pop, self.pop_x.ptr, self.pop_y.ptr,
                                 self.rank.ptr, self.perm.ptr), "remove_worst")
        L.round_f32(self.pop_y.ptr, pop * M)
        chk(lib.dmo_hypervolume_ranked(ctx, self.pop_y.ptr, pop, M, self.ref.ctypes.data, self.rank.ptr, ctypes.byref(out)), "hypervolume")
        self.hv = out.value
        return P


def dump_outputs(out_dir, rs, limit_bytes=64 << 20, seed=0):
    """What the timed step hands its caller after the last step -- the population (decision vectors, objectives, ranks)
    and its hypervolume -- as ``out_dir/<name>.npy`` in float64.  Above ``limit_bytes`` a fixed, seeded sample of
    population rows is written instead, with their indices in ``rows.npy``."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"population_x": rs.pop_x.download(), "population_y": rs.pop_y.download(), "rank": rs.rank.download().astype(np.float64)}
    row_bytes = 8 * sum(a[0].size for a in arrays.values())  # written as float64
    max_rows = max(1, (limit_bytes - 1024) // (row_bytes + 8))
    if rs.pop > max_rows:
        rows = np.sort(np.random.default_rng(seed).choice(rs.pop, size=max_rows, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    arrays["hypervolume"] = np.array([rs.hv], dtype=np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def time_device(L, fn, reps=3, warm=1):
    for _ in range(warm):
        fn()
    L.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    L.synchronize()
    return (time.perf_counter() - t0) / reps


def sort_hv_legs(L, pop, M, y_gp_merged, ref_gp):
    """rank + stable truncation (dmo_remove_worst) and exact hypervolume (dmo_hypervolume) of the merged 2*pop set, data
    resident, on SURVEY section 8d's three objective sets."""
    import ctypes

    lib, ctx = L.load_library(), L.context()
    n = 2 * pop
    sets = {"gp_predicted": (y_gp_merged, ref_gp)}
    for k, Y in objective_sets(n, M).items():
        sets[k] = (Y, Y.max(axis=0) + 0.1)
    out = {}
    d = 4
    Xd = L.DeviceArray((n, d)).upload(np.random.default_rng(0).random((n, d)))
    xo, yo = L.DeviceArray((pop, d)), L.DeviceArray((pop, M))
    rk, pm = L.DeviceArray((pop,), np.int32), L.DeviceArray((pop,), np.int64)
    for name, (Y, ref) in sets.items():
        Yd = L.DeviceArray((n, M)).upload(np.ascontiguousarray(Y[:n], dtype=np.float64))
        refc = np.ascontiguousarray(ref, dtype=np.float64)
        hv = ctypes.c_double(0.0)

        def do_sort():
            L._check(lib.dmo_remove_worst(ctx, Xd.ptr, Yd.ptr, n, d, M, L.METRIC_NONE, None, 0, pop, xo.ptr, yo.ptr, rk.ptr, pm.ptr), "remove_worst")

        def do_hv():
            L._check(lib.dmo_hypervolume(ctx, yo.ptr, pop, M, refc.ctypes.data, ctypes.byref(hv)), "hypervolume")

        t_sort = time_device(L, do_sort)
        t_hv = time_device(L, do_hv)
        ranks = rk.download()
        out[name] = {"n": n, "rank_truncate_ms": t_sort * 1e3, "hv_ms": t_hv * 1e3, "front0_in_population": int((ranks == 0).sum()),
                     "max_rank_kept": int(ranks.max()), "hv": hv.value,
                     # algorithmic bytes of the rank (SURVEY 8d): 4 n M read + 4 n written, vs the measured HBM peak
                     "rank_algorithmic_gbs": (4.0 * n * M + 4.0 * n) / t_sort / 1e9}
        Yd.free()
    return out


def run_ours(args):
    import dmosopt_b200 as b2
    from dmosopt_b200 import _lib as L
    from dmosopt_b200.indicators import Hypervolume

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = torch = None
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L.context(local_rank)
    # started now (spawning nvidia-smi can take longer than a short timed region); rows are time-stamped and filtered later
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    pop, d, M, N = args.pop, args.dim, args.obj, args.ntrain
    prec = {"auto": L.GP_AUTO, "tensor": L.GP_TENSOR, "fp64": L.GP_FP64}[args.precision]
    w = workload(pop, d, M, N)
    t0 = time.time()
    sm = b2.GPR_Matern(w["Xtr"], w["Ytr"], d, M, w["xlb"], w["xub"], optimizer=None, precision=args.precision)
    t_fit = time.time() - t0
    mdl = b2.Model(objective=sm)
    y0 = sm.evaluate(w["X0"]).astype(np.float32)
    ref = y0.max(axis=0).astype(np.float64) + 0.1 * (y0.max(axis=0) - y0.min(axis=0))
    peaks, peak_kind = load_peaks()
    auto = sm._gp.auto_info() if prec == L.GP_AUTO else None

    def barrier():
        L.synchronize()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ e2e: plugin API, host buffers
    from dmosopt_b200.parallel import ShardedSurrogate

    sm_e2e = ShardedSurrogate(sm, device=torch.device("cuda", local_rank)) if world > 1 else sm
    opt = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=mdl, distance_metric=None if args.distance_metric == "none" else args.distance_metric)
    opt.initialize_strategy(w["X0"], y0, np.column_stack((w["xlb"], w["xub"])), np.random.default_rng(args.seed))
    hv_ind = Hypervolume(ref_point=ref)

    def plugin_step():
        x_gen, st = opt.generate()  # MOASMO.py:105
        y_gen, y_var = sm_e2e.predict(x_gen)  # posterior mean AND variance, as the reference computes (model.py:1254-1268)
        opt.update(x_gen, y_gen, st)  # MOASMO.py:116
        _, py = opt.population_objectives  # termination criterion reads the population ... (MOASMO.py:93-97)
        return hv_ind.do(py.astype(np.float64)), x_gen.shape[0]  # ... and computes its hypervolume

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    for _ in range(min(args.warmup, 3) if args.e2e_warmup is None else args.e2e_warmup):
        plugin_step()
    barrier()
    h0, d0 = L.transfer_bytes()
    n_e2e = 0
    t0 = time.perf_counter()
    L.timer_begin()
    for _ in range(e2e_steps):
        _, P = plugin_step()
        n_e2e += P
    ms_e2e_dev = L.timer_end()
    barrier()
    t_e2e = max_over_ranks(time.perf_counter() - t0)
    h1, d1 = L.transfer_bytes()
    e2e_val = n_e2e / t_e2e

    # ------------------------------------------------------------------ value: resident step
    rank0 = opt.state.rank.copy()
    rs = ResidentStep(L, sm._gp, pop, d, M, w["xlb"], w["xub"], opt.state.population_parm, opt.state.population_obj.astype(np.float64), rank0, ref,
                      args.seed, world, rank, dist, torch)
    rs.precision = prec
    rs.metric = {"none": L.METRIC_NONE, "crowding": L.METRIC_CROWDING, "euclidean": L.METRIC_EUCLIDEAN}[args.distance_metric]
    for _ in range(args.warmup):
        rs.step()
    barrier()
    clocks.mark_begin()
    L.profile_enable(True)
    launches0 = L.launch_count()
    n_val = 0
    t0 = time.perf_counter()
    L.timer_begin()
    for _ in range(args.steps):
        n_val += rs.step()
    ms_dev = L.timer_end()
    barrier()
    clocks.mark_end()
    t_val = max_over_ranks(max(time.perf_counter() - t0, ms_dev * 1e-3))
    launches = L.launch_count() - launches0
    prof = L.profile_report()
    L.profile_enable(False)
    clk = clocks.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, rs)
    value = n_val / t_val
    refined = sm._gp.auto_info()["last_refined"] if prec == L.GP_AUTO else 0

    # ------------------------------------------------------------------ roofline of the dominant kernel (GP variance)
    var_ms, var_cnt = prof.get("gp_var", (0.0, 0))
    P_local = (n_val / args.steps) / world
    flops_per_launch = 2.0 * N * N * M * P_local  # SURVEY section 8d: GEMM form 2 N^2 M per candidate
    tensor_path = prec == L.GP_TENSOR or (prec == L.GP_AUTO and auto["var_tensor"])
    version = "v2" if os.environ.get("DMO_GP_TC") == "2" else "v3"
    roof = None
    if var_cnt:
        avg_s = var_ms * 1e-3 / var_cnt
        ach = flops_per_launch / avg_s / 1e12
        peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
        tr = NCU_TRAFFIC.get((version, pop, d, M, N)) if (tensor_path and world == 1) else None
        roof = {"bound": "tensor", "kernel": "gp_var (V = L^-1 K_*^T, column sums of V^2)", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": ach / peak, "traffic": tr[1] if tr else None, "traffic_source": tr[0] if tr else None,
                "peak_kind": f"bf16 dense, sustained, {peak_kind}", "avg_launch_ms": avg_s * 1e3, "flops_per_launch": flops_per_launch,
                "arithmetic": "tcgen05 split-fp16" if tensor_path else "float64 CUDA cores"}
    shares = {k: v[0] / (ms_dev if ms_dev > 0 else 1.0) for k, v in prof.items()}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ------------------------------------------------------------------ second half of the metric: HV contributions / s
    # (A17, indicators.HypervolumeImprovement._do -> select_candidates): expected-HV-improvement scores of one offspring
    # population against the current front, candidates' mean / variance from the surrogate, host buffers in and out.
    hvc = None
    try:
        px, py = opt.population_objectives
        front = py[opt.state.rank == 0].astype(np.float64)[:512]
        xc = w["rng"].random((pop, d))
        mu, var = sm.predict(xc)
        kk = min(pop, 1024)
        dt = time_device(L, lambda: L.ehvi_select(front, mu, var, ref, kk))
        sel_g, sc_g = L.ehvi_select(front, mu, var, ref, kk, return_scores=True)
        nb = max(int(front.shape[0]) - 1, 1)  # valid boxes between consecutive front points (hv_box_decomposition.py:418-437)
        evals = float(pop) * nb * M  # (candidate, box, objective) terms, each 2 Phi + 2 phi in float64
        hvc = {"value": pop / dt, "unit": "HV contributions/s", "candidates": pop, "front": int(front.shape[0]), "select_k": kk, "ms": dt * 1e3,
               "roofline": {"bound": "fp64 ALU / SFU (erfc + exp per term; 4 M (nc + 2 nb) bytes of input: not HBM bound)",
                            "achieved": evals / dt / 1e9, "unit": "G (candidate, box, objective) terms/s",
                            "note": "each term = 2 normcdf + 2 exp + ~12 flop in float64; no tensor-core or HBM roofline applies"}}
        if have_reference():  # the reference's own selector on a bounded sample, same inputs
            if REF_DIR not in sys.path:
                sys.path.insert(0, REF_DIR)
            from dmosopt import indicators as rind

            ncs = 2048
            t0 = time.perf_counter()
            sel_r = rind.HypervolumeImprovement(ref_point=ref, nds=False).do(front, mu[:ncs], var[:ncs], 64)
            dtr = time.perf_counter() - t0
            sel_s, _ = L.ehvi_select(front, mu[:ncs], var[:ncs], ref, 64, nds=False, return_scores=True)
            hvc["cpu_baseline"] = {"value": ncs / dtr, "unit": "HV contributions/s", "cores": 1, "kind": "reference",
                                   "sample": f"indicators.HypervolumeImprovement.do on {ncs} of the {pop} candidates, same {front.shape[0]}-point front, k=64",
                                   "selection_matches_gpu": bool(np.array_equal(np.asarray(sel_r), np.asarray(sel_s)))}
    except Exception as e:  # the headline metric does not depend on it
        hvc = {"error": repr(e)[:300]}

    # ------------------------------------------------------------------ sort / HV on the three objective sets of SURVEY 8d
    sort_hv = None
    if not args.no_sort_hv:
        try:
            P_last = min(pop, n_val // args.steps)
            y_m = np.vstack((sm.evaluate(np.asarray(opt.generate()[0])[:P_last]), opt.state.population_obj.astype(np.float64)))
            if y_m.shape[0] < 2 * pop:
                y_m = np.vstack((y_m, y_m[: 2 * pop - y_m.shape[0]]))
            sort_hv = sort_hv_legs(L, pop, M, y_m, ref)
        except Exception as e:
            sort_hv = {"error": repr(e)[:300]}

    # ------------------------------------------------------------------ CPU baseline beside it (rank 0, bounded sample)
    cpu = None
    if not args.no_cpu_baseline:
        try:
            cores = use_all_host_threads()
            gen, kind, sample = cpu_arm(w, args.cpu_sample, d, M, N, smlist=sm.smlist)
            gen.step()
            ts = [gen.step() for _ in range(3)]
            tot = float(np.mean([t["total"] for t in ts]))
            cpu = {"value": float(np.mean([t["children"] for t in ts])) / tot, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample + " (mean of 3 generations)",
                   "breakdown_s": {k: float(np.mean([t[k] for t in ts])) for k in ("variation", "gp", "sort", "hv")}}
        except Exception as e:
            cpu = {"error": repr(e)[:300]}

    if prec == L.GP_FP64:
        dtype = "f64"
    elif tensor_path:
        dtype = ("f64 results; GP variance contraction in split-fp16 tcgen05 with fp32 accumulation"
                 + (f" (precision=auto: calibrated against the float64 path, {refined} of {int(P_local)} rows of the last step recomputed in float64)" if auto else "")
                 + "; ranks on u32 ids")
    else:
        dtype = "f64 (precision=auto chose the float64 path for this model)"
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_val * 1e3 / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": dtype, "data": "synthetic",
        "config": {"workload": f"NSGA2 surrogate generation pop={pop} dim={d} obj={M} N_train={N} GPR_Matern fixed theta (DTLZ2-shaped targets), "
                               f"distance_metric={args.distance_metric} (MOASMO.epoch constructs the optimizer with None, MOASMO.py:365-373)",
                   "parallelism": f"candidates sharded over {world} GPU(s), one all-gather of predicted objectives" if world > 1 else "single GPU",
                   "gp_precision": args.precision, "gp_auto": auto,
                   "l2": "inputs larger than L2 (L^-1 split-fp16: %.0f MB, K_*: %.0f MB, streamed every step)" % (M * N * N * 4 / 1e6, M * N * pop * 4 / 1e6),
                   "surrogate_fit_s": t_fit},
        "roofline": roof, "cpu_baseline": cpu,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": (h1 - h0) / e2e_steps, "d2h_bytes_per_step": (d1 - d0) / e2e_steps,
                "steps": e2e_steps, "ms_per_step": t_e2e * 1e3 / e2e_steps, "device_ms_per_step": ms_e2e_dev / e2e_steps},
        "gpu_launches": int(launches), "clocks": clk, "kernel_share_of_step": shares, "hypervolume": rs.hv, "hv_contrib": hvc, "sort_hv": sort_hv,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=160)  # ~2 s timed region at ~13 ms / step
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pop", type=int, default=65536)
    ap.add_argument("--dim", type=int, default=30)
    ap.add_argument("--obj", type=int, default=3)
    ap.add_argument("--ntrain", type=int, default=4096)
    # auto = the plugin default: tensor path where the per-model calibration admits it, float64 rows where it does not;
    # tensor = the tcgen05 split-fp16 variance kernel unconditionally (<= 1e-5 of the prior variance); fp64 = the float64
    # CUDA-core path that matches scikit-learn to 1e-8 (parity anchor, ~15x slower)
    ap.add_argument("--precision", default=os.environ.get("DMOSOPT_B200_GP", "auto"), choices=["auto", "fp64", "tensor"])
    # MOASMO.epoch constructs its optimizer with distance_metric=None (dmosopt/MOASMO.py:365-373): rank ties keep
    # children-first index order.  "crowding" is NSGA2's stand-alone default (NSGA2.py:25).
    ap.add_argument("--distance-metric", default="none", choices=["none", "crowding", "euclidean"])
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--cpu-sample", type=int, default=512)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--e2e-warmup", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sort-hv", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (population, ranks, hypervolume) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
