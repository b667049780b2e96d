#!/usr/bin/env python
"""Generate golden input/output vectors from the *reference itself*.

Run in the build container, where the reference checkout is mounted read-only:

    PYTHONPATH=<dmosopt checkout> PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [name ...]

It imports dmosopt's own modules (dda, indicators, MOEA, NSGA2, AGEMOEA, SMPSO,
CMAES, hv, hv_box_decomposition, model + scikit-learn) and records seeded
inputs together with the outputs the reference produces, as small ``.npz``
files next to this script.  The reference cannot travel to the GPU box, the
fixtures do; ``tests/test_oracle_golden.py`` pins the oracle to them and the
``-m gpu`` tests pin the CUDA path to the same files.

Nothing outside ``tests/golden/`` is written.
"""

import os
import sys
import warnings

import numpy as np

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))

from dmosopt import dda, indicators, MOEA, NSGA2, AGEMOEA, SMPSO, CMAES  # noqa: E402
from dmosopt import hv as hv_mod  # noqa: E402
from dmosopt import hv_box_decomposition as hvbd  # noqa: E402
from dmosopt import model as model_mod  # noqa: E402


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {name}.npz  ({os.path.getsize(path)} bytes)")


class ReplayRng:
    """Generator stand-in whose .random(n) replays pre-drawn uniforms (for operator goldens)."""

    def __init__(self, u):
        self.u = np.asarray(u, dtype=np.float64)
        self.k = 0

    def random(self, n=None):
        if n is None:
            v = self.u.ravel()[self.k]
            self.k += 1
            return v
        v = self.u.ravel()[self.k : self.k + n]
        self.k += n
        return v.copy()


def zdt1(x):
    f1 = x[:, 0]
    g = 1.0 + 9.0 / (x.shape[1] - 1) * x[:, 1:].sum(axis=1)
    return np.column_stack((f1, g * (1.0 - np.sqrt(f1 / g))))


def dtlz2(x, M):
    g = ((x[:, M - 1 :] - 0.5) ** 2).sum(axis=1)
    f = np.ones((x.shape[0], M)) * (1.0 + g)[:, None]
    for i in range(M):
        for j in range(M - 1 - i):
            f[:, i] *= np.cos(0.5 * np.pi * x[:, j])
        if i > 0:
            f[:, i] *= np.sin(0.5 * np.pi * x[:, M - 1 - i])
    return f


# ---------------------------------------------------------------------------
def gen_dda(rng):
    out = {}
    # the reference's own known-answer example (tests/test_dda.py:162-171): expected [0 2 1 1 0 0]
    Y1 = np.asarray(
        [
            [0.2031, 0.7894, 0.5678, 0.4940, 0.1343, 0.2031],
            [0.4031, 0.8041, 0.4940, 0.4954, 0.4131, 0.4031],
            [0.3946, 0.9640, 0.4947, 0.5494, 0.4113, 0.3946],
        ]
    ).T
    out["ex_Y"] = Y1
    out["ex_rank_ens"] = dda.dda_ens(Y1)
    out["ex_rank_ns"] = dda.dda_non_dominated_sort(Y1)
    out["ex_D"] = dda.dominance_degree_matrix(Y1)
    k = 0
    for n, M in [(1, 2), (2, 2), (7, 3), (50, 2), (200, 2), (200, 3), (333, 5), (600, 3), (400, 4)]:
        Y = rng.random((n, M))
        out[f"c{k}_Y"] = Y
        out[f"c{k}_rank"] = dda.dda_ens(Y)
        out[f"c{k}_rank_ns"] = dda.dda_non_dominated_sort(Y)
        k += 1
    # near-single-front (DTLZ2 sphere) and ZDT1-like data
    x = rng.random((300, 12))
    Y = dtlz2(x, 3) * (1 + 0.01 * rng.random((300, 1)))
    out[f"c{k}_Y"] = Y
    out[f"c{k}_rank"] = dda.dda_ens(Y)
    out[f"c{k}_rank_ns"] = dda.dda_non_dominated_sort(Y)
    k += 1
    Y = zdt1(rng.random((250, 30)))
    out[f"c{k}_Y"] = Y
    out[f"c{k}_rank"] = dda.dda_ens(Y)
    out[f"c{k}_rank_ns"] = dda.dda_non_dominated_sort(Y)
    k += 1
    # duplicates (identical vectors are mutually non-dominating) with objective 0 tie-free otherwise
    Y = rng.random((60, 3))
    Y[10] = Y[3]
    Y[44] = Y[3]
    out[f"c{k}_Y"] = Y
    out[f"c{k}_rank"] = dda.dda_ens(Y)
    out[f"c{k}_rank_ns"] = dda.dda_non_dominated_sort(Y)
    k += 1
    # integer grid: many ties in every objective -> canonical (dda_non_dominated_sort) is the contract
    Y = rng.integers(0, 6, size=(150, 3)).astype(float)
    out[f"c{k}_Y"] = Y
    out[f"c{k}_rank"] = dda.dda_ens(Y)
    out[f"c{k}_rank_ns"] = dda.dda_non_dominated_sort(Y)
    k += 1
    out["ncases"] = np.array(k)
    # the objective-0 tie quirk (SURVEY section 8a row A2)
    Yq = np.array([[0.5, 0.9], [0.5, 0.1]])
    out["quirk_Y"] = Yq
    out["quirk_rank_ens"] = dda.dda_ens(Yq)
    out["quirk_rank_ns"] = dda.dda_non_dominated_sort(Yq)
    save("dda", **out)


def gen_distance(rng):
    out = {}
    k = 0
    for n, M in [(1, 3), (2, 2), (3, 3), (17, 2), (100, 3), (257, 5), (500, 2), (64, 4)]:
        Y = rng.random((n, M)) * rng.uniform(0.1, 10.0, size=(1, M))
        out[f"c{k}_Y"] = Y
        out[f"c{k}_crowd"] = indicators.crowding_distance_metric(Y)
        out[f"c{k}_eucl"] = indicators.euclidean_distance_metric(Y)
        k += 1
    # a constant column (zero range -> 1.0)
    Y = rng.random((40, 3))
    Y[:, 1] = 0.25
    out[f"c{k}_Y"] = Y
    out[f"c{k}_crowd"] = indicators.crowding_distance_metric(Y)
    out[f"c{k}_eucl"] = indicators.euclidean_distance_metric(Y)
    k += 1
    out["ncases"] = np.array(k)
    save("distance", **out)


def gen_sortmo(rng):
    out = {}
    k = 0
    for n, d, M, pop, metric in [
        (40, 5, 2, 20, None),
        (40, 5, 2, 20, "crowding"),
        (300, 8, 3, 150, "crowding"),
        (300, 8, 3, 150, "euclidean"),
        (300, 8, 3, 100, None),
        (128, 4, 5, 64, "crowding"),
    ]:
        x = rng.random((n, d))
        y = rng.random((n, M))
        ym = None if metric is None else [metric]
        xs, ys, rank, perm = MOEA.remove_worst(x, y, pop, y_distance_metrics=ym, return_perm=True)
        perm_full, rank_full, _ = MOEA.orderMO(x, y, y_distance_metrics=ym)
        out[f"c{k}_x"] = x
        out[f"c{k}_y"] = y
        out[f"c{k}_pop"] = np.array(pop)
        out[f"c{k}_metric"] = np.array(metric if metric else "none")
        out[f"c{k}_xs"] = xs
        out[f"c{k}_ys"] = ys
        out[f"c{k}_rank"] = rank
        out[f"c{k}_perm"] = perm
        out[f"c{k}_perm_full"] = perm_full
        out[f"c{k}_rank_full"] = rank_full
        k += 1
    out["ncases"] = np.array(k)
    save("sortmo", **out)


def gen_variation(rng):
    out = {}
    k = 0
    for d, rate, dim, dic in [(30, 1.0 / 30, 20.0, 1.0), (12, 1.0 / 12, 20.0, 1.0), (5, 0.5, 7.0, 3.0), (8, 0.25, 30.0, 15.0)]:
        npar = 64
        xlb = -rng.random(d) * 2.0
        xub = 1.0 + rng.random(d) * 3.0
        parents = xlb + rng.random((npar, d)) * (xub - xlb)
        parents2 = xlb + rng.random((npar, d)) * (xub - xlb)
        u_m = rng.random((npar, d))
        u_c = rng.random((npar, d))
        # a few exact edge draws
        u_m[0, 0] = 0.0
        u_c[0, 0] = 0.5
        u_c[0, 1] = 0.0
        di_m = np.asarray([dim] * d)
        di_c = np.asarray([dic] * d)
        if k == 3:  # per-dimension distribution indices (sa.py consumers, SURVEY row 21)
            di_m = rng.uniform(5.0, 40.0, size=d)
            di_c = rng.uniform(0.5, 20.0, size=d)
        mut = np.vstack([MOEA.mutation(ReplayRng(u_m[i]), parents[i], di_m, xlb, xub, mutation_rate=rate)[0] for i in range(npar)])
        c1 = []
        c2 = []
        for i in range(npar):
            a, b = MOEA.crossover_sbx(ReplayRng(u_c[i]), parents[i], parents2[i], di_c, xlb, xub)
            c1.append(a[0])
            c2.append(b[0])
        out[f"c{k}_xlb"] = xlb
        out[f"c{k}_xub"] = xub
        out[f"c{k}_p1"] = parents
        out[f"c{k}_p2"] = parents2
        out[f"c{k}_um"] = u_m
        out[f"c{k}_uc"] = u_c
        out[f"c{k}_dim"] = di_m
        out[f"c{k}_dic"] = di_c
        out[f"c{k}_rate"] = np.array(rate)
        out[f"c{k}_mut"] = mut
        out[f"c{k}_c1"] = np.vstack(c1)
        out[f"c{k}_c2"] = np.vstack(c2)
        k += 1
    out["ncases"] = np.array(k)
    save("variation", **out)


def gen_tournament(rng):
    """Inclusion frequencies of the reference's tournament_selection (distributional golden)."""
    out = {}
    k = 0
    for pop, pool, trials in [(12, 6, 40000), (30, 15, 20000), (9, 4, 40000)]:
        rank = rng.integers(0, 4, size=pop)
        crowd = rng.random(pop)
        counts1 = np.zeros(pop)
        counts2 = np.zeros(pop)
        first1 = np.zeros(pop)
        r = np.random.default_rng(1234 + k)
        for _ in range(trials):
            idx = MOEA.tournament_selection(r, pop, pool, rank)
            counts1[idx] += 1
            first1[idx[0]] += 1
            idx = MOEA.tournament_selection(r, pop, pool, -crowd, rank)
            counts2[idx] += 1
        out[f"c{k}_rank"] = rank
        out[f"c{k}_crowd"] = crowd
        out[f"c{k}_pool"] = np.array(pool)
        out[f"c{k}_trials"] = np.array(trials)
        out[f"c{k}_freq_rank"] = counts1 / trials
        out[f"c{k}_first_rank"] = first1 / trials
        out[f"c{k}_freq_rank_crowd"] = counts2 / trials
        out[f"c{k}_order_rank"] = np.lexsort((rank,))
        out[f"c{k}_order_rank_crowd"] = np.lexsort((-crowd, rank))
        k += 1
    out["ncases"] = np.array(k)
    save("tournament", **out)


def gen_duplicates(rng):
    out = {}
    X = rng.random((80, 6))
    X[7] = X[2]
    X[50] = X[2]
    X[51] = X[30]
    out["X"] = X
    out["dup"] = MOEA.get_duplicates(X)
    # the two-set form of MOASMO's resample step (MOASMO.py:442): rows of X against EARLIER rows of Y
    Y = rng.random((60, 6))
    Y[3] = X[10]   # j = 3 < i = 10: duplicate
    Y[40] = X[12]  # j = 40 > i = 12: masked by the upper triangle, not a duplicate
    Y[5] = X[5]    # j == i: the diagonal is masked too
    Y[0] = X[79]
    out["Y"] = Y
    out["dup_xy"] = MOEA.get_duplicates(X, Y)
    save("duplicates", **out)


def gen_gp(rng):
    """GPR_Matern / GPR_RBF posterior: fitted state (from sklearn) + predictions."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import ConstantKernel, Matern, RBF, WhiteKernel

    out, factors = {}, {}
    k = 0
    cases = [
        # (N, d, M, P, kind, length_scale (None = fixed initial theta), anisotropic)
        (64, 5, 2, 40, "matern", None, False),
        (200, 12, 3, 96, "matern", None, False),
        (150, 30, 2, 64, "matern", None, False),
        (120, 6, 2, 50, "matern", "fit", False),
        (100, 4, 2, 50, "matern", "fit", True),
        (90, 5, 2, 40, "rbf", None, False),
    ]
    for N, d, M, P, kind, mode, aniso in cases:
        xlb = -rng.random(d)
        xub = 1.0 + rng.random(d)
        xin = xlb + rng.random((N, d)) * (xub - xlb)
        xn = (xin - xlb) / (xub - xlb)
        yin = dtlz2(xn, M) if M > 2 else zdt1(xn)
        xtest = xlb + rng.random((P, d)) * (xub - xlb)
        # a few test points very close to training points (small posterior variance)
        xtest[:4] = xin[:4] + 1e-4 * (xub - xlb) * rng.standard_normal((4, d))
        xtest = np.clip(xtest, xlb, xub)
        if mode == "fit":
            # the reference's own class: SCE-UA optimised hyper-parameters (model.py:1182-1252)
            mdl = model_mod.GPR_Matern(xin, yin, d, M, xlb, xub, optimizer="sceua", seed=7, anisotropic=aniso)
            mean, var = mdl.predict(xtest)
            smlist = mdl.smlist
        else:
            # fixed initial theta, sklearn optimizer=None (BASELINE.md section 3 item 1), then the
            # reference's own predict() body run on these regressors
            if kind == "matern":
                kern = ConstantKernel(1, (1e-4, 1e3)) * Matern(length_scale=0.5, length_scale_bounds=(1e-3, 100.0), nu=2.5) + WhiteKernel(
                    noise_level=1e-6, noise_level_bounds=(1e-9, 1e-2)
                )
                cls = model_mod.GPR_Matern
            else:
                kern = ConstantKernel(1, (1e-4, 1e3)) * RBF(length_scale=0.5, length_scale_bounds=(1e-3, 100.0)) + WhiteKernel(
                    noise_level=1e-5, noise_level_bounds=(1e-9, 1e-2)
                )
                cls = model_mod.GPR_RBF
            smlist = []
            for m in range(M):
                g = GaussianProcessRegressor(kernel=kern, optimizer=None, normalize_y=True)
                g.fit(xn, yin[:, m])
                smlist.append(g)
            mdl = cls.__new__(cls)
            mdl.nInput, mdl.nOutput, mdl.xlb, mdl.xub, mdl.xrg = d, M, xlb, xub, xub - xlb
            mdl.smlist = smlist
            mdl.return_mean_variance = False
            mean, var = mdl.predict(xtest)
        out[f"c{k}_kind"] = np.array(kind)
        out[f"c{k}_xlb"] = xlb
        out[f"c{k}_xub"] = xub
        out[f"c{k}_xin"] = xin
        out[f"c{k}_yin"] = yin
        out[f"c{k}_xtest"] = xtest
        out[f"c{k}_mean"] = mean
        out[f"c{k}_var"] = var
        out[f"c{k}_Xtrain"] = np.asarray(smlist[0].X_train_)
        out[f"c{k}_alpha"] = np.stack([np.ravel(g.alpha_) for g in smlist])
        factors[f"c{k}_L"] = np.stack([g.L_ for g in smlist])
        out[f"c{k}_const"] = np.array([g.kernel_.k1.k1.constant_value for g in smlist])
        out[f"c{k}_ls"] = np.stack([np.broadcast_to(np.asarray(g.kernel_.k1.k2.length_scale, float), (d,)) for g in smlist])
        out[f"c{k}_noise"] = np.array([g.kernel_.k2.noise_level for g in smlist])
        out[f"c{k}_ymean"] = np.array([np.ravel(g._y_train_mean)[0] for g in smlist])
        out[f"c{k}_ystd"] = np.array([np.ravel(g._y_train_std)[0] for g in smlist])
        k += 1
    out["ncases"] = np.array(k)
    save("gp", **out)
    save("gp_factors", **factors)  # the Cholesky factors in a file of their own: each file stays under 1 MB


def gen_hv(rng):
    out = {}
    # analytic known answers from the reference's tests (tests/test_hv_box_decomposition.py:29-67,100-108)
    ka = [
        (np.array([[1.0, 1.0]]), np.array([3.0, 3.0]), 4.0),
        (np.array([[1.0, 3.0], [2.0, 2.0], [3.0, 1.0]]), np.array([4.0, 4.0]), 6.0),
        (np.array([[1.0, 2.0], [2.0, 1.0]]), np.array([3.0, 3.0]), 3.0),
        (np.array([[1.0, 1.0, 1.0]]), np.array([2.0, 2.0, 2.0]), 1.0),
        (np.array([[2.0]]), np.array([5.0]), 3.0),
    ]
    for i, (P, r, v) in enumerate(ka):
        out[f"ka{i}_P"] = P
        out[f"ka{i}_ref"] = r
        out[f"ka{i}_expected"] = np.array(v)
        out[f"ka{i}_refimpl"] = np.array(hvbd.HyperVolumeBoxDecomposition(r).compute_hypervolume(P))
    out["nka"] = np.array(len(ka))
    k = 0
    for n, d in [(1, 2), (5, 2), (60, 2), (300, 2), (30, 3), (120, 3), (40, 4), (60, 4), (25, 5), (12, 6)]:
        P = 0.05 + rng.random((n, d))
        ref = np.full(d, 1.0 + 0.1 * rng.random())
        if k % 3 == 2:  # a non-dominated-ish cloud
            P = dtlz2(rng.random((n, d + 4)), d) + 0.05
            ref = np.full(d, 1.3)
        out[f"c{k}_P"] = P
        out[f"c{k}_ref"] = ref
        out[f"c{k}_hv_box"] = np.array(hvbd.HyperVolumeBoxDecomposition(ref).compute_hypervolume(P))
        out[f"c{k}_hv_adaptive"] = np.array(hv_mod.AdaptiveHyperVolume(ref).compute_hypervolume(P, algorithm="box"))
        k += 1
    # reference point cutting through the cloud (hv.py:159 mask)
    P = rng.random((80, 3)) + 0.05
    ref = np.array([0.8, 0.9, 0.7])
    out[f"c{k}_P"] = P
    out[f"c{k}_ref"] = ref
    out[f"c{k}_hv_box"] = np.array(np.nan)  # box algorithm alone is not defined for points outside ref
    out[f"c{k}_hv_adaptive"] = np.array(hv_mod.AdaptiveHyperVolume(ref).compute_hypervolume(P, algorithm="box"))
    k += 1
    out["ncases"] = np.array(k)
    # the documented <=0 coordinate divergence (SURVEY row A16)
    out["quirk_P"] = np.array([[-1.0, -1.0]])
    out["quirk_ref"] = np.array([1.0, 1.0])
    out["quirk_refimpl"] = np.array(hvbd.HyperVolumeBoxDecomposition(np.array([1.0, 1.0])).compute_hypervolume(np.array([[-1.0, -1.0]])))
    save("hv", **out)


def gen_hv_many(rng):
    """Exact hypervolume for 6 .. 8 objectives from the reference's box decomposition (the branch hv.py:160-170 takes for
    every M < 10): random clouds and DTLZ2-shaped (mostly non-dominated) sets, sized so that the Python reference finishes."""
    import time

    out = {}
    k = 0
    for n, d, shaped in [(14, 6, False), (40, 6, False), (36, 6, True), (30, 7, False), (24, 7, True), (22, 8, False), (18, 8, True),
                         (200, 6, False), (120, 6, True), (100, 7, True), (150, 7, False), (80, 8, True)]:
        if shaped:
            P = dtlz2(rng.random((n, d + 4)), d) + 0.05
            ref = np.full(d, 1.3)
        else:
            P = 0.05 + rng.random((n, d))
            ref = np.full(d, 1.0 + 0.1 * rng.random())
        t0 = time.time()
        out[f"c{k}_P"], out[f"c{k}_ref"] = P, ref
        out[f"c{k}_hv_box"] = np.array(hvbd.HyperVolumeBoxDecomposition(ref).compute_hypervolume(P))
        out[f"c{k}_hv_adaptive"] = np.array(hv_mod.AdaptiveHyperVolume(ref).compute_hypervolume(P, algorithm="box"))
        print(f"  hv_many case {k}: n={n} d={d} shaped={shaped}: {time.time() - t0:.1f} s, hv={float(out[f'c{k}_hv_box']):.6g}", flush=True)
        k += 1
    out["ncases"] = np.array(k)
    save("hv_many", **out)


def gen_ehvi(rng):
    out = {}
    k = 0
    for nf, nc, d, kk in [(30, 50, 2, 10), (100, 200, 3, 40), (60, 120, 5, 25), (8, 20, 4, 5)]:
        chosen = dtlz2(rng.random((nf, d + 5)), d) * (1.0 + 0.3 * rng.random((nf, 1)))
        cand = dtlz2(rng.random((nc, d + 5)), d) * (1.0 + 0.3 * rng.random((nc, 1)))
        ref = np.max(np.vstack((chosen, cand)), axis=0) + 1
        variances = np.ones_like(cand) if k % 2 == 0 else 0.05 + rng.random(cand.shape)
        ind = indicators.HypervolumeImprovement(ref_point=ref, nds=True)
        sel = ind.do(chosen, cand, variances, kk)
        # intermediate values straight from the reference's box code
        rank = dda.dda_ens(chosen)
        front = chosen[rank == 0]
        hvo = hvbd.HyperVolumeBoxDecomposition(ref)
        boxes = hvo._decompose_dominated_space(front)
        ehvi = hvo._compute_batch_ehvi(boxes, cand, variances)
        out[f"c{k}_chosen"] = chosen
        out[f"c{k}_cand"] = cand
        out[f"c{k}_var"] = variances
        out[f"c{k}_ref"] = ref
        out[f"c{k}_k"] = np.array(kk)
        out[f"c{k}_sel"] = np.asarray(sel)
        out[f"c{k}_ehvi"] = ehvi
        out[f"c{k}_lower"] = np.array([b.lower for b in boxes])
        out[f"c{k}_upper"] = np.array([b.upper for b in boxes])
        k += 1
    out["ncases"] = np.array(k)
    save("ehvi", **out)


def gen_nsga2(rng):
    """Reference NSGA2 plugin: initialize_state + update_strategy on recorded offspring."""
    out = {}
    k = 0
    # ZDT1's f1 = x0 ties exactly at clipped genes, which makes the reference's own result depend on
    # numpy's unstable sorts (crowding argsort, dda_ens order); those cases are flagged ``ties`` and only
    # pin the oracle on this machine.  The other cases add a small random linear term to DTLZ2 so that
    # every objective is tie-free even at clipped genes.
    for pop, d, M, metric, fname in [(40, 6, 2, "crowding", "dtlz2"), (100, 12, 3, None, "dtlz2"), (64, 30, 2, None, "zdt1"),
                                     (64, 30, 2, "crowding", "dtlz2"), (50, 10, 3, "euclidean", "dtlz2")]:
        bounds = np.column_stack((np.zeros(d), np.ones(d)))
        W = rng.random((d, M))
        f = (lambda x: zdt1(x)) if fname == "zdt1" else (lambda x, M=M, W=W: dtlz2(x, M) + 0.01 * (x @ W))
        out[f"c{k}_ties"] = np.array(fname == "zdt1")
        x0 = rng.random((pop + 17, d))
        y0 = f(x0).astype(np.float32)  # MOASMO.optimize casts the initial objectives (MOASMO.py:64)
        opt = NSGA2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=model_mod.Model(), distance_metric=metric)
        r = np.random.default_rng(99 + k)
        opt.initialize_strategy(x0, y0, bounds, r)
        out[f"c{k}_x0"] = x0
        out[f"c{k}_y0"] = y0
        out[f"c{k}_metric"] = np.array(metric if metric else "none")
        out[f"c{k}_init_px"] = opt.state.population_parm.copy()
        out[f"c{k}_init_py"] = opt.state.population_obj.copy()
        out[f"c{k}_init_rank"] = opt.state.rank.copy()
        for g in range(3):
            x_gen, st = opt.generate()
            y_gen = f(x_gen)
            opt.update(x_gen, y_gen, st)
            out[f"c{k}_g{g}_xgen"] = x_gen
            out[f"c{k}_g{g}_ygen"] = y_gen
            out[f"c{k}_g{g}_cidx"] = st["crossover_indices"]
            out[f"c{k}_g{g}_midx"] = st["mutation_indices"]
            out[f"c{k}_g{g}_px"] = opt.state.population_parm.copy()
            out[f"c{k}_g{g}_py"] = opt.state.population_obj.copy()
            out[f"c{k}_g{g}_rank"] = opt.state.rank.copy()
        # offspring-count distribution of the serial variation loop (NSGA2.py:142-178)
        counts = []
        ncross = []
        for _ in range(300):
            xg, st = opt.generate()
            counts.append(xg.shape[0])
            ncross.append(len(st["crossover_indices"]) // 2)
        out[f"c{k}_count_hist"] = np.bincount(np.asarray(counts), minlength=pop + 2)
        out[f"c{k}_ncross_mean"] = np.array(np.mean(ncross))
        k += 1
    out["ncases"] = np.array(k)
    save("nsga2", **out)


def gen_agemoea(rng):
    out = {}
    k = 0
    for n, d, M, pop in [(60, 5, 2, 30), (200, 8, 3, 100), (150, 6, 3, 120), (120, 5, 4, 40)]:
        x = rng.random((n, d))
        y = dtlz2(x, M) * (1.0 + (0.0 if k == 2 else 0.4) * rng.random((n, 1)))
        xs, ys, rank, cd = AGEMOEA.environmental_selection(np.random.default_rng(5), x, y, pop, d, M)
        out[f"c{k}_x"] = x
        out[f"c{k}_y"] = y
        out[f"c{k}_pop"] = np.array(pop)
        out[f"c{k}_xs"] = xs
        out[f"c{k}_ys"] = ys
        out[f"c{k}_rank"] = rank
        out[f"c{k}_cd"] = cd
        # survival score of the first front on its own
        r = dda.dda_ens(y)
        idxr = r.argsort()
        ys_sorted = y[idxr]
        front = np.argwhere(r[idxr] == 0).ravel()
        ideal = np.min(ys_sorted[front], axis=0)
        norm_, p_, cd_ = AGEMOEA.survival_score(ys_sorted, front, ideal)
        out[f"c{k}_front_y"] = ys_sorted[front]
        out[f"c{k}_ss_norm"] = np.asarray(norm_, dtype=float)
        out[f"c{k}_ss_p"] = np.array(p_, dtype=float)
        out[f"c{k}_ss_cd"] = cd_
        k += 1
    out["ncases"] = np.array(k)
    save("agemoea", **out)


def gen_smpso(rng):
    out = {}

    class FixedRng:
        """Replays the scalar draws of velocity_vector (SMPSO.py:316-321, 332)."""

        def __init__(self, vals, ints):
            self.vals = list(vals)
            self.ints = ints

        def uniform(self, low=0.0, high=1.0, size=1):
            v = self.vals.pop(0)
            return np.array([low + (high - low) * v])

        def integers(self, low=0, high=None, size=None):
            return np.asarray(self.ints)

    k = 0
    for n, d, M in [(40, 6, 2), (100, 10, 3)]:
        xlb = -rng.random(d)
        xub = 1 + rng.random(d)
        pos = (xlb + rng.random((n, d)) * (xub - xlb)).astype(np.float32)
        vel = xlb + rng.random((n, d)) * (xub - xlb)
        arch = (xlb + rng.random((n, d)) * (xub - xlb)).astype(np.float32)
        y = rng.random((n, M))
        crowd = indicators.crowding_distance_metric(y)
        u5 = rng.random(5)
        if k == 1:
            u5[3] = 0.9
            u5[4] = 0.95  # c1 + c2 > 4 -> constriction active
        ints = rng.integers(0, n, size=2)
        v = SMPSO.velocity_vector(FixedRng(u5, ints), pos, vel, arch, crowd, xlb, xub)
        out[f"c{k}_xlb"] = xlb
        out[f"c{k}_xub"] = xub
        out[f"c{k}_pos"] = pos
        out[f"c{k}_vel"] = vel
        out[f"c{k}_arch"] = arch
        out[f"c{k}_crowd"] = crowd
        out[f"c{k}_u5"] = u5
        out[f"c{k}_ints"] = ints
        out[f"c{k}_vout"] = v
        out[f"c{k}_newpos"] = SMPSO.update_position(pos, v, xlb, xub)
        k += 1
    out["ncases"] = np.array(k)
    save("smpso", **out)


def gen_cmaes(rng):
    """CMAES._select masks (fronts + HV-improvement split) on recorded candidates."""
    out = {}
    k = 0
    for pop, d, M in [(40, 6, 2), (60, 8, 3)]:
        opt = CMAES.CMAES(popsize=pop, nInput=d, nOutput=M, model=model_mod.Model(), distance_metric=None)
        n = pop + pop // 2
        cx = rng.random((n, d))
        cy = dtlz2(cx, M) * (1.0 + 0.5 * rng.random((n, 1)))
        inds = np.arange(n)
        chosen, not_chosen, rank = opt._select(cx, cy, None, inds)
        out[f"c{k}_pop"] = np.array(pop)
        out[f"c{k}_cx"] = cx
        out[f"c{k}_cy"] = cy
        out[f"c{k}_chosen"] = chosen
        out[f"c{k}_not_chosen"] = not_chosen
        out[f"c{k}_rank"] = rank
        k += 1
    out["ncases"] = np.array(k)
    save("cmaes", **out)


def gen_plugins(rng):
    """Full update steps of the reference AGEMOEA / SMPSO / CMAES plugins on recorded offspring."""
    out = {}
    d, M, pop = 8, 3, 40
    bounds = np.column_stack((np.zeros(d), np.ones(d)))
    W = rng.random((d, M))
    f = lambda x: dtlz2(x, M) + 0.01 * (x @ W)  # noqa: E731  (tie-free objectives)
    # ---- AGEMOEA: initialize + two updates (set-level parity: row order inside a front is unstable in the reference)
    x0 = rng.random((pop + 10, d))
    y0 = f(x0).astype(np.float32)
    opt = AGEMOEA.AGEMOEA(popsize=pop, nInput=d, nOutput=M, model=model_mod.Model())
    out["age_x0"], out["age_y0"] = x0.copy(), y0.copy()  # the reference keeps views of its inputs and writes into them
    opt.initialize_strategy(x0, y0, bounds, np.random.default_rng(3))
    out["age_init_rank"], out["age_init_cd"] = opt.state.rank.copy(), opt.state.crowd_dist.copy()
    for g in range(2):
        xg = np.clip(opt.state.population_parm + 0.05 * rng.standard_normal((pop, d)), 0, 1)
        yg = f(xg)
        opt.update(xg, yg, {})
        out[f"age_g{g}_xgen"], out[f"age_g{g}_ygen"] = xg, yg
        out[f"age_g{g}_px"], out[f"age_g{g}_py"] = opt.state.population_parm.copy(), opt.state.population_obj.copy()
        out[f"age_g{g}_rank"], out[f"age_g{g}_cd"] = opt.state.rank.copy(), opt.state.crowd_dist.copy()
    # ---- SMPSO: initialize (velocity from the generator) + one update with a fresh generator
    pop_s, sw = 24, 5
    x0 = rng.random((pop_s * sw, d))
    y0 = f(x0).astype(np.float32)
    opt = SMPSO.SMPSO(popsize=pop_s, nInput=d, nOutput=M, model=model_mod.Model(), distance_metric=None)
    opt.initialize_strategy(x0, y0, bounds, np.random.default_rng(11))
    out["smpso_x0"], out["smpso_y0"] = x0, y0
    out["smpso_init_px"], out["smpso_init_py"], out["smpso_init_vel"] = opt.state.population_parm.copy(), opt.state.population_obj.copy(), opt.state.velocity.copy()
    xg, _ = opt.generate()
    out["smpso_xgen_shape"] = np.array(xg.shape)
    out["smpso_xgen_positions"] = xg.reshape(sw, 2 * pop_s, d)[:, :pop_s].copy()  # deterministic half of x_gen
    yg = f(xg.astype(np.float64))
    opt.local_random = np.random.default_rng(12)
    opt.update(xg, yg, {})
    out["smpso_xgen"], out["smpso_ygen"] = xg, yg
    out["smpso_g0_px"], out["smpso_g0_py"], out["smpso_g0_vel"] = opt.state.population_parm.copy(), opt.state.population_obj.copy(), opt.state.velocity.copy()
    out["smpso_g0_ranks"] = np.stack(opt.state.ranks)
    out["smpso_succ"] = np.array(opt.state.successful_children)
    # ---- CMAES: initialize + two full updates on recorded offspring / parent indices
    popc = 30
    x0 = rng.random((popc + 8, d))
    y0 = f(x0)
    opt = CMAES.CMAES(popsize=popc, nInput=d, nOutput=M, model=model_mod.Model(), distance_metric=None)
    opt.initialize_strategy(x0, y0, bounds, np.random.default_rng(21))
    out["cma_x0"], out["cma_y0"] = x0, y0
    out["cma_init_px"], out["cma_init_sig"] = opt.state.parents_x.copy(), opt.state.sigmas.copy()
    for g in range(3):
        xg, stg = opt.generate()
        yg = f(xg)
        if g == 0:  # sampling golden: record the normal draws by replaying the generator
            out["cma_g0_parents_x"], out["cma_g0_sigmas"], out["cma_g0_A"] = opt.state.parents_x.copy(), opt.state.sigmas.copy(), opt.state.A.copy()
        opt.update(xg, yg, stg)
        out[f"cma_g{g}_xgen"], out[f"cma_g{g}_ygen"], out[f"cma_g{g}_pidx"] = xg, yg, stg["p_idx"]
        out[f"cma_g{g}_px"], out[f"cma_g{g}_py"] = opt.state.parents_x.copy(), opt.state.parents_y.copy()
        out[f"cma_g{g}_sig"], out[f"cma_g{g}_A"], out[f"cma_g{g}_Ainv"] = opt.state.sigmas.copy(), opt.state.A.copy(), opt.state.Ainv.copy()
        out[f"cma_g{g}_pc"], out[f"cma_g{g}_psucc"], out[f"cma_g{g}_rank"] = opt.state.pc.copy(), opt.state.psucc.copy(), opt.state.rank.copy()
    save("plugins", **out)


def gen_adaptive(rng):
    """The adaptive helpers of the optimizers (host control logic, off the hot path, but part of the plugin contract):
    update_population_size of NSGA2 / AGEMOEA / SMPSO / CMAES / TRS and update_operator_rates of NSGA2 / SMPSO on crafted
    states that reach every branch (few / many first-front members, small / large crowding spread, low / high success)."""
    from dmosopt import TRS

    out = {}
    d, M, pop = 6, 2, 60
    bounds = np.column_stack((np.zeros(d), np.ones(d)))

    def states():
        """(rank, objectives) pairs: every point on one front / a tiny first front / clustered first front / generic."""
        t = np.sort(rng.random(pop))
        yield np.zeros(pop, dtype=int), np.column_stack((t, 1.0 - t))
        r = np.ones(pop, dtype=int)
        r[:3] = 0
        yield r, rng.random((pop, M))
        r = (np.arange(pop) % 2).astype(int)
        y = rng.random((pop, M))
        y[r == 0] = 0.5 + 1e-3 * rng.random((int((r == 0).sum()), M))
        yield r, y
        yield rng.integers(0, 4, size=pop), rng.random((pop, M))
        r = np.zeros(pop, dtype=int)
        r[pop // 3:] = 1
        y = rng.random((pop, M)) ** 3
        yield r, y

    cases = list(states())
    out["n_cases"] = np.array(len(cases))
    for k, (r, y) in enumerate(cases):
        out[f"c{k}_rank"], out[f"c{k}_obj"] = r, y
    x0 = rng.random((pop, d))
    y0 = zdt1(x0)
    for name, cls, kw in (("nsga2", NSGA2.NSGA2, {}), ("age", AGEMOEA.AGEMOEA, {}), ("cma", CMAES.CMAES, {"distance_metric": None}),
                          ("trs", TRS.TRS, {})):
        for k, (r, y) in enumerate(cases):
            opt = cls(popsize=pop, nInput=d, nOutput=M, model=model_mod.Model(), **kw)
            opt.initialize_strategy(x0.copy(), y0.copy(), bounds, np.random.default_rng(1))
            st = opt.state
            st.rank = r.copy()
            if name == "cma":
                st.parents_y = y.copy()
            else:
                st.population_obj = y.copy()
            opt.opt_params.max_population_size, opt.opt_params.min_population_size = 90, 20
            opt.update_population_size()
            out[f"{name}_c{k}_popsize"] = np.array(opt.opt_params.popsize)
    # SMPSO keeps one rank array per swarm
    for k, (r, y) in enumerate(cases):
        opt = SMPSO.SMPSO(popsize=pop // 5, nInput=d, nOutput=M, model=model_mod.Model(), distance_metric=None)
        opt.initialize_strategy(x0.copy(), y0.astype(np.float32), bounds, np.random.default_rng(1))
        opt.state.ranks = [r[s * (pop // 5):(s + 1) * (pop // 5)].copy() for s in range(5)]
        opt.state.population_obj = y.copy()
        opt.opt_params.max_population_size, opt.opt_params.min_population_size = 30, 4
        opt.update_population_size()
        out[f"smpso_c{k}_popsize"] = np.array(opt.opt_params.popsize)
    # operator rates: (successful, total) counters below / inside / above the success band, twice in a row
    rates = [(0, 50, 1, 40), (10, 50, 8, 40), (40, 50, 30, 40), (0, 0, 0, 0), (50, 50, 0, 40)]
    out["n_rates"] = np.array(len(rates))
    for k, (sc, tc, smu, tmu) in enumerate(rates):
        opt = NSGA2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=model_mod.Model())
        opt.initialize_strategy(x0.copy(), y0.copy(), bounds, np.random.default_rng(1))
        rec = []
        for _ in range(2):
            st = opt.state
            st.successful_crossovers, st.total_crossovers, st.successful_mutations, st.total_mutations = sc, tc, smu, tmu
            opt.update_operator_rates()
            p = opt.opt_params
            rec.append(np.concatenate((np.atleast_1d(np.asarray(p.di_crossover, dtype=float)).ravel()[:1], [float(p.crossover_prob)],
                                       np.atleast_1d(np.asarray(p.di_mutation, dtype=float)).ravel()[:1], [float(p.mutation_prob), float(p.mutation_rate)],
                                       [st.successful_crossovers, st.total_crossovers, st.successful_mutations, st.total_mutations])))
        out[f"nsga2_rates{k}"] = np.stack(rec)
        out[f"nsga2_rates{k}_in"] = np.array([sc, tc, smu, tmu])
        opt = SMPSO.SMPSO(popsize=pop // 5, nInput=d, nOutput=M, model=model_mod.Model(), distance_metric=None)
        opt.initialize_strategy(x0.copy(), y0.astype(np.float32), bounds, np.random.default_rng(1))
        rec = []
        for _ in range(2):
            opt.state.successful_children = sc
            opt.update_operator_rates()
            p = opt.opt_params
            rec.append([float(np.atleast_1d(np.asarray(p.di_mutation, dtype=float)).ravel()[0]), float(p.mutation_rate), float(opt.state.successful_children)])
        out[f"smpso_rates{k}"] = np.array(rec)
    out["x0"], out["y0"] = x0, y0
    save("adaptive", **out)


def gen_trs(rng):
    """Trust-region search (dmosopt/TRS.py): initialize, then three generate / update rounds driven by one NumPy generator
    (Sobol perturbations come from scipy's sampler seeded by that generator, so the plugin reproduces them exactly), and
    the vectorised benchmark functions (dmosopt/benchmarks/moo_benchmarks.py) evaluated row by row."""
    from dmosopt import TRS
    from dmosopt.benchmarks import moo_benchmarks as mb

    out = {}
    d, M, pop = 8, 3, 36
    bounds = np.column_stack((np.zeros(d), np.ones(d)))
    W = rng.random((d, M))
    f = lambda x: dtlz2(x, M) + 0.01 * (x @ W)  # noqa: E731
    x0 = rng.random((pop + 12, d))
    y0 = f(x0)
    opt = TRS.TRS(popsize=pop, nInput=d, nOutput=M, model=model_mod.Model())
    out["x0"], out["y0"] = x0.copy(), y0.copy()
    opt.initialize_strategy(x0, y0, bounds, np.random.default_rng(31))
    out["init_px"], out["init_py"], out["init_rank"] = opt.state.population_parm.copy(), opt.state.population_obj.copy(), opt.state.rank.copy()
    for g in range(3):
        xg, stg = opt.generate()
        yg = f(xg)
        opt.update(xg, yg, stg)
        out[f"g{g}_xgen"], out[f"g{g}_ygen"] = xg.copy(), yg.copy()
        out[f"g{g}_px"], out[f"g{g}_py"], out[f"g{g}_rank"] = opt.state.population_parm.copy(), opt.state.population_obj.copy(), opt.state.rank.copy()
        out[f"g{g}_length"] = np.array(opt.state.tr.length)
    # benchmark functions: the reference evaluates one row at a time
    names = ["dtlz1", "dtlz2", "dtlz3", "dtlz4", "dtlz5", "dtlz7", "wfg4"]
    got = []
    for nm in names:
        fn = getattr(mb, nm, None)
        if fn is None:
            continue
        for m_obj, n_var in ((2, 10),) if nm.startswith("zdt") else ((3, 12), (5, 22)):
            X = rng.random((17, n_var))
            try:
                Y = np.vstack([np.asarray(fn(x, m_obj) if not nm.startswith("zdt") else fn(x), dtype=np.float64).ravel() for x in X])
            except Exception:  # signature differs: skip, the test only covers what was recorded
                continue
            key = f"bm_{nm}_{m_obj}_{n_var}"
            out[key + "_X"], out[key + "_Y"] = X, Y
            got.append(key)
    # ZDT1 / ZDT3: the objective functions of the reference's examples (examples/example_dmosopt_zdt1.py:9-20, _zdt3.py:9-21)
    import importlib.util

    for nm in ("zdt1", "zdt3"):
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(MOEA.__file__))), "examples", f"example_dmosopt_{nm}.py")
        text = open(path).read()
        src = text[text.index(f"def {nm}(") : text.index("def obj_fun")]  # the objective function only (the rest needs MPI / dmosopt.run)
        ns = {"np": np}
        exec(compile(src, path, "exec"), ns)
        X = rng.random((17, 30))
        out[f"bm_{nm}_2_30_X"], out[f"bm_{nm}_2_30_Y"] = X, np.vstack([np.asarray(ns[nm](x), dtype=np.float64).ravel() for x in X])
        got.append(f"bm_{nm}_2_30")
    out["bm_keys"] = np.array(got)
    save("trs", **out)


def gen_reference_loop(rng):
    """The reference's results for tests/test_gpu_reference_loop.py: three NSGA2 generations (its own generate / update) and
    the controller helpers MOASMO.get_best, MOEA.get_duplicates / crowding_distance_metric and hv.AdaptiveHyperVolume."""
    from dmosopt import MOASMO
    from dmosopt import model as rmodel

    out = {}
    # ---- NSGA2: same initial state, the reference's offspring, the reference's survivors after each update
    d, M, pop = 10, 3, 300
    r = np.random.default_rng(3)
    bounds = np.column_stack((np.zeros(d), np.ones(d)))
    x0 = r.random((pop, d))

    def f(x):
        return np.column_stack((x[:, 0] + x[:, 3:].sum(1) * 0.1, (1 - x[:, 0]) * (1 + x[:, 1]), x[:, 2] ** 2 + 0.5 * x[:, 1]))

    y0 = f(x0).astype(np.float32)
    out["nsga2_x0"], out["nsga2_y0"] = x0, y0
    ro = NSGA2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=rmodel.Model(), distance_metric=None)
    ro.initialize_strategy(x0.astype(np.float32), y0.copy(), bounds, np.random.default_rng(1))
    out["nsga2_init_rank"] = np.array(ro.state.rank)  # copies: the reference updates its state arrays in place
    for gi in range(3):
        x_gen, st = ro.generate()
        x_gen = np.array(x_gen)
        ro.update(x_gen, f(x_gen), st)
        out[f"nsga2_g{gi}_xgen"] = x_gen
        out[f"nsga2_g{gi}_cidx"] = np.array(st["crossover_indices"])
        out[f"nsga2_g{gi}_midx"] = np.array(st["mutation_indices"])
        out[f"nsga2_g{gi}_rank"] = np.array(ro.state.rank)
        out[f"nsga2_g{gi}_py"] = np.array(ro.state.population_obj)
    # ---- controller helpers on a set with duplicated objective rows and shared decision rows
    r = np.random.default_rng(21)
    n, d, M = 700, 9, 3
    x = r.random((n, d))
    y = np.column_stack((x[:, 0] + 0.1, (1.1 - x[:, 0]) * (1 + x[:, 1]), 0.2 + x[:, 2] ** 2 + x[:, 1]))
    y[50] = y[3]
    y[400] = y[3]
    x0 = r.random((300, d))
    x0[:40] = x[100:140]
    ref_pt = y.max(axis=0) + 0.1
    out["help_x"], out["help_y"], out["help_x0"], out["help_ref"] = x, y, x0, ref_pt
    best_x, best_y, best_f, best_c, best_epoch, perm = MOASMO.get_best(x, y, None, None, d, M, return_perm=True)
    assert best_f is None and best_c is None and best_epoch is None
    out["help_best_x"], out["help_best_y"], out["help_best_perm"] = best_x, best_y, np.asarray(perm)
    out["help_dup"] = MOEA.get_duplicates(x, x0)
    out["help_cd"] = MOEA.crowding_distance_metric(y[np.r_[0:50, 51:400, 401:n]])
    out["help_hv"] = np.array(hv_mod.AdaptiveHyperVolume(ref_pt).compute_hypervolume(y[:300]))
    save("reference_loop", **out)


def main():
    which = sys.argv[1:] or ["dda", "distance", "sortmo", "variation", "tournament", "duplicates", "gp", "hv", "ehvi", "nsga2", "agemoea", "smpso", "cmaes", "plugins", "trs", "adaptive", "hv_many", "reference_loop"]
    gens = {
        "dda": gen_dda,
        "distance": gen_distance,
        "sortmo": gen_sortmo,
        "variation": gen_variation,
        "tournament": gen_tournament,
        "duplicates": gen_duplicates,
        "gp": gen_gp,
        "hv": gen_hv,
        "ehvi": gen_ehvi,
        "nsga2": gen_nsga2,
        "agemoea": gen_agemoea,
        "smpso": gen_smpso,
        "cmaes": gen_cmaes,
        "plugins": gen_plugins,
        "trs": gen_trs,
        "adaptive": gen_adaptive,
        "hv_many": gen_hv_many,
        "reference_loop": gen_reference_loop,
    }
    for i, name in enumerate(which):
        gens[name](np.random.default_rng(20260921 + i * 0 + sum(map(ord, name))))


if __name__ == "__main__":
    main()
