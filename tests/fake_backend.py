"""Oracle-backed stand-in for ``dmosopt_b200._lib`` -- TEST SEAM ONLY.

The product has no CPU path.  To exercise the *host* logic of the plugins (argument marshalling,
state handling, dtype flow) on a machine without a GPU,
tests monkeypatch the thin ``_lib`` functions with these NumPy implementations built on ``oracle/``.
"""

import numpy as np

from oracle import dda, gp, hv, indicators, moea, nsga2

METRIC_NONE, METRIC_CROWDING, METRIC_EUCLIDEAN = 0, 1, 2


def rank_nd(Y):
    return dda.rank_canonical(np.asarray(Y, dtype=np.float64)).astype(np.intp)


def crowding_distance(Y):
    return indicators.crowding_distance_metric(np.asarray(Y, dtype=np.float64))


def euclidean_distance(Y):
    return indicators.euclidean_distance_metric(np.asarray(Y, dtype=np.float64))


def _order(Y, metric, extra):
    Y = np.asarray(Y, dtype=np.float64)
    rank = rank_nd(Y)
    keys = [-np.asarray(e, dtype=np.float64) for e in (extra or [])]
    dist = None
    if metric == METRIC_CROWDING:
        dist = crowding_distance(Y)
    elif metric == METRIC_EUCLIDEAN:
        dist = euclidean_distance(Y)
    if dist is not None:
        keys.append(-dist)
    perm = np.lexsort(keys + [rank])
    return perm, rank, dist


def order_mo(Y, metric=METRIC_NONE, extra_desc_keys=None):
    perm, rank, dist = _order(Y, metric, extra_desc_keys)
    return perm.astype(np.int64), rank[perm], (None if dist is None else dist[perm])


def remove_worst(X, Y, keep, metric=METRIC_NONE, extra_desc_keys=None):
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    perm, rank, _ = _order(Y, metric, extra_desc_keys)
    perm = perm[:keep]
    return X[perm], Y[perm], rank[perm], perm.astype(np.int64)


def remove_worst_pair(Xa, Ya, Xb, Yb, keep, metric=METRIC_NONE, out_X=None):
    Xo, Yo, rank, perm = remove_worst(np.vstack((Xa, Xb)), np.vstack((Ya, Yb)), keep, metric)
    if out_X is not None and out_X.dtype == np.float64 and out_X.shape == Xo.shape:
        out_X[:] = Xo
        Xo = out_X
    return Xo, Yo, rank, perm


def _rng(seed, stream_id):
    return np.random.default_rng([int(seed) & (2**63 - 1), int(stream_id)])


def tournament(rank, poolsize, seed, stream_id, crowd=None, return_uniforms=False):
    rank = np.asarray(rank)
    u = _rng(seed, stream_id).random(rank.shape[0])
    u = np.clip(u, 1e-300, 1 - 1e-16)
    metrics = (rank,) if crowd is None else (-np.asarray(crowd), rank)
    pool = moea.tournament_selection_gumbel(u, poolsize, *metrics).astype(np.int64)
    return (pool, u) if return_uniforms else pool


def mutation_u(parents, u, di_mutation, xlb, xub, mutation_rate):
    return moea.mutation_u(np.atleast_2d(parents), np.atleast_2d(u), di_mutation, np.asarray(xlb), np.asarray(xub), mutation_rate)


def sbx_u(parent1, parent2, u, di_crossover, xlb, xub):
    return moea.crossover_sbx_u(np.atleast_2d(parent1), np.atleast_2d(parent2), np.atleast_2d(u), di_crossover, np.asarray(xlb), np.asarray(xub))


def nsga2_generate(pop_x, pool_idx, popsize, crossover_prob, mutation_prob, mutation_rate, di_crossover, di_mutation, xlb, xub, seed, stream_id, return_draws=False):
    pop_x = np.asarray(pop_x, dtype=np.float64)
    d = pop_x.shape[1]
    T = 2 * popsize + 64
    r = _rng(seed, stream_id)
    poolsize = len(pool_idx)
    u_cross, u_mut = r.random(T), r.random(T)
    i1 = r.integers(0, poolsize, size=T)
    i2 = r.integers(0, max(poolsize - 1, 1), size=T)
    i2 = np.where(i2 >= i1, i2 + 1, i2) if poolsize > 1 else i2
    pair = np.stack((i1, i2), axis=1)
    single = r.integers(0, poolsize, size=T)
    u_genes = r.random((T, 2, d))
    pool = pop_x[np.asarray(pool_idx)]
    x_gen, cidx, midx = nsga2.generate_given_draws(pool, u_cross, u_mut, pair, single, u_genes, popsize, np.asarray(di_crossover), np.asarray(di_mutation),
                                                   np.asarray(xlb), np.asarray(xub), mutation_rate, crossover_prob, mutation_prob)
    kind = np.full(x_gen.shape[0], 2, dtype=np.int32)
    kind[cidx[0::2]] = 0
    kind[cidx[1::2]] = 1
    if return_draws:
        return x_gen, kind, {"u_cross": u_cross, "u_mut": u_mut, "pair": pair, "single": single, "u_genes": u_genes}
    return x_gen, kind


class GPHandle:
    def __init__(self, X_train, alpha, factor, constant, length_scale, noise, y_mean, y_std, xlb, xub, kernel=0, factor_is_inverse=False):
        if factor_is_inverse:  # the plugin uploads L^-1; the oracle works with L
            factor = [np.linalg.inv(np.asarray(f)) for f in factor]
        self.st = gp.GPState(X_train=np.asarray(X_train, float), xlb=np.asarray(xlb, float), xub=np.asarray(xub, float))
        self.M = len(alpha)
        for m in range(self.M):
            self.st.objectives.append(gp.GPObjective(np.asarray(alpha[m]), np.asarray(factor[m]), float(constant[m]), np.asarray(length_scale[m]),
                                                     float(noise[m]), float(y_mean[m]), float(y_std[m]), int(kernel)))

    def predict(self, X, return_var=True, precision=0):
        mean, var = gp.predict(self.st, X)
        return mean, (var if return_var else None)

    def close(self):
        pass


def hypervolume(F, ref):
    return hv.hypervolume(np.atleast_2d(F), ref)


def ehvi_select(F, means, variances, ref, k, nds=True, return_scores=False):
    F = np.asarray(F, dtype=np.float64)
    if nds:
        r0 = dda.rank_canonical(F)
        if np.any(r0 == 0):
            F = F[r0 == 0]
    sel, score = hv.select_candidates(F, means, variances, ref, k)
    return (sel.astype(np.int64), score) if return_scores else sel.astype(np.int64)


def get_duplicates(X, eps=1e-16, Y=None):
    return moea.get_duplicates(X, eps, Y=Y)


def age_survival(yn, nn, p, extreme):
    """Greedy loop of AGEMOEA.survival_score restated with the kernel's incremental two-smallest update."""
    from oracle import agemoea

    yn = np.asarray(yn, dtype=np.float64)
    m = yn.shape[0]
    dist = agemoea.minkowski(yn, yn, p) / np.asarray(nn)[:, None]
    crowd = np.zeros(m)
    selected = np.zeros(m, dtype=bool)
    selected[np.asarray(extreme)] = True
    crowd[selected] = np.inf
    remaining = [i for i in range(m) if not selected[i]]
    while remaining:
        sel = np.flatnonzero(selected)
        D = dist[np.ix_(sel, remaining)].T
        score = np.partition(D, 1, axis=1)[:, :2].sum(axis=1) if D.shape[1] > 1 else D[:, 0]
        j = int(np.argmax(score))
        best = remaining.pop(j)
        selected[best] = True
        crowd[best] = score[j]
    return crowd


def smpso_velocity(position, velocity, leader1, leader2, w, c1, r1, c2, r2, chi, xlb, xub):
    pos = np.asarray(position)
    d1 = np.asarray(np.asarray(leader1) - pos, dtype=np.float64)  # NumPy's own dtype promotion
    d2 = np.asarray(np.asarray(leader2) - pos, dtype=np.float64)
    delta = (np.asarray(xub, float) - np.asarray(xlb, float)) / 2
    out = (w * np.asarray(velocity, dtype=np.float64) + c1 * r1 * d1 + c2 * r2 * d2) * chi
    return np.clip(out, -delta, delta)


def mutate_groups(pop_x, group_size, n_groups, per_group, di_mutation, xlb, xub, mutation_rate, seed, stream_id, return_parents=False):
    pop_x = np.asarray(pop_x, dtype=np.float64)
    d = pop_x.shape[1]
    r = _rng(seed, stream_id)
    total = n_groups * per_group
    pi = r.integers(0, group_size, size=total) + np.repeat(np.arange(n_groups), per_group) * group_size
    u = r.random((total, d))
    out = moea.mutation_u(pop_x[pi], u, np.asarray(di_mutation), np.asarray(xlb), np.asarray(xub), mutation_rate)
    return (out, pi) if return_parents else out


def gp_fit(X_train, y, constant, length_scale, noise, kernel=0, jitter=1e-10, want_L=True, want_alpha=True):
    """dmo_gp_fit on the CPU: kernel matrix, Cholesky, alpha, log marginal likelihood per objective (oracle/gp.py)."""
    from scipy.linalg import cho_solve, cholesky

    X = np.asarray(X_train, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    M, N = y.shape
    Ls, als, lml = [], [], np.empty(M)
    for m in range(M):
        K = constant[m] * gp.kernel_matrix(X, X, np.asarray(length_scale[m], dtype=np.float64), kernel)
        K[np.diag_indices_from(K)] += noise[m] + jitter
        Lm = cholesky(K, lower=True, check_finite=False)
        a = cho_solve((Lm, True), y[m], check_finite=False)
        lml[m] = -0.5 * y[m] @ a - np.log(np.diag(Lm)).sum() - 0.5 * N * np.log(2 * np.pi)
        Ls.append(Lm)
        als.append(a)
    return (np.stack(Ls) if want_L else None), (np.stack(als) if want_alpha else None), lml


class ResidentRows:
    """NumPy-backed stand-in for _lib.ResidentRows (same surface: shape, __array__, indexing, copy)."""

    def __init__(self, a):
        self.a = np.array(a, dtype=np.float64)
        self.shape, self.dtype, self.ndim = self.a.shape, self.a.dtype, self.a.ndim

    def __len__(self):
        return self.shape[0]

    def __array__(self, dtype=None, copy=None):
        return self.a if dtype is None else self.a.astype(dtype)

    def __getitem__(self, key):
        return self.a[key]

    def copy(self):
        return ResidentRows(self.a)


def resident_rows(a):
    return a if isinstance(a, ResidentRows) else ResidentRows(a)


def gather_rows(src, idx, alt=None, sel=None):
    idx = np.asarray(idx, dtype=np.int64)
    out = np.asarray(src)[idx] if len(idx) else np.zeros((0,) + src.shape[1:])
    if sel is not None and len(idx):
        sel = np.asarray(sel, dtype=bool)
        out = out.copy()
        out[sel] = np.asarray(alt)[idx[sel]]
    return ResidentRows(out)


def identity_rows(n, d):
    return ResidentRows(np.broadcast_to(np.identity(d), (n, d, d)))


def rows_of(a):
    return resident_rows(a)


def scale_rows(rows, factors, seg_row=None, seg_start=None):
    f = np.asarray(factors, dtype=np.float64)
    if seg_row is None:
        rows.a *= f.reshape((-1,) + (1,) * (rows.a.ndim - 1))
        return rows
    for s, r in enumerate(np.asarray(seg_row)):
        for e in range(int(seg_start[s]), int(seg_start[s + 1])):
            rows.a[r] = rows.a[r] * f[e]
    return rows


def cmaes_generate(parents_x, sigmas, A, p_idx, z, xlb, xub):
    ind = cmaes_sample(parents_x, sigmas, A, p_idx, z)
    xlb, xub = np.asarray(xlb, dtype=np.float64), np.asarray(xub, dtype=np.float64)
    return np.clip((ind / np.max(np.abs(ind))) * (xub - xlb) + xlb, xlb, xub)


def cmaes_step_z(x_gen, cand_idx, parents_x, par_idx, xlb, xub, steps):
    z = np.divide(np.asarray(x_gen)[np.asarray(cand_idx)] - np.asarray(parents_x)[np.asarray(par_idx)], np.asarray(xub) - np.asarray(xlb)) / np.asarray(steps)
    return ResidentRows(z)


def cmaes_sample(parents_x, sigmas, A, p_idx, z):
    p_idx = np.asarray(p_idx)
    return np.asarray(parents_x)[p_idx] + np.asarray(sigmas)[p_idx] * np.einsum("ijk,ik->ij", np.asarray(A)[p_idx], np.asarray(z))


def cmaes_update_cholesky(A, Ainv, pc, z, psucc, cc, ccov, pthresh):
    from oracle import cmaes

    resident = isinstance(A, ResidentRows)
    A, Ainv, pc = np.array(A, dtype=float), np.array(Ainv, dtype=float), np.array(pc, dtype=float)
    for i in range(pc.shape[0]):
        A[i], Ainv[i], pc[i] = cmaes.update_cholesky(A[i], Ainv[i], np.asarray(z)[i], float(np.asarray(psucc)[i]), pc[i], cc, ccov, pthresh)
    return (ResidentRows(A), ResidentRows(Ainv), ResidentRows(pc)) if resident else (A, Ainv, pc)


SmpsoSwarms = None  # the CPU seam exercises the per-swarm host path of the SMPSO plugin; the resident path is a GPU test

FUNCTIONS = ["rank_nd", "crowding_distance", "euclidean_distance", "order_mo", "remove_worst", "remove_worst_pair", "tournament", "mutation_u", "sbx_u",
             "nsga2_generate", "GPHandle", "hypervolume", "ehvi_select", "get_duplicates", "age_survival", "smpso_velocity", "mutate_groups",
             "cmaes_sample", "cmaes_update_cholesky", "ResidentRows", "resident_rows", "gather_rows", "identity_rows", "rows_of", "scale_rows",
             "cmaes_generate", "cmaes_step_z", "SmpsoSwarms", "gp_fit"]


def install(monkeypatch):
    """Patch dmosopt_b200._lib in place for one test."""
    import sys

    from dmosopt_b200 import _lib

    me = sys.modules[__name__]
    for name in FUNCTIONS:
        monkeypatch.setattr(_lib, name, getattr(me, name))
