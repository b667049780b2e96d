"""GPU micro-timings of the individual hot-path kernels (CUDA events through the library's profile timers)."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dmosopt_b200 import _lib as L  # noqa: E402


def timed(fn, reps=3):
    fn()
    L.synchronize()
    best = 1e9
    for _ in range(reps):
        L.timer_begin()
        fn()
        best = min(best, L.timer_end())
    return best


def main():
    L.context()
    rng = np.random.default_rng(0)
    what = sys.argv[1] if len(sys.argv) > 1 else "rank"
    if what == "rank":
        for n, M, kind in [(131072, 3, "uniform"), (131072, 3, "sphere"), (131072, 2, "uniform"), (16384, 2, "uniform"), (65536, 5, "uniform")]:
            Y = rng.random((n, M))
            if kind == "sphere":
                Y = Y / np.linalg.norm(Y, axis=1, keepdims=True) * (1 + 0.01 * rng.random((n, 1)))
            d = L.DeviceArray((n, M)).upload(Y)
            r = L.DeviceArray((n,), np.int32)
            lib, ctx = L.load_library(), L.context()
            L.profile_enable(True)
            ms = timed(lambda: L._check(lib.dmo_rank_nd(ctx, d.ptr, n, M, r.ptr), "rank"))
            rep = L.profile_report()
            L.profile_enable(False)
            rk = r.download()
            print(f"rank n={n} M={M} {kind}: total {ms:.3f} ms, chain {rep['rank_chain'][0] / rep['rank_chain'][1]:.3f} ms, fronts {rk.max() + 1}, OCC={os.environ.get('DMO_RANK_OCC', 'default')}", flush=True)


def gp_sweep():
    """GP posterior at the BASELINE shape: fp64 vs tensor path, accuracy and time."""
    L.context()
    rng = np.random.default_rng(1)
    N, d, M, P = 4096, 30, 3, 65536
    from oracle import gp as ogp

    Xtr = rng.random((N, d))
    Ytr = np.column_stack([np.sin(3 * Xtr[:, :4].sum(axis=1) + k) + Xtr[:, 4 + k] ** 2 for k in range(M)])
    st = ogp.fit_fixed(Xtr, Ytr, np.zeros(d), np.ones(d), 1.0, 0.5, 1e-6)
    h = L.GPHandle(st.X_train, np.stack([o.alpha for o in st.objectives]), np.stack([o.L for o in st.objectives]), [o.constant for o in st.objectives],
                   [np.full(d, 0.5)] * M, [o.noise for o in st.objectives], [o.y_mean for o in st.objectives], [o.y_std for o in st.objectives],
                   np.zeros(d), np.ones(d))
    X = rng.random((P, d))
    Xd = L.DeviceArray((P, d)).upload(X)
    md, vd = L.DeviceArray((P, M)), L.DeviceArray((P, M))
    lib, ctx = L.load_library(), L.context()
    prior = np.array([(o.constant + o.noise) * o.y_std**2 for o in st.objectives])
    ref = None
    for name, prec in (("fp64", L.GP_FP64), ("tensor", L.GP_TENSOR)):
        L.profile_enable(True)
        ms = timed(lambda: L._check(lib.dmo_gp_predict(ctx, h._h, Xd.ptr, P, md.ptr, vd.ptr, prec), "gp"), reps=2)
        rep = L.profile_report()
        L.profile_enable(False)
        mean, var = md.download(), vd.download()
        if ref is None:
            ref = (mean, var)
            err = ""
        else:
            err = f" | vs fp64: var err/prior {np.max(np.abs(var - ref[1]) / prior):.2e}, mean err {np.max(np.abs(mean - ref[0])):.2e}"
        parts = ", ".join(f"{k} {v[0] / v[1]:.3f}" for k, v in rep.items())
        print(f"gp {name}: total {ms:.3f} ms [{parts}]{err}", flush=True)


def stream_sweep():
    """The HBM-bound kernels at the BASELINE shape: crowding / euclidean distance (n = 131072, M = 3), SBX + mutation
    (pop 65536, d 30), mean kernel's neighbours, hypervolume of a 65536-point 3-D front.  Prints time and the achieved
    fraction of the algorithmic bytes; run under ncu for the DRAM counters (profiles/README.md)."""
    L.context()
    rng = np.random.default_rng(2)
    lib, ctx = L.load_library(), L.context()
    n, M = 131072, 3
    Y = L.DeviceArray((n, M)).upload(rng.random((n, M)))
    D = L.DeviceArray((n,))
    for name, fn in (("crowding", lib.dmo_crowding_distance), ("euclidean", lib.dmo_euclidean_distance)):
        ms = timed(lambda: L._check(fn(ctx, Y.ptr, n, M, D.ptr), name))
        print(f"{name} n={n} M={M}: {ms:.3f} ms; minimum bytes 8nM + 8n = {(8 * n * M + 8 * n) / 1e6:.1f} MB -> {(8 * n * M + 8 * n) / ms / 1e6:.1f} GB/s on the algorithmic bytes", flush=True)
    pop, d = 65536, 30
    X = L.DeviceArray((pop, d)).upload(rng.random((pop, d)))
    pool = L.DeviceArray((pop // 2,), np.int64).upload(rng.permutation(pop)[: pop // 2].astype(np.int64))
    Xg = L.DeviceArray((pop + 1, d))
    kind = L.DeviceArray((pop + 1,), np.int32)
    nch = np.zeros(1, dtype=np.int64)
    one, twenty = L.DeviceArray((d,)).upload(np.full(d, 1.0)), L.DeviceArray((d,)).upload(np.full(d, 20.0))
    lb, ub = L.DeviceArray((d,)).upload(np.zeros(d)), L.DeviceArray((d,)).upload(np.ones(d))
    ms = timed(lambda: L._check(lib.dmo_nsga2_generate(ctx, X.ptr, pop, d, pool.ptr, pop // 2, pop, 0.9, 0.1, 1.0 / d, one.ptr, twenty.ptr, lb.ptr, ub.ptr,
                                                      7, 1, Xg.ptr, kind.ptr, nch.ctypes.data, None), "generate"))
    by = 8 * d * 2 * int(nch[0])
    print(f"variation pop={pop} d={d}: {ms:.3f} ms for {int(nch[0])} children; 8d B read + 8d B written per child = {by / 1e6:.1f} MB -> {by / ms / 1e6:.1f} GB/s", flush=True)
    x = rng.random((pop, 3))
    F = L.DeviceArray((pop, 3)).upload(x / np.linalg.norm(x, axis=1, keepdims=True))
    import ctypes

    out = ctypes.c_double(0.0)
    ref = np.full(3, 1.1)
    ms = timed(lambda: L._check(lib.dmo_hypervolume(ctx, F.ptr, pop, 3, ref.ctypes.data, ctypes.byref(out)), "hv"), reps=2)
    print(f"hypervolume n={pop} M=3 (whole set non-dominated): {ms:.3f} ms, value {out.value:.6f}", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "stream":
        stream_sweep()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "gp":
        gp_sweep()
        sys.exit(0)
    main()
