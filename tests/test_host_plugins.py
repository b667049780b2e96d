"""Host-side logic of the plugins (no GPU): the ``_lib`` calls are replaced by the oracle-backed test seam.

Checks the state handling / dtype flow of the plugins against golden vectors recorded from the reference plugins.
"""

import numpy as np
import pytest

import fake_backend
from conftest import load_golden


@pytest.fixture
def fake(monkeypatch):
    fake_backend.install(monkeypatch)


def test_nsga2_plugin_reproduces_reference_state_sequence(fake):
    import dmosopt_b200 as b2

    g = load_golden("nsga2")
    for k in range(int(g["ncases"])):
        if bool(g[f"c{k}_ties"]):
            continue  # objective ties: the reference's own result depends on unstable sorts
        metric = str(g[f"c{k}_metric"])
        metric = None if metric == "none" else metric
        x0, y0 = g[f"c{k}_x0"], g[f"c{k}_y0"]
        pop = g[f"c{k}_init_px"].shape[0]
        d, M = x0.shape[1], y0.shape[1]
        bounds = np.column_stack((np.zeros(d), np.ones(d)))
        opt = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=b2.Model(), distance_metric=metric)
        opt.initialize_strategy(x0, y0, bounds, np.random.default_rng(1))
        assert np.array_equal(opt.state.population_parm, g[f"c{k}_init_px"])
        assert np.array_equal(opt.state.population_obj, g[f"c{k}_init_py"])
        assert opt.state.population_obj.dtype == np.float32
        assert np.array_equal(opt.state.rank, g[f"c{k}_init_rank"])
        for gi in range(3):
            st = {"crossover_indices": g[f"c{k}_g{gi}_cidx"], "mutation_indices": g[f"c{k}_g{gi}_midx"]}
            opt.update(g[f"c{k}_g{gi}_xgen"], g[f"c{k}_g{gi}_ygen"], st)
            assert np.array_equal(opt.state.population_parm, g[f"c{k}_g{gi}_px"]), (k, gi)
            assert np.array_equal(opt.state.population_obj, g[f"c{k}_g{gi}_py"]), (k, gi)
            assert np.array_equal(opt.state.rank, g[f"c{k}_g{gi}_rank"]), (k, gi)


def test_nsga2_plugin_generate_contract(fake):
    import dmosopt_b200 as b2

    pop, d, M = 50, 7, 2
    rng = np.random.default_rng(0)
    bounds = np.column_stack((-np.ones(d), 2 * np.ones(d)))
    x0 = rng.uniform(-1, 2, size=(pop, d))
    y0 = rng.random((pop, M)).astype(np.float32)
    opt = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
    opt.initialize_strategy(x0, y0, bounds, rng)
    x_gen, st = opt.generate()
    assert x_gen.shape[1] == d and pop - 1 <= x_gen.shape[0] <= pop + 1  # NSGA2.py:142
    assert np.all(x_gen >= bounds[:, 0]) and np.all(x_gen <= bounds[:, 1])
    ci, mi = st["crossover_indices"], st["mutation_indices"]
    assert len(ci) % 2 == 0 and len(ci) + len(mi) == x_gen.shape[0]
    assert sorted(np.concatenate((ci, mi)).tolist()) == list(range(x_gen.shape[0]))
    assert opt.state.total_crossovers == len(ci) // 2 and opt.state.total_mutations == len(mi)
    px, py = opt.population_objectives
    assert px.shape == (pop, d) and py.shape == (pop, M)
    # same seed -> same offspring (Philox seed is drawn from the caller's generator)
    opt2 = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
    opt2.initialize_strategy(x0, y0, bounds, np.random.default_rng(0))
    opt3 = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
    opt3.initialize_strategy(x0, y0, bounds, np.random.default_rng(0))
    assert np.array_equal(opt2.generate()[0], opt3.generate()[0])


def test_gpr_matern_plugin_matches_reference_predictions(fake):
    import dmosopt_b200 as b2

    g = load_golden("gp")
    for k in (0, 1, 5):
        cls = b2.GPR_Matern if str(g[f"c{k}_kind"]) == "matern" else b2.GPR_RBF
        M = g[f"c{k}_yin"].shape[1]
        d = g[f"c{k}_xin"].shape[1]
        sm = cls(g[f"c{k}_xin"], g[f"c{k}_yin"], d, M, g[f"c{k}_xlb"], g[f"c{k}_xub"], optimizer=None)
        mean, var = sm.predict(g[f"c{k}_xtest"])
        np.testing.assert_allclose(mean, g[f"c{k}_mean"], rtol=1e-7, atol=1e-9)
        assert sm.evaluate(g[f"c{k}_xtest"]).shape == mean.shape
        sm.return_mean_variance = True
        assert len(sm.evaluate(g[f"c{k}_xtest"])) == 2


def _run_plugin_goldens(b2):
    """Shared by the CPU (oracle-backed seam) and GPU runs: reference plugin state sequences (tests/golden/plugins.npz)."""
    from conftest import sort_rows

    g = load_golden("plugins")
    d, M = 8, 3
    bounds = np.column_stack((np.zeros(d), np.ones(d)))
    # ---- AGE-MOEA: the selected set, ranks and crowding values (row order inside a front is unstable in the reference)
    pop = g["age_g0_px"].shape[0]
    opt = b2.AGEMOEA(popsize=pop, nInput=d, nOutput=M, model=b2.Model())
    opt.initialize_strategy(g["age_x0"], g["age_y0"], bounds, np.random.default_rng(3))
    assert np.array_equal(np.sort(opt.state.rank), np.sort(g["age_init_rank"]))
    np.testing.assert_allclose(np.sort(opt.state.crowd_dist), np.sort(g["age_init_cd"]), rtol=1e-5)
    # from here on continue from the reference's own state (its initial row order is implementation defined)
    for gi in range(2):
        opt.update(g[f"age_g{gi}_xgen"], g[f"age_g{gi}_ygen"], {})
        assert np.array_equal(sort_rows(opt.state.population_parm), sort_rows(g[f"age_g{gi}_px"])), gi
        assert np.array_equal(sort_rows(opt.state.population_obj), sort_rows(g[f"age_g{gi}_py"])), gi
        assert np.array_equal(np.sort(opt.state.rank), np.sort(g[f"age_g{gi}_rank"]))
        np.testing.assert_allclose(np.sort(opt.state.crowd_dist), np.sort(g[f"age_g{gi}_cd"]), rtol=1e-5)
        opt.state.population_parm[:] = g[f"age_g{gi}_px"]
        opt.state.population_obj[:] = g[f"age_g{gi}_py"]
        opt.state.rank[:] = g[f"age_g{gi}_rank"]
        opt.state.crowd_dist[:] = g[f"age_g{gi}_cd"]
    x_gen, _ = opt.generate()
    assert pop - 1 <= x_gen.shape[0] <= pop + 1
    # ---- SMPSO: exact state after initialize and after one update driven by the same NumPy generator
    pop_s = g["smpso_init_px"].shape[0] // 5
    opt = b2.SMPSO(popsize=pop_s, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
    opt.initialize_strategy(g["smpso_x0"], g["smpso_y0"], bounds, np.random.default_rng(11))
    assert np.array_equal(opt.state.population_parm, g["smpso_init_px"]) and np.array_equal(opt.state.population_obj, g["smpso_init_py"])
    assert np.array_equal(opt.state.velocity, g["smpso_init_vel"])
    xg, _ = opt.generate()
    assert list(xg.shape) == list(g["smpso_xgen_shape"]) and xg.dtype == g["smpso_xgen"].dtype
    assert np.array_equal(xg.reshape(5, 2 * pop_s, d)[:, :pop_s], g["smpso_xgen_positions"])
    assert np.all(xg >= 0) and np.all(xg <= 1)
    opt.local_random = np.random.default_rng(12)
    opt.update(g["smpso_xgen"], g["smpso_ygen"], {})
    np.testing.assert_allclose(opt.state.velocity, g["smpso_g0_vel"], rtol=1e-13, atol=1e-15)
    assert np.array_equal(opt.state.population_parm, g["smpso_g0_px"]) and np.array_equal(opt.state.population_obj, g["smpso_g0_py"])
    assert np.array_equal(np.stack(opt.state.ranks), g["smpso_g0_ranks"]) and opt.state.successful_children == int(g["smpso_succ"])
    # ---- MO-CMA-ES: three full updates on the recorded offspring
    popc = g["cma_init_px"].shape[0]
    opt = b2.CMAES(popsize=popc, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
    opt.initialize_strategy(g["cma_x0"], g["cma_y0"], bounds, np.random.default_rng(21))
    assert np.array_equal(opt.state.parents_x, g["cma_init_px"]) and np.array_equal(opt.state.sigmas, g["cma_init_sig"])
    for gi in range(3):
        opt.update(g[f"cma_g{gi}_xgen"], g[f"cma_g{gi}_ygen"], {"p_idx": g[f"cma_g{gi}_pidx"]})
        assert np.array_equal(opt.state.parents_x, g[f"cma_g{gi}_px"]), gi
        assert np.array_equal(opt.state.parents_y, g[f"cma_g{gi}_py"]) and np.array_equal(opt.state.rank, g[f"cma_g{gi}_rank"])
        np.testing.assert_allclose(opt.state.psucc, g[f"cma_g{gi}_psucc"], rtol=1e-13)
        np.testing.assert_allclose(opt.state.sigmas, g[f"cma_g{gi}_sig"], rtol=1e-13)
        np.testing.assert_allclose(opt.state.A, g[f"cma_g{gi}_A"], rtol=1e-11, atol=1e-13)
        np.testing.assert_allclose(opt.state.Ainv, g[f"cma_g{gi}_Ainv"], rtol=1e-11, atol=1e-13)
        np.testing.assert_allclose(opt.state.pc, g[f"cma_g{gi}_pc"], rtol=1e-12, atol=1e-15)
    x_new, stg = opt.generate()
    assert x_new.shape == (opt.opt_params.mu, d) and len(stg["p_idx"]) == opt.opt_params.mu
    px, py = opt.population_objectives
    assert px.shape[1] == d and py.shape[1] == M


def _run_trs_golden(b2):
    """Trust-region search: exact state sequence of the reference over three generate / update rounds (tests/golden/trs.npz).
    The Sobol perturbations come from scipy's sampler seeded by the caller's generator, so generate() itself is reproduced."""
    g = load_golden("trs")
    d, M = g["x0"].shape[1], g["y0"].shape[1]
    pop = g["init_px"].shape[0]
    bounds = np.column_stack((np.zeros(d), np.ones(d)))
    opt = b2.TRS(popsize=pop, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
    opt.initialize_strategy(g["x0"].copy(), g["y0"].copy(), bounds, np.random.default_rng(31))
    assert np.array_equal(opt.state.population_parm, g["init_px"]) and np.array_equal(opt.state.population_obj, g["init_py"])
    assert np.array_equal(opt.state.rank, g["init_rank"])
    for gi in range(3):
        xg, stg = opt.generate()
        assert np.array_equal(xg, g[f"g{gi}_xgen"]), gi
        opt.update(xg, g[f"g{gi}_ygen"], stg)
        assert np.array_equal(opt.state.population_parm, g[f"g{gi}_px"]), gi
        assert np.array_equal(opt.state.population_obj, g[f"g{gi}_py"]), gi
        assert np.array_equal(opt.state.rank, g[f"g{gi}_rank"]), gi
        assert opt.state.tr.length == float(g[f"g{gi}_length"])


def test_trs_plugin_reproduces_reference(fake):
    import dmosopt_b200 as b2

    _run_trs_golden(b2)


def test_age_smpso_cmaes_plugins_reproduce_reference(fake):
    import dmosopt_b200 as b2

    _run_plugin_goldens(b2)


def test_adaptive_helpers_reproduce_reference(fake):
    """update_population_size (NSGA2 / AGEMOEA / SMPSO / CMAES / TRS) and update_operator_rates (NSGA2 / SMPSO) against
    the reference's own results on crafted states (tests/golden/adaptive.npz): host control logic of the plugin contract."""
    import dmosopt_b200 as b2

    g = load_golden("adaptive")
    x0, y0 = g["x0"], g["y0"]
    pop, d, M = x0.shape[0], x0.shape[1], y0.shape[1]
    bounds = np.column_stack((np.zeros(d), np.ones(d)))
    n = int(g["n_cases"])
    for name, cls, kw in (("nsga2", b2.NSGA2, {}), ("age", b2.AGEMOEA, {}), ("cma", b2.CMAES, {"distance_metric": None}), ("trs", b2.TRS, {})):
        for k in range(n):
            opt = cls(popsize=pop, nInput=d, nOutput=M, model=b2.Model(), **kw)
            opt.initialize_strategy(x0.copy(), y0.copy(), bounds, np.random.default_rng(1))
            opt.state.rank = g[f"c{k}_rank"].copy()
            if name == "cma":
                opt.state.parents_y = g[f"c{k}_obj"].copy()
            else:
                opt.state.population_obj = g[f"c{k}_obj"].copy()
            opt.opt_params.max_population_size, opt.opt_params.min_population_size = 90, 20
            opt.update_population_size()
            assert opt.opt_params.popsize == int(g[f"{name}_c{k}_popsize"]), (name, k)
            if name == "nsga2":
                assert opt.opt_params.poolsize == int(round(opt.opt_params.popsize / 2.0))
    for k in range(n):
        opt = b2.SMPSO(popsize=pop // 5, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
        opt.initialize_strategy(x0.copy(), y0.astype(np.float32), bounds, np.random.default_rng(1))
        r = g[f"c{k}_rank"]
        opt.state.ranks = [r[s * (pop // 5) : (s + 1) * (pop // 5)].copy() for s in range(5)]
        opt.state.population_obj = g[f"c{k}_obj"].copy()
        opt.opt_params.max_population_size, opt.opt_params.min_population_size = 30, 4
        opt.update_population_size()
        assert opt.opt_params.popsize == int(g[f"smpso_c{k}_popsize"]), k
    first = lambda v: float(np.atleast_1d(np.asarray(v, dtype=float)).ravel()[0])  # noqa: E731
    for k in range(int(g["n_rates"])):
        sc, tc, smu, tmu = (int(v) for v in g[f"nsga2_rates{k}_in"])
        opt = b2.NSGA2(popsize=pop, nInput=d, nOutput=M, model=b2.Model())
        opt.initialize_strategy(x0.copy(), y0.copy(), bounds, np.random.default_rng(1))
        for rnd in range(2):
            st, p = opt.state, opt.opt_params
            st.successful_crossovers, st.total_crossovers, st.successful_mutations, st.total_mutations = sc, tc, smu, tmu
            opt.update_operator_rates()
            got = [first(p.di_crossover), float(p.crossover_prob), first(p.di_mutation), float(p.mutation_prob), float(p.mutation_rate),
                   st.successful_crossovers, st.total_crossovers, st.successful_mutations, st.total_mutations]
            np.testing.assert_allclose(got, g[f"nsga2_rates{k}"][rnd], rtol=1e-15, atol=0, err_msg=str((k, rnd)))
        opt = b2.SMPSO(popsize=pop // 5, nInput=d, nOutput=M, model=b2.Model(), distance_metric=None)
        opt.initialize_strategy(x0.copy(), y0.astype(np.float32), bounds, np.random.default_rng(1))
        for rnd in range(2):
            opt.state.successful_children = sc
            opt.update_operator_rates()
            got = [first(opt.opt_params.di_mutation), float(opt.opt_params.mutation_rate), float(opt.state.successful_children)]
            np.testing.assert_allclose(got, g[f"smpso_rates{k}"][rnd], rtol=1e-15, atol=0, err_msg=str((k, rnd)))
