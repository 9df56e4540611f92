"""The reference-shaped Python API (`src` package) on the GPU: DoCalculus closures, GaussianProcessFactory models,
CausalExpectedImprovement / Cost / find_next_y_point, the batched CBO.compute_best_acquisition_values, and a short
end-to-end run of the agent -- each checked against the oracle restatement of the reference's arithmetic."""
import os
import types

import numpy as np
import pytest

from helpers import RTOL, rel_err
from oracle import cbo_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def in_tmp(tmp_path, monkeypatch):
    """The agent saves its results under ./data/: keep them in a per-test directory."""
    monkeypatch.chdir(tmp_path)


def make_agent(experiment="toy_graph", n_obs=60, trials=4, causal=True, p=40):
    from src.CBO import CBO
    from src.DataLoader import DataLoader
    args = types.SimpleNamespace(exploration_set="MIS", initial_num_obs_samples=n_obs, num_interventions=10, type_cost=1,
                                 num_additional_observations=20, num_trials=trials, name_index=0, seed=9, causal_prior=causal,
                                 experiment=experiment, task="min", grid_points=p, device="cuda:0", num_sem_samples=2000)
    np.random.seed(args.seed)
    return CBO(args, DataLoader(experiment, n_obs), verbose=False)


def oracle_inputs(cbo, s):
    pr = cbo.do_calculus.set_problem(s)
    X = np.hstack([pr.x_obs_int, pr.x_obs_cond])
    gp = dict(X=X, variance=pr.s2, lengthscale=np.concatenate([pr.ls_int, pr.ls_cond]), noise=pr.noise, alpha=pr.alpha_obs,
              Kyinv=pr.kyinv, form="diff")
    gp["L"] = np.linalg.cholesky(np.linalg.inv(pr.kyinv))  # only for the direct (loop) form
    return pr, gp, X


def bounded_gps(cbo):
    """Observational GPs with a lengthscale floor (see tests/golden/make_golden.py for why)."""
    from cbo_with_oop_b200.obs_gp import fit_state, optimize_hyperparameters
    from src.utils_functions.utils import ObservationalGP
    g = cbo.graph
    meas = {v: np.asarray(cbo.measurements[v], np.float64).reshape(-1, 1) for v in g.var_names}
    gps = {}
    for s in cbo.exploration_set:
        cols = g.prior_columns(s)
        x, y = np.hstack([meas[c] for c in cols]), meas["Y"].reshape(-1)
        s2, ls = optimize_hyperparameters(x, y, 1.0, 1.0, False, 1e-2, min_lengthscale=float(0.5 * x.std(0).max()), max_variance=20.0)
        alpha, kyinv = fit_state(x, y, s2, ls, 1e-2)
        gps[g.get_gp_name(cols)] = ObservationalGP(x, y.reshape(-1, 1), s2, ls, 1e-2, alpha, kyinv, False)
    return gps


def test_do_functions_match_direct_form(cuda_engine_ready):
    """mean_fn / var_fn closures (DoCalculus.py:14-66) against the reference-faithful per-candidate loop."""
    cbo = make_agent("complete_graph", n_obs=50)
    mean_fns, var_fns = cbo.do_calculus.update_all_do_functions(bounded_gps(cbo))
    rng = np.random.default_rng(3)
    for s in [0, 1, 3, 5]:
        pr, gp, X = oracle_inputs(cbo, s)
        lo = np.array([t[0] for t in pr.grid]); hi = np.array([t[-1] for t in pr.grid])
        vals = rng.uniform(lo, hi, (9, pr.d))
        m_ref, v_ref = O.do_prior_direct(gp, X, list(range(pr.d)), vals)
        m, v = mean_fns[s](vals), var_fns[s](vals)
        assert m.shape == (9, 1) and v.shape == (9, 1) and m.dtype == np.float64
        assert rel_err(m[:, 0], m_ref, 1e-6).max() <= RTOL
        assert rel_err(v[:, 0], v_ref, 1e-6).max() <= RTOL
        # memo keyed by str(value), as in the reference (cbo.x_mean / cbo.x_var)
        assert str(vals[0]) in cbo.x_mean[cbo.intervention_names[s]]
        np.testing.assert_array_equal(mean_fns[s](vals[:3]), m[:3])


def test_factory_models_and_single_set_api(cuda_engine_ready):
    """GaussianProcessFactory.create -> model.predict, CausalExpectedImprovement.evaluate, Cost, find_next_y_point
    (single-set form) and the batched CBO.compute_best_acquisition_values agree with each other and the oracle."""
    from src.GaussianProcessFactory import GaussianProcessFactory, GaussianProcessType
    from src.utils_functions import CausalExpectedImprovement, Cost, find_next_y_point
    cbo = make_agent("complete_graph", n_obs=50, p=100)
    cbo.mean_functions, cbo.var_functions = cbo.do_calculus.update_all_do_functions(bounded_gps(cbo))
    cbo.update_all_gaussian_processes()
    best = float(cbo.current_best_solution())
    xs, ys = cbo.compute_best_acquisition_values(best)
    rng = np.random.default_rng(5)
    for s in range(cbo.es_size):
        pr, gp, X = oracle_inputs(cbo, s)
        ref = O.sweep_set(gp, X, list(range(pr.d)), pr.x_int, pr.y_int, pr.grid, best, "min", fix_costs=np.array([pr.cost_fix]),
                          form="diff")
        assert xs[s].shape == (1, pr.d) and ys[s].shape == (1, 1)
        np.testing.assert_array_equal(xs[s][0], ref["x"])
        np.testing.assert_allclose(ys[s][0, 0], ref["val"], rtol=RTOL)
        # explicit points through the model object
        lo = np.array([t[0] for t in pr.grid]); hi = np.array([t[-1] for t in pr.grid])
        Xq = rng.uniform(lo, hi, (17, pr.d))
        f = O.prior_factors(gp, X, list(range(pr.d)))
        mq, vq = O.do_prior_factorised(gp, f, list(range(pr.d)), Xq)
        post = O.posterior_fit(pr.x_int, pr.y_int, ref["mI"], ref["vI"], form="diff")
        mu_ref, var_ref = O.posterior_predict(post, Xq, mq, vq)
        mu, var = cbo.models[s].predict(Xq)
        assert mu.shape == (17, 1) and var.shape == (17, 1)
        assert rel_err(mu[:, 0], mu_ref, 1e-4).max() <= RTOL
        assert rel_err(var[:, 0], var_ref, 1e-4 * (1 + vq)).max() <= RTOL
        acq = CausalExpectedImprovement(best, "min", cbo.models[s]) / Cost(cbo.costs, cbo.exploration_set[s])
        ei_ref = O.expected_improvement(mu_ref, var_ref, best, "min") / pr.cost_fix
        assert rel_err(acq.evaluate(Xq)[:, 0], ei_ref, 1e-6 * np.abs(ei_ref).max()).max() <= RTOL
        # single-set search == batched search
        y1, x1 = find_next_y_point(cbo.monitor.space_list[s], cbo.models[s], best, cbo.exploration_set[s], cbo.costs, task="min")
        np.testing.assert_array_equal(x1, xs[s])
        np.testing.assert_array_equal(y1, ys[s])
    sel_set, sel = cbo.select_next_intervention(ys)
    assert sel == int(np.argmax([y[0, 0] for y in ys])) and sel_set == cbo.exploration_set[sel]
    # a model built from plain Python callables (not DoCalculus closures) goes through the external-prior path
    s = 3
    pr, gp, X = oracle_inputs(cbo, s)
    f = O.prior_factors(gp, X, list(range(pr.d)))
    mean_fn = lambda v: O.do_prior_factorised(gp, f, list(range(pr.d)), v)[0].reshape(-1, 1)
    var_fn = lambda v: O.do_prior_factorised(gp, f, list(range(pr.d)), v)[1].reshape(-1, 1)
    generic = GaussianProcessFactory.create(GaussianProcessType.CAUSAL_GP, pr.x_int, pr.y_int.reshape(-1, 1), [mean_fn, var_fn], True)
    Xq = rng.uniform(-1, 1, (5, pr.d))
    mu_g, var_g = generic.predict(Xq)
    mu_s, var_s = cbo.models[s].predict(Xq)
    assert rel_err(mu_g, mu_s, 1e-4).max() <= RTOL and rel_err(var_g, var_s, 1e-4).max() <= RTOL
    y2, x2 = find_next_y_point(cbo.monitor.space_list[s], generic, best, cbo.exploration_set[s], cbo.costs, task="min")
    np.testing.assert_array_equal(x2, xs[s])
    np.testing.assert_allclose(y2, ys[s], rtol=RTOL)


@pytest.mark.parametrize("causal", [True, False])
def test_agent_runs_end_to_end(cuda_engine_ready, causal):
    """runCBO.py's loop on the toy graph: observe / intervene trials, results saved with the reference's file names."""
    cbo = make_agent("toy_graph", n_obs=60, trials=5, causal=causal, p=50)
    cbo.run()
    m = cbo.monitor
    assert len(m.global_opt) == 1 + cbo.num_trials and len(m.current_cost) == 1 + cbo.num_trials
    assert m.type_trial[0] == 0 and m.type_trial[1] == 1
    assert np.all(np.diff(m.global_opt) <= 1e-12)           # the incumbent never gets worse (task = min)
    n_int = int(np.sum(m.type_trial))
    assert sum(len(x) for x in m.data_x) == 10 * cbo.es_size + n_int
    index = f"{cbo.exploration_set}_{cbo.gp_type}_{cbo.name_index}"
    assert os.path.exists(cbo.saving_dir + f"global_opt_{index}.npy")
