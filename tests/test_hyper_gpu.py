"""K8 and the consumers of `cbo_set_desc.hyper` on the GPU: bit-identity of hyper = NULL and hyper = (1, 1) on every path,
cbo_posterior_nll and the sweep / gradients at non-unit (s2, l) against oracle/hyper_oracle.py, the fit on the four golden
configurations against the oracle's multi-start L-BFGS-B, determinism, and the agent with --optimize_surrogates."""
import os

import numpy as np
import pytest

from helpers import make_case, rel_err
from oracle import cbo_oracle as O
from oracle import hyper_oracle as H

pytestmark = pytest.mark.gpu

# one set per K3 launch class: FMA separable / not, MMA separable / not, generic n > 48, non-causal, variable cost
CLASS_CASES = [dict(seed=601, N=120, d=2, c=1, n=9, p=(20, 24)), dict(seed=602, N=90, d=2, c=2, n=11, p=(7, 11)),
               dict(seed=603, N=150, d=2, c=1, n=20, p=(30, 32)), dict(seed=604, N=100, d=3, c=1, n=30, p=(8, 8, 8)),
               dict(seed=605, N=110, d=2, c=1, n=60, p=(20, 20)), dict(seed=606, N=50, d=2, c=1, n=12, p=(18, 18), causal=False),
               dict(seed=607, N=70, d=1, c=1, n=14, p=(40,), cost_variable=True)]
ARRAYS = ("mu", "var", "ei", "acq")


def engine(cases, **kw):
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    return SweepEngine([SetProblem(**k) for k, _ in cases], device="cuda:0", keep=ARRAYS, **kw)


def sweep_at(eng, best, task="min", hyper=None):
    """A full trial with the hyper buffers holding `hyper` (g -> (s2, l)) and no fit: K8 does not run."""
    import torch
    for g, v in (hyper or {}).items():
        eng.buf[eng.local_of[g]]["hyper"].copy_(torch.tensor(v, dtype=torch.float64))
    fit, eng.fit_hyper = eng.fit_hyper, False
    try:
        return eng.sweep(best, task)
    finally:
        eng.fit_hyper = fit


def oracle_state(ora, eng, g, s2, l):
    """Oracle posterior of set g at (s2, l) from the device's own prior at x_int (the input both sides share)."""
    if ora["causal"]:
        f = O.prior_factors(ora["gp"], ora["cond"], ora["cols"])
        mI, vI = eng.fetch("m_int", g), eng.fetch("v_int", g)
        post = H.posterior_fit(ora["XI"], ora["yI"], mI, vI, s2, l)
        kw = dict(gp=ora["gp"], factors=f, intervened_cols=ora["cols"])
    else:
        post, kw = H.posterior_fit(ora["XI"], ora["yI"], s2=s2, l=l), {}
    return post, dict(kw, fix_costs=ora["fix"], variable_cost=ora["variable"])


def test_null_and_unit_hyper_are_bit_identical(cuda_engine_ready):
    cases = [make_case(**s) for s in CLASS_CASES]
    best = float(min(np.min(k["y_int"]) for k, _ in cases))
    a, b = engine(cases), engine(cases, fit_hyperparameters=True)
    assert all(a.h_sets[i].hyper is None for i in range(len(cases))) and all(b.h_sets[i].hyper for i in range(len(cases)))
    oa, ob = a.sweep(best, "min"), sweep_at(b, best)
    assert oa.set_values.tobytes() == ob.set_values.tobytes() and list(oa.set_indices) == list(ob.set_indices)
    for g in range(len(cases)):
        for n in ("L", "alpha") + ARRAYS:
            assert a.fetch(n, g).tobytes() == b.fetch(n, g).tobytes(), (g, n)
        X = np.random.default_rng(g).uniform(-2, 2, (9, cases[g][0]["x_int"].shape[1]))
        ga, gb = a.acquisition_gradients(g, X, best), b.acquisition_gradients(g, X, best)
        for n in ga:
            assert ga[n].tobytes() == gb[n].tobytes(), (g, n)
        pa, pb = a.evaluate_points(g, X, best), b.evaluate_points(g, X, best)
        for n in pa:
            assert pa[n].tobytes() == pb[n].tobytes(), (g, n)
    ra, rb = a.refine(oa, best, "min", max_iter=8), b.refine(ob, best, "min", max_iter=8)
    assert ra.set_values.tobytes() == rb.set_values.tobytes()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(ra.set_x, rb.set_x))
    # post-intervention trial: the fused refresh (NULL) and the staged one (hyper = (1, 1), K8 not run): cached EI included
    g = oa.set
    kw = cases[g][0]
    x_new, y_new = np.vstack([kw["x_int"], oa.x[None, :]]), np.append(kw["y_int"], best - 0.3)
    for e in (a, b):
        e.set_interventional(g, x_new, y_new)
    fa = a.refresh(best - 0.3, "min", refit=[g])
    fit, b.fit_hyper = b.fit_hyper, False
    b.timing = True                                  # the staged path, as the engine takes it with the fit on
    fb = b.refresh(best - 0.3, "min", refit=[g])
    b.timing, b.fit_hyper = False, fit
    assert fa.set_values.tobytes() == fb.set_values.tobytes() and list(fa.set_indices) == list(fb.set_indices)
    for h in range(len(cases)):
        for n in ARRAYS:
            assert a.fetch(n, h).tobytes() == b.fetch(n, h).tobytes(), (h, n)


NLL_NS = [1, 2, 10, 17, 33, 48, 49, 100, 128]


@pytest.mark.parametrize("causal", [True, False])
def test_posterior_nll_and_fit_against_oracle(cuda_engine_ready, causal):
    rng = np.random.default_rng(611 + causal)
    specs = [dict(seed=620 + i, N=80, d=1 + i % 3, c=1, n=n, p=(6,) * (1 + i % 3), causal=causal) for i, n in enumerate(NLL_NS)]
    cases = [make_case(**s) for s in specs]
    hyp = [(float(np.exp(rng.uniform(np.log(0.05), np.log(50.0)))), float(np.exp(rng.uniform(np.log(0.2), np.log(3.0)))))
           for _ in cases]
    eng = engine(cases, fit_hyperparameters=True)
    sweep_at(eng, 0.0, hyper=dict(enumerate(hyp)))
    for g, ((kw, ora), (s2, l)) in enumerate(zip(cases, hyp)):
        assert eng.hyperparameters(g) == (s2, l)
        got = eng.posterior_nll(g)
        mI, vI = (eng.fetch("m_int", g), eng.fetch("v_int", g)) if causal else (None, None)
        resid = ora["yI"] - mI if causal else ora["yI"]
        f, gr, tries = H.nll(ora["XI"], resid, s2, l, vI)
        post = H.posterior_fit(ora["XI"], ora["yI"], mI, vI, s2, l)
        assert int(eng.buf[g]["fit_info"][0].item()) == tries == post["tries"], g
        cond = np.linalg.cond(H.gram(ora["XI"], s2, l, vI))
        scale = 1.0 if cond < 1e6 else cond * 1e-9
        assert abs(got[0] - f) <= 1e-6 * max(abs(f), 1.0) * scale, (g, got[0], f, cond)
        assert np.all(np.abs(got[1:] - gr) <= 1e-6 * max(np.abs(gr).max(), len(resid)) * scale), (g, got, gr, cond)
        L, alpha = eng.fetch("L", g), eng.fetch("alpha", g)
        Ky = H.gram(ora["XI"], s2, l, vI)
        assert np.abs(L @ L.T - Ky).max() <= 1e-12 * np.abs(Ky).max(), g
        if cond < 1e6:
            assert rel_err(L, post["L"], 1e-6).max() <= 1e-6 and rel_err(alpha, post["alpha"], 1e-6 * np.abs(post["alpha"]).max()).max() <= 1e-6
    # duplicated rows at a large variance and a long lengthscale: the Gram sits at the noise floor
    kw, ora = make_case(seed=630, N=60, d=1, c=1, n=100, p=(50,), causal=causal)
    kw["x_int"][1] = kw["x_int"][0]
    ora["XI"] = kw["x_int"]
    e2 = engine([(kw, ora)], fit_hyperparameters=True)
    sweep_at(e2, 0.0, hyper={0: (1e6, 40.0)})
    got = e2.posterior_nll(0)
    mI, vI = (e2.fetch("m_int", 0), e2.fetch("v_int", 0)) if causal else (None, None)
    f, _, tries = H.nll(ora["XI"], ora["yI"] - mI if causal else ora["yI"], 1e6, 40.0, vI)
    # the Gram's condition number is ~1e16 here, so the NLL itself is rounding noise: K2's factor must be backward stable for
    # the Gram plus whatever jitter it needed, and the NLL finite
    t = int(e2.buf[0]["fit_info"][0].item())
    Ky = H.gram(ora["XI"], 1e6, 40.0, vI)
    if t:
        Ky = Ky + np.eye(Ky.shape[0]) * np.mean(np.diag(Ky)) * 1e-6 * 10.0 ** (t - 1)
    L = e2.fetch("L", 0)
    assert np.abs(L @ L.T - Ky).max() <= 1e-12 * np.abs(Ky).max(), (t, tries)
    assert np.all(np.isfinite(got)), (got, f, t, tries)


def test_sweep_at_fitted_hyperparameters_against_oracle(cuda_engine_ready):
    cases = [make_case(**s) for s in CLASS_CASES]
    best = float(min(np.min(k["y_int"]) for k, _ in cases))
    hyp = {g: v for g, v in enumerate([(2.5, 0.7), (0.3, 1.9), (12.0, 0.45), (0.8, 2.5), (4.0, 0.9), (7.0, 0.6), (0.5, 1.3)])}
    eng = engine(cases, fit_hyperparameters=True)
    out = sweep_at(eng, best, hyper=hyp)

    def check(g, b):
        kw, ora = cases[g]
        s2, l = hyp[g]
        post, okw = oracle_state(ora, eng, g, s2, l)
        Xg = O.tensor_grid(ora["tables"])
        mg, vg = (eng.fetch("m", g), eng.fetch("v", g)) if ora["causal"] else (None, None)
        mu, var = H.posterior_predict(post, Xg, mg, vg)
        ei = O.expected_improvement(mu, var, b)
        acq = ei / O.point_cost(Xg, ora["fix"], ora["variable"])
        kd = s2 + (vg if vg is not None else 0.0)
        assert rel_err(eng.fetch("mu", g), mu, max(1e-4, 1e-3 * np.abs(mu).max())).max() <= 1e-6, g
        assert rel_err(eng.fetch("var", g), var, 1e-4 * kd).max() <= 1e-6, g
        scale = max(np.nanmax(np.abs(ei)), 1e-300)
        assert np.nanmax(rel_err(eng.fetch("acq", g), acq, 1e-6 * scale)) <= 1e-6, g
        return O.first_argmax(acq), acq

    for g in range(len(cases)):
        (i, v, _), acq = check(g, best)
        if out.set_indices[g] != i:                        # flat maximum: the two maxima agree to rounding
            assert abs(acq[out.set_indices[g]] - v) <= 1e-9 * abs(v), g
    # explicit points: the same arithmetic at arbitrary candidates
    for g in (1, 3, 5):
        kw, ora = cases[g]
        X = np.random.default_rng(g).uniform(-2, 2, (37, kw["x_int"].shape[1]))
        post, okw = oracle_state(ora, eng, g, *hyp[g])
        mg, vg = (eng.evaluate_points(g, X, stages="prior")["m"], eng.evaluate_points(g, X, stages="prior")["v"]) \
            if ora["causal"] else (None, None)
        mu, var = H.posterior_predict(post, X, mg, vg)
        got = eng.evaluate_points(g, X, best)
        assert rel_err(got["mu"], mu, max(1e-4, 1e-3 * np.abs(mu).max())).max() <= 1e-6
        assert rel_err(got["var"], var, 1e-4 * (hyp[g][0] + (vg if vg is not None else 0.0))).max() <= 1e-6
    # post-intervention trial: the refitted set and the cached EI refresh of the others, at the new incumbent
    g = out.set
    kw, ora = cases[g]
    x_new, y_new = np.vstack([kw["x_int"], out.x[None, :]]), np.append(kw["y_int"], best - 0.25)
    eng.set_interventional(g, x_new, y_new)
    cases[g] = (dict(kw, x_int=x_new, y_int=y_new), dict(ora, XI=x_new, yI=y_new))
    fit, eng.fit_hyper = eng.fit_hyper, False
    eng.timing = True
    out2 = eng.refresh(best - 0.25, "min", refit=[g])
    eng.timing, eng.fit_hyper = False, fit
    for h in range(len(cases)):
        (i, v, _), acq = check(h, best - 0.25)
        assert out2.set_indices[h] == i or abs(acq[out2.set_indices[h]] - v) <= 1e-9 * abs(v), h


def golden_engine(cfg, **kw):
    from cbo_with_oop_b200.engine import SweepEngine
    from cbo_with_oop_b200.fixtures import golden_path, load_golden_problems
    if not os.path.exists(golden_path(cfg)):
        pytest.fail("golden fixture missing")
    problems, best, task = load_golden_problems(cfg, device_fit=False)
    return problems, best, task, SweepEngine(problems, device="cuda:0", fit_hyperparameters=True, **kw)


@pytest.mark.parametrize("cfg", ["toy", "complete", "simplified_coral", "coral_synth"])
def test_fit_on_golden_configurations(cuda_engine_ready, cfg):
    from cbo_with_oop_b200.engine import hyper_bounds
    problems, best, task, eng = golden_engine(cfg)
    out = eng.sweep(best, task)
    worse = []
    for g, pr in enumerate(problems):
        r = eng.hyper_result(g)
        b = hyper_bounds(pr.grid)
        s2, l = eng.hyperparameters(g)
        assert (s2, l) == (r["variance"], r["lengthscale"]) and r["status"] != "not_positive_definite", (g, r)
        assert b[0] <= s2 <= b[1] and b[2] <= l <= b[3], (g, s2, l, b)
        if b[0] <= 1.0 <= b[1] and b[2] <= 1.0 <= b[3]:
            assert r["nll"] <= r["nll_start"], (g, r)
        mI, vI = eng.fetch("m_int", g), eng.fetch("v_int", g)
        resid = pr.y_int - mI
        f, gr, _ = H.nll(pr.x_int, resid, s2, l, vI)
        scale = max(1.0, np.linalg.cond(H.gram(pr.x_int, s2, l, vI)) * 1e-10)    # forward error grows with cond(Ky)
        assert abs(f - r["nll"]) <= 1e-6 * max(abs(f), 1.0) * scale, (g, f, r["nll"], scale)
        if r["status"] == "converged":
            pg = H.projected_gradient(np.log([s2, l]), gr, b)
            assert np.abs(pg).max() <= 1e-5 * scale, (g, pg, r)
        ref = H.fit(pr.x_int, resid, b, vI)["best"][0]
        if r["nll"] > ref + max(1e-6 * abs(ref), 1e-6):
            worse.append((g, r["nll"], ref, r["start"], r["status"]))
        # the posterior the sweep used is K2's at the fitted values
        assert int(eng.buf[g]["fit_info"][0].item()) == r["jitter_tries"] or r["jitter_tries"] < 0
    assert not worse, worse
    assert np.all(np.isfinite(out.set_values))


def test_fit_is_deterministic_and_independent_of_the_call(cuda_engine_ready):
    problems, best, task, eng = golden_engine("complete")
    eng.sweep(best, task)
    first = [eng.hyperparameters(g) for g in range(len(problems))]
    res1 = [str(eng.hyper_result(g)) for g in range(len(problems))]      # (repr of a float is exact; NaN compares equal)
    eng.sweep(best, task)
    assert [eng.hyperparameters(g) for g in range(len(problems))] == first
    assert [str(eng.hyper_result(g)) for g in range(len(problems))] == res1
    from cbo_with_oop_b200.engine import SweepEngine
    for g in (0, 3, 5):
        alone = SweepEngine([problems[g]], device="cuda:0", fit_hyperparameters=True)
        alone.sweep(best, task)
        assert alone.hyperparameters(0) == first[g] and str(alone.hyper_result(0)) == res1[g]
    # a 2-way partition on one GPU: set 4 is split between the ranks, each runs K8 on it redundantly
    ranks = [SweepEngine(problems, device="cuda:0", rank=r, world_size=2, fit_hyperparameters=True) for r in range(2)]
    split = [g for g in range(len(problems)) if all(g in e.local_of for e in ranks)]
    assert split
    for e in ranks:
        e.build_tables(); e.prior_precompute(); e.prior_eval(1); e.fit_hyperparameters()
    for g in set(ranks[0].local_of) | set(ranks[1].local_of):
        for e in ranks:
            if g in e.local_of:
                assert e.hyperparameters(g) == first[g], g


def test_gradients_and_refinement_at_fitted_hyperparameters(cuda_engine_ready):
    cases = [make_case(**s) for s in (CLASS_CASES[0], CLASS_CASES[2], CLASS_CASES[5], CLASS_CASES[6])]
    best = float(min(np.min(k["y_int"]) for k, _ in cases))
    eng = engine(cases, fit_hyperparameters=True)
    grid = eng.sweep(best, "min")
    for g, (kw, ora) in enumerate(cases):
        s2, l = eng.hyperparameters(g)
        assert eng.hyper_result(g)["start"] >= 0
        post, okw = oracle_state(ora, eng, g, s2, l)
        X = np.random.default_rng(g).uniform(-2, 2, (19, kw["x_int"].shape[1]))
        got = eng.acquisition_gradients(g, X, best)
        ref = H.acquisition_gradients(post, X, best, "min", **okw)
        for n in ("mu", "var", "ei", "acq", "dmu", "dvar", "dei", "dacq"):
            floor = max(1e-6 * np.max(np.abs(ref[n])), 1e-300)
            assert np.max(np.abs(got[n] - ref[n]) / np.maximum(np.abs(ref[n]), floor)) <= 1e-6, (g, n)
    out = eng.refine(grid, best, "min")
    for g, pr in enumerate(eng.problems):
        assert out.set_values[g] >= grid.set_values[g]
        assert all(min(t) <= v <= max(t) for t, v in zip(pr.grid, out.set_x[g]))


@pytest.fixture
def in_tmp(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)


@pytest.mark.parametrize("experiment,causal,trials", [("toy_graph", True, 10), ("simplified_coral_graph", True, 3),
                                                      ("toy_graph", False, 6)])
def test_agent_with_fitted_surrogates(cuda_engine_ready, in_tmp, experiment, causal, trials):
    from src.ArgumentParser import ArgumentParser
    from src.CBO import CBO
    from src.DataLoader import DataLoader
    # (--causal_prior is the reference's bool flag: any non-empty value enables it, so the non-causal run leaves it out)
    argv = ["--experiment", experiment, "--num_trials", str(trials), "--optimize_surrogates"] + (["--causal_prior", "1"] if causal else [])
    args = ArgumentParser().parse(argv=argv)
    assert args.optimize_surrogates
    args.grid_points, args.num_sem_samples = 40, 2000
    np.random.seed(args.seed)
    cbo = CBO(args, DataLoader(experiment, args.initial_num_obs_samples), verbose=False)
    if experiment == "simplified_coral_graph":
        # the reference's result file names spell out all 25 exploration sets: longer than a file name may be on Linux
        cbo.monitor.save_results = lambda: None
    cbo.run()
    session = cbo.get_session()
    assert session.engine.fit_hyper
    fitted = 0
    for s, model in enumerate(cbo.models):
        s2, l = model.kern.variance, model.kern.lengthscale
        r = session.engine.hyper_result(s)
        assert (s2, l) == session.engine.hyperparameters(s) == (r["variance"], r["lengthscale"])
        assert np.isfinite(model.log_likelihood())
        fitted += (s2, l) != (1.0, 1.0)
    assert fitted >= 1
