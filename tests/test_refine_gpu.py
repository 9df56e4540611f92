"""K7 on the GPU: cbo_acq_grad against the oracle's analytic gradients, cbo_refine against the oracle's L-BFGS-B refinement,
its invariants (box, bounds, determinism, independence of the other sets, bit-exact fall-back to the grid result) and the
agent with --refine_acquisition."""
import ctypes as C
import os
import types

import numpy as np
import pytest

from helpers import make_case
from oracle import cbo_oracle as O
from oracle import refine_oracle as R

pytestmark = pytest.mark.gpu


def rule(got, ref, rtol=1e-6):
    """max relative error with a floor of 1e-6 max|ref| (the 1e-6 rule of the feature)."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    floor = max(1e-6 * np.max(np.abs(ref)), 1e-300)
    return float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), floor)))


def oracle_state(ora):
    if ora["causal"]:
        f = O.prior_factors(ora["gp"], ora["cond"], ora["cols"])
        mI, vI = O.do_prior_factorised(ora["gp"], f, ora["cols"], ora["XI"], precise=True)
        post = O.posterior_fit(ora["XI"], ora["yI"], mI, vI, form="diff")
        kw = dict(gp=ora["gp"], factors=f, intervened_cols=ora["cols"])
    else:
        post = O.posterior_fit(ora["XI"], ora["yI"], form="diff")
        kw = {}
    return post, dict(kw, fix_costs=ora["fix"], variable_cost=ora["variable"])


def engine(cases, **kw):
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    return SweepEngine([SetProblem(**k) for k, _ in cases], device="cuda:0", **kw)


GRAD_CASES = [dict(seed=401, N=1, d=1, c=1, n=5, p=(30,)), dict(seed=402, N=127, d=2, c=1, n=15, p=(20, 20)),
              dict(seed=403, N=128, d=3, c=2, n=17, p=(8, 8, 8)), dict(seed=404, N=129, d=4, c=1, n=47, p=(5, 5, 5, 5)),
              dict(seed=405, N=1000, d=2, c=2, n=49, p=(30, 30), cost_variable=True), dict(seed=406, N=4000, d=3, c=1, n=20, p=(10, 10, 10)),
              dict(seed=407, N=300, d=1, c=0, n=8, p=(50,), ard=False), dict(seed=408, N=50, d=2, c=1, n=30, p=(20, 20), causal=False),
              dict(seed=409, N=50, d=4, c=1, n=12, p=(4, 4, 4, 4), causal=False, cost_variable=True)]


@pytest.mark.parametrize("spec", GRAD_CASES, ids=lambda s: f"N{s['N']}-d{s['d']}-n{s['n']}{'' if s.get('causal', True) else '-plain'}")
@pytest.mark.parametrize("task", ["min", "max"])
def test_acq_grad_matches_oracle(cuda_engine_ready, spec, task):
    kw, ora = make_case(**spec)
    best = float(np.min(ora["yI"]) if task == "min" else np.max(ora["yI"]))
    eng = engine([(kw, ora)])
    eng.sweep(best, task)
    rng = np.random.default_rng(spec["seed"])
    X = rng.uniform(-2.0, 2.0, (19, spec["d"]))           # three batches of 8, the last one partial
    got = eng.acquisition_gradients(0, X, best, task)
    post, okw = oracle_state(ora)
    ref = R.acquisition_gradients(post, X, best, task, **okw)
    for n in ("m", "v", "mu", "var", "ei", "acq", "dm", "dv", "dmu", "dvar", "dei", "dacq"):
        assert got[n].shape == ref[n].shape, n
        if not ora["causal"] and n in ("m", "v", "dm", "dv"):
            assert np.all(got[n] == 0.0), n
            continue
        assert rule(got[n], ref[n]) <= 1e-6, (n, rule(got[n], ref[n]))
    # the values are the sweep's own arithmetic at explicit points
    pts = eng.evaluate_points(0, X, best, task)
    assert rule(got["acq"], pts["acq"]) <= 1e-6


REFINE_CASES = [dict(seed=411, N=200, d=1, c=1, n=6, p=(25,)), dict(seed=412, N=300, d=2, c=2, n=9, p=(15, 15)),
                dict(seed=413, N=150, d=3, c=1, n=12, p=(9, 9, 9), cost_variable=True),
                dict(seed=414, N=60, d=2, c=1, n=10, p=(12, 12), causal=False)]


def box(pr):
    return np.array([t.min() for t in pr.grid]), np.array([t.max() for t in pr.grid])


def test_refine_against_oracle(cuda_engine_ready):
    cases = [make_case(**s) for s in REFINE_CASES]
    best = float(min(np.min(k["y_int"]) for k, _ in cases))
    eng = engine(cases)
    grid = eng.sweep(best, "min")
    out = eng.refine(grid, best, "min")
    for g, (kw, ora) in enumerate(cases):
        pr = eng.problems[g]
        lo, hi = box(pr)
        x, val = out.set_x[g], out.set_values[g]
        assert val >= grid.set_values[g], g
        assert np.all(x >= lo) and np.all(x <= hi)
        assert abs(eng.evaluate_points(g, x[None, :], best, "min")["acq"][0] - val) <= 1e-6 * abs(val)
        post, okw = oracle_state(ora)
        assert abs(R.acquisition_gradients(post, x[None, :], best, "min", **okw)["acq"][0] - val) <= 1e-6 * abs(val)
        ref = R.refine_set(post, eng_grid_x(pr, grid.set_indices[g]), pr.grid, best, "min", **okw)
        assert abs(ref["value"] - val) <= 1e-6 * abs(ref["value"]), (g, ref["value"], val, out.refine_status[g])
        if ref["interior"] and ref["hess_negdef"]:
            assert np.all(np.abs(ref["x"] - x) <= 1e-4 * (hi - lo)), (g, ref["x"], x)
    # global selection: first maximum over the refined per-set values
    assert out.set == int(np.argmax(out.set_values)) and out.value == out.set_values[out.set]
    np.testing.assert_array_equal(out.x, out.set_x[out.set])


def eng_grid_x(pr, idx):
    ii = np.unravel_index(int(idx), [len(t) for t in pr.grid])
    return np.array([pr.grid[k][ii[k]] for k in range(pr.d)])


def test_refine_pins_bound_exactly(cuda_engine_ready):
    """A set whose constrained maximum lies on the upper bound of dimension 1 and inside the box in dimension 0: the pinned
    coordinate equals the bound exactly while the free one moves off the grid."""
    kw, ora = make_case(seed=421, N=40, d=2, c=1, n=8, p=(40, 40), causal=False)
    best = float(np.min(kw["y_int"]))
    eng = engine([(kw, ora)])
    grid = eng.sweep(best, "min")
    out = eng.refine(grid, best, "min")
    x = out.set_x[0]
    assert out.set_values[0] > grid.set_values[0]
    assert x[1] == kw["grid"][1][-1], (x, out.refine_status)
    assert kw["grid"][0][0] < x[0] < kw["grid"][0][-1] and not np.any(kw["grid"][0] == x[0])


def test_refine_deterministic_and_independent_of_other_sets(cuda_engine_ready):
    cases = [make_case(**s) for s in REFINE_CASES]
    best = float(min(np.min(k["y_int"]) for k, _ in cases))
    eng = engine(cases)
    grid = eng.sweep(best, "min")
    a = eng.refine(grid, best, "min")
    b = eng.refine(grid, best, "min")
    for g in range(len(cases)):
        assert a.set_values[g].tobytes() == b.set_values[g].tobytes()
        assert a.set_x[g].tobytes() == b.set_x[g].tobytes()
    for g in (1, 2):
        alone = engine([cases[g]])
        ga = alone.sweep(best, "min")
        assert ga.set_indices[0] == grid.set_indices[g]
        r = alone.refine(ga, best, "min")
        assert r.set_values[0].tobytes() == a.set_values[g].tobytes()
        assert r.set_x[0].tobytes() == a.set_x[g].tobytes()


def test_skipped_and_non_improving_sets_keep_the_grid_result(cuda_engine_ready):
    from cbo_with_oop_b200 import _lib
    from cbo_with_oop_b200.engine import SetProblem
    kw, ora = make_case(seed=431, N=150, d=2, c=1, n=9, p=(15, 15))
    res = O.sweep_set(ora["gp"], ora["cond"], ora["cols"], ora["XI"], ora["yI"], ora["tables"], float(np.min(kw["y_int"])),
                      fix_costs=ora["fix"], form="diff", precise_int=True)
    ext = SetProblem.with_external_prior(kw["grid"], kw["x_int"], kw["y_int"], res["mI"], res["vI"], res["mg"], res["vg"],
                                         cost_fix=2.0)
    best = float(np.min(kw["y_int"]))
    from cbo_with_oop_b200.engine import SweepEngine
    eng = SweepEngine([SetProblem(**kw), ext], device="cuda:0")
    grid = eng.sweep(best, "min")
    out = eng.refine(grid, best, "min")
    assert out.refine_status[1] == "skipped_external_prior"
    assert out.set_values[1].tobytes() == grid.set_values[1].tobytes()
    np.testing.assert_array_equal(out.set_x[1], eng_grid_x(eng.problems[1], grid.set_indices[1]))
    # no iteration: nothing improves, the grid result stays bit for bit
    none = eng.refine(grid, best, "min", max_iter=0)
    for g in range(2):
        assert none.set_values[g].tobytes() == grid.set_values[g].tobytes()
        assert none.set_x[g].tobytes() == eng_grid_x(eng.problems[g], grid.set_indices[g]).tobytes()
    assert none.set == grid.set and none.index == grid.index and none.value == grid.value
    # explicit points: the set is skipped before anything else of it is read
    import torch
    h = (_lib.SetDesc * 1).from_buffer_copy(bytes(eng.h_sets)[:C.sizeof(_lib.SetDesc)])
    dummy = torch.zeros(8, dtype=torch.float64, device="cuda:0")
    h[0].points = dummy.data_ptr()
    h[0].p[0], h[0].p[1] = h[0].g_total, 1
    d_h = torch.frombuffer(bytearray(bytes(h)), dtype=torch.uint8).to("cuda:0")
    x0 = torch.tensor([0.5, -0.25, 0.0, 0.0], dtype=torch.float64, device="cuda:0")
    ws = torch.empty((eng.lib.cbo_refine_workspace_bytes(h, 1),), dtype=torch.uint8, device="cuda:0")
    r = torch.empty((C.sizeof(_lib.RefineResult),), dtype=torch.uint8, device="cuda:0")
    _lib.check(eng.lib.cbo_refine(h, C.c_void_p(d_h.data_ptr()), 1, best, 1, C.c_void_p(x0.data_ptr()), 10, 1e-7,
                                  C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(r.data_ptr()), eng._stream()), "cbo_refine")
    rr = _lib.RefineResult.from_buffer_copy(r.cpu().numpy().tobytes())
    assert rr.status == 4 and list(rr.x)[:2] == [0.5, -0.25] and rr.iterations == 0 and np.isnan(rr.value)


def test_simplified_coral_all_sets(cuda_engine_ready):
    from cbo_with_oop_b200.engine import SweepEngine
    from cbo_with_oop_b200.fixtures import golden_path, load_golden_problems
    if not os.path.exists(golden_path("simplified_coral")):
        pytest.fail("golden fixture missing")
    problems, best, task = load_golden_problems("simplified_coral", device_fit=False)
    eng = SweepEngine(problems, device="cuda:0")
    grid = eng.sweep(best, task)
    out = eng.refine(grid, best, task)
    scale = float(np.nanmax(np.abs(grid.set_values)))
    for g, pr in enumerate(problems):
        assert out.set_values[g] >= grid.set_values[g], g
        X = np.hstack([pr.x_obs_int, pr.x_obs_cond])
        gp = dict(X=X, variance=pr.s2, lengthscale=np.concatenate([pr.ls_int, pr.ls_cond]), noise=pr.noise, alpha=pr.alpha_obs,
                  Kyinv=pr.kyinv, form="diff")
        cols = list(range(pr.d))
        f = O.prior_factors(gp, X, cols)
        mI, vI = O.do_prior_factorised(gp, f, cols, pr.x_int, precise=True)
        post = O.posterior_fit(pr.x_int, pr.y_int, mI, vI, form="diff")
        ref = R.refine_set(post, eng_grid_x(pr, grid.set_indices[g]), pr.grid, best, task, fix_costs=np.array([pr.cost_fix]),
                           gp=gp, factors=f, intervened_cols=cols)
        assert abs(ref["value"] - out.set_values[g]) <= 1e-6 * max(abs(ref["value"]), 1e-6 * scale), \
            (g, ref["value"], out.set_values[g], out.refine_status[g])


@pytest.fixture
def in_tmp(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)


@pytest.mark.parametrize("experiment", ["toy_graph", "complete_graph"])
def test_agent_with_refinement(cuda_engine_ready, in_tmp, experiment):
    from src.CBO import CBO
    from src.DataLoader import DataLoader
    args = types.SimpleNamespace(exploration_set="MIS", initial_num_obs_samples=60, num_interventions=10, type_cost=1,
                                 num_additional_observations=20, num_trials=6, name_index=0, seed=9, causal_prior=True,
                                 experiment=experiment, task="min", grid_points=40, device="cuda:0", num_sem_samples=2000,
                                 refine_acquisition=True)
    np.random.seed(args.seed)
    cbo = CBO(args, DataLoader(experiment, 60), verbose=False)
    cbo.run()
    ranges = cbo.graph.get_interventional_ranges()
    off_grid = 0
    for s, variables in enumerate(cbo.exploration_set):
        tables = cbo.monitor.space_list[s].grid_tables(args.grid_points)
        for x in np.asarray(cbo.monitor.data_x[s])[args.num_interventions:]:
            for k, v in enumerate(variables):
                assert ranges[v][0] <= x[k] <= ranges[v][1], (v, x)
            off_grid += int(any(not np.any(tables[k] == x[k]) for k in range(len(variables))))
    assert int(np.sum(cbo.monitor.type_trial)) >= 1
    assert off_grid >= 1
