"""CPU checks of oracle/hyper_oracle.py, the checker of the hyper-parameter fit (K8) and of the kernels that read
`cbo_set_desc.hyper`: at (1, 1) it is the existing oracle bit for bit, its NLL gradient and acquisition x-gradients agree
with central differences at fitted-looking (s2, l), and the bounds and start lattice are what K8 is documented to use."""
import os

import numpy as np
import pytest

from helpers import make_case
from oracle import cbo_oracle as O
from oracle import hyper_oracle as H
from oracle import refine_oracle as R


def causal_state(seed, n=12, d=2, causal=True):
    kw, ora = make_case(seed=seed, N=80, d=d, c=1, n=n, p=(15,) * d, causal=causal)
    if not causal:
        return ora, None, None, None
    f = O.prior_factors(ora["gp"], ora["cond"], ora["cols"])
    mI, vI = O.do_prior_factorised(ora["gp"], f, ora["cols"], ora["XI"], precise=True)
    return ora, f, mI, vI


@pytest.mark.parametrize("causal", [True, False])
def test_unit_hyperparameters_equal_the_existing_oracle_bit_for_bit(causal):
    ora, f, mI, vI = causal_state(501, causal=causal)
    Xg = O.tensor_grid(ora["tables"])
    a = O.posterior_fit(ora["XI"], ora["yI"], mI, vI, form="diff")
    b = H.posterior_fit(ora["XI"], ora["yI"], mI, vI, 1.0, 1.0)
    assert a["L"].tobytes() == b["L"].tobytes() and a["alpha"].tobytes() == b["alpha"].tobytes() and a["tries"] == b["tries"]
    mg, vg = O.do_prior_factorised(ora["gp"], f, ora["cols"], Xg) if causal else (None, None)
    mu_a, var_a = O.posterior_predict(a, Xg, mg, vg)
    mu_b, var_b = H.posterior_predict(b, Xg, mg, vg)
    assert mu_a.tobytes() == mu_b.tobytes() and var_a.tobytes() == var_b.tobytes()
    kw = dict(gp=ora["gp"], factors=f, intervened_cols=ora["cols"]) if causal else {}
    X = np.random.default_rng(1).uniform(-2, 2, (6, 2))
    best = float(np.min(ora["yI"]))
    ra = R.acquisition_gradients(a, X, best, "min", **kw)
    rb = H.acquisition_gradients(b, X, best, "min", **kw)
    for k in ra:
        assert ra[k].tobytes() == rb[k].tobytes(), k


@pytest.mark.parametrize("causal", [True, False])
@pytest.mark.parametrize("s2,l", [(1.0, 1.0), (37.0, 0.35), (0.3, 1.8)])
def test_nll_gradient_matches_central_differences(causal, s2, l):
    ora, f, mI, vI = causal_state(502, n=15, causal=causal)
    resid = ora["yI"] - mI if causal else ora["yI"]
    f0, g, tries = H.nll(ora["XI"], resid, s2, l, vI)
    assert np.isfinite(f0) and tries == 0
    h = 2e-6
    for k in range(2):
        th = np.log([s2, l])
        tp, tm = th.copy(), th.copy()
        tp[k] += h
        tm[k] -= h
        fp = H.nll(ora["XI"], resid, *np.exp(tp), vI, grad=False)[0]
        fm = H.nll(ora["XI"], resid, *np.exp(tm), vI, grad=False)[0]
        fd = (fp - fm) / (2 * h)
        assert abs(fd - g[k]) <= 1e-5 * max(1.0, abs(g[k])), (k, fd, g[k])


@pytest.mark.parametrize("causal", [True, False])
def test_acquisition_x_gradients_match_central_differences(causal):
    ora, f, mI, vI = causal_state(503, n=10, causal=causal)
    post = H.posterior_fit(ora["XI"], ora["yI"], mI, vI, 5.0, 0.6)
    kw = dict(gp=ora["gp"], factors=f, intervened_cols=ora["cols"]) if causal else {}
    best = float(np.min(ora["yI"]))
    X = np.random.default_rng(2).uniform(-1.5, 1.5, (4, 2))
    r = H.acquisition_gradients(post, X, best, "min", **kw)
    h = 1e-6
    for a in range(X.shape[0]):
        for k in range(2):
            xp, xm = X[a].copy(), X[a].copy()
            xp[k] += h
            xm[k] -= h
            rp = H.acquisition_gradients(post, xp[None], best, "min", **kw)
            rm = H.acquisition_gradients(post, xm[None], best, "min", **kw)
            for name in ("mu", "var", "ei", "acq"):
                fd = (rp[name][0] - rm[name][0]) / (2 * h)
                an = r["d" + name][a, k]
                assert abs(fd - an) <= 1e-5 * max(1e-3, abs(an), np.abs(r["d" + name]).max()), (name, a, k, fd, an)


def test_bounds_follow_the_grid():
    from cbo_with_oop_b200.engine import hyper_bounds
    b = hyper_bounds([np.linspace(-5.0, 5.0, 101), np.linspace(0.0, 2.0, 5)])
    assert b[0] == 1e-6 and b[1] == 1e6
    assert b[2] == pytest.approx(0.1) and b[3] == pytest.approx(100.0)
    assert list(hyper_bounds([np.zeros(1)])) == [1e-6, 1e6, 1.0, 1.0]
    from cbo_with_oop_b200.fixtures import golden_path
    for cfg in ("toy", "complete", "simplified_coral", "coral_synth"):
        if not os.path.exists(golden_path(cfg)):
            pytest.fail("golden fixture missing")
        z = np.load(golden_path(cfg))
        for s in range(int(z["num_sets"])):
            grid = [np.linspace(lo, hi, int(p)) for lo, hi, p in z[f"set{s}_grid_lo_hi_p"]]
            b = hyper_bounds(grid)
            assert np.all(np.isfinite(b)) and np.all(b > 0) and b[0] <= b[1] and b[2] <= b[3]
            assert b[2] == min((t[-1] - t[0]) / (len(t) - 1) for t in grid)


def test_start_lattice():
    bounds = np.array([1e-6, 1e6, 0.1, 100.0])
    rng = np.random.default_rng(3)
    r = rng.standard_normal(12) * 3.0
    st = H.starts(bounds, r)
    assert len(st) == H.NUM_STARTS == 9
    assert np.all(st[0] == 0.0)                                  # (1, 1): the reference's model
    lo, hi = H.log_box(bounds)
    assert all(np.all(t >= lo) and np.all(t <= hi) for t in st)
    assert len({tuple(t) for t in st}) == 9
    ls = sorted({t[1] for t in st[1:]})
    assert np.allclose(np.diff(ls), (hi[1] - lo[1]) / 4) and ls[0] == pytest.approx(lo[1] + (hi[1] - lo[1]) / 8)
    assert np.allclose(sorted({t[0] for t in st[1:]}), np.log(r.var()) + np.array([0.0, np.log(10.0)]))
    # a box that excludes (1, 1) clips start 0 onto it; a constant residual starts s2 at the lower bound
    st = H.starts(np.array([2.0, 3.0, 1.5, 4.0]), np.ones(5))
    assert np.allclose(st[0], np.log([2.0, 1.5])) and all(np.isclose(t[0], np.log(2.0)) for t in st[1:5])
