"""The table stage (K0) and the prior precompute (K1a) give every set the same bits whichever sets share the call: a set
alone, all sets in one launch per stage, and sets whose descriptors share one P scratch buffer (then they run one after
the other).  The explicit-point table and the appended-row table of a post-intervention trial go through the same kernel
and must agree with it bit for bit."""
import numpy as np
import pytest

from helpers import make_case

pytestmark = pytest.mark.gpu

SPECS = [dict(seed=401, N=150, d=2, c=2, n=9, p=(12, 10)),
         dict(seed=402, N=260, d=3, c=1, n=7, p=(6, 5, 4)),        # three 128-row blocks
         dict(seed=403, N=90, d=2, c=0, n=6, p=(8, 7)),             # no conditioning columns: M = s2^2 Ky^-1
         dict(seed=404, N=100, d=1, c=3, n=5, p=(40,), S_mc=33)]    # S_mc != N, ragged 16-column padding
N_COND = sum(1 for s in SPECS if s["c"] > 0)


def _arrays(eng, g):
    names = [f"tab{k}" for k in range(eng.problems[g].d)] + ["u_int", "pbar", "w", "M"]
    return {n: eng.fetch(n, g) for n in names}


def _points(s):
    return np.random.default_rng(s["seed"]).uniform(-2.5, 2.5, (300, s["d"]))


def _assert_same(eng, alone):
    for g, s in enumerate(SPECS):
        ref_arrays, ref_prior = alone[g]
        for n, a in _arrays(eng, g).items():
            assert np.array_equal(a, ref_arrays[n]), f"set {g}: {n} differs from the set computed alone"
        prior = eng.evaluate_points(g, _points(s), stages="prior")
        for n in ("m", "v"):
            assert np.array_equal(prior[n], ref_prior[n]), f"set {g}: explicit-point {n} differs"


def test_stage_arrays_do_not_depend_on_which_sets_share_the_call(cuda_engine_ready):
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    cases = [make_case(**s) for s in SPECS]
    alone = []
    for g, (kw, _) in enumerate(cases):
        eng = SweepEngine([SetProblem(**kw)])
        eng.build_tables()
        eng.prior_precompute()
        alone.append((_arrays(eng, 0), eng.evaluate_points(0, _points(SPECS[g]), stages="prior")))
        del eng

    eng = SweepEngine([SetProblem(**kw) for kw, _ in cases])
    assert eng._private_P
    l0 = eng.launches
    eng.build_tables()
    eng.prior_precompute()
    # one table launch; one launch for the c = 0 set; pgen + syrk shared by the sets with conditioning columns
    assert eng.launches - l0 == 1 + 1 + 2
    _assert_same(eng, alone)

    # the same sets on one shared P buffer: each set with conditioning columns gets its own pgen + syrk, in set order
    for li, s in enumerate(SPECS):
        if s["c"] > 0:
            eng.h_sets[li].P = eng.P.data_ptr()
        for n in ("pbar", "w", "M"):
            eng.buf[li][n].fill_(float("nan"))
    eng._descs_dirty = True
    l0 = eng.launches
    eng.prior_precompute()
    assert eng.launches - l0 == 1 + 2 * N_COND
    _assert_same(eng, alone)


def test_appended_row_table_matches_a_fresh_build(cuda_engine_ready):
    """A post-intervention trial writes only the appended row of u_int; the whole table must equal a fresh build's."""
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    cases = [make_case(**s) for s in SPECS]
    best = float(min(np.min(kw["y_int"]) for kw, _ in cases))
    eng = SweepEngine([SetProblem(**kw) for kw, _ in cases])
    eng.sweep(best, "min")
    for g in (0, 2):
        kw = cases[g][0]
        x_new = np.vstack([kw["x_int"], np.full((1, SPECS[g]["d"]), 0.3)])
        y_new = np.append(kw["y_int"], best - 0.1)
        eng.set_interventional(g, x_new, y_new)
        eng.refresh(best - 0.1, "min", refit=[g])
        fresh = SweepEngine([SetProblem(**dict(kw, x_int=x_new, y_int=y_new))])
        fresh.build_tables()
        assert np.array_equal(eng.fetch("u_int", g), fresh.fetch("u_int", 0))
