"""SweepEngine.refine on multi-rank engines, every rank in one process on one GPU: the all-gathers of the sweep and of the
refinement are replaced by stacking the ranks' tables rank-major, and every rank's refined output must equal, bit for bit,
what a single-GPU engine's refine returns on the same problems (set, index, value, x, set_values, set_x, refine_status).
tools/multi_gpu_refine_check.py runs the same comparison over NCCL with one GPU per rank."""
import copy

import numpy as np
import pytest

from helpers import make_case
from oracle import cbo_oracle as O

pytestmark = pytest.mark.gpu

MIXED = [dict(seed=701, N=120, d=1, c=1, n=8, p=(1500,)), dict(seed=702, N=200, d=2, c=2, n=10, p=(30, 30)),
         dict(seed=703, N=150, d=3, c=1, n=12, p=(10, 10, 10), cost_variable=True),
         dict(seed=704, N=90, d=4, c=1, n=9, p=(6, 6, 6, 6)),
         dict(seed=705, N=60, d=2, c=1, n=10, p=(40, 25), causal=False, cost_variable=True),
         dict(seed=707, N=100, d=2, c=0, n=7, p=(20, 20))]


def mixed_problems():
    from cbo_with_oop_b200.engine import SetProblem
    return [SetProblem(**make_case(**s)[0]) for s in MIXED]


def engines(problems, world, **kw):
    """A world-1 engine and the `world` ranks of a partitioned one, each with its own copy of the problems (set_interventional
    changes the caller's SetProblem in place)."""
    from cbo_with_oop_b200.engine import SweepEngine
    whole = SweepEngine(copy.deepcopy(problems), device="cuda:0", **kw)
    ranks = [SweepEngine(copy.deepcopy(problems), device="cuda:0", rank=r, world_size=world, **kw) for r in range(world)]
    return whole, ranks


def _stack(ranks, run):
    """Runs run(e) on every rank, each ending in one all-gather, and stacks the tables each rank would send."""
    import torch
    tables = [None] * len(ranks)
    for r, e in enumerate(ranks):
        def record(table, gathered, r=r):
            tables[r] = table.clone()
            gathered.view(len(ranks), -1).copy_(table.view(1, -1).expand(len(ranks), -1))
        e._all_gather = record
        try:
            run(e)
        finally:
            del e._all_gather
    return torch.cat(tables)


def _replayed(e, stacked, run):
    """run(e) with its all-gather filled from the stacked tables of every rank."""
    e._all_gather = lambda table, gathered: gathered.copy_(stacked)
    try:
        return run(e)
    finally:
        del e._all_gather


def sweep_ranks(ranks, run):
    """Every rank's SweepOutput of a sweep() or refresh() as NCCL would leave it."""
    stacked = _stack(ranks, run)
    return [_replayed(e, stacked, lambda e: e._finish([])) for e in ranks]


def refine_ranks(ranks, grids, best, task, **kw):
    """Every rank's refine(): the local steps' tables stacked rank-major, then each rank's refine() with that gather."""
    import torch
    max_iter, gtol = kw.get("max_iter", 30), kw.get("gtol", 1e-7)
    stacked = torch.cat([e._refine_local(g, best, task, max_iter, gtol, []) for e, g in zip(ranks, grids)])
    outs = []
    for e, g in zip(ranks, grids):
        e.timing = True
        outs.append(_replayed(e, stacked, lambda e: e.refine(g, best, task, **kw)))
        e.timing = False
        if e.active:
            assert {"refine", "refine_gather"} <= set(outs[-1].stage_ms)
    return outs


def same_grid(a, b):
    assert (a.set, a.index, a.n_nan) == (b.set, b.index, b.n_nan)
    assert np.float64(a.value).tobytes() == np.float64(b.value).tobytes()
    assert a.set_values.tobytes() == b.set_values.tobytes() and list(a.set_indices) == list(b.set_indices)


def same_refined(a, b):
    same_grid(a, b)
    assert (a.x is None) == (b.x is None) and (a.x is None or a.x.tobytes() == b.x.tobytes())
    assert a.refine_status == b.refine_status
    for g, (u, v) in enumerate(zip(a.set_x, b.set_x)):
        assert (u is None) == (v is None) and (u is None or u.tobytes() == v.tobytes()), g


def split_sets(ranks):
    return [g for g in range(len(ranks[0].problems)) if sum(g in e.local_of for e in ranks) > 1]


def argmax_off_owner(ranks, grid):
    """Split sets whose grid argmax lies outside their owner rank's slice."""
    out = []
    for g in split_sets(ranks):
        b, c = ranks[ranks[0].refine_owner[g]].slices[g]
        if not b <= grid.set_indices[g] < b + c:
            out.append(g)
    return out


def check(problems, world, best, task="min", **kw):
    """Sweep and refine on a world-1 engine and on `world` ranks; returns (ranks, world-1 grid output, refined output)."""
    whole, ranks = engines(problems, world, **kw)
    grid = whole.sweep(best, task)
    ref = whole.refine(grid, best, task)
    grids = sweep_ranks(ranks, lambda e: e.sweep(best, task))
    for g in grids:
        same_grid(g, grid)
    for out in refine_ranks(ranks, grids, best, task):
        same_refined(out, ref)
    assert ref.refine_status.count("converged") + ref.refine_status.count("max_iter") >= 1
    return whole, ranks, grid, ref


@pytest.mark.parametrize("world", [2, 3])
def test_mixed_sets_match_one_gpu(cuda_engine_ready, world):
    problems = mixed_problems()
    best = float(min(np.min(p.y_int) for p in problems))
    _, ranks, grid, ref = check(problems, world, best)
    assert split_sets(ranks), "no set is split between the ranks"
    assert any(ref.set_values[g] > grid.set_values[g] for g in split_sets(ranks))


def test_split_set_argmax_in_a_later_slice(cuda_engine_ready):
    problems = mixed_problems()
    best = float(min(np.min(p.y_int) for p in problems))
    reached = []
    for world in (2, 3):
        _, ranks, grid, _ = check(problems, world, best)
        reached += argmax_off_owner(ranks, grid)
    assert reached, "no split set has its grid argmax outside its owner's slice"


def test_rank_without_sets(cuda_engine_ready):
    from cbo_with_oop_b200.engine import SetProblem
    problems = [SetProblem(**make_case(seed=121, N=70, d=1, c=1, n=5, p=(100,))[0]),
                SetProblem(**make_case(seed=122, N=90, d=2, c=1, n=6, p=(13, 10))[0])]
    best = float(min(np.min(p.y_int) for p in problems))
    _, ranks, _, _ = check(problems, 3, best)
    assert any(not e.active for e in ranks)


def test_external_prior_set(cuda_engine_ready):
    from cbo_with_oop_b200.engine import SetProblem
    kw, ora = make_case(seed=431, N=150, d=2, c=1, n=9, p=(15, 15))
    res = O.sweep_set(ora["gp"], ora["cond"], ora["cols"], ora["XI"], ora["yI"], ora["tables"], float(np.min(kw["y_int"])),
                      fix_costs=ora["fix"], form="diff", precise_int=True)
    ext = SetProblem.with_external_prior([np.linspace(-2.0, 2.0, 60), np.linspace(-2.0, 2.0, 60)], kw["x_int"], kw["y_int"],
                                         res["mI"], res["vI"], np.tile(res["mg"].reshape(15, 15), (4, 4)).reshape(-1),
                                         np.tile(res["vg"].reshape(15, 15), (4, 4)).reshape(-1), cost_fix=2.0)
    problems = [SetProblem(**kw), ext, SetProblem(**make_case(seed=432, N=80, d=1, c=1, n=7, p=(500,))[0])]
    best = float(np.min(kw["y_int"]))
    _, ranks, _, ref = check(problems, 2, best)
    assert ref.refine_status[1] == "skipped_external_prior"
    assert split_sets(ranks)


def test_fitted_hyperparameters(cuda_engine_ready):
    problems = mixed_problems()
    best = float(min(np.min(p.y_int) for p in problems))
    whole, ranks, _, _ = check(problems, 2, best, fit_hyperparameters=True)
    for g in split_sets(ranks):
        assert all(e.hyperparameters(g) == whole.hyperparameters(g) for e in ranks if g in e.local_of)


def test_refine_after_refresh_with_an_appended_row(cuda_engine_ready):
    problems = mixed_problems()
    best = float(min(np.min(p.y_int) for p in problems))
    whole, ranks, _, _ = check(problems, 2, best)
    g = split_sets(ranks)[0]
    pr = whole.problems[g]
    x_new = np.vstack([pr.x_int, [[float(t[len(t) // 3]) for t in pr.grid]]])
    y_new = np.append(pr.y_int, float(np.mean(pr.y_int)))
    best = min(best, float(y_new[-1]))
    for e in [whole] + ranks:
        e.set_interventional(g, x_new, y_new)
    grid = whole.refresh(best, "min", refit=[g])
    ref = whole.refine(grid, best, "min")
    grids = sweep_ranks(ranks, lambda e: e.refresh(best, "min", refit=[g]))
    for out in grids:
        same_grid(out, grid)
    for out in refine_ranks(ranks, grids, best, "min"):
        same_refined(out, ref)


def test_max_task(cuda_engine_ready):
    problems = mixed_problems()
    best = float(max(np.max(p.y_int) for p in problems))
    check(problems, 3, best, task="max")
