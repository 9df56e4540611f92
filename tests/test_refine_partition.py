"""CPU tests of the multi-GPU refinement's host logic: which rank refines each exploration set (partition.refine_owners) and,
with two gloo processes, the all-gather of the cbo_refine_result tables followed on every rank by the same assembly
(engine.refined_output)."""
import ctypes as C
import os
import pickle
import socket

import numpy as np
import pytest

from cbo_with_oop_b200.partition import SetSize, partition, refine_owners


def random_sizes(rng):
    S = int(rng.integers(1, 12))
    return [SetSize(int(rng.choice([1, 7, 128, 129, 1000, 20_000, 10 ** 6])), int(rng.choice([0, 50, 1000, 10_000])),
                    int(rng.integers(1, 129))) for _ in range(S)]


@pytest.mark.parametrize("seed", range(40))
def test_refine_owner_is_the_lowest_rank_holding_the_set(seed):
    rng = np.random.default_rng(seed)
    sizes = random_sizes(rng)
    for world in range(1, 9):
        sl = partition(sizes, world, tile=int(rng.choice([1, 128])))
        owners = refine_owners(sl)
        assert len(owners) == len(sizes)
        for s in range(len(sizes)):
            holders = [r for r in range(world) if sl[r][s][1] > 0]
            assert holders, (s, world)                               # every set with candidates has a slice somewhere
            assert owners[s] == holders[0]                           # exactly one owner: the lowest rank that holds the set
            assert sl[owners[s]][s][1] > 0
        if world == 1:
            assert owners == [0] * len(sizes)


def test_refine_owner_worked_examples():
    big = SetSize(10 ** 6, 10 ** 4, 32)
    assert refine_owners(partition([big] * 3, 8)) == [0, 2, 5]
    assert refine_owners(partition([big] * 3, 4)) == [0, 1, 2]
    assert refine_owners(partition([big] * 16, 8)) == [r for r in range(8) for _ in range(2)]
    # a set no rank holds has no owner
    assert refine_owners([[(0, 10), (0, 0)], [(10, 5), (0, 0)]]) == [0, -1]


# ---- two gloo ranks ------------------------------------------------------------------------------------------------------
S_GLOO = 6


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _problems():
    from cbo_with_oop_b200.engine import SetProblem
    rng = np.random.default_rng(5)
    out = []
    for s, p in enumerate([(1000,), (30, 30), (12, 12, 12), (4000,), (50, 50), (10, 10, 10)]):   # on 2 ranks set 3 is split
        grid = [np.linspace(-1.0 - s, 1.0 + s, n) for n in p]
        out.append(SetProblem.non_causal(grid, rng.uniform(-1, 1, (4, len(p))), rng.normal(size=4), name=f"set{s}"))
    return out


def _sweep_output(problems):
    """A grid result as the sweep leaves it: global indices; set 4 has no finite maximum, sets 1 and 3 share the largest
    grid value (the refinement decides which set is selected)."""
    from cbo_with_oop_b200.engine import SweepOutput
    vals = np.array([0.3, 0.9, 0.1, 0.9, np.nan, 0.2])
    idx = np.array([p.g_total // 3 for p in problems], dtype=np.int64)
    return SweepOutput(1, int(idx[1]), 0.9, None, vals, idx, 2)


def _records(problems, world):
    """What each rank's K7 call would leave in its global-indexed table: the owner of a set writes its refined record, any
    other rank holding the set writes the record of a set started at a NaN row (skipped), and the rest stays zero."""
    from cbo_with_oop_b200._lib import RefineResult
    sizes = [SetSize(p.g_total, 0, p.x_int.shape[0]) for p in problems]
    sl = partition(sizes, world, tile=1)
    owners = refine_owners(sl)
    out = _sweep_output(problems)
    tables = [(RefineResult * len(problems))() for _ in range(world)]
    for s, p in enumerate(problems):
        for r in range(world):
            if not sl[r][s][1]:
                continue
            rec = tables[r][s]
            if r == owners[s] and np.isfinite(out.set_values[s]):
                x = [float(np.mean(t)) + 0.01 * (s + 1) for t in p.grid]
                gain = {1: 0.05, 2: 0.0, 3: 0.2}.get(s, 0.01)                # set 2: no step improved
                rec.value, rec.start_value = out.set_values[s] + gain, out.set_values[s]
                rec.iterations, rec.status = 3 + s, 0 if s % 2 else 1
            else:
                x = [np.nan] * p.d
                rec.value = rec.start_value = np.nan
                rec.iterations, rec.status = 0, 5
            for k in range(p.d):
                rec.x[k] = x[k]
    return sl, owners, out, tables


def _worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist
    from cbo_with_oop_b200.dist import gather_set_bests
    from cbo_with_oop_b200.engine import refined_output
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    problems = _problems()
    _, owners, out, tables = _records(problems, world)
    local = torch.frombuffer(bytearray(bytes(tables[rank])), dtype=torch.uint8)
    gathered = torch.empty(world * local.numel(), dtype=torch.uint8)
    gather_set_bests(local, gathered, world)
    res = refined_output(out, problems, owners, gathered.numpy().tobytes())
    with open(os.path.join(out_dir, f"refined_{rank}.pkl"), "wb") as f:
        pickle.dump((gathered.numpy(), res), f)
    dist.destroy_process_group()


def test_refined_records_all_gathered_with_two_gloo_ranks(tmp_path):
    import torch.multiprocessing as mp
    from cbo_with_oop_b200._lib import REFINE_STATUS, RefineResult
    from cbo_with_oop_b200.engine import grid_point
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    (g0, r0), (g1, r1) = [pickle.load(open(tmp_path / f"refined_{r}.pkl", "rb")) for r in range(world)]
    assert C.sizeof(RefineResult) == 56 and g0.size == world * S_GLOO * 56
    np.testing.assert_array_equal(g0, g1)
    problems = _problems()
    sl, owners, out, tables = _records(problems, world)
    for r in range(world):                                                  # rank-major layout
        assert g0.reshape(world, -1)[r].tobytes() == bytes(tables[r])
    assert any(all(sl[r][s][1] for r in range(world)) for s in range(S_GLOO)), "no set is split between the ranks"
    assert sorted(set(owners)) == [0, 1]
    # both ranks assemble the same output, bit for bit
    for name in ("set", "index", "value", "n_nan", "refine_status"):
        assert getattr(r0, name) == getattr(r1, name), name
    assert r0.set_values.tobytes() == r1.set_values.tobytes() and r0.x.tobytes() == r1.x.tobytes()
    assert all((a is None and b is None) or a.tobytes() == b.tobytes() for a, b in zip(r0.set_x, r1.set_x))
    # each set's record is its owner's
    for s, p in enumerate(problems):
        rec = tables[owners[s]][s]
        assert r0.refine_status[s] == REFINE_STATUS[rec.status]
        if rec.value > rec.start_value:
            assert r0.set_values[s] == rec.value and list(r0.set_x[s]) == list(rec.x)[:p.d]
        else:
            assert r0.set_values[s].tobytes() == np.float64(out.set_values[s]).tobytes()
            np.testing.assert_array_equal(r0.set_x[s], grid_point(p, out.set_indices[s]))
    # selection: first maximum of the refined values, NaN = -inf; the grid tie of sets 1 and 3 is broken by set 3's gain
    assert r0.set == 3 and r0.value == r0.set_values[3] and r0.index == out.set_indices[3]
    assert r0.x.tobytes() == r0.set_x[3].tobytes()
