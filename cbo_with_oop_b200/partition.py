"""Multi-GPU partition of a sweep: the flattened (exploration set x grid tile) list is cut into contiguous,
FLOP-weighted chunks, one per rank (SURVEY.md §8e).  Pure Python / integers: every rank computes the same
cuts from the same sizes, no communication.  Candidates are independent given the per-set state, so the
only exchange of a sweep is the all-gather of each rank's per-set best (dist.py)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence, Tuple


@dataclass(frozen=True)
class SetSize:
    g_total: int      # candidates of the set
    n_obs: int        # N (0 for a non-causal set)
    n_int: int        # n

    @property
    def weight(self) -> int:
        """Executed FP64 multiply-adds per candidate: N^2/2-ish prior quadratic form + n^2/2 forward
        substitution + n kernel evaluations (integer proxy, only ratios matter)."""
        return self.n_obs * self.n_obs // 2 + self.n_int * self.n_int // 2 + 32 * self.n_int + 64


def _cuts(sizes: Sequence[SetSize], world: int, tile: int, snap: float) -> List[Tuple[int, int]]:
    """world+1 cut points (set, first candidate), in units the ranks agree on."""
    weights = [s.g_total * s.weight for s in sizes]
    total = sum(weights)
    cuts: List[Tuple[int, int]] = [(0, 0)]
    for r in range(1, world):
        target = total * r // world
        s, cum = 0, 0
        while s < len(sizes) - 1 and cum + weights[s] <= target:
            cum += weights[s]
            s += 1
        w = sizes[s].weight
        pt = (target - cum + w // 2) // w          # nearest candidate
        pt = (pt + tile // 2) // tile * tile       # nearest tile boundary
        pt = max(0, min(pt, sizes[s].g_total))
        # prefer whole sets: a split set costs both ranks its one-off prior precompute and its M matrix
        share = total / world
        if pt * w <= snap * share:
            pt = 0
        elif (sizes[s].g_total - pt) * w <= snap * share:
            pt = sizes[s].g_total
        if pt == sizes[s].g_total and s < len(sizes) - 1:
            s, pt = s + 1, 0
        if (s, pt) < cuts[-1]:
            s, pt = cuts[-1]
        cuts.append((s, pt))
    cuts.append((len(sizes), 0))
    return cuts


def partition(sizes: Sequence[SetSize], world: int, tile: int = 128, snap: float = 0.05) -> List[List[Tuple[int, int]]]:
    """Returns slices[rank][set] = (g_begin, g_count).  The slices of one set over all ranks tile
    [0, g_total) exactly once and in rank order."""
    if world < 1:
        raise ValueError("world must be >= 1")
    cuts = _cuts(sizes, world, tile, snap)
    out: List[List[Tuple[int, int]]] = []
    for r in range(world):
        (s0, p0), (s1, p1) = cuts[r], cuts[r + 1]
        sl = []
        for s, sz in enumerate(sizes):
            if s < s0 or s > s1 or (s == s1 and p1 == 0):
                sl.append((0, 0))
                continue
            b = p0 if s == s0 else 0
            e = p1 if s == s1 else sz.g_total
            sl.append((b, max(0, e - b)) if e > b else (0, 0))
        out.append(sl)
    return out


def refine_owners(slices: Sequence[Sequence[Tuple[int, int]]]) -> List[int]:
    """The rank that refines each set off the grid (SweepEngine.refine): the lowest rank whose slice of the set is
    non-empty, or -1 when no rank holds any of it.  Every rank that touches a set holds the set's whole state, so any of
    them could; a pure function of the partition lets every rank agree without communicating."""
    num_sets = len(slices[0]) if slices else 0
    owners = [-1] * num_sets
    for r in reversed(range(len(slices))):
        for s, (_, count) in enumerate(slices[r]):
            if count > 0:
                owners[s] = r
    return owners
