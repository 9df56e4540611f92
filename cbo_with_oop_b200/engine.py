"""Host side of the B200 acquisition sweep: owns device memory (PyTorch tensors), builds the cbo_set_desc
array, and drives libcbo_b200.so through its C ABI.  PyTorch is plumbing here (allocation, streams, NCCL);
every number is produced by the hand-written kernels in csrc/.

One SweepEngine = one rank's share of one trial's sweep over every exploration set.
Stages (reference call sites in include/cbo_b200.h):
    build_tables -> prior_precompute -> prior_eval(x_int) -> posterior_fit -> prior_eval(grid) -> sweep
`sweep(best, task)` runs all of them (a post-observation trial); `refresh(best, task, refit=[...])` reuses the
cached prior and only refits the listed sets (a post-intervention trial).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import AcqGradOut, HyperResult, RefineResult, SetBest, SetDesc, SweepResult
from .dist import gather_set_bests
from .partition import SetSize, partition, refine_owners

HYPER_S2_BOUNDS = (1e-6, 1e6)


def hyper_bounds(grid: Sequence[np.ndarray]) -> np.ndarray:
    """(s2_lo, s2_hi, l_lo, l_hi) of the marginal-likelihood fit of one exploration set's GP (cbo_posterior_hyper_fit):
    s2 in [1e-6, 1e6]; l from the smallest grid spacing of the set (a shorter lengthscale only fits noise between
    candidates the sweep never evaluates: unbounded, the fit runs to white-noise spikes far below one spacing) to ten
    times the largest box span (beyond that the kernel is flat over the box).  A set whose box has no extent keeps l = 1."""
    spans = [float(np.max(t) - np.min(t)) for t in grid]
    steps = [sp / (len(t) - 1) for sp, t in zip(spans, grid) if len(t) > 1 and sp > 0.0]
    if not steps:
        return np.array([HYPER_S2_BOUNDS[0], HYPER_S2_BOUNDS[1], 1.0, 1.0])
    return np.array([HYPER_S2_BOUNDS[0], HYPER_S2_BOUNDS[1], min(steps), 10.0 * max(spans)])


@dataclass
class SetProblem:
    """Host description of one exploration set's share of a trial (all float64 NumPy, caller-owned)."""
    x_obs_int: np.ndarray            # (N, d) intervened columns of the observational GP's training design
    x_obs_cond: np.ndarray           # (N, c) conditioning columns (c may be 0)
    mc_cond: np.ndarray              # (S_mc, c) conditioning samples (reference: the same observational rows)
    alpha_obs: Optional[np.ndarray]  # (N,)  Ky^-1 y of the observational GP   } both None + y_obs given: computed on the
    kyinv: Optional[np.ndarray]      # (N, N) Ky^-1                             } device by cbo_obs_gp_fit (K5)
    ls_int: np.ndarray               # (d,) lengthscales of the intervened columns
    ls_cond: np.ndarray              # (c,)
    s2: float                        # RBF variance
    grid: List[np.ndarray]           # d coordinate tables (np.linspace from the host)
    x_int: np.ndarray                # (n, d) interventional inputs
    y_int: np.ndarray                # (n,)   interventional outputs
    noise: float = 1e-2              # utils.py:43
    cost_fix: float = 1.0
    cost_variable: bool = False
    causal: bool = True
    name: str = ""
    # Caller-supplied causal prior (e.g. produced by DoCalculus closures): m_int, v_int on x_int and, for a grid sweep,
    # m_grid / v_grid over the whole tensor grid.  When set, the observational-GP fields above are ignored.
    y_obs: Optional[np.ndarray] = None   # (N,) training targets of the observational GP (only needed for the device fit)
    prior_external: bool = False
    m_int: Optional[np.ndarray] = None
    v_int: Optional[np.ndarray] = None
    m_grid: Optional[np.ndarray] = None
    v_grid: Optional[np.ndarray] = None

    @property
    def d(self) -> int:
        return len(self.grid)

    @property
    def computes_prior(self) -> bool:
        return self.causal and not self.prior_external

    @property
    def device_fit(self) -> bool:
        """alpha_obs / kyinv are produced on the device from (x_obs, y_obs) instead of being supplied."""
        return self.computes_prior and self.kyinv is None

    @staticmethod
    def with_external_prior(grid, x_int, y_int, m_int, v_int, m_grid=None, v_grid=None, cost_fix=1.0, cost_variable=False,
                            name=""):
        d = len(grid)
        return SetProblem(np.zeros((0, d)), np.zeros((0, 0)), np.zeros((0, 0)), np.zeros(0), np.zeros((0, 0)), np.ones(d),
                          np.zeros(0), 1.0, list(grid), x_int, y_int, cost_fix=cost_fix, cost_variable=cost_variable,
                          causal=True, name=name, prior_external=True, m_int=m_int, v_int=v_int, m_grid=m_grid, v_grid=v_grid)

    @property
    def g_total(self) -> int:
        g = 1
        for t in self.grid:
            g *= len(t)
        return g

    @staticmethod
    def non_causal(grid, x_int, y_int, cost_fix=1.0, cost_variable=False, name=""):
        d = len(grid)
        z = np.zeros((0, d))
        return SetProblem(z, np.zeros((0, 0)), np.zeros((0, 0)), np.zeros(0), np.zeros((0, 0)), np.ones(d), np.zeros(0),
                          1.0, list(grid), x_int, y_int, cost_fix=cost_fix, cost_variable=cost_variable, causal=False,
                          name=name)


@dataclass
class SweepOutput:
    set: int                 # global exploration-set index of the next intervention (-1: nothing evaluated)
    index: int               # flat grid index inside that set
    value: float             # acquisition value there
    x: Optional[np.ndarray]  # (d,) coordinates
    set_values: np.ndarray   # (S,) best acquisition per set (the reference's `ys`)
    set_indices: np.ndarray  # (S,) flat index of each set's best candidate
    n_nan: int
    stage_ms: Dict[str, float] = field(default_factory=dict)
    # filled by SweepEngine.refine: per-set coordinates of set_values ((d_s,) each; None for a set without a maximum) and
    # the per-set outcome of the refinement (_lib.REFINE_STATUS names)
    set_x: Optional[List[Optional[np.ndarray]]] = None
    refine_status: Optional[List[str]] = None


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def grid_point(pr: SetProblem, index: int) -> np.ndarray:
    """(d,) coordinates of flat grid index `index` of a set."""
    ii = np.unravel_index(int(index), [len(t) for t in pr.grid])
    return np.array([pr.grid[k][ii[k]] for k in range(pr.d)])


def refined_output(out: SweepOutput, problems: Sequence[SetProblem], owners: Sequence[int], gathered: bytes) -> SweepOutput:
    """Host assembly of SweepEngine.refine from the all-gathered cbo_refine_result tables (rank-major, one row of S records
    per rank): set g's record is the one in the row of owners[g] (partition.refine_owners; -1: no record, the set keeps its
    grid result).  A set whose record strictly improved on its start takes the refined value and coordinates; the selection
    is the sweep's rule (first maximum, NaN = -inf)."""
    S = len(problems)
    rows = (RefineResult * (len(gathered) // C.sizeof(RefineResult))).from_buffer_copy(gathered)
    grid_x = [grid_point(problems[g], out.set_indices[g]) if out.set_indices[g] >= 0 else None for g in range(S)]
    values = np.array(out.set_values, np.float64, copy=True)
    set_x = list(grid_x)
    status = ["skipped_nonfinite"] * S
    for g in range(S):
        if owners[g] < 0:
            continue
        r = rows[owners[g] * S + g]
        status[g] = _lib.REFINE_STATUS.get(r.status, str(r.status))
        if r.value > r.start_value:          # strictly improved (both finite)
            values[g] = r.value
            set_x[g] = np.array(r.x[:problems[g].d])
    valid = np.flatnonzero(np.asarray(out.set_indices) >= 0)
    s, value, x = -1, out.value, None
    if valid.size:
        v = np.where(np.isnan(values[valid]), -np.inf, values[valid])
        s = int(valid[int(np.argmax(v))])
        value, x = float(values[s]), set_x[s]
    return SweepOutput(s, int(out.set_indices[s]) if s >= 0 else out.index, value, x, values,
                       np.array(out.set_indices, copy=True), out.n_nan, dict(out.stage_ms), set_x=set_x, refine_status=status)


class SweepEngine:
    def __init__(self, problems: Sequence[SetProblem], device: str | torch.device = "cuda:0", rank: int = 0,
                 world_size: int = 1, keep: Sequence[str] = (), process_group=None, n_int_capacity: int = _lib.CBO_MAX_NINT,
                 pinned_staging: bool = False, fit_hyperparameters: bool = False):
        """fit_hyperparameters: fit each set's GP variance and lengthscale by marginal likelihood on the device (K8) before
        every posterior fit, instead of the reference's fixed (1, 1) (opt-in; off, every path and output is unchanged)."""
        if not torch.cuda.is_available():
            raise RuntimeError("SweepEngine needs a CUDA device: the CUDA library is the product, there is no CPU path")
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.rank, self.world = rank, world_size
        self.group = process_group
        self.problems = list(problems)
        # mu / var are always kept: they are the cache behind the post-intervention EI refresh (refresh())
        self.keep = tuple(dict.fromkeys(("mu", "var") + tuple(keep)))
        self.ncap = int(n_int_capacity)
        self._posterior_valid = set()     # global ids whose mu / var arrays match their current interventional data
        self._prior_rows_valid = set()    # global ids whose m_int / v_int match the rows that were on the device last
        self._row_begin = {}              # global id -> first interventional row without a prior yet (appended rows)
        self.timing = False
        self._launch0 = self.lib.cbo_launch_count()
        self.pinned_staging = pinned_staging
        self.fit_hyper = bool(fit_hyperparameters)
        for k in self.keep:
            if k not in ("mu", "var", "ei", "acq"):
                raise ValueError(f"unknown array {k!r}")
        S = len(self.problems)
        sizes = [SetSize(p.g_total, p.x_obs_int.shape[0] if p.computes_prior else 0, p.x_int.shape[0]) for p in self.problems]
        slices = partition(sizes, world_size)
        self.slices = slices[rank]
        self.refine_owner = refine_owners(slices)                       # global id -> the rank that refines the set
        self.active = [s for s in range(S) if self.slices[s][1] > 0]   # global ids of the sets this rank touches
        self.local_of = {g: i for i, g in enumerate(self.active)}
        self._alloc()
        self.upload()

    @property
    def launches(self) -> int:
        """Kernels of libcbo_b200 launched from this thread since the engine was built (the library tallies every
        launch site itself: cbo_launch_count; bench.py reports the per-step difference)."""
        return int(self.lib.cbo_launch_count() - self._launch0)

    # ------------------------------------------------------------------------------------------------
    def _dev(self, shape, dtype=torch.float64, zero=False):
        f = torch.zeros if zero else torch.empty
        return f(shape, dtype=dtype, device=self.device)

    def _alloc(self):
        A = len(self.active)
        self.h_sets = (SetDesc * max(A, 1))()
        self.buf: List[Dict[str, torch.Tensor]] = []
        self.stage: List[Dict[str, torch.Tensor]] = []   # pinned host staging of the inputs (e2e path)
        p_rows = p_cols = 0
        for g in self.active:
            pr = self.problems[g]
            if pr.computes_prior and pr.x_obs_cond.shape[1] > 0:
                p_rows = max(p_rows, _round_up(pr.x_obs_int.shape[0], _lib.CBO_NPAD))
                p_cols = max(p_cols, _round_up(pr.mc_cond.shape[0], _lib.CBO_SPAD))
        # P scratch of the prior precompute: one buffer per set when that is small (the library then runs every set in one
        # launch per stage), one shared stream-ordered buffer when the sets are large (0.8 GB each at N = 1e4)
        self.P = self._dev((p_rows * p_cols,)) if p_rows else None
        n_cond = sum(1 for g in self.active if self.problems[g].computes_prior and self.problems[g].x_obs_cond.shape[1] > 0)
        self._private_P = p_rows > 0 and n_cond > 1 and n_cond * p_rows * p_cols * 8 <= (1 << 30)
        for li, g in enumerate(self.active):
            pr = self.problems[g]
            d, n = pr.d, pr.x_int.shape[0]
            if n > self.ncap or self.ncap > _lib.CBO_MAX_NINT:
                raise ValueError(f"set {g}: n_int={n} exceeds the capacity {self.ncap} (max {_lib.CBO_MAX_NINT})")
            gb, gc = self.slices[g]
            b: Dict[str, torch.Tensor] = {}
            b["x_int"] = self._dev((self.ncap * d,))
            b["y_int"] = self._dev((self.ncap,))
            b["L"] = self._dev((self.ncap * self.ncap,))
            b["alpha"] = self._dev((self.ncap,))
            b["sqrt_v_int"] = self._dev((self.ncap,), zero=True)
            b["m_int"] = self._dev((self.ncap,), zero=True)
            b["v_int"] = self._dev((self.ncap,), zero=True)
            b["fit_info"] = self._dev((2,), dtype=torch.int32, zero=True)
            if self.fit_hyper:
                b["hyper"] = torch.ones((2,), dtype=torch.float64, device=self.device)
            for k in range(d):
                b[f"grid{k}"] = self._dev((len(pr.grid[k]),))
            for name in self.keep:
                b[name] = self._dev((gc,))
            if pr.causal and pr.prior_external:
                b["m"] = self._dev((gc,), zero=True)
                b["v"] = self._dev((gc,), zero=True)
            if pr.computes_prior:
                N, c, Smc = pr.x_obs_int.shape[0], pr.x_obs_cond.shape[1], pr.mc_cond.shape[0]
                Np = _round_up(N, _lib.CBO_NPAD)
                b["x_obs_int"] = self._dev((d * N,))
                b["x_obs_cond"] = self._dev((max(c * N, 1),))
                b["mc_cond"] = self._dev((max(c * Smc, 1),))
                b["alpha_obs"] = self._dev((N,))
                b["kyinv"] = self._dev((N * N,))
                if pr.device_fit:
                    if pr.y_obs is None:
                        raise ValueError(f"set {g}: neither (alpha_obs, kyinv) nor y_obs was given")
                    b["y_obs"] = self._dev((N,))
                for k in range(d):
                    b[f"tab{k}"] = self._dev((len(pr.grid[k]) * Np,))
                b["u_int"] = self._dev((self.ncap * Np,))
                b["pbar"] = self._dev((Np,))
                b["w"] = self._dev((Np,))
                b["M"] = self._dev((Np * Np,))
                if self._private_P and c > 0:
                    b["P"] = self._dev((Np * _round_up(max(Smc, 1), _lib.CBO_SPAD),))
                b["m"] = self._dev((gc,))
                b["v"] = self._dev((gc,))
            self.buf.append(b)
        # sweep scratch / outputs
        self._fill_descs()
        n_items = self.lib.cbo_sweep_num_items(self.h_sets, A) if A else 0
        # prior-eval workspace: one scratch slot per SM (persistent kernel, one CTA per SM)
        self.num_sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        ws = self.lib.cbo_prior_workspace_bytes(self.h_sets, A, self.num_sms) if A else 0
        self.prior_ws = torch.empty((max(ws, 256),), dtype=torch.uint8, device=self.device)
        self.tile_best = torch.empty((max(n_items, 1) * C.sizeof(SetBest),), dtype=torch.uint8, device=self.device)
        S = len(self.problems)
        # [cbo_sweep_result | S x cbo_set_best]: the step's whole result, read back with ONE device -> host copy into pinned
        # memory (an event, not a blocking .cpu()).  On a single rank that touches every set the sweep's own per-set
        # reduction writes straight into the global table (local ids == global ids): no scatter, no second combine.
        self.out_buf = torch.empty((C.sizeof(SweepResult) + S * C.sizeof(SetBest),), dtype=torch.uint8, device=self.device)
        self.out_host = torch.empty((self.out_buf.numel(),), dtype=torch.uint8).pin_memory()
        self._out_event = torch.cuda.Event()
        self.result = self.out_buf[:C.sizeof(SweepResult)]
        self.global_best = self.out_buf[C.sizeof(SweepResult):]
        self._direct = self.world == 1 and self.active == list(range(S))
        self.local_best = self.global_best if self._direct else \
            torch.empty((max(A, 1) * C.sizeof(SetBest),), dtype=torch.uint8, device=self.device)
        self.gathered = torch.empty((self.world * S * C.sizeof(SetBest),), dtype=torch.uint8, device=self.device)
        empty = (SetBest * S)()
        for s in range(S):
            empty[s].value, empty[s].index = -np.inf, -1
        self._empty_best = torch.frombuffer(bytearray(bytes(empty)), dtype=torch.uint8).to(self.device)

    def _fill_descs(self):
        for li, g in enumerate(self.active):
            pr, b, D = self.problems[g], self.buf[li], self.h_sets[li]
            d, n = pr.d, pr.x_int.shape[0]
            gb, gc = self.slices[g]
            D.d, D.n_int, D.causal = d, n, int(pr.causal)
            for k in range(_lib.CBO_MAX_D):
                D.p[k] = len(pr.grid[k]) if k < d else 1
            D.g_total, D.g_begin, D.g_count = pr.g_total, gb, gc
            D.cost_fix, D.cost_variable = float(pr.cost_fix), int(bool(pr.cost_variable))
            D.prior_external = int(bool(pr.causal and pr.prior_external))
            ptr = lambda name: b[name].data_ptr() if name in b else None
            for k in range(d):
                D.grid[k] = ptr(f"grid{k}")
            D.x_int, D.y_int, D.L, D.alpha = ptr("x_int"), ptr("y_int"), ptr("L"), ptr("alpha")
            D.sqrt_v_int, D.m_int, D.v_int, D.fit_info = ptr("sqrt_v_int"), ptr("m_int"), ptr("v_int"), ptr("fit_info")
            D.mu, D.var, D.ei, D.acq = ptr("mu"), ptr("var"), ptr("ei"), ptr("acq")
            D.m, D.v = ptr("m"), ptr("v")
            D.hyper = ptr("hyper")
            if pr.computes_prior:
                N, c, Smc = pr.x_obs_int.shape[0], pr.x_obs_cond.shape[1], pr.mc_cond.shape[0]
                D.c, D.n_obs, D.n_obs_pad = c, N, _round_up(N, _lib.CBO_NPAD)
                D.n_mc, D.n_mc_pad = Smc, _round_up(max(Smc, 1), _lib.CBO_SPAD)
                D.s2, D.noise = float(pr.s2), float(pr.noise)
                ls_int = np.broadcast_to(np.asarray(pr.ls_int, np.float64).reshape(-1), (d,)) if np.size(pr.ls_int) in (1, d) else None
                if ls_int is None:
                    raise ValueError(f"set {g}: ls_int must have 1 or d entries")
                ls_cond = np.asarray(pr.ls_cond, np.float64).reshape(-1)
                if c and ls_cond.size == 1:
                    ls_cond = np.repeat(ls_cond, c)
                if ls_cond.size != c:
                    raise ValueError(f"set {g}: ls_cond must have c={c} entries")
                for k in range(d):
                    D.ls_int[k] = float(ls_int[k])
                for k in range(c):
                    D.ls_cond[k] = float(ls_cond[k])
                D.x_obs_int, D.x_obs_cond, D.mc_cond = ptr("x_obs_int"), ptr("x_obs_cond"), ptr("mc_cond")
                D.alpha_obs, D.kyinv, D.y_obs = ptr("alpha_obs"), ptr("kyinv"), ptr("y_obs")
                for k in range(d):
                    D.tab[k] = ptr(f"tab{k}")
                D.u_int, D.pbar, D.w, D.M = ptr("u_int"), ptr("pbar"), ptr("w"), ptr("M")
                D.P = ptr("P") if "P" in b else (self.P.data_ptr() if (self.P is not None and c > 0) else None)
        A = len(self.active)
        self.d_sets = torch.empty((max(A, 1) * C.sizeof(SetDesc),), dtype=torch.uint8, device=self.device)
        self._descs_dirty = True
        self._push_descs()

    def _push_descs(self):
        """Upload the host descriptor array if it changed since the last upload.  Flag and size changes only touch the
        host copy; every stage call starts with this, so a trial uploads the descriptors once, not once per change."""
        if self._descs_dirty:
            raw = bytearray(bytes(self.h_sets))
            self.d_sets.copy_(torch.frombuffer(raw, dtype=torch.uint8))
            self._descs_dirty = False

    # ------------------------------------------------------------------------------------------------
    def _h2d(self, dst: torch.Tensor, arr: np.ndarray, key, restage: bool):
        """One input array to the device.  With pinned staging the host copy lives in page-locked memory (filled
        when the array is (re)staged) and the transfer is an asynchronous DMA on the current stream."""
        if not self.pinned_staging:
            arr = np.ascontiguousarray(arr, dtype=np.float64).reshape(-1)
            if arr.size:
                dst[:arr.size].copy_(torch.from_numpy(arr))
            return arr.nbytes
        st = self._pins.get(key)
        if st is None or restage:
            arr = np.ascontiguousarray(arr, dtype=np.float64).reshape(-1)
            if st is None or st.numel() != arr.size:
                st = torch.empty((arr.size,), dtype=torch.float64).pin_memory()
                self._pins[key] = st
            if arr.size:
                st.numpy()[:] = arr
        if st.numel():
            dst[:st.numel()].copy_(st, non_blocking=True)
        return st.numel() * 8

    def upload(self, what: str = "all", restage: bool = False) -> int:
        """Copy the host inputs to the device; returns the bytes moved.  what = 'all' | 'interventional'.
        restage=True re-reads the caller's NumPy arrays into the pinned staging buffers first (needed after the
        caller changed them in place); otherwise the staged copies are what is transferred."""
        if not hasattr(self, "_pins"):
            self._pins: Dict[object, torch.Tensor] = {}
        total = 0
        for li, g in enumerate(self.active):
            pr, b = self.problems[g], self.buf[li]
            total += self._h2d(b["x_int"], pr.x_int, (li, "x_int"), restage)
            total += self._h2d(b["y_int"], pr.y_int, (li, "y_int"), restage)
            if pr.causal and pr.prior_external:
                total += self._h2d(b["m_int"], pr.m_int, (li, "m_int"), restage)
                total += self._h2d(b["v_int"], pr.v_int, (li, "v_int"), restage)
            if what == "interventional":
                continue
            if pr.causal and pr.prior_external and pr.m_grid is not None:
                gb, gc = self.slices[g]
                total += self._h2d(b["m"], np.asarray(pr.m_grid).reshape(-1)[gb:gb + gc], (li, "m"), restage)
                total += self._h2d(b["v"], np.asarray(pr.v_grid).reshape(-1)[gb:gb + gc], (li, "v"), restage)
            for k in range(pr.d):
                total += self._h2d(b[f"grid{k}"], pr.grid[k], (li, f"grid{k}"), restage)
            if pr.computes_prior:
                total += self._h2d(b["x_obs_int"], np.asarray(pr.x_obs_int).T, (li, "x_obs_int"), restage)
                total += self._h2d(b["x_obs_cond"], np.asarray(pr.x_obs_cond).T, (li, "x_obs_cond"), restage)
                total += self._h2d(b["mc_cond"], np.asarray(pr.mc_cond).T, (li, "mc_cond"), restage)
                if pr.device_fit:
                    total += self._h2d(b["y_obs"], pr.y_obs, (li, "y_obs"), restage)
                    self._obs_fit_stale = True
                else:
                    total += self._h2d(b["alpha_obs"], pr.alpha_obs, (li, "alpha_obs"), restage)
                    total += self._h2d(b["kyinv"], pr.kyinv, (li, "kyinv"), restage)
        return total

    def fit_observational(self):
        """K5 for every set whose observational-GP state is produced on the device (SetProblem.device_fit): Gram, blocked
        Cholesky, Ky^-1 and alpha from (x_obs, y_obs), with GPy's jitter-retry rule driven from here
        (fit_gaussian_process, utils.py:40-45, for frozen hyper-parameters)."""
        self._obs_fit_stale = False
        todo = [li for li, g in enumerate(self.active) if self.problems[g].device_fit]
        if not todo:
            return
        self._push_descs()
        if getattr(self, "fit_ws", None) is None:
            self.fit_ws = torch.empty((self.lib.cbo_obs_gp_workspace_bytes(self.h_sets, len(self.active)),), dtype=torch.uint8,
                                      device=self.device)
            self.fit_info = torch.zeros((max(len(self.active), 1),), dtype=torch.int32, device=self.device)
        self.obs_fit_tries = {}
        for li in todo:       # one set at a time: each has its own jitter history
            pr = self.problems[self.active[li]]
            h = C.cast(C.byref(self.h_sets, li * C.sizeof(SetDesc)), C.POINTER(SetDesc))
            jitter, tries = 0.0, 0
            while True:
                _lib.check(self.lib.cbo_obs_gp_fit(h, 1, jitter, C.c_void_p(self.fit_ws.data_ptr()), self.fit_ws.numel(),
                                                   C.c_void_p(self.fit_info.data_ptr()), self._stream()), "cbo_obs_gp_fit")
                if int(self.fit_info[0].item()) == 0:
                    break
                if tries == 5:
                    raise np.linalg.LinAlgError(f"set {self.active[li]}: observational Gram matrix not positive definite, even with jitter")
                jitter = (pr.s2 + pr.noise + 1e-8) * 1e-6 if tries == 0 else jitter * 10.0
                tries += 1
            self.obs_fit_tries[self.active[li]] = tries

    def set_interventional(self, g: int, x_int: np.ndarray, y_int: np.ndarray):
        """Replace the interventional data of global set g (Monitor.add_intervention_data, Monitor.py:148-160)."""
        pr = self.problems[g]
        old_x = pr.x_int
        pr.x_int = np.asarray(x_int, np.float64).reshape(-1, pr.d)
        pr.y_int = np.asarray(y_int, np.float64).reshape(-1)
        if pr.x_int.shape[0] > self.ncap:
            raise ValueError(f"set {g}: n_int={pr.x_int.shape[0]} exceeds capacity {self.ncap}")
        if g in self.local_of:
            li = self.local_of[g]
            # rows appended to an unchanged prefix whose prior is on the device: the next refresh() evaluates the prior of
            # the new rows only (cbo_set_desc.int_row_begin); anything else re-evaluates every row
            n_old = old_x.shape[0]
            appended = (g in self._prior_rows_valid and pr.x_int.shape[0] > n_old and np.array_equal(pr.x_int[:n_old], old_x))
            self._row_begin[g] = min(self._row_begin.get(g, n_old), n_old) if appended else 0
            self.h_sets[li].n_int = pr.x_int.shape[0]
            self._h2d(self.buf[li]["x_int"], pr.x_int, (li, "x_int"), True)
            self._h2d(self.buf[li]["y_int"], pr.y_int, (li, "y_int"), True)
            self._descs_dirty = True
            self._posterior_valid.discard(g)

    # ------------------------------------------------------------------------------------------------
    @property
    def d2h_bytes_per_sweep(self) -> int:
        return C.sizeof(SweepResult) + len(self.problems) * C.sizeof(SetBest)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _subset(self, local_ids: Optional[Sequence[int]]):
        """(host descriptor pointer, device descriptor pointer, count) for all active sets or a contiguous run."""
        self._push_descs()
        A = len(self.active)
        if local_ids is None:
            return self.h_sets, C.c_void_p(self.d_sets.data_ptr()), A
        ids = list(local_ids)
        if ids != list(range(ids[0], ids[0] + len(ids))):
            raise ValueError("subset must be a contiguous run of local set ids")
        h = C.cast(C.byref(self.h_sets, ids[0] * C.sizeof(SetDesc)), C.POINTER(SetDesc))
        return h, C.c_void_p(self.d_sets.data_ptr() + ids[0] * C.sizeof(SetDesc)), len(ids)

    def _timed(self, name, fn, out):
        if not self.timing:
            fn()
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(self.device))
        fn()
        e1.record(torch.cuda.current_stream(self.device))
        out.append((name, e0, e1))

    def build_tables(self, local_ids=None):
        h, dptr, n = self._subset(local_ids)
        if n:
            _lib.check(self.lib.cbo_build_tables(h, dptr, n, self._stream()), "cbo_build_tables")

    def prior_precompute(self, local_ids=None):
        h, dptr, n = self._subset(local_ids)
        if n:
            _lib.check(self.lib.cbo_prior_precompute(h, dptr, n, self._stream()), "cbo_prior_precompute")

    def prior_eval(self, which: int, local_ids=None):
        h, dptr, n = self._subset(local_ids)
        if n:
            _lib.check(self.lib.cbo_prior_eval(h, dptr, n, which, C.c_void_p(self.prior_ws.data_ptr()),
                                               self.prior_ws.numel(), self._stream()), "cbo_prior_eval")

    def posterior_fit(self, local_ids=None):
        h, dptr, n = self._subset(local_ids)
        if n:
            _lib.check(self.lib.cbo_posterior_fit(h, dptr, n, self._stream()), "cbo_posterior_fit")

    def fit_hyperparameters(self, local_ids=None, max_iter: int = 100, gtol: float = 1e-6):
        """K8 (cbo_posterior_hyper_fit) for all active sets or a contiguous run of local ids: the variance and lengthscale of
        each set's GP by marginal likelihood on its current interventional data and prior at x_int (needs prior_eval(1)),
        within hyper_bounds(grid), written to the set's hyper buffer that the posterior fit, the sweep and the refinement
        read.  This is where the reference's models[i].optimize() (CBO.py:173) takes effect."""
        if not self.fit_hyper:
            raise ValueError("the engine was built with fit_hyperparameters=False: its sets have no hyper-parameter buffers")
        h, dptr, n = self._subset(local_ids)
        if not n:
            return
        first = 0 if local_ids is None else list(local_ids)[0]
        ids = self.active[first:first + n]
        bounds = np.ascontiguousarray(np.concatenate([hyper_bounds(self.problems[g].grid) for g in ids]), np.float64)
        if getattr(self, "_hyper_res", None) is None:
            self._hyper_res = torch.zeros((max(len(self.active), 1) * C.sizeof(HyperResult),), dtype=torch.uint8, device=self.device)
            self._hyper_ws = torch.empty((max(self.lib.cbo_posterior_hyper_workspace_bytes(self.h_sets, len(self.active)), 256),),
                                         dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.cbo_posterior_hyper_fit(h, dptr, n, bounds.ctypes.data_as(C.POINTER(C.c_double)), int(max_iter),
                                                    float(gtol), C.c_void_p(self._hyper_ws.data_ptr()), self._hyper_ws.numel(),
                                                    C.c_void_p(self._hyper_res.data_ptr() + first * C.sizeof(HyperResult)),
                                                    self._stream()), "cbo_posterior_hyper_fit")

    def hyperparameters(self, g: int):
        """(variance, lengthscale) of global set g's GP: what K8 last fitted, or the reference's (1.0, 1.0)."""
        if not self.fit_hyper:
            return 1.0, 1.0
        h = self.buf[self.local_of[g]]["hyper"].cpu().numpy()
        return float(h[0]), float(h[1])

    def hyper_result(self, g: int) -> Optional[dict]:
        """K8's cbo_hyper_result of global set g from its last fit (None before the first fit)."""
        if getattr(self, "_hyper_res", None) is None:
            return None
        li = self.local_of[g]
        raw = self._hyper_res[li * C.sizeof(HyperResult):(li + 1) * C.sizeof(HyperResult)].cpu().numpy().tobytes()
        r = HyperResult.from_buffer_copy(raw)
        out = {n: getattr(r, n) for n, _ in HyperResult._fields_}
        out["status"] = _lib.HYPER_STATUS.get(r.status, str(r.status))
        return out

    def posterior_nll(self, g: int) -> np.ndarray:
        """(-log p(y), d/dlog s2, d/dlog l) of global set g's GP at its current hyper-parameters (cbo_posterior_nll); needs
        the set's prior at x_int on the device."""
        h, dptr = self._local_desc(self.local_of[g])
        out = torch.empty((3,), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.cbo_posterior_nll(h, dptr, 1, C.c_void_p(out.data_ptr()), self._stream()), "cbo_posterior_nll")
        return out.cpu().numpy()

    def log_marginal_likelihood(self, g: int) -> float:
        """log p(y) of global set g's GP (GPy's model.log_likelihood()), from cbo_posterior_nll."""
        return -float(self.posterior_nll(g)[0])

    def _sweep_local(self, best: float, task: str):
        A = len(self.active)
        if task not in ("min", "max"):
            raise ValueError("task must be 'min' or 'max'")
        self._push_descs()
        if A:
            _lib.check(self.lib.cbo_sweep(self.h_sets, C.c_void_p(self.d_sets.data_ptr()), A, float(best),
                                          1 if task == "min" else -1, C.c_void_p(self.tile_best.data_ptr()),
                                          C.c_void_p(self.local_best.data_ptr()), C.c_void_p(self.result.data_ptr()),
                                          self._stream()), "cbo_sweep")

    def _to_global(self, local: torch.Tensor, table: torch.Tensor, rec: int):
        """Scatter this rank's records of its active sets (local ids, `rec` bytes each) into a global-indexed table."""
        if self.active:
            if not hasattr(self, "_active_idx"):
                self._active_idx = torch.as_tensor(self.active, device=self.device, dtype=torch.long)
            table.view(-1, rec).index_copy_(0, self._active_idx, local.view(-1, rec)[:len(self.active)])

    def _all_gather(self, table: torch.Tensor, gathered: torch.Tensor):
        """All-gather of a global-indexed per-set table over the engine's ranks, rank-major (NCCL; one rank: a copy)."""
        gather_set_bests(table, gathered, self.world, self.group)

    def _finish(self, events) -> SweepOutput:
        """Scatter the local per-set bests into the global table, all-gather over ranks (NCCL), combine on
        the device with the same deterministic rule on every rank, and read the 24-byte result back."""
        S, sb = len(self.problems), C.sizeof(SetBest)
        gb = self.global_best
        if not self._direct:
            gb.copy_(self._empty_best)
            self._to_global(self.local_best, gb, sb)
            # combine_kernel's input and output must not alias (both are __restrict__): one rank stages its table by a copy
            self._all_gather(gb, self.gathered)
            _lib.check(self.lib.cbo_argmax_combine(C.c_void_p(self.gathered.data_ptr()), self.world, S, C.c_void_p(gb.data_ptr()),
                                                   C.c_void_p(self.result.data_ptr()), self._stream()), "cbo_argmax_combine")
        # ONE device -> host read of the step's result, into pinned memory; wait on its event only
        self.out_host.copy_(self.out_buf, non_blocking=True)
        self._out_event.record(torch.cuda.current_stream(self.device))
        self._out_event.synchronize()
        out_h = self.out_host.numpy().tobytes()
        res_h, best_h = out_h[:C.sizeof(SweepResult)], out_h[C.sizeof(SweepResult):]
        r = SweepResult.from_buffer_copy(res_h)
        bests = (SetBest * S).from_buffer_copy(best_h)
        x = None
        if r.set >= 0:
            pr = self.problems[r.set]
            ii = np.unravel_index(r.index, [len(t) for t in pr.grid])
            x = np.array([pr.grid[k][ii[k]] for k in range(pr.d)])
        ms = {}
        for name, e0, e1 in events:
            ms[name] = ms.get(name, 0.0) + e0.elapsed_time(e1)
        return SweepOutput(r.set, r.index, r.value, x, np.array([b.value for b in bests]),
                           np.array([b.index for b in bests], dtype=np.int64), r.n_nan, ms)

    def sweep(self, best: float, task: str = "min") -> SweepOutput:
        """Full post-observation trial: prior precompute + prior on x_int and on the grid + posterior fit +
        EI / cost + argmax (reference CBO.intervene after an observe(), CBO.py:143-173)."""
        ev: list = []
        if getattr(self, "_obs_fit_stale", False):
            self._timed("obs_gp_fit", self.fit_observational, ev)
        self._timed("tables", self.build_tables, ev)
        self._timed("prior_precompute", self.prior_precompute, ev)
        self._set_row_begin({})
        self._timed("prior_eval_train", lambda: self.prior_eval(1), ev)
        self._prior_rows_valid = {g for g in self.active if self.problems[g].computes_prior}
        self._row_begin = {}
        if self.fit_hyper:
            self._timed("hyper_fit", self.fit_hyperparameters, ev)
        self._timed("posterior_fit", self.posterior_fit, ev)
        self._timed("prior_eval_grid", lambda: self.prior_eval(0), ev)
        self._timed("sweep", lambda: self._sweep_local(best, task), ev)
        self._posterior_valid = set(self.active)
        return self._finish(ev)

    def _set_row_begin(self, begins):
        """Write int_row_begin (global id -> first row to evaluate; missing = 0) into the host descriptors."""
        changed = False
        for li, g in enumerate(self.active):
            rb = int(begins.get(g, 0))
            if self.h_sets[li].int_row_begin != rb:
                self.h_sets[li].int_row_begin = rb
                changed = True
        self._descs_dirty |= changed

    def _mark_cached(self, cached_globals):
        """Set posterior_cached on the given sets (and clear it on the others) in the host descriptors."""
        changed = False
        for li, g in enumerate(self.active):
            flag = 1 if g in cached_globals else 0
            if self.h_sets[li].posterior_cached != flag:
                self.h_sets[li].posterior_cached = flag
                changed = True
        self._descs_dirty |= changed

    def refresh(self, best: float, task: str = "min", refit: Sequence[int] = ()) -> SweepOutput:
        """Post-intervention trial: the prior on the grid is cached; only the sets in `refit` (global ids) get
        their interventional table, prior at x_int and posterior refreshed
        (CBO.update_gaussian_process_of_last_intervention, CBO.py:224-235), then EI everywhere."""
        ev: list = []
        if task not in ("min", "max"):
            raise ValueError("task must be 'min' or 'max'")
        # sets that are not refitted keep their posterior: their share of the sweep is a 16 B/candidate EI refresh.
        # Both flags go into the descriptors before the first kernel: one upload for the whole trial.
        self._set_row_begin({g: self._row_begin.get(g, 0) for g in refit if g in self._prior_rows_valid})
        self._mark_cached(self._posterior_valid - set(refit))
        refit_local = [self.local_of[g] for g in refit if g in self.local_of]
        if not self.timing and not self.fit_hyper and len(refit_local) <= 1 and self.active:
            # the whole trial in one library call (cbo_refresh_trial): descriptor upload, the appended rows' table and prior,
            # the refit, the sweep and its reductions -- six launches, no Python between them
            li = refit_local[0] if refit_local else -1
            _lib.check(self.lib.cbo_refresh_trial(self.h_sets, C.c_void_p(self.d_sets.data_ptr()), len(self.active), li, float(best),
                                                  1 if task == "min" else -1, C.c_void_p(self.prior_ws.data_ptr()),
                                                  self.prior_ws.numel(), C.c_void_p(self.tile_best.data_ptr()),
                                                  C.c_void_p(self.local_best.data_ptr()), C.c_void_p(self.result.data_ptr()),
                                                  self._stream()), "cbo_refresh_trial")
            self._descs_dirty = False
            for g in refit:
                if g in self.local_of and self.problems[g].computes_prior:
                    self._prior_rows_valid.add(g)
                    self._row_begin.pop(g, None)
            self._set_row_begin({})
            self._mark_cached(set())
            self._posterior_valid = set(self.active)
            return self._finish(ev)
        for g in refit:
            if g not in self.local_of:
                continue
            li = [self.local_of[g]]
            if self.problems[g].computes_prior:
                self._timed("tables", lambda: self.build_tables(li), ev)
                self._timed("prior_eval_train", lambda: self.prior_eval(1, li), ev)
                self._prior_rows_valid.add(g)
                self._row_begin.pop(g, None)
            if self.fit_hyper:
                self._timed("hyper_fit", lambda: self.fit_hyperparameters(li), ev)
            self._timed("posterior_fit", lambda: self.posterior_fit(li), ev)
        self._timed("sweep", lambda: self._sweep_local(best, task), ev)
        self._set_row_begin({})      # host flags back to neutral; the device copy follows with the next trial's upload
        self._mark_cached(set())
        self._posterior_valid = set(self.active)
        return self._finish(ev)

    # ------------------------------------------------------------------------------------------------
    def evaluate_points(self, g: int, X: np.ndarray, best: float = 0.0, task: str = "min", stages: str = "all",
                        m_pts: Optional[np.ndarray] = None, v_pts: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
        """Evaluate global set g at arbitrary candidates X (m, d) with the set's CURRENT device state -- the explicit-point
        twin of the grid sweep, behind model.predict(X), acquisition.evaluate(X) and the DoCalculus closures
        (DoCalculus.py:34-66, causal_acquisition_functions.py:27-43).
        stages = 'prior': only m(X), v(X) (needs tables + prior_precompute done);
        stages = 'all'  : also mu, var, ei, acq (needs the posterior fit done).
        A set with an external prior takes m_pts / v_pts from the caller."""
        li = self.local_of[g]
        pr, D0 = self.problems[g], self.h_sets[li]
        X = np.ascontiguousarray(np.asarray(X, np.float64).reshape(-1, pr.d))
        mtot = X.shape[0]
        names = ["m", "v"] + (["mu", "var", "ei", "acq"] if stages == "all" else [])
        out = {k: np.empty(mtot) for k in names}
        if mtot == 0:
            return out
        Np = D0.n_obs_pad if pr.computes_prior else 0
        chunk = mtot if not Np else max(_lib.CBO_PRIOR_TILE, min(mtot, (256 << 20) // (8 * Np) // 128 * 128))
        dev = self.device
        for a in range(0, mtot, chunk):
            mc = min(chunk, mtot - a)
            D = SetDesc.from_buffer_copy(bytes(D0))
            pts = torch.from_numpy(X[a:a + mc].reshape(-1)).to(dev)
            bufs = {k: torch.empty((mc,), dtype=torch.float64, device=dev) for k in names}
            D.points = pts.data_ptr()
            D.p[0] = mc
            for k in range(1, _lib.CBO_MAX_D):
                D.p[k] = 1
            D.g_total, D.g_begin, D.g_count = mc, 0, mc
            D.m, D.v = bufs["m"].data_ptr(), bufs["v"].data_ptr()
            D.mu = bufs["mu"].data_ptr() if "mu" in bufs else None
            D.var = bufs["var"].data_ptr() if "var" in bufs else None
            D.ei = bufs["ei"].data_ptr() if "ei" in bufs else None
            D.acq = bufs["acq"].data_ptr() if "acq" in bufs else None
            tab0 = None
            if pr.computes_prior:
                tab0 = torch.empty((mc * Np,), dtype=torch.float64, device=dev)
                D.tab[0] = tab0.data_ptr()
            elif pr.causal:
                if m_pts is None or v_pts is None:
                    raise ValueError("a set with an external prior needs m_pts and v_pts")
                bufs["m"].copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(m_pts, np.float64).reshape(-1)[a:a + mc])))
                bufs["v"].copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(v_pts, np.float64).reshape(-1)[a:a + mc])))
            h = (SetDesc * 1)(D)
            d_desc = torch.frombuffer(bytearray(bytes(h)), dtype=torch.uint8).to(dev)
            dptr, st = C.c_void_p(d_desc.data_ptr()), self._stream()
            if pr.computes_prior:
                _lib.check(self.lib.cbo_build_tables(h, dptr, 1, st), "cbo_build_tables")
                _lib.check(self.lib.cbo_prior_eval(h, dptr, 1, 0, C.c_void_p(self.prior_ws.data_ptr()), self.prior_ws.numel(), st),
                           "cbo_prior_eval")
            if stages == "all":
                n_items = self.lib.cbo_sweep_num_items(h, 1)
                scratch = torch.empty(((n_items + 2) * C.sizeof(SetBest) + C.sizeof(SweepResult),), dtype=torch.uint8, device=dev)
                base = scratch.data_ptr()
                _lib.check(self.lib.cbo_sweep(h, dptr, 1, float(best), 1 if task == "min" else -1, C.c_void_p(base),
                                              C.c_void_p(base + n_items * C.sizeof(SetBest)),
                                              C.c_void_p(base + (n_items + 1) * C.sizeof(SetBest)), st), "cbo_sweep")
            for k in names:
                out[k][a:a + mc] = bufs[k].cpu().numpy()
        return out

    # ------------------------------------------------------------------------------------------------
    _GRAD_DTYPE = np.dtype([(n, "f8") for n in ("m", "v", "mu", "var", "ei", "acq")] +
                           [(n, "f8", (_lib.CBO_MAX_D,)) for n in ("dm", "dv", "dmu", "dvar", "dei", "dacq")])

    def _local_desc(self, li: int):
        self._push_descs()
        h = C.cast(C.byref(self.h_sets, li * C.sizeof(SetDesc)), C.POINTER(SetDesc))
        return h, C.c_void_p(self.d_sets.data_ptr() + li * C.sizeof(SetDesc))

    def _refine_workspace(self, nbytes: int) -> torch.Tensor:
        """K7's workspace, grown on demand and kept (stream-ordered reuse)."""
        ws = getattr(self, "_refine_ws", None)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty((max(nbytes, 256),), dtype=torch.uint8, device=self.device)
            self._refine_ws = ws
        return ws

    def acquisition_gradients(self, g: int, X: np.ndarray, best: float = 0.0, task: str = "min") -> Dict[str, np.ndarray]:
        """Value and gradient with respect to x of the prior, posterior, EI and EI / cost of global set g at the rows of X
        (m, d), with the set's CURRENT device state (cbo_acq_grad, K7): the gradient behind
        CausalExpectedImprovement.evaluate_with_gradients (causal_acquisition_functions.py:45-67).  Scalars come back with
        shape (m,), gradients (dm, dv, dmu, dvar, dei, dacq) with shape (m, d)."""
        if task not in ("min", "max"):
            raise ValueError("task must be 'min' or 'max'")
        li = self.local_of[g]
        pr = self.problems[g]
        X = np.ascontiguousarray(np.asarray(X, np.float64).reshape(-1, pr.d))
        m = X.shape[0]
        if m == 0:
            return {n: np.empty((0,) + ((pr.d,) if n.startswith("d") else ())) for n in self._GRAD_DTYPE.names}
        h, dptr = self._local_desc(li)
        one = self.lib.cbo_refine_workspace_bytes(h, 1)
        ws = self._refine_workspace(one * min(16, (m + 7) // 8))
        pts = torch.from_numpy(X.reshape(-1)).to(self.device)
        out = torch.empty((m * C.sizeof(AcqGradOut),), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.cbo_acq_grad(h, dptr, C.c_void_p(pts.data_ptr()), m, float(best), 1 if task == "min" else -1,
                                         C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(out.data_ptr()), self._stream()),
                   "cbo_acq_grad")
        rec = np.frombuffer(out.cpu().numpy().tobytes(), dtype=self._GRAD_DTYPE)
        return {n: (rec[n][:, :pr.d].copy() if n.startswith("d") else rec[n].copy()) for n in self._GRAD_DTYPE.names}

    def refine(self, out: SweepOutput, best: float, task: str = "min", max_iter: int = 30, gtol: float = 1e-7) -> SweepOutput:
        """Refine every set's acquisition maximum off the grid (cbo_refine, K7): a projected quasi-Newton ascent of EI / cost
        inside the set's box [min grid[k], max grid[k]], started at the set's grid argmax in `out` (the output of the sweep
        that left the current device state).  Replaces the L-BFGS polish of the reference's anchor search
        (causal_optimizer.py:52-62).  Returns a copy of `out` whose set_values, set_x and refine_status are per set and whose
        set / value / x are chosen by the sweep's rule (first maximum, NaN = -inf); `index` stays the grid index the chosen
        set started from.  A set that is skipped (external prior, explicit points, no finite grid maximum) or that no step
        improved keeps its grid index, value and coordinates bit for bit.

        On a multi-GPU engine this is a collective call, like sweep(), and `out` is the sweep's output (global indices):
        each set is refined by one rank that holds it (partition.refine_owners), the refined records are all-gathered
        (56 B per set and rank, stage_ms "refine_gather"), and every rank returns the same output, the one a single-GPU
        engine returns."""
        ev: list = []
        table = self._refine_local(out, best, task, max_iter, gtol, ev)
        gathered = torch.empty((self.world * table.numel(),), dtype=torch.uint8, device=self.device)
        self._timed("refine_gather", lambda: self._all_gather(table, gathered), ev)
        return self._refine_finish(out, gathered, ev)

    def _refine_local(self, out: SweepOutput, best: float, task: str, max_iter: int, gtol: float, ev: list) -> torch.Tensor:
        """This rank's share of refine(): one cbo_refine call over its active sets, in which each set the rank owns starts
        at its grid argmax in `out` and every other set at a NaN row (K7 skips it).  Returns the records scattered into a
        global-indexed device table of S cbo_refine_result (zeros where the rank has no record)."""
        if task not in ("min", "max"):
            raise ValueError("task must be 'min' or 'max'")
        S, A, rb = len(self.problems), len(self.active), C.sizeof(RefineResult)
        x0 = np.full((max(A, 1), _lib.CBO_MAX_D), np.nan)
        for li, g in enumerate(self.active):
            if self.refine_owner[g] == self.rank and out.set_indices[g] >= 0 and np.isfinite(out.set_values[g]):
                x0[li, :self.problems[g].d] = grid_point(self.problems[g], out.set_indices[g])
        table = torch.zeros((S * rb,), dtype=torch.uint8, device=self.device)
        if A:
            self._push_descs()
            ws = self._refine_workspace(self.lib.cbo_refine_workspace_bytes(self.h_sets, A))
            d_x0 = torch.from_numpy(x0.reshape(-1)).to(self.device)
            d_res = torch.empty((A * rb,), dtype=torch.uint8, device=self.device)
            self._timed("refine", lambda: _lib.check(self.lib.cbo_refine(
                self.h_sets, C.c_void_p(self.d_sets.data_ptr()), A, float(best), 1 if task == "min" else -1,
                C.c_void_p(d_x0.data_ptr()), int(max_iter), float(gtol), C.c_void_p(ws.data_ptr()), ws.numel(),
                C.c_void_p(d_res.data_ptr()), self._stream()), "cbo_refine"), ev)
            self._to_global(d_res, table, rb)
        return table

    def _refine_finish(self, out: SweepOutput, gathered: torch.Tensor, ev: list) -> SweepOutput:
        """Read the all-gathered tables back once and assemble the output (refined_output), the same on every rank."""
        res = refined_output(out, self.problems, self.refine_owner, gathered.cpu().numpy().tobytes())
        for name, e0, e1 in ev:
            e1.synchronize()
            res.stage_ms[name] = res.stage_ms.get(name, 0.0) + e0.elapsed_time(e1)
        return res

    def fetch(self, name: str, g: int) -> np.ndarray:
        """Device array of global set g as NumPy (parity tests / debugging)."""
        li = self.local_of[g]
        pr, b, D = self.problems[g], self.buf[li], self.h_sets[li]
        t = b["L" if name == "Linv" else name].cpu().numpy()
        n = D.n_int
        if name in ("m", "v", "mu", "var", "ei", "acq"):
            return t[:D.g_count]
        if name == "L":      # the factor; for n <= 48 K2 leaves L^-T in the strict upper triangle (K3's tensor-pipe path): "Linv"
            return np.tril(t[:n * n].reshape(n, n))
        if name == "Linv":
            A = t[:n * n].reshape(n, n)
            return np.triu(A, 1).T + np.diag(1.0 / np.diag(A))
        if name in ("alpha", "sqrt_v_int", "m_int", "v_int", "y_int"):
            return t[:n]
        if name == "x_int":
            return t[:n * pr.d].reshape(n, pr.d)
        if name == "M":   # stored blocked ([row block][k block][k4 group][row][4], see include/cbo_b200.h)
            Np = D.n_obs_pad
            return t.reshape(Np // 128, Np // 16, 4, 128, 4).transpose(0, 3, 1, 2, 4).reshape(Np, Np)[:D.n_obs, :D.n_obs]
        if name in ("w", "pbar"):
            return t[:D.n_obs]
        if name == "u_int":
            return t[:n * D.n_obs_pad].reshape(n, D.n_obs_pad)[:, :D.n_obs]
        if name.startswith("tab"):
            k = int(name[3:])
            return t.reshape(D.p[k], D.n_obs_pad)[:, :D.n_obs]
        return t
