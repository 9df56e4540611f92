"""AcquisitionSession: a SweepEngine plus the bookkeeping of what is stale, shared by the objects of the
reference-shaped API (DoCalculus closures, per-set models, CBO.compute_best_acquisition_values).

State machine per trial (reference CBO.intervene, CBO.py:143-173):
  new observational GPs  -> new session: everything stale
  first acquisition      -> engine.sweep()    (tables, prior precompute, prior on x_int + grid, fits, EI, argmax)
  new interventional row -> mark_interventional(g): only set g's fit is stale
  next acquisition       -> engine.refresh(refit=stale sets)   (prior on the grid stays cached)
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

from .engine import SetProblem, SweepEngine, SweepOutput


class AcquisitionSession:
    def __init__(self, problems: Sequence[SetProblem], device="cuda:0", keep: Sequence[str] = (), fit_hyperparameters: bool = False):
        self.engine = SweepEngine(list(problems), device=device, keep=keep, fit_hyperparameters=fit_hyperparameters)
        self.num_sets = len(problems)
        self.prior_ready = False          # tables + prior precompute done
        self.grid_ready = False           # prior on the grid cached
        self.stale_fit = set(range(self.num_sets))
        self.last_output: Optional[SweepOutput] = None
        self._last_key = None

    # ---- stage guards ------------------------------------------------------------------------------
    def _ensure_prior(self):
        if not self.prior_ready:
            if getattr(self.engine, "_obs_fit_stale", False):
                self.engine.fit_observational()
            self.engine.build_tables()
            self.engine.prior_precompute()
            self.prior_ready = True

    def ensure_fit(self, g: int):
        """Bring global set g's posterior (and, when fitted, its hyper-parameters) up to date with its data."""
        self._ensure_fit(g)

    def _ensure_fit(self, g: int):
        self._ensure_prior()
        if g in self.stale_fit:
            li = [self.engine.local_of[g]]
            if self.engine.problems[g].computes_prior:
                self.engine.build_tables(li)           # the interventional-row table follows x_int
                self.engine.prior_eval(1, li)
            if self.engine.fit_hyper:
                self.engine.fit_hyperparameters(li)
            self.engine.posterior_fit(li)
            self.stale_fit.discard(g)

    # ---- data changes -------------------------------------------------------------------------------
    def mark_interventional(self, g: int, x_int: np.ndarray, y_int: np.ndarray):
        pr = self.engine.problems[g]
        x_int = np.asarray(x_int, np.float64).reshape(-1, pr.d)
        y_int = np.asarray(y_int, np.float64).reshape(-1)
        # unchanged data: nothing to do, whether or not the set is already waiting for a refit (Monitor.add_intervention_data
        # -> model.set_data marks the set first; the next compute_best_acquisition_values then passes the same arrays again
        # and must not reset the appended-row bookkeeping of the engine)
        if x_int.shape == pr.x_int.shape and np.array_equal(x_int, pr.x_int) and np.array_equal(y_int, pr.y_int):
            return
        self.engine.set_interventional(g, x_int, y_int)
        self.stale_fit.add(g)
        self.last_output = None

    # ---- evaluation ---------------------------------------------------------------------------------
    def prior_points(self, g: int, X: np.ndarray):
        """(m(X), v(X)) of global set g: the Monte-Carlo do-calculus average (DoCalculus.py:34-89) on the GPU."""
        self._ensure_prior()
        r = self.engine.evaluate_points(g, X, stages="prior")
        return r["m"], r["v"]

    def predict_points(self, g: int, X: np.ndarray, best: float = 0.0, task: str = "min", m_pts=None, v_pts=None
                       ) -> Dict[str, np.ndarray]:
        self._ensure_fit(g)
        return self.engine.evaluate_points(g, X, best=best, task=task, stages="all", m_pts=m_pts, v_pts=v_pts)

    def gradient_points(self, g: int, X: np.ndarray, best: float = 0.0, task: str = "min") -> Dict[str, np.ndarray]:
        """Values and x-gradients of the prior, posterior, EI and EI / cost of global set g at the rows of X (cbo_acq_grad)."""
        self._ensure_fit(g)
        return self.engine.acquisition_gradients(g, X, best=best, task=task)

    def best_per_set(self, best: float, task: str = "min", refine: bool = False) -> SweepOutput:
        """The batched form of CBO.compute_best_acquisition_values (CBO.py:237-260): every set's acquisition maximum --
        on the grid, or with refine=True refined off the grid from the grid maximum (SweepEngine.refine)."""
        key = (float(best), task, bool(refine))
        if self.grid_ready and not self.stale_fit and self.last_output is not None and self._last_key == key:
            return self.last_output      # nothing changed since the last sweep (per-set callers share one device pass)
        if refine:
            out = self.engine.refine(self.best_per_set(best, task), best, task)
            self._last_key, self.last_output = key, out
            return out
        self._last_key = key
        if not self.grid_ready:
            out = self.engine.sweep(best, task)
            self.prior_ready = self.grid_ready = True
            self.stale_fit.clear()
        else:
            refit = sorted(self.stale_fit)
            out = self.engine.refresh(best, task, refit=refit)
            self.stale_fit.clear()
        self.last_output = out
        return out

    def grid_point(self, g: int, flat_index: int) -> np.ndarray:
        pr = self.engine.problems[g]
        ii = np.unravel_index(int(flat_index), [len(t) for t in pr.grid])
        return np.array([pr.grid[k][ii[k]] for k in range(pr.d)])
