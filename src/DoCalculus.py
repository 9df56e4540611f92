"""Do-calculus engine (reference: src/DoCalculus.py): the causal prior E[Y | do(X = x)] and its variance for every
exploration set, as the Monte-Carlo average of observational-GP predictions over the observed samples.

Same surface as the reference -- `update_all_do_functions(gps)` returns [mean_functions, var_functions], one callable
per exploration set, f(values (m, d)) -> float64 (m, 1), memoised in cbo.x_mean / cbo.x_var by str(value) -- but the
arithmetic runs on the GPU: update_all_do_functions packs the fitted GPs into an AcquisitionSession (exp tables +
prior precompute kernels) and every closure call is one explicit-point pass of the prior kernel (mean and variance
together, so the two closures never repeat each other's work as they do in the reference, DoCalculus.py:59).
Deviations from the literal reference code, all listed in SURVEY.md Appendix B: the set -> GP table is explicit
(#3-#5), `np.mean` of the per-sample predictions is what is returned (#6), the memo is cleared when new observational
GPs arrive (#15)."""
from __future__ import annotations

import numpy as np


class DoFunction:
    """Prior mean (index 0) or variance (index 1) of one exploration set, callable like the reference's partials."""

    def __init__(self, do_calculus, set_index, index):
        self.do_calculus, self.set_index, self.index = do_calculus, set_index, index

    def __call__(self, values):
        dc = self.do_calculus
        return dc.update_do_function(dc.gaussian_processes, dc.cbo.exploration_set[self.set_index], self.index, values)


class DoCalculus:
    def __init__(self, cbo):
        self.cbo = cbo
        self.gaussian_processes = None
        self.session = None

    # ---- reference API --------------------------------------------------------------------------------
    def update_all_do_functions(self, gaussian_processes):
        self.gaussian_processes = gaussian_processes
        self.session = None                       # built lazily: the monitor may not exist yet at construction time
        for name in self.cbo.intervention_names:  # stale priors must not survive new observations
            self.cbo.x_mean[name].clear()
            self.cbo.x_var[name].clear()
        return [self.update_do_functions(index, gaussian_processes) for index in [0, 1]]

    def update_do_functions(self, index, gaussian_processes):
        return [DoFunction(self, s, index) for s in range(self.cbo.es_size)]

    def update_do_function(self, gaussian_processes, intervention, index, values):
        name = "".join(intervention)
        s = self.cbo.intervention_names.index(name)
        values = np.atleast_2d(np.asarray(values, np.float64))
        means, variances = self.cbo.x_mean[name], self.cbo.x_var[name]
        keys = [str(v) for v in values]
        missing = [i for i, k in enumerate(keys) if k not in means]
        if missing:
            m, v = self.compute_do_batch(s, values[missing])
            for i, mi, vi in zip(missing, m, v):
                means[keys[i]] = np.float64(mi)
                variances[keys[i]] = np.float64(vi)
        table = means if index == 0 else variances
        return np.float64(np.array([table[k] for k in keys]).reshape(-1, 1))

    def compute_do(self, measurements, gp, value, input_vars, intervention_vars):
        """(mean, variance) of the do-prior at ONE value (reference :68-78 returns the per-sample predictions whose
        mean the caller takes; the build returns the averages directly)."""
        s = self.cbo.exploration_set.index(list(intervention_vars))
        m, v = self.compute_do_batch(s, np.asarray(value, np.float64).reshape(1, -1))
        return m.reshape(1, 1), v.reshape(1, 1)

    @staticmethod
    def get_intervened_inputs(measurements, input_var, intervention_vars, value):
        """One column of the intervened design (reference :80-89); kept for API parity / tests."""
        col = np.asarray(measurements[input_var], np.float64).reshape(-1, 1)
        if input_var in intervention_vars:
            col = np.ones_like(col) * value[intervention_vars.index(input_var)]
        return col

    # ---- GPU path -------------------------------------------------------------------------------------
    def compute_do_batch(self, set_index, values):
        return self.get_session().prior_points(set_index, values)

    def set_problem(self, s):
        """Pack exploration set s for the sweep: columns of its observational GP split into intervened / conditioning."""
        from cbo_with_oop_b200.engine import SetProblem
        cbo = self.cbo
        variables = cbo.exploration_set[s]
        cols = cbo.graph.prior_columns(variables)
        gp = self.gaussian_processes[cbo.graph.get_gp_name(cols)]
        pos = [cols.index(v) for v in variables]
        rest = [i for i in range(len(cols)) if i not in pos]
        ls = np.broadcast_to(np.asarray(gp.lengthscale, np.float64).reshape(-1), (len(cols),)) if np.size(gp.lengthscale) in (1, len(cols)) \
            else np.asarray(gp.lengthscale, np.float64)
        fix, variable = cbo.graph.fixed_cost_of(variables, cbo.type_cost)
        mon = cbo.monitor
        # a GP fitted by the agent carries no host-side Ky^-1: the engine forms alpha and Ky^-1 in HBM from (X, y)
        # (cbo_obs_gp_fit), so no N x N array crosses PCIe
        on_device = getattr(gp, "device_fit", False)
        state = dict(alpha_obs=None, kyinv=None, y_obs=np.asarray(gp.Y, np.float64).reshape(-1)) if on_device else \
            dict(alpha_obs=gp.alpha, kyinv=gp.kyinv)
        return SetProblem(x_obs_int=gp.X[:, pos], x_obs_cond=gp.X[:, rest], mc_cond=gp.X[:, rest], **state,
                          ls_int=ls[pos], ls_cond=ls[rest], s2=gp.variance, noise=gp.noise,
                          grid=mon.space_list[s].grid_tables(cbo.grid_points_per_dim), x_int=mon.data_x[s],
                          y_int=mon.data_y[s].reshape(-1), cost_fix=fix, cost_variable=variable, causal=True, name="".join(variables))

    def get_session(self):
        if self.session is None:
            from cbo_with_oop_b200.session import AcquisitionSession
            self.session = AcquisitionSession([self.set_problem(s) for s in range(self.cbo.es_size)], device=self.cbo.device,
                                              fit_hyperparameters=getattr(self.cbo, "optimize_surrogates", False))
        return self.session
