"""Factory of the per-exploration-set surrogates (reference: src/GaussianProcessFactory.py).

The reference returns GPy GPRegression objects (optionally inside emukit's GPyModelWrapper); this build returns
`SurrogateModel`, which has the surface the agent uses -- predict / set_data / optimize / X / Y -- and evaluates
everything with the CUDA kernels: Gram + Cholesky + solves in csrc/posterior_fit.cu, predictive mean / variance / EI
in csrc/sweep.cu.  Hyper-parameters are the reference's: lengthscale 1, variance 1, noise 1e-10 (:57-73), unless the agent
runs with --optimize_surrogates: then the variance and lengthscale of every set are fitted by marginal likelihood on the
device (csrc/posterior_hyper.cu) at each refit, and `kern` / `log_likelihood()` report them."""
from types import SimpleNamespace

from enum import IntEnum

import numpy as np


class GaussianProcessType(IntEnum):
    GRAPH_GP = 0
    CAUSAL_GP = 1
    NON_CAUSAL_GP = 2


class SurrogateModel:
    """GP on one exploration set's interventional data.  causal: prior mean m(.) and CausalRBF kernel built from the
    prior variance v(.) (reference :63-73); non-causal: zero mean, RBF (:57-60).
    If the mean / variance functions are DoCalculus closures the model shares the agent's AcquisitionSession (one
    device state for all sets); with arbitrary Python callables it keeps a private single-set session and feeds the
    callables' values to the kernels as an external prior."""

    def __init__(self, x, y, mean_function=None, var_function=None, device="cuda:0"):
        self.X = np.atleast_2d(np.asarray(x, np.float64))
        self.Y = np.asarray(y, np.float64).reshape(-1, 1)
        self.mean_function, self.var_function = mean_function, var_function
        self.causal = mean_function is not None
        self.device = device
        self._attached = None

    def attach(self, session_provider, set_index):
        """Bind the model to a session shared with other sets (used by the agent for its non-causal surrogates, whose
        constructor arguments carry no reference to the agent)."""
        self._attached = (session_provider, set_index)

    # ---- which device state ---------------------------------------------------------------------------
    def _shared(self):
        from src.DoCalculus import DoFunction
        if self._attached is not None:
            return self._attached[0](), self._attached[1]
        if isinstance(self.mean_function, DoFunction) and isinstance(self.var_function, DoFunction):
            dc = self.mean_function.do_calculus
            return dc.get_session(), self.mean_function.set_index
        return None

    def _private_session(self, tables, cost_fix=1.0, cost_variable=False, with_grid=False):
        from cbo_with_oop_b200.engine import SetProblem
        from cbo_with_oop_b200.session import AcquisitionSession
        y = self.Y.reshape(-1)
        if not self.causal:
            pr = SetProblem.non_causal(tables, self.X, y, cost_fix, cost_variable)
        else:
            m_int = np.asarray(self.mean_function(self.X), np.float64).reshape(-1)
            v_int = np.asarray(self.var_function(self.X), np.float64).reshape(-1)
            m_grid = v_grid = None
            if with_grid:
                mesh = np.meshgrid(*tables, indexing="ij")
                Xg = np.stack([g.reshape(-1) for g in mesh], axis=1)
                m_grid = np.concatenate([np.asarray(self.mean_function(Xg[a:a + 65536]), np.float64).reshape(-1)
                                         for a in range(0, len(Xg), 65536)])
                v_grid = np.concatenate([np.asarray(self.var_function(Xg[a:a + 65536]), np.float64).reshape(-1)
                                         for a in range(0, len(Xg), 65536)])
            pr = SetProblem.with_external_prior(tables, self.X, y, m_int, v_int, m_grid, v_grid, cost_fix, cost_variable)
        return AcquisitionSession([pr], device=self.device)

    # ---- reference surface ----------------------------------------------------------------------------
    def predict(self, X):
        """(mean (m,1), variance (m,1)) including the 1e-10 likelihood noise, no clipping (GPy GP.predict)."""
        r = self.acquisition_points(X, 0.0, "min")
        return r["mu"].reshape(-1, 1), r["var"].reshape(-1, 1)

    def acquisition_points(self, X, best, task):
        X = np.atleast_2d(np.asarray(X, np.float64))
        shared = self._shared()
        if shared is not None:
            session, g = shared
            session.mark_interventional(g, self.X, self.Y)
            return session.predict_points(g, X, best, task)
        d = self.X.shape[1]
        session = self._private_session([np.zeros(1)] * d)
        m_pts = v_pts = None
        if self.causal:
            m_pts = np.asarray(self.mean_function(X), np.float64).reshape(-1)
            v_pts = np.asarray(self.var_function(X), np.float64).reshape(-1)
        return session.predict_points(0, X, best, task, m_pts=m_pts, v_pts=v_pts)

    @property
    def has_gradients(self):
        """x-gradients come from the device prior (DoCalculus closures) or need no prior (non-causal); arbitrary Python
        mean / variance callables have no gradient."""
        return not self.causal or self._shared() is not None

    def acquisition_gradients(self, X, best, task):
        """Values and x-gradients of m, v, mu, var, EI and EI / cost at the rows of X (cbo_acq_grad); gradients (m, d)."""
        X = np.atleast_2d(np.asarray(X, np.float64))
        shared = self._shared()
        if shared is not None:
            session, g = shared
            session.mark_interventional(g, self.X, self.Y)
            return session.gradient_points(g, X, best, task)
        if self.causal:
            raise ValueError("gradients need the device prior: this model's mean / variance are arbitrary callables")
        session = self._private_session([np.zeros(1)] * self.X.shape[1])
        return session.gradient_points(0, X, best, task)

    def get_prediction_gradients(self, X):
        """(d mean / dx (m, d), d variance / dx (m, d)) at the rows of X (emukit's IDifferentiable interface)."""
        r = self.acquisition_gradients(X, 0.0, "min")
        return r["dmu"], r["dvar"]

    def grid_argmax(self, tables, best, task, cost_fix=1.0, cost_variable=False, refine=False):
        """(max of EI / cost over the tensor grid, its coordinates (d,)): the per-set form of the batched sweep.
        refine=True: the maximum refined off the grid inside the grid's box (SweepEngine.refine)."""
        def result(session, out, g):
            x = out.set_x[g] if refine and out.set_x[g] is not None else session.grid_point(g, out.set_indices[g])
            return float(out.set_values[g]), np.asarray(x, np.float64)
        shared = self._shared()
        if shared is not None:
            session, g = shared
            pr = session.engine.problems[g]
            same = len(tables) == pr.d and all(len(a) == len(b) and np.array_equal(a, b) for a, b in zip(tables, pr.grid)) \
                and float(cost_fix) == float(pr.cost_fix) and bool(cost_variable) == bool(pr.cost_variable)
            if same:
                session.mark_interventional(g, self.X, self.Y)
                return result(session, session.best_per_set(best, task, refine=refine), g)
        session = self._private_session(tables, cost_fix, cost_variable, with_grid=True)
        return result(session, session.best_per_set(best, task, refine=refine), 0)

    def set_data(self, X, Y):
        """emukit GPyModelWrapper.set_data (reference call site Monitor.py:160)."""
        self.X = np.atleast_2d(np.asarray(X, np.float64))
        self.Y = np.asarray(Y, np.float64).reshape(-1, 1)
        shared = self._shared()
        if shared is not None:
            shared[0].mark_interventional(shared[1], self.X, self.Y)

    def optimize(self):
        """The reference re-optimises this GP's hyper-parameters after every intervention (CBO.py:173) and discards
        them when the model is rebuilt with lengthscale 1 / variance 1 before the next acquisition (CBO.py:229-235,
        SURVEY.md Appendix B #16); keeping the fixed values is therefore behaviour-preserving.  With --optimize_surrogates
        the fit the reference meant to keep moves to the refit itself: the session's next posterior fit of this set runs the
        marginal-likelihood search first (SweepEngine.fit_hyperparameters), on the same data this call would have seen."""
        return None

    @property
    def hyperparameters(self):
        """(variance, lengthscale) of the per-set GP as the kernels use them: the fitted values when the shared session
        fits them (--optimize_surrogates), otherwise the reference's (1.0, 1.0)."""
        shared = self._shared()
        if shared is None:
            return 1.0, 1.0
        session, g = shared
        session.mark_interventional(g, self.X, self.Y)
        session.ensure_fit(g)
        return session.engine.hyperparameters(g)

    @property
    def kern(self):
        """GPy-shaped read access: model.kern.variance, model.kern.lengthscale."""
        s2, l = self.hyperparameters
        return SimpleNamespace(variance=s2, lengthscale=l)

    def log_likelihood(self):
        """log p(Y) of this GP at its current hyper-parameters (GPy's model.log_likelihood()), from cbo_posterior_nll."""
        shared = self._shared()
        if shared is not None:
            session, g = shared
            session.mark_interventional(g, self.X, self.Y)
        else:
            session, g = self._private_session([np.zeros(1)] * self.X.shape[1]), 0
        session.ensure_fit(g)
        return session.engine.log_marginal_likelihood(g)

    @property
    def model(self):          # emukit wrapper exposes the wrapped GPy model as .model
        return self


class GaussianProcessFactory:
    @staticmethod
    def create(gp_type, x, y, parameters=None, emukit_wrapper=False):
        """gp_type CAUSAL_GP: parameters = [mean_function, var_function]; NON_CAUSAL_GP: parameters ignored;
        GRAPH_GP: parameters = [lengthscale, variance, noise, ARD] (observational GP, not optimised).
        `emukit_wrapper` is accepted for compatibility: SurrogateModel already has the wrapper's interface."""
        makers = {
            GaussianProcessType.GRAPH_GP: GaussianProcessFactory.create_graph_gp,
            GaussianProcessType.CAUSAL_GP: GaussianProcessFactory.create_causal_gp,
            GaussianProcessType.NON_CAUSAL_GP: GaussianProcessFactory.create_non_causal_gp,
        }
        return makers[GaussianProcessType(gp_type)](x, y, parameters)

    @staticmethod
    def create_graph_gp(x, y, parameters):
        from src.utils_functions.utils import fit_gaussian_process
        return fit_gaussian_process(x, y, parameters, optimize=False)

    @staticmethod
    def create_non_causal_gp(x, y, _):
        return SurrogateModel(x, y)

    @staticmethod
    def create_causal_gp(x, y, parameters):
        mean_function, var_function = parameters
        return SurrogateModel(x, y, mean_function, var_function)
