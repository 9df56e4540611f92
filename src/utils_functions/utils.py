"""Helpers of the agent (reference: src/utils_functions/utils.py)."""
import numpy as np

from .cost_functions import *                                         # noqa: F401,F403  (the reference star-exports these)
from .causal_acquisition_functions import CausalExpectedImprovement   # noqa: F401
from .causal_optimizer import CausalGradientAcquisitionOptimizer


def find_current_global(current_y, dict_interventions, task):
    """Best observed target value over all exploration sets (reference :8-26)."""
    pick = np.min if task == "min" else np.max
    per_set = {name: [] for name in dict_interventions}
    for variable, value in current_y.items():
        if len(value) > 0:
            per_set[variable] = pick(value)
    choose = min if task == "min" else max
    return per_set[choose(per_set, key=per_set.get)]


def find_next_y_point(space, model, current_global_best, evaluated_set, costs_functions, task="min", refine=False):
    """Maximise EI / cost over the set's candidates and return (acquisition value (1,1), x_new (1,d)) (reference :29-37).
    The reference scores 100 random anchors and refines the best with L-BFGS; this build takes the argmax of the dense
    tensor-product grid (100 points per dimension), evaluated by the CUDA sweep; refine=True refines that maximum off the
    grid with on-device gradients."""
    cost_acquisition = Cost(costs_functions, evaluated_set)
    optimizer = CausalGradientAcquisitionOptimizer(space, refine=refine)
    acquisition = CausalExpectedImprovement(current_global_best, task, model) / cost_acquisition
    x_new, y_acquisition = optimizer.optimize(acquisition)
    return np.asarray(y_acquisition, np.float64).reshape(1, 1), x_new


class ObservationalGP:
    """State of one observational GP (RBF, Gaussian noise fixed to 1e-2): what DoCalculus needs of the GPRegression
    object the reference builds at utils.py:40-45.  When the agent fits on the device (`device_fit`), the O(N^3) state
    (alpha = Ky^-1 y, Ky^-1) is never formed on the host: DoCalculus hands X, y and the hyper-parameters to the engine and
    cbo_obs_gp_fit produces the state in HBM.  `alpha` / `kyinv` stay available as host arrays on demand (fixtures, tests)."""

    def __init__(self, X, Y, variance, lengthscale, noise, alpha=None, kyinv=None, ARD=False, device_fit=False):
        self.X, self.Y = X, Y
        self.variance, self.lengthscale, self.noise = float(variance), np.asarray(lengthscale, np.float64), float(noise)
        self._alpha, self._kyinv, self.ARD = alpha, kyinv, bool(ARD)
        self.device_fit = bool(device_fit) and alpha is None and kyinv is None
        self.columns = None

    def _host_state(self):
        if self._alpha is None or self._kyinv is None:
            from cbo_with_oop_b200.obs_gp import fit_state
            self._alpha, self._kyinv = fit_state(self.X, self.Y, self.variance, self.lengthscale, self.noise)
        return self._alpha, self._kyinv

    @property
    def alpha(self):
        return self._host_state()[0]

    @property
    def kyinv(self):
        return self._host_state()[1]


def fit_gaussian_process(x, y, parameter_list, optimize=True, device=None):
    """RBF GP regression of y on x with the likelihood variance fixed to 1e-2 (the `noise_var=parameter_list[2]`
    argument is overwritten in the reference too, utils.py:43), hyper-parameters optimised from
    lengthscale = parameter_list[0], variance = parameter_list[1], ARD = parameter_list[3].
    With a `device` the marginal-likelihood search evaluates its objective and gradient on the GPU (cbo_obs_gp_fit +
    cbo_obs_gp_nll) and the returned object carries no host-side Ky^-1: the engine refits on the device."""
    from cbo_with_oop_b200.obs_gp import optimize_hyperparameters
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64).reshape(-1)
    ls0, s20, ard = parameter_list[0], parameter_list[1], bool(parameter_list[3])
    if optimize:
        s2, ls = optimize_hyperparameters(x, y, s2=s20, ls=ls0, ard=ard, noise=1e-2, device=device)
    else:
        s2, ls = float(s20), np.repeat(float(ls0), x.shape[1])
    return ObservationalGP(x, y.reshape(-1, 1), s2, ls, 1e-2, ARD=ard, device_fit=device is not None)
