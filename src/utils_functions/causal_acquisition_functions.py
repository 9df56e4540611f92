"""Causal Expected Improvement (reference: src/utils_functions/causal_acquisition_functions.py).

`evaluate(x)` keeps the reference signature, but the arithmetic -- posterior mean/variance at x, sd (u Phi(u) + phi(u))
with u = (best - mu) / sd, sign flipped for task 'max' -- runs in the CUDA sweep kernel (csrc/sweep.cu) through
`model.acquisition_points`.  `evaluate_with_gradients(x)` differentiates the same quantity on the device
(csrc/refine.cu, cbo_acq_grad) when the model provides gradients."""
import numpy as np
import scipy.stats


class _Quotient:
    """acquisition / cost (emukit's Acquisition.__truediv__ in the reference, utils.py:34)."""

    def __init__(self, numerator, denominator):
        self.numerator, self.denominator = numerator, denominator

    def evaluate(self, x):
        return self.numerator.evaluate(x) / self.denominator.evaluate(x)

    @property
    def has_gradients(self):
        return False


class CausalExpectedImprovement:
    def __init__(self, current_global_min, task, model, jitter=0.0):
        self.model = model
        self.jitter = jitter
        self.current_global_min = current_global_min
        self.task = task

    def evaluate(self, x):
        """EI at the rows of x, shape (m, 1) (reference :27-43).  A jitter on the mean is a shift of the incumbent."""
        x = np.atleast_2d(np.asarray(x, np.float64))
        out = self.model.acquisition_points(x, float(self.current_global_min) - float(self.jitter), self.task)
        return out["ei"].reshape(-1, 1)

    def evaluate_with_gradients(self, x):
        """(EI (m, 1), dEI/dx (m, d)) at the rows of x (reference :45-67)."""
        x = np.atleast_2d(np.asarray(x, np.float64))
        out = self.model.acquisition_gradients(x, float(self.current_global_min) - float(self.jitter), self.task)
        return out["ei"].reshape(-1, 1), out["dei"].reshape(x.shape[0], -1)

    def __truediv__(self, cost):
        return _Quotient(self, cost)

    @property
    def has_gradients(self):
        return bool(getattr(self.model, "has_gradients", False))


def get_standard_normal_pdf_cdf(x, mean, standard_deviation):
    """(u, phi(u), Phi(u)) with u = (x - mean) / sd (reference :77-88); host helper kept for API parity."""
    u = (x - mean) / standard_deviation
    return u, scipy.stats.norm.pdf(u), scipy.stats.norm.cdf(u)
