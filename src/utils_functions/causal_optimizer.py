"""Acquisition maximiser (reference: src/utils_functions/causal_optimizer.py).  The reference draws
`num_anchor_points` = 100 uniform anchors, keeps the best and refines it with L-BFGS (:19, :52-62); the build's
deterministic replacement is the dense tensor-product grid with `num_anchor_points` points per dimension and the
first argmax (SURVEY.md §0).  With a model that is backed by the CUDA sweep the whole search is one device pass;
`refine=True` then polishes the grid maximum off the grid with on-device gradients (the reference's L-BFGS step)."""
import numpy as np


class CausalGradientAcquisitionOptimizer:
    def __init__(self, space, num_anchor_points=100, refine=False):
        self.space = space
        self.num_anchor_points = num_anchor_points
        self.refine = refine

    def optimize(self, acquisition, context=None):
        """Returns (x (1, d), acquisition value there)."""
        tables = self.space.grid_tables(self.num_anchor_points)
        ei, cost = getattr(acquisition, "numerator", acquisition), getattr(acquisition, "denominator", None)
        model = getattr(ei, "model", None)
        if model is not None and hasattr(model, "grid_argmax"):
            fix, variable = cost.kernel_form() if cost is not None else (1.0, False)
            value, x = model.grid_argmax(tables, float(ei.current_global_min) - float(ei.jitter), ei.task, fix, variable,
                                         refine=self.refine)
            return np.asarray(x, np.float64).reshape(1, -1), value
        # generic acquisition object: score the grid in chunks through its evaluate()
        mesh = np.meshgrid(*tables, indexing="ij")
        X = np.stack([g.reshape(-1) for g in mesh], axis=1)
        best_v, best_x = -np.inf, X[:1]
        for a in range(0, len(X), 1 << 16):
            v = np.asarray(acquisition.evaluate(X[a:a + (1 << 16)]), np.float64).reshape(-1)
            v = np.where(np.isnan(v), -np.inf, v)
            i = int(np.argmax(v))
            if v[i] > best_v:
                best_v, best_x = v[i], X[a + i:a + i + 1]
        return best_x, best_v
