"""CPU oracle of the acquisition's x-gradients and of the continuous refinement -- TEST INFRASTRUCTURE, NOT THE PRODUCT.

Restates in NumPy / SciPy float64 what csrc/refine.cu (K7) computes: the analytic gradients of the causal prior, the per-set
posterior, Expected Improvement and EI / cost (formulas as stated in the header of csrc/refine.cu), and the reference's
continuous polish of the best anchor (causal_optimizer.py:52-62, with the gradient of causal_acquisition_functions.py:45-67)
as SciPy L-BFGS-B.  Built on the values of oracle/cbo_oracle.py, which it leaves untouched; only tests/ import it.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg
import scipy.optimize
import scipy.stats

from oracle import cbo_oracle as O


def prior_gradients(gp, factors, intervened_cols, values):
    """m, v (m,) and dm/dx, dv/dx (m, d) of the factorised causal prior at the rows of ``values``:
    a_kj = u_j (x_k - X_jk) / l_k^2,  dm/dx_k = -sum_j a_kj w_j,  dv/dx_k = 2 a_k^T M u."""
    values = np.atleast_2d(np.asarray(values, np.float64))
    X = gp["X"]
    ls = gp["lengthscale"] if gp["lengthscale"].size > 1 else np.repeat(gp["lengthscale"], X.shape[1])
    U = O.intervened_u(gp, intervened_cols, values)
    MU = U @ factors["M"]
    m = U @ factors["w"]
    v = gp["variance"] + gp["noise"] - np.einsum("gj,gj->g", MU, U)
    d = len(intervened_cols)
    dm, dv = np.empty((values.shape[0], d)), np.empty((values.shape[0], d))
    for k, col in enumerate(intervened_cols):
        A = U * (values[:, k][:, None] - X[:, col][None, :]) / ls[col] ** 2
        dm[:, k] = -(A @ factors["w"])
        dv[:, k] = 2.0 * np.einsum("gj,gj->g", A, MU)
    return m, v, dm, dv


def acquisition_gradients(post, values, best, task="min", fix_costs=None, variable_cost=False, gp=None, factors=None,
                          intervened_cols=None):
    """Values and x-gradients of m, v, mu, var, EI and EI / cost at the rows of ``values`` (per-set GP distances from
    coordinate differences).  Causal sets need (gp, factors, intervened_cols); a non-causal set has m = v = 0.
      k*_i = e_i + sv_i sqrt(v),  dk*_i = -e_i (x - x_i) + sv_i dv / (2 sqrt v)
      dmu = dm + sum_i alpha_i dk*_i,  dvar = dv - 2 beta^T dk*,  beta = L^-T L^-1 k*
      dEI = -sign Phi(u) dmu + sign phi(u) dsd,  dacq = (dEI - acq dc) / c,  dc_k = [variable] sign(x_k)"""
    values = np.atleast_2d(np.asarray(values, np.float64))
    npts, d = values.shape
    if post["causal"]:
        m, v, dm, dv = prior_gradients(gp, factors, intervened_cols, values)
    else:
        m, v, dm, dv = np.zeros(npts), np.zeros(npts), np.zeros((npts, d)), np.zeros((npts, d))
    XI, L, alpha = post["XI"], post["L"], post["alpha"]
    sv = np.sqrt(post["vI"]) if post["causal"] else np.zeros(XI.shape[0])
    out = {k: np.empty(npts) for k in ("m", "v", "mu", "var", "ei", "acq")}
    out.update({k: np.empty((npts, d)) for k in ("dm", "dv", "dmu", "dvar", "dei", "dacq")})
    fix = float(np.sum(np.ones(d) if fix_costs is None else fix_costs))
    sign = 1.0 if task == "min" else -1.0
    with np.errstate(invalid="ignore", divide="ignore"):
        for a, x in enumerate(values):
            diff = x[None, :] - XI
            e = np.exp(-0.5 * np.sum(diff * diff, axis=1))
            sq = np.sqrt(v[a])
            ks = e + sv * sq
            dks = -e[:, None] * diff + (np.outer(sv, dv[a]) / (2.0 * sq) if post["causal"] else 0.0)
            mu = m[a] + ks @ alpha
            dmu = dm[a] + alpha @ dks
            t = scipy.linalg.solve_triangular(L, ks, lower=True)
            var = (1.0 + v[a]) - t @ t + O.POST_NOISE
            beta = scipy.linalg.solve_triangular(L, t, lower=True, trans="T")
            dvar = dv[a] - 2.0 * (beta @ dks)
            sd = np.sqrt(var)
            u = (best - mu) / sd
            pdf, cdf = scipy.stats.norm.pdf(u), scipy.stats.norm.cdf(u)
            ei = sign * sd * (u * cdf + pdf)
            dei = sign * (pdf * dvar / (2.0 * sd) - cdf * dmu)
            c = fix + (np.sum(np.abs(x)) if variable_cost else 0.0)
            dc = np.sign(x) if variable_cost else np.zeros(d)
            acq = ei / c
            for k, val in (("m", m[a]), ("v", v[a]), ("mu", mu), ("var", var), ("ei", ei), ("acq", acq)):
                out[k][a] = val
            for k, val in (("dm", dm[a]), ("dv", dv[a]), ("dmu", dmu), ("dvar", dvar), ("dei", dei), ("dacq", (dei - acq * dc) / c)):
                out[k][a] = val
    return out


def refine_set(post, x0, tables, best, task="min", fix_costs=None, variable_cost=False, gp=None, factors=None,
               intervened_cols=None, max_iter=500):
    """SciPy L-BFGS-B on -acq with the analytic gradient above, from x0 inside the box [min table_k, max table_k]
    (the reference's continuous polish, causal_optimizer.py:52-62).  Never returns a point worse than x0.
    Returns dict(x, value, start_value, hess_negdef): hess_negdef reports a negative-definite finite-difference Hessian of
    acq at an interior maximiser (where the maximiser is well determined)."""
    kw = dict(fix_costs=fix_costs, variable_cost=variable_cost, gp=gp, factors=factors, intervened_cols=intervened_cols)
    lo = np.array([np.min(t) for t in tables])
    hi = np.array([np.max(t) for t in tables])

    def f(x):
        r = acquisition_gradients(post, x[None, :], best, task, **kw)
        val, g = r["acq"][0], r["dacq"][0]
        if not np.isfinite(val):
            return np.inf, np.zeros_like(x)
        return -val, -g

    x0 = np.clip(np.asarray(x0, np.float64), lo, hi)
    start = -f(x0)[0]
    res = scipy.optimize.minimize(f, x0, jac=True, method="L-BFGS-B", bounds=list(zip(lo, hi)),
                                  options=dict(maxiter=max_iter, ftol=1e-15, gtol=1e-12))
    x, value = (res.x, -res.fun) if -res.fun > start else (x0, start)
    interior = bool(np.all((x > lo + 1e-9 * (hi - lo)) & (x < hi - 1e-9 * (hi - lo))))
    negdef = False
    if interior:
        h = 1e-5 * (hi - lo)
        d = x.size
        Hs = np.empty((d, d))
        for k in range(d):
            e = np.zeros(d)
            e[k] = h[k]
            Hs[k] = (f(x + e)[1] - f(x - e)[1]) / (2 * h[k])
        Hs = -0.5 * (Hs + Hs.T)
        negdef = bool(np.all(np.linalg.eigvalsh(Hs) < 0))
    return dict(x=x, value=float(value), start_value=float(start), hess_negdef=negdef, interior=interior)
