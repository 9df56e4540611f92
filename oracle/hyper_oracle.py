"""CPU oracle of the per-set GP with fitted hyper-parameters -- TEST INFRASTRUCTURE, NOT THE PRODUCT.

Restates in NumPy / SciPy float64 what csrc/posterior_hyper.cu (K8) and the consumers of `cbo_set_desc.hyper` (K2, K3, K7)
compute once the per-set kernel has a variance s2 and a lengthscale l instead of the reference's (1, 1):
  K(X, X') = s2 exp(-.5 |x - x'|^2 / l^2) [+ sqrt(v(X)) sqrt(v(X'))^T]   (coordinate differences, as the CUDA path)
  Ky = K + (1e-10 + 1e-8) I (+ GPy's jitter) ,  NLL = .5 r^T Ky^-1 r + sum log L_ii + .5 n log(2 pi)
  dNLL / d(log s2, log l) = .5 tr((Ky^-1 - alpha alpha^T) dK)
the posterior, EI and EI / cost with their x-gradients at (s2, l), K8's start lattice, and a multi-start SciPy L-BFGS-B over
the same starts and bounds.  Built on oracle/cbo_oracle.py (whose rbf_K takes (s2, l) already) and oracle/refine_oracle.py,
which it leaves unchanged; at (1, 1) every value is bit-identical to theirs.  Only tests/ and tools/ import it.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg
import scipy.optimize
import scipy.stats

from oracle import cbo_oracle as O
from oracle import refine_oracle as R

NUM_STARTS = 9


def kernel(X, X2, s2, l, vX=None, vX2=None, form="diff"):
    """s2 exp(-.5 r^2 / l^2) (+ sqrt(vX) sqrt(vX2)^T for a causal set)."""
    K = O.rbf_K(X, X2, s2, l, form)
    if vX is not None:
        K = K + np.outer(np.sqrt(vX), np.sqrt(vX2))
    return K


def gram(XI, s2, l, vI=None, form="diff"):
    """Ky = K(X_I, X_I) + (1e-10 + 1e-8) I; a non-causal set zeroes the diagonal of r^2 (RBF.K(X)), as cbo_oracle does."""
    XI = np.asarray(XI, np.float64)
    if vI is None:
        K = O.rbf_K(XI, XI, s2, l, form, same=True)
    else:
        K = kernel(XI, XI, s2, l, vI, vI, form)
    return K + (O.POST_NOISE + O.GPY_JITTER) * np.eye(XI.shape[0])


def nll(XI, resid, s2, l, vI=None, grad=True):
    """(NLL, gradient in (log s2, log l) or None, jitter retries); NLL = +inf when Ky is not positive definite."""
    XI = np.asarray(XI, np.float64)
    r = np.asarray(resid, np.float64).reshape(-1)
    n = r.size
    Ky = gram(XI, s2, l, vI)
    try:
        L, tries = O.jitchol(Ky)
    except np.linalg.LinAlgError:
        return np.inf, (np.full(2, np.nan) if grad else None), -1
    alpha = scipy.linalg.cho_solve((L, True), r)
    z = scipy.linalg.solve_triangular(L, r, lower=True)
    f = 0.5 * (z @ z) + np.sum(np.log(np.diag(L))) + 0.5 * n * np.log(2.0 * np.pi)
    if not grad:
        return f, None, tries
    d = (XI[:, None, :] - XI[None, :, :]) / l
    r2 = np.sum(d * d, axis=2)
    G1 = s2 * np.exp(-0.5 * r2)
    W = scipy.linalg.cho_solve((L, True), np.eye(n)) - np.outer(alpha, alpha)
    g = 0.5 * np.array([np.sum(W * G1), np.sum(W * G1 * r2)])
    return f, g, tries


def posterior_fit(XI, yI, mI=None, vI=None, s2=1.0, l=1.0, form="diff"):
    """cbo_oracle.posterior_fit with (s2, l): what K2 computes from `hyper`."""
    XI = np.asarray(XI, np.float64)
    yI = np.asarray(yI, np.float64).reshape(-1)
    causal = mI is not None
    resid = yI - mI if causal else yI
    Ky = gram(XI, s2, l, vI if causal else None, form)
    L, tries = O.jitchol(Ky)
    alpha = scipy.linalg.cho_solve((L, True), resid)
    return dict(XI=XI, L=L, alpha=alpha, tries=tries, vI=(np.asarray(vI, np.float64) if causal else None), causal=causal,
                form=form, s2=float(s2), l=float(l))


def posterior_predict(post, Xg, mg=None, vg=None):
    """k* = K(X_I, x) at (s2, l); mu = m + k*.alpha; var = (s2 + v) - |L^-1 k*|^2 + 1e-10 (cbo_oracle.posterior_predict at (1, 1))."""
    Xg = np.atleast_2d(np.asarray(Xg, np.float64))
    s2, l = post["s2"], post["l"]
    if post["causal"]:
        Ks = kernel(post["XI"], Xg, s2, l, post["vI"], vg, post["form"])
        kdiag, mean0 = s2 + vg, mg
    else:
        Ks = O.rbf_K(post["XI"], Xg, s2, l, post["form"])
        kdiag, mean0 = s2 * np.ones(Xg.shape[0]), 0.0
    mu = Ks.T @ post["alpha"] + mean0
    tmp = scipy.linalg.solve_triangular(post["L"], Ks, lower=True)
    return mu, kdiag - np.sum(np.square(tmp), 0) + O.POST_NOISE


def acquisition_gradients(post, values, best, task="min", fix_costs=None, variable_cost=False, gp=None, factors=None,
                          intervened_cols=None):
    """refine_oracle.acquisition_gradients at (s2, l) = (post['s2'], post['l']):
    k*_i = s2 e_i + sv_i sqrt(v),  dk*_i = -s2 e_i (x - x_i) / l^2 + sv_i dv / (2 sqrt v),  var = (s2 + v) - |L^-1 k*|^2 + 1e-10."""
    values = np.atleast_2d(np.asarray(values, np.float64))
    npts, d = values.shape
    s2, l = post["s2"], post["l"]
    if post["causal"]:
        m, v, dm, dv = R.prior_gradients(gp, factors, intervened_cols, values)
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
            diff = (x[None, :] - XI) / l
            e = s2 * np.exp(-0.5 * np.sum(diff * diff, axis=1))
            sq = np.sqrt(v[a])
            ks = e + sv * sq
            dks = -e[:, None] * diff / l + (np.outer(sv, dv[a]) / (2.0 * sq) if post["causal"] else 0.0)
            mu = m[a] + ks @ alpha
            dmu = dm[a] + alpha @ dks
            t = scipy.linalg.solve_triangular(L, ks, lower=True)
            var = (s2 + v[a]) - t @ t + O.POST_NOISE
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


def log_box(bounds):
    """(lo, hi) of the search box in (log s2, log l) from (s2_lo, s2_hi, l_lo, l_hi)."""
    b = np.log(np.asarray(bounds, np.float64))
    return np.array([b[0], b[2]]), np.array([b[1], b[3]])


def starts(bounds, resid):
    """K8's starts in (log s2, log l): start 0 = (1, 1); starts 1..8 = {log var(r), log var(r) + log 10} x the centres of the
    four quarters of [log l_lo, log l_hi] (the lengthscale fastest); all clipped to the box."""
    lo, hi = log_box(bounds)
    r = np.asarray(resid, np.float64).reshape(-1)
    mean = 0.0
    for x in r:
        mean += x
    mean /= r.size
    var = 0.0
    for x in r:
        var += (x - mean) * (x - mean)
    var /= r.size
    out = [np.zeros(2)]
    for k in range(1, NUM_STARTS):
        a, b = (k - 1) % 4, (k - 1) // 4
        out.append(np.array([(np.log(var) if var > 0 else lo[0]) + b * np.log(10.0), lo[1] + (a + 0.5) * 0.25 * (hi[1] - lo[1])]))
    return [np.clip(t, lo, hi) for t in out]


def projected_gradient(theta, g, bounds):
    """The gradient with the components that point out of the box at an active bound zeroed (K8's convergence test)."""
    lo, hi = log_box(bounds)
    pg = np.array(g, np.float64, copy=True)
    for k in range(2):
        if hi[k] <= lo[k] or (theta[k] <= lo[k] and g[k] > 0) or (theta[k] >= hi[k] and g[k] < 0):
            pg[k] = 0.0
    return pg


def fit(XI, resid, bounds, vI=None):
    """SciPy L-BFGS-B on the NLL in (log s2, log l) from every start of `starts`; returns dict(best=(f, theta), runs)."""
    lo, hi = log_box(bounds)

    def fun(th):
        f, g, _ = nll(XI, resid, np.exp(th[0]), np.exp(th[1]), vI)
        if not np.isfinite(f):
            return 1e300, np.zeros(2)
        return f, g

    runs = []
    for t0 in starts(bounds, resid):
        res = scipy.optimize.minimize(fun, t0, jac=True, method="L-BFGS-B", bounds=list(zip(lo, hi)),
                                      options=dict(maxiter=1000, ftol=1e-15, gtol=1e-10))
        runs.append((float(res.fun), np.asarray(res.x, np.float64)))
    best = min(runs, key=lambda t: t[0])
    return dict(best=best, runs=runs)
