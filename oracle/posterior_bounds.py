"""Reference values and proven error bounds for the per-set surrogate GP kernels.

    K2 (csrc/posterior_fit.cu): Ky = K + kSurrogateDiag I (+ jitter), L = jitchol(Ky), alpha = Ky^-1 r, W = L^-1 (n <= 48);
    K3 (csrc/sweep.cu): mu = m + k*.alpha, var = ((s2 + v) - |L^-1 k*|^2) + 1e-10, EI, acq = EI / cost, on six launch
        classes (forward substitution by the staged reciprocal diagonal, or t = W k* on DMMA; k* direct or from the
        separable tables);
    K7 (csrc/refine.cu, acq_grad_kernel): the same values at explicit points, by a column-oriented substitution.

Every builder takes the kernel's own inputs as fetched from the device (x_int, y_int, m_int, sqrt_v_int, L, W, alpha, the
candidates' m / v, hyper, best, the cost), so a check covers one kernel and none of the rounding of the stages that produced
its inputs.  u = 2^-53, gamma_k = k u / (1 - k u).  References are evaluated in np.longdouble (u_ld = 2^-64 on x86) and the
reference's own gamma(.., u_ld) is added to each bound, as in oracle/prior_bounds.py.  1 / l is formed once by the kernels
(fl(1 / l), IEEE division); the references use that same double, and sqrt(v) of a candidate is the IEEE-rounded double both
sides form.

Results in or below the subnormal range (exp(-r2 / 2) of distant points, products of tiny entries) lose up to 2^-1074
each; every bound carries a matching absolute term, which is negligible wherever the result is normal.

Two assumptions are stated rather than proven, as in prior_bounds: a DMMA.8x8x4 and an FMA each count as one IEEE rounding
of their result (a DMMA adds four products and the accumulator), and -fmad contraction is covered because every bound below
holds for any order of the additions and any fusing of a multiplication into the following addition (fusing removes a
rounding, it never adds one).  Where a bound is first order in u it is multiplied by SLACK = 2, which covers the neglected
O(n^2 u^2) terms many times over at n <= 128.

Gram entry (K2).  K_ij = s2 exp(-r2 / 2) + sv_i sv_j, r2 = sum_k ((x_ik - x_jk) il)^2.  The kernel rounds x_ik - x_jk, the
product by il, each square and each addition (d + 4 roundings on every term of r2: |r2^ - r2| <= gamma_{d+5} r2), evaluates
exp with at most EXP_ULP ulp (relative 2 EXP_ULP u), rounds s2 e (__dmul_rn) and fma(sv_i, sv_j, .), and adds
fl(kSurrogateDiag + jitter) to the diagonal with one more rounding:
    E_gram_ij = SLACK [s2 e_ij (r2_ij gamma_{d+5} / 2 + (2 EXP_ULP + 1) u) + u |K_ij|]  (+ u |Ky_ii| on the diagonal).

K2 factor.  surrogate_jitchol is LAPACK's right-looking Cholesky, but it multiplies by fl(1 / fl(sqrt(pivot))) instead of
dividing: l_ij carries two roundings where Higham's Theorem 10.3 (Accuracy and Stability, 2nd ed.) assumes one.  Repeating
his proof with the extra rounding, every entry satisfies |a_ij - sum_{k <= j} l_ik l_jk| <= gamma_{j+2} sum |l_ik||l_jk|, so
    |L^ L^T - Ky_ref| <= gamma_{n+3} |L^| |L^T| + E_gram,      c = 3 (one spare rounding).
Jitter: when fit_info[0] > 0 the reference forms the kernel's jitter bit for bit: diagonal entries fma(sv, sv, s2) rounded
once (exact rational -> float), + kSurrogateDiag, a sequential sum, / n, * 1e-6, then * 10 per further retry.

K2 alpha.  Higham Theorem 10.4 for the factor above and two substitutions by division: (Ky^ + dA) alpha^ = r^ with
|dA| <= gamma_{3n+4} |L^||L^T|.  With r^ = fl(y - m_int) (|dr| <= u |r|):
    |Ky_ref alpha^ - r_ref| <= gamma_{3n+4} |L^||L^T||alpha^| + E_gram |alpha^| + u |r|.
K2 W = L^-1 (n <= 48, surrogate_lower_inverse): W_cc = fl(1 / L_cc); W_ic = -fl(s_ic) * fl(1 / L_ii), s_ic the dot product of
row i of L with column c of W by four FMA partials and a butterfly.  Each entry is one forward substitution step, so the LEFT
residual has a bound free of cond(L):
    |L^ W^ - I| <= gamma_{n+4} |L^||W^|.

k* (K3, K7).  Direct form (FMA / generic / class 3 / K7): q_k = fl(fl(x_k il) - fl(x_int,ik il)), r2 = sum q_k^2 by FMA.
The staged products carry an absolute error u(|x_k| + |x_int,ik|) il each, and the subtraction u |q_k|, so
    dq_k = SLACK u ((|x_k| + |x_int,ik|) il + |q_k|),  dr2 = sum_k (2 |q_k| dq_k + dq_k^2) + gamma_d r2,
    |dk*_i| <= SLACK [s2 e_i (dr2 / 2 + (2 EXP_ULP + 1) u) + u (|sv_i svg| + |k*_i|)].
Separable form (classes 1, 2): eLead = __dmul_rn(s2, exp(-r2_lead / 2)), r2_lead from d - 1 rounded differences (gamma_{d+4});
eLast = exp(-q^2 / 2), q = fl(fl(g - x_int) il) (gamma_5 on q^2); k* = fma(eLead, eLast, fl(sv svg)):
    |dk*_i| <= SLACK [s2 e_i ((gamma_{d+4} r2_lead + gamma_5 q^2) / 2 + (4 EXP_ULP + 2) u) + u |sv_i svg| + u |k*_i|].
At d = 1 there are no leading dimensions: eLead = s2 exactly.

mu = m + sum k*_i alpha_i (any order, n + 1 additions, FMA products):
    |mu^ - mu_ref| <= gamma_{n+2} (|m| + sum |k*_i alpha_i|) + sum |dk*_i| |alpha_i|.
ss = |t|^2.  Substitution (FMA, generic: t_i = fl(four partials) * fl(1 / L_ii); K7: division by L_ii): L^ t^ = k^* + e with
|e| <= gamma_{n+3} |L^||t^|, so |t^ - L^-1 k*_ref| <= |L^-1| (gamma_{n+3} |L^||t| + |dk*|), L^-1 in longdouble.
DMMA (classes 2, 3): t^ = W^ k^* with the kernel's own W^ (K2's output, diagonal fl(1 / L_ii)):
|t^ - W^ k*_ref| <= gamma_{n+2} |W^||k*| + |W^||dk*|.  Either way, with dt the bound on t,
    |ss^ - ss_ref| <= sum (2 |t_i| dt_i + dt_i^2) + gamma_{n+4} sum t_i^2.
var = ((s2 + v) - ss) + 1e-10: three roundings, |dvar| <= |dss| + SLACK u (|s2 + v| + |s2 + v - ss| + |var|).

EI.  The reference is exact: EI = sign sd (u Phi(u) + phi(u)), sd = sqrt(var^), u = (best - mu^) / sd, evaluated in mpmath at
the kernel's own (best, mu^, var^).  The kernel's error, first order in u and multiplied by SLACK:
    sd: 1 rounding (IEEE sqrt);  u: (best - mu), / sd and sd's own -> eps_u = 3 u;
    phi: a = -u^2 / 2 rounded once (eps_a = 2 eps_u + u), exp with EXP_ULP ulp, the constant 1/sqrt(2 pi) as a double and the
         product: eps_phi = |a| eps_a + (2 EXP_ULP + 2) u;
    Phi: z = -u fl(1/sqrt 2) (eps_z = eps_u + 2 u), erfc with ERFC_ULP ulp and condition kappa(z) = 2 |z| / (sqrt(pi) erfcx(z)):
         eps_Phi = kappa eps_z + 2 ERFC_ULP u;
    g = fl(fl(u Phi) + phi): |dg| <= |u Phi| (eps_u + eps_Phi + u) + phi eps_phi + u |g|   (u Phi + phi cancels in the tail:
         the absolute terms keep the bound faithful there);
    EI = sign sd g: |dEI| <= sd |dg| + 2 u |EI|, plus an absolute 8 (1 + sd) 2^-1022 for results that underflow.
EXP_ULP = 1 and ERFC_ULP = 5 are the maximum ulp errors of CUDA's double-precision exp(x) and erfc(x) listed in the CUDA C++
Programming Guide, appendix "Mathematical Functions", double-precision table (CUDA 12.9); sqrt and / are IEEE-rounded there.
acq = EI / cost needs no bound: NumPy forms cost_fix + sum |x_k| in candidate_cost's order and the IEEE quotient, bit for bit.
A candidate whose reference var is within its own bound of 0 gets no EI check (the callers count them).
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

from oracle.prior_bounds import ETA, U, U_LD, _ratio, gamma

LD = np.longdouble
SLACK = 2.0
EXP_ULP = 1
ERFC_ULP = 5
K_DIAG = np.float64(1e-10) + np.float64(1e-8)      # csrc/surrogate.cuh kSurrogateDiag
VAR_NOISE = np.float64(1e-10)


def g2(k):
    """gamma_k of the kernel plus the reference's own gamma_k in longdouble."""
    return gamma(k) + gamma(k, U_LD)


def inv_l(l):
    return np.float64(1.0) / np.float64(l)


# --------------------------------------------------------------------------------------------------
# K2
# --------------------------------------------------------------------------------------------------
def jitter(tries, sv, s2):
    """The jitter K2 added on its successful attempt, bit for bit (0.0 when tries == 0)."""
    if tries <= 0:
        return np.float64(0.0)
    n = len(sv)
    diag = np.array([float(Fraction(float(a)) ** 2 + Fraction(float(s2))) for a in sv]) + K_DIAG
    t = np.float64(0.0)
    for a in diag:
        t = t + a
    j = (t / np.float64(n)) * np.float64(1e-6)
    for _ in range(tries - 1):
        j = j * np.float64(10.0)
    return j


def gram_ref(x_int, sv, s2, l, jit=0.0):
    """Ky_ref (n x n, longdouble) and E_gram (float64) of the module docstring."""
    X = np.asarray(x_int, np.float64)
    n, d = X.shape
    il = LD(inv_l(l))
    Dl = (X[:, None, :].astype(LD) - X[None, :, :].astype(LD)) * il
    r2 = np.einsum("ijk,ijk->ij", Dl, Dl)
    e = np.exp(-0.5 * r2)
    svl = np.asarray(sv, np.float64).astype(LD)
    K = LD(s2) * e + np.outer(svl, svl)
    dg = LD(np.float64(K_DIAG) + np.float64(jit))
    K[np.diag_indices(n)] += dg
    a = (LD(s2) * e).astype(np.float64)
    r2f = r2.astype(np.float64)
    Kabs = np.abs(K).astype(np.float64)
    E = SLACK * (a * (0.5 * gamma(d + 5) * r2f + (2 * EXP_ULP + 1) * U) + U * Kabs)
    E += g2(d + 10) * (a * (1.0 + r2f) + Kabs)                         # the reference's own rounding
    E += 4.0 * ETA * max(1.0, float(s2))                                # exp(-r2 / 2) in or below the subnormal range
    E[np.diag_indices(n)] += U * np.diag(Kabs)
    return K, E


def lower_inverse_ld(L):
    """L^-1 of the fp64 lower-triangular L in longdouble (row-wise substitution)."""
    Ll = np.tril(np.asarray(L, np.float64)).astype(LD)
    n = Ll.shape[0]
    X = np.zeros((n, n), LD)
    for i in range(n):
        s = -(Ll[i, :i] @ X[:i, :]) if i else np.zeros(n, LD)
        s[i] += 1
        X[i] = s / Ll[i, i]
    return X


def check_fit(L, alpha, x_int, y_int, sv, s2, l, tries, m_int=None, W=None):
    """Worst |error| / bound of K2's factor, alpha and (n <= 48) W against the Gram of the kernel's own inputs.  Returns
    dict(L=, alpha=, W=) ratios (<= 1 passes) and the bounds' size relative to the quantity (L_scale, alpha_scale)."""
    L = np.tril(np.asarray(L, np.float64))
    n = L.shape[0]
    Ky, E = gram_ref(x_int, sv, s2, l, jitter(tries, sv, s2))
    Ll, Lab = L.astype(LD), np.abs(L)
    LLt = Lab @ Lab.T
    res = np.abs(Ll @ Ll.T - Ky).astype(np.float64)
    bL = g2(n + 3) * LLt + E + 4.0 * (n + 4) * ETA                     # (products that underflow: 2^-1074 each)
    out = dict(L=float(np.tril(_ratio(res, bL)).max()), L_scale=float((bL / np.abs(Ky).astype(np.float64).max()).max()))
    y = np.asarray(y_int, np.float64)
    r = y.astype(LD) - (np.asarray(m_int, np.float64).astype(LD) if m_int is not None else 0)
    a = np.asarray(alpha, np.float64)
    ra = np.abs(Ky @ a.astype(LD) - r).astype(np.float64)
    ba = g2(3 * n + 4) * (LLt @ np.abs(a)) + E @ np.abs(a) + U * np.abs(r).astype(np.float64)
    ba += 4.0 * (3 * n + 4) * ETA * (1.0 + np.abs(a).max()) * (1.0 + Lab.max()) ** 2
    out["alpha"] = float(_ratio(ra, ba).max())
    out["alpha_scale"] = float(ba.max() / max((np.abs(Ky).astype(np.float64) @ np.abs(a)).max(), 1e-300))
    if W is not None:
        W = np.tril(np.asarray(W, np.float64))
        rw = np.abs(Ll @ W.astype(LD) - np.eye(n, dtype=LD)).astype(np.float64)
        bw = g2(n + 4) * (Lab @ np.abs(W)) + 4.0 * (n + 4) * ETA * (1.0 + np.abs(W).max()) * (1.0 + Lab.max()) ** 2
        out["W"] = float(np.tril(_ratio(rw, bw)).max())
    return out


# --------------------------------------------------------------------------------------------------
# K3 / K7: mu, var
# --------------------------------------------------------------------------------------------------
def kstar_ref(X, x_int, sv, svg, s2, l, separable):
    """k*_ref (g x n, longdouble) and its bound dk* (float64) for candidates X (g x d), in the direct or separable form."""
    X, XI = np.asarray(X, np.float64), np.asarray(x_int, np.float64)
    d = XI.shape[1]
    ilf = inv_l(l)
    il = LD(ilf)
    Q = (X[:, None, :].astype(LD) - XI[None, :, :].astype(LD)) * il        # g x n x d
    Q2 = Q * Q
    r2 = Q2.sum(-1)
    e = np.exp(-0.5 * r2)
    svl = np.asarray(sv, np.float64).astype(LD)
    svgl = np.asarray(svg, np.float64).astype(LD)
    ssv = np.abs(svgl[:, None] * svl[None, :]).astype(np.float64)
    k = LD(s2) * e + svgl[:, None] * svl[None, :]
    a = (LD(s2) * e).astype(np.float64)
    kab = np.abs(k).astype(np.float64)
    r2f = r2.astype(np.float64)
    if separable:
        lead = Q2[..., :d - 1].sum(-1).astype(np.float64)
        last = Q2[..., d - 1].astype(np.float64)
        dk = SLACK * (a * (0.5 * (gamma(d + 4) * lead + gamma(5) * last) + (4 * EXP_ULP + 2) * U) + U * ssv + U * kab)
    else:
        Qf = np.abs(Q).astype(np.float64)
        dq = SLACK * U * ((np.abs(X)[:, None, :] + np.abs(XI)[None, :, :]) * ilf + Qf)
        dr2 = (2.0 * Qf * dq + dq * dq).sum(-1) + gamma(d) * r2f
        dk = SLACK * (a * (0.5 * dr2 + (2 * EXP_ULP + 1) * U) + U * (ssv + kab))
    dk += g2(d + 10) * (a * (1.0 + r2f) + kab)                         # the reference's own rounding
    dk += 4.0 * ETA * max(1.0, float(s2))                               # exp(-r2 / 2) in or below the subnormal range
    return k, dk


def posterior_ref(X, m, v, st, path, separable=False, block=2048):
    """posterior_ref_block over blocks of `block` candidates (bounded memory); same result."""
    X = np.asarray(X, np.float64).reshape(len(m), -1)
    parts = [posterior_ref_block(X[a:a + block], np.asarray(m)[a:a + block], np.asarray(v)[a:a + block], st, path, separable)
             for a in range(0, len(m), block)]
    out = {k: np.concatenate([p[k] for p in parts]) for k in ("mu", "var", "e_mu", "e_var", "ss")}
    out["n"] = parts[0]["n"] if parts else 0
    return out


def posterior_ref_block(X, m, v, st, path, separable=False):
    """Reference mu, var (longdouble) and their bounds (float64) at candidates X with prior m, v (zeros for a non-causal set).
    st: dict(x_int, sv, alpha, L, W (path 'mma'), s2, l) as fetched; path: 'subst' (forward substitution) or 'mma' (t = W k*).
    Also returns ss_ref (the quantity var cancels against) for the informativeness report."""
    m, v = np.asarray(m, np.float64), np.asarray(v, np.float64)
    svg = np.sqrt(v)
    k, dk = kstar_ref(X, st["x_int"], st["sv"], svg, st["s2"], st["l"], separable)
    n = k.shape[1]
    al = np.asarray(st["alpha"], np.float64)
    kab = np.abs(k).astype(np.float64)
    mu = m.astype(LD) + k @ al.astype(LD)
    e_mu = g2(n + 2) * (np.abs(m) + kab @ np.abs(al)) + dk @ np.abs(al)
    if path == "mma":
        W = np.tril(np.asarray(st["W"], np.float64))
        t = k @ W.T.astype(LD)
        Wab = np.abs(W)
        dt = g2(n + 2) * (kab @ Wab.T) + (dk + 4.0 * (n + 4) * ETA) @ Wab.T
    else:
        L = np.tril(np.asarray(st["L"], np.float64))
        Li = st.get("Linv_ld")
        if Li is None:
            Li = st["Linv_ld"] = lower_inverse_ld(L)
        t = k @ Li.T
        tab = np.abs(t).astype(np.float64)
        dt = (g2(n + 3) * (tab @ np.abs(L).T) * SLACK + dk + 4.0 * (n + 4) * ETA) @ np.abs(Li).astype(np.float64).T
    tab = np.abs(t).astype(np.float64)
    ss = (t * t).sum(-1)
    e_ss = (2.0 * tab * dt + dt * dt).sum(-1) + g2(n + 4) * ss.astype(np.float64)
    a = np.float64(st["s2"]) + v                                        # fl(s2 + v): a kernel rounding, bounded below
    base = LD(st["s2"]) + v.astype(LD)
    var = (base - ss) + LD(VAR_NOISE)
    e_var = e_ss + SLACK * U * (np.abs(a) + np.abs(base - ss).astype(np.float64) + np.abs(var).astype(np.float64))
    return dict(mu=mu, var=var, e_mu=e_mu, e_var=e_var, ss=ss.astype(np.float64), n=n)


def check_posterior(mu, var, ref):
    """Worst |error| / bound of the kernel's mu, var against posterior_ref (NaN counts as infinitely wrong)."""
    em = np.abs(np.asarray(mu, np.float64).astype(LD) - ref["mu"]).astype(np.float64)
    ev = np.abs(np.asarray(var, np.float64).astype(LD) - ref["var"]).astype(np.float64)
    return float(_ratio(em, ref["e_mu"]).max(initial=0.0)), float(_ratio(ev, ref["e_var"]).max(initial=0.0))


# --------------------------------------------------------------------------------------------------
# EI, acq
# --------------------------------------------------------------------------------------------------
def ei_bound(best, mu, var, task_sign):
    """Bound on |EI^ - EI(best, mu, var)| of the kernel's expected_improvement at its own (mu, var) (module docstring)."""
    from scipy.special import erfc, erfcx, ndtr
    mu, var = np.asarray(mu, np.float64), np.asarray(var, np.float64)
    with np.errstate(all="ignore"):
        sd = np.sqrt(var)
        u = (best - mu) / sd
        phi = np.exp(-0.5 * u * u) / np.sqrt(2.0 * np.pi)
        z = -u / np.sqrt(2.0)
        Phi = ndtr(u)
        zp = np.maximum(z, 0.0)
        kappa = np.where(z >= 0, 2.0 * zp / (np.sqrt(np.pi) * erfcx(zp)),
                         2.0 * np.abs(z) * np.exp(-z * z) / (np.sqrt(np.pi) * erfc(np.minimum(z, 0.0))))
        eps_u = 3.0 * U
        eps_phi = 0.5 * u * u * (2.0 * eps_u + U) + (2 * EXP_ULP + 2) * U
        eps_Phi = kappa * (eps_u + 2.0 * U) + 2 * ERFC_ULP * U
        g = u * Phi + phi
        dg = np.abs(u * Phi) * (eps_u + eps_Phi + U) + phi * eps_phi + U * np.abs(g)
        # (+ an absolute floor for results in or below the subnormal range: phi, Phi and EI underflow far in the tail)
        return SLACK * (sd * dg + 2.0 * U * sd * np.abs(g)) + 8.0 * 2.0 ** -1022 * (1.0 + sd)


def ei_exact(best, mu, var, task_sign, dps=40):
    """EI = sign sd (u Phi(u) + phi(u)) at each (mu, var) in mpmath (mpf list)."""
    import mpmath as mp
    mp.mp.dps = dps
    out = []
    b = mp.mpf(float(best))
    for m_, v_ in zip(np.asarray(mu, np.float64), np.asarray(var, np.float64)):
        sd = mp.sqrt(mp.mpf(float(v_)))
        u = (b - mp.mpf(float(m_))) / sd
        g = u * mp.erfc(-u / mp.sqrt(2)) / 2 + mp.exp(-u * u / 2) / mp.sqrt(2 * mp.pi)
        out.append(task_sign * sd * g)
    return out


def check_ei(ei, best, mu, var, task_sign, idx):
    """Worst |EI^ - EI_exact| / bound over the candidates idx (kernel's own mu, var)."""
    import mpmath as mp
    idx = np.asarray(idx, np.int64)
    if idx.size == 0:
        return 0.0
    ex = ei_exact(best, mu[idx], var[idx], task_sign)
    b = ei_bound(best, mu[idx], var[idx], task_sign)
    e = np.array([float(abs(mp.mpf(float(a)) - r)) if np.isfinite(a) else np.inf for a, r in zip(ei[idx], ex)])
    return float(_ratio(e, b).max())


def candidate_cost(X, cost_fix, cost_variable):
    """csrc/surrogate.cuh candidate_cost in its order: cost_fix, then + |x_k| for k = 0 .. d - 1."""
    X = np.asarray(X, np.float64)
    c = np.full(X.shape[0], np.float64(cost_fix))
    if cost_variable:
        for k in range(X.shape[1]):
            c = c + np.abs(X[:, k])
    return c


def first_argmax(acq):
    """(value, index, n_nan) by the kernels' rule: np.argmax with NaN as -inf; index -1 when nothing is finite-or-inf."""
    a = np.asarray(acq, np.float64)
    nn = int(np.isnan(a).sum())
    if nn == a.size:
        return -np.inf, -1, nn
    w = np.where(np.isnan(a), -np.inf, a)
    i = int(np.argmax(w))
    return float(w[i]), i, nn
