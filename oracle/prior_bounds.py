"""Reference values and proven error bounds for the causal-prior kernels.

    K1b (csrc/prior_eval.cu) and K1p (csrc/prior_pair.cu): m(x) = u.w and v(x) = (s2 + noise) - u^T M u in plain fp64,
        in whatever order the work decomposition adds things up (DMMA, folded column blocks, segment partials added by
        prior_finalize_kernel, the pair regrouping);
    K1c (csrc/prior_rows.cu): m_int, v_int at the interventional rows in compensated (Dot2) arithmetic.

The builders take the kernels' own inputs as fetched from the device (the tab{k} or u_int tables, M, w, s2, noise), so a
check covers one kernel and none of the rounding of the stages that produced its inputs.  u = 2^-53 throughout.

Bound A (K1b / K1p).  For a sum of products evaluated with n roundings on any path from an exact product to the result,
in ANY order of IEEE operations, |computed - exact| <= gamma_n * sum |terms|, gamma_n = n u / (1 - n u) (Higham,
Accuracy and Stability of Numerical Algorithms, Lemma 3.1 applied to each term's path).  A term of q = u^T M u is
u_j M_jk u_k, with u_j formed from d table entries:
    n_q = N^2 + 2 d + 2:  2 (d - 1) roundings forming u_j and u_k from the tables, 2 multiplications (FMA or DMMA products
                          count as one rounding with the following addition, which only lowers the count), and at most
                          N^2 - 1 additions, the depth bound of any summation tree over at most N^2 nonzero products (the
                          kernels visit M's lower block triangle and double it exactly, the pair path sums N (N + 1) / 2
                          pair products); the last 3 are slack.
    n_m = N + d:          d - 1 roundings forming u_j, 1 multiplication by w_j, at most N - 1 additions.
    v:                    the kernels compute fl(fl(s2 + noise) - q); the reference applies the same fl(s2 + noise) and
                          the subtraction costs one more rounding: e_v = e_q + u (|v_ref| + e_q).
The reference itself is evaluated in np.longdouble (u_ld = eps(longdouble) / 2, 2^-64 on x86) with the same n, so its
own gamma_n(u_ld) sum|terms| is added; on a platform whose longdouble is fp64 the bound simply doubles.

Bound C (K1c).  Every product is split exactly (TwoProd) and every sum carries its rounding error (TwoSum), so the only
losses are (i) the fp64 additions that accumulate the captured errors in the low words and (ii) the final rounding.  There
are fewer than n_e = 2 N^2 + 4 N + 256 captured errors (one TwoProd and one TwoSum per term, plus the reductions over
rows, warps and partials), each at most u (1 + gamma) sum|terms|, and the low words add them with chains no longer than
n_e.  Following the Dot2 analysis of Ogita, Rump and Oishi ("Accurate sum and dot product", SISC 2005):
    |v_gpu - v_ref| <= 3 u |v_ref| + 2 (n_e u)^2 sum|terms| + 8 N^2 2^-1074 max(1, |M|_max),
where 3 u |v_ref| covers the kernel's ((a - q_hi) - q_lo) (two roundings; a - q_hi is exact under cancellation by
Sterbenz's lemma, otherwise its error is u (|v| + |q_lo|)) and the reference's own correct rounding.  The last term is
underflow: a TwoProd whose error term falls below 2^-1074 is no longer exact, and each of the N^2 terms can lose at most
an absolute 2^-1074 times the remaining factors (all u_j <= 1) in the kernel and in the reference.  m_int likewise with
n_m = 2 N + 256 and one final rounding (m_hi + m_lo).

The exact K1c reference splits each term u_n M_nk u_k into four doubles with Dekker's TwoProd (Veltkamp splitting, no FMA
needed, vectorised in NumPy) and sums them with math.fsum, which is correctly rounded.
"""
from __future__ import annotations

import math

import numpy as np

U = 2.0 ** -53
U_LD = float(np.finfo(np.longdouble).eps) / 2.0
ETA = 2.0 ** -1074          # smallest subnormal


def gamma(n, u=U):
    nu = float(n) * u
    if nu >= 1.0:
        raise ValueError(f"gamma_{n} is undefined for u = {u}")
    return nu / (1.0 - nu)


# --------------------------------------------------------------------------------------------------
# Bound A: K1b / K1p
# --------------------------------------------------------------------------------------------------
def grid_u(tabs, rows):
    """u (len(rows), N) in np.longdouble for flat C-order indices `rows` of the tensor grid whose per-dimension tables
    (p_k, N) are `tabs` (one table of explicit points: its rows)."""
    p = [t.shape[0] for t in tabs]
    idx = np.unravel_index(np.asarray(rows, np.int64), p)
    u = tabs[0][idx[0]].astype(np.longdouble)
    for k in range(1, len(tabs)):
        u = u * tabs[k][idx[k]].astype(np.longdouble)
    return u


def prior_ref(u, M, w, s2, noise, d):
    """Reference m, v (np.longdouble) of the candidates whose u rows (np.longdouble, from grid_u) are given, with the
    sums of |terms| that scale bound A.  d: tables multiplied into each u_j (1 for explicit points)."""
    u = np.asarray(u, np.longdouble)
    Ml, wl = np.asarray(M, np.float64).astype(np.longdouble), np.asarray(w, np.float64).astype(np.longdouble)
    q = np.einsum("gj,gj->g", u @ Ml, u)
    a = np.float64(s2) + np.float64(noise)            # the kernels' fl(s2 + noise)
    ua = np.abs(u).astype(np.float64)
    return dict(m=u @ wl, v=np.longdouble(a) - q, q_abs=np.einsum("gj,gj->g", ua @ np.abs(M), ua), m_abs=ua @ np.abs(w),
                N=int(u.shape[1]), d=int(d), Mmax=float(np.abs(M).max(initial=0.0)), wmax=float(np.abs(w).max(initial=0.0)))


def prior_bounds(ref):
    """Bound A (module docstring) for every candidate of `ref`: dict(m=..., v=...) as float64 arrays."""
    N, d = ref["N"], ref["d"]
    nq, nm = N * N + 2 * d + 2, N + d
    uf_q = 4.0 * N * N * ETA * max(1.0, ref["Mmax"])
    uf_m = 4.0 * N * ETA * max(1.0, ref["wmax"])
    e_q = (gamma(nq) + gamma(nq, U_LD)) * ref["q_abs"] + uf_q
    e_m = (gamma(nm) + gamma(nm, U_LD)) * ref["m_abs"] + uf_m
    e_v = e_q + U * (np.abs(ref["v"]).astype(np.float64) + e_q)
    return dict(m=e_m, v=e_v)


def _ratio(err, bound):
    err, bound = np.asarray(err, np.float64), np.asarray(bound, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
    return np.where(np.isnan(err), np.inf, r)


def check_prior(m, v, ref):
    """Worst |error| / bound A of computed m, v against `ref` (a NaN counts as infinitely wrong).  <= 1 passes."""
    b = prior_bounds(ref)
    em = np.abs(np.asarray(m, np.float64).astype(np.longdouble) - ref["m"]).astype(np.float64)
    ev = np.abs(np.asarray(v, np.float64).astype(np.longdouble) - ref["v"]).astype(np.float64)
    return float(_ratio(em, b["m"]).max(initial=0.0)), float(_ratio(ev, b["v"]).max(initial=0.0))


# --------------------------------------------------------------------------------------------------
# Bound C: K1c (exact reference)
# --------------------------------------------------------------------------------------------------
_SPLIT = 134217729.0        # 2^27 + 1


def _split(a):
    c = _SPLIT * a
    hi = c - (c - a)
    return hi, a - hi


def two_prod(a, b):
    """Dekker's TwoProd without FMA: p + e == a * b exactly (barring underflow and overflow), elementwise."""
    a, b = np.broadcast_arrays(np.asarray(a, np.float64), np.asarray(b, np.float64))
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    e = al * bl - (((p - ah * bh) - al * bh) - ah * bl)
    return p, e


def rows_ref(u_int, M, w, s2, noise):
    """Exact-then-correctly-rounded m_int, v_int for the rows of u_int (R, N), with the sums of |terms| of bound C.
    v_ref = round((fl(s2 + noise)) - sum_nk u_n M_nk u_k), m_ref = round(sum_n u_n w_n)."""
    u_int = np.asarray(u_int, np.float64)
    M, w = np.asarray(M, np.float64), np.asarray(w, np.float64)
    a = np.float64(s2) + np.float64(noise)
    R, N = u_int.shape
    m, v, q_abs, m_abs = (np.empty(R) for _ in range(4))
    for r in range(R):
        x = u_int[r]
        p1, e1 = two_prod(x[:, None], M)                 # u_n M_nk = p1 + e1
        h1, l1 = two_prod(p1, x[None, :])                # (p1 + e1) u_k = h1 + l1 + h2 + l2
        h2, l2 = two_prod(e1, x[None, :])
        neg = np.concatenate([h1.ravel(), l1.ravel(), h2.ravel(), l2.ravel()])
        np.negative(neg, out=neg)
        v[r] = math.fsum(np.concatenate([[a], neg]))
        q_abs[r] = float(np.abs(x) @ np.abs(M) @ np.abs(x))
        ph, pl = two_prod(x, w)
        m[r] = math.fsum(np.concatenate([ph, pl]))
        m_abs[r] = float(np.abs(x) @ np.abs(w))
    return dict(m=m, v=v, q_abs=q_abs, m_abs=m_abs, N=N, Mmax=float(np.abs(M).max(initial=0.0)),
                wmax=float(np.abs(w).max(initial=0.0)))


def rows_bounds(ref):
    """Bound C (module docstring): dict(m=..., v=...)."""
    N = ref["N"]
    ne, nm = 2 * N * N + 4 * N + 256, 2 * N + 256
    e_v = 3.0 * U * np.abs(ref["v"]) + 2.0 * (ne * U) ** 2 * ref["q_abs"] + 8.0 * N * N * ETA * max(1.0, ref["Mmax"])
    e_m = 2.0 * U * np.abs(ref["m"]) + 2.0 * (nm * U) ** 2 * ref["m_abs"] + 8.0 * N * ETA * max(1.0, ref["wmax"])
    return dict(m=e_m, v=e_v)


def check_rows(m_int, v_int, ref):
    """Worst |error| / bound C of computed m_int, v_int (a NaN counts as infinitely wrong).  <= 1 passes."""
    b = rows_bounds(ref)
    em = np.abs(np.asarray(m_int, np.float64) - ref["m"])
    ev = np.abs(np.asarray(v_int, np.float64) - ref["v"])
    return float(_ratio(em, b["m"]).max(initial=0.0)), float(_ratio(ev, b["v"]).max(initial=0.0))


def cancellation(ref):
    """sum |u_j M_jk u_k| / |v| per row: how much of the quadratic form cancels (the factor a plain fp64 evaluation
    loses)."""
    return np.asarray(ref["q_abs"], np.float64) / np.maximum(np.abs(np.asarray(ref["v"], np.float64)), 1e-300)
