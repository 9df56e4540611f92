"""The checkers of oracle/posterior_bounds.py are sharp: NumPy emulations of the surrogate kernels in their own order of
operations pass them, and each fault a wrong block, fragment, staging or formula would cause fails them.  CPU only.

Emulated: K2's right-looking Cholesky with the scaled column, its substitutions and its 4-lane L^-1; the sweep's
four-partial forward substitution by the staged reciprocal diagonal; W k* in k4 steps of 8-row blocks (sweep_mma_kernel);
the separable k* tables; K7's column-oriented substitution.  Every fault is also judged by the parity rule the oracle tests
apply (helpers.sweep_errors floors, the normwise backward error of L, |W L - I| <= 1e-9 cond(L)); test_current_rule prints
which faults that rule lets through."""
import numpy as np
import pytest
from scipy.special import erf, erfc

from helpers import BACKWARD_TOL
from oracle import posterior_bounds as P

TILE = 1024


# ---- a set's inputs ---------------------------------------------------------------------------------------------------
def _state(n, d, seed, s2=1.0, l=1.0, causal=True, spread=1.1):
    """x_int on a jittered lattice of spacing ~ spread l (a fit whose bounds stay informative), y, m_int, v_int."""
    rng = np.random.default_rng(seed)
    side = int(np.ceil(n ** (1.0 / d)))
    pts = np.stack(np.meshgrid(*[np.arange(side)] * d, indexing="ij"), -1).reshape(-1, d)[:n].astype(float)
    X = (pts - (side - 1) / 2.0) * spread * l + rng.uniform(-0.15, 0.15, (n, d)) * l
    y = np.sin(X.sum(1)) + 0.1 * rng.standard_normal(n)
    m_int = 0.2 * np.cos(X[:, 0]) if causal else None
    v_int = rng.uniform(0.05, 0.4, n) if causal else np.zeros(n)
    return dict(x_int=X, y=y, m_int=m_int, sv=np.sqrt(v_int), s2=s2, l=l, d=d, n=n, causal=causal)


def _gram(st, jit=0.0):
    """K2's Gram in its order: differences, * il, squares summed, s2 exp, + sv sv, + (kSurrogateDiag + jitter)."""
    X, il = st["x_int"], P.inv_l(st["l"])
    r2 = np.zeros((st["n"], st["n"]))
    for k in range(st["d"]):
        t = (X[:, None, k] - X[None, :, k]) * il
        r2 = r2 + t * t
    K = np.outer(st["sv"], st["sv"]) + st["s2"] * np.exp(-0.5 * r2)
    K[np.diag_indices(st["n"])] += P.K_DIAG + jit
    return K


def _cholesky(A, drop=None):
    """surrogate_jitchol's arithmetic: piv, sq = sqrt(piv), inv = 1 / sq, column *= inv, trailing -= l_ij l_kj.
    drop = (i, k, j): that one trailing-update product is skipped."""
    A = np.tril(A.copy())
    n = A.shape[0]
    for j in range(n):
        sq = np.sqrt(A[j, j])
        inv = 1.0 / sq
        A[j, j] = sq
        A[j + 1:, j] *= inv
        c = A[j + 1:, j]
        upd = np.tril(np.outer(c, c))
        if drop is not None and drop[2] == j:
            upd[drop[0] - j - 1, drop[1] - j - 1] = 0.0
        A[j + 1:, j + 1:] -= upd
    return np.tril(A)


def _solve_lower(L, b):
    z = b.copy()
    for j in range(len(z)):
        z[j] = z[j] / L[j, j]
        z[j + 1:] -= L[j + 1:, j] * z[j]
    return z


def _lower_inverse(L):
    """surrogate_lower_inverse: W_cc = 1 / L_cc, W_ic = -(four partial dot products, butterfly) * (1 / L_ii)."""
    n = L.shape[0]
    rinv = 1.0 / np.diag(L)
    W = np.diag(rinv)
    for c in range(n):
        for i in range(c + 1, n):
            a = np.zeros(4)
            for j in range(c + 1, i):
                a[(j - c - 1) % 4] += L[i, j] * W[j, c]
            a[0] += L[i, c] * rinv[c]
            W[i, c] = -(((a[0] + a[1]) + (a[2] + a[3])) * rinv[i])
    return W


def _fit(st, drop=None):
    K = _gram(st)
    L = _cholesky(K, drop)
    r = st["y"] - st["m_int"] if st["causal"] else st["y"].copy()
    alpha = _solve_lower(L.T[::-1, ::-1], _solve_lower(L, r)[::-1])[::-1]
    W = _lower_inverse(L) if st["n"] <= 48 else None
    return L, alpha, W


# ---- candidates, k*, the sweep's solves -------------------------------------------------------------------------------
def _grid(st, p_last, rows, seed):
    """A tensor grid of `rows` leading rows x p_last: the candidates, their flat (row, j) and a prior m, v."""
    d, rng = st["d"], np.random.default_rng(seed)
    span = np.abs(st["x_int"]).max() + 0.5 * st["l"]
    last = np.linspace(-span, span, p_last)
    if d == 1:
        X = last[:, None]
        row = np.zeros(p_last, int)
    else:
        lead = rng.uniform(-span, span, (rows, d - 1))
        X = np.hstack([np.repeat(lead, p_last, 0), np.tile(last, rows)[:, None]])
        row = np.repeat(np.arange(rows), p_last)
    g = X.shape[0]
    v = rng.uniform(0.05, 0.5, g) if st["causal"] else np.zeros(g)
    m = 0.3 * np.sin(X[:, 0]) if st["causal"] else np.zeros(g)
    return X, row, m, v


def _kstar_direct(st, X, svg, lost_sv=None):
    il = P.inv_l(st["l"])
    xs = st["x_int"] * il
    xl = X * il
    r2 = np.zeros((X.shape[0], st["n"]))
    for k in range(st["d"]):
        q = xl[:, None, k] - xs[None, :, k]
        r2 = r2 + q * q
    sv = np.outer(svg, st["sv"])
    if lost_sv is not None:
        sv[:, lost_sv] = 0.0
    return sv + st["s2"] * np.exp(-0.5 * r2)


def _kstar_separable(st, X, row, svg, lead_shift=None):
    """eLead[row] * eLast[j] + sv svg.  lead_shift = (first candidate, count): those candidates read the next row's eLead
    (a lead-row table indexed one row off from where an item starts)."""
    il, d = P.inv_l(st["l"]), st["d"]
    XI = st["x_int"]
    q = (X[:, None, d - 1] - XI[None, :, d - 1]) * il
    eLast = np.exp(-0.5 * (q * q))
    r2 = np.zeros_like(eLast)
    for k in range(d - 2, -1, -1):
        t = (X[:, None, k] - XI[None, :, k]) * il
        r2 = r2 + t * t
    eLead = st["s2"] * np.exp(-0.5 * r2)
    if lead_shift is not None:
        a, c = lead_shift
        nxt = np.searchsorted(row, row[a] + 1)
        eLead[a:a + c] = eLead[nxt]
    return eLead * eLast + np.outer(svg, st["sv"])


def _subst_four(L, K, recip_off=None):
    """posterior_at / posterior_sep: t_i = ((a0 + a1) + (a2 + a3)) * Li[i], Li[i] = 1 / L_ii staged (recip_off: that row's
    diagonal staged as L_ii itself)."""
    n = L.shape[0]
    Li = 1.0 / np.diag(L)
    if recip_off is not None:
        Li[recip_off] = L[recip_off, recip_off]
    T = np.zeros_like(K)
    for i in range(n):
        a = [K[:, i].copy(), 0.0, 0.0, 0.0]
        for j in range(i):
            a[j & 3] = a[j & 3] - L[i, j] * T[:, j]
        T[:, i] = ((a[0] + a[1]) + (a[2] + a[3])) * Li[i]
    return T


def _subst_column(L, K):
    """K7: column-oriented forward substitution by division."""
    R = K.copy()
    for j in range(L.shape[0]):
        R[:, j] = R[:, j] / L[j, j]
        R[:, j + 1:] -= np.outer(R[:, j], L[j + 1:, j])
    return R


def _mma(W, K, skip_last_k4=False, drop_block=None):
    """sweep_mma_kernel: t = W k* as 8 x 4 blocks of W's block lower triangle, k4 step outermost, each DMMA one rounding of
    (accumulator + four products).  skip_last_k4: the last k4 step of the last 8-row block is not issued; drop_block =
    (ib, ks): that B fragment is missing."""
    n = W.shape[0]
    nb, ksn = (n + 7) // 8, (n + 3) // 4
    Wp = np.zeros((8 * nb, 4 * ksn))
    Wp[:n, :n] = np.tril(W)
    Kp = np.zeros((K.shape[0], 4 * ksn))
    Kp[:, :n] = K
    T = np.zeros((K.shape[0], 8 * nb))
    for ks in range(ksn):
        for ib in range(ks >> 1, nb):
            if skip_last_k4 and ib == nb - 1 and ks == ksn - 1:
                continue
            if drop_block == (ib, ks):
                continue
            T[:, 8 * ib:8 * ib + 8] += Kp[:, 4 * ks:4 * ks + 4] @ Wp[8 * ib:8 * ib + 8, 4 * ks:4 * ks + 4].T
    return T[:, :n]


def _finish(st, T, K, alpha, m, v):
    mu = K @ alpha + m
    ss = np.einsum("gi,gi->g", T, T)
    var = ((st["s2"] + v) - ss) + 1e-10
    return mu, var


def _ref(st, X, m, v, L, alpha, W, path, separable):
    s = dict(x_int=st["x_int"], sv=st["sv"], alpha=alpha, L=L, W=W, s2=st["s2"], l=st["l"])
    return P.posterior_ref(X, m, v, s, path, separable)


# ---- the parity rule of the oracle tests (helpers.sweep_errors / test_parity_gpu._check_set) -------------------------
def _rule_posterior(mu, var, ref, v):
    mr, vr = ref["mu"].astype(np.float64), ref["var"].astype(np.float64)
    e_mu = np.abs(mu - mr) / np.maximum(np.abs(mr), max(1e-4, 1e-3 * np.abs(mr).max()))
    e_var = np.abs(var - vr) / np.maximum(np.abs(vr), 1e-4 * (1.0 + v))
    return max(e_mu.max(), e_var.max()) <= 1e-6


def _rule_fit(L, Ky):
    return np.abs(L @ L.T - Ky).max() / np.abs(Ky).max() <= BACKWARD_TOL


def _rule_inverse(L, W):
    return np.abs(W @ L - np.eye(L.shape[0])).max() <= 1e-9 * np.linalg.cond(L)


CURRENT_RULE = {}


# ---- K2 ------------------------------------------------------------------------------------------------------------------
K2_CASES = [(1, 1, 1), (17, 2, 2), (33, 2, 3), (48, 3, 4), (64, 2, 5), (96, 2, 8), (128, 4, 6)]   # (96 at l = 0.3: Gram entries underflow)


@pytest.mark.parametrize("n,d,seed", K2_CASES, ids=[f"n{c[0]}_d{c[1]}" for c in K2_CASES])
@pytest.mark.parametrize("hyper", [(1.0, 1.0), (50.0, 0.3)], ids=["unit", "s2_50_l0.3"])
def test_fit_checker_accepts_k2_order(n, d, seed, hyper):
    st = _state(n, d, seed, s2=hyper[0], l=hyper[1])
    L, alpha, W = _fit(st)
    r = P.check_fit(L, alpha, st["x_int"], st["y"], st["sv"], st["s2"], st["l"], 0, st["m_int"], W)
    print(f"K2 n={n} d={d} hyper={hyper}: {r}")
    assert r["L"] <= 1.0 and r["alpha"] <= 1.0 and r.get("W", 0.0) <= 1.0
    assert r["L_scale"] <= 1e-8


def test_fit_checker_rejects_a_missing_trailing_product():
    st = _state(33, 2, 3)
    K = _gram(st)
    L0 = _cholesky(K)
    j = 5
    col = np.abs(L0[j + 1:, j])
    i = j + 1 + int(np.argmax(col))
    L, alpha, W = _fit(st, drop=(i, j + 1, j))
    r = P.check_fit(L, alpha, st["x_int"], st["y"], st["sv"], st["s2"], st["l"], 0, st["m_int"], W)
    print(f"K2 fault missing trailing product: {r}")
    assert r["L"] > 1.0
    CURRENT_RULE["cholesky: one trailing-update product missing"] = _rule_fit(L, K)


def test_fit_checker_rejects_an_inverse_entry_off_by_1e3_ulp():
    st = _state(48, 3, 4)
    L, alpha, W = _fit(st)
    W2 = W.copy()
    W2[47, 46] += 1e3 * np.spacing(W2[47, 46])
    r = P.check_fit(L, alpha, st["x_int"], st["y"], st["sv"], st["s2"], st["l"], 0, st["m_int"], W2)
    print(f"K2 fault L^-T entry + 1e3 ulp: W {r['W']:.2e}")
    assert r["W"] > 1.0
    CURRENT_RULE["L^-T: one entry off by 1e3 ulp"] = _rule_inverse(L, W2)


def test_jitter_is_reproduced_bit_for_bit():
    """Two identical rows at s2 = 2^40 make the first attempt meet a zero pivot exactly; the retry's jitter follows the
    kernel's order (sequential sum of fl(fma(sv, sv, s2) + kSurrogateDiag), / n, * 1e-6)."""
    st = _state(6, 1, 7, s2=2.0 ** 40, causal=False)
    st["x_int"][1] = st["x_int"][0]
    st["x_int"] *= 8.0
    with np.errstate(invalid="ignore", divide="ignore"):
        assert np.isnan(_cholesky(_gram(st))).any()
    jit = P.jitter(1, st["sv"], st["s2"])
    diag = np.full(6, 2.0 ** 40) + P.K_DIAG
    assert jit == (np.sum(diag) / 6) * 1e-6 and P.jitter(3, st["sv"], st["s2"]) == jit * 10.0 * 10.0
    L = _cholesky(_gram(st, jit))
    r = P.check_fit(L, _solve_lower(L.T[::-1, ::-1], _solve_lower(L, st["y"])[::-1])[::-1], st["x_int"], st["y"], st["sv"],
                    st["s2"], st["l"], 1, None, _lower_inverse(L))
    assert r["L"] <= 1.0 and r["alpha"] <= 1.0 and r["W"] <= 1.0, r
    r_wrong = P.check_fit(L, np.zeros(6), st["x_int"], st["y"], st["sv"], st["s2"], st["l"], 2, None)
    assert r_wrong["L"] > 1.0, "a wrong retry count must show in the factor"


# ---- K3 / K7 --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sep_sets():
    """n = 17, 25, 33, 48 (d = 2, causal) and n = 16 (FMA path): fit, separable grid of 3 items."""
    out = {}
    for n, seed in ((16, 21), (17, 22), (25, 23), (33, 24), (48, 25)):
        st = _state(n, 2, seed)
        L, alpha, W = _fit(st)
        X, row, m, v = _grid(st, 100, 31, seed)
        out[n] = (st, L, alpha, W, X, row, m, v)
    return out


def _sweep(sep, n, path, fault=None):
    st, L, alpha, W, X, row, m, v = sep[n]
    svg = np.sqrt(v)
    lost = None
    if fault == "lost_sv":
        lost = n // 2
    if fault == "lead_row":
        K = _kstar_separable(st, X, row, svg, lead_shift=(TILE, 100 - TILE % 100))   # item 1 starts mid-row
    else:
        K = _kstar_separable(st, X, row, svg)
        if lost is not None:
            K[:, lost] -= svg * st["sv"][lost]
    if path == "mma":
        T = _mma(W, K, skip_last_k4=fault == "skip_k4", drop_block=(1, 0) if fault == "drop_block" else None)
    else:
        T = _subst_four(L, K, recip_off=int(np.argmin(np.diag(L))) if fault == "recip" else None)
    mu, var = _finish(st, T, K, alpha, m, v)
    ref = _ref(st, X, m, v, L, alpha, W, path, True)
    return mu, var, ref, v


@pytest.mark.parametrize("n,path", [(16, "subst"), (17, "mma"), (25, "mma"), (33, "mma"), (48, "mma"), (48, "subst")])
def test_posterior_checker_accepts_sweep_order(sep_sets, n, path):
    mu, var, ref, _ = _sweep(sep_sets, n, path)
    rm, rv = P.check_posterior(mu, var, ref)
    scale = max((ref["e_var"] / (1.0 + ref["ss"])).max(), (ref["e_mu"] / np.abs(ref["mu"].astype(float)).max()).max())
    print(f"sweep n={n} {path}: mu {rm:.2e} var {rv:.2e} of bound, bound / scale {scale:.1e}")
    assert rm <= 1.0 and rv <= 1.0
    assert scale <= 1e-8


FAULTS = [("skip_k4", 17, "mma"), ("skip_k4", 25, "mma"), ("skip_k4", 33, "mma"), ("drop_block", 33, "mma"),
          ("drop_block", 48, "mma"), ("recip", 16, "subst"), ("recip", 48, "subst"), ("lost_sv", 17, "mma"),
          ("lost_sv", 16, "subst"), ("lead_row", 33, "mma"), ("lead_row", 16, "subst")]


@pytest.mark.parametrize("fault,n,path", FAULTS, ids=[f"{f}_n{n}" for f, n, _ in FAULTS])
def test_posterior_checker_rejects_faults(sep_sets, fault, n, path):
    mu, var, ref, v = _sweep(sep_sets, n, path, fault)
    rm, rv = P.check_posterior(mu, var, ref)
    print(f"sweep fault {fault} n={n} {path}: mu {rm:.2e} var {rv:.2e} of bound")
    assert max(rm, rv) > 1.0
    CURRENT_RULE[f"sweep: {fault} (n = {n}, {path})"] = _rule_posterior(mu, var, ref, v)


@pytest.mark.parametrize("n,d", [(1, 1), (33, 2), (128, 4)])
def test_points_checker_accepts_direct_form_and_column_substitution(n, d):
    """Explicit points through the direct k* (x il - x_int il) with the sweep's substitution and K7's."""
    st = _state(n, d, 40 + n)
    L, alpha, W = _fit(st)
    rng = np.random.default_rng(n)
    span = np.abs(st["x_int"]).max() + 0.5
    X = rng.uniform(-span, span, (293, d))
    X[:3] = st["x_int"][:3] if n >= 3 else X[:3]
    m, v = 0.3 * np.sin(X[:, 0]), rng.uniform(0.05, 0.5, 293)
    K = _kstar_direct(st, X, np.sqrt(v))
    for name, T in (("four-partial", _subst_four(L, K)), ("column", _subst_column(L, K))):
        mu, var = _finish(st, T, K, alpha, m, v)
        rm, rv = P.check_posterior(mu, var, _ref(st, X, m, v, L, alpha, W, "subst", False))
        print(f"points n={n} d={d} {name}: mu {rm:.2e} var {rv:.2e}")
        assert rm <= 1.0 and rv <= 1.0
    if W is not None and n > 16:
        mu, var = _finish(st, _mma(W, K), K, alpha, m, v)
        rm, rv = P.check_posterior(mu, var, _ref(st, X, m, v, L, alpha, W, "mma", False))
        assert rm <= 1.0 and rv <= 1.0


def test_points_checker_rejects_a_lost_sv_term():
    st = _state(33, 2, 73)
    L, alpha, W = _fit(st)
    X = np.random.default_rng(3).uniform(-4, 4, (200, 2))
    m, v = np.zeros(200), np.full(200, 0.3)
    K = _kstar_direct(st, X, np.sqrt(v), lost_sv=7)
    mu, var = _finish(st, _subst_column(L, K), K, alpha, m, v)
    rm, rv = P.check_posterior(mu, var, _ref(st, X, m, v, L, alpha, W, "subst", False))
    assert max(rm, rv) > 1.0


# ---- EI, acq ---------------------------------------------------------------------------------------------------------------
def _ei(best, mu, var, sign, cdf="erfc"):
    sd = np.sqrt(var)
    u = (best - mu) / sd
    pdf = 0.3989422804014326779 * np.exp(-0.5 * u * u)
    c = 0.5 * erfc(-u * 0.7071067811865475244) if cdf == "erfc" else 0.5 * (1.0 - erf(-u * 0.7071067811865475244))
    return sign * (sd * (u * c + pdf))


@pytest.fixture(scope="module")
def ei_case():
    """mu from the incumbent to 9 sd beyond it (the tail where u Phi + phi cancels), both tasks; EI underflowing at
    u = -40 and u Phi ~ u at u = 45."""
    rng = np.random.default_rng(5)
    var = rng.uniform(1e-3, 2.0, 604)
    u = np.concatenate([rng.uniform(-9.0, 3.0, 500), rng.uniform(-9.0, -5.0, 100), [-40.0, -38.5, 30.0, 45.0]])
    return 0.25, 0.25 - u * np.sqrt(var), var


@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_ei_checker_accepts_the_formula(ei_case, sign):
    best, mu, var = ei_case
    if sign < 0:
        mu = 2 * best - mu
    ei = _ei(best, mu, var, sign)
    r = P.check_ei(ei, best, mu, var, sign, np.arange(len(mu)))
    print(f"EI (sign {sign}): {r:.2e} of bound")
    assert r <= 1.0


def test_ei_checker_rejects_one_minus_erf(ei_case):
    best, mu, var = ei_case
    ei = _ei(best, mu, var, 1.0, cdf="erf")
    r = P.check_ei(ei, best, mu, var, 1.0, np.arange(len(mu)))
    print(f"EI with 1 - erf: {r:.2e} of bound")
    assert r > 1.0
    exact = np.array([float(e) for e in P.ei_exact(best, mu, var, 1.0)])
    rel = np.abs(ei - exact) / np.abs(exact).max()
    CURRENT_RULE["EI: Phi as 1 - erf"] = bool(np.nanmax(rel) <= 1e-6)


def test_cost_matches_candidate_cost_order():
    X = np.array([[0.1, -0.2, 0.3], [1e-17, 1.0, -1e-17]])
    assert np.array_equal(P.candidate_cost(X, 3.0, True), (((3.0 + 0.1) + 0.2) + 0.3, ((3.0 + 1e-17) + 1.0) + 1e-17))
    assert np.array_equal(P.candidate_cost(X, 3.0, False), [3.0, 3.0])
    assert P.first_argmax([np.nan, 1.0, 1.0, 0.5]) == (1.0, 1, 1)
    assert P.first_argmax([np.nan, np.nan]) == (-np.inf, -1, 2)


def test_current_rule(sep_sets, ei_case):
    """Every fault above once more, printing which of them the parity rule of the oracle tests accepts (the bounds reject
    them all)."""
    CURRENT_RULE.clear()
    test_fit_checker_rejects_a_missing_trailing_product()
    test_fit_checker_rejects_an_inverse_entry_off_by_1e3_ulp()
    for fault, n, path in FAULTS:
        test_posterior_checker_rejects_faults(sep_sets, fault, n, path)
    test_ei_checker_rejects_one_minus_erf(ei_case)
    print("\nfaults the current parity rule accepts:")
    for k, ok in CURRENT_RULE.items():
        print(f"  {'ACCEPTED' if ok else 'rejected'}  {k}")
