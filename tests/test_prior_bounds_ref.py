"""The checkers of oracle/prior_bounds.py are sharp: they accept a correct evaluation done in the kernels' own order and
reject each fault a wrong tile, ownership or carry would cause.  CPU only.

K1b (prior_eval.cu) is mimicked by a blocked fp64 evaluation: per 128-column block jb of M, the strictly-lower k range
doubled plus the diagonal block, optionally cut into segments of `chunk` column blocks whose partial row sums are added
in item order (prior_finalize_kernel).  K1c (prior_rows.cu) is mimicked by a vectorised Dot2: TwoProd / TwoSum along k,
then TwoProd against u_n and a double-double reduction over n."""
import numpy as np
import pytest

from helpers import make_case
from oracle import cbo_oracle as O
from oracle import prior_bounds as B

BLK = 128


# ---- K1b ---------------------------------------------------------------------------------------------
def _k1b_case(seed=11, N=2 * BLK + 17, p=(13, 11)):
    """Fp64 tables (p_k, N) of a d = 2 grid, M, w, s2, noise: the inputs K1b reads.  N = 273: the last column block has
    17 live columns (the ragged variant <8,1,2,4>)."""
    kw, ora = make_case(seed=seed, N=N, d=len(p), c=1, n=3, p=p)
    gp = ora["gp"]
    f = O.prior_factors(gp, ora["cond"], ora["cols"])
    tabs = [O.intervened_u(gp, [k], kw["grid"][k][:, None]) for k in range(len(p))]
    return tabs, f["M"], f["w"], kw["s2"], 1e-2


def _blocked(tabs, M, w, s2, noise, chunk=0, mutate=None):
    """K1b's order in fp64: returns m, v of every grid row.  chunk > 0: segments of `chunk` column blocks (partials added
    in item order).  mutate: 'drop_ragged' (one 16 x 16 block of M missing from the last column block), 'once' (an
    off-diagonal block of column block 1 counted once), 'dup_segment' (one segment's partial added twice)."""
    G = int(np.prod([t.shape[0] for t in tabs]))
    N = M.shape[0]
    Np = -(-N // BLK) * BLK
    nJ = Np // BLK
    U = np.asarray(B.grid_u(tabs, np.arange(G)), np.float64)     # (the fp64 rounding of the products K1b forms)
    U = np.pad(U, ((0, 0), (0, Np - N)))
    Mp = np.pad(M, ((0, Np - N), (0, Np - N)))
    if mutate == "drop_ragged":
        Mp = Mp.copy()
        Mp[16:32, (nJ - 1) * BLK:(nJ - 1) * BLK + 16] = 0.0     # k slab 1 x the first 16 live columns of the last block
    parts = []
    for jb in range(nJ):
        J = slice(jb * BLK, (jb + 1) * BLK)
        segs = []
        if jb:
            step = chunk * BLK if chunk else jb * BLK
            segs += [(k0, min(k0 + step, jb * BLK), True) for k0 in range(0, jb * BLK, step)]
        segs.append((jb * BLK, (jb + 1) * BLK, False))
        for k0, k1, lower in segs:
            T = U[:, k0:k1] @ Mp[k0:k1, J]
            if lower and not (mutate == "once" and jb == 1 and k0 == 0):
                T = T * 2.0
            parts.append(np.einsum("gj,gj->g", T, U[:, J]))
    if mutate == "dup_segment":
        parts.insert(len(parts) // 2, parts[len(parts) // 2])
    q = np.zeros(G)
    for pq in parts:
        q = q + pq
    return U @ np.pad(w, (0, Np - N)), (np.float64(s2) + np.float64(noise)) - q


@pytest.fixture(scope="module")
def k1b():
    tabs, M, w, s2, noise = _k1b_case()
    G = int(np.prod([t.shape[0] for t in tabs]))
    ref = B.prior_ref(B.grid_u(tabs, np.arange(G)), M, w, s2, noise, d=len(tabs))
    return tabs, M, w, s2, noise, ref


@pytest.mark.parametrize("chunk", [0, 1, 2])
def test_bound_a_accepts_the_blocked_order(k1b, chunk):
    tabs, M, w, s2, noise, ref = k1b
    rm, rv = B.check_prior(*_blocked(tabs, M, w, s2, noise, chunk=chunk), ref)
    print(f"K1b blocked chunk={chunk}: m {rm:.2e}  v {rv:.2e} of bound A")
    assert rm <= 1.0 and rv <= 1.0


@pytest.mark.parametrize("mutate,chunk", [("drop_ragged", 0), ("once", 0), ("dup_segment", 1), ("dup_segment", 2)])
def test_bound_a_rejects_faults(k1b, mutate, chunk):
    tabs, M, w, s2, noise, ref = k1b
    _, rv = B.check_prior(*_blocked(tabs, M, w, s2, noise, chunk=chunk, mutate=mutate), ref)
    print(f"K1b fault {mutate} chunk={chunk}: v {rv:.2e} of bound A")
    assert rv > 1.0, f"{mutate}: the fault stayed inside bound A"


def test_bound_a_rejects_a_nan_and_a_wrong_mean(k1b):
    tabs, M, w, s2, noise, ref = k1b
    m, v = _blocked(tabs, M, w, s2, noise)
    v2 = v.copy()
    v2[5] = np.nan
    assert B.check_prior(m, v2, ref)[1] == np.inf
    m2 = m.copy()
    m2[7] += 1e3 * B.prior_bounds(ref)["m"][7]
    assert B.check_prior(m2, v, ref)[0] > 1.0


def test_bound_a_counts_the_documented_roundings():
    N, d = 300, 3
    ref = dict(N=N, d=d, q_abs=np.ones(1), m_abs=np.ones(1), v=np.zeros(1, np.longdouble), Mmax=1.0, wmax=1.0)
    b = B.prior_bounds(ref)
    assert b["m"][0] == pytest.approx(B.gamma(N + d) + B.gamma(N + d, B.U_LD), rel=1e-12)
    assert b["v"][0] >= B.gamma(N * N + 2 * d + 2)


# ---- K1c ---------------------------------------------------------------------------------------------
def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _dot2_rows(u, M, w, s2, noise, drop_low=False):
    """prior_rows.cu's arithmetic, vectorised over rows r and observations n (Dekker TwoProd in place of the DFMA one:
    both are exact).  drop_low: the final store without its low word (v = a - q_hi, m = m_hi)."""
    R, N = u.shape
    S, C = np.zeros((R, N)), np.zeros((R, N))
    for k in range(N):                               # s_n[r] = sum_k M[n][k] u_r[k] in Dot2
        p, pe = B.two_prod(M[None, :, k], u[:, k:k + 1])
        S, te = _two_sum(S, p)
        C = C + (te + pe)
    qh_n, ql_n = B.two_prod(u, S)
    ql_n = ql_n + u * C
    mh_n, ml_n = B.two_prod(u, w[None, :])
    qh, ql, mh, ml = (np.zeros(R) for _ in range(4))
    for n in range(N):                               # double-double reduction over n
        qh, te = _two_sum(qh, qh_n[:, n])
        ql = ql + (te + ql_n[:, n])
        mh, te = _two_sum(mh, mh_n[:, n])
        ml = ml + (te + ml_n[:, n])
    a = np.float64(s2) + np.float64(noise)
    if drop_low:
        return mh, a - qh
    return mh + ml, (a - qh) - ql


def _dense_1d():
    """Dense 1-D observational data, noise 1e-4: the prior variance at rows inside the data cancels ~1e10-fold."""
    rng = np.random.default_rng(0)
    N = 200
    X = np.sort(rng.uniform(-2.0, 2.0, N))[:, None]
    y = np.sin(2.0 * X[:, 0]) + 0.01 * rng.standard_normal(N)
    gp = O.obs_gp_fit(X, y, 1.0, np.array([0.8]), noise=1e-4, form="diff")
    f = O.prior_factors(gp, X, [0])
    u = O.intervened_u(gp, [0], rng.uniform(-1.8, 1.8, (6, 1)))
    return u, f["M"], f["w"], 1.0, 1e-4


def _coral_set2():
    """Set 2 of the simplified coral fixture (the 4e8 cancellation DESIGN §4 quotes) at its interventional rows."""
    from cbo_with_oop_b200.fixtures import golden_path
    from cbo_with_oop_b200.obs_gp import fit_state
    z = np.load(golden_path("simplified_coral"))
    k = "set2_"
    X = np.hstack([z[k + "x_obs_int"], z[k + "x_obs_cond"]])
    d = z[k + "x_obs_int"].shape[1]
    ls = np.concatenate([z[k + "ls_int"], z[k + "ls_cond"]])
    s2 = float(z[k + "s2"])
    alpha, kyinv = fit_state(X, z[k + "y_obs"], s2, ls, 1e-2)
    gp = dict(X=X, variance=s2, lengthscale=ls, noise=1e-2, alpha=alpha, Kyinv=kyinv, form="diff")
    f = O.prior_factors(gp, X, list(range(d)))
    return O.intervened_u(gp, list(range(d)), z[k + "x_int"]), f["M"], f["w"], s2, 1e-2


CANCELLED = {"dense_1d": (_dense_1d, 1e9), "coral_set2": (_coral_set2, 1e8)}


@pytest.fixture(scope="module", params=sorted(CANCELLED))
def cancelled(request):
    build, min_cancel = CANCELLED[request.param]
    u, M, w, s2, noise = build()
    ref = B.rows_ref(u, M, w, s2, noise)
    assert B.cancellation(ref).max() >= min_cancel, "the case was meant to cancel"
    return request.param, u, M, w, s2, noise, ref


def test_bound_c_accepts_dot2(cancelled):
    name, u, M, w, s2, noise, ref = cancelled
    rm, rv = B.check_rows(*_dot2_rows(u, M, w, s2, noise), ref)
    print(f"K1c Dot2 {name} (cancellation {B.cancellation(ref).max():.1e}): m {rm:.2e}  v {rv:.2e} of bound C")
    assert rm <= 1.0 and rv <= 1.0


def test_bound_c_rejects_plain_fp64(cancelled):
    name, u, M, w, s2, noise, ref = cancelled
    v = (np.float64(s2) + np.float64(noise)) - np.einsum("rj,rj->r", u @ M, u)
    _, rv = B.check_rows(ref["m"], v, ref)
    print(f"K1c plain fp64 {name}: v {rv:.2e} of bound C")
    assert rv > 1.0


def test_bound_c_rejects_a_lost_low_word(cancelled):
    name, u, M, w, s2, noise, ref = cancelled
    _, rv = B.check_rows(*_dot2_rows(u, M, w, s2, noise, drop_low=True), ref)
    print(f"K1c without its low word {name}: v {rv:.2e} of bound C")
    assert rv > 1.0


def test_rows_reference_is_exact_on_representable_sums():
    """Terms chosen so that the exact sum is known: the reference must return it although fp64 summation loses it."""
    u = np.array([[1.0, 1.0, 1.0]])
    M = np.array([[1e16, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, -1e16]])
    ref = B.rows_ref(u, M, np.array([1e16, 1.0, -1e16]), 0.0, 0.0)
    assert ref["v"][0] == -1.0 and ref["m"][0] == 1.0
