"""The checkers of oracle/state_bounds.py are sharp: NumPy emulations of K0, K1a and K5 in their own order of operations pass
them, and each fault a wrong tile, partial, constant or store would cause fails them.  CPU only.

Emulated: K5's Gram, the panelled Cholesky (left-looking updates inside a panel of two block columns, the diagonal block by
a right-looking Cholesky that scales by 1 / sqrt(pivot), its inverse by column substitution on 32 x 32 sub-blocks and the
recursion W21 = -W22 (L21 W11), the rows below multiplied by that inverse, one deep update behind each panel), the blocked
solve for Wt = L^-T, Ky^-1 = Wt Wt^T, z by 256-row chunks, alpha, the NLL and its gradient; K1a's P, its row sums by 256
thread partials and 8 warp partials, w and M; the K0 tables.  test_current_rule shows which faults the rules of
tests/test_obs_gp_gpu.py (test_fit_matches_oracle) let through."""
import numpy as np
import pytest

from oracle import cbo_oracle as O
from oracle import state_bounds as B

FB = 128


# ---- K5 emulation ---------------------------------------------------------------------------------------------------
def _data(seed=3, N=300, D=3):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    y = np.sin(X @ rng.uniform(-1, 1, D)) + 0.1 * rng.standard_normal(N)
    return X, y, float(rng.uniform(0.6, 1.6)), rng.uniform(0.7, 1.8, D), 1e-2


def _gram(X, s2, ls, dadd, npad):
    N = X.shape[0]
    il = 1.0 / np.asarray(ls, np.float64)
    r2 = np.zeros((N, N))
    for k in range(X.shape[1]):
        t = (X[:, None, k] - X[None, :, k]) * il[k]
        r2 = r2 + t * t
    A = np.eye(npad)
    A[:N, :N] = s2 * np.exp(-0.5 * r2)
    A[np.arange(N), np.arange(N)] += dadd
    return A


def _diag_factor(Bk):
    """Cholesky of one 128 x 128 block scaled by invd = 1 / sqrt(pivot), then its inverse: column substitution on the
    32 x 32 diagonal sub-blocks and W21 = -W22 (L21 W11) on 32- and 64-wide halves."""
    Bk = np.tril(Bk.copy())
    for j in range(FB):
        piv = Bk[j, j]
        inv = 1.0 / np.sqrt(piv)
        Bk[j, j] = piv * inv
        Bk[j + 1:, j] *= inv
        c = Bk[j + 1:, j]
        Bk[j + 1:, j + 1:] -= np.tril(np.outer(c, c))
    L = np.tril(Bk)
    W = np.zeros((FB, FB))
    for b in range(4):
        o = 32 * b
        Lb = L[o:o + 32, o:o + 32]
        for c in range(32):
            x = np.zeros(32)
            for i in range(c, 32):
                x[i] = ((1.0 if i == c else 0.0) - Lb[i, :i] @ x[:i]) / Lb[i, i]
            W[o:o + 32, o + c] = x
    for h in range(2):
        b0, b1 = 64 * h, 64 * h + 32
        T = L[b1:b1 + 32, b0:b0 + 32] @ W[b0:b0 + 32, b0:b0 + 32]
        W[b1:b1 + 32, b0:b0 + 32] = -(W[b1:b1 + 32, b1:b1 + 32] @ T)
    T = L[64:, :64] @ W[:64, :64]
    W[64:, :64] = -(W[64:, 64:] @ T)
    return L, W


def k5(X, y, s2, ls, noise, width=2, fault=None):
    """Every output and the workspace of one cbo_obs_gp_fit + cbo_obs_gp_nll in the kernels' order (NumPy float64)."""
    N = X.shape[0]
    npad = -(-N // FB) * FB
    nb = npad // FB
    dadd = B.diag_add(noise, 0.0)
    A = _gram(X, s2, ls, dadd, npad)
    Linv = np.zeros((nb, FB, FB))
    Wt = np.zeros((npad, npad))
    blk = lambda q: slice(q * FB, (q + 1) * FB)
    for p0 in range(0, nb, width):
        we = min(width, nb - p0)
        for q in range(p0, p0 + we):
            if q > p0:
                Ap = A[q * FB:, p0 * FB:q * FB]
                prod = Ap @ A[blk(q), p0 * FB:q * FB].T
                if fault == "slab":                 # tile 0 (rows of block q) loses the 16-deep slab 16..31
                    prod[:FB] -= Ap[:FB, 16:32] @ A[blk(q), p0 * FB + 16:p0 * FB + 32].T
                A[q * FB:, blk(q)] -= prod
            L, W = _diag_factor(A[blk(q), blk(q)])
            if fault == "linv" and q == 1:          # one entry of Linv_1 off by 10^3 ulp
                W[37, 35] += 1000 * np.spacing(W[37, 35])
            A[blk(q), blk(q)] = L
            Linv[q] = W
            Wt[blk(q), blk(q)] = W.T
            if q + 1 < nb:
                new = A[(q + 1) * FB:, blk(q)] @ W.T
                if fault == "half" and q == 0:      # the second 64-row half of tile 0 left unwritten
                    new[64:FB] = A[FB + 64:2 * FB, blk(q)]
                A[(q + 1) * FB:, blk(q)] = new
        T = nb - p0 - we
        for bi in range(T):
            for bj in range(bi + 1):
                I, J = p0 + we + bi, p0 + we + bj
                A[blk(I), blk(J)] -= A[blk(I), p0 * FB:(p0 + we) * FB] @ A[blk(J), p0 * FB:(p0 + we) * FB].T
    for K0 in range(0, nb, width):
        we = min(width, nb - K0)
        for K in range(K0, K0 + we):
            if K > K0:
                Wt[:K * FB, blk(K)] -= Wt[:K * FB, K0 * FB:K * FB] @ A[blk(K), K0 * FB:K * FB].T
            if K > 0:
                Wt[:K * FB, blk(K)] = Wt[:K * FB, blk(K)] @ Linv[K].T
        if nb - K0 - we > 0:
            c = (K0 + we) * FB
            Wt[:c, c:] -= Wt[:c, K0 * FB:c] @ A[c:, K0 * FB:c].T
    Wl = Wt[:N, :N]
    kyinv = np.tril(Wl @ Wl.T)
    kyinv = kyinv + np.tril(kyinv, -1).T
    if fault == "kyinv":
        kyinv[5, 5] += 1000 * np.spacing(kyinv[5, 5])
    yp = np.zeros(npad)
    yp[:N] = y
    parts = [Wt[c:c + 256].T @ yp[c:c + 256] for c in range(0, npad, 256)]
    if fault == "wty":
        parts.append(parts[0])
    z = np.zeros(npad)
    for pt in parts:
        z = z + pt
    Wz = np.triu(Wl) if fault != "wz" else np.triu(Wl, 1)
    alpha = Wz @ z[:N]
    # NLL and gradient (cbo_obs_gp_nll)
    Ld = np.diag(A)[:N]
    logs = np.log(Ld if fault != "log" else Ld[:-1])
    nll = 0.5 * float(y @ alpha) + 0.5 * N * float(B.LOG_2PI) + float(logs.sum())
    il = 1.0 / ls
    r2 = np.zeros((N, N))
    dks = []
    for k in range(X.shape[1]):
        t = (X[:, None, k] - X[None, :, k]) * il[k]
        dks.append(t * t)
        r2 = r2 + dks[-1]
    wk = (np.outer(alpha, alpha) - kyinv) * (s2 * np.exp(-0.5 * r2))
    g = [-0.5 * wk.sum()]
    for k, dk in enumerate(dks):
        term = wk * dk
        if fault == "dk" and k == 1:
            term[7, 3] = 0.0
        g.append(-0.5 * term.sum())
    return dict(A=A, Wt=Wt, Linv=Linv, z=z, kyinv=kyinv, alpha=alpha, out=np.array([nll] + g), npad=npad, dadd=dadd)


def k5_checks(st, X, y, s2, ls):
    """Every K5 check on the whole matrix; returns {name: ratio} (an AssertionError counts as an infinite ratio)."""
    N = X.shape[0]
    rows = cols = np.arange(N)
    out = {}
    L = np.tril(st["A"])
    calls = {
        "gram": lambda: B.check_gram_upper(st["A"], X, s2, ls, st["dadd"], rows, cols)[0],
        "linv": lambda: B.check_linv(L, st["Linv"], range(st["npad"] // FB)),
        "chol": lambda: B.check_chol(st["A"], st["Linv"], X, s2, ls, st["dadd"], rows, cols),
        "wt": lambda: B.check_wt(st["A"], st["Wt"], st["Linv"], rows, cols),
        "kyinv": lambda: B.check_kyinv(st["kyinv"], st["Wt"], rows, cols),
        "z": lambda: B.check_alpha(st["Wt"], y, st["z"], st["alpha"])[0],
        "alpha": lambda: B.check_alpha(st["Wt"], y, st["z"], st["alpha"])[1],
        "nll": lambda: B.check_nll(st["out"], st["alpha"], y, np.diag(st["A"])[:N], X, st["kyinv"], s2, ls)[0],
        "grad": lambda: B.check_nll(st["out"], st["alpha"], y, np.diag(st["A"])[:N], X, st["kyinv"], s2, ls)[1],
    }
    for k, f in calls.items():
        try:
            out[k] = f()
        except AssertionError:
            out[k] = np.inf
    return out


@pytest.fixture(scope="module")
def k5_case():
    X, y, s2, ls, noise = _data()
    return X, y, s2, ls, noise, k5(X, y, s2, ls, noise)


def test_k5_emulation_passes(k5_case):
    X, y, s2, ls, noise, st = k5_case
    r = k5_checks(st, X, y, s2, ls)
    print("K5 emulation, worst error / bound:", {k: f"{v:.2e}" for k, v in r.items()})
    assert all(v <= 1.0 for v in r.values()), r


K5_FAULTS = {"linv": "linv", "slab": "chol", "half": "chol", "kyinv": "kyinv", "wty": "z", "wz": "alpha", "log": "nll",
             "dk": "grad"}


@pytest.mark.parametrize("fault", sorted(K5_FAULTS))
def test_k5_fault_fails(k5_case, fault):
    X, y, s2, ls, noise, _ = k5_case
    with np.errstate(invalid="ignore"):      # (the "half" fault meets a negative pivot)
        st = k5(X, y, s2, ls, noise, fault=fault)
    r = k5_checks(st, X, y, s2, ls)
    assert r[K5_FAULTS[fault]] > 1.0, (fault, r)


def _old_rule(X, y, s2, ls, noise, alpha, kyinv):
    """test_fit_matches_oracle's rules: residuals of alpha and Ky^-1, symmetry, the 1e-6 forward rule."""
    from helpers import RTOL, rel_err
    ref = O.obs_gp_fit(X, y, s2, ls, form="diff")
    N = X.shape[0]
    Ky = O.rbf_K(X, X, s2, ls, "diff", same=True) + (noise + 1e-8) * np.eye(N)
    nrm = np.abs(Ky).sum(1).max()
    return bool(np.abs(Ky @ alpha - y).max() <= 1e-12 * (nrm * np.abs(alpha).max() + np.abs(y).max())
                and np.abs(Ky @ kyinv - np.eye(N)).max() <= 1e-11 * nrm * np.abs(kyinv).max()
                and np.array_equal(kyinv, kyinv.T)
                and rel_err(alpha, ref["alpha"], 1e-6 * np.abs(ref["alpha"]).max()).max() <= RTOL
                and rel_err(kyinv, ref["Kyinv"], 1e-6 * np.abs(ref["Kyinv"]).max()).max() <= RTOL)


def test_current_rule(k5_case):
    """The normwise rules accept a Ky^-1 entry 10^3 ulp off (and the other faults that change alpha or Ky^-1 by little);
    the bounds above reject every one of them."""
    X, y, s2, ls, noise, st = k5_case
    assert _old_rule(X, y, s2, ls, noise, st["alpha"], st["kyinv"])
    accepted = []
    for fault in ("linv", "slab", "half", "kyinv", "wty", "wz"):
        with np.errstate(invalid="ignore"):
            f = k5(X, y, s2, ls, noise, fault=fault)
        if _old_rule(X, y, s2, ls, noise, f["alpha"], f["kyinv"]):
            accepted.append(fault)
    print("faults the rules of test_fit_matches_oracle accept:", accepted)
    assert "kyinv" in accepted and "linv" in accepted


def test_jitter_reproduced():
    """jitter_k5 repeats DeviceObsGP.fit's ladder in its order of operations."""
    s2, noise = 1e12, 0.0
    j = 0.0
    for t in range(4):
        assert B.jitter_k5(t, s2, noise) == j
        j = (s2 + noise + 1e-8) * 1e-6 if t == 0 else j * 10.0


# ---- K1a emulation ----------------------------------------------------------------------------------------------------
def k1a(seed=5, N=300, c=3, n_mc=40, fault=None):
    rng = np.random.default_rng(seed)
    xc, mc = rng.standard_normal((N, c)), rng.standard_normal((n_mc, c))
    ls = rng.uniform(0.7, 1.8, c)
    s2 = float(rng.uniform(0.6, 1.6))
    alpha = rng.standard_normal(N)
    Kq = rng.standard_normal((N, N))
    kyinv = Kq @ Kq.T / N + np.eye(N)
    kyinv = np.tril(kyinv) + np.tril(kyinv, -1).T
    npad, spad = -(-N // FB) * FB, -(-n_mc // 16) * 16
    il = 1.0 / ls
    r2 = np.zeros((N, n_mc))
    for k in range(c):
        t = (mc[None, :, k] - xc[:, None, k]) * il[k]
        r2 += t * t
    P = np.zeros((npad, spad))
    P[:N, :n_mc] = np.exp(-0.5 * r2)
    # row sums: thread partials (stride 256), 8 warp partials, then their sum
    thr = np.zeros((npad, 256))
    for i in range(spad):
        thr[:, i % 256] += P[:, i]
    warps = thr.reshape(npad, 8, 32).sum(2)
    if fault == "warp":
        warps[:, 1] = 0.0
    tot = np.zeros(npad)
    for x in range(8):
        tot = tot + warps[:, x]
    pbar = tot[:N] / n_mc
    w = (s2 * alpha) * pbar
    coef = (s2 * s2) / n_mc if fault != "coef" else s2 / n_mc
    a = P @ P.T
    M = np.zeros((npad, npad))
    M[:N, :N] = (coef * kyinv) * a[:N, :N]
    M = np.tril(M) + np.tril(M, -1).T
    if fault == "mirror":          # tile (0, 1) receives the mirror of tile (2, 0)
        M[:FB, FB:2 * FB] = M[2 * FB:3 * FB, :FB].T
    if fault == "pad":
        M[N + 3, 7] = M[7, N + 3] = 1e-300
    return dict(P=P, pbar=pbar, w=w, M=M, kyinv=kyinv, s2=s2, n_mc=n_mc, alpha=alpha, xc=xc, mc=mc, ls=ls, N=N)


def k1a_checks(st):
    N = st["N"]
    out = {}
    calls = {"P": lambda: B.check_p(st["P"], st["mc"], st["xc"], st["ls"], st["n_mc"]),
             "pbar": lambda: B.check_pbar_w(st["P"][:N], st["pbar"], st["w"], st["n_mc"], st["s2"], st["alpha"]),
             "M": lambda: B.check_m(st["M"], st["P"][:N], st["kyinv"], st["s2"], st["n_mc"])}
    for k, f in calls.items():
        try:
            out[k] = f()
        except AssertionError:
            out[k] = np.inf
    return out


def test_k1a_emulation_passes():
    r = k1a_checks(k1a())
    print("K1a emulation, worst error / bound:", {k: f"{v:.2e}" for k, v in r.items()})
    assert all(v <= 1.0 for v in r.values()), r


@pytest.mark.parametrize("fault,check", [("warp", "pbar"), ("coef", "M"), ("mirror", "M"), ("pad", "M")])
def test_k1a_fault_fails(fault, check):
    assert k1a_checks(k1a(fault=fault))[check] > 1.0


def test_nocond_bit_for_bit():
    rng = np.random.default_rng(9)
    N, npad, s2 = 130, 256, 1.3
    kyinv = rng.standard_normal((N, N))
    kyinv = kyinv + kyinv.T
    alpha = rng.standard_normal(N)
    M = np.zeros((npad, npad))
    M[:N, :N] = (s2 * s2) * kyinv
    B.check_nocond(M, np.ones(N), s2 * alpha, kyinv, s2, alpha)
    M[:N, :N] = s2 * kyinv
    with pytest.raises(AssertionError):
        B.check_nocond(M, np.ones(N), s2 * alpha, kyinv, s2, alpha)


# ---- K0 -----------------------------------------------------------------------------------------------------------------
def test_k0_tables():
    rng = np.random.default_rng(11)
    N, npad, d = 129, 256, 3
    X = rng.standard_normal((N, d))
    ls = rng.uniform(0.5, 2.0, d)
    g = np.linspace(-2, 2, 17)
    tab = np.zeros((17, npad))
    tab[:, :N] = np.exp(-0.5 * (((g[:, None] - X[None, :, 0]) * (1.0 / ls[0])) ** 2))
    assert B.check_table(tab, g[:, None], X[:, :1], ls[:1]) <= 1.0
    pts = rng.uniform(-2, 2, (5, d))
    u = np.zeros((5, npad))
    r2 = np.zeros((5, N))
    for q in range(d):
        t = (pts[:, None, q] - X[None, :, q]) * (1.0 / ls[q])
        r2 += t * t
    u[:, :N] = np.exp(-0.5 * r2)
    assert B.check_table(u, pts, X, ls) <= 1.0
    bad = u.copy()
    bad[2, 9] *= 1 + 64 * 2.0 ** -52
    assert B.check_table(bad, pts, X, ls) > 1.0
    bad = u.copy()
    bad[1, N] = 1e-310
    with pytest.raises(AssertionError):
        B.check_table(bad, pts, X, ls)


# ---- the launch mirror --------------------------------------------------------------------------------------------------
def test_k5_plan_split_thresholds():
    """On 148 SMs the in-panel products first run as panel_tile_kernel<4> at nb = 39 and as <8> at nb = 76."""
    assert B.k5_plan(38 * 128, 148)["variants"] == {2}
    assert B.k5_plan(38 * 128 + 1, 148)["variants"] == {2, 4}
    assert 8 not in B.k5_plan(9600, 148)["variants"]
    assert B.k5_plan(9601, 148)["variants"] == {2, 4, 8}
    p = B.k5_plan(1, 148)
    assert p["launches"] == 1 + 1 + 4 and p["tma"] == []
    p = B.k5_plan(513, 148)
    assert p["tma"] == ["syrk", "winv"]
