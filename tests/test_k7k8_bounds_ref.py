"""CPU checks of oracle/k7k8_bounds.py: NumPy emulations of K7's prior-gradient pass (per item and slab, the butterfly, the
4-warp sum, the per-lane item sum), of eval_point (k*, dk*, the warp substitutions, EI and its gradient) and of K8's NLL and
gradient (substitutions by rinv, X = L^-1 from the right, W) pass their checkers; each injected fault fails its checker.
Run with -s to see every fault, its worst error / bound, and whether the older rules (the 1e-6 rule of test_refine_gpu, the
cond-scaled rule of test_hyper_gpu) accept it."""
import numpy as np
import pytest
from scipy.special import erf, erfc

from oracle import cbo_oracle as O
from oracle import k7k8_bounds as K
from oracle import posterior_bounds as P


def _bfly(x):
    """Fixed xor butterfly over the last axis (32 lanes); the result of lane 0."""
    x = x.copy()
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        x = x + x[..., lanes ^ o]
    return x[..., 0]


# ---- K7 prior-gradient pass ------------------------------------------------------------------------------------------------
def emulate_pass(pts, X, ls, M, w, s2, noise, fault=None):
    """refine_prior_kernel + eval_point's reduction of the partials, in the kernels' order (an FMA is a multiply and an add)."""
    pts, X = np.atleast_2d(pts), np.atleast_2d(X)
    N, d = X.shape
    R, C = K.m_row_blocks(N), K.m_chunks(N)
    Np = R * K.PASS_THREADS
    il = 1.0 / np.asarray(ls, np.float64)
    z = (pts[:, None, :] - X[None, :, :]) * il                       # P x N x d
    r2 = np.zeros(z.shape[:2])
    for k in range(d):
        r2 = r2 + z[..., k] * z[..., k]
    u = np.exp(-0.5 * r2)
    a = u[..., None] * z * (1.0 if fault == "a_no_il" else il)      # P x N x d
    T = np.zeros((len(pts), 1 + d, Np))
    T[:, 0, :N] = u
    T[:, 1:, :N] = a.transpose(0, 2, 1)
    Mp = np.zeros((Np, Np))
    Mp[:N, :N] = M
    wp = np.zeros(Np)
    wp[:N] = w
    nf = 2 + 2 * d
    part = np.zeros((R * C, len(pts), nf))
    for I in range(R):
        rows = slice(I * 128, I * 128 + 128)
        for c in range(C):
            if not K.m_item_exists(I, c):
                continue
            kt0, kt1, diag0 = K.item_slabs(I, c)
            acc = np.zeros((len(pts), 1 + d, 128))
            for kt in range(kt0, kt1):
                if fault == "skip_last_slab" and c > 0 and kt == kt1 - 1:
                    continue
                sc = 2.0 if kt < diag0 or (fault == "diag_scale2" and kt == diag0) else 1.0
                for col in range(kt * 16, kt * 16 + 16):
                    acc = acc + (Mp[rows, col] * sc)[None, None, :] * T[:, :, col][:, :, None]
            un, an = T[:, 0, rows], T[:, 1:, rows]
            wn = wp[rows] if c == 0 else np.zeros(128)
            v = np.zeros((len(pts), nf, 128))
            v[:, 0] = un * wn
            v[:, 1] = un * acc[:, 0]
            v[:, 2:2 + d] = an * wn
            v[:, 2 + d:] = an * acc[:, 0:1] + un[:, None] * acc[:, 1:]
            warps = _bfly(v.reshape(len(pts), nf, 4, 32))                  # P x nf x 4
            s = (warps[..., 0] + warps[..., 1]) + warps[..., 2]
            full = s + warps[..., 3]
            if fault == "sred_drop_w3_dv":
                full[:, 2 + d:] = s[:, 2 + d:]
            part[I * C + c] = full
    lane = np.zeros((len(pts), nf, 32))
    for e in range(R * C):
        if K.m_item_exists(e // C, e % C):
            lane[:, :, e % 32] = lane[:, :, e % 32] + part[e]
    tot = _bfly(lane)
    return dict(m=tot[:, 0], v=(np.float64(s2) + np.float64(noise)) - tot[:, 1], dm=-tot[:, 2:2 + d], dv=tot[:, 2 + d:])


def _obs_case(N, d, seed, noise=1e-2):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, d))
    ls = np.array([0.7, 1.3, 0.9, 1.6])[:d]                          # l_k != 1: a fault in il is visible
    y = np.sin(X.sum(1)) + 0.1 * rng.standard_normal(N)
    gp = O.obs_gp_fit(X, y, 1.2, ls, noise=noise, form="diff")
    s2 = 1.2
    M = (s2 * s2) * gp["Kyinv"]
    M = 0.5 * (M + M.T)
    w = s2 * gp["alpha"]
    pts = np.vstack([X[:3], rng.uniform(-1.5, 1.5, (5, d))])
    return pts, X, ls, M, w, s2, noise


def old_rule(got, ref):
    """test_refine_gpu.rule: max relative error with a floor of 1e-6 max|ref|; <= 1e-6 accepts."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    floor = max(1e-6 * np.max(np.abs(ref)), 1e-300)
    return float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), floor)))


PASS_CASES = [(200, 2, 1), (641, 1, 2)]


@pytest.fixture(scope="module", params=PASS_CASES, ids=lambda c: f"N{c[0]}-d{c[1]}")
def pass_case(request):
    N, d, seed = request.param
    case = _obs_case(N, d, seed)
    pts, X, ls, M, w, s2, noise = case
    return case, K.prior_pass_ref(pts, X, ls, M, w, s2, noise)


def test_pass_emulation_meets_bounds(pass_case):
    case, ref = pass_case
    r = K.check_prior_pass(emulate_pass(*case), ref)
    print(f"  pass N={len(case[1])}: " + "  ".join(f"{k} {v:.2e}" for k, v in r.items()), K.pass_counts(len(case[1])))
    assert max(r.values()) <= 1.0, r


PASS_FAULTS = {"diag_scale2": ("v", "dv"), "sred_drop_w3_dv": ("dv",), "skip_last_slab": ("v", "dv"), "a_no_il": ("dm", "dv")}


@pytest.mark.parametrize("fault", sorted(PASS_FAULTS))
def test_pass_faults_are_caught(pass_case, fault):
    case, ref = pass_case
    N = len(case[1])
    if fault == "skip_last_slab" and K.m_chunks(N) < 2:
        pytest.skip("needs a second chunk (N > 512)")
    got = emulate_pass(*case, fault=fault)
    r = K.check_prior_pass(got, ref)
    old = {k: old_rule(got[k], ref[k].astype(np.float64)) <= 1e-6 for k in PASS_FAULTS[fault]}
    print(f"  fault {fault} N={N}: " + "  ".join(f"{k} {r[k]:.1e}" for k in PASS_FAULTS[fault]) + f"; 1e-6 rule accepts {old}")
    assert max(r[k] for k in PASS_FAULTS[fault]) > 1.0, (fault, r)


# ---- eval_point ----------------------------------------------------------------------------------------------------------------
def emulate_eval(S, x, m, v, dm, dv, best, sign, fault=None):
    """eval_point for one point x (d) from the prior's m, v, dm, dv; S: x_int, sv, alpha, L, s2, l, causal, cost."""
    n, d = S["x_int"].shape
    il = 1.0 / S["l"]
    xs = S["x_int"] * il
    causal = S["causal"]
    sqv = np.sqrt(v) if causal else 0.0
    hv = (1.0 / sqv if fault == "hv_no_half" else 0.5 / sqv) if causal else 0.0
    zz = x * il - xs                                                 # n x d
    r2 = np.zeros(n)
    for k in range(d):
        r2 = r2 + zz[:, k] * zz[:, k]
    e = S["s2"] * np.exp(-0.5 * r2)
    ks = S["sv"] * sqv + e
    dks = -e[:, None] * (zz * il) + ((S["sv"][:, None] * dv[None, :]) * hv)
    al = S["alpha"]
    pad = lambda a: np.concatenate([a, np.zeros((128 - n,) + a.shape[1:])]).reshape((4, 32) + a.shape[1:])

    def wsum(terms):                                                 # 4-slot chain per lane, then warp_sum
        t = pad(terms)
        s = np.zeros(t.shape[1:])
        for r in range(4):
            s = s + t[r]
        return _bfly(np.moveaxis(s, 0, -1))

    mu = m + wsum(ks * al)
    dmu = dm + wsum(al[:, None] * dks)
    L = S["L"]
    rr = ks.copy()
    for j in range(n):
        rr[j] = rr[j] / L[j, j]
        rr[j + 1:] = rr[j + 1:] - L[j + 1:, j] * rr[j]
    ss = wsum(rr * rr)
    var = ((S["s2"] + v) - ss) + 1e-10
    order = []
    for rb in (3, 2, 1, 0):
        jj = list(range(32 * rb, min(n, 32 * rb + 32)))
        order += jj if (fault == "beta_forward_slot" and rb == 0) else jj[::-1]
    for j in order:
        rr[j] = rr[j] / L[j, j]
        rr[:j] = rr[:j] - L[j, :j] * rr[j]
    dvar = dv - 2.0 * wsum(rr[:, None] * dks)
    sd = np.sqrt(var)
    u = (best - mu) / sd
    pdf = 0.3989422804014326779 * np.exp(-0.5 * u * u)
    z = -u * 0.7071067811865475244
    cdf = 0.5 * (1.0 - erf(z)) if fault == "Phi_1_minus_erf" else 0.5 * erfc(z)     # the fault: erfc(z) as 1 - erf(z)
    ei = sign * (sd * (u * cdf + pdf))
    cost = P.candidate_cost(x[None, :], S["cost_fix"], S["cost_variable"])[0]
    acq = ei / cost
    dei = sign * (pdf * dvar / (2.0 * sd) - cdf * dmu)
    if S["cost_variable"]:
        dc = np.where(x > 0, 1.0, np.where(x < 0, -1.0, 1.0 if fault == "sign0_is_1" else 0.0))
    else:
        dc = np.zeros(d)
    return dict(mu=mu, var=var, ei=ei, acq=acq, dmu=dmu, dvar=dvar, dei=dei, dacq=(dei - acq * dc) / cost)


def _surrogate(n, d, seed, causal=True, s2=1.0, l=1.0, cost_variable=True):
    rng = np.random.default_rng(seed)
    XI = rng.uniform(-1.5, 1.5, (n, d)) * l
    sv = np.sqrt(rng.uniform(0.05, 0.5, n)) if causal else np.zeros(n)
    y = np.sin(XI.sum(1) / l) + 0.05 * rng.standard_normal(n)
    Ky = np.array(P.gram_ref(XI, sv, s2, l)[0], np.float64)
    L = np.linalg.cholesky(Ky)
    alpha = np.linalg.solve(Ky, y)
    return dict(x_int=XI, sv=sv, alpha=alpha, L=L, s2=s2, l=l, causal=causal, cost_fix=float(d), cost_variable=cost_variable,
                y=y)


def _eval_all(S, X, m, v, dm, dv, best, sign, fault=None):
    best = np.broadcast_to(np.asarray(best, np.float64), (len(X),))
    outs = [emulate_eval(S, X[p], m[p], v[p], dm[p], dv[p], best[p], sign, fault) for p in range(len(X))]
    return {k: np.array([o[k] for o in outs]) for k in outs[0]}


EVAL_CASES = [(40, 2, True, 1.0, 1.0), (100, 3, True, 50.0, 4.0), (33, 1, False, 1e-3, 0.3)]


@pytest.fixture(scope="module", params=EVAL_CASES, ids=lambda c: f"n{c[0]}-d{c[1]}-{'causal' if c[2] else 'plain'}")
def eval_case(request):
    n, d, causal, s2, l = request.param
    S = _surrogate(n, d, 300 + n, causal, s2, l)
    rng = np.random.default_rng(n)
    X = rng.uniform(-1.5, 1.5, (9, d)) * l
    X[0, 0] = 0.0                                                    # x_k = 0 with a variable cost
    X[1] = S["x_int"][0]
    P_ = len(X)
    if causal:
        m, v = rng.standard_normal(P_) * 0.3, rng.uniform(0.2, 0.8, P_)
        dm, dv = rng.standard_normal((P_, d)), rng.standard_normal((P_, d)) * 0.2
    else:
        m = v = np.zeros(P_)
        dm = dv = np.zeros((P_, d))
    # an incumbent per point, u = (best - mu) / sd from -1 to -8 (u Phi + phi cancels; Phi as 1 - erf loses digits) and
    # one point at u = -40, where phi, Phi and dei underflow
    post = _eval_all(S, X, m, v, dm, dv, 0.0, 1.0)
    u = np.array([-1.0, -2.0, -3.0, -4.0, -5.0, -6.0, -7.0, -8.0, -40.0])
    best = post["mu"] + u * np.sqrt(post["var"])
    ref = K.grad_ref(X, m, v, dm, dv, dict(S))
    return S, X, m, v, dm, dv, best, ref


@pytest.mark.parametrize("task", ["min", "max"])
def test_eval_emulation_meets_bounds(eval_case, task):
    S, X, m, v, dm, dv, best, ref = eval_case
    sign = 1.0 if task == "min" else -1.0
    got = _eval_all(S, X, m, v, dm, dv, best, sign)
    uu = (best - got["mu"]) / np.sqrt(got["var"])
    assert np.all(uu[:8] < -0.9) and np.all(uu[:8] > -8.1) and uu[8] < -39.0, uu
    assert np.count_nonzero(got["dei"][:8]) == got["dei"][:8].size      # the checked dei are not underflowed
    r = K.check_grad(got, ref)
    r["dei"] = K.check_dei(got["dei"], best, got["mu"], got["var"], got["dmu"], got["dvar"], sign)
    dacq = K.dacq_ref(got["dei"], got["acq"], X, S["cost_fix"], S["cost_variable"])
    assert dacq.tobytes() == got["dacq"].tobytes()
    print(f"  eval n={len(S['y'])} {task}: " + "  ".join(f"{k} {v_:.2e}" for k, v_ in r.items()))
    assert max(r.values()) <= 1.0, r


EVAL_FAULTS = {"hv_no_half": "dmu", "beta_forward_slot": "dvar", "Phi_1_minus_erf": "dei", "sign0_is_1": "dacq"}


@pytest.mark.parametrize("fault", sorted(EVAL_FAULTS))
def test_eval_faults_are_caught(eval_case, fault):
    S, X, m, v, dm, dv, best, ref = eval_case
    if fault == "hv_no_half" and not S["causal"]:
        pytest.skip("a non-causal set has no sqrt(v) term")
    q = EVAL_FAULTS[fault]
    got = _eval_all(S, X, m, v, dm, dv, best, 1.0, fault)
    good = _eval_all(S, X, m, v, dm, dv, best, 1.0)
    if q == "dei":
        r = K.check_dei(got["dei"], best, got["mu"], got["var"], got["dmu"], got["dvar"], 1.0)
        caught = r > 1.0
    elif q == "dacq":
        r = float(np.abs(K.dacq_ref(got["dei"], got["acq"], X, S["cost_fix"], S["cost_variable"]) - got["dacq"]).max())
        caught = r > 0.0
    else:
        r = K._worst(got[q], ref[q], ref["e_" + q])
        caught = r > 1.0
    old = old_rule(got[q], good[q]) <= 1e-6
    print(f"  fault {fault} ({q}): {'error / bound' if q != 'dacq' else 'bit difference'} {r:.1e}; 1e-6 rule accepts {old}")
    assert caught, (fault, r)


# ---- K8 ----------------------------------------------------------------------------------------------------------------------
def emulate_k8(L, x_int, res, s2, l, fault=None):
    """hyp_nll + hyp_grad from the factor L (K2's), in the kernel's order."""
    n, d = x_int.shape
    dsq = np.diag(L).copy()
    rinv = 1.0 / dsq
    z = res.copy()
    for j in range(n):
        z[j] = z[j] * rinv[j]
        z[j + 1:] = z[j + 1:] - L[j + 1:, j] * z[j]
    pad = lambda a: np.concatenate([a, np.zeros(128 - n)]).reshape(4, 32)
    zp, lgp = pad(z), pad(np.log(dsq))
    zz, lg = np.zeros(32), np.zeros(32)
    for r in range(4):
        zz = zz + zp[r] * zp[r]
        if not (fault == "lg_missing_slot3" and r == 3):
            lg = lg + lgp[r]
    zz, lg = _bfly(zz), _bfly(lg)
    al = z.copy()
    for j in range(n - 1, -1, -1):
        al[j] = al[j] * rinv[j]
        al[:j] = al[:j] - L[j, :j] * al[j]
    nll = (0.5 * zz + lg) + n * K.HALF_LOG_2PI
    X = np.diag(rinv)
    for j in range(n - 2, -1, -1):
        a = L[j + 1:, j] * rinv[j + 1:]
        for k in range(j + 1, n):
            a[k - j:] = a[k - j:] + X[k + 1:, k] * L[k, j]          # rows i > k: X_ik L_kj
        X[j + 1:, j] = -a * rinv[j]
    il = 1.0 / l
    t0, t1 = np.zeros(K.HYP_THREADS), np.zeros(K.HYP_THREADS)
    W = np.where(np.eye(n, dtype=bool), rinv * rinv, np.tril(X, -1) * rinv[:, None])     # W_ij starts at X_ij X_ii
    k0 = 0 if fault == "w_from_k_eq_i" else 1
    for i in range(n):
        for k in range(i + k0, n):
            W[i, :i + 1] = W[i, :i + 1] + X[k, i] * X[k, :i + 1]
    for e in range(n * n):
        i, j = divmod(e, n)
        if j > i:
            continue
        r2 = 0.0
        for k in range(d):
            t = (x_int[i, k] - x_int[j, k]) * il
            r2 = r2 + t * t
        h = 0.5 if (i == j and fault != "diag_not_halved") else 1.0
        c = h * (W[i, j] - al[i] * al[j]) * (s2 * np.exp(-0.5 * r2))
        t0[e % K.HYP_THREADS] += c
        t1[e % K.HYP_THREADS] = t1[e % K.HYP_THREADS] + c * r2
    w0, w1 = _bfly(t0.reshape(8, 32)), _bfly(t1.reshape(8, 32))
    g0 = g1 = 0.0
    for k in range(8):
        g0, g1 = g0 + w0[k], g1 + w1[k]
    return np.array([nll, g0, g1])


def old_hyper_rule(got, ref, cond, n):
    """test_hyper_gpu's rule: 1e-6 max(|f|, 1) and 1e-6 max(|g|, n), times cond 1e-9 when cond >= 1e6."""
    scale = 1.0 if cond < 1e6 else cond * 1e-9
    return bool(abs(got[0] - ref[0]) <= 1e-6 * max(abs(ref[0]), 1.0) * scale
                and np.all(np.abs(got[1:] - ref[1:]) <= 1e-6 * max(np.abs(ref[1:]).max(), n) * scale))


K8_CASES = [(31, 2, True, 1.0, 1.0), (97, 3, True, 1e-3, 0.2), (65, 1, False, 50.0, 4.0), (128, 4, False, 1.0, 0.5)]


@pytest.fixture(scope="module", params=K8_CASES, ids=lambda c: f"n{c[0]}-d{c[1]}-s2{c[3]}-l{c[4]}")
def k8_case(request):
    n, d, causal, s2, l = request.param
    S = _surrogate(n, d, 500 + n, causal, s2, l)
    res = S["y"] - 0.1
    ref = K.k8_ref(S["L"], S["x_int"], res, s2, l)
    return S, res, ref


def test_k8_emulation_meets_bounds(k8_case):
    S, res, ref = k8_case
    got = emulate_k8(S["L"], S["x_int"], res, S["s2"], S["l"])
    r = K.check_k8(got, ref)
    print(f"  K8 n={len(res)}: " + "  ".join(f"{k} {v:.2e}" for k, v in r.items()))
    assert max(r.values()) <= 1.0, r


K8_FAULTS = ["w_from_k_eq_i", "lg_missing_slot3", "diag_not_halved"]


@pytest.mark.parametrize("fault", K8_FAULTS)
def test_k8_faults_are_caught(k8_case, fault):
    S, res, ref = k8_case
    n = len(res)
    if fault == "lg_missing_slot3" and n <= 96:
        pytest.skip("the fourth register slot holds rows 96..127")
    got = emulate_k8(S["L"], S["x_int"], res, S["s2"], S["l"], fault)
    good = emulate_k8(S["L"], S["x_int"], res, S["s2"], S["l"])
    r = K.check_k8(got, ref)
    cond = float(np.linalg.cond(S["L"] @ S["L"].T))
    old = old_hyper_rule(got, good, cond, n)
    print(f"  fault {fault} n={n} cond {cond:.0e}: " + "  ".join(f"{k} {v:.1e}" for k, v in r.items())
          + f"; cond-scaled rule accepts {old}")
    assert max(r.values()) > 1.0, (fault, r)
