"""Reference values and proven error bounds for the kernels that produce the causal prior's state.

    K0 (csrc/tables.cu): tab{k}[i][j] = exp(-1/2 ((g_k[i] - X_jk) il_k)^2), u_int and the explicit-point table (rows of d
        coordinates), zero for N <= j < Npad;
    K1a (csrc/prior_precompute.cu): P_ji = exp(-1/2 sum_k ((mc_ik - X_jk) il_k)^2), pbar = sum_i P_ji / n_mc,
        w = s2 alpha pbar, M = coef Ky^-1 o (P P^T) with coef = fl(s2 s2) / n_mc, or M = (s2 s2) Ky^-1 without conditioning
        columns (nocond_kernel);
    K5 (csrc/obs_gp_fit.cu): the Gram, the blocked Cholesky with explicit diagonal-block inverses Linv_p, Wt = L^-T,
        Ky^-1 = Wt Wt^T, alpha = Wt (Wt^T y) and the NLL with its gradient (cbo_obs_gp_nll).

Every builder takes the kernel's own inputs as fetched from the device (the coordinates, alpha_obs, Ky^-1, P, and for K5
the workspace: A holding L, Wt, the Linv blocks and z), so a check covers one kernel and none of the rounding of the stages
that produced its inputs.  This module is test infrastructure; the package does not import it.

Notation and conventions (as in oracle/prior_bounds.py and oracle/posterior_bounds.py): u = 2^-53, gamma_k = k u / (1 - k u).
References are evaluated in np.longdouble (u_ld = 2^-64 on x86) and the reference's own gamma(.., u_ld) is added to each
bound.  A DMMA.8x8x4 and an FMA each count as one IEEE rounding of their result; every bound holds for any order of the
additions and any fusing of a multiplication into the following addition (-fmad contraction removes roundings, it never
adds one).  A bound that is first order in u is multiplied by SLACK = 2.  Results in or below the subnormal range lose up
to ETA = 2^-1074 each: every bound carries a matching absolute term.  libdevice: double exp and log have at most 1 ulp of
error (EXP_ULP = LOG_ULP = 1), double rsqrt at most 1 ulp (RSQRT_ULP = 1) (CUDA C++ Programming Guide, "Mathematical
Functions", double-precision table, CUDA 12.9); one ulp is at most 2 u relative.

RBF entry (K0, K1a's P, K5's Gram).  e = exp(-r2 / 2), r2 = sum_k t_k^2, t_k = (a_k - b_k) il_k with il_k = fl(1 / l_k)
formed once on the device (or host) by IEEE division.  The reference uses the exact 1 / l_k, so that rounding is counted:
t_k carries three roundings (difference, il_k, the product), t_k^2 seven, and the sum of d squares d - 1 more:
|r2^ - r2| <= gamma_{d+6} r2.  -1/2 r2 is exact; exp adds EXP_ULP ulp and propagates the argument error with factor 1:
    |e^ - e| <= SLACK e (gamma_{d+6} r2 / 2 + 2 EXP_ULP u) + 4 ETA.
The Gram multiplies by s2 (one rounding) and adds diag_add = fl(fl(noise + 1e-8) + jitter) on the diagonal (one more);
diag_add and the jitter of a retry are reproduced bit for bit (jitter_k5):
    E_gram_ij = s2 |e^ - e|_bound + u s2 e + u |Ky_ii| [i = j] + 4 ETA s2.
Pads (N <= j < Npad, rows past N, columns past n_mc) must be exactly 0.

K1a.  pbar_j = fl(sum_i P^_ji) / n_mc: at most n_mc_pad - 1 additions in any tree, one division:
    |pbar^ - sum P^ / n_mc| <= gamma_{S} sum |P^| / n_mc,   S = n_mc_pad.
w_j = fl(fl(s2 alpha_j) pbar^_j) is reproduced bit for bit from the fetched pbar.  M_jk = fl(fl(coef Ky^-1_jk) a_jk),
a = fl(P^ P^T) (S-deep DMMA), coef = fl(fl(s2 s2) / n_mc) as a double (store_m_pair):
    |M^_jk - coef Ky^-1_jk (P^ P^T)_jk| <= gamma_{S+3} |coef Ky^-1_jk| (|P^| |P^|^T)_jk.
The mirrored store makes M exactly symmetric, and every entry of the blocked layout outside the live N x N corner is 0.
nocond_kernel is reproduced bit for bit: M = fl(fl(s2 s2) Ky^-1), w = fl(s2 alpha), pbar = 1.

K5 Cholesky.  L is formed block column by block column: block column q is brought up to date by tile products (each a
fl(sum) of up to 128 w products subtracted once per panel), its diagonal block is factored in shared memory by a
right-looking Cholesky over 32-column sub-blocks that scales by invd = rsqrt(pivot) (l_jj = fl(pivot invd),
l_ij = fl(s invd): l_ij l_jj = s (1 + theta), |theta| <= 3 (2 RSQRT_ULP u) + 2 u, i.e. six roundings), and the rows below
are NOT found by substitution but multiplied by the computed inverse Ŵ_p = Linv_p of the diagonal block:
L^_Ip = fl(S_Ip Ŵ_p^T).  Repeating Higham's proof of Thm 10.3 (Accuracy and Stability, 2nd ed.) for the sums of all
products and subtractions, every entry meets |S - sum_k l_ik l_jk| <= gamma_{n_chol} sum_k |l_ik||l_jk| with
n_chol = Npad + nb + 16 (products, one subtraction per panel and per 32-sub-block, the six of the scaling, spare), and the
multiplication by Ŵ_p adds, for i in a block I > p (first order, S_Ip ~ L^_Ip L^_pp^T):
    S_Ip - L^_Ip L^_pp^T = S_Ip (I - Ŵ_p^T L^_pp^T) - E L^_pp^T,  |E| <= gamma_128 |S_Ip||Ŵ_p^T|, so
    |Ky_ref - L^ L^T|_ij <= SLACK gamma_{n_chol} (|L^||L^T|)_ij + E_gram_ij
                           + (|L^_Ip| (|L^_pp^T| |R_p^T| + gamma_128 |L^_pp^T||Ŵ_p^T||L^_pp^T|))_ij,   R_p = L^_pp Ŵ_p - I,
R_p evaluated in longdouble from the fetched Linv_p, so the term needs no assumption on cond(L_pp).
Diagonal-block inverse.  Ŵ_p comes from column-oriented forward substitution on the four 32 x 32 diagonal sub-blocks
(L x = e_c: a right residual, Higham Thm 8.5, with the rsqrt scaling: gamma_40) and the recursion W21 = -W22 (L21 W11) on
32- and then 64-wide halves.  Expanding (L W - I)_21 = -R_22 L21 W11 - (I + R_22) E_T - L22 E_W for the two rounded
products E_T, E_W gives, with X = |L^_pp||Ŵ_p|, the RIGHT residual bound (first order)
    |R_p| <= SLACK gamma_40 X                                  inside the 32 x 32 diagonal sub-blocks,
    |R_p| <= SLACK gamma_{176} (X + X^2 + X^3)                 elsewhere (level-1 and level-2 blocks).
Wt.  Block row K of W = L^-1 is Ŵ_K S_KJ with S_KJ = -sum_{P<K} L^_KP Ŵ_PJ (tile products), so (L^ Ŵ - I)_KJ =
R_K S_KJ + E1 + L^_KK E2 and the blocked solve satisfies a RIGHT residual (Higham §14.2.2) for K > J:
    |L^ Ŵ - I|_KJ <= SLACK gamma_{n_chol} (|L^||Ŵ|)_KJ + (|R_K||L^_KK| + gamma_128 |L^_KK||Ŵ_K||L^_KK|) |Ŵ_KJ|,
and the diagonal blocks of Wt are Linv_K^T bit for bit.
Ky^-1_ij = sum_{k >= max(i,j)} Ŵ_ik Ŵ_jk from the fetched Wt: |error| <= gamma_{Npad} (|Wt||Wt|^T)_ij; the mirrored
store makes it exactly symmetric.
alpha.  z = Wt^T y by FMA chains over 256-row chunks, the chunks added in order: |z^ - Wt^T y| <= gamma_{Npad+chunks}
|Wt|^T |y|.  alpha = Wt z^ by warp-strided FMA chains and a butterfly: |alpha^ - Wt z^| <= gamma_{Npad} |Wt||z^|.
NLL.  out0 = fl(fl(0.5 fl(sum y alpha)) + fl(0.5 n c)) + fl(sum log L_ii), c = log(2 pi) as a double:
    |nll^ - nll_ref| <= SLACK [gamma_{n+2} (0.5 sum |y alpha| + sum |log L_ii|) + 2 LOG_ULP u sum |log L_ii| + 3 u 0.5 n c
                              + u |nll|]
with nll_ref = 0.5 y.alpha + sum log L_ii + 0.5 n log(2 pi) from the fetched alpha, y and diag(L^).  Gradient: terms
w_ij K_ij (1) and w_ij K_ij dk_ij, w_ij = alpha_i alpha_j - Ky^-1_ij from the fetched alpha and Ky^-1.  Each term carries the
rounding of w (2 u (|alpha_i alpha_j| + |w|)), of K (E_gram without the diagonal part), of dk_ij = t_k^2 (gamma_7), of the
products (2 u); the sums run per row over 256 threads, a butterfly and 8 warps, then over the rows the same way: depth
n_g = 2 ceil(n / 256) + 20, so |g^ - g_ref| <= 0.5 (gamma_{n_g} sum |terms| + SLACK sum |term errors|).
"""
from __future__ import annotations

import numpy as np

from oracle.prior_bounds import ETA, U, U_LD, _ratio, gamma

LD = np.longdouble
SLACK = 2.0
EXP_ULP = 1
LOG_ULP = 1
RSQRT_ULP = 1
FB = 128                 # K5 block / tile size
WTY_ROWS = 256           # rows per z partial (wty_kernel)
LOG_2PI = np.float64(1.8378770664093454836)


def g2(k):
    """gamma_k of the kernel plus the reference's own gamma_k in longdouble."""
    return gamma(k) + gamma(k, U_LD)


def worst(err, bound):
    return float(np.max(_ratio(err, bound), initial=0.0))


# --------------------------------------------------------------------------------------------------
# RBF entries (K0, P, the Gram)
# --------------------------------------------------------------------------------------------------
def rbf_ref(A, B, ls):
    """e_ref = exp(-r2 / 2) (len(A) x len(B), longdouble) with exact 1 / l, r2 (float64) and the bound on |e^ - e_ref|."""
    A, B = np.atleast_2d(np.asarray(A, np.float64)), np.atleast_2d(np.asarray(B, np.float64))
    ls = np.asarray(ls, np.float64).reshape(-1)
    d = A.shape[1]
    r2 = np.zeros((A.shape[0], B.shape[0]), LD)
    for k in range(d):
        t = (A[:, k].astype(LD)[:, None] - B[:, k].astype(LD)[None, :]) / LD(ls[k])
        r2 += t * t
    e = np.exp(-0.5 * r2)
    ef, r2f = e.astype(np.float64), r2.astype(np.float64)
    bound = SLACK * ef * (0.5 * gamma(d + 6) * r2f + 2 * EXP_ULP * U) + g2(d + 8) * ef * (1.0 + r2f) + 4.0 * ETA
    return e, r2f, bound


def check_table(tab, A, X, ls):
    """tab: rows x Npad as written (rows of coordinates A against the N observational rows X).  Returns the worst
    |error| / bound of the live entries; the pads N <= j < Npad must be exactly 0 (asserted)."""
    tab = np.asarray(tab, np.float64)
    N = X.shape[0]
    pad = tab[:, N:]
    assert np.all(pad == 0.0) and not np.any(np.signbit(pad)), "a table pad is not exactly +0"
    e, _, b = rbf_ref(A, X, ls)
    return worst(np.abs(tab[:, :N].astype(LD) - e).astype(np.float64), b)


# --------------------------------------------------------------------------------------------------
# K1a
# --------------------------------------------------------------------------------------------------
def unblock_m(raw, npad):
    """M's blocked layout ([row block][k block][k4 group][row][4], include/cbo_b200.h) -> Npad x Npad."""
    return np.asarray(raw, np.float64).reshape(npad // 128, npad // 16, 4, 128, 4).transpose(0, 3, 1, 2, 4).reshape(npad, npad)


def check_p(P, mc, xc, ls_cond, n_mc, rows=None):
    """P (Npad x S_pad as written) against exp(-r2 / 2) of the conditioning samples at `rows` (all by default); every pad
    (rows past N, columns past n_mc) exactly 0.  Returns the ratio."""
    P = np.asarray(P, np.float64)
    N = xc.shape[0]
    assert np.all(P[N:] == 0.0) and np.all(P[:N, n_mc:] == 0.0), "P has a nonzero pad"
    rows = np.arange(N) if rows is None else np.asarray(rows)
    live = P[rows, :n_mc]
    e, _, b = rbf_ref(xc[rows], mc, ls_cond)
    return worst(np.abs(live.astype(LD) - e).astype(np.float64), b)


def check_pbar_w(P, pbar, w, n_mc, s2, alpha):
    """pbar against the fetched P's row sums / n_mc (summation bound); w bit for bit.  P: N x S_pad (pads included)."""
    P = np.asarray(P, np.float64)
    S = P.shape[1]
    ref = P.astype(LD).sum(1) / LD(n_mc)
    b = g2(S) * np.abs(P).sum(1) / n_mc + 4.0 * S * ETA
    r = worst(np.abs(np.asarray(pbar, np.float64).astype(LD) - ref).astype(np.float64), b)
    wr = (np.float64(s2) * np.asarray(alpha, np.float64)) * np.asarray(pbar, np.float64)
    np.testing.assert_array_equal(w, wr, err_msg="w != fl(fl(s2 alpha) pbar)")
    return r


def m_coef(s2, n_mc):
    return (np.float64(s2) * np.float64(s2)) / np.float64(n_mc)


def check_m(Mfull, P, kyinv, s2, n_mc, rows=None, cols=None):
    """M (Npad x Npad, unblocked) against coef Ky^-1 o (P P^T) on rows x cols of the live corner (all by default).
    Asserts exact symmetry and zero pads.  P: N x S_pad as fetched."""
    Mfull = np.asarray(Mfull, np.float64)
    P = np.asarray(P, np.float64)
    N = kyinv.shape[0]
    np.testing.assert_array_equal(Mfull, Mfull.T, err_msg="M is not exactly symmetric")
    pad = Mfull.copy()
    pad[:N, :N] = 0.0
    assert np.all(pad == 0.0), "M has a nonzero entry outside the live N x N corner"
    rows = np.arange(N) if rows is None else np.asarray(rows)
    cols = np.arange(N) if cols is None else np.asarray(cols)
    S = P.shape[1]
    coef = m_coef(s2, n_mc)
    PP = P[rows].astype(LD) @ P[cols].astype(LD).T
    ck = np.abs(coef * kyinv[np.ix_(rows, cols)])
    ref = LD(coef) * kyinv[np.ix_(rows, cols)].astype(LD) * PP
    ppf = np.abs(PP).astype(np.float64)
    b = g2(S + 3) * ck * ppf + 4.0 * (S + 3) * ETA * (1.0 + ck)
    return worst(np.abs(Mfull[np.ix_(rows, cols)].astype(LD) - ref).astype(np.float64), b)


def check_nocond(Mfull, pbar, w, kyinv, s2, alpha):
    """nocond_kernel bit for bit: M = fl(s2 s2) Ky^-1 in the live corner, 0 elsewhere, w = s2 alpha, pbar = 1."""
    N = kyinv.shape[0]
    ref = np.zeros_like(Mfull)
    ref[:N, :N] = (np.float64(s2) * np.float64(s2)) * kyinv
    np.testing.assert_array_equal(Mfull, ref, err_msg="nocond M")
    np.testing.assert_array_equal(pbar, np.ones(N), err_msg="nocond pbar")
    np.testing.assert_array_equal(w, np.float64(s2) * alpha, err_msg="nocond w")


# --------------------------------------------------------------------------------------------------
# K5
# --------------------------------------------------------------------------------------------------
def jitter_k5(tries, s2, noise):
    """The jitter of the attempt after `tries` failures, as DeviceObsGP.fit / SweepEngine.fit_observational form it."""
    j = np.float64(0.0)
    for t in range(tries):
        j = (np.float64(s2) + np.float64(noise) + np.float64(1e-8)) * np.float64(1e-6) if t == 0 else j * np.float64(10.0)
    return j


def diag_add(noise, jit):
    return (np.float64(noise) + np.float64(1e-8)) + np.float64(jit)


def split_ws(ws, npad):
    """(A, Wt, Linv blocks (nb x 128 x 128), z) of the fit workspace (obs_gp_fit_impl's layout)."""
    ws = np.asarray(ws).view(np.float64) if np.asarray(ws).dtype != np.float64 else np.asarray(ws)
    nb = npad // FB
    o = 0
    A = ws[o:o + npad * npad].reshape(npad, npad); o += npad * npad
    Wt = ws[o:o + npad * npad].reshape(npad, npad); o += npad * npad
    Linv = ws[o:o + nb * FB * FB].reshape(nb, FB, FB); o += nb * FB * FB
    z = ws[o:o + npad]
    return A, Wt, Linv, z


def gram_ref(X, s2, ls, dadd, rows, cols):
    """Ky_ref (rows x cols, longdouble) and E_gram (float64)."""
    e, _, be = rbf_ref(X[rows], X[cols], ls)
    K = LD(s2) * e
    Kf = np.abs(K).astype(np.float64)
    E = s2 * be + U * Kf + g2(2) * Kf + 4.0 * ETA * max(1.0, s2)
    eq = np.asarray(rows)[:, None] == np.asarray(cols)[None, :]
    K = K + np.where(eq, LD(dadd), LD(0))
    E = E + np.where(eq, U * np.abs(K).astype(np.float64), 0.0)
    return K, E


def n_chol(npad):
    return npad + npad // FB + 16


def check_gram_upper(A, X, s2, ls, dadd, rows, cols):
    """The strictly upper blocks of A are never touched by the factorisation: they hold the Gram as gram_kernel wrote it.
    rows / cols: sampled indices; pairs with block(row) < block(col) are checked.  Returns (ratio, pairs checked)."""
    rows, cols = np.asarray(rows), np.asarray(cols)
    K, E = gram_ref(X, s2, ls, dadd, rows, cols)
    m = (rows[:, None] // FB) < (cols[None, :] // FB)
    err = np.abs(A[np.ix_(rows, cols)].astype(LD) - K).astype(np.float64)
    return worst(np.where(m, err, 0.0), np.where(m, E, 1.0)), int(m.sum())


def _lrows(A, idx):
    """Rows idx of L = tril(A) (A holds L in its lower triangle and the untouched Gram above the diagonal blocks)."""
    idx = np.asarray(idx)
    return np.where(np.arange(A.shape[1])[None, :] <= idx[:, None], A[idx], 0.0)


def _block_terms(L, Linv, p):
    """(R_p longdouble, |L_pp|, |Linv_p|) of block p (L: the workspace A or the factor; only its lower triangle is read)."""
    Lpp = np.tril(L[p * FB:(p + 1) * FB, p * FB:(p + 1) * FB])
    Wp = np.asarray(Linv[p], np.float64)
    R = Lpp.astype(LD) @ Wp.astype(LD) - np.eye(FB, dtype=LD)
    return R, np.abs(Lpp), np.abs(Wp)


def check_linv(L, Linv, blocks):
    """RIGHT residual of each diagonal-block inverse (module docstring).  L: the Npad x Npad factor (tril of A)."""
    out = 0.0
    sub = (np.arange(FB)[:, None] // 32) == (np.arange(FB)[None, :] // 32)
    for p in blocks:
        R, La, Wa = _block_terms(L, Linv, p)
        X = La @ Wa
        X2 = X @ X
        b = np.where(sub, SLACK * g2(40) * X, SLACK * g2(176) * (X + X2 + X2 @ X)) + 4.0 * FB * ETA * (1.0 + X)
        out = max(out, worst(np.abs(R).astype(np.float64), b))
    return out


def check_chol(A, Linv, X, s2, ls, dadd, rows, cols):
    """|Ky_ref - L^ L^T| on the pairs rows x cols with row >= col (the live corner), against the bound of the module
    docstring.  Returns the worst ratio."""
    npad = A.shape[0]
    L = A
    rows, cols = np.asarray(rows), np.asarray(cols)
    K, E = gram_ref(X, s2, ls, dadd, rows, cols)
    Lr, Lc = _lrows(A, rows), _lrows(A, cols)
    res = np.abs(Lr.astype(LD) @ Lc.T.astype(LD) - K).astype(np.float64)
    b = SLACK * g2(n_chol(npad)) * (np.abs(Lr) @ np.abs(Lc).T) + E + 4.0 * npad * ETA
    pb = cols // FB
    for p in np.unique(pb):
        R, La, Wa = _block_terms(L, Linv, p)
        G = La.T @ np.abs(R).astype(np.float64).T + gamma(FB) * (La.T @ Wa.T @ La.T)
        T = np.abs(Lr[:, p * FB:(p + 1) * FB]) @ G                 # rows x 128
        sel = pb == p
        extra = T[:, cols[sel] - p * FB]
        below = (rows[:, None] // FB) > p
        b[:, sel] += SLACK * np.where(below, extra, 0.0)
    m = rows[:, None] >= cols[None, :]
    return worst(np.where(m, res, 0.0), np.where(m, b, 1.0))


def check_wt(A, Wt, Linv, rows, cols):
    """RIGHT residual of the blocked solve L W = I (W = Wt^T) on rows x cols with block(row) > block(col); the diagonal
    blocks of Wt must equal Linv_K^T bit for bit and Wt's strictly lower blocks must be 0 (asserted)."""
    npad = A.shape[0]
    nb = npad // FB
    L = A
    for K in range(nb):
        blk = Wt[K * FB:(K + 1) * FB, K * FB:(K + 1) * FB]
        np.testing.assert_array_equal(blk, np.asarray(Linv[K]).T, err_msg=f"Wt's diagonal block {K} != Linv_K^T")
        assert np.all(Wt[(K + 1) * FB:, K * FB:(K + 1) * FB] == 0.0), f"Wt has a nonzero entry below block {K}"
    rows, cols = np.asarray(rows), np.asarray(cols)
    Lr, Wc = _lrows(A, rows), Wt[cols]                      # W[:, j] = Wt[j, :]
    res = (Lr.astype(LD) @ Wc.T.astype(LD)).astype(LD)
    res -= (rows[:, None] == cols[None, :])
    res = np.abs(res).astype(np.float64)
    b = SLACK * g2(n_chol(npad)) * (np.abs(Lr) @ np.abs(Wc).T) + 4.0 * npad * ETA
    rb = rows // FB
    for K in np.unique(rb):
        R, La, Wa = _block_terms(L, Linv, K)
        H = np.abs(R).astype(np.float64) @ La + gamma(FB) * (La @ Wa @ La)
        sel = rb == K
        b[sel] += SLACK * (H[rows[sel] - K * FB] @ np.abs(Wt[cols, K * FB:(K + 1) * FB]).T)
    m = rb[:, None] > (cols[None, :] // FB)
    return worst(np.where(m, res, 0.0), np.where(m, b, 1.0))


def check_kyinv(kyinv, Wt, rows, cols):
    """Forward error of Ky^-1 on rows x cols against sum_k Wt_ik Wt_jk; exact symmetry of the whole matrix."""
    N = kyinv.shape[0]
    npad = Wt.shape[0]
    np.testing.assert_array_equal(kyinv, kyinv.T, err_msg="Ky^-1 is not exactly symmetric")
    rows, cols = np.asarray(rows), np.asarray(cols)
    Wr, Wc = Wt[rows, :N], Wt[cols, :N]
    ref = Wr.astype(LD) @ Wc.T.astype(LD)
    b = g2(npad) * (np.abs(Wr) @ np.abs(Wc).T) + 4.0 * npad * ETA
    return worst(np.abs(kyinv[np.ix_(rows, cols)].astype(LD) - ref).astype(np.float64), b)


def check_alpha(Wt, y, z, alpha, ks=None, rows=None):
    """z^ against Wt^T y at the columns ks, alpha^ against Wt z^ at the rows `rows` (all by default): (ratio z, ratio alpha)."""
    N = len(y)
    npad = Wt.shape[0]
    chunks = -(-npad // WTY_ROWS)
    ks = np.arange(N) if ks is None else np.asarray(ks)
    rows = np.arange(N) if rows is None else np.asarray(rows)
    y = np.asarray(y, np.float64)
    Wk = Wt[:N, ks]
    zr = Wk.T.astype(LD) @ y.astype(LD)
    bz = g2(npad + chunks) * (np.abs(Wk).T @ np.abs(y)) + 4.0 * npad * ETA
    rz = worst(np.abs(z[ks].astype(LD) - zr).astype(np.float64), bz)
    zn = np.asarray(z[:N], np.float64)
    Wr = Wt[rows, :N]
    ar = Wr.astype(LD) @ zn.astype(LD)
    ba = g2(npad) * (np.abs(Wr) @ np.abs(zn)) + 4.0 * npad * ETA
    ra = worst(np.abs(np.asarray(alpha, np.float64)[rows].astype(LD) - ar).astype(np.float64), ba)
    return rz, ra


def check_nll(out, alpha, y, Ldiag, X, kyinv, s2, ls):
    """cbo_obs_gp_nll's out = (nll, d/dlog s2, d/dlog l_k) against references from the fetched alpha, y, diag(L), Ky^-1.
    Returns (ratio nll, ratio gradient)."""
    alpha, y, Ldiag = (np.asarray(a, np.float64) for a in (alpha, y, Ldiag))
    n = len(y)
    D = X.shape[1]
    logl = np.log(Ldiag.astype(LD))
    ya = y.astype(LD) * alpha.astype(LD)
    nll = 0.5 * ya.sum() + logl.sum() + 0.5 * n * np.log(LD(2) * LD(np.pi))
    sa, sl = float(np.abs(ya).sum()), float(np.abs(logl).sum())
    c = 0.5 * n * float(LOG_2PI)
    bn = SLACK * (gamma(n + 2) * (0.5 * sa + sl) + 2 * LOG_ULP * U * sl + 3 * U * c + U * abs(float(nll)))
    bn += g2(n + 4) * (sa + sl + c) + 1e-19 * c       # the reference's own rounding and its log(2 pi)
    rn = worst(abs(float(out[0]) - nll), bn)
    # gradient
    ls = np.asarray(ls, np.float64).reshape(-1)
    e, r2, be = rbf_ref(X, X, ls)
    K = LD(s2) * e
    Kf = np.abs(K).astype(np.float64)
    dK = s2 * be + U * Kf + 4.0 * ETA * max(1.0, s2)
    aa = np.outer(alpha, alpha).astype(LD)
    w = aa - kyinv.astype(LD)
    wf = np.abs(w).astype(np.float64)
    dw = 2 * U * (np.abs(aa).astype(np.float64) + wf)
    ng = 2 * (-(-n // 256)) + 20
    rg = 0.0
    for t in range(1 + D):
        if t == 0:
            dk, ddk = np.ones((n, n), LD), np.zeros((n, n))
        else:
            q = (X[:, t - 1].astype(LD)[:, None] - X[:, t - 1].astype(LD)[None, :]) / LD(ls[t - 1])
            dk = q * q
            ddk = gamma(7) * np.abs(dk).astype(np.float64)
        term = w * K * dk
        tf = np.abs(term).astype(np.float64)
        dkf = np.abs(dk).astype(np.float64)
        terr = dw * Kf * dkf + wf * dK * dkf + wf * Kf * ddk + 2 * U * tf
        ref = -0.5 * term.sum()
        b = 0.5 * (g2(ng) * tf.sum() + SLACK * terr.sum()) + 4.0 * n * n * ETA
        rg = max(rg, worst(abs(float(out[1 + t]) - ref), b))
    return rn, rg


# --------------------------------------------------------------------------------------------------
# K5 launch plan (a Python mirror of obs_gp_fit_impl / launch_panel_op) and the samples of a large fit
# --------------------------------------------------------------------------------------------------
def panel_variant(tiles, sms):
    """launch_panel_op's split: panel_tile_kernel<2> (4 CTAs a tile), <4> (2) or <8> (1); None launches nothing."""
    if tiles <= 0:
        return None
    return 2 if 4 * tiles <= sms else (4 if 2 * tiles <= sms else 8)


def k5_plan(N, sms, width=4):
    """Launches of one cbo_obs_gp_fit and the panel_tile_kernel variants / TMA plans it runs."""
    npad = -(-N // FB) * FB
    nb = npad // FB
    launches, variants, tma = 1, set(), []
    for p0 in range(0, nb, width):
        we = min(width, nb - p0)
        for q in range(p0, p0 + we):
            for t in ([nb - q] if q > p0 else []) + [nb - q - 1]:
                v = panel_variant(t, sms)
                if v:
                    launches += 1
                    variants.add(v)
            launches += 1                                         # potrf_diag_kernel
        T = nb - p0 - we
        if T > 0:
            launches += 1
            tma.append("syrk")
    for K0 in range(0, nb, width):
        we = min(width, nb - K0)
        for K in range(K0, K0 + we):
            for t in ([K] if K > K0 else []) + [K]:
                v = panel_variant(t, sms)
                if v:
                    launches += 1
                    variants.add(v)
        if nb - K0 - we > 0:
            launches += 1
            tma.append("winv")
    launches += 4                                                 # Ky^-1, wty, wty_reduce, wz
    return dict(launches=launches, variants=variants, tma=tma, nb=nb, npad=npad)


def k5_samples(N, seed=0, per_block_rows=4, per_block_cols=2):
    """Sampled rows and columns of a large fit: in every 128-block one row in each quarter (every per-CTA row range of
    panel_tile_kernel<2>, <4> and <8>) and the block's first / last live columns, so that the pairs cover the diagonal
    blocks, the in-panel tiles, the tiles behind each panel and the ragged last block without covering the matrix."""
    rng = np.random.default_rng(seed)
    nb = -(-N // FB)
    rows, cols = [], []
    for b in range(nb):
        hi = min(N, (b + 1) * FB)
        for q in range(per_block_rows):
            lo_q, hi_q = b * FB + q * FB // per_block_rows, min(hi, b * FB + (q + 1) * FB // per_block_rows)
            if lo_q < hi_q:
                rows.append(int(rng.integers(lo_q, hi_q)))
        cols += [b * FB, hi - 1][:per_block_cols]
    rows += [N - 1]
    return np.unique(rows), np.unique(cols)
