"""Reference values and proven error bounds for K7's gradients (csrc/refine.cu) and K8's likelihood (csrc/posterior_hyper.cu).

Test infrastructure; the package does not import it.  Conventions as in oracle/prior_bounds.py, posterior_bounds.py and
state_bounds.py: u = 2^-53, gamma_k = k u / (1 - k u); references in np.longdouble with their own gamma(.., u_ld) added; an
FMA or a DMMA counts as one rounding; every bound holds for any order of the additions and any fusing of a multiplication
into the following addition; first-order terms carry SLACK = 2; results in or below the subnormal range get absolute
ETA = 2^-1074 terms.  Each check covers one stage, from the inputs that stage itself read, fetched from the device.

A. Prior-gradient pass (refine_prior_kernel, one item (I, c) per CTA of m_triangle_pass.cuh).  Inputs: the points, x_obs_int,
   ls_int, M, w, s2, noise.  u_j = exp(-1/2 sum_k t_k^2), t_k = (x_k - X_kj) / l_k; the kernel forms z_k = fl(fl(x_k - X_kj) il_k)
   with il_k = fl(1 / l_k), so u carries state_bounds' RBF-entry bound du (gamma_{d+6}), and a_kj = fl(fl(u_j z_k) il_k)
   carries |da| <= du |t_k| / l_k + SLACK gamma_6 |a|.  The chain of one output, counted from m_chunks / m_row_blocks:
       the FMA chain over the item's slabs           16 min(kPassSlabs, 8 m_row_blocks)   (S_u, S_a of row n; x2 is exact)
       the row product                               1 (m, q, a.w), 2 for dv = fma(a_n, S_u, u_n S_a)
       the 5-step butterfly, the 4-warp sred sum     5 + 3
       the per-lane sum over items in index order    ceil(m_row_blocks m_chunks / 32)
       warp_sum                                      5
   m:  gamma_{n_m} sum |u||w| + sum du |w|;   dm_k = -sum a_kj w_j likewise with a, da;
   q:  gamma_{n_q} |u|^T |M| |u| + 2 du^T |M| |u|   (the u are formed in the kernel, not read from a table);
   v = fl(fl(s2 + noise) - q): two roundings more, SLACK u (|s2 + noise| + |v|);
   dv_k = sum_n a_kn S_u[n] + u_n S_a,k[n] over the lower block triangle (scale 2 left of the diagonal block) = 2 a_k^T M u:
       gamma_{n_dv} 2 |a_k|^T |M| |u| + 2 (da_k^T |M| |u| + |a_k|^T |M| du).
   M is exactly symmetric (state_bounds), so the reference uses the full matrix.

B. Posterior gradients (eval_point).  Inputs: K7's own m, v, dm, dv, the fetched L, alpha, sqrt_v_int, x_int and hyper.
   dk*_ik = fma(-e_i, fl(z_k il), fl(sv_i dv_k) hv), hv = fl(0.5 / fl(sqrt v)); the reference uses the exact 0.5 / sqrt(v)
   and posterior_bounds' k* and its bound for e (z_k = fl(fl(x_k il) - fl(x_ik il)): dq of posterior_bounds, one rounding
   more for z_k il).  The sv term carries four roundings (sqrt, /, two products), the fma one:
       |ddk*| <= de |q| il + e (dq il + SLACK u |q| il) + SLACK gamma_4 |sv dv hv| + SLACK u |dk*| + 4 ETA.
   dmu_k = dm_k + warp_sum(4-slot FMA chain of alpha_i dk*_ik): gamma_10 (|dm| + sum |alpha||dk*|) + sum |alpha| ddk*.
   beta = L^-T t by backward substitution with division, t = L^-1 k* as in posterior_bounds (dt): with L^T beta^ = t^ + e,
   |e| <= gamma_{n+3} |L^T||beta|,  |beta^ - beta_ref| <= |L^-T| (SLACK gamma_{n+3} |L^T||beta| + dt), L^-1 evaluated in
   longdouble: sharp at cond(L) = 1e10, no scaled tolerance.
   dvar_k = dv_k - 2 warp_sum(sum_r beta_i dk*_ik): gamma_10 (|dv| + 2 sum |beta||dk*|) + 2 sum (dbeta (|dk*| + ddk*) + |beta| ddk*).

C. dei = sign (phi dvar / (2 sd) - Phi dmu) from the device's (best, mu, var, dmu, dvar); phi, Phi exact in mpmath at the
   kernel's own mu^, var^.  posterior_bounds.ei_terms gives the relative errors of the kernel's phi (exp at 1 ulp, du through
   |u| phi) and Phi (erfc at 5 ulp, du through erfc's condition number), with sd's and u's roundings; then
       A = phi |dvar| / (2 sd): eps_phi + 3 u (sd, the product, the division);  B = Phi |dmu|: eps_Phi + u;
       |ddei| <= SLACK (A eps_A + B eps_B + u |A - B|) + 8 ETA (1 + (1 + |dvar|) / (2 sd) + |dmu|).
   The last term covers results in the subnormal range (u below about -37.5): phi, Phi and each product lose up to ETA, and
   the kernel forms fl(phi dvar) BEFORE dividing by 2 sd, so that product's rounding reaches dei as ETA / (2 sd).

D. dacq = (dei - acq dc) / cost, dc = sign(x_k) when the cost is variable (exactly 0 at x_k = 0), else 0: bit for bit from
   the device's dei and acq and candidate_cost's order.

E. K8 (cbo_posterior_nll).  K8's L lives in shared memory only, but it is surrogate_jitchol<256> on the same
   (x_int, sqrt(v_int), hyper) as K2's: both kernels stage x_int and sv = IEEE sqrt(v_int) unchanged, read hyper through
   surrogate_hyper, use kFitThreads == kHypThreads == 256, and jitchol's arithmetic does not depend on the row pitch (K2: n,
   K8: n | 1) nor on which thread updates an entry (each entry's updates run in column order).  So with the same hyper and the
   same jitter count (fit_info) K8's factor is K2's fetched L^, bit for bit, and K8 is bounded from it.  res = fl(y - m_int).
   z = L^-1 res and alpha = L^-T z by substitutions multiplying by rinv = fl(1 / L_ii) (one rounding more than division):
       |z^ - z| <= |L^-1| SLACK gamma_{n+3} |L^||z|,   |alpha^ - alpha| <= |L^-T| (SLACK gamma_{n+3} |L^T||alpha| + dz);
   NLL = fl(fl(0.5 zz + lg) + fl(n c)), zz = |z|^2 and lg = sum log L_ii by 4-slot chains and warp_sum (9 roundings), log at
   LOG_ULP = 1 ulp per term, c = 0.5 log(2 pi) as a double:
       |dNLL| <= SLACK [0.5 (2 sum |z| dz + gamma_9 zz) + (gamma_9 + 2 u) sum |log L_ii| + u |0.5 zz + lg| + 2 u n c + u |NLL|].
   Gradient.  X = L^-1 column by column from the right (X_ij L_jj = -sum_{j<k<=i} X_ik L_kj, by rinv): the LEFT residual
   |X^ L^ - I| <= gamma_{n+3} |X^||L^| gives |X^ - L^-1| <= SLACK gamma_{n+3} |X^||L^||L^-1|, evaluated with the longdouble L^-1.
   W_ij = sum_{k >= i} X_ki X_kj (an FMA chain): |W^ - W| <= gamma_n |X^|^T|X^| + |dX|^T |X^| + |X^|^T |dX|.  Each pair i >= j
   contributes c_ij = h (W_ij - alpha_i alpha_j) s2 E_ij (h = 1/2 on the diagonal, exact) and c_ij r2_ij, r2 with
   gamma_{d+5} (posterior_bounds' Gram), s2 E with its E_gram; the rounding of alpha_i alpha_j and of the difference, of the
   product by s2 E, and of c r2 are one each.  The sums run per thread over ceil(n^2 / 256) pairs, a butterfly and 8 warps:
   n_g = ceil(n^2 / 256) + 5 + 8, and |dg| <= gamma_{n_g} sum |terms| + sum |term errors|.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import posterior_bounds as P
from oracle import state_bounds as SB
from oracle.prior_bounds import ETA, U, U_LD, _ratio, gamma

LD = np.longdouble
SLACK = 2.0
LOG_ULP = 1
HALF_LOG_2PI = np.float64(0.91893853320467274178)

# csrc/m_triangle_pass.cuh and refine.cu
PASS_THREADS = 128            # kPassThreads = kMBlkRows
BK = 16                       # columns per slab
SLABS_PER_BLOCK = PASS_THREADS // BK
PASS_SLABS = 32               # kPassSlabs
WARPS = PASS_THREADS // 32
REF_B = 8                     # kRefB
HYP_THREADS = 256             # kHypThreads


def g2(k, k_ld=None):
    return gamma(k) + gamma(k if k_ld is None else k_ld, U_LD)


# ---- geometry of the pass (m_triangle_pass.cuh) -------------------------------------------------------------------------
def m_row_blocks(N):
    return -(-N // PASS_THREADS)


def m_chunks(N):
    return -(-(m_row_blocks(N) * SLABS_PER_BLOCK) // PASS_SLABS)


def m_item_exists(I, c):
    return c * PASS_SLABS < (I + 1) * SLABS_PER_BLOCK


def item_slabs(I, c):
    """(kt0, kt1, diag0) of item (I, c)."""
    kt0 = c * PASS_SLABS
    return kt0, min(kt0 + PASS_SLABS, (I + 1) * SLABS_PER_BLOCK), I * SLABS_PER_BLOCK


def pass_counts(N):
    """Roundings on the path of one term of m (and dm), q and dv (module docstring, A)."""
    R, C = m_row_blocks(N), m_chunks(N)
    chain = BK * min(PASS_SLABS, SLABS_PER_BLOCK * R)
    tail = 5 + (WARPS - 1) + -(-(R * C) // 32) + 5
    return dict(m=1 + tail, q=chain + 1 + tail, dv=chain + 2 + tail)


# ---- A: the prior-gradient pass ------------------------------------------------------------------------------------------
def prior_pass_ref(X, x_obs, ls, M, w, s2, noise):
    """Reference m, v, dm, dv (longdouble) at points X (P x d) and their bounds (float64)."""
    X, x_obs = np.atleast_2d(np.asarray(X, np.float64)), np.atleast_2d(np.asarray(x_obs, np.float64))
    ls = np.asarray(ls, np.float64).reshape(-1)
    N, d = x_obs.shape
    M, w = np.asarray(M, np.float64), np.asarray(w, np.float64)
    u, _, du = SB.rbf_ref(X, x_obs, ls)                                       # P x N
    t = (X[:, None, :].astype(LD) - x_obs[None, :, :].astype(LD)) / ls.astype(LD)
    a = u[:, :, None] * t / ls.astype(LD)                                     # P x N x d
    Ml = M.astype(LD)
    Mu = u @ Ml
    base = LD(s2) + LD(noise)
    ref = dict(m=u @ w.astype(LD), v=base - (u * Mu).sum(1), dm=-np.einsum("pnk,n->pk", a, w.astype(LD)),
               dv=2 * np.einsum("pnk,pn->pk", a, Mu))
    uf, af = np.abs(u).astype(np.float64) + du, np.abs(a).astype(np.float64)
    da = du[:, :, None] * np.abs(t).astype(np.float64) / ls + SLACK * gamma(6) * af + 4.0 * ETA
    af = af + da
    aM = np.abs(M)
    Mabs_u = uf @ aM
    Mabs_du = du @ aM
    n = pass_counts(N)
    own = N + d + 16                                                          # the longdouble reference's own depth
    wa = np.abs(w)
    Mmax, wmax = float(aM.max(initial=0.0)), float(wa.max(initial=0.0))
    e_m = g2(n["m"], own) * (uf @ wa) + du @ wa + 4.0 * N * ETA * max(1.0, wmax)
    e_q = g2(n["q"], own) * (uf * Mabs_u).sum(1) + 2.0 * (du * Mabs_u).sum(1) + 4.0 * N * N * ETA * max(1.0, Mmax)
    e_v = e_q + SLACK * U * (abs(float(s2) + float(noise)) + np.abs(ref["v"]).astype(np.float64))
    e_dm = g2(n["m"], own) * np.einsum("pnk,n->pk", af, wa) + np.einsum("pnk,n->pk", da, wa) + 4.0 * N * ETA * max(1.0, wmax)
    e_dv = (g2(n["dv"], own) * 2.0 * np.einsum("pnk,pn->pk", af, Mabs_u)
            + 2.0 * (np.einsum("pnk,pn->pk", da, Mabs_u) + np.einsum("pnk,pn->pk", af, Mabs_du))
            + 8.0 * N * N * ETA * max(1.0, Mmax))
    ref.update(e_m=e_m, e_v=e_v, e_dm=e_dm, e_dv=e_dv, q_abs=(uf * Mabs_u).sum(1))
    return ref


def _worst(got, ref, bound):
    err = np.abs(np.asarray(got, np.float64).astype(LD) - ref).astype(np.float64)
    return float(np.max(_ratio(err, bound), initial=0.0))


def check_prior_pass(out, ref):
    """Worst |error| / bound of m, v, dm, dv (dicts of arrays; dm, dv P x d)."""
    return {k: _worst(out[k], ref[k], ref["e_" + k]) for k in ("m", "v", "dm", "dv")}


# ---- B: eval_point -----------------------------------------------------------------------------------------------------------
def grad_ref(X, m, v, dm, dv, st):
    """Reference mu, var, dmu, dvar (longdouble) and bounds at points X from K7's own m, v, dm, dv.
    st: dict(x_int, sv, alpha, L, s2, l, causal) as fetched."""
    X = np.atleast_2d(np.asarray(X, np.float64))
    m, v = np.asarray(m, np.float64), np.asarray(v, np.float64)
    dm, dv = np.asarray(dm, np.float64), np.asarray(dv, np.float64)
    XI = np.asarray(st["x_int"], np.float64)
    n, d = XI.shape
    sv = np.asarray(st["sv"], np.float64)
    s2, il = float(st["s2"]), P.inv_l(st["l"])
    causal = bool(st["causal"])
    post = P.posterior_ref_block(X, m, v, st, "subst")
    e, de = P.kstar_ref(X, XI, np.zeros(n), np.zeros(len(X)), s2, st["l"], False)      # s2 exp(-r2 / 2) alone
    ilL = LD(il)
    q = (X[:, None, :].astype(LD) * ilL - XI[None, :, :].astype(LD) * ilL)              # P x n x d
    hv = (LD(0.5) / np.sqrt(v.astype(LD))) if causal else np.zeros(len(X), LD)
    sec = sv.astype(LD)[None, :, None] * dv.astype(LD)[:, None, :] * hv[:, None, None]
    dks = -e[:, :, None] * q * ilL + sec
    qf, ef = np.abs(q).astype(np.float64), np.abs(e).astype(np.float64)
    dq = SLACK * U * ((np.abs(X)[:, None, :] + np.abs(XI)[None, :, :]) * il + qf)
    ddk = (de[:, :, None] * qf * il + ef[:, :, None] * (dq * il + SLACK * U * qf * il)
           + SLACK * gamma(4) * np.abs(sec).astype(np.float64) + SLACK * U * np.abs(dks).astype(np.float64) + 4.0 * ETA)
    al = np.asarray(st["alpha"], np.float64)
    dkf = np.abs(dks).astype(np.float64) + ddk
    dmu = dm.astype(LD) + np.einsum("i,pik->pk", al.astype(LD), dks)
    e_dmu = g2(10, n + 16) * (np.abs(dm) + np.einsum("i,pik->pk", np.abs(al), dkf)) + np.einsum("i,pik->pk", np.abs(al), ddk)
    L = np.tril(np.asarray(st["L"], np.float64))
    Li = st.get("Linv_ld")
    if Li is None:
        Li = st["Linv_ld"] = P.lower_inverse_ld(L)
    beta = post["t"] @ Li                                                                # L^-T t, row per point
    bf = np.abs(beta).astype(np.float64)
    dbeta = (SLACK * g2(n + 3) * (bf @ np.abs(L)) + post["dt"]) @ np.abs(Li).astype(np.float64)
    bf = bf + dbeta
    dvar = dv.astype(LD) - 2 * np.einsum("pi,pik->pk", beta, dks)
    e_dvar = (g2(10, n + 16) * (np.abs(dv) + 2.0 * np.einsum("pi,pik->pk", bf, dkf))
              + 2.0 * (np.einsum("pi,pik->pk", dbeta, dkf) + np.einsum("pi,pik->pk", bf, ddk)))
    return dict(mu=post["mu"], var=post["var"], e_mu=post["e_mu"], e_var=post["e_var"], dmu=dmu, dvar=dvar, e_dmu=e_dmu,
                e_dvar=e_dvar, beta=beta)


def check_grad(out, ref):
    return {k: _worst(out[k], ref[k], ref["e_" + k]) for k in ("mu", "var", "dmu", "dvar")}


# ---- C: dei --------------------------------------------------------------------------------------------------------------------
def dei_exact(best, mu, var, dmu, dvar, task_sign, dps=40):
    """sign (phi(u) dvar / (2 sd) - Phi(u) dmu) at the kernel's own (mu, var), exactly (mpf, P x d nested lists).  best: one
    incumbent, or one per point."""
    import mpmath as mp
    mp.mp.dps = dps
    out = []
    mu = np.asarray(mu, np.float64)
    bests = np.broadcast_to(np.asarray(best, np.float64), mu.shape)
    for b_, m_, v_, gm, gv in zip(bests, mu, np.asarray(var, np.float64), np.atleast_2d(dmu), np.atleast_2d(dvar)):
        sd = mp.sqrt(mp.mpf(float(v_)))
        u = (mp.mpf(float(b_)) - mp.mpf(float(m_))) / sd
        phi = mp.exp(-u * u / 2) / mp.sqrt(2 * mp.pi)
        Phi = mp.erfc(-u / mp.sqrt(2)) / 2
        out.append([task_sign * (phi * mp.mpf(float(a)) / (2 * sd) - Phi * mp.mpf(float(c))) for c, a in zip(gm, gv)])
    return out


def dei_bound(best, mu, var, dmu, dvar):
    t = P.ei_terms(best, mu, var)
    sd, phi, Phi = t["sd"][:, None], t["phi"][:, None], t["Phi"][:, None]
    dmu, dvar = np.abs(np.atleast_2d(dmu)), np.abs(np.atleast_2d(dvar))
    with np.errstate(all="ignore"):
        A = phi * dvar / (2.0 * sd)
        B = Phi * dmu
        return (SLACK * (A * (t["eps_phi"][:, None] + 3.0 * U) + B * (t["eps_Phi"][:, None] + U) + U * np.abs(A - B))
                + 8.0 * ETA * (1.0 + (1.0 + dvar) / (2.0 * sd) + dmu))


def check_dei(dei, best, mu, var, dmu, dvar, task_sign):
    import mpmath as mp
    dei = np.atleast_2d(np.asarray(dei, np.float64))
    ex = dei_exact(best, mu, var, dmu, dvar, task_sign)
    err = np.array([[float(abs(mp.mpf(float(g)) - r)) if np.isfinite(g) else np.inf for g, r in zip(gr, rr)]
                    for gr, rr in zip(dei, ex)])
    return float(np.max(_ratio(err, dei_bound(best, mu, var, dmu, dvar)), initial=0.0))


# ---- D: dacq -------------------------------------------------------------------------------------------------------------------
def dacq_ref(dei, acq, X, cost_fix, cost_variable):
    """(dei - acq dc) / cost in eval_point's order, bit for bit."""
    X = np.atleast_2d(np.asarray(X, np.float64))
    cost = P.candidate_cost(X, cost_fix, cost_variable)
    dc = np.sign(X) if cost_variable else np.zeros_like(X)
    return (np.asarray(dei, np.float64) - np.asarray(acq, np.float64)[:, None] * dc) / cost[:, None]


# ---- E: K8 ---------------------------------------------------------------------------------------------------------------------
def k8_ref(L, x_int, res, s2, l):
    """Reference NLL, g0, g1 (longdouble) from K2's fetched factor L^ and their bounds.  res = fl(y - m_int) (or y)."""
    L = np.tril(np.asarray(L, np.float64))
    n = L.shape[0]
    d = np.asarray(x_int).shape[1]
    res = np.asarray(res, np.float64)
    Li = P.lower_inverse_ld(L)
    Lab, Lia = np.abs(L), np.abs(Li).astype(np.float64)
    z = Li @ res.astype(LD)
    zf = np.abs(z).astype(np.float64)
    dz = Lia @ (SLACK * g2(n + 3) * (Lab @ zf))
    al = Li.T @ z
    af = np.abs(al).astype(np.float64)
    dal = Lia.T @ (SLACK * g2(n + 3) * (Lab.T @ af) + dz)
    zz = (z * z).sum()
    lgs = np.log(np.diag(L).astype(LD))
    lg = lgs.sum()
    nc = LD(n) * LD(HALF_LOG_2PI)
    nll = 0.5 * zz + lg + nc
    lga = float(np.abs(lgs).sum())
    e_nll = SLACK * (0.5 * (float((2.0 * zf + dz) @ dz) + g2(9, n + 8) * float(zz)) + (g2(9, n + 8) + 2 * LOG_ULP * U) * lga
                     + U * abs(float(0.5 * zz + lg)) + 2.0 * U * float(nc) + U * abs(float(nll)))
    # gradient
    X = Li                                                                   # the longdouble L^-1 stands for X^ to first order
    Xa = Lia
    dX = SLACK * g2(n + 3) * (Xa @ Lab @ Lia) + 4.0 * (n + 4) * ETA
    Xa2 = Xa + dX
    W = X.T @ X
    dW = g2(n, n + 8) * (Xa2.T @ Xa2) + dX.T @ Xa2 + Xa2.T @ dX
    Kref, E = P.gram_ref(x_int, np.zeros(n), s2, l, 0.0)
    sE = Kref - np.diag(np.full(n, LD(P.K_DIAG)))
    sEf = np.abs(sE).astype(np.float64)
    XI = np.asarray(x_int, np.float64)
    Dl = (XI[:, None, :].astype(LD) - XI[None, :, :].astype(LD)) * LD(P.inv_l(l))
    r2 = np.einsum("ijk,ijk->ij", Dl, Dl)
    r2f = r2.astype(np.float64)
    aa = np.outer(al, al)
    D = W - aa
    Df = np.abs(D).astype(np.float64)
    aaf = np.outer(af, af)
    dD = dW + np.outer(dal, af) + np.outer(af, dal) + 2.0 * U * (np.abs(W).astype(np.float64) + aaf) + U * Df
    h = np.tril(np.ones((n, n))) - 0.5 * np.eye(n)
    c = LD(1) * h * D * sE
    cf = np.abs(c).astype(np.float64)
    dc = h * (dD * (sEf + E) + Df * E + U * Df * sEf)
    dr2 = SLACK * gamma(d + 5) * r2f
    ng = -(-n * n // HYP_THREADS) + 5 + 8 + 2
    g0 = c.sum()
    g1 = (c * r2).sum()
    e_g0 = g2(ng, n * n + 8) * float(cf.sum()) + float(dc.sum()) + 4.0 * n * n * ETA
    e_g1 = g2(ng + 1, n * n + 8) * float((cf * r2f).sum()) + float((dc * r2f + cf * dr2).sum()) + 4.0 * n * n * ETA
    return dict(nll=nll, g0=g0, g1=g1, e_nll=e_nll, e_g0=e_g0, e_g1=e_g1, z=z, alpha=al, W=W)


def check_k8(out, ref):
    """Worst |error| / bound of (NLL, g0, g1) = out."""
    return {k: _worst(np.array([out[i]]), np.array([ref[k]]), np.array([ref["e_" + k]])) for i, k in enumerate(("nll", "g0", "g1"))}


# ---- cancellation at the interventional rows ------------------------------------------------------------------------------
def exact_v_dv(x, x_obs, ls, M, s2, noise, with_dv=True):
    """v = fl(s2 + noise) - u^T M u and dv_k = 2 a_k^T M u at the point x, correctly rounded from u and a evaluated in
    longdouble (exact 1 / l) and carried as double-double (hi + lo) into math.fsum over TwoProd splits."""
    from oracle.prior_bounds import two_prod
    x, x_obs = np.asarray(x, np.float64), np.atleast_2d(np.asarray(x_obs, np.float64))
    ls, M = np.asarray(ls, np.float64).reshape(-1), np.asarray(M, np.float64)
    t = (x[None, :].astype(LD) - x_obs.astype(LD)) / ls.astype(LD)
    u = np.exp(-0.5 * (t * t).sum(1))
    a = (u[:, None] * t / ls.astype(LD)).T

    def split(z):
        hi = z.astype(np.float64)
        return hi, (z - hi.astype(LD)).astype(np.float64)

    def quad(p, q):
        out = []
        for x_ in split(p):
            for y_ in split(q):
                p1, e1 = two_prod(x_[:, None], M)
                h1, l1 = two_prod(p1, y_[None, :])
                h2, l2 = two_prod(e1, y_[None, :])
                out += [h1.ravel(), l1.ravel(), h2.ravel(), l2.ravel()]
        return np.concatenate(out)

    v = math.fsum(np.concatenate([[np.float64(s2) + np.float64(noise)], -quad(u, u)]))
    if not with_dv:
        return v
    return v, np.array([2.0 * math.fsum(quad(ak, u)) for ak in a])
