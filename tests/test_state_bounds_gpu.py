"""The kernels that produce the causal prior's state against the error bounds of oracle/state_bounds.py, on every launch
shape they have: K5 (obs_gp_fit.cu: Gram, panelled Cholesky, Wt = L^-T, Ky^-1, alpha, NLL), K1a (prior_precompute.cu: P,
pbar, w, M) and K0 (tables.cu).

Every output, the K5 workspace, P, M and the tables start as NaN, so an unwritten entry fails instead of passing on stale
memory, and every case runs twice with bit-identical results.  state_bounds.k5_plan mirrors obs_gp_fit_impl's panel loop
and launch_panel_op's split of a tile over 4, 2 or 1 CTAs (panel_tile_kernel<2>, <4>, <8>); _own mirrors
prior_precompute's own_launches; each case asserts the path it was built for and the launch count that goes with it.  The
K5 sizes that reach <4> and <8> are derived from the SM count.  Large fits are checked on sampled rows and columns that
cover every tile class (state_bounds.k5_samples).  Run with -s to see each case's worst error as a fraction of its bound."""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from helpers import make_case
from oracle import state_bounds as B

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FB = 128
FULL_N = 641          # up to here every entry is checked; beyond, k5_samples


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _nb_for(sms, variant):
    """The smallest number of blocks whose in-panel products reach panel_tile_kernel<variant> (2 tiles <= sms < 4 tiles:
    <4>; 2 tiles > sms: <8>); the products launch at most nb - 1 tiles."""
    return (sms // 4 + 1) + 1 if variant == 4 else (sms // 2 + 1) + 1


# ---- K5 -----------------------------------------------------------------------------------------------------------------
def _data(seed, N, D):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    y = np.sin(X @ rng.uniform(-1, 1, D)) + 0.1 * rng.standard_normal(N)
    return X, y, float(rng.uniform(0.6, 1.6)), rng.uniform(0.7, 1.8, D)


def _fit(X, y, s2, ls, noise):
    """Two fits from NaN (workspace, alpha, Ky^-1); identical bits.  Returns the state on the host and launches per fit."""
    import torch
    from cbo_with_oop_b200.obs_gp import DeviceObsGP
    gp = DeviceObsGP(X, y, noise)
    runs = []
    for _ in range(2):
        gp.ws.fill_(0xFF)
        gp.alpha.fill_(float("nan"))
        gp.kyinv.fill_(float("nan"))
        gp.out.fill_(float("nan"))
        l0 = gp.lib.cbo_launch_count()
        tries = gp.fit(s2, ls)
        torch.cuda.synchronize()
        launches = gp.lib.cbo_launch_count() - l0
        nll = gp.nll_grad()
        runs.append((tries, launches, gp.ws.clone(), gp.alpha.clone(), gp.kyinv.clone(), gp.out.clone(), nll))
    (t1, l1, w1, a1, k1, o1, _), (t2, l2, w2, a2, k2, o2, _) = runs
    assert t1 == t2 and l1 == l2
    for a, b, name in ((w1, w2, "workspace"), (a1, a2, "alpha"), (k1, k2, "Ky^-1"), (o1, o2, "nll")):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), f"{name} differs between two identical fits"
    npad = gp.h[0].n_obs_pad
    nws = B.split_ws(w1.view(torch.float64)[:2 * npad * npad + (npad // FB) * FB * FB + npad].cpu().numpy(), npad)
    del runs, w2
    return dict(tries=t1, launches=l1, A=nws[0], Wt=nws[1], Linv=nws[2], z=nws[3], alpha=a1.cpu().numpy(),
                kyinv=k1.cpu().numpy(), out=o1.cpu().numpy(), npad=npad)


def _check_k5(st, X, y, s2, ls, noise, label, nll=False):
    N = X.shape[0]
    npad = st["npad"]
    jit = B.jitter_k5(st["tries"], s2, noise)
    dadd = B.diag_add(noise, jit)
    if N <= FULL_N:
        rows = cols = np.arange(N)
    else:
        rows, cols = B.k5_samples(N, seed=N)
    blocks = range(npad // FB)
    r = {}
    r["gram"], pairs = B.check_gram_upper(st["A"], X, s2, ls, dadd, rows, cols)
    r["linv"] = B.check_linv(st["A"], st["Linv"], blocks)
    r["chol"] = B.check_chol(st["A"], st["Linv"], X, s2, ls, dadd, rows, cols)
    r["wt"] = B.check_wt(st["A"], st["Wt"], st["Linv"], rows, cols)
    r["kyinv"] = B.check_kyinv(st["kyinv"], st["Wt"], rows, cols)
    r["z"], r["alpha"] = B.check_alpha(st["Wt"], y, st["z"], st["alpha"], ks=cols if N > FULL_N else None,
                                       rows=rows if N > FULL_N else None)
    if nll:
        r["nll"], r["grad"] = B.check_nll(st["out"], st["alpha"], y, np.diag(st["A"])[:N], X, st["kyinv"], s2, ls)
    print(f"  K5 {label} (N={N}, D={X.shape[1]}, tries={st['tries']}, upper Gram pairs {pairs}): "
          + "  ".join(f"{k} {v:.2e}" for k, v in r.items()))
    bad = {k: v for k, v in r.items() if not v <= 1.0}
    assert not bad, (label, bad)
    return r


def _k5_cases():
    sms = _sms()
    n4 = _nb_for(sms, 4) * FB - 100          # nb = first <4> block count, a ragged last block
    n8 = max(10000, _nb_for(sms, 8) * FB - 100)
    return sms, [1, 2, 127, 128, 129, 511, 512, 513, 641, 1025, 2049, n4, n8]


K5_N = ["1", "2", "127", "128", "129", "511", "512", "513", "641", "1025", "2049", "first_4", "first_8"]
NLL_N = {1, 129, 641, 2049}


@pytest.mark.parametrize("case", K5_N)
def test_k5_launch_shapes(cuda_engine_ready, case):
    sms, ns = _k5_cases()
    N = ns[K5_N.index(case)]
    D = 12 if K5_N.index(case) % 2 or N in (129, 2049) else 1
    X, y, s2, ls = _data(3000 + N, N, D)
    st = _fit(X, y, s2, ls, 1e-2)
    plan = B.k5_plan(N, sms)
    assert st["tries"] == 0
    assert st["launches"] == plan["launches"], (st["launches"], plan)
    if case == "513":
        assert plan["tma"] == ["syrk", "winv"]               # first trailing TMA syrk and winv update; last panel of one block
    if case == "641":
        assert plan["nb"] % 4 == 2                           # a last panel of two blocks
    if case == "first_4":
        assert 4 in plan["variants"] and 8 not in plan["variants"]
    if case == "first_8":
        assert plan["variants"] == {2, 4, 8}
    _check_k5(st, X, y, s2, ls, 1e-2, case, nll=N in NLL_N)


def test_k5_jitter_retry(cuda_engine_ready):
    """test_jitter_retry_rule's case: the jitter of the successful attempt is reproduced bit for bit in Ky_ref."""
    X, y, _, ls = _data(8, 140, 2)
    X[70:] = X[:70]
    st = _fit(X, y, 1e12, ls, 0.0)
    assert st["tries"] >= 1
    assert st["launches"] == B.k5_plan(140, _sms())["launches"] * (st["tries"] + 1)
    _check_k5(st, X, y, 1e12, ls, 0.0, "jitter retry")


_PANEL_SCRIPT = r"""
import json, sys
import numpy as np
import torch
from cbo_with_oop_b200.obs_gp import DeviceObsGP
a = json.loads(sys.argv[1])
X, y = np.load(a["x"]), np.load(a["y"])
gp = DeviceObsGP(X, y, a["noise"])
out = []
for _ in range(2):
    gp.ws.fill_(0xFF); gp.alpha.fill_(float("nan")); gp.kyinv.fill_(float("nan"))
    l0 = gp.lib.cbo_launch_count()
    tries = gp.fit(a["s2"], np.array(a["ls"]))
    torch.cuda.synchronize()
    out.append((tries, gp.lib.cbo_launch_count() - l0, gp.ws.cpu().numpy().copy(), gp.alpha.cpu().numpy(), gp.kyinv.cpu().numpy()))
assert out[0][0] == out[1][0] and out[0][1] == out[1][1]
for k in (2, 3, 4):
    assert np.array_equal(out[0][k], out[1][k])
np.savez(a["out"], tries=out[0][0], launches=out[0][1], ws=out[0][2], alpha=out[0][3], kyinv=out[0][4])
"""


@pytest.mark.parametrize("width", [1, 3])
def test_k5_panel_width(cuda_engine_ready, width):
    """CBO_FIT_PANEL = 1 and 3 at N = 1025 (read once per process, so each runs in a subprocess): the same bounds hold."""
    N = 1025
    X, y, s2, ls = _data(4000 + width, N, 5)
    with tempfile.TemporaryDirectory() as td:
        np.save(os.path.join(td, "x.npy"), X)
        np.save(os.path.join(td, "y.npy"), y)
        arg = dict(x=os.path.join(td, "x.npy"), y=os.path.join(td, "y.npy"), noise=1e-2, s2=s2, ls=list(ls),
                   out=os.path.join(td, "o.npz"))
        env = dict(os.environ, CBO_FIT_PANEL=str(width), PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
        subprocess.run([sys.executable, "-c", _PANEL_SCRIPT, json.dumps(arg)], cwd=ROOT, env=env, check=True, timeout=600)
        o = np.load(arg["out"])
        npad = -(-N // FB) * FB
        A, Wt, Linv, z = B.split_ws(o["ws"].view(np.float64), npad)
        st = dict(tries=int(o["tries"]), A=A, Wt=Wt, Linv=Linv, z=z, alpha=o["alpha"], kyinv=o["kyinv"], npad=npad)
        assert st["tries"] == 0
        assert int(o["launches"]) == B.k5_plan(N, _sms(), width)["launches"]
        _check_k5(st, X, y, s2, ls, 1e-2, f"panel width {width}")


# ---- K1a ----------------------------------------------------------------------------------------------------------------
def _engine(specs):
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    eng = SweepEngine([SetProblem(**make_case(**s)[0]) for s in specs])
    return eng


def _nan_k1a(eng):
    for li, g in enumerate(eng.active):
        for k in ("M", "pbar", "w", "P"):
            if k in eng.buf[li]:
                eng.buf[li][k].fill_(float("nan"))
    if eng.P is not None:
        eng.P.fill_(float("nan"))


def _precompute(eng, ids=None):
    import torch
    _nan_k1a(eng)
    l0 = eng.launches
    eng.prior_precompute(ids)
    torch.cuda.synchronize()
    return eng.launches - l0


def _k1a_state(eng, li):
    D, b = eng.h_sets[li], eng.buf[li]
    npad, spad = D.n_obs_pad, D.n_mc_pad
    out = dict(M=B.unblock_m(b["M"].cpu().numpy(), npad), pbar=b["pbar"].cpu().numpy()[:D.n_obs], w=b["w"].cpu().numpy()[:D.n_obs])
    if D.c:
        nbytes = npad * spad
        out["P"] = _view(D.P, npad * spad).cpu().numpy().reshape(npad, spad)
    return out


def _view(ptr, n):
    """The float64 tensor view of n doubles at device address ptr (the P scratch a descriptor points to)."""
    for t in _P_OWNERS:
        base = t.data_ptr()
        if base <= ptr and ptr + 8 * n <= base + 8 * t.numel():
            off = (ptr - base) // 8
            return t[off:off + n]
    raise LookupError("P pointer of no known buffer")


_P_OWNERS = []


def _register_p(eng):
    _P_OWNERS.clear()
    if eng.P is not None:
        _P_OWNERS.append(eng.P)
    for b in eng.buf:
        if "P" in b:
            _P_OWNERS.append(b["P"])


def _own(eng, li, sms):
    """prior_precompute.cu own_launches."""
    D = eng.h_sets[li]
    nT = D.n_obs_pad // FB
    if nT * (nT + 1) // 2 >= sms:
        return True
    e0 = D.P + D.n_obs_pad * D.n_mc_pad * 8
    for t in range(len(eng.active)):
        T = eng.h_sets[t]
        if t == li or not T.c:
            continue
        if D.P < T.P + T.n_obs_pad * T.n_mc_pad * 8 and T.P < e0:
            return True
    return False


def _check_k1a(eng, li, label, rows=None):
    D = eng.h_sets[li]
    pr = eng.problems[eng.active[li]]
    st = _k1a_state(eng, li)
    kyinv = eng.fetch("kyinv", eng.active[li]).reshape(D.n_obs, D.n_obs)
    alpha = eng.fetch("alpha_obs", eng.active[li])[:D.n_obs]
    if D.c == 0:
        B.check_nocond(st["M"], st["pbar"], st["w"], kyinv, D.s2, alpha)
        print(f"  K1a {label} set {li} (c=0, N={D.n_obs}): bit for bit")
        return
    N = D.n_obs
    xc, mc = np.asarray(pr.x_obs_cond), np.asarray(pr.mc_cond)
    ls = np.array([D.ls_cond[k] for k in range(D.c)])
    rp = B.check_p(st["P"], mc, xc, ls, D.n_mc, rows=rows)
    rb = B.check_pbar_w(st["P"][:N] if rows is None else st["P"][rows], st["pbar"] if rows is None else st["pbar"][rows],
                        st["w"] if rows is None else st["w"][rows], D.n_mc, D.s2, alpha if rows is None else alpha[rows])
    rm = B.check_m(st["M"], st["P"][:N], kyinv, D.s2, D.n_mc, rows=rows, cols=rows)
    print(f"  K1a {label} set {li} (c={D.c}, N={N}, S_mc={D.n_mc}): P {rp:.2e}  pbar {rb:.2e}  M {rm:.2e}")
    assert rp <= 1.0 and rb <= 1.0 and rm <= 1.0, (label, li, rp, rb, rm)
    return st


def _alone(eng, ids, first):
    """Each set run alone gives the bits it had among the others."""
    for li in ids:
        _precompute(eng, [li])
        st = _k1a_state(eng, li)
        for k, v in first[li].items():
            np.testing.assert_array_equal(st[k], v, err_msg=f"set {li}: {k} alone differs")


def test_k1a_batched_and_nocond(cuda_engine_ready):
    """Batched cp.async sets with c = 1..8 and S_mc in {1, 15, 16, 17, 33}, mixed with two sets without conditioning
    columns (nocond_kernel): one nocond launch, one pgen and one syrk launch for all conditioned sets."""
    smc = [1, 15, 16, 17, 33, 17, 16, 15]
    specs = [dict(seed=1100 + c, N=90 + 37 * c, d=1 + c % 3, c=c, n=2, p=(4,) * (1 + c % 3), S_mc=smc[c - 1]) for c in range(1, 9)]
    specs.insert(3, dict(seed=1190, N=140, d=2, c=0, n=2, p=(4, 4)))
    specs.append(dict(seed=1191, N=129, d=1, c=0, n=2, p=(6,)))
    eng = _engine(specs)
    _register_p(eng)
    sms = _sms()
    ids = list(range(len(specs)))
    assert not any(_own(eng, i, sms) for i in ids if eng.h_sets[i].c)
    runs = []
    for _ in range(2):
        launches = _precompute(eng)
        assert launches == 3, launches
        runs.append({li: _k1a_state(eng, li) for li in ids})
    for li in ids:
        for k in runs[0][li]:
            np.testing.assert_array_equal(runs[0][li][k], runs[1][li][k], err_msg=f"set {li} {k}: two runs differ")
    for li in ids:
        _check_k1a(eng, li, "batched")
    _alone(eng, ids, runs[0])


def test_k1a_shared_p_own_launches(cuda_engine_ready):
    """Three conditioned sets whose descriptors point at ONE P scratch (the engine's layout for large sets): each takes
    launches of its own (pgen + syrk), stream-ordered."""
    import torch
    specs = [dict(seed=1200 + j, N=150 + 100 * j, d=2, c=1 + j, n=2, p=(4, 4), S_mc=17 + 16 * j) for j in range(3)]
    eng = _engine(specs)
    npad = max(eng.h_sets[i].n_obs_pad for i in range(3))
    spad = max(eng.h_sets[i].n_mc_pad for i in range(3))
    shared = torch.empty((npad * spad,), dtype=torch.float64, device=eng.device)
    for i in range(3):
        eng.h_sets[i].P = shared.data_ptr()
    eng._descs_dirty = True
    eng.P = shared
    _P_OWNERS.clear()
    _P_OWNERS.append(shared)
    sms = _sms()
    assert all(_own(eng, i, sms) for i in range(3))
    assert _precompute(eng) == 6
    Ms = []
    for i in range(3):       # P holds the last set's rows only; check M / pbar of each set from its own rerun
        _precompute(eng, [i])
        st = _check_k1a(eng, i, "shared P")
        Ms.append(st["M"])
    assert _precompute(eng) == 6
    for i in range(3):
        np.testing.assert_array_equal(_k1a_state(eng, i)["M"], Ms[i], err_msg=f"set {i}: M differs from the set run alone")


@pytest.mark.parametrize("N,S_mc", [(2049, 17), (2049, 10000), (2176, 17), (2176, 10000)])
def test_k1a_tma_syrk(cuda_engine_ready, N, S_mc):
    """A set whose block triangle fills the GPU: pgen + the TMA syrk (PriorSyrkPlan).  N = 2049 has one live row in its
    last block.  Checked on sampled rows x columns of every block (all tile classes, mirrored tiles included)."""
    eng = _engine([dict(seed=1300 + N + S_mc, N=N, d=1, c=2, n=2, p=(5,), S_mc=S_mc)])
    _register_p(eng)
    sms = _sms()
    D = eng.h_sets[0]
    nT = D.n_obs_pad // FB
    assert nT * (nT + 1) // 2 >= sms and _own(eng, 0, sms)
    first = None
    for _ in range(2):
        assert _precompute(eng) == 2
        st = _k1a_state(eng, 0)
        if first is None:
            first = st
        else:
            for k in st:
                np.testing.assert_array_equal(st[k], first[k])
    rows, _ = B.k5_samples(N, seed=N, per_block_rows=2)
    _check_k1a(eng, 0, f"TMA syrk N={N}", rows=rows)


# ---- K0 -----------------------------------------------------------------------------------------------------------------
def _tables_check(eng, li, label):
    D, b, pr = eng.h_sets[li], eng.buf[li], eng.problems[eng.active[li]]
    npad = D.n_obs_pad
    X = np.asarray(pr.x_obs_int)
    ls = np.array([D.ls_int[k] for k in range(D.d)])
    worst = 0.0
    for k in range(D.d):
        tab = b[f"tab{k}"].cpu().numpy().reshape(D.p[k], npad)
        worst = max(worst, B.check_table(tab, np.asarray(pr.grid[k])[:, None], X[:, k:k + 1], ls[k:k + 1]))
    u = b["u_int"].cpu().numpy()[:D.n_int * npad].reshape(D.n_int, npad)
    worst = max(worst, B.check_table(u, np.asarray(pr.x_int), X, ls))
    print(f"  K0 {label} set {li} (d={D.d}, N={D.n_obs}, p={[D.p[k] for k in range(D.d)]}): {worst:.2e}")
    assert worst <= 1.0, (label, li, worst)


def test_k0_tables(cuda_engine_ready):
    """d = 1..4, grids with p = 1, 128, 129, N = 127 and 129, in one launch; the same bits twice."""
    import torch
    specs = []
    for d in range(1, 5):
        for N in (127, 129):
            p = tuple([1, 128, 129, 7][(d + j + N) % 4] if d < 4 else [1, 128, 3, 129][j] for j in range(d))
            specs.append(dict(seed=1400 + 10 * d + N % 2, N=N, d=d, c=1, n=5, p=p))
    eng = _engine(specs)
    runs = []
    for _ in range(2):
        for b in eng.buf:
            for k, v in b.items():
                if k.startswith("tab") or k == "u_int":
                    v.fill_(float("nan"))
        l0 = eng.launches
        eng.build_tables()
        torch.cuda.synchronize()
        assert eng.launches - l0 == 1
        runs.append([{k: v.cpu().numpy().copy() for k, v in b.items() if k.startswith("tab") or k == "u_int"} for b in eng.buf])
    for a, b in zip(*runs):
        for k in a:
            np.testing.assert_array_equal(a[k], b[k])
    for li in range(len(specs)):
        _tables_check(eng, li, "grid")


def test_k0_explicit_points(cuda_engine_ready):
    """The explicit-point table (table 0, one row per point) of a 3-D set, from NaN."""
    import torch
    from cbo_with_oop_b200 import _lib
    from cbo_with_oop_b200._lib import SetDesc
    eng = _engine([dict(seed=1450, N=129, d=3, c=1, n=2, p=(3, 3, 3))])
    D0, dev = eng.h_sets[0], eng.device
    Xp = np.random.default_rng(1450).uniform(-2.5, 2.5, (293, 3))
    mc = Xp.shape[0]
    D = SetDesc.from_buffer_copy(bytes(D0))
    pts = torch.from_numpy(np.ascontiguousarray(Xp).reshape(-1)).to(dev)
    tab0 = torch.full((mc * D0.n_obs_pad,), float("nan"), dtype=torch.float64, device=dev)
    D.points, D.tab[0] = pts.data_ptr(), tab0.data_ptr()
    D.p[0] = mc
    for k in range(1, _lib.CBO_MAX_D):
        D.p[k] = 1
    D.g_total, D.g_begin, D.g_count = mc, 0, mc
    h = (SetDesc * 1)(D)
    d_desc = torch.frombuffer(bytearray(bytes(h)), dtype=torch.uint8).to(dev)
    l0 = eng.launches
    _lib.check(eng.lib.cbo_build_tables(h, C.c_void_p(d_desc.data_ptr()), 1, eng._stream()), "cbo_build_tables")
    torch.cuda.synchronize()
    assert eng.launches - l0 == 1
    ls = np.array([D0.ls_int[k] for k in range(3)])
    r = B.check_table(tab0.cpu().numpy().reshape(mc, D0.n_obs_pad), Xp, np.asarray(eng.problems[0].x_obs_int), ls)
    print(f"  K0 explicit points: {r:.2e}")
    assert r <= 1.0


def test_k0_rows_appended_by_refresh(cuda_engine_ready):
    """Rows appended through set_interventional + refresh (the int_rows_only launch): the new rows of u_int meet the bound
    from NaN, the earlier rows keep their bits."""
    import torch
    eng = _engine([dict(seed=1460, N=129, d=2, c=1, n=4, p=(6, 6)), dict(seed=1461, N=127, d=3, c=2, n=3, p=(3, 4, 5))])
    best = float(min(np.min(p.y_int) for p in eng.problems))
    eng.sweep(best, "min")
    rng = np.random.default_rng(1460)
    for g, add in ((0, 1), (1, 3)):
        pr, D = eng.problems[g], eng.h_sets[g]
        n_old = pr.x_int.shape[0]
        npad = D.n_obs_pad
        before = eng.buf[g]["u_int"][:n_old * npad].clone()
        x_new = np.vstack([pr.x_int, rng.uniform(-2.0, 2.0, (add, pr.d))])
        eng.set_interventional(g, x_new, np.append(pr.y_int, best - 0.05 * rng.random(add)))
        eng.buf[g]["u_int"][n_old * npad:].fill_(float("nan"))
        eng.refresh(best, "min", refit=[g])
        torch.cuda.synchronize()
        assert torch.equal(eng.buf[g]["u_int"][:n_old * npad], before)
        _tables_check(eng, g, f"appended {add}")
