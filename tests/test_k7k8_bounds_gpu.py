"""K7's gradients (refine.cu) and K8's likelihood (posterior_hyper.cu) against the error bounds of oracle/k7k8_bounds.py.

Stage A (refine_prior_kernel: m, v, dm, dv) is checked from the points, x_obs_int, ls_int, M, w, s2 and noise; stage B
(eval_point: mu, var, dmu, dvar) from K7's own m, v, dm, dv and the fetched L, alpha, sqrt_v_int, x_int, hyper; stage C (dei)
from the device's best, mu, var, dmu, dvar; stage D (dacq) bit for bit; stage E (cbo_posterior_nll) from K2's fetched factor.
_pass_grid / _acq_launches mirror m_pass_grid, m_chunks, m_item_exists and acq_grad_impl's per-launch batch split, and every
case asserts its geometry and launch count.  Outputs and the workspace start as NaN, every call runs twice with identical
bits.  Run with -s to see the worst error / bound of every quantity."""
import ctypes as C

import numpy as np
import pytest

from helpers import make_case
from oracle import k7k8_bounds as K
from oracle import posterior_bounds as P

pytestmark = pytest.mark.gpu

WORST = {}


def _note(r):
    for k, v in r.items():
        WORST[k] = max(WORST.get(k, 0.0), v)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\n  worst error / bound: " + "  ".join(f"{k} {v:.2e}" for k, v in sorted(WORST.items())))


# ---- mirrors ----------------------------------------------------------------------------------------------------------------
def _pass_grid(descs, per_set):
    live = [D for D in descs if D.causal and not D.prior_external]
    return (max((K.m_chunks(D.n_obs) for D in live), default=0), max((K.m_row_blocks(D.n_obs) for D in live), default=0),
            len(descs) * per_set)


def _items(D):
    return K.m_row_blocks(D.n_obs) * K.m_chunks(D.n_obs) if (D.causal and not D.prior_external) else 0


def _acq_launches(lib, h, D, npts, ws_bytes):
    """(launches, batches per launch) of one cbo_acq_grad call (acq_grad_impl)."""
    per_batch = _items(D) * K.REF_B * (2 + 2 * 4)
    state = lib.cbo_refine_workspace_bytes(h, 1) - 256 - per_batch * 8
    nbatch = -(-npts // K.REF_B)
    room = ((ws_bytes - 256 - state) // 8) // per_batch if per_batch else nbatch
    per_launch = min(room, nbatch, 65535)
    calls = -(-nbatch // per_launch)
    return calls * (2 if per_batch else 1), per_launch


# ---- running ------------------------------------------------------------------------------------------------------------------
def _engine(problems, **kw):
    from cbo_with_oop_b200.engine import SweepEngine
    return SweepEngine(problems, fit_hyperparameters=True, **kw)


def _fit(eng, hyper=None):
    import torch
    for li in range(len(eng.active)):
        eng.buf[li]["hyper"].copy_(torch.tensor((hyper or {}).get(eng.active[li], (1.0, 1.0)), dtype=torch.float64))
    eng.build_tables()
    eng.prior_precompute()
    eng.prior_eval(1)
    eng.posterior_fit()


def _grads_once(eng, g, X, best, task, ws_bytes):
    """One cbo_acq_grad call from a NaN workspace of ws_bytes into NaN outputs; the outputs and the launches it made."""
    import torch
    from cbo_with_oop_b200 import _lib
    h, dptr = eng._local_desc(eng.local_of[g])
    m = len(X)
    ws = eng._refine_workspace(ws_bytes)
    ws.view(torch.uint8).fill_(0xFF)                                    # NaN in every double
    pts = torch.from_numpy(np.ascontiguousarray(X, np.float64).reshape(-1)).to(eng.device)
    raw = torch.full((m * C.sizeof(_lib.AcqGradOut) // 8,), float("nan"), dtype=torch.float64, device=eng.device)
    torch.cuda.synchronize()
    l0 = eng.launches
    _lib.check(eng.lib.cbo_acq_grad(h, dptr, C.c_void_p(pts.data_ptr()), m, float(best), 1 if task == "min" else -1,
                                    C.c_void_p(ws.data_ptr()), ws_bytes, C.c_void_p(raw.data_ptr()), eng._stream()), "cbo_acq_grad")
    torch.cuda.synchronize()
    rec = np.frombuffer(raw.cpu().numpy().tobytes(), dtype=eng._GRAD_DTYPE)
    d = eng.problems[g].d
    return {n: (rec[n][:, :d].copy() if n.startswith("d") else rec[n].copy()) for n in eng._GRAD_DTYPE.names}, eng.launches - l0


def _grads(eng, g, X, best, task, ws_bytes=None):
    """Two calls from NaN with identical bits and the launch count of the mirror.  ws_bytes None: the workspace
    acquisition_gradients sizes, and acquisition_gradients itself must return the same bits."""
    D = eng.h_sets[eng.local_of[g]]
    h, _ = eng._local_desc(eng.local_of[g])
    engine_size = ws_bytes is None
    if engine_size:
        ws_bytes = eng.lib.cbo_refine_workspace_bytes(h, 1) * min(16, -(-len(X) // K.REF_B))
    (o1, l1), (o2, l2) = (_grads_once(eng, g, X, best, task, ws_bytes) for _ in range(2))
    for k in o1:
        assert o1[k].tobytes() == o2[k].tobytes(), f"{k} differs between two identical calls"
    want, per_launch = _acq_launches(eng.lib, h, D, len(X), ws_bytes)
    assert l1 == l2 == want, (l1, want)
    if engine_size:
        e = eng.acquisition_gradients(g, X, best, task)
        for k in o1:
            assert e[k].tobytes() == o1[k].tobytes(), f"{k}: acquisition_gradients differs from cbo_acq_grad"
    return o1, per_launch


def _state(eng, g, hyper=(1.0, 1.0)):
    D = eng.h_sets[eng.local_of[g]]
    return dict(x_int=eng.fetch("x_int", g), alpha=eng.fetch("alpha", g), L=eng.fetch("L", g), s2=hyper[0], l=hyper[1],
                sv=eng.fetch("sqrt_v_int", g) if D.causal else np.zeros(D.n_int), causal=bool(D.causal))


def _check(eng, g, X, o, best, task, hyper=(1.0, 1.0), label=""):
    """Stages A-D at the points X from the device outputs o."""
    pr, D = eng.problems[g], eng.h_sets[eng.local_of[g]]
    r = {}
    if pr.computes_prior:
        ref = K.prior_pass_ref(X, eng.fetch("x_obs_int", g).reshape(pr.d, -1).T, np.array(D.ls_int[:pr.d]), eng.fetch("M", g),
                               eng.fetch("w", g), D.s2, D.noise)
        r.update(K.check_prior_pass(o, ref))
    else:
        for k in ("m", "v", "dm", "dv"):
            assert not np.any(o[k]), f"{label}: a non-causal set has {k} != 0"
    st = _state(eng, g, hyper)
    r.update(K.check_grad(o, K.grad_ref(X, o["m"], o["v"], o["dm"], o["dv"], st)))
    sign = 1.0 if task == "min" else -1.0
    ok = o["var"] > 0
    r["dei"] = K.check_dei(o["dei"][ok], best, o["mu"][ok], o["var"][ok], o["dmu"][ok], o["dvar"][ok], sign)
    dacq = K.dacq_ref(o["dei"], o["acq"], X, pr.cost_fix, pr.cost_variable)
    assert dacq.tobytes() == o["dacq"].tobytes(), f"{label}: dacq is not (dei - acq dc) / cost bit for bit"
    print(f"  {label}: " + "  ".join(f"{k} {v:.2e}" for k, v in r.items()))
    _note(r)
    assert max(r.values()) <= 1.0, (label, r)
    return r


def _points(pr, npts, seed, obs=True):
    """npts points in the set's box: observational rows (u = 1 for that row, a = 0), box faces, x_k = 0, random."""
    rng = np.random.default_rng(seed)
    lo, hi = np.array([t.min() for t in pr.grid]), np.array([t.max() for t in pr.grid])
    X = rng.uniform(lo, hi, (npts, pr.d))
    fixed = []
    if obs and pr.computes_prior:
        fixed += [np.clip(pr.x_obs_int[j], lo, hi) for j in range(min(2, pr.x_obs_int.shape[0]))]
        fixed[0] = pr.x_obs_int[0]
    fixed += [lo, hi, np.where(np.arange(pr.d) == 0, 0.0, X[0])]
    for i, f in enumerate(fixed[:npts]):
        X[i] = f
    return X


# ---- A: pass geometry ---------------------------------------------------------------------------------------------------------
GEOMETRY = [(1, 1), (16, 2), (127, 3), (128, 4), (129, 1), (192, 2), (255, 3), (512, 4), (513, 1), (641, 2), (1153, 3),
            (4000, 2)]


def _geometry_expect(N):
    R, Cc = K.m_row_blocks(N), K.m_chunks(N)
    return dict(R=R, C=Cc, ragged=N - (R - 1) * 128,
                mixed=any(K.item_slabs(I, c)[0] < K.item_slabs(I, c)[2] < K.item_slabs(I, c)[1]
                          for I in range(R) for c in range(1, Cc) if K.m_item_exists(I, c)),
                all_diag=any(K.item_slabs(I, c)[0] >= K.item_slabs(I, c)[2] for I in range(R) for c in range(1, Cc)
                             if K.m_item_exists(I, c)))


@pytest.mark.parametrize("N,d", GEOMETRY, ids=[f"N{n}-d{d}" for n, d in GEOMETRY])
def test_pass_geometry(cuda_engine_ready, N, d):
    from cbo_with_oop_b200.engine import SetProblem
    kw, _ = make_case(seed=1000 + N, N=N, d=d, c=1, n=12, p=(6,) * d, cost_variable=N % 2 == 1)
    pr = SetProblem(**kw)
    eng = _engine([pr])
    _fit(eng)
    e = _geometry_expect(N)
    assert _pass_grid([eng.h_sets[0]], 2) == (e["C"], e["R"], 2)
    if N == 513:
        assert e["C"] == 2 and e["all_diag"] and not e["mixed"]
    if N == 641:
        assert e["C"] == 2 and e["mixed"]
    if N == 1153:
        assert e["C"] == 3
    if N in (129, 192, 255):
        assert e["ragged"] == {129: 1, 192: 64, 255: 127}[N]
    X = _points(pr, 9, N)
    best = float(np.min(pr.y_int))
    o, _ = _grads(eng, 0, X, best, "min")
    _check(eng, 0, X, o, best, "min", label=f"geometry N={N} d={d} R={e['R']} C={e['C']}")


# ---- points and launches ------------------------------------------------------------------------------------------------------
def test_point_counts_and_launches(cuda_engine_ready):
    """1, 7, 8, 9, 83 and 200 points on a set with three items (200 points need a second acq_grad_impl launch); a raw call
    whose workspace holds exactly one batch (one batch per launch) gives the engine's bits."""
    from cbo_with_oop_b200.engine import SetProblem
    kw, _ = make_case(seed=1101, N=300, d=2, c=1, n=20, p=(10, 10), cost_variable=True)
    pr = SetProblem(**kw)
    eng = _engine([pr])
    _fit(eng)
    D = eng.h_sets[0]
    assert _items(D) == 3
    best = float(np.min(pr.y_int))
    per = {}
    for npts in (1, 7, 8, 9, 83, 200):
        X = _points(pr, npts, npts)
        o, per[npts] = _grads(eng, 0, X, best, "min")
        if npts in (9, 200):
            _check(eng, 0, X, o, best, "min", label=f"{npts} points")
    assert per[200] < 25, "200 points were meant to need a second launch"
    X = _points(pr, 83, 83)
    full, _ = _grads(eng, 0, X, best, "min")
    h, _ = eng._local_desc(0)
    one = eng.lib.cbo_refine_workspace_bytes(h, 1)
    raw, pl = _grads(eng, 0, X, best, "min", ws_bytes=one)
    assert pl == 1
    for k in full:
        assert full[k].tobytes() == raw[k].tobytes(), f"{k}: one batch per launch differs from the engine's call"


# ---- B: posterior slots ---------------------------------------------------------------------------------------------------------
POST_N = [1, 31, 32, 33, 64, 65, 96, 97, 128]
HYPER = [(1.0, 1.0), (1e-3, 0.3), (50.0, 4.0)]


@pytest.mark.parametrize("task", ["min", "max"])
def test_posterior_slots(cuda_engine_ready, task):
    from cbo_with_oop_b200.engine import SetProblem
    probs, hyper = [], {}
    for j, n in enumerate(POST_N):
        d = 1 + j % 4
        kw, _ = make_case(seed=1200 + n, N=150, d=d, c=1, n=n, p=(6,) * d, causal=j % 3 != 2, cost_variable=j % 2 == 0)
        s2, l = HYPER[j % 3]
        kw["x_int"] = kw["x_int"] * l
        probs.append(SetProblem(**kw))
        hyper[j] = (s2, l)
    eng = _engine(probs)
    _fit(eng, hyper)
    n_sub = 0
    for g, pr in enumerate(probs):
        assert int(eng.fetch("fit_info", g)[1]) == 0
        X = _points(pr, 9, g)
        inc = float(pr.y_int.min() if task == "min" else pr.y_int.max())
        o, _ = _grads(eng, g, X, inc, task)
        _check(eng, g, X, o, inc, task, hyper[g], f"n={pr.x_int.shape[0]} d={pr.d} causal={pr.causal} hyper={hyper[g]} {task} "
                                                  "best=incumbent")
        # the EI tail for either task: best below every point's mean, u <= -6 (u Phi + phi cancels) and u <= -38 at
        # every point, -38 at one (phi, Phi and dei subnormal)
        sd = np.sqrt(np.maximum(o["var"], 0.0))
        for depth in (6.0, 38.0):
            best = float(np.min(o["mu"] - depth * sd))
            ot, _ = _grads(eng, g, X, best, task)
            assert np.all(ot["mu"] == o["mu"]) and np.all(ot["var"] == o["var"])
            _check(eng, g, X, ot, best, task, hyper[g], f"n={pr.x_int.shape[0]} d={pr.d} causal={pr.causal} hyper={hyper[g]} "
                                                         f"{task} u<=-{depth:g}")
            n_sub += int(np.count_nonzero((ot["dei"] != 0) & (np.abs(ot["dei"]) < np.finfo(np.float64).tiny)))
    print(f"  {n_sub} subnormal dei checked")
    assert n_sub > 0, "the u = -38 points were meant to give subnormal dei"


# ---- refine ---------------------------------------------------------------------------------------------------------------------
def _raw_refine(eng, x0, best, max_iter):
    import torch
    from cbo_with_oop_b200 import _lib
    A = len(eng.active)
    eng._push_descs()
    ws = eng._refine_workspace(eng.lib.cbo_refine_workspace_bytes(eng.h_sets, A))
    ws.view(torch.uint8).fill_(0xFF)
    d_x0 = torch.from_numpy(np.ascontiguousarray(x0, np.float64).reshape(-1)).to(eng.device)
    res = torch.zeros((A * C.sizeof(_lib.RefineResult),), dtype=torch.uint8, device=eng.device)
    torch.cuda.synchronize()
    l0 = eng.launches
    _lib.check(eng.lib.cbo_refine(eng.h_sets, C.c_void_p(eng.d_sets.data_ptr()), A, float(best), 1, C.c_void_p(d_x0.data_ptr()),
                                  int(max_iter), 1e-7, C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(res.data_ptr()),
                                  eng._stream()), "cbo_refine")
    torch.cuda.synchronize()
    return (_lib.RefineResult * A).from_buffer_copy(res.cpu().numpy().tobytes()), eng.launches - l0


def test_refine_reads_the_slots_acq_grad_reads(cuda_engine_ready):
    """One refine over sets with d = 1..4 and different N (four pass launches per iteration; the smaller sets' CTAs find no
    item): with max_iter = 0 every start value is acquisition_gradients(x0).acq bit for bit, and after a refine every set's
    value is acquisition_gradients(x).acq at its returned x bit for bit."""
    from cbo_with_oop_b200.engine import SetProblem
    specs = [(700, 1), (130, 2), (40, 3), (300, 4)]
    probs = [SetProblem(**make_case(seed=1300 + d, N=N, d=d, c=1, n=10 + d, p=(8,) * d)[0]) for N, d in specs]
    eng = _engine(probs)
    _fit(eng)
    best = float(min(np.min(p.y_int) for p in probs))
    x0 = np.zeros((len(probs), 4))
    for g, pr in enumerate(probs):
        x0[g, :pr.d] = _points(pr, 3, g, obs=False)[2]
    for max_iter in (0, 30):
        (r1, l1), (r2, l2) = (_raw_refine(eng, x0, best, max_iter) for _ in range(2))
        assert bytes(r1) == bytes(r2) and l1 == l2
        if max_iter == 0:
            assert l1 == 1 + 4 + 1 + 1, l1          # init, one pass per d, the step, finish
        for g, pr in enumerate(probs):
            x = np.array(r1[g].x[:pr.d]) if max_iter else x0[g, :pr.d]
            o, _ = _grads(eng, g, x[None, :], best, "min")
            want = r1[g].start_value if max_iter == 0 else r1[g].value
            assert np.float64(want).tobytes() == o["acq"][0].tobytes(), (g, max_iter, want, o["acq"][0])
    # each set alone gives the bits it gave in the mixed call
    for g, pr in enumerate(probs):
        alone = _engine([pr])
        _fit(alone)
        ra, _ = _raw_refine(alone, x0[g:g + 1], best, 30)
        assert bytes(ra[0]) == bytes(r1[g]), g


# ---- cancellation at the interventional rows -------------------------------------------------------------------------------------
def _dense_1d_problem():
    from cbo_with_oop_b200.engine import SetProblem
    from oracle import cbo_oracle as O
    rng = np.random.default_rng(0)
    N = 200
    X = np.sort(rng.uniform(-2.0, 2.0, N))[:, None]
    y = np.sin(2.0 * X[:, 0]) + 0.01 * rng.standard_normal(N)
    gp = O.obs_gp_fit(X, y, 1.0, np.array([0.8]), noise=1e-4, form="diff")
    z = np.zeros((N, 0))
    return SetProblem(x_obs_int=X, x_obs_cond=z, mc_cond=z, alpha_obs=gp["alpha"], kyinv=gp["Kyinv"], ls_int=np.array([0.8]),
                      ls_cond=np.zeros(0), s2=1.0, grid=[np.linspace(-2, 2, 9)], x_int=rng.uniform(-1.8, 1.8, (6, 1)),
                      y_int=rng.standard_normal(6), noise=1e-4, name="dense_1d")


def test_cancellation_at_the_interventional_rows(cuda_engine_ready):
    """Dense 1-D data with noise 1e-4 and set 2 of the simplified coral fixture, where u^T M u cancels 1e8..1e10-fold: K7's
    v and dv at every x_int row and at 1e-3 l from it, against the exact value and against K1c's v_int (Dot2)."""
    from cbo_with_oop_b200.fixtures import load_golden_problems
    coral = load_golden_problems("simplified_coral", device_fit=False)[0][2]
    probs = [_dense_1d_problem(), coral]
    eng = _engine(probs)
    _fit(eng)
    worst = {}
    for g, pr in enumerate(probs):
        D = eng.h_sets[g]
        XI = eng.fetch("x_int", g)
        ls = np.array(D.ls_int[:pr.d])
        Xo = eng.fetch("x_obs_int", g).reshape(pr.d, -1).T
        M = eng.fetch("M", g)
        X = np.vstack([XI, XI + 1e-3 * ls])
        best = float(np.min(pr.y_int))
        o, _ = _grads(eng, g, X, best, "min")
        _check(eng, g, X, o, best, "min", label=f"cancelled set {g}")
        ev = np.zeros(len(X))
        edv = np.zeros(len(X))
        for p, x in enumerate(X):
            v, dv = K.exact_v_dv(x, Xo, ls, M, D.s2, D.noise)
            ev[p] = abs(o["v"][p] - v) / abs(v)
            edv[p] = np.max(np.abs(o["dv"][p] - dv) / np.maximum(np.abs(dv), 1e-300))
        n = len(XI)
        vint = eng.fetch("v_int", g)
        k1c = np.abs(o["v"][:n] - vint) / np.abs(vint)
        print(f"  cancelled set {g} (N={D.n_obs}): K7 v rel. error at x_int {ev[:n].max():.2e}, at 1e-3 l {ev[n:].max():.2e}; "
              f"dv {edv[:n].max():.2e} / {edv[n:].max():.2e}; |v_K7 - v_int_K1c| / v_int {k1c.max():.2e}")
        worst[g] = (ev.max(), edv.max(), k1c.max())
        assert ev.max() <= 1e-6, (g, ev.max())


@pytest.mark.parametrize("cfg", ["toy", "complete", "simplified_coral", "coral_synth"])
def test_cancellation_on_golden_configurations(cuda_engine_ready, cfg):
    """K7's v at every interventional row of every set of the golden configurations against the exact value: below 1e-6
    relative, the accuracy K1c's compensated v_int was introduced for, so the pass needs no compensation."""
    from cbo_with_oop_b200.fixtures import load_golden_problems
    problems, best, task = load_golden_problems(cfg, device_fit=False)
    eng = _engine(problems)
    _fit(eng)
    worst, n_rows = 0.0, 0
    for g, pr in enumerate(problems):
        if not pr.computes_prior:
            continue
        D = eng.h_sets[eng.local_of[g]]
        XI = eng.fetch("x_int", g)
        o, _ = _grads(eng, g, XI, best, task)
        Xo = eng.fetch("x_obs_int", g).reshape(pr.d, -1).T
        M, ls = eng.fetch("M", g), np.array(D.ls_int[:pr.d])
        for p, x in enumerate(XI):
            v = K.exact_v_dv(x, Xo, ls, M, D.s2, D.noise, with_dv=False)
            worst = max(worst, abs(o["v"][p] - v) / abs(v))
        n_rows += len(XI)
    print(f"  {cfg}: worst relative error of K7's v at {n_rows} interventional rows {worst:.2e}")
    assert n_rows > 0 and worst <= 1e-6, (cfg, worst)


# ---- E: K8 ---------------------------------------------------------------------------------------------------------------------
K8_N = [1, 2, 31, 32, 33, 63, 64, 65, 96, 97, 127, 128]
K8_HYPER = [(1e-3, 0.2), (1.0, 1.0), (50.0, 4.0), (0.3, 0.6)]


def _nll_all(eng):
    import torch
    from cbo_with_oop_b200 import _lib
    A = len(eng.active)
    eng._push_descs()
    out = torch.full((3 * A,), float("nan"), dtype=torch.float64, device=eng.device)
    l0 = eng.launches
    _lib.check(eng.lib.cbo_posterior_nll(eng.h_sets, C.c_void_p(eng.d_sets.data_ptr()), A, C.c_void_p(out.data_ptr()),
                                         eng._stream()), "cbo_posterior_nll")
    torch.cuda.synchronize()
    assert eng.launches - l0 == 1
    return out.cpu().numpy().reshape(A, 3)


def _check_k8(eng, g, got, hyper, label):
    D = eng.h_sets[eng.local_of[g]]
    assert int(eng.fetch("fit_info", g)[1]) == 0, "K2 failed: its factor cannot stand for K8's"
    y = eng.fetch("y_int", g)
    res = y - eng.fetch("m_int", g) if D.causal else y
    ref = K.k8_ref(eng.fetch("L", g), eng.fetch("x_int", g), res, hyper[0], hyper[1])
    r = K.check_k8(got, ref)
    print(f"  K8 {label} tries={int(eng.fetch('fit_info', g)[0])}: " + "  ".join(f"{k} {v:.2e}" for k, v in r.items()))
    _note(r)
    assert max(r.values()) <= 1.0, (label, r)


def test_k8_every_row_slot(cuda_engine_ready):
    from cbo_with_oop_b200.engine import SetProblem
    probs, hyper = [], {}
    for j, n in enumerate(K8_N):
        d = 1 + j % 4
        s2, l = K8_HYPER[j % 4]
        kw, _ = make_case(seed=1400 + n, N=60, d=d, c=1, n=n, p=(5,) * d, causal=j % 2 == 0)
        kw["x_int"] = kw["x_int"] * l
        probs.append(SetProblem(**kw))
        hyper[j] = (s2, l)
    eng = _engine(probs)
    _fit(eng, hyper)
    a, b = _nll_all(eng), _nll_all(eng)
    assert a.tobytes() == b.tobytes()
    for g, pr in enumerate(probs):
        _check_k8(eng, g, a[g], hyper[g], f"n={pr.x_int.shape[0]} d={pr.d} causal={pr.causal} hyper={hyper[g]}")


def test_k8_jitter_retry_and_not_positive_definite(cuda_engine_ready):
    """Two identical rows at s2 = 2^40: the first Cholesky meets an exactly zero pivot and the retry's factor is K2's; a
    negative variance keeps every pivot negative (the jitter is negative too) and K8 returns three NaNs."""
    from cbo_with_oop_b200.engine import SetProblem
    kw, _ = make_case(seed=1501, N=40, d=1, c=1, n=6, p=(20,), causal=False)
    kw["x_int"] = kw["x_int"] * 8.0
    kw["x_int"][1] = kw["x_int"][0]
    kw["grid"] = [np.linspace(-30.0, 30.0, 20)]
    pr = SetProblem(**kw)
    kw2, _ = make_case(seed=1502, N=40, d=2, c=1, n=9, p=(5, 5), causal=False)
    eng = _engine([pr, SetProblem(**kw2)])
    _fit(eng, {0: (2.0 ** 40, 1.0), 1: (1.0, 1.0)})
    assert int(eng.fetch("fit_info", 0)[0]) == 1
    import torch
    eng.buf[1]["hyper"].copy_(torch.tensor((-1.0, 1.0), dtype=torch.float64))
    out = _nll_all(eng)
    _check_k8(eng, 0, out[0], (2.0 ** 40, 1.0), "jitter retry")
    assert np.all(np.isnan(out[1])), out[1]
