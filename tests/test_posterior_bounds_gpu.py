"""The per-set surrogate kernels against the error bounds of oracle/posterior_bounds.py, on every branch they have.

K2 (posterior_fit.cu) is checked from its own inputs (x_int, y_int, m_int, sqrt_v_int, hyper, the retry count), K3
(sweep.cu) from the fetched L, L^-1, alpha and the candidates' prior, K7 (refine.cu) from its own m, v outputs.  Which of
the six sweep launches takes a set, and the chunk length of the tensor-pipe launch, are decided on the host;
_class / _chunk repeat those decisions in Python and every case asserts the path it was built for, with the launch count
that goes with it.  Cases are sized from the SM count so that the intended chunk occurs on any B200 configuration.

Every sweep starts from NaN in mu / var / ei / acq and runs twice with bit-identical results; every set of a mixed call is
also run alone and must give the same bits.  acq = ei / cost is reproduced bit for bit, the per-set argmax and NaN count
exactly.  Sets of up to 2^15 candidates are checked on every candidate; larger ones on every candidate of their first,
a middle and their last item plus a seeded sample of 2^14 (the argmax and NaN checks always see every candidate).  EI is
checked against mpmath on a seeded sample of 512 candidates plus the 64 deepest in the tail.  Run with -s to see the
worst error / bound and bound / scale of every case."""
import ctypes as C

import numpy as np
import pytest

from helpers import make_case
from oracle import posterior_bounds as P

pytestmark = pytest.mark.gpu

TILE = 1024
ARRAYS = ("mu", "var", "ei", "acq")
FULL = 1 << 15
SAMPLE = 1 << 14
SEP_MAX_P, MMA_MAX_N, FMA_MAX_N, MAX_CHUNK = 256, 48, 16, 64
HYPERS = [(1e-3, 0.3), (50.0, 4.0), (1e-3, 4.0), (50.0, 0.3)]


# ---- Python mirror of sweep_class / sweep_separable / sweep_impl's chunk (csrc/sweep.cu) -----------------------------------
def _separable(D):
    return not D.points and D.n_int <= MMA_MAX_N and 16 <= D.p[D.d - 1] <= SEP_MAX_P


def _class(D):
    if D.posterior_cached:
        return 0 if D.cost_variable else 5
    if D.n_int <= FMA_MAX_N:
        return 1 if _separable(D) else 0
    if D.n_int <= MMA_MAX_N:
        return 2 if _separable(D) else 3
    return 4


def _items(D):
    return -(-D.g_count // TILE)


def _chunk(descs, sms):
    c2 = [D for D in descs if D.g_count > 0 and _class(D) == 2]
    if not c2:
        return 1
    chunk = min(-(-sum(_items(D) for D in c2) // sms), MAX_CHUNK)
    base = (42 * 32 + 2 * 48 + 48 * 4) * 8
    while True:
        tab = max(((D.n_int + 3) & ~3) * ((((D.p[D.d - 1] + 3) // 8) * 8 + 4) + ((chunk * TILE // D.p[D.d - 1] + 2) | 1))
                  for D in c2)
        if chunk == 1 or base + tab * 8 <= 160 * 1024:
            return chunk
        chunk -= 1


def _descs(eng):
    return [eng.h_sets[i] for i in range(len(eng.active))]


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- problems ---------------------------------------------------------------------------------------------------------------
def _lattice(n, d, seed, l):
    rng = np.random.default_rng(seed)
    side = int(np.ceil(n ** (1.0 / d) - 1e-9))
    pts = np.stack(np.meshgrid(*[np.arange(side)] * d, indexing="ij"), -1).reshape(-1, d)[:n].astype(float)
    return (pts - (side - 1) / 2.0) * 1.1 * l + rng.uniform(-0.15, 0.15, (n, d)) * l


def _problem(seed, n, p, causal=True, cost_variable=False, l=1.0, N=48):
    """A set whose interventional rows sit on a jittered lattice of spacing ~1.1 l (an informative bound), on a grid that
    covers them."""
    from cbo_with_oop_b200.engine import SetProblem
    d = len(p)
    kw, _ = make_case(seed=seed, N=N, d=d, c=1, n=n, p=p, causal=causal, cost_variable=cost_variable)
    X = _lattice(n, d, seed, l)
    span = float(np.abs(X).max()) + 0.5 * l
    kw["x_int"] = X
    kw["y_int"] = np.sin(X.sum(1) / l) + 0.1 * np.random.default_rng(seed).standard_normal(n)
    kw["grid"] = [np.linspace(-span * (1 + 0.01 * k), span, pk) for k, pk in enumerate(p)]
    return SetProblem(**kw)


def _engine(problems, **kw):
    from cbo_with_oop_b200.engine import SweepEngine
    return SweepEngine(problems, keep=ARRAYS, fit_hyperparameters=True, **kw)


def _best(eng):
    return float(min(np.min(eng.problems[g].y_int) for g in eng.active))


# ---- running ------------------------------------------------------------------------------------------------------------------
def _fit(eng, hyper=None):
    """Every stage up to the sweep, with the hyper buffers holding `hyper` (global id -> (s2, l)); K8 does not run."""
    import torch
    for li in range(len(eng.active)):
        eng.buf[li]["hyper"].copy_(torch.tensor((hyper or {}).get(eng.active[li], (1.0, 1.0)), dtype=torch.float64))
    eng.build_tables()
    eng.prior_precompute()
    eng.prior_eval(1)
    eng.posterior_fit()
    eng.prior_eval(0)
    eng._posterior_valid = set(eng.active)


def _bests(eng):
    from cbo_with_oop_b200._lib import SetBest
    A = len(eng.active)
    raw = eng.local_best[:A * C.sizeof(SetBest)].cpu().numpy().tobytes()
    return [(b.value, b.index, b.n_nan) for b in (SetBest * A).from_buffer_copy(raw)]


def _sweep_once(eng, best, task, names=ARRAYS):
    import torch
    for b in eng.buf:
        for k in names:
            b[k].fill_(float("nan"))
    l0 = eng.launches
    eng._sweep_local(best, task)
    torch.cuda.synchronize()
    return eng.launches - l0, {g: {k: eng.fetch(k, g).copy() for k in ARRAYS} for g in eng.active}, _bests(eng)


def _sweep(eng, best, task):
    """Two sweeps from NaN: the launch count and the outputs must agree bit for bit.  Asserts the launch count the mirror
    predicts (one launch per class present, the set and global reductions)."""
    (l1, o1, b1), (l2, o2, b2) = _sweep_once(eng, best, task), _sweep_once(eng, best, task)
    assert l1 == l2 and b1 == b2
    for g in o1:
        for k in ARRAYS:
            assert o1[g][k].tobytes() == o2[g][k].tobytes(), f"set {g}: {k} differs between two identical runs"
    classes = {_class(D) for D in _descs(eng) if D.g_count > 0}
    assert l1 == len(classes) + 2, (l1, classes)
    return o1, b1


# ---- checks ---------------------------------------------------------------------------------------------------------------
def _hyper(eng, g):
    s2, l = eng.buf[eng.local_of[g]]["hyper"].cpu().numpy()
    return float(s2), float(l)


def _state(eng, g):
    D = eng.h_sets[eng.local_of[g]]
    s2, l = _hyper(eng, g)
    st = dict(x_int=eng.fetch("x_int", g), alpha=eng.fetch("alpha", g), L=eng.fetch("L", g), s2=s2, l=l,
              sv=eng.fetch("sqrt_v_int", g) if D.causal else np.zeros(D.n_int))
    if D.n_int <= MMA_MAX_N:
        st["W"] = eng.fetch("Linv", g)
    return st


def _check_fit(eng, g, label=""):
    D = eng.h_sets[eng.local_of[g]]
    n = D.n_int
    info = eng.fetch("fit_info", g)
    assert info[1] == 0, (g, info)
    st = _state(eng, g)
    m_int = None
    if D.causal:
        m_int = eng.fetch("m_int", g)
        assert st["sv"].tobytes() == np.sqrt(eng.fetch("v_int", g)).tobytes(), "sqrt_v_int is not the IEEE sqrt of v_int"
    raw = eng.buf[eng.local_of[g]]["L"][:n * n].cpu().numpy().reshape(n, n)
    if n > MMA_MAX_N:
        assert not np.triu(raw, 1).any(), f"set {g}: the strict upper triangle is not zero for n = {n} > 48"
    r = P.check_fit(st["L"], st["alpha"], st["x_int"], eng.fetch("y_int", g), st["sv"], st["s2"], st["l"], int(info[0]),
                    m_int, st.get("W"))
    print(f"  K2 {label} set {g} n={n} d={D.d} tries={info[0]}: " + "  ".join(f"{k} {v:.2e}" for k, v in r.items()))
    assert r["L"] <= 1.0 and r["alpha"] <= 1.0 and r.get("W", 0.0) <= 1.0, (g, r)
    return r


def _coords(eng, g, idx):
    pr, D = eng.problems[g], eng.h_sets[eng.local_of[g]]
    ii = np.unravel_index(D.g_begin + np.asarray(idx, np.int64), [len(t) for t in pr.grid])
    return np.stack([pr.grid[k][ii[k]] for k in range(pr.d)], 1)


def _checked(gc, seed):
    if gc <= FULL:
        return np.arange(gc)
    it = -(-gc // TILE)
    parts = [np.arange(0, TILE), np.arange((it // 2) * TILE, (it // 2 + 1) * TILE), np.arange((it - 1) * TILE, gc),
             np.random.default_rng(seed).choice(gc, SAMPLE, replace=False)]
    return np.unique(np.concatenate(parts))


def _check_values(st, X, m, v, out, best, task, cost_fix, cost_var, path, separable, label, informative=False):
    """mu, var against their bounds, EI against mpmath on a sample, acq bit for bit, at candidates X."""
    ref = P.posterior_ref(X, m, v, st, path, separable)
    rm, rv = P.check_posterior(out["mu"], out["var"], ref)
    mu_scale = float(np.abs(ref["mu"].astype(np.float64)).max())
    b_mu = float(ref["e_mu"].max() / max(mu_scale, 1e-300))
    b_var = float((ref["e_var"] / (st["s2"] + np.asarray(v))).max())
    sign = 1.0 if task == "min" else -1.0
    var_ref = ref["var"].astype(np.float64)
    ok = (var_ref > ref["e_var"]) & (out["var"] > 0)
    skipped = int((~ok).sum())
    cand = np.flatnonzero(ok)
    re = 0.0
    if cand.size:
        rng = np.random.default_rng(len(cand))
        u = (best - out["mu"][cand]) / np.sqrt(out["var"][cand])
        tail = cand[np.argsort(u)[:64]]
        pick = np.unique(np.concatenate([rng.choice(cand, min(512, cand.size), replace=False), tail]))
        re = P.check_ei(out["ei"], best, out["mu"], out["var"], sign, pick)
    acq = out["ei"] / P.candidate_cost(X, cost_fix, cost_var)
    assert acq.tobytes() == out["acq"].tobytes(), f"{label}: acq is not ei / cost bit for bit"
    print(f"  {label}: mu {rm:.2e} var {rv:.2e} ei {re:.2e} of bound; bound/scale mu {b_mu:.1e} var {b_var:.1e}; "
          f"{skipped} without EI check")
    assert rm <= 1.0 and rv <= 1.0 and re <= 1.0, (label, rm, rv, re)
    assert skipped <= max(2, 0.01 * len(X)), (label, skipped)
    if informative:
        assert b_mu <= 1e-8 and b_var <= 1e-8, (label, b_mu, b_var)
    return rm, rv, re


def _path(D):
    return "mma" if FMA_MAX_N < D.n_int <= MMA_MAX_N else "subst"


def _check_set(eng, g, out, best_tuple, best, task, label="", informative=False):
    """Bounds on the checked candidates of set g's sweep, argmax / NaN count on all of them."""
    D = eng.h_sets[eng.local_of[g]]
    pr = eng.problems[g]
    idx = _checked(D.g_count, g)
    X = _coords(eng, g, idx)
    if pr.computes_prior:
        m, v = eng.fetch("m", g)[idx], eng.fetch("v", g)[idx]
    else:
        m = v = np.zeros(len(idx))
    o = {k: out[g][k][idx] for k in ARRAYS}
    cls = _class(D)
    _check_values(_state(eng, g), X, m, v, o, best, task, pr.cost_fix, pr.cost_variable, _path(D), cls in (1, 2),
                  f"{label} set {g} class {cls} n={D.n_int} d={D.d} p_last={D.p[D.d - 1]} g={D.g_count}", informative)
    val, i, nn = P.first_argmax(out[g]["acq"])
    assert best_tuple == (val, D.g_begin + i if i >= 0 else -1, nn), (g, best_tuple, val, i, nn)


def _alone_matches(problems, hyper, best, task, mixed):
    """Every set run alone gives the bits it gave inside the mixed call."""
    for g, pr in enumerate(problems):
        e = _engine([pr])
        _fit(e, {0: hyper[g]} if hyper and g in hyper else None)
        o, _ = _sweep(e, best, task)
        for k in ARRAYS:
            assert o[0][k].tobytes() == mixed[g][k].tobytes(), f"set {g}: {k} alone != {k} in the mixed call"


# ---- K2 ---------------------------------------------------------------------------------------------------------------------
K2_N = [1, 2, 31, 32, 33, 48, 49, 64, 65, 96, 97, 127, 128]


def test_fit_every_row_slot(cuda_engine_ready):
    """n on both sides of the warp's row slots (32, 64, 96) and of the L^-T cut-off (48), causal and not, unit hyper and
    (50, 0.3); the factor, alpha and L^-1 against the Gram of the kernel's own inputs."""
    probs = [_problem(100 + j, n, (8, 9), causal=j % 2 == 0) for j, n in enumerate(K2_N)]
    hyper = {g: (50.0, 0.3) for g in range(0, len(probs), 3)}
    eng = _engine(probs)
    _fit(eng, hyper)
    for g in range(len(probs)):
        _check_fit(eng, g, "row slots")


def test_fit_jitter_retry(cuda_engine_ready):
    """Two identical rows at s2 = 2^40: fma(sv, sv, s2) + kSurrogateDiag rounds to 2^40 and the second pivot is exactly 0,
    so the first attempt fails on every order of the trailing update; the retry's jitter is reproduced bit for bit."""
    pr = _problem(131, 6, (20,), causal=False, l=1.0)
    pr.x_int = pr.x_int * 8.0
    pr.x_int[1] = pr.x_int[0]
    pr.grid = [np.linspace(-30.0, 30.0, 20)]
    eng = _engine([pr])
    _fit(eng, {0: (2.0 ** 40, 1.0)})
    assert int(eng.fetch("fit_info", 0)[0]) == 1
    _check_fit(eng, 0, "jitter")
    o, b = _sweep(eng, 0.0, "min")
    _check_set(eng, 0, o, b[0], 0.0, "min", "jitter")


# ---- K3: every class in one call, then alone ----------------------------------------------------------------------------------
def _class_problems():
    """(problem, expected class, informative) for one mixed call."""
    S = []
    add = lambda cls, inf, *a, **k: S.append((_problem(*a, **k), cls, inf))
    # class 0: n <= 16 without tables (p_last 15 / 257), d = 1..4
    add(0, False, 201, 1, (15,))
    add(0, False, 202, 2, (9, 257), causal=False)
    add(0, False, 203, 15, (5, 4, 15), cost_variable=True)
    add(0, True, 204, 16, (3, 3, 3, 257))
    # class 1: p_last 16, 17, 255, 256; d = 1 and 4; 66 lead rows per item; g = 1025
    add(1, False, 211, 16, (16,))
    add(1, False, 212, 7, (256,), causal=False)
    add(1, False, 213, 16, (4, 4, 4, 17), cost_variable=True)
    add(1, False, 214, 9, (200, 16))
    add(1, False, 215, 12, (41, 25))
    add(1, False, 216, 10, (30, 255), causal=False)
    # class 2: n on and off the 8-row blocks and k4 steps; g = 391 (dead tail lanes, 7 mod 32)
    for j, (n, p) in enumerate([(17, (37, 100)), (20, (10, 64)), (24, (23, 17)), (25, (20, 64)), (31, (23, 17)),
                                (32, (6, 7, 50)), (33, (6, 7, 50)), (40, (12, 100)), (47, (30, 33)), (48, (70, 16))]):
        add(2, n in (17, 25, 33, 48), 220 + j, n, p, causal=j % 3 != 2, cost_variable=n == 33)
    # class 3: grids with p_last 15 and 300
    add(3, False, 241, 20, (30, 15))
    add(3, False, 242, 40, (4, 300), causal=False)
    # class 4: n > 48, d = 1..4 (n = 128 at d = 4: the largest shared-memory launch); cost variable at n = 100
    for j, (n, p) in enumerate([(49, (300,)), (64, (20, 20)), (65, (8, 8, 8)), (100, (4, 4, 4, 6)), (127, (30, 31)),
                                (128, (4, 5, 6, 7))]):
        add(4, n == 128, 250 + j, n, p, causal=j % 2 == 0, cost_variable=n == 100)
    return S


@pytest.fixture(scope="module")
def mixed(cuda_engine_ready):
    S = _class_problems()
    probs = [s[0] for s in S]
    eng = _engine(probs)
    for g, (_, cls, _) in enumerate(S):
        assert _class(eng.h_sets[g]) == cls, f"set {g} was built for class {cls}, the mirror says {_class(eng.h_sets[g])}"
    _fit(eng)
    return S, probs, eng


@pytest.mark.parametrize("task", ["min", "max"])
def test_every_class_in_one_call(mixed, task):
    S, probs, eng = mixed
    best = _best(eng) if task == "min" else float(max(np.max(p.y_int) for p in probs))
    assert _chunk(_descs(eng), eng.num_sms) == 1
    out, bests = _sweep(eng, best, task)
    for g, (_, cls, inf) in enumerate(S):
        _check_fit(eng, g, "mixed")
        _check_set(eng, g, out, bests[g], best, task, f"mixed {task}", informative=inf)
    if task == "min":
        _alone_matches(probs, None, best, task, out)


def test_cached_sets_refresh(mixed):
    """A staged refresh (no refit): fixed-cost sets go to ei_refresh_kernel (class 5), variable-cost ones to
    sweep_kernel<16, false> (class 0, also at n = 33 and 100).  At the same incumbent EI and acq keep the sweeping class's
    bits; at a new incumbent they meet the EI bound at the cached mu, var and acq = ei / cost bit for bit."""
    import torch
    S, probs, eng = mixed
    best = _best(eng)
    base, _ = _sweep(eng, best, "min")
    eng.timing = True
    try:
        for b2 in (best, best - 0.3):
            eng._posterior_valid = set(eng.active)
            for b in eng.buf:
                b["ei"].fill_(float("nan"))
                b["acq"].fill_(float("nan"))
            l0 = eng.launches
            eng.refresh(b2, "min", refit=[])
            torch.cuda.synchronize()
            classes = {0 if p.cost_variable else 5 for p in probs}
            assert eng.launches - l0 == len(classes) + 2
            bests = _bests(eng)
            for g, pr in enumerate(probs):
                mu, var, ei, acq = (eng.fetch(k, g) for k in ARRAYS)
                assert mu.tobytes() == base[g]["mu"].tobytes() and var.tobytes() == base[g]["var"].tobytes()
                if b2 == best:
                    assert ei.tobytes() == base[g]["ei"].tobytes() and acq.tobytes() == base[g]["acq"].tobytes(), g
                    continue
                X = _coords(eng, g, np.arange(len(mu)))
                acq_ref = ei / P.candidate_cost(X, pr.cost_fix, pr.cost_variable)
                assert acq_ref.tobytes() == acq.tobytes(), g
                pick = np.random.default_rng(g).choice(len(mu), min(256, len(mu)), replace=False)
                pick = pick[var[pick] > 1e-12]
                r = P.check_ei(ei, b2, mu, var, 1.0, pick)
                assert r <= 1.0, (g, r)
                val, i, nn = P.first_argmax(acq)
                assert bests[g] == (val, i, nn), g
    finally:
        eng.timing = False


@pytest.mark.parametrize("task", ["min", "max"])
@pytest.mark.parametrize("causal", [True, False], ids=["causal", "non_causal"])
def test_non_unit_hyper_every_class(cuda_engine_ready, task, causal):
    """s2 in {1e-3, 50}, l in {0.3, 4} on classes 0-4 (the lattice and the box scale with l)."""
    specs = [(1, (15,)), (9, (17, 20)), (17, (12, 64)), (33, (5, 300)), (64, (9, 10))]
    probs, hyper = [], {}
    for j, (n, p) in enumerate(specs):
        s2, l = HYPERS[(j + (0 if causal else 1)) % 4]
        probs.append(_problem(300 + j + 10 * causal, n, p, causal=causal, l=l, cost_variable=j == 1))
        hyper[j] = (s2, l)
    eng = _engine(probs)
    assert sorted(_class(D) for D in _descs(eng)) == [0, 1, 2, 3, 4]
    _fit(eng, hyper)
    best = _best(eng) if task == "min" else float(max(np.max(p.y_int) for p in probs))
    out, bests = _sweep(eng, best, task)
    for g in range(len(probs)):
        _check_fit(eng, g, f"hyper {hyper[g]}")
        _check_set(eng, g, out, bests[g], best, task, f"hyper {hyper[g]} {task}")
    _alone_matches(probs, hyper, best, task, out)


# ---- K3: chunks of the tensor-pipe launch ------------------------------------------------------------------------------------
def _chunk_case(sms, chunk):
    """Class-2 sets whose items make the chunk `chunk`: a long set of L items with a partial last chunk (L % chunk != 0)
    and a one-item set, shorter than one chunk, in the same launch."""
    L = (chunk - 1) * sms + 1 if chunk > 1 else 3
    if L % chunk == 0:
        L += 1
    rows = (L * TILE - 1) // 100            # rows * 100 candidates: exactly L items
    return [_problem(400 + chunk, 33, (rows, 100)), _problem(410 + chunk, 17, (7, 64), causal=False)]


@pytest.mark.parametrize("chunk", [1, 2, 3])
def test_mma_chunks(cuda_engine_ready, chunk):
    sms = _sms()
    probs = _chunk_case(sms, chunk)
    eng = _engine(probs)
    descs = _descs(eng)
    assert [_class(D) for D in descs] == [2, 2]
    assert _chunk(descs, eng.num_sms) == chunk
    if chunk > 1:
        assert _items(descs[0]) % chunk != 0 and _items(descs[1]) < chunk
    _fit(eng)
    best = _best(eng)
    out, bests = _sweep(eng, best, "min")
    for g in range(2):
        _check_set(eng, g, out, bests[g], best, "min", f"chunk {chunk}", informative=True)
    _alone_matches(probs, None, best, "min", out)


def test_mma_chunk_lowered_by_shared_memory(cuda_engine_ready):
    """n = 48, p_last = 16: the lead-row table of a chunk of more than 5 items exceeds 160 KB, so the host lowers the chunk."""
    sms = _sms()
    items = 6 * sms + 3
    probs = [_problem(420, 48, (items * TILE // 16, 16))]
    eng = _engine(probs)
    D = eng.h_sets[0]
    want = min(-(-_items(D) // eng.num_sms), MAX_CHUNK)
    got = _chunk(_descs(eng), eng.num_sms)
    assert got < want, (got, want)
    print(f"  chunk lowered from {want} to {got} by the shared-memory loop")
    _fit(eng)
    best = _best(eng)
    out, bests = _sweep(eng, best, "min")
    _check_set(eng, 0, out, bests[0], best, "min", f"chunk {got} (lowered)", informative=True)


# ---- K3: rank slices --------------------------------------------------------------------------------------------------------
def test_rank_slices(cuda_engine_ready):
    """World size 3 over a class-1 and a class-2 set (non-causal; p_last = 97): slices that begin inside a grid row
    (off0 != 0), rank shares that take chunk > 1.  Every slice is bit-identical to the whole-set sweep (whose chunk is
    different: the chunk does not change the bits)."""
    sms = _sms()
    scale = sms / 148.0
    p_last = 97
    probs = [_problem(501, 10, (int(1.2e6 * scale) // p_last, p_last), causal=False),
             _problem(502, 30, (int(6e5 * scale) // p_last, p_last), causal=False)]
    whole = _engine(probs)
    assert [_class(D) for D in _descs(whole)] == [1, 2]
    _fit(whole)
    best = _best(whole)
    wout, wbests = _sweep(whole, best, "min")
    for g in range(2):
        _check_set(whole, g, wout, wbests[g], best, "min", "whole")
    chunks, mid_row = {_chunk(_descs(whole), whole.num_sms)}, set()
    for r in range(3):
        eng = _engine(probs, rank=r, world_size=3)
        _fit(eng)
        out, _ = _sweep(eng, best, "min")
        chunks.add(_chunk(_descs(eng), eng.num_sms))
        for g in eng.active:
            D = eng.h_sets[eng.local_of[g]]
            if D.g_begin % p_last:
                mid_row.add((g, r))
            for k in ARRAYS:
                assert out[g][k].tobytes() == wout[g][k][D.g_begin:D.g_begin + D.g_count].tobytes(), (r, g, k)
    print(f"  rank slices: chunks {sorted(chunks)}, slices starting mid-row {sorted(mid_row)}")
    assert {g for g, _ in mid_row} == {0, 1}
    assert len([c for c in chunks if c > 1]) >= 2


# ---- explicit points: classes 0, 3, 4 and K7 --------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 15, 16, 17, 33, 48, 64, 128])
def test_explicit_points(cuda_engine_ready, n):
    """evaluate_points at 293 points (class 0 for n <= 16, 3 for n <= 48, 4 beyond), d = 1..4."""
    d = 1 + n % 4
    pr = _problem(600 + n, n, (5,) * d, cost_variable=n % 2 == 1)
    eng = _engine([pr])
    _fit(eng)
    rng = np.random.default_rng(n)
    lo, hi = [t[0] for t in pr.grid], [t[-1] for t in pr.grid]
    X = rng.uniform(lo, hi, (293, d))
    X[:2] = pr.x_int[:2] if n >= 2 else X[:2]
    best = _best(eng)
    runs = [eng.evaluate_points(0, X, best, "min") for _ in range(2)]
    for k in runs[0]:
        assert runs[0][k].tobytes() == runs[1][k].tobytes(), k
    o = runs[0]
    path = "mma" if FMA_MAX_N < n <= MMA_MAX_N else "subst"
    _check_fit(eng, 0, "points")
    _check_values(_state(eng, 0), X, o["m"], o["v"], o, best, "min", pr.cost_fix, pr.cost_variable, path, False,
                  f"points n={n} d={d} ({path})")


@pytest.mark.parametrize("n", [1, 31, 32, 33, 64, 65, 128])
def test_k7_values(cuda_engine_ready, n):
    """acquisition_gradients' mu, var, ei, acq at 83 points (a partial last batch of 8), from K7's own m, v and the fetched
    L, alpha (column-oriented substitution by division)."""
    d = 1 + n % 4
    pr = _problem(700 + n, n, (6,) * d, causal=n != 32, cost_variable=n % 2 == 0)
    eng = _engine([pr])
    _fit(eng, {0: (50.0, 0.3)} if n == 65 else None)
    lo, hi = [t[0] for t in pr.grid], [t[-1] for t in pr.grid]
    X = np.random.default_rng(n).uniform(lo, hi, (83, d))
    best = _best(eng)
    for task in ("min", "max"):
        o = eng.acquisition_gradients(0, X, best, task)
        o2 = eng.acquisition_gradients(0, X, best, task)
        for k in ARRAYS:
            assert o[k].tobytes() == o2[k].tobytes(), k
        _check_values(_state(eng, 0), X, o["m"], o["v"], o, best, task, pr.cost_fix, pr.cost_variable, "subst", False,
                      f"K7 n={n} d={d} {task}")
