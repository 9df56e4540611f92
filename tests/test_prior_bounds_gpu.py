"""The causal-prior kernels against the error bounds of oracle/prior_bounds.py, on every work decomposition they have.

K1b (prior_eval.cu) chooses its decomposition from the number of CTAs its workspace holds.  A workspace of
cbo_prior_workspace_bytes(sets, n, c) bytes holds exactly c of them (the grid layout is the larger one for every case
here, test_workspace_step_is_one_scratch_slot), so tiny grids reach every branch: one item per tile (grid mode), segments
of M's triangle (chunk = 1, 2, 3, with a partial last piece), folded column blocks (nsplit = 2, 3, 4, the ragged last
block owned by sp = 0 and by sp != 0).  _mirror repeats the host's choice in Python; every case asserts the branch it was
built for, and the launch count that goes with it.  K1p (prior_pair.cu) and K1c (prior_rows.cu) are held to the same
kind of bound.

Every evaluation starts from NaN in m, v (m_int, v_int) and in the workspace -- an unwritten output or an unread
partial then fails instead of passing on stale memory -- and runs twice with bit-identical results.  Run with -s to see
the worst error of each case as a fraction of its bound."""
import ctypes as C

import numpy as np
import pytest

from helpers import make_case
from oracle import cbo_oracle as O
from oracle import prior_bounds as B

pytestmark = pytest.mark.gpu

TILE = BLK = 128
PARTIAL_FLOOR = 1024


# ---- Python mirror of prior_eval_impl's decomposition (csrc/prior_eval.cu) -----------------------------------------
def _G(n, chunk):
    if n <= 0:
        return 0
    q, r = divmod(n, chunk)
    return chunk * q * (q + 1) // 2 + r * (q + 1)


def _F(nJ, chunk):
    return _G(nJ - 1, chunk) + nJ


def _mirror(sets, ctas):
    """sets: [(tiles, nJ)] of the sets the general kernel evaluates; ctas: CTAs the workspace holds (<= SMs)."""
    tiles = sum(t for t, _ in sets)
    chunk, nsplit = 0, 1
    if tiles < 2 * ctas:
        nJmax = max([nJ for t, nJ in sets if t] + [1])
        budget = min(4 * ctas + PARTIAL_FLOOR, 4 * ctas)
        for c in range(1, nJmax + 1 if nJmax > 1 else 1):
            if sum(t * _F(nJ, c) for t, nJ in sets) <= budget:
                chunk = c
                break
        if chunk == 0:
            nsplit = -(-2 * ctas // tiles)
            while nsplit > 1 and sum(t * min(nsplit, max(nJ // 2, 1)) for t, nJ in sets) > 4 * ctas + PARTIAL_FLOOR:
                nsplit -= 1
    mode = "chunk" if chunk else ("fold" if nsplit > 1 else "grid")
    ns = [min(nsplit, max(nJ // 2, 1)) for _, nJ in sets]
    owner = []
    for n, (_, nJ) in zip(ns, sets):
        r = (nJ - 1) % (2 * n)
        owner.append(r if r < n else 2 * n - 1 - r)
    return dict(mode=mode, chunk=chunk, nsplit=nsplit, ns=ns, owner=owner, launches=1 if mode == "grid" else 2)


# ---- engine plumbing ----------------------------------------------------------------------------------------------
def _engine(specs, **kw):
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    problems = [s if isinstance(s, SetProblem) else SetProblem(**make_case(**s)[0]) for s in specs]
    eng = SweepEngine(problems, **kw)
    eng.build_tables()
    eng.prior_precompute()
    return eng


def _shape(eng, ids):
    return [(-(-eng.h_sets[i].g_count // TILE), -(-eng.h_sets[i].n_obs // BLK)) for i in ids]


def _ws_bytes(eng, ids, c):
    h, _, n = eng._subset(ids)
    return int(eng.lib.cbo_prior_workspace_bytes(h, n, c))


def _nan_ws(eng, nbytes):
    import torch
    return torch.full((-(-nbytes // 8),), float("nan"), dtype=torch.float64, device=eng.device)


def _eval0(eng, ids, ws, nbytes):
    """One cbo_prior_eval(which = 0) over the sets `ids` from NaN outputs; returns (launches, {id: (m, v)})."""
    import torch
    from cbo_with_oop_b200 import _lib
    for i in ids:
        eng.buf[i]["m"].fill_(float("nan"))
        eng.buf[i]["v"].fill_(float("nan"))
    h, dptr, n = eng._subset(ids)
    l0 = eng.launches
    _lib.check(eng.lib.cbo_prior_eval(h, dptr, n, 0, C.c_void_p(ws.data_ptr()), nbytes, eng._stream()), "cbo_prior_eval")
    torch.cuda.synchronize()
    return eng.launches - l0, {i: (eng.fetch("m", i).copy(), eng.fetch("v", i).copy()) for i in ids}


def _run(eng, ids, c=None):
    """Evaluate the sets `ids` on a workspace of c CTAs (None: the engine's own), twice from NaN; the two runs must agree
    bit for bit.  Returns (launches per run, {id: (m, v)})."""
    if c is None:
        ws, nbytes = eng.prior_ws, eng.prior_ws.numel()
    else:
        nbytes = _ws_bytes(eng, ids, c)
        ws = _nan_ws(eng, nbytes)
    runs = []
    for _ in range(2):
        ws.fill_(0xFF if c is None else float("nan"))     # (0xFF bytes: the engine's uint8 workspace reads as NaN)
        runs.append(_eval0(eng, ids, ws, nbytes))
    (l1, o1), (l2, o2) = runs
    assert l1 == l2
    for i in ids:
        np.testing.assert_array_equal(o1[i][0], o2[i][0], err_msg=f"set {i}: m differs between two identical runs")
        np.testing.assert_array_equal(o1[i][1], o2[i][1], err_msg=f"set {i}: v differs between two identical runs")
    return l1, o1


def _check_bound_a(eng, i, m, v, rows=None, label=""):
    """Bound A for set i (whole grid, or the flat grid indices `rows`) from the tables, M and w on the device."""
    D = eng.h_sets[i]
    tabs = [eng.fetch(f"tab{k}", i) for k in range(D.d)]
    rows = np.arange(D.g_count) if rows is None else np.asarray(rows)
    ref = B.prior_ref(B.grid_u(tabs, rows), eng.fetch("M", i), eng.fetch("w", i), D.s2, D.noise, D.d)
    rm, rv = B.check_prior(m[rows], v[rows], ref)
    print(f"  {label} set {i} (N={D.n_obs}, d={D.d}, g={D.g_count}): m {rm:.2e}  v {rv:.2e} of bound A")
    assert rm <= 1.0 and rv <= 1.0, (label, i, rm, rv)
    return rm, rv


def _branch(eng, ids, c, expect, launches):
    """Assert the decomposition the mirror predicts for `ids` on c CTAs, and the launch count that goes with it."""
    got = _mirror(_shape(eng, ids), min(c, eng.num_sms))
    for k, want in expect.items():
        assert got[k] == want, f"the case was built for {k} = {want}, the mirror says {got[k]}"
    assert launches == got["launches"], f"{launches} launches for a {got['mode']} launch"
    return got


# ---- workspace sizing ---------------------------------------------------------------------------------------------
def test_workspace_step_is_one_scratch_slot(cuda_engine_ready):
    """bytes(c + 1) - bytes(c) is one CTA's partial slots plus its U scratch slot: a workspace of bytes(c) holds c CTAs."""
    eng = _engine([dict(seed=501, N=300, d=2, c=1, n=3, p=(9, 11)), dict(seed=502, N=1216, d=1, c=1, n=2, p=(128,))])
    for ids in ([0], [1], [0, 1]):
        npad = max(eng.h_sets[i].n_obs_pad for i in ids)
        per_cta = (4 * 2 * TILE + TILE * npad) * 8
        steps = {_ws_bytes(eng, ids, c + 1) - _ws_bytes(eng, ids, c) for c in range(1, 9)}
        assert steps == {per_cta}, (ids, steps, per_cta)


# ---- grid mode: every ragged variant, more than 32 sets in one call -------------------------------------------------
LC = [1, 15, 16, 17, 31, 32, 33, 48, 63, 64, 65, 127, 128]
LIVE_LAST = [0, 1, 8, 9, 57, 64, 65, 120, 127]


def _grid_specs():
    specs = []
    for k in (1, 2):
        for j, lc in enumerate(LC):
            r = LIVE_LAST[(j + 4 * k) % len(LIVE_LAST)]
            specs.append(dict(seed=600 + 20 * k + j, N=BLK * k + lc, d=1, c=1, n=2, p=(TILE * (1 + (j % 2)) + (r or TILE),)))
    # ten more pair-ineligible sets: d = 4, and d = 2 / 3 with N > 256; one set of a single column block
    more = [(150, (3, 4, 5, 4)), (193, (2, 3, 4, 8)), (257, (3, 3, 3, 5)), (270, (15, 13)), (300, (5, 6, 7)), (320, (16, 16)),
            (380, (3, 7, 7)), (100, (2, 2, 4, 16)), (129, (321,)), (64, (200,))]
    for j, (N, p) in enumerate(more):
        specs.append(dict(seed=660 + j, N=N, d=len(p), c=1 + j % 2, n=2, p=p))
    return specs


def test_grid_mode_every_ragged_variant_in_one_call_of_36_sets(cuda_engine_ready):
    """36 sets, N = 128 k + Lc for every Lc class (all three consume_ragged_block variants, the regular tiling just past
    64, the 16-slab padding), last tiles with 0..127 live rows, d = 1..4, through ONE CTA (items of different LIVE and
    ragged state back to back in its ring) and past the 32 sets PriorBases holds (the descriptor walk).  Each set must be
    bit-identical to the same set run alone: an item's arithmetic depends only on its set and tile."""
    specs = _grid_specs()
    assert len(specs) == 36
    eng = _engine(specs)
    ids = list(range(len(specs)))
    assert int(eng.lib.cbo_prior_pair_items(eng.h_sets, len(ids), eng.num_sms)) == 0
    launches, out = _run(eng, ids, c=1)
    _branch(eng, ids, 1, dict(mode="grid"), launches)
    worst = [0.0, 0.0]
    for i in ids:
        rm, rv = _check_bound_a(eng, i, *out[i], label="grid c=1, 36 sets:")
        worst = [max(worst[0], rm), max(worst[1], rv)]
    print(f"grid mode, 36 sets: worst m {worst[0]:.2e}, v {worst[1]:.2e} of bound A")
    for i in ids:
        launches, alone = _eval0(eng, [i], _nan_ws(eng, _ws_bytes(eng, [i], 1)), _ws_bytes(eng, [i], 1))
        _branch(eng, [i], 1, dict(mode="grid"), launches)
        np.testing.assert_array_equal(alone[i][0], out[i][0], err_msg=f"set {i}: m alone != m among 36 sets")
        np.testing.assert_array_equal(alone[i][1], out[i][1], err_msg=f"set {i}: v alone != v among 36 sets")


# ---- small launches: segments and folded column blocks --------------------------------------------------------------
SPLIT_CASES = {
    # id: (set spec, CTAs, expected decomposition)
    "chunk1": (dict(seed=701, N=300, d=2, c=1, n=2, p=(9, 11)), 2, dict(mode="chunk", chunk=1)),
    "chunk2_partial_piece": (dict(seed=702, N=400, d=3, c=1, n=2, p=(4, 5, 6)), 2, dict(mode="chunk", chunk=2)),
    "chunk3_partial_pieces": (dict(seed=703, N=801, d=1, c=2, n=2, p=(100,)), 4, dict(mode="chunk", chunk=3)),
    "fold_ns1": (dict(seed=704, N=321, d=1, c=1, n=2, p=(100,)), 1, dict(mode="fold", nsplit=2, ns=[1])),
    "fold2_ragged_sp0": (dict(seed=705, N=401, d=2, c=1, n=2, p=(8, 16)), 1, dict(mode="fold", ns=[2], owner=[0])),
    "fold2_ragged_sp1": (dict(seed=706, N=680, d=1, c=2, n=2, p=(128,)), 1, dict(mode="fold", ns=[2], owner=[1])),
    "fold3_ragged_sp1": (dict(seed=707, N=905, d=4, c=1, n=2, p=(4, 4, 4, 4)), 3, dict(mode="fold", ns=[3], owner=[1])),
    "fold4_ragged_sp0": (dict(seed=708, N=927, d=3, c=1, n=2, p=(4, 4, 8)), 2, dict(mode="fold", ns=[4], owner=[0])),
    "fold4_ragged_sp1": (dict(seed=709, N=1216, d=1, c=1, n=2, p=(128,)), 2, dict(mode="fold", ns=[4], owner=[1])),
}


@pytest.mark.parametrize("case", sorted(SPLIT_CASES))
def test_split_decompositions(cuda_engine_ready, case):
    spec, c, expect = SPLIT_CASES[case]
    eng = _engine([spec])
    launches, out = _run(eng, [0], c=c)
    _branch(eng, [0], c, expect, launches)
    _check_bound_a(eng, 0, *out[0], label=f"{case} (c={c}):")


def _points_eval(eng, X, c):
    """Explicit points X through the table and prior kernels on a workspace of c CTAs, from NaN; returns (launches of the
    prior call, m, v, the points' table (mc, N))."""
    import torch
    from cbo_with_oop_b200 import _lib
    from cbo_with_oop_b200._lib import SetDesc
    D0, dev = eng.h_sets[0], eng.device
    mc = X.shape[0]
    D = SetDesc.from_buffer_copy(bytes(D0))
    pts = torch.from_numpy(np.ascontiguousarray(X).reshape(-1)).to(dev)
    m = torch.full((mc,), float("nan"), dtype=torch.float64, device=dev)
    v = torch.full((mc,), float("nan"), dtype=torch.float64, device=dev)
    tab0 = torch.full((mc * D0.n_obs_pad,), float("nan"), dtype=torch.float64, device=dev)
    D.points, D.tab[0] = pts.data_ptr(), tab0.data_ptr()
    D.p[0] = mc
    for k in range(1, _lib.CBO_MAX_D):
        D.p[k] = 1
    D.g_total, D.g_begin, D.g_count = mc, 0, mc
    D.m, D.v, D.mu, D.var, D.ei, D.acq = m.data_ptr(), v.data_ptr(), None, None, None, None
    h = (SetDesc * 1)(D)
    d_desc = torch.frombuffer(bytearray(bytes(h)), dtype=torch.uint8).to(dev)
    dptr, st = C.c_void_p(d_desc.data_ptr()), eng._stream()
    _lib.check(eng.lib.cbo_build_tables(h, dptr, 1, st), "cbo_build_tables")
    nbytes = int(eng.lib.cbo_prior_workspace_bytes(h, 1, c))
    ws = _nan_ws(eng, nbytes)
    l0 = eng.launches
    _lib.check(eng.lib.cbo_prior_eval(h, dptr, 1, 0, C.c_void_p(ws.data_ptr()), nbytes, st), "cbo_prior_eval")
    torch.cuda.synchronize()
    nl = eng.launches - l0
    shape = [(-(-mc // TILE), -(-D0.n_obs // BLK))]
    tab = tab0.cpu().numpy().reshape(mc, D0.n_obs_pad)[:, :D0.n_obs]
    return nl, shape, m.cpu().numpy(), v.cpu().numpy(), tab


@pytest.mark.parametrize("c,expect", [(1, dict(mode="grid")), (2, dict(mode="fold", ns=[1])), (4, dict(mode="chunk", chunk=2))],
                         ids=["grid", "fold_ns1", "chunk2"])
def test_explicit_points(cuda_engine_ready, c, expect):
    """293 explicit points (three tiles, 37 live rows in the last) of an N = 300 set: the points' own table is fetched
    and u is its rows (d = 1 for the kernel)."""
    eng = _engine([dict(seed=711, N=300, d=3, c=1, n=2, p=(3, 3, 3))])
    X = np.random.default_rng(711).uniform(-2.5, 2.5, (293, 3))
    runs = [_points_eval(eng, X, c) for _ in range(2)]
    np.testing.assert_array_equal(runs[0][2], runs[1][2])
    np.testing.assert_array_equal(runs[0][3], runs[1][3])
    nl, shape, m, v, tab = runs[0]
    got = _mirror(shape, c)
    for k, want in expect.items():
        assert got[k] == want, (k, got[k], want)
    assert nl == got["launches"]
    ref = B.prior_ref(tab.astype(np.longdouble), eng.fetch("M", 0), eng.fetch("w", 0), eng.h_sets[0].s2, eng.h_sets[0].noise, 1)
    rm, rv = B.check_prior(m, v, ref)
    print(f"  explicit points (c={c}, {got['mode']}): m {rm:.2e}  v {rv:.2e} of bound A")
    assert rm <= 1.0 and rv <= 1.0


# ---- the production configuration -----------------------------------------------------------------------------------
def test_production_workspace(cuda_engine_ready):
    """The engine's own workspace (one CTA per SM) with >= 2 x SMs tiles: three 1-D sets of ~40 000 candidates at
    N = 145, 160, 192 and a 3-D set at N = 304 (no pair path).  Bound A on every row of the first and last tiles and on 8
    rows of every other tile; a run on one CTA must give the same bits."""
    specs = [dict(seed=721, N=145, d=1, c=2, n=2, p=(40000,)), dict(seed=722, N=160, d=1, c=1, n=2, p=(40001,)),
             dict(seed=723, N=192, d=1, c=2, n=2, p=(39999,)), dict(seed=724, N=304, d=3, c=1, n=2, p=(40, 32, 32))]
    eng = _engine(specs)
    ids = list(range(len(specs)))
    assert int(eng.lib.cbo_prior_pair_items(eng.h_sets, len(ids), eng.num_sms)) == 0
    ctas = eng.num_sms
    assert eng.prior_ws.numel() >= _ws_bytes(eng, ids, ctas)
    launches, out = _run(eng, ids)
    _branch(eng, ids, ctas, dict(mode="grid"), launches)
    rng = np.random.default_rng(720)
    for i in ids:
        g = eng.h_sets[i].g_count
        tiles = -(-g // TILE)
        rows = [np.arange(min(TILE, g)), np.arange((tiles - 1) * TILE, g)]
        rows += [t * TILE + rng.choice(TILE, 8, replace=False) for t in range(1, tiles - 1)]
        _check_bound_a(eng, i, *out[i], rows=np.unique(np.concatenate(rows)), label=f"production ({ctas} CTAs):")
    launches1, one = _run(eng, ids, c=1)
    _branch(eng, ids, 1, dict(mode="grid"), launches1)
    for i in ids:
        np.testing.assert_array_equal(one[i][0], out[i][0], err_msg=f"set {i}: m on 1 CTA != m on {ctas}")
        np.testing.assert_array_equal(one[i][1], out[i][1], err_msg=f"set {i}: v on 1 CTA != v on {ctas}")


# ---- K1p: more than 32 sets ------------------------------------------------------------------------------------------
def test_pair_path_beyond_32_sets(cuda_engine_ready):
    """40 pair-eligible 3-D sets: two pair launches (32 + 8 sets, the second offset into the pair area), 4 kernels.  Bound A
    on every row, and the same bits as the sets run as two engines of 20 (each still >= 148 pair items)."""
    specs = [dict(seed=800 + j, N=20 + 6 * j, d=3, c=1 + j % 2, n=2, p=(8, 5 + j % 3, 6)) for j in range(40)]
    eng = _engine(specs)
    ids = list(range(40))
    assert int(eng.lib.cbo_prior_pair_items(eng.h_sets, 40, eng.num_sms)) >= eng.num_sms
    launches, out = _run(eng, ids)
    assert launches == 4, f"{launches} launches: expected two pair batches of table + GEMM kernels"
    worst = [0.0, 0.0]
    for i in ids:
        rm, rv = _check_bound_a(eng, i, *out[i], label="pair, 40 sets:")
        worst = [max(worst[0], rm), max(worst[1], rv)]
    print(f"pair path, 40 sets: worst m {worst[0]:.2e}, v {worst[1]:.2e} of bound A")
    for half in (0, 1):
        sub = _engine(specs[20 * half:20 * half + 20])
        assert int(sub.lib.cbo_prior_pair_items(sub.h_sets, 20, sub.num_sms)) >= sub.num_sms
        nl, o = _run(sub, list(range(20)))
        assert nl == 2
        for j in range(20):
            np.testing.assert_array_equal(o[j][0], out[20 * half + j][0], err_msg=f"set {20 * half + j}: m")
            np.testing.assert_array_equal(o[j][1], out[20 * half + j][1], err_msg=f"set {20 * half + j}: v")
        del sub


# ---- K1c: the interventional rows ------------------------------------------------------------------------------------
def _eval_rows(eng):
    import torch
    for b in eng.buf:
        if "m_int" in b:
            b["m_int"].fill_(float("nan"))
            b["v_int"].fill_(float("nan"))
    eng.prior_ws.fill_(0xFF)
    l0 = eng.launches
    eng.prior_eval(1)
    torch.cuda.synchronize()
    return eng.launches - l0


def _check_bound_c(eng, i, label):
    D = eng.h_sets[i]
    ref = B.rows_ref(eng.fetch("u_int", i), eng.fetch("M", i), eng.fetch("w", i), D.s2, D.noise)
    rm, rv = B.check_rows(eng.fetch("m_int", i), eng.fetch("v_int", i), ref)
    print(f"  {label} set {i} (N={D.n_obs}, rows={D.n_int}, cancellation {B.cancellation(ref).max():.1e}): "
          f"m {rm:.2e}  v {rv:.2e} of bound C")
    assert rm <= 1.0 and rv <= 1.0, (label, i, rm, rv)


ROWS_CASES = {
    "narrow_1row": [dict(seed=901, N=50, d=1, c=1, n=1, p=(5,))],
    "narrow_4rows_3blocks": [dict(seed=902, N=300, d=2, c=1, n=4, p=(4, 4))],
    "wide_5rows": [dict(seed=903, N=200, d=2, c=2, n=5, p=(4, 4))],
    "wide_32rows": [dict(seed=904, N=130, d=3, c=1, n=32, p=(3, 3, 3))],
    "wide_33rows_2passes": [dict(seed=905, N=129, d=1, c=1, n=33, p=(5,))],
    "wide_128rows_4passes": [dict(seed=906, N=40, d=2, c=1, n=128, p=(4, 4))],
    # one launch, sets of different nJ, k-chunk counts (N = 520, 700: two 32-slab chunks) and row counts
    "mixed_launch": [dict(seed=907, N=1, d=1, c=1, n=3, p=(5,)), dict(seed=908, N=100, d=2, c=2, n=40, p=(4, 4)),
                     dict(seed=909, N=700, d=1, c=1, n=2, p=(5,)), dict(seed=910, N=520, d=3, c=1, n=7, p=(2, 2, 2))],
}


@pytest.mark.parametrize("case", sorted(ROWS_CASES))
def test_rows_kernel(cuda_engine_ready, case):
    eng = _engine(ROWS_CASES[case])
    got = []
    for _ in range(2):
        assert _eval_rows(eng) == 2
        got.append([(eng.fetch("m_int", i).copy(), eng.fetch("v_int", i).copy()) for i in range(len(eng.active))])
    for (m1, v1), (m2, v2) in zip(*got):
        np.testing.assert_array_equal(m1, m2)
        np.testing.assert_array_equal(v1, v2)
    for i in range(len(eng.active)):
        _check_bound_c(eng, i, case)


def test_rows_appended_by_refresh(cuda_engine_ready):
    """Rows appended through set_interventional + refresh (int_row_begin > 0): 1, 2 and 5 at once.  The new rows must meet
    bound C and the earlier rows keep their bits."""
    import torch
    specs = [dict(seed=921, N=150, d=2, c=1, n=4, p=(6, 6)), dict(seed=922, N=600, d=1, c=1, n=3, p=(20,))]
    eng = _engine(specs)
    best = float(min(np.min(p.y_int) for p in eng.problems))
    eng.sweep(best, "min")
    rng = np.random.default_rng(920)
    for g, add in ((0, 1), (0, 2), (1, 5), (1, 1)):
        pr = eng.problems[g]
        n_old = pr.x_int.shape[0]
        before = (eng.fetch("m_int", g).copy(), eng.fetch("v_int", g).copy())
        x_new = np.vstack([pr.x_int, rng.uniform(-2.0, 2.0, (add, pr.d))])
        y_new = np.append(pr.y_int, best - 0.05 * rng.random(add))
        eng.set_interventional(g, x_new, y_new)
        eng.buf[g]["m_int"][n_old:].fill_(float("nan"))
        eng.buf[g]["v_int"][n_old:].fill_(float("nan"))
        eng.prior_ws.fill_(0xFF)
        best = float(min(best, y_new.min()))
        eng.refresh(best, "min", refit=[g])
        torch.cuda.synchronize()
        np.testing.assert_array_equal(eng.fetch("m_int", g)[:n_old], before[0])
        np.testing.assert_array_equal(eng.fetch("v_int", g)[:n_old], before[1])
        _check_bound_c(eng, g, f"appended {add}")


def _dense_1d_problem():
    from cbo_with_oop_b200.engine import SetProblem
    rng = np.random.default_rng(0)
    N = 200
    X = np.sort(rng.uniform(-2.0, 2.0, N))[:, None]
    y = np.sin(2.0 * X[:, 0]) + 0.01 * rng.standard_normal(N)
    gp = O.obs_gp_fit(X, y, 1.0, np.array([0.8]), noise=1e-4, form="diff")
    z = np.zeros((N, 0))
    return SetProblem(x_obs_int=X, x_obs_cond=z, mc_cond=z, alpha_obs=gp["alpha"], kyinv=gp["Kyinv"], ls_int=np.array([0.8]),
                      ls_cond=np.zeros(0), s2=1.0, grid=[np.linspace(-2, 2, 9)], x_int=rng.uniform(-1.8, 1.8, (6, 1)),
                      y_int=rng.standard_normal(6), noise=1e-4, name="dense_1d")


def test_rows_cancelled_cases(cuda_engine_ready):
    """Dense 1-D data with noise 1e-4 (~1e10-fold cancellation) and set 2 of the simplified coral fixture (4e8): a plain
    fp64 sum, or Dot2 without its low word, is far outside bound C here."""
    from cbo_with_oop_b200.fixtures import load_golden_problems
    coral = load_golden_problems("simplified_coral", device_fit=False)[0][2]
    eng = _engine([_dense_1d_problem(), coral])
    assert _eval_rows(eng) == 2
    for i in range(2):
        D = eng.h_sets[i]
        ref = B.rows_ref(eng.fetch("u_int", i), eng.fetch("M", i), eng.fetch("w", i), D.s2, D.noise)
        assert B.cancellation(ref).max() > 1e8, "the case was meant to cancel"
        _check_bound_c(eng, i, "cancelled")
