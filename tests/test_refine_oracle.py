"""CPU checks of the acquisition-gradient feature (K7): the oracle's analytic gradients against central differences of the
existing oracle functions, the oracle's L-BFGS-B refinement, the ctypes mirrors of the new ABI structs, the agent's flag
and the new entry points' failure without a device."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from helpers import make_case
from oracle import cbo_oracle as O
from oracle import refine_oracle as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_state(ora):
    """(posterior, keyword arguments of R.acquisition_gradients) of a make_case oracle dict."""
    if ora["causal"]:
        f = O.prior_factors(ora["gp"], ora["cond"], ora["cols"])
        mI, vI = O.do_prior_factorised(ora["gp"], f, ora["cols"], ora["XI"], precise=True)
        post = O.posterior_fit(ora["XI"], ora["yI"], mI, vI, form="diff")
        kw = dict(gp=ora["gp"], factors=f, intervened_cols=ora["cols"])
    else:
        post = O.posterior_fit(ora["XI"], ora["yI"], form="diff")
        kw = {}
    return post, dict(kw, fix_costs=ora["fix"], variable_cost=ora["variable"])


def values_at(post, kw, X, best, task):
    """m, v, mu, var, ei, acq at X from the EXISTING oracle functions (the quantities the gradients differentiate)."""
    X = np.atleast_2d(X)
    if post["causal"]:
        m, v = O.do_prior_factorised(kw["gp"], kw["factors"], kw["intervened_cols"], X)
        mu, var = O.posterior_predict(post, X, m, v)
    else:
        m, v = np.zeros(len(X)), np.zeros(len(X))
        mu, var = O.posterior_predict(post, X)
    ei = O.expected_improvement(mu, var, best, task)
    acq = ei / O.point_cost(X, kw["fix_costs"], kw["variable_cost"])
    return dict(m=m, v=v, mu=mu, var=var, ei=ei, acq=acq)


def central_difference(post, kw, X, best, task, h=1e-5):
    d = X.shape[1]
    out = {k: np.empty(X.shape) for k in ("m", "v", "mu", "var", "ei", "acq")}
    for k in range(d):
        e = np.zeros(d)
        e[k] = h
        a, b = values_at(post, kw, X + e, best, task), values_at(post, kw, X - e, best, task)
        for n in out:
            out[n][:, k] = (a[n] - b[n]) / (2 * h)
    return out


def grad_rule_ok(got, ref, rtol=1e-6):
    """1e-6 relative with a floor of 1e-6 max|grad| (per quantity)."""
    floor = max(1e-6 * np.max(np.abs(ref)), 1e-300)
    return np.max(np.abs(got - ref) / np.maximum(np.abs(ref), floor)) <= rtol


CASES = [dict(seed=s, d=d, c=c, N=N, n=n, p=(9,) * d, causal=causal, ard=ard, cost_variable=cv)
         for s, d, c, N, n, causal, ard, cv in [
             (301, 1, 1, 60, 6, True, True, False), (302, 2, 2, 80, 9, True, True, True), (303, 3, 1, 70, 11, True, False, False),
             (304, 4, 2, 50, 12, True, True, True), (305, 1, 0, 40, 5, False, True, True), (306, 2, 1, 40, 8, False, True, False),
             (307, 3, 0, 40, 10, False, False, True), (308, 4, 1, 40, 14, False, True, False)]]


@pytest.mark.parametrize("spec", CASES, ids=lambda s: f"seed{s['seed']}-d{s['d']}-{'causal' if s['causal'] else 'plain'}")
@pytest.mark.parametrize("task", ["min", "max"])
def test_oracle_gradients_match_central_differences(spec, task):
    kw0, ora = make_case(**spec)
    post, kw = oracle_state(ora)
    rng = np.random.default_rng(spec["seed"])
    X = rng.uniform(-1.8, 1.8, (6, spec["d"]))
    best = float(np.min(ora["yI"]) if task == "min" else np.max(ora["yI"]))
    got = R.acquisition_gradients(post, X, best, task, **kw)
    ref = values_at(post, kw, X, best, task)
    for n in ref:      # the values themselves are the existing oracle's
        np.testing.assert_allclose(got[n], ref[n], rtol=1e-9, atol=1e-12 * max(1.0, np.max(np.abs(ref[n]))))
    fd = central_difference(post, kw, X, best, task)
    for n in ("m", "v", "mu", "var", "ei", "acq"):
        if not post["causal"] and n in ("m", "v"):
            assert np.all(got["d" + n] == 0.0)
            continue
        assert grad_rule_ok(got["d" + n], fd[n]), (n, got["d" + n], fd[n])


@pytest.mark.parametrize("spec", CASES[:4] + CASES[5:6], ids=lambda s: f"seed{s['seed']}-d{s['d']}")
def test_oracle_refine_never_lowers_and_stays_in_box(spec):
    kw0, ora = make_case(**spec)
    post, kw = oracle_state(ora)
    best = float(np.min(ora["yI"]))
    ref = O.sweep_set(ora["gp"], ora["cond"], ora["cols"], ora["XI"], ora["yI"], ora["tables"], best, "min",
                      fix_costs=ora["fix"], variable_cost=ora["variable"], causal=ora["causal"], form="diff")
    r = R.refine_set(post, ref["x"], ora["tables"], best, "min", **kw)
    assert r["value"] >= r["start_value"]
    assert r["value"] >= ref["val"] * (1 - 1e-9)
    lo = np.array([t.min() for t in ora["tables"]])
    hi = np.array([t.max() for t in ora["tables"]])
    assert np.all(r["x"] >= lo) and np.all(r["x"] <= hi)


def test_struct_mirrors_match_the_header(tmp_path):
    from cbo_with_oop_b200 import _lib
    cc = shutil.which("cc") or shutil.which("gcc") or shutil.which("g++")
    if cc is None:
        pytest.skip("no host C compiler")
    fields = {"cbo_acq_grad_out": _lib.AcqGradOut, "cbo_refine_result": _lib.RefineResult}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "cbo_b200.h"', "int main(void) {"]
    for st, py in fields.items():
        lines.append(f'printf("{st} sizeof %zu\\n", sizeof({st}));')
        for f, _ in py._fields_:
            lines.append(f'printf("{st} {f} %zu\\n", offsetof({st}, {f}));')
    enums = ["CONVERGED", "MAX_ITER", "LINE_SEARCH_FAILED", "SKIPPED_EXTERNAL", "SKIPPED_POINTS", "SKIPPED_NONFINITE"]
    for e in enums:
        lines.append(f'printf("enum {e} %d\\n", (int)CBO_REFINE_{e});')
    lines.append("return 0; }")
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = {}
    for line in subprocess.check_output([str(exe)], text=True).splitlines():
        a, b, c = line.split()
        got[(a, b)] = int(c)
    for st, py in fields.items():
        assert got[(st, "sizeof")] == C.sizeof(py)
        for f, _ in py._fields_:
            assert got[(st, f)] == getattr(py, f).offset, (st, f)
    assert [got[("enum", e)] for e in enums] == sorted(_lib.REFINE_STATUS)


def test_argument_parser_refinement_defaults_off():
    from src.ArgumentParser import ArgumentParser
    assert ArgumentParser().parse(argv=[]).refine_acquisition is False
    assert ArgumentParser().parse(argv=["--refine_acquisition"]).refine_acquisition is True


NO_DEVICE = r"""
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from cbo_with_oop_b200 import _lib
lib = _lib.load()
h = (_lib.SetDesc * 1)()
h[0].d, h[0].n_int, h[0].p[0], h[0].g_total, h[0].g_count, h[0].cost_fix = 1, 3, 4, 4, 4, 1.0
h[0].grid[0] = 256
h[0].L, h[0].alpha, h[0].x_int = 256, 256, 256
ws = lib.cbo_refine_workspace_bytes(h, 1)
assert ws >= 256, ws
rc1 = lib.cbo_refine(h, C.c_void_p(256), 1, 0.0, 1, C.c_void_p(256), 5, 1e-7, C.c_void_p(256), ws, C.c_void_p(256), None)
e1 = lib.cbo_last_error().decode()
rc2 = lib.cbo_acq_grad(h, C.c_void_p(256), C.c_void_p(256), 3, 0.0, 1, C.c_void_p(256), ws, C.c_void_p(256), None)
e2 = lib.cbo_last_error().decode()
print(rc1, rc2, e1, "|", e2)
assert rc1 > 0 and rc2 > 0, (rc1, rc2, e1, e2)
"""


def test_entry_points_fail_without_a_device():
    """With no visible CUDA device the new entry points return a CUDA error (no CPU fallback).  Run in a child process with
    the devices hidden, so that the placeholder pointers can never reach a real GPU."""
    from cbo_with_oop_b200.build import build_library
    build_library()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", NO_DEVICE, ROOT], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_argument_validation_of_the_new_entry_points():
    from cbo_with_oop_b200.build import build_library
    build_library()
    from cbo_with_oop_b200 import _lib
    lib = _lib.load()
    h = (_lib.SetDesc * 1)()
    h[0].d, h[0].n_int, h[0].p[0], h[0].g_total, h[0].g_count, h[0].cost_fix = 1, 3, 4, 4, 4, 1.0
    assert lib.cbo_refine(h, None, 1, 0.0, 1, None, 5, 1e-7, None, 0, None, None) == -1
    assert b"d_sets" in lib.cbo_last_error()
    assert lib.cbo_refine(h, C.c_void_p(256), 1, 0.0, 2, C.c_void_p(256), 5, 1e-7, None, 0, C.c_void_p(256), None) == -1
    assert b"task_sign" in lib.cbo_last_error()
    assert lib.cbo_refine(h, C.c_void_p(256), 1, 0.0, 1, C.c_void_p(256), -1, 1e-7, None, 0, C.c_void_p(256), None) == -1
    assert b"max_iter" in lib.cbo_last_error()
    assert lib.cbo_acq_grad(h, C.c_void_p(256), None, 3, 0.0, 1, None, 0, None, None) == -1
    assert b"NULL" in lib.cbo_last_error()
    h[0].causal, h[0].prior_external = 1, 1
    assert lib.cbo_acq_grad(h, C.c_void_p(256), C.c_void_p(256), 3, 0.0, 1, None, 0, C.c_void_p(256), None) == -1
    assert b"supplied by the caller" in lib.cbo_last_error()
