"""Measured cost of the opt-in acquisition refinement (K7, csrc/refine.cu) on one GPU:

  * BASELINE.json configs[4] with 2 exploration sets (N = 1e4 observational rows, 1e6-point grids, d = 3): wall time of
    SweepEngine.refine after a post-observation sweep, iterations and gain value / start_value per set, and the time of
    one prior-gradient pass (refine_prior_kernel, torch.profiler) against its HBM-byte and FP64 bounds;
  * the shipped-data configurations (inputs from tests/golden/golden_*.npz, as bench.py's small_configs): trial time, refine
    time, iterations and gains per set;
  * the card name and power limit, queried in the same run.

    python tools/refine_probe.py --out DIR        (writes DIR/refine_probe.json and prints it)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12          # HGX B200 data sheet, one GPU
FP64_FLOPS = 36.4e12      # measured DFMA issue rate of a B200 (profiles/fp64_peak_r01.json)
STEP_MS_N1E4 = 5880.0     # the post-observation step of BASELINE configs[4] the 1 % target refers to


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def events_ms(fn, n, warm):
    import torch
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts)), r


def per_set(grid, out):
    return [{"grid_value": float(g), "value": float(v), "gain": (float(v / g) if g else None), "status": st}
            for g, v, st in zip(grid.set_values, out.set_values, out.refine_status)]


def iterations(eng, grid, best, task):
    """Iterations per set of one refine call (read from the library's result records)."""
    import ctypes as C
    import torch
    from cbo_with_oop_b200 import _lib
    A = len(eng.active)
    x0 = np.full((A, _lib.CBO_MAX_D), np.nan)
    for li, g in enumerate(eng.active):
        pr = eng.problems[g]
        ii = np.unravel_index(int(grid.set_indices[g]), [len(t) for t in pr.grid])
        x0[li, :pr.d] = [pr.grid[k][ii[k]] for k in range(pr.d)]
    ws = torch.empty((eng.lib.cbo_refine_workspace_bytes(eng.h_sets, A),), dtype=torch.uint8, device=eng.device)
    d_x0 = torch.from_numpy(x0.reshape(-1)).to(eng.device)
    res = torch.empty((A * C.sizeof(_lib.RefineResult),), dtype=torch.uint8, device=eng.device)
    _lib.check(eng.lib.cbo_refine(eng.h_sets, C.c_void_p(eng.d_sets.data_ptr()), A, float(best), 1 if task == "min" else -1,
                                  C.c_void_p(d_x0.data_ptr()), 30, 1e-7, C.c_void_p(ws.data_ptr()), ws.numel(),
                                  C.c_void_p(res.data_ptr()), eng._stream()), "cbo_refine")
    rr = (_lib.RefineResult * A).from_buffer_copy(res.cpu().numpy().tobytes())
    return [int(r.iterations) for r in rr]


def prior_pass(eng, g):
    """refine_prior_kernel time of one pass over set g (8 points, cbo_acq_grad) by torch.profiler, with its bounds."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    pr = eng.problems[g]
    rng = np.random.default_rng(7)
    X = rng.uniform(-2, 2, (8, pr.d))
    for _ in range(3):
        eng.acquisition_gradients(g, X)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            eng.acquisition_gradients(g, X)
        torch.cuda.synchronize()
    us = [e.device_time for e in prof.events() if "refine_prior_kernel" in e.name and e.device_time > 0]
    t = float(np.median(us)) * 1e-6
    npad = (pr.x_obs_int.shape[0] + 127) // 128
    slabs = npad * (npad + 1) // 2 * 8
    nbytes = slabs * 128 * 16 * 8
    flops = slabs * 128 * 16 * 8 * (1 + pr.d) * 2
    tb, tf = nbytes / HBM_BPS, flops / FP64_FLOPS
    return {"kernel_ms": t * 1e3, "launches_profiled": len(us), "bytes": nbytes, "flops": flops,
            "byte_bound_ms": tb * 1e3, "fp64_bound_ms": tf * 1e3, "bound": "fp64" if tf > tb else "hbm",
            "share_of_bound": max(tb, tf) / t, "achieved_tbps": nbytes / t * 1e-12, "achieved_tflops": flops / t * 1e-12}


def targets(res):
    """The bars the refinement is held to, with what was measured against each."""
    t = {}
    b = res.get("baseline_config4_2sets")
    if b:
        t["refine_le_1pct_of_5880ms_step"] = {"measured_pct": 100 * b["refine_share_of_step_5880ms"],
                                              "met": b["refine_share_of_step_5880ms"] <= 0.01}
        pp = b["prior_gradient_pass"]
        t["prior_pass_ge_50pct_of_bound"] = {"measured_pct": 100 * pp["share_of_bound"], "bound": pp["bound"],
                                             "met": pp["share_of_bound"] >= 0.5}
    for row in res.get("small_configs", []):
        if row["config"].startswith("simplified_coral"):
            t["simplified_coral_refine_le_1ms"] = {"measured_ms": row["refine_ms"], "met": row["refine_ms"] <= 1.0}
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--skip-large", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("refine_probe.py needs a CUDA device")
    from cbo_with_oop_b200.engine import SweepEngine
    from cbo_with_oop_b200.fixtures import CONFIGS, golden_path, load_golden_problems
    from cbo_with_oop_b200.synthetic import best_of, scaled_set
    res = {"card": card(), "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
           "bounds": {"hbm_bytes_per_s": HBM_BPS, "fp64_flops_per_s": FP64_FLOPS}}
    rows = []
    for config, label in CONFIGS.items():
        if not os.path.exists(golden_path(config)):
            continue
        problems, best, task = load_golden_problems(config, device_fit=True)
        eng = SweepEngine(problems, device="cuda:0")
        eng.sweep(best, task)
        trial_ms, _, grid = events_ms(lambda: eng.sweep(best, task), 10, 3)
        ref_ms, ref_min, out = events_ms(lambda: eng.refine(grid, best, task), 10, 3)
        rows.append({"config": label, "sets": len(problems), "trial_ms": trial_ms, "refine_ms": ref_ms, "refine_ms_min": ref_min,
                     "iterations": iterations(eng, grid, best, task), "sets_detail": per_set(grid, out)})
        del eng
    res["small_configs"] = rows
    if not args.skip_large:
        problems = [scaled_set(s, n_obs=10_000, p=100, d=3, c=3, n_int=32, device_fit=True) for s in range(2)]
        best = best_of(problems)
        eng = SweepEngine(problems, device="cuda:0")
        eng.sweep(best, "min")
        step_ms, _, grid = events_ms(lambda: eng.sweep(best, "min"), 2, 1)
        ref_ms, ref_min, out = events_ms(lambda: eng.refine(grid, best, "min"), 5, 2)
        res["baseline_config4_2sets"] = {
            "what": "BASELINE.json configs[4] with 2 exploration sets: N = 1e4, 1e6-point grid (d = 3), n_int = 32",
            "post_observation_step_ms": step_ms, "refine_ms": ref_ms, "refine_ms_min": ref_min,
            "refine_share_of_step_5880ms": ref_ms / STEP_MS_N1E4, "refine_share_of_measured_step": ref_ms / step_ms,
            "iterations": iterations(eng, grid, best, "min"), "sets_detail": per_set(grid, out),
            "prior_gradient_pass": prior_pass(eng, 0)}
    res["targets"] = targets(res)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "refine_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
