"""Measured cost of the opt-in hyper-parameter fit of the per-set GPs (K8, csrc/posterior_hyper.cu) on one GPU:

  * the shipped-data configurations (inputs from tests/golden/golden_*.npz, as bench.py's small_configs): time of one
    SweepEngine.fit_hyperparameters call over every set, and per set the fitted (s2, l), the NLL at (1, 1) and at the fit,
    the winning start, its line searches and status;
  * BASELINE.json configs[4] with 2 exploration sets (n_int = 32): the same call, and the post-observation step;
  * one set with n_int = 128 (the largest Gram the library holds);
  * a post-intervention trial (SweepEngine.refresh of one set on simplified_coral) with the fit on and off;
  * the card name and power limit, queried in the same run.

    python tools/hyper_probe.py --out DIR        (writes DIR/hyper_probe.json and prints it)
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

TARGET_CORAL_MS = 2.0        # simplified_coral, 25 sets
TARGET_N128_MS = 10.0        # one set at n_int = 128


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
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def fit_row(eng, label, reps=10):
    """Time of one fit over every set of the engine (the fit's result does not depend on the values it overwrites, so
    repeated calls do identical work), and what it found."""
    ms, ms_min = events_ms(eng.fit_hyperparameters, reps, 2)
    sets = []
    for g in eng.active:
        r = eng.hyper_result(g)
        sets.append({k: r[k] for k in ("variance", "lengthscale", "nll", "nll_start", "start", "iterations", "status",
                                       "jitter_tries")} | {"n_int": int(eng.problems[g].x_int.shape[0])})
    return {"config": label, "sets": len(eng.active), "fit_ms": ms, "fit_ms_min": ms_min, "sets_detail": sets,
            "max_iterations": max(s["iterations"] for s in sets)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--skip-large", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("hyper_probe.py needs a CUDA device")
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    from cbo_with_oop_b200.fixtures import CONFIGS, golden_path, load_golden_problems
    from cbo_with_oop_b200.synthetic import best_of, scaled_set
    res = {"card": card(), "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())}
    rows = []
    for config, label in CONFIGS.items():
        if not os.path.exists(golden_path(config)):
            continue
        problems, best, task = load_golden_problems(config, device_fit=True)
        eng = SweepEngine(problems, device="cuda:0", fit_hyperparameters=True)
        eng.sweep(best, task)
        rows.append(fit_row(eng, label))
        if config == "simplified_coral":
            # a post-intervention trial, the fit on and off (one appended row on set 0, as bench's post_intervention_trial)
            trial = {}
            for on in (False, True):
                probs, best, task = load_golden_problems(config, device_fit=True)
                e = SweepEngine(probs, device="cuda:0", fit_hyperparameters=on)
                out = e.sweep(best, task)
                pr = probs[0]
                x_new = np.vstack([pr.x_int, pr.x_int[-1:] * 0.5])
                y_new = np.append(pr.y_int, pr.y_int[-1])

                def step(e=e, x=x_new, y=y_new, p=pr):
                    e.set_interventional(0, x[:-1], y[:-1])
                    e.set_interventional(0, x, y)
                    return e.refresh(best, task, refit=[0])
                trial["fit_on_ms" if on else "fit_off_ms"] = events_ms(step, 20, 3)[0]
                del e
            res["simplified_coral_post_intervention_trial"] = trial
        del eng
    res["small_configs"] = rows
    rng = np.random.default_rng(5)
    x = np.sort(rng.uniform(-3.0, 3.0, (128, 2)), axis=0)
    y = np.sin(x[:, 0]) * np.cos(x[:, 1]) + 0.05 * rng.standard_normal(128)
    grid = [np.linspace(-3.0, 3.0, 60), np.linspace(-3.0, 3.0, 60)]
    eng = SweepEngine([SetProblem.non_causal(grid, x, y, name="n128")], device="cuda:0", fit_hyperparameters=True)
    eng.sweep(float(y.min()), "min")
    res["one_set_n128"] = fit_row(eng, "one non-causal set, n_int = 128, d = 2", reps=5)
    del eng
    if not args.skip_large:
        problems = [scaled_set(s, n_obs=10_000, p=100, d=3, c=3, n_int=32, device_fit=True) for s in range(2)]
        best = best_of(problems)
        eng = SweepEngine(problems, device="cuda:0", fit_hyperparameters=True)
        eng.sweep(best, "min")
        step_ms, _ = events_ms(lambda: eng.sweep(best, "min"), 2, 1)
        row = fit_row(eng, "BASELINE.json configs[4] with 2 exploration sets: N = 1e4, 1e6-point grid (d = 3), n_int = 32")
        row["post_observation_step_ms_with_fit"] = step_ms
        res["baseline_config4_2sets"] = row
    coral = [r for r in rows if r["config"].startswith("simplified_coral")]
    res["targets"] = {
        "simplified_coral_fit_le_2ms": {"measured_ms": coral[0]["fit_ms"] if coral else None,
                                        "met": bool(coral and coral[0]["fit_ms"] <= TARGET_CORAL_MS)},
        "n128_fit_le_10ms": {"measured_ms": res["one_set_n128"]["fit_ms"], "met": res["one_set_n128"]["fit_ms"] <= TARGET_N128_MS}}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "hyper_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
