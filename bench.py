#!/usr/bin/env python
"""Benchmark of the per-trial acquisition sweep (BASELINE.json metric: EI grid-points/s per trial, all
exploration sets) on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--sets-per-gpu S] [--strong [--sets T]]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload: BASELINE.json configs[4], the synthetic scaled sweep (1e6-point intervention grid per exploration
set, 1e4 observational samples, 32 interventional rows, d = 3 + 3 conditioning columns; SURVEY.md §8d row 5),
weak-scaled: every GPU sweeps `--sets-per-gpu` (default 2) exploration sets, so 8 GPUs run exactly the
16-set configuration.  `--strong` sweeps a fixed number of sets (`--sets`, default 16) on however many GPUs there are
(a count that does not divide by the GPUs makes the partition cut inside sets).
A step = one full post-observation trial: exp tables, prior precompute, prior on x_int and on the grid,
posterior fit, EI / cost, argmax, and (N > 1) the NCCL all-gather + combine of the per-set bests.
`e2e` is the same trial from HOST buffers: upload of the observational design, its targets and the interventional
data, the observational GP fit on the device (the reference's trial starts with it, CBO.py:135), the sweep, and the
read-back of the result.

At N = 1 the same run also reports, in their own blocks (none of them enters `value`):
  full_config   -- one timed step of the FULL 16-set configuration on the one GPU;
  small_configs -- one full trial of each shipped-data configuration (BASELINE.json configs 1-4, tests/golden fixtures);
  cpu_baseline  -- the CPU restatement of the reference on the box's host cores.
One JSON line on stdout (rank 0).  `--impl reference` times the CPU restatement of the reference's arithmetic
(oracle/, the reference itself cannot be installed offline -- DESIGN.md) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sets-per-gpu", type=int, default=2)
    ap.add_argument("--strong", action="store_true", help="fixed total work: --sets exploration sets split over the GPUs")
    ap.add_argument("--sets", type=int, default=16, help="exploration sets of a --strong run")
    ap.add_argument("--n-obs", type=int, default=10_000)
    ap.add_argument("--p", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-config", action="store_true", help="skip the one-step 16-set block of an N = 1 run (about 100 s)")
    ap.add_argument("--no-small-configs", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--direct-candidates", type=int, default=None,
                    help="candidates timed in the reference-faithful one-at-a-time form (default: 16 in the reference arm, 2 in cpu_baseline)")
    ap.add_argument("--strict-selection", action="store_true", help="exit non-zero when the selected intervention differs from profiles/expected_selection.json")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


ARGS = parse()
if ARGS.impl == "reference":
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm must use the box's cores at every N (set before NumPy
    # loads its BLAS; threadpoolctl raises the limit again at run time in case a pool was already created)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "EI grid-points/sec per trial (all exploration sets)"
UNIT = "grid-points/s"
D_INT, C_COND, N_INT = 3, 3, 32
FP64_PEAK_FILE = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r01_prior_eval_traffic.json")
EXPECTED_FILE = os.path.join(ROOT, "profiles", "expected_selection.json")


def workload_config(args, world):
    S = args.sets if args.strong else args.sets_per_gpu * world
    return {
        "workload": "synthetic scaled sweep (BASELINE.json configs[4]): %d exploration sets x %d^3 grid points x %d "
                    "observational samples, d=3 intervened + 3 conditioning columns, %d interventional rows%s"
                    % (S, args.p, args.n_obs, N_INT, "" if args.strong else
                       " -- weak-scaled, %d sets per GPU (16 sets at 8 GPUs is the full configuration; at N = 1 the "
                       "`full_config` block times all 16 sets on the one GPU)" % args.sets_per_gpu),
        "exploration_sets": S, "grid_points_per_set": args.p ** D_INT, "n_obs": args.n_obs, "n_int": N_INT,
        "step": "full post-observation trial: tables + prior precompute + prior(x_int) + posterior fit + prior(grid) + EI/cost + argmax"
                + (" + NCCL all-gather/combine" if world > 1 else ""),
        "l2": "inputs larger than L2: every set streams its 0.8 GB prior matrix M (L2 is 126 MB); no explicit flush",
        "partition": "contiguous FLOP-weighted chunks of (set x grid tile), one per GPU (cbo_with_oop_b200/partition.py)",
    }, S


def blas_threads(n=None):
    """Context manager pinning the BLAS / OpenMP pools to n threads (default: every host core); yields the count."""
    import contextlib
    n = n or os.cpu_count() or 1

    @contextlib.contextmanager
    def cm():
        try:
            from threadpoolctl import threadpool_info, threadpool_limits
            with threadpool_limits(limits=n):
                got = max([i.get("num_threads", 1) for i in threadpool_info()] or [1])
                yield int(got)
        except ImportError:
            yield int(n)
    return cm()


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/cbo_oracle.py) on the host cores.  Only this function touches oracle/.
# ---------------------------------------------------------------------------------------------------------
def cpu_port(problem, alpha_obs, kyinv, sample_pts, seed=0, direct_pts=0, direct_budget_s=150.0):
    """Time the best-effort vectorised CPU port (factorised prior + batched posterior/EI in NumPy/BLAS) on a
    bounded sample of one exploration set and extrapolate linearly to the set's full grid; optionally also the
    reference-faithful form (DoCalculus.py:50-89: one candidate at a time, mean and variance closures separately)."""
    from oracle import cbo_oracle as O
    X = np.hstack([problem.x_obs_int, problem.x_obs_cond])
    d = problem.d
    N = X.shape[0]
    ls = np.concatenate([problem.ls_int, problem.ls_cond])
    gp = dict(X=X, variance=problem.s2, lengthscale=ls, noise=problem.noise, alpha=alpha_obs, Kyinv=kyinv, form="diff")
    cols = list(range(d))
    with blas_threads() as nthreads:
        t0 = time.perf_counter()
        factors = O.prior_factors(gp, X, cols)                      # one-off per set (K1a's work)
        mI, vI = O.do_prior_factorised(gp, factors, cols, problem.x_int)
        post = O.posterior_fit(problem.x_int, problem.y_int, mI, vI, form="diff")
        t_once = time.perf_counter() - t0
        rng = np.random.default_rng(seed)
        G = problem.g_total
        flat = np.sort(rng.choice(G, size=min(sample_pts, G), replace=False))
        ii = np.unravel_index(flat, [len(t) for t in problem.grid])
        Xg = np.stack([problem.grid[k][ii[k]] for k in range(d)], axis=1)
        best = float(problem.y_int.min())
        t0 = time.perf_counter()
        mg, vg = O.do_prior_factorised(gp, factors, cols, Xg, chunk=2048)
        mu, var = O.posterior_predict(post, Xg, mg, vg)
        acq = O.expected_improvement(mu, var, best, "min") / O.point_cost(Xg, np.ones(d), False)
        O.first_argmax(acq)
        t_pts = time.perf_counter() - t0
        per_pt = t_pts / len(flat)
        out = {"points_per_s": G / (t_once + per_pt * G), "one_off_s": t_once, "per_point_s": per_pt, "sample_points": int(len(flat)),
               "sample_s": t_once + t_pts, "threads": nthreads, "host_cores": os.cpu_count()}
        if direct_pts > 0:
            # needs the Cholesky factor of the observational Gram (the reference's GPRegression holds it)
            t0 = time.perf_counter()
            gp_full = O.obs_gp_fit(X, np.zeros(N), problem.s2, ls, problem.noise, form="diff", want_inverse=False)
            gp_full["alpha"] = alpha_obs
            t_fit = time.perf_counter() - t0
            t0, done = time.perf_counter(), 0
            for x in Xg[:direct_pts]:
                O.do_prior_direct(gp_full, X, cols, x[None, :])   # mean closure
                O.do_prior_direct(gp_full, X, cols, x[None, :])   # variance closure (the reference runs predict twice)
                done += 1
                if time.perf_counter() - t0 > direct_budget_s:
                    break
            t_dir = (time.perf_counter() - t0) / done
            out["direct_form"] = {"points_per_s": 1.0 / t_dir, "candidates_timed": done, "s_per_candidate": t_dir,
                                  "obs_gp_factorisation_s": t_fit, "threads": nthreads}
    return out


def run_reference(args, world, rank):
    if rank != 0:
        return
    from cbo_with_oop_b200.obs_gp import fit_state
    from cbo_with_oop_b200.synthetic import scaled_set
    cfg, S = workload_config(args, world)
    # the observational-GP state comes from host LAPACK here: none of this repository's kernels runs in this arm
    pr = scaled_set(0, n_obs=args.n_obs, p=args.p, d=D_INT, c=C_COND, n_int=N_INT, device=None, device_fit=True)
    with blas_threads():
        alpha, kyinv = fit_state(np.hstack([pr.x_obs_int, pr.x_obs_cond]), pr.y_obs, pr.s2, np.ones(D_INT + C_COND), pr.noise)
    sample = 2048 if args.n_obs >= 5000 else 16384
    vals, times = [], []
    for i in range(args.warmup + args.steps):
        r = cpu_port(pr, alpha, kyinv, sample, seed=i)
        if i >= args.warmup:
            vals.append(r["points_per_s"])
            times.append(r["sample_s"])
    v = float(np.mean(vals))
    ndirect = 16 if args.direct_candidates is None else args.direct_candidates
    direct = cpu_port(pr, alpha, kyinv, sample, seed=0, direct_pts=ndirect).get("direct_form") if ndirect > 0 else None
    total_pts = S * args.p ** D_INT
    sample_txt = ("each step: one-off precompute of 1 exploration set + %d seeded candidates of its grid, "
                  "extrapolated linearly to the set's %d candidates; all sets have the same cost" % (r["sample_points"], args.p ** D_INT))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_pts / v * 1e3, "sample_ms_per_step": float(np.mean(times) * 1e3),
            "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": r["threads"], "threads": r["threads"], "host_cores": r["host_cores"],
                             "kind": "port", "sample": sample_txt, "reference_faithful_direct_form": direct},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement of the reference's arithmetic (oracle/cbo_oracle.py, factorised vectorised form) on the "
                    "host cores, BLAS pinned to every core at every N; `ms_per_step` is the extrapolated time of a whole step, "
                    "`sample_ms_per_step` what was actually timed; the reference itself needs GPy/emukit/paramz, which cannot be "
                    "installed offline"}
    emit(line)


# ---------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            for ln in self.proc.stdout:
                self.rows.append([c.strip() for c in ln.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            self.proc.wait()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)]
        return {"sm_mhz": float(np.median(busy or sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# stdout carries exactly ONE line, the JSON record: the process-wide fd 1 is pointed at stderr before any library loads
# (NCCL prints its version banner to fd 1 from C), and the record goes to a private duplicate of the original stdout.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def measure_fp64_peak(gpu_index):
    """FP64 DMMA issue rate of THIS box, measured before the timed region with the micro-benchmark of tools/fp64_peak.cu
    (built by __graft_entry__.build(); otherwise compiled into a temporary directory: the tree may be read-only).  Falls back to
    the round-1 measurement."""
    import tempfile
    from cbo_with_oop_b200.build import _nvcc
    exe = os.path.join(ROOT, "tools", "fp64_peak")
    tmp = None
    try:
        if not os.path.exists(exe):
            tmp = tempfile.TemporaryDirectory(prefix="cbo_fp64_peak_")
            exe = os.path.join(tmp.name, "fp64_peak")
            subprocess.check_call([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe,
                                   os.path.join(ROOT, "tools", "fp64_peak.cu")], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[gpu_index]
                   if os.environ.get("CUDA_VISIBLE_DEVICES") else str(gpu_index))
        res = json.loads(subprocess.check_output([exe], env=env, stderr=subprocess.DEVNULL, timeout=120).decode())
        rows = [r for r in res["results"] if r["kind"].startswith("dmma")]
        return max(r["tflops"] for r in rows), "measured in this run, before the timed region: DMMA issue-rate micro-benchmark tools/fp64_peak.cu (DFMA %.2f)" \
            % max(r["tflops"] for r in res["results"] if r["kind"] == "dfma")
    except Exception as e:  # noqa: BLE001
        try:
            pk = json.load(open(FP64_PEAK_FILE))
            return max(r["tflops"] for r in pk["issue_rate"]["results"] if r["kind"].startswith("dmma")), \
                "round-1 measurement on this pool's B200 (profiles/fp64_peak_r01.json); the in-run probe failed: %s" % type(e).__name__
        except Exception:  # noqa: BLE001
            return 36.97, "fallback constant (round-1 measurement)"
    finally:
        if tmp is not None:
            tmp.cleanup()


DUMP_SAMPLE = 1 << 20      # candidates whose posterior is written, over all sets: 4 arrays x 8 B x 2^20 = 32 MB


def dump_outputs(path, eng, out):
    """Write what one SweepEngine.sweep computed as float64 .npy files under `path` (about 32 MB at most), so that two
    builds can be compared output for output on the same seeded inputs:
      selected.npy                         [set, flat index, acquisition value, NaN count] of the next intervention
      selected_x.npy                       its coordinates
      set_values.npy, set_indices.npy      every exploration set's best acquisition value and its flat index
      sample_set.npy, sample_index.npy,    posterior mean and variance (the device arrays the sweep leaves behind) at a
      mu.npy, var.npy                      fixed seeded sample of each set's candidates, or at all of them when they fit
    Only candidates this rank holds are written; which ones are sampled does not depend on the partition."""
    os.makedirs(path, exist_ok=True)
    arrays = {"selected": [out.set, out.index, out.value, out.n_nan],
              "selected_x": out.x if out.x is not None else np.zeros(0),
              "set_values": out.set_values, "set_indices": out.set_indices}
    per_set = DUMP_SAMPLE // len(eng.problems)
    cols = {"sample_set": [], "sample_index": [], "mu": [], "var": []}
    for g in eng.active:
        G = eng.problems[g].g_total
        idx = np.arange(G) if G <= per_set else np.sort(np.random.default_rng([0, g]).choice(G, per_set, replace=False))
        gb, gc = eng.slices[g]
        idx = idx[(idx >= gb) & (idx < gb + gc)]
        cols["sample_set"].append(np.full(len(idx), g))
        cols["sample_index"].append(idx)
        for k in ("mu", "var"):
            cols[k].append(eng.fetch(k, g)[idx - gb])
    arrays.update({k: np.concatenate(v) if v else np.zeros(0) for k, v in cols.items()})
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def timed_trials(eng, best, dev, n, warm):
    """min / median milliseconds of n full trials (CUDA events around SweepEngine.sweep incl. the result read-back)."""
    import torch
    for _ in range(warm):
        out = eng.sweep(best, "min")
    ms, stages = [], []
    for _ in range(n):
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(dev))
        out = eng.sweep(best, "min")
        e1.record(torch.cuda.current_stream(dev))
        torch.cuda.synchronize(dev)
        ms.append(e0.elapsed_time(e1))
        stages.append(out.stage_ms)
    k = int(np.argsort(ms)[len(ms) // 2])
    return float(np.min(ms)), float(ms[k]), stages[k], out


def small_configs_block(dev, peak):
    """One full post-observation trial of every shipped-data configuration (BASELINE.json configs 1-4)."""
    from cbo_with_oop_b200.engine import SweepEngine
    from cbo_with_oop_b200.fixtures import CONFIGS, golden_path, load_golden_problems
    rows = []
    for config, label in CONFIGS.items():
        if not os.path.exists(golden_path(config)):
            continue
        problems, best, task = load_golden_problems(config, device_fit=True)
        eng = SweepEngine(problems, device=dev)
        eng.timing = True
        eng.sweep(best, task)                       # the observational fit (K5) happens here, outside the timed trials
        lo, med, st, out = timed_trials(eng, best, dev, 10, 3)
        G = sum(p.g_total for p in problems)
        A = len(eng.active)
        flops = float(eng.lib.cbo_prior_eval_flops(eng.h_sets, A, eng.num_sms))
        pair = int(eng.lib.cbo_prior_pair_items(eng.h_sets, A, eng.num_sms))
        k_ms = st["prior_eval_grid"]
        rows.append({"config": label, "exploration_sets": len(problems), "candidates": G,
                     "n_obs": int(max(p.x_obs_int.shape[0] for p in problems)), "ms_per_trial": med, "ms_per_trial_min": lo,
                     "value": G / (med * 1e-3), "unit": UNIT,
                     "dominant_kernel": "cbo::prior_pair_kernel (+ pair_tables_kernel)" if pair else "cbo::prior_eval_kernel",
                     "dominant_kernel_ms": k_ms, "share_of_trial": k_ms / med,
                     "executed_tflops": flops / (k_ms * 1e-3) * 1e-12, "executed_frac": flops / (k_ms * 1e-3) * 1e-12 / peak,
                     "stage_ms": {k: round(v, 4) for k, v in st.items()}, "selected": {"set": out.set, "index": out.index}})
        del eng
    return rows


def run_ours(args, world, rank, local_rank):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    from cbo_with_oop_b200.partition import SetSize, partition
    from cbo_with_oop_b200.synthetic import scaled_set

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    peak, peak_src = (measure_fp64_peak(local_rank) if rank == 0 else (None, None))
    barrier()

    cfg, S = workload_config(args, world)
    G_set = args.p ** D_INT

    def build_engine(num_sets, w, r, pinned):
        sizes = [SetSize(G_set, args.n_obs, N_INT)] * num_sets
        mine = partition(sizes, w)[r]
        problems = []
        for s in range(num_sets):
            if mine[s][1] > 0:   # the observational state (alpha, Ky^-1) is produced on the device from (X, y): cbo_obs_gp_fit
                problems.append(scaled_set(s, n_obs=args.n_obs, p=args.p, d=D_INT, c=C_COND, n_int=N_INT, device_fit=True))
            else:  # shape-only placeholder: this rank never touches the set
                z = lambda *sh: np.broadcast_to(np.zeros(1), sh)
                problems.append(SetProblem(z(args.n_obs, D_INT), z(args.n_obs, C_COND), z(args.n_obs, C_COND), z(args.n_obs), z(1, 1),
                                           np.ones(D_INT), np.ones(C_COND), 1.0, [np.linspace(-2, 2, args.p)] * D_INT,
                                           z(N_INT, D_INT), z(N_INT), cost_fix=float(D_INT)))
        # the incumbent every rank would hold: min over the interventional outputs of ALL sets
        b = float(min([np.min(p.y_int) for p in problems if p.y_obs is not None] or [np.inf]))
        if w > 1:
            t = torch.tensor([b], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            b = float(t.item())
        e = SweepEngine(problems, device=dev, rank=r, world_size=w, pinned_staging=pinned)
        e.timing = True
        return e, problems, mine, b

    t_setup = time.time()
    eng, problems, mine, best = build_engine(S, world, rank, True)
    t_setup = time.time() - t_setup

    def timed(e, b, nsteps, with_upload):
        stage_ms, launches, h2d = {}, 0, 0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(dev))
        out = None
        for _ in range(nsteps):
            if with_upload:
                h2d = e.upload()        # (X, y) of the observational GPs, interventional data, grids; marks the fit stale
            l0 = e.launches
            out = e.sweep(b, "min")
            launches = e.launches - l0
            for k, v in out.stage_ms.items():
                stage_ms[k] = stage_ms.get(k, 0.0) + v
        e1.record(torch.cuda.current_stream(dev))
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out, {k: v / nsteps for k, v in stage_ms.items()}, launches, h2d

    for _ in range(args.warmup):        # the first warm-up also runs the one-off observational fit (inputs resident afterwards)
        eng.sweep(best, "min")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    try:
        ms, out, stage_ms, launches, _ = timed(eng, best, args.steps, False)
    finally:
        clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:     # before the post-intervention trials below overwrite mu / var
        dump_outputs(args.dump_outputs, eng, out)
    total_pts = S * G_set
    value = total_pts / (ms / args.steps * 1e-3)

    # secondary metric: the post-intervention trial (prior on the grid cached; one set gets a new interventional row and
    # is refitted, every other set only refreshes EI from its cached posterior).  Reported apart from the headline.
    refresh = None
    if eng.active:
        g0 = eng.active[0]
        pr0 = eng.problems[g0]
        x_old, y_old = pr0.x_int.copy(), pr0.y_int.copy()
        rng = np.random.default_rng(7)
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x_cur, y_cur = x_old, y_old
        nref = 10
        for it in range(nref + 3):          # every trial appends one interventional row to the set, as CBO.intervene does
            if it == 2:
                r0.record(torch.cuda.current_stream(dev))
            if it == nref + 2:              # one more trial through the per-stage entry points, for the stage breakdown only
                r1.record(torch.cuda.current_stream(dev))
            eng.timing = it == nref + 2     # timed trials: one library call each (cbo_refresh_trial)
            x_cur = np.vstack([x_cur, rng.uniform(-2, 2, (1, D_INT))])
            y_cur = np.append(y_cur, 0.0)
            eng.set_interventional(g0, x_cur, y_cur)
            out_r = eng.refresh(best, "min", refit=[g0])
        barrier()
        eng.timing = True
        eng.set_interventional(g0, x_old, y_old)
        ms_r = torch.tensor([r0.elapsed_time(r1) / nref], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms_r, op=dist.ReduceOp.MAX)
        my_pts = sum(c for _, c in mine)
        refresh = {"ms_per_trial": float(ms_r.item()), "value": total_pts / (float(ms_r.item()) * 1e-3), "unit": UNIT,
                   "stage_ms_of_one_staged_trial": out_r.stage_ms,
                   "hbm_bound_ms": (16.0 * my_pts + 8.0 * eng.h_sets[0].n_obs_pad ** 2 / 2) / 6535.4e9 * 1e3,
                   "hbm_frac": (16.0 * my_pts + 8.0 * eng.h_sets[0].n_obs_pad ** 2 / 2) / 6535.4e9 * 1e3 / float(ms_r.item()),
                   "what": "post-intervention trial through ONE library call (cbo_refresh_trial), host data in, host result out: "
                           "one interventional row appended to a set -> its interventional table, the prior "
                           "of the NEW row (u^T M u streams M once: HBM-bound), refit of that set, full posterior + EI for it, EI "
                           "refresh from cached mu/var (16 B/candidate) for the other sets, argmax; hbm_bound_ms = (16 B x this "
                           "GPU's candidates + one pass over M's triangle) / 6535 GB/s"}

    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    ms_e, out_e, stage_e, _, h2d = timed(eng, best, e2e_steps, True)
    e2e_value = total_pts / (ms_e / e2e_steps * 1e-3)
    if world > 1:
        hb = torch.tensor([float(h2d)], dtype=torch.float64, device=dev)
        dist.all_reduce(hb, op=dist.ReduceOp.SUM)
        h2d = int(hb.item())
    d2h = world * eng.d2h_bytes_per_sweep

    line = None
    if rank == 0:
        # roofline of the dominant kernel (prior_eval on the grid): flops the DMMA pipe executes per launch / live duration
        my_pts = sum(c for _, c in mine)
        N, d = args.n_obs, D_INT
        flops_dense = my_pts * (2.0 * N * N + 2.0 * N + d * N)          # SURVEY.md §8(d) F_prior, dense-counted
        flops_exec = float(eng.lib.cbo_prior_eval_flops(eng.h_sets, len(eng.active), eng.num_sms))
        dur_s = stage_ms["prior_eval_grid"] * 1e-3
        traffic, traffic_src = None, None
        try:
            traffic = json.load(open(TRAFFIC_FILE)).get("dram_bytes_per_launch")
            traffic_src = ("quoted from profiles/r01_prior_eval_traffic.json (one `ncu --set full` capture of this kernel on the "
                           "2-set workload), not measured in this run")
        except Exception:  # noqa: BLE001
            pass
        roof = {"bound": "tensor", "kernel": "cbo::prior_eval_kernel (which=0, grid)", "achieved": flops_exec / dur_s * 1e-12,
                "peak": peak, "unit": "TFLOP/s", "frac": flops_exec / dur_s * 1e-12 / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "achieved_dense_counted": flops_dense / dur_s * 1e-12, "frac_dense_counted": flops_dense / dur_s * 1e-12 / peak,
                "flops_per_launch_executed": flops_exec, "flops_per_launch_dense_counted": flops_dense,
                "kernel_ms_per_launch": stage_ms["prior_eval_grid"], "share_of_step": stage_ms["prior_eval_grid"] / (ms / args.steps),
                "peak_source": peak_src,
                "note": "FP64 tensor pipe (DMMA.8x8x4), not the bf16 figure of MEASURED_PEAKS.json.  `achieved`/`frac` count the "
                        "flops the kernel EXECUTES (the lower block triangle of the symmetric M: about N^2 per candidate, "
                        "cbo_prior_eval_flops) -- the hardware utilisation of the FP64 pipe; the `*_dense_counted` keys use "
                        "SURVEY.md 8(d)'s 2N^2+2N+dN per candidate and can approach 2 because of the symmetry."}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "steps": e2e_steps, "ms_per_step": ms_e / e2e_steps, "obs_gp_fit_ms": stage_e.get("obs_gp_fit"),
                        "api": "observe + intervene from host buffers: SweepEngine.upload() (pinned host -> device of the observational "
                               "design X, its targets y, the interventional data and the grids -- no N x N array crosses PCIe) + "
                               "the observational GP fit on the device (cbo_obs_gp_fit; the reference's trial starts with it, "
                               "CBO.py:135) + SweepEngine.sweep() -> host result"},
                "gpu_launches": int(launches) * args.steps, "gpu_launches_per_step": int(launches),
                "roofline": roof, "clocks": clocks, "stage_ms_per_step": stage_ms, "post_intervention_trial": refresh,
                "selected": {"set": out.set, "index": out.index, "value": out.value}, "setup_s": round(t_setup, 1)}
        key = "sets%d_nobs%d_p%d" % (S, args.n_obs, args.p)
        try:
            exp = json.load(open(EXPECTED_FILE)).get(key)
        except Exception:  # noqa: BLE001
            exp = None
        if exp is not None:
            line["selected_expected"] = exp
            line["selected_matches_expected"] = bool(exp["set"] == out.set and exp["index"] == out.index)
        first_li = 0
        alpha_h = eng.buf[first_li]["alpha_obs"].cpu().numpy() if eng.active else None
        kyinv_h = eng.buf[first_li]["kyinv"].cpu().numpy().reshape(args.n_obs, args.n_obs) if eng.active else None
        first_problem = eng.problems[eng.active[0]] if eng.active else None
    del eng
    torch.cuda.empty_cache()

    if rank == 0 and world == 1:
        if not args.strong and not args.no_full_config and S != 16:
            # the FULL named configuration on this one GPU: all 16 sets, one warm-up step (the kernels themselves are warm
            # from the steps above) and one timed step
            engF, _, mineF, bestF = build_engine(16, 1, 0, False)
            engF.sweep(bestF, "min")
            msF, outF, stF, lF, _ = timed(engF, bestF, 1, False)
            flF = float(engF.lib.cbo_prior_eval_flops(engF.h_sets, len(engF.active), engF.num_sms))
            line["full_config"] = {"exploration_sets": 16, "grid_points": 16 * G_set, "steps": 1, "warmup": 1, "ms_per_step": msF,
                                   "value": 16 * G_set / (msF * 1e-3), "unit": UNIT, "gpu_launches_per_step": int(lF),
                                   "stage_ms": stF, "roofline_frac": flF / (stF["prior_eval_grid"] * 1e-3) * 1e-12 / peak,
                                   "selected": {"set": outF.set, "index": outF.index, "value": outF.value},
                                   "what": "BASELINE.json configs[4] in full (16 sets x 1e6 candidates x 1e4 observational samples) on one "
                                           "B200, inputs resident; same kernels and per-set work as the weak-scaled headline"}
            try:
                expF = json.load(open(EXPECTED_FILE)).get("sets16_nobs%d_p%d" % (args.n_obs, args.p))
            except Exception:  # noqa: BLE001
                expF = None
            if expF is not None:
                line["full_config"]["selected_matches_expected"] = bool(expF["set"] == outF.set and expF["index"] == outF.index)
            del engF
            torch.cuda.empty_cache()
        if not args.no_small_configs:
            try:
                line["small_configs"] = small_configs_block(dev, peak)
            except Exception as e:  # noqa: BLE001
                line["small_configs"] = {"error": "%s: %s" % (type(e).__name__, e)}
        if not args.no_cpu_baseline and first_problem is not None:
            nd = 2 if args.direct_candidates is None else args.direct_candidates
            r = cpu_port(first_problem, alpha_h, kyinv_h, 2048 if args.n_obs >= 5000 else 16384,
                         direct_pts=nd if args.n_obs <= 10_000 else 0, direct_budget_s=40.0)
            line["cpu_baseline"] = {
                "value": r["points_per_s"], "unit": UNIT, "cores": r["threads"], "threads": r["threads"], "kind": "port",
                "sample": "one-off precompute of 1 exploration set + %d seeded candidates of its grid with the vectorised factorised "
                          "NumPy/BLAS port (oracle/cbo_oracle.py), extrapolated linearly to the set's %d candidates"
                          % (r["sample_points"], G_set),
                "one_off_s": r["one_off_s"], "per_point_s": r["per_point_s"], "host_cores": r["host_cores"],
                "reference_faithful_direct_form": r.get("direct_form")}
    if rank == 0:
        emit(line)
        if args.strict_selection and line.get("selected_matches_expected") is False:
            raise SystemExit("selected intervention %s differs from the expected %s" % (line["selected"], line["selected_expected"]))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = ARGS
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    if args.impl == "reference":
        run_reference(args, world, rank)
    else:
        run_ours(args, world, rank, local_rank)


if __name__ == "__main__":
    main()
