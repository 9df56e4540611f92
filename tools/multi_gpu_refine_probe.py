"""Measured cost of the off-grid refinement (K7, SweepEngine.refine) on multi-GPU engines; launch with torchrun, one rank
per GPU (also with one process):

  * --shape weak:   BASELINE.json configs[4] weak-scaled, 2 exploration sets per GPU (N = 1e4 observational rows, 1e6-point
                    grids, d = 3; synthetic.scaled_sweep(device_fit=True));
  * --shape split3: the 3-set strong-scaling shape of the same sets, which splits sets between ranks on more than 3 GPUs.

Per rank: milliseconds per refine call (CUDA events, median of 10 after 2 warm-up calls), with the K7 call ("refine") and
the all-gather of the refined records ("refine_gather") taken apart from stage_ms.  The refined per-set values and
coordinates are compared bit for bit with a single-GPU engine built on the rank's own GPU over the sets the rank refines (a
set's refinement reads nothing of the other sets).  The card's name and power limit are read in the same run.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29581 \\
        tools/multi_gpu_refine_probe.py --shape weak --out DIR        (rank 0 writes DIR/multi_gpu_refine_<shape>_n<W>.json)

With --gloo the records travel over gloo and the ranks may outnumber the GPUs (rank r runs on GPU r mod the device count):
the refined values and their comparison are then those of the multi-rank path, but the times are of ranks sharing a GPU and
the file is named ..._n<W>_gloo_<G>gpu.json.
"""
from __future__ import annotations

import argparse
import datetime
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(local: int) -> str:
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", choices=("weak", "split3"), required=True)
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--gloo", action="store_true")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("multi_gpu_refine_probe.py needs a CUDA device")
    from cbo_with_oop_b200.engine import SweepEngine
    from cbo_with_oop_b200.synthetic import best_of, scaled_sweep
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local, gpus = int(os.environ.get("LOCAL_RANK", "0")), torch.cuda.device_count()
    if args.gloo:
        local %= gpus
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    timeout = datetime.timedelta(seconds=600)
    if args.gloo:
        dist.init_process_group("gloo", timeout=timeout)
    else:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=timeout)
    S = 2 * world if args.shape == "weak" else 3
    problems = scaled_sweep(S, n_obs=10_000, p=100, d=3, c=3, n_int=32, device_fit=True)
    best = best_of(problems)
    eng = SweepEngine(problems, device=dev, rank=rank, world_size=world)
    grid = eng.sweep(best, "min")
    eng.timing = True
    calls, k7, gather = [], [], []
    for i in range(args.warmup + args.calls):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = eng.refine(grid, best, "min")
        e1.record()
        torch.cuda.synchronize()
        if i >= args.warmup:
            calls.append(e0.elapsed_time(e1))
            k7.append(out.stage_ms.get("refine", 0.0))
            gather.append(out.stage_ms["refine_gather"])
    eng.timing = False
    # single-GPU engine over the sets this rank refines: the same refined values and coordinates, bit for bit
    owned = [g for g in range(S) if eng.refine_owner[g] == rank]
    matches = None
    if owned:
        one = SweepEngine([problems[g] for g in owned], device=dev)
        ref = one.refine(one.sweep(best, "min"), best, "min")
        matches = all(ref.set_values[i].tobytes() == out.set_values[g].tobytes() and ref.set_x[i].tobytes() == out.set_x[g].tobytes()
                      and ref.refine_status[i] == out.refine_status[g] for i, g in enumerate(owned))
    row = {"rank": rank, "card": card(local), "active_sets": eng.active, "owned_sets": owned, "slices": eng.slices,
           "refine_call_ms_median": float(np.median(calls)), "refine_call_ms_min": float(np.min(calls)),
           "k7_ms_median": float(np.median(k7)) if eng.active else None, "gather_ms_median": float(np.median(gather)),
           "matches_single_gpu": matches}
    rows = [None] * world
    dist.all_gather_object(rows, row)
    if rank == 0:
        res = {"what": ("BASELINE.json configs[4] weak-scaled: 2 sets per GPU" if args.shape == "weak" else
                        "3 sets of BASELINE.json configs[4] (strong scaling)") +
                       ", N = 1e4, 1e6-point grid (d = 3), n_int = 32, device_fit=True",
               "shape": args.shape, "ranks_n": world, "backend": "gloo" if args.gloo else "nccl",
               "gpus_used": min(world, gpus) if args.gloo else world, "sets": S, "calls": args.calls, "warmup": args.warmup,
               "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
               "refine_call_ms_median_max_over_ranks": max(r["refine_call_ms_median"] for r in rows),
               "gather_ms_median_max_over_ranks": max(r["gather_ms_median"] for r in rows),
               "all_ranks_match_single_gpu": all(r["matches_single_gpu"] is not False for r in rows),
               "refined": [{"set": g, "grid_value": float(grid.set_values[g]), "value": float(out.set_values[g]),
                            "x": [float(v) for v in out.set_x[g]], "status": out.refine_status[g], "owner": eng.refine_owner[g]}
                           for g in range(S)],
               "selected": {"set": out.set, "value": float(out.value)},
               "ranks": rows}
        os.makedirs(args.out, exist_ok=True)
        tag = f"_gloo_{min(world, gpus)}gpu" if args.gloo else ""
        path = os.path.join(args.out, f"multi_gpu_refine_{args.shape}_n{world}{tag}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({k: v for k, v in res.items() if k != "ranks"}, indent=1), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
