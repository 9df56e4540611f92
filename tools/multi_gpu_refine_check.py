"""Multi-GPU check of the off-grid refinement (launch with torchrun, one rank per GPU): a mixed list of exploration sets is
partitioned over the ranks (some sets split between ranks), every rank sweeps its share and refines the sets it owns, and the
refined records are all-gathered over NCCL.  Every rank must return, bit for bit, what a single-GPU engine built on its own
GPU returns (set, index, value, x, set_values, set_x, refine_status), and all ranks must return the same output.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29562 tools/multi_gpu_refine_check.py

With --gloo the tables travel over gloo and the ranks may outnumber the GPUs (rank r runs on GPU r mod the device count): the
same check of the partitioned path on a machine with fewer GPUs than ranks.
"""
import datetime
import hashlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import make_case  # noqa: E402
from cbo_with_oop_b200.engine import SetProblem, SweepEngine  # noqa: E402


def digest(out) -> bytes:
    """Every field the refinement returns, as bytes (NaNs compare by their bits)."""
    parts = [np.array([out.set, out.index, out.n_nan], np.int64).tobytes(), np.float64(out.value).tobytes(),
             b"-" if out.x is None else out.x.tobytes(), out.set_values.tobytes(), np.asarray(out.set_indices, np.int64).tobytes(),
             "|".join(out.refine_status).encode()]
    parts += [b"-" if x is None else x.tobytes() for x in out.set_x]
    return hashlib.sha256(b"#".join(parts)).digest()


rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
gloo = "--gloo" in sys.argv[1:]
if gloo:
    local %= torch.cuda.device_count()
torch.cuda.set_device(local)
dev = f"cuda:{local}"
timeout = datetime.timedelta(seconds=300)
if gloo:
    dist.init_process_group("gloo", timeout=timeout)
else:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=timeout)
specs = [dict(seed=61, N=96, d=1, c=1, n=8, p=(300,)), dict(seed=62, N=140, d=2, c=2, n=10, p=(40, 40)),
         dict(seed=63, N=200, d=3, c=1, n=12, p=(20, 20, 20), cost_variable=True), dict(seed=64, N=70, d=2, c=0, n=9, p=(60, 30)),
         dict(seed=65, N=90, d=1, c=2, n=10, p=(640,), causal=False), dict(seed=66, N=150, d=4, c=1, n=11, p=(8, 8, 8, 8))]
cases = [make_case(**s) for s in specs]
chosen = []
for task in ("min", "max"):
    best = float(min(np.min(k["y_int"]) for k, _ in cases) if task == "min" else max(np.max(k["y_int"]) for k, _ in cases))
    eng = SweepEngine([SetProblem(**k) for k, _ in cases], device=dev, rank=rank, world_size=world)
    one = SweepEngine([SetProblem(**k) for k, _ in cases], device=dev)
    ref = one.refine(one.sweep(best, task), best, task)
    out = eng.refine(eng.sweep(best, task), best, task)
    t = torch.frombuffer(bytearray(digest(out)), dtype=torch.uint8).to(dev)
    g = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(g, t)
    assert bytes(t.cpu().numpy()) == digest(ref), (task, out, ref)       # the single-GPU engine's output
    assert all(torch.equal(g[0], x) for x in g), task                     # the same on every rank
    chosen.append(f"{task}: set {out.set} value {out.value!r} {out.refine_status}")
split = [s for s in range(len(cases)) if 0 < eng.slices[s][1] < eng.problems[s].g_total]
print(f"rank {rank}/{world}: slices {eng.slices} split sets {split} owners {eng.refine_owner} -> {'; '.join(chosen)} OK", flush=True)
dist.barrier()
dist.destroy_process_group()
