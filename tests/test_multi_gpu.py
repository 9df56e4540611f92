"""Multi-GPU parity on real devices (NCCL): tools/multi_gpu_check.py under torchrun -- six exploration sets partitioned over
the ranks with sets split between ranks, per-set bests all-gathered and combined on every rank, compared with the oracle
(per-set maxima to 1e-6, indices and the selected intervention bit-exact, identical on all ranks).  Skipped on a box
with fewer than two GPUs; the CPU suite covers the same host logic with two gloo processes (tests/test_partition.py)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_multi_gpu_check_under_torchrun(cuda_engine_ready, tmp_path):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    for world in sorted({2, min(n, 4), n}):
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
               "--master-port", str(29530 + world), os.path.join(ROOT, "tools", "multi_gpu_check.py")]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
        ok = [ln for ln in r.stdout.splitlines() if ln.startswith("rank ") and ln.rstrip().endswith("OK")]
        with open(tmp_path / f"multi_gpu_check_n{world}.log", "w") as f:
            f.write(r.stdout + "\n---- stderr ----\n" + r.stderr[-4000:])
        assert r.returncode == 0, r.stderr[-2000:]
        assert len(ok) == world, r.stdout
        assert any("split sets [" in ln and "split sets []" not in ln for ln in ok), "no set was split between ranks"
