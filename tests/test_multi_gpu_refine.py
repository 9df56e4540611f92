"""Off-grid refinement on real devices (NCCL): tools/multi_gpu_refine_check.py under torchrun -- six exploration sets
partitioned over the ranks with sets split between ranks, each set refined by its owner rank, the refined records
all-gathered, and every rank's output equal bit for bit to a single-GPU engine's and to every other rank's.  Skipped on a box
with fewer than two GPUs; tests/test_refine_multi_rank_gpu.py runs the same comparison with all ranks on one GPU."""
import os
import signal
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_in_own_session(cmd, timeout):
    """subprocess.run that kills the launcher's whole process group on a timeout, so that no rank outlives the test."""
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, start_new_session=True)
    try:
        out, err = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        out, err = p.communicate()
        pytest.fail(f"torchrun did not finish in {timeout} s:\n{out[-2000:]}\n{err[-2000:]}")
    return p.returncode, out, err


def test_multi_gpu_refine_under_torchrun(cuda_engine_ready, tmp_path):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    for world in sorted({2, min(n, 4), n}):
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
               "--master-port", str(29560 + world), os.path.join(ROOT, "tools", "multi_gpu_refine_check.py")]
        rc, out, err = run_in_own_session(cmd, 600)
        ok = [ln for ln in out.splitlines() if ln.startswith("rank ") and ln.rstrip().endswith("OK")]
        with open(tmp_path / f"multi_gpu_refine_check_n{world}.log", "w") as f:
            f.write(out + "\n---- stderr ----\n" + err[-4000:])
        assert rc == 0, err[-2000:]
        assert len(ok) == world, out
        assert any("split sets [" in ln and "split sets []" not in ln for ln in ok), "no set was split between ranks"
