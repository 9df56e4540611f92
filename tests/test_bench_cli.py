"""bench.py's contract: the reference arm prints exactly one JSON line on stdout with the keys a caller reads, `ours`
refuses to run without a CUDA device (no CPU fallback), malformed arguments are refused, build() compiles -- and, on
the GPU, --dump-outputs writes the same outputs for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT,
                          timeout=600, env=env)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--n-obs", "300", "--p", "12", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "grid-points/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["metric"].startswith("EI grid-points/sec") and "workload" in d["config"]


def test_ours_arm_needs_a_gpu():
    # (on a machine with a GPU the device is hidden from the child process)
    r = _run("--steps", "1", "--warmup", "0", env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0 and "CUDA" in (r.stderr + r.stdout)
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]      # nothing that looks like a result


def test_build_entry_compiles_and_loads():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()
    from cbo_with_oop_b200 import _lib
    assert _lib.load().cbo_abi_version() == _lib.CBO_ABI_VERSION


def test_malformed_arguments_are_refused():
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        r = _run(*args, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        assert r.returncode == 2 and "error" in r.stderr, (args, r.stderr[-500:])


@pytest.mark.gpu
def test_dump_outputs_repeat_for_the_same_inputs(cuda_engine_ready, tmp_path):
    """Two runs with different step counts dump the same last-step outputs: the inputs are seeded, the kernels
    deterministic.  The files are float64 and within the 64 MB budget; selected.npy agrees with the JSON line."""
    small = ["--n-obs", "1000", "--p", "24", "--no-full-config", "--no-small-configs", "--no-cpu-baseline", "--e2e-steps", "1"]
    runs = []
    for steps, warmup in ((2, 1), (1, 0)):
        out = tmp_path / f"steps{steps}"
        r = _run(*small, "--steps", str(steps), "--warmup", str(warmup), "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout)
        assert line["steps"] == steps
        files = sorted(out.iterdir())
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        arrays = {f.stem: np.load(f) for f in files}
        assert all(a.dtype == np.float64 for a in arrays.values())
        sel = arrays["selected"]
        assert (int(sel[0]), int(sel[1])) == (line["selected"]["set"], line["selected"]["index"])
        assert sel[2] == line["selected"]["value"] and np.array_equal(arrays["set_values"][int(sel[0])], sel[2])
        assert len(arrays["mu"]) == len(arrays["var"]) == len(arrays["sample_index"]) == 2 * 24 ** 3   # every candidate fits
        runs.append(arrays)
    assert runs[0].keys() == runs[1].keys()
    for name in runs[0]:
        np.testing.assert_array_equal(runs[0][name], runs[1][name], err_msg=name)
