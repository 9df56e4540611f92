"""CPU checks of the C-ABI boundary: the library builds and loads without a GPU, exports every symbol that
include/cbo_b200.h declares, the ctypes mirror of cbo_set_desc matches, argument validation reports errors through
cbo_last_error -- and the compute entry points fail loudly (no silent CPU fallback) when there is no device."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from cbo_with_oop_b200.build import build_library
    build_library()
    from cbo_with_oop_b200 import _lib
    return _lib.load()


def declared_functions():
    text = open(os.path.join(ROOT, "include", "cbo_b200.h")).read()
    return sorted(set(re.findall(r"CBO_API\s+[\w\s\*]+?\b(cbo_\w+)\s*\(", text)))


def test_every_declared_symbol_is_exported(lib):
    names = declared_functions()
    assert len(names) >= 12 and "cbo_sweep" in names and "cbo_prior_eval" in names
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/cbo_b200.h but not exported"
    from cbo_with_oop_b200 import _lib
    assert sorted(_lib.EXPORTS) == names, "ctypes binding and header disagree on the function list"


def test_struct_mirror_and_version(lib):
    from cbo_with_oop_b200 import _lib
    assert lib.cbo_abi_version() == _lib.CBO_ABI_VERSION
    assert lib.cbo_sizeof_set_desc() == C.sizeof(_lib.SetDesc)
    for name, _ in _lib.SetDesc._fields_:
        assert lib.cbo_offsetof_set_desc(name.encode()) == getattr(_lib.SetDesc, name).offset
    assert lib.cbo_offsetof_set_desc(b"no_such_field") == -1
    assert C.sizeof(_lib.SetBest) == 24 and C.sizeof(_lib.SweepResult) == 24
    header = open(os.path.join(ROOT, "include", "cbo_b200.h")).read()
    for macro, val in [("CBO_MAX_D", _lib.CBO_MAX_D), ("CBO_MAX_C", _lib.CBO_MAX_C), ("CBO_MAX_NINT", _lib.CBO_MAX_NINT),
                       ("CBO_NPAD", _lib.CBO_NPAD), ("CBO_SPAD", _lib.CBO_SPAD), ("CBO_PRIOR_TILE", _lib.CBO_PRIOR_TILE),
                       ("CBO_SWEEP_TILE", _lib.CBO_SWEEP_TILE), ("CBO_ABI_VERSION", _lib.CBO_ABI_VERSION)]:
        assert re.search(rf"#define\s+{macro}\s+{val}\b", header), macro


def test_argument_validation_reports_through_last_error(lib):
    from cbo_with_oop_b200 import _lib
    h = (_lib.SetDesc * 1)()
    assert lib.cbo_build_tables(h, None, 1, None) == -1
    assert b"d=0" in lib.cbo_last_error()
    h[0].d, h[0].n_int, h[0].p[0], h[0].g_total, h[0].g_count = 1, 5, 10, 10, 10
    h[0].causal, h[0].n_obs, h[0].n_obs_pad = 1, 100, 100          # pad not a multiple of 128
    h[0].cost_fix = 1.0
    assert lib.cbo_prior_precompute(h, None, 1, None) == -1
    assert b"n_obs_pad" in lib.cbo_last_error()
    h[0].g_total = 11
    assert lib.cbo_sweep(h, None, 1, 0.0, 1, None, None, None, None) == -1
    assert b"g_total" in lib.cbo_last_error()
    assert lib.cbo_sweep_num_items(h, 1) == 1
    h[0].g_total, h[0].n_obs_pad = 10, 128
    # header + the (empty) pair-table area's 16 ones, rounded to 256 B + partials + one scratch slot per CTA
    assert lib.cbo_prior_workspace_bytes(h, 1, 148) == 256 + 256 + (4 * 148 + 1024) * 2 * 128 * 8 + 148 * 128 * 128 * 8
    assert lib.cbo_prior_pair_items(h, 1, 148) == 0
    with pytest.raises(_lib.CboError):
        _lib.check(-1, "demo")


def test_tables_and_prior_precompute_refuse_host_only_descriptors(lib):
    """Both stages read every set from the device copy of the descriptors: a NULL d_sets is refused, with a message,
    after the descriptors themselves have passed validation."""
    from cbo_with_oop_b200 import _lib
    h = (_lib.SetDesc * 1)()
    h[0].d, h[0].n_int, h[0].p[0], h[0].g_total, h[0].g_count, h[0].cost_fix = 1, 5, 10, 10, 10, 1.0
    h[0].causal, h[0].n_obs, h[0].n_obs_pad, h[0].ls_int[0] = 1, 100, 128, 1.0
    assert lib.cbo_sweep(h, None, 1, 0.0, 1, None, None, None, None) == -1
    assert lib.cbo_last_error() == b"cbo_sweep: d_sets is NULL"      # validate_sets accepted the descriptor
    for fn in (lib.cbo_build_tables, lib.cbo_prior_precompute):
        assert fn(h, None, 1, None) == -1
        assert b"d_sets" in lib.cbo_last_error()


def test_no_cpu_fallback(monkeypatch):
    """Without a CUDA device the engine refuses to start (the product path is the CUDA library).  On a machine with a
    GPU the device is hidden from the engine."""
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    import numpy as np
    from cbo_with_oop_b200.engine import SetProblem, SweepEngine
    pr = SetProblem.non_causal([np.linspace(0, 1, 4)], np.zeros((2, 1)), np.zeros(2))
    with pytest.raises(RuntimeError, match="no CPU path"):
        SweepEngine([pr])


def test_product_never_imports_the_oracle():
    for base in ("cbo_with_oop_b200", "src"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    text = open(os.path.join(dirpath, f)).read()
                    assert "cbo_oracle" not in text and "from oracle" not in text and "import oracle" not in text, os.path.join(dirpath, f)
