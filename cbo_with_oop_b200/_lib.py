"""ctypes binding of libcbo_b200.so (include/cbo_b200.h).  There is no fallback: if the library is missing
or a call fails this module raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CBO_B200_LIB") or os.path.join(HERE, "libcbo_b200.so")   # (the override is for kernel experiments)

CBO_ABI_VERSION = 9
CBO_MAX_D = 4
CBO_MAX_C = 8
CBO_MAX_NINT = 128
CBO_NPAD = 128
CBO_SPAD = 16
CBO_PRIOR_TILE = 128
CBO_SWEEP_TILE = 1024

_dp = C.c_void_p  # device pointer


class SetDesc(C.Structure):
    """Mirror of cbo_set_desc; field order and types must match include/cbo_b200.h (checked at load time
    against cbo_offsetof_set_desc)."""
    _fields_ = [
        ("d", C.c_int32), ("c", C.c_int32), ("n_obs", C.c_int32), ("n_obs_pad", C.c_int32),
        ("n_mc", C.c_int32), ("n_mc_pad", C.c_int32), ("n_int", C.c_int32), ("causal", C.c_int32),
        ("p", C.c_int32 * CBO_MAX_D),
        ("g_total", C.c_int64), ("g_begin", C.c_int64), ("g_count", C.c_int64),
        ("x_obs_int", _dp), ("x_obs_cond", _dp), ("mc_cond", _dp), ("alpha_obs", _dp), ("kyinv", _dp),
        ("ls_int", C.c_double * CBO_MAX_D), ("ls_cond", C.c_double * CBO_MAX_C),
        ("s2", C.c_double), ("noise", C.c_double),
        ("tab", _dp * CBO_MAX_D), ("u_int", _dp), ("P", _dp), ("pbar", _dp), ("w", _dp), ("M", _dp),
        ("grid", _dp * CBO_MAX_D), ("x_int", _dp), ("y_int", _dp), ("m_int", _dp), ("v_int", _dp),
        ("L", _dp), ("alpha", _dp), ("sqrt_v_int", _dp), ("fit_info", _dp),
        ("cost_fix", C.c_double), ("cost_variable", C.c_int32), ("prior_external", C.c_int32),
        ("m", _dp), ("v", _dp), ("mu", _dp), ("var", _dp), ("ei", _dp), ("acq", _dp),
        ("posterior_cached", C.c_int32), ("int_row_begin", C.c_int32), ("y_obs", C.c_void_p),
        ("points", _dp), ("hyper", _dp),
    ]


class SetBest(C.Structure):
    _fields_ = [("value", C.c_double), ("index", C.c_int64), ("n_nan", C.c_int32), ("reserved", C.c_int32)]


class SweepResult(C.Structure):
    _fields_ = [("value", C.c_double), ("index", C.c_int64), ("set", C.c_int32), ("n_nan", C.c_int32)]


class AcqGradOut(C.Structure):
    """Mirror of cbo_acq_grad_out (value and gradient of the acquisition at one point)."""
    _fields_ = [(n, C.c_double) for n in ("m", "v", "mu", "var", "ei", "acq")] + \
               [(n, C.c_double * CBO_MAX_D) for n in ("dm", "dv", "dmu", "dvar", "dei", "dacq")]


class RefineResult(C.Structure):
    """Mirror of cbo_refine_result (one exploration set's refined maximum)."""
    _fields_ = [("x", C.c_double * CBO_MAX_D), ("value", C.c_double), ("start_value", C.c_double),
                ("iterations", C.c_int32), ("status", C.c_int32)]


class HyperResult(C.Structure):
    """Mirror of cbo_hyper_result (one exploration set's marginal-likelihood fit)."""
    _fields_ = [("variance", C.c_double), ("lengthscale", C.c_double), ("nll", C.c_double), ("nll_start", C.c_double),
                ("iterations", C.c_int32), ("status", C.c_int32), ("start", C.c_int32), ("jitter_tries", C.c_int32)]


CBO_HYPER_STARTS = 9
HYPER_STATUS = {0: "converged", 1: "max_iter", 2: "line_search_failed", 3: "not_positive_definite"}

REFINE_STATUS = {0: "converged", 1: "max_iter", 2: "line_search_failed", 3: "skipped_external_prior",
                 4: "skipped_explicit_points", 5: "skipped_nonfinite"}

EXPORTS = [
    "cbo_abi_version", "cbo_sizeof_set_desc", "cbo_offsetof_set_desc", "cbo_last_error", "cbo_sweep_num_items",
    "cbo_prior_workspace_bytes", "cbo_launch_count", "cbo_obs_gp_workspace_bytes", "cbo_prior_pair_items",
    "cbo_prior_eval_flops",
    "cbo_obs_gp_fit", "cbo_obs_gp_nll",
    "cbo_build_tables", "cbo_prior_precompute", "cbo_prior_eval", "cbo_posterior_fit", "cbo_sweep",
    "cbo_argmax_combine", "cbo_sem_eval", "cbo_refresh_trial", "cbo_acq_grad", "cbo_refine",
    "cbo_refine_workspace_bytes", "cbo_posterior_nll", "cbo_posterior_hyper_fit", "cbo_posterior_hyper_workspace_bytes",
]
CBO_SEM_MAX_NODES, CBO_SEM_MAX_TERMS, CBO_SEM_BLOCKS = 16, 96, 64
SEM_FUNCS = {"id": 0, "exp": 1, "cos": 2, "sin": 3, "square": 4}


class SemTerm(C.Structure):
    _fields_ = [("src", C.c_int32), ("func", C.c_int32), ("coef", C.c_double), ("scale", C.c_double)]


class SemNode(C.Structure):
    _fields_ = [("first_term", C.c_int32), ("num_terms", C.c_int32), ("constant", C.c_double)]

_lib = None


class CboError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once) and verify the ABI mirror."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m cbo_with_oop_b200.build` "
            "(the CUDA library is the product; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise ImportError(f"{LIB_PATH} does not export {name}")
    lib.cbo_abi_version.restype = C.c_int
    lib.cbo_sizeof_set_desc.restype = C.c_size_t
    lib.cbo_offsetof_set_desc.restype = C.c_long
    lib.cbo_offsetof_set_desc.argtypes = [C.c_char_p]
    lib.cbo_last_error.restype = C.c_char_p
    lib.cbo_launch_count.restype = C.c_ulonglong
    P = C.POINTER(SetDesc)
    lib.cbo_sweep_num_items.restype = C.c_long
    lib.cbo_sweep_num_items.argtypes = [P, C.c_int]
    lib.cbo_build_tables.argtypes = [P, C.c_void_p, C.c_int, C.c_void_p]
    lib.cbo_prior_precompute.argtypes = [P, C.c_void_p, C.c_int, C.c_void_p]
    lib.cbo_prior_workspace_bytes.restype = C.c_size_t
    lib.cbo_prior_workspace_bytes.argtypes = [P, C.c_int, C.c_int]
    lib.cbo_prior_eval_flops.restype = C.c_double
    lib.cbo_prior_eval_flops.argtypes = [P, C.c_int, C.c_int]
    lib.cbo_prior_pair_items.restype = C.c_long
    lib.cbo_prior_pair_items.argtypes = [P, C.c_int, C.c_int]
    lib.cbo_obs_gp_workspace_bytes.restype = C.c_size_t
    lib.cbo_obs_gp_workspace_bytes.argtypes = [P, C.c_int]
    lib.cbo_obs_gp_fit.argtypes = [P, C.c_int, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.cbo_obs_gp_nll.argtypes = [P, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.cbo_prior_eval.argtypes = [P, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.cbo_posterior_fit.argtypes = [P, C.c_void_p, C.c_int, C.c_void_p]
    lib.cbo_sweep.argtypes = [P, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]
    lib.cbo_argmax_combine.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cbo_refresh_trial.argtypes = [P, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cbo_sem_eval.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cbo_acq_grad.argtypes = [P, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                 C.c_void_p]
    lib.cbo_refine.argtypes = [P, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p,
                               C.c_size_t, C.c_void_p, C.c_void_p]
    for name in EXPORTS[10:]:
        getattr(lib, name).restype = C.c_int
    lib.cbo_posterior_nll.argtypes = [P, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.cbo_posterior_hyper_fit.argtypes = [P, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_double, C.c_void_p,
                                            C.c_size_t, C.c_void_p, C.c_void_p]
    lib.cbo_posterior_hyper_workspace_bytes.restype = C.c_size_t
    lib.cbo_posterior_hyper_workspace_bytes.argtypes = [P, C.c_int]
    lib.cbo_refine_workspace_bytes.restype = C.c_size_t
    lib.cbo_refine_workspace_bytes.argtypes = [P, C.c_int]
    if lib.cbo_abi_version() != CBO_ABI_VERSION:
        raise ImportError(f"ABI version mismatch: library {lib.cbo_abi_version()} != binding {CBO_ABI_VERSION}")
    if lib.cbo_sizeof_set_desc() != C.sizeof(SetDesc):
        raise ImportError(f"cbo_set_desc size mismatch: C {lib.cbo_sizeof_set_desc()} vs ctypes {C.sizeof(SetDesc)}")
    for fname, _ in SetDesc._fields_:
        off = lib.cbo_offsetof_set_desc(fname.encode())
        if off != getattr(SetDesc, fname).offset:
            raise ImportError(f"cbo_set_desc.{fname}: C offset {off} != ctypes {getattr(SetDesc, fname).offset}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cbo_last_error().decode(errors="replace")
        raise CboError(f"{what} failed with status {rc}: {msg}")
