"""CPU checks of the C ABI of the hyper-parameter fit (K8): the descriptor field, the result mirror, and the refusals of
cbo_posterior_nll / cbo_posterior_hyper_fit, each with a message.  The calls run in a child process with the device hidden:
every refusal happens before anything touches a GPU."""
import ctypes as C
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_descriptor_field_and_result_mirror():
    from cbo_with_oop_b200.build import build_library
    build_library()
    from cbo_with_oop_b200 import _lib
    lib = _lib.load()
    assert _lib.CBO_ABI_VERSION == 9
    assert lib.cbo_offsetof_set_desc(b"hyper") == _lib.SetDesc.hyper.offset == C.sizeof(_lib.SetDesc) - 8
    assert lib.cbo_offsetof_set_desc(b"points") == _lib.SetDesc.points.offset == 472    # every earlier offset unchanged
    assert C.sizeof(_lib.SetDesc) == 488 and C.sizeof(_lib.HyperResult) == 48
    assert lib.cbo_posterior_hyper_workspace_bytes(None, 1) == 0


def test_refusals_with_the_device_hidden():
    script = textwrap.dedent("""
        import ctypes as C, sys
        sys.path.insert(0, %r)
        from cbo_with_oop_b200 import _lib
        lib = _lib.load()
        h = (_lib.SetDesc * 1)()
        h[0].d, h[0].n_int, h[0].p[0], h[0].g_total, h[0].g_count, h[0].cost_fix = 1, 5, 10, 10, 10, 1.0
        h[0].x_int = h[0].y_int = 16          # never dereferenced: every call below is refused first
        fake = C.c_void_p(64)
        ok = [1e-6, 1e6, 0.1, 10.0]
        B = lambda v: (C.c_double * 4)(*v)
        def refused(rc, needle):
            msg = lib.cbo_last_error().decode()
            assert rc == -1 and needle in msg, (rc, msg)
        refused(lib.cbo_posterior_nll(h, None, 1, fake, None), "d_sets is NULL")
        refused(lib.cbo_posterior_hyper_fit(h, None, 1, B(ok), 10, 1e-6, fake, 1 << 20, fake, None), "d_sets is NULL")
        refused(lib.cbo_posterior_hyper_fit(h, fake, 1, B(ok), 10, 1e-6, fake, 1 << 20, fake, None), "hyper == NULL")
        h[0].hyper = 32
        for bad in ([1e-6, 1e6, 0.0, 10.0], [1e-6, float("inf"), 0.1, 10.0], [1e-6, 1e6, 10.0, 0.1], [2.0, 1.0, 0.1, 1.0],
                    [1e-6, 1e6, float("nan"), 1.0], [-1.0, 1e6, 0.1, 1.0]):
            refused(lib.cbo_posterior_hyper_fit(h, fake, 1, B(bad), 10, 1e-6, fake, 1 << 20, fake, None), "must be finite and positive")
        refused(lib.cbo_posterior_hyper_fit(h, fake, 1, None, 10, 1e-6, fake, 1 << 20, fake, None), "h_bounds is NULL")
        refused(lib.cbo_posterior_hyper_fit(h, fake, 1, B(ok), -1, 1e-6, fake, 1 << 20, fake, None), "max_iter")
        refused(lib.cbo_posterior_hyper_fit(h, fake, 1, B(ok), 10, 1e-6, fake, 8, fake, None), "too small")
        print("refusals ok")
    """ % ROOT)
    from cbo_with_oop_b200.build import build_library
    build_library()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, env=env, cwd=ROOT)
    assert r.returncode == 0 and "refusals ok" in r.stdout, r.stdout + r.stderr
