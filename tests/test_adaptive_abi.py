"""rc_render_adaptive without a GPU: the struct's layout, argument checks that come before the context is used, and the
C++ host's flags."""
import ctypes as C
import os
import subprocess
import tempfile

from conftest import ROOT
from racer_tracer_b200 import capi, harness
from test_host_cpp import CONFIG, racer_render, run  # noqa: F401  (racer_render: the fixture that builds the binary)


def test_rc_adaptive_layout_matches_the_header():
    src = r'''
    #include <stddef.h>
    #include <stdio.h>
    #include "racer_cuda.h"
    int main(void) {
      printf("%zu %zu %zu\n", sizeof(rc_adaptive), offsetof(rc_adaptive, min_samples), offsetof(rc_adaptive, threshold));
      return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(capi.rc_adaptive), capi.rc_adaptive.min_samples.offset, capi.rc_adaptive.threshold.offset]


def test_null_arguments_are_rejected(cuda_lib):
    """Each NULL is refused before the context is looked at, so an opaque stand-in for the context will do here."""
    fake_ctx = C.cast(C.create_string_buffer(64), C.c_void_p)
    p = harness.make_params(8, 8, 4, 2)
    a = capi.rc_adaptive(min_samples=2, threshold=0.01)
    rgb = (C.c_double * (8 * 8 * 3))()
    for args, what in (((None, C.byref(p), C.byref(a), rgb), "ctx"),
                       ((fake_ctx, None, C.byref(a), rgb), "params"),
                       ((fake_ctx, C.byref(p), None, rgb), "adaptive"),
                       ((fake_ctx, C.byref(p), C.byref(a), None), "out_rgb")):
        assert cuda_lib.rc_render_adaptive(*args, None, None, None) == capi.RC_ERR_INVALID, what
        assert what.encode() in cuda_lib.rc_last_error()


def test_min_samples_flag_needs_adaptive(racer_render, tmp_path):
    r = run(racer_render, "--config", CONFIG, "--min-samples", "8", "--dump-flat", str(tmp_path / "flat.json"), check=False)
    assert r.returncode != 0 and "--min-samples needs --adaptive" in r.stderr
