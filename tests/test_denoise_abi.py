"""rc_render_denoised / rc_denoise_filter without a GPU: the structs' layouts, argument checks that come before the
context is used, the C++ host's flags, and properties of the f64 restatement the GPU tests compare the filter with."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np

from conftest import ROOT, scene_path
from racer_tracer_b200 import capi, harness
from test_gpu_denoise import f32, restate, synthetic
from test_host_cpp import CONFIG, racer_render, run  # noqa: F401  (racer_render: the fixture that builds the binary)

STRUCTS = {"rc_denoise": ["levels", "reserved", "sigma_l", "sigma_n", "sigma_z"],
           "rc_denoise_aux": ["mean", "var", "albedo", "normal", "depth", "id"]}


def test_layouts_match_the_header():
    lines = [f'printf("%zu\\n", sizeof({s}));' for s in STRUCTS] + \
            [f'printf("%zu\\n", offsetof({s}, {f}));' for s, fs in STRUCTS.items() for f in fs]
    src = '#include <stddef.h>\n#include <stdio.h>\n#include "racer_cuda.h"\nint main(void) {\n' + "\n".join(lines) + "\nreturn 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(getattr(capi, s)) for s in STRUCTS] + \
           [getattr(getattr(capi, s), f).offset for s, fs in STRUCTS.items() for f in fs]
    assert got == want


def test_rust_structs_follow_the_header():
    sys_rs = open(os.path.join(ROOT, "racer_tracer_b200", "rust_shim", "racer-cuda-sys", "src", "lib.rs")).read()
    for name, fields in STRUCTS.items():
        body = re.search(r"pub struct %s \{(.*?)\n?\}" % name, sys_rs, flags=re.S).group(1)
        assert re.findall(r"pub (\w+)\s*:", body) == fields, name


def test_null_arguments_are_rejected(cuda_lib):
    """Each NULL is refused before the context is looked at, so an opaque stand-in for the context will do here."""
    fake_ctx = C.cast(C.create_string_buffer(64), C.c_void_p)
    p = harness.make_params(8, 8, 4, 2)
    dn = harness.default_denoise()
    rgb = (C.c_double * (8 * 8 * 3))()
    for args, what in (((None, C.byref(p), C.byref(dn), rgb), "ctx"),
                       ((fake_ctx, None, C.byref(dn), rgb), "params"),
                       ((fake_ctx, C.byref(p), None, rgb), "denoise"),
                       ((fake_ctx, C.byref(p), C.byref(dn), None), "out_rgb")):
        assert cuda_lib.rc_render_denoised(*args, None, None) == capi.RC_ERR_INVALID, what
        assert what.encode() in cuda_lib.rc_last_error()
    f = (C.c_double * (8 * 8 * 3))()
    ids = (C.c_uint32 * 64)()
    full = [fake_ctx, C.byref(dn), 8, 8, f, f, f, f, f, ids, rgb]
    for k in (0, 1, 4, 5, 6, 7, 8, 9, 10):
        args = list(full)
        args[k] = None
        assert cuda_lib.rc_denoise_filter(*args) == capi.RC_ERR_INVALID, k
        assert b"NULL" in cuda_lib.rc_last_error()


def test_denoise_flag_errors(racer_render, tmp_path):  # noqa: F811
    flat = ["--dump-flat", str(tmp_path / "flat.json")]
    r = run(racer_render, "--config", CONFIG, "--denoise", "--adaptive", "0.01", *flat, check=False)
    assert r.returncode != 0 and "--denoise and --adaptive exclude each other" in r.stderr
    r = run(racer_render, "--config", CONFIG, "--denoise-levels", "3", *flat, check=False)
    assert r.returncode != 0 and "--denoise-levels needs --denoise" in r.stderr
    cfg_file = tmp_path / "config.yml"
    cfg_file.write_text(open(CONFIG).read() + "gpu:\n  adaptive:\n    threshold: 0.01\n  denoise:\n    levels: 3\n")
    r = run(racer_render, "--config", str(cfg_file), *flat, check=False)
    assert r.returncode != 0 and "exclude each other" in r.stderr
    assert run(racer_render, "--config", CONFIG, "--scene", scene_path("cornell_box"), "--denoise", "--denoise-levels", "3",
               *flat, check=False).returncode == 0


# ---------------------------------------------------------------------------
# The restatement itself
# ---------------------------------------------------------------------------
def test_restatement_levels_0_is_the_identity():
    mean, var, albedo, normal, depth, ids = synthetic(40, 30, 1)
    np.testing.assert_allclose(restate(mean, var, albedo, normal, depth, ids, levels=0), np.sqrt(f32(mean)), rtol=1e-12)


def test_restatement_keeps_a_constant_image_constant():
    """mean = albedo / 2 exactly (a power of two survives the fp32 rounding): c = 1/2 everywhere, and so after the filter."""
    mean, var, albedo, normal, depth, ids = synthetic(50, 37, 2)
    albedo = np.maximum(albedo, 0.01)
    out = restate(albedo / 2, var, albedo, normal, depth, ids, levels=6)
    np.testing.assert_allclose(out, np.sqrt(f32(albedo) / 2), rtol=1e-12)


def test_restatement_never_mixes_across_ids():
    """Two ids whose colours differ wildly: filtered, each keeps exactly its own (constant) colour."""
    mean, var, albedo, normal, depth, ids = synthetic(48, 32, 3)
    ids = np.where(np.arange(48)[None, :] < 20, 5, 9).repeat(32, axis=0).astype(np.uint32)
    albedo[:] = 1.0
    normal[:] = (0.0, 0.0, 1.0)
    depth[:] = 3.0
    mean[ids == 5] = 0.1
    mean[ids == 9] = 2.5
    out = restate(mean, var, albedo, normal, depth, ids, levels=5, sigma_l=1e6, sigma_n=0.0, sigma_z=1e6)
    np.testing.assert_allclose(out[ids == 5], np.sqrt(f32(0.1)), rtol=1e-12)
    np.testing.assert_allclose(out[ids == 9], np.sqrt(f32(2.5)), rtol=1e-12)
    # ... while with one id the same parameters blur the edge
    blurred = restate(mean, var, albedo, normal, depth, np.full_like(ids, 5), levels=5, sigma_l=1e6, sigma_n=0.0, sigma_z=1e6)
    assert np.abs(blurred - out).max() > 0.1
