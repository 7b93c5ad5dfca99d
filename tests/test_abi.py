"""The C-ABI shared library loads and exports every symbol include/racer_cuda.h
declares; without a GPU the entry points fail loudly instead of falling back."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from racer_tracer_b200 import capi, harness

HEADER = os.path.join(ROOT, "include", "racer_cuda.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rc_[a-z0-9_]+)\s*\(", text)))


def test_header_and_python_binding_agree():
    assert declared_symbols() == sorted(capi.ABI_SYMBOLS)


def test_library_exports_every_declared_symbol(cuda_lib):
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    for name in declared_symbols():
        assert name in exported, f"{name} is declared in racer_cuda.h but not exported"
        assert hasattr(cuda_lib, name)
    assert cuda_lib.rc_abi_version() == 2
    assert not any(s.startswith("oracle_") for s in exported), "the product must not contain the oracle"


def test_struct_layouts_match_the_header(cuda_lib):
    """sizeof of every ctypes mirror equals the C compiler's sizeof."""
    src = r'''
    #include <stdio.h>
    #include "racer_cuda.h"
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(rc_material), sizeof(rc_texture),
             sizeof(rc_image), sizeof(rc_perlin), sizeof(rc_instance), sizeof(rc_bvh_node), sizeof(rc_scene),
             sizeof(rc_camera), sizeof(rc_params), sizeof(rc_tone_map), sizeof(rc_stats));
      return 0; }'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        sizes = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    mirrors = [capi.rc_material, capi.rc_texture, capi.rc_image, capi.rc_perlin, capi.rc_instance,
               capi.rc_bvh_node, capi.rc_scene, capi.rc_camera, capi.rc_params, capi.rc_tone_map, capi.rc_stats]
    assert sizes == [C.sizeof(m) for m in mirrors]


def test_no_gpu_means_a_loud_error_not_a_fallback(cuda_lib):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    ctx = C.c_void_p()
    st = cuda_lib.rc_create(None, 1, C.byref(ctx))
    assert st == capi.RC_ERR_NO_DEVICE
    assert b"no CPU fallback" in cuda_lib.rc_last_error()
    with pytest.raises(capi.RacerCudaError):
        harness.CudaRenderer([0])


def test_null_arguments_are_rejected(cuda_lib):
    assert cuda_lib.rc_create(None, 1, None) == capi.RC_ERR_INVALID
    assert cuda_lib.rc_upload_scene(None, None) == capi.RC_ERR_INVALID
    assert cuda_lib.rc_destroy(None) == capi.RC_OK
    p = harness.make_params(4, 4, 1, 1)
    assert cuda_lib.rc_render(None, C.byref(p), None, None) == capi.RC_ERR_INVALID


def test_product_never_touches_the_oracle():
    """Nothing under racer_tracer_b200/ may import, link or open oracle/."""
    pkg = os.path.join(ROOT, "racer_tracer_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h", ".sh")):
                text = open(os.path.join(d, f), errors="replace").read()
                assert "liboracle" not in text and "from oracle" not in text and "import oracle" not in text, f
    out = subprocess.run(["ldd", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_specialised_source_compiles_for_sm_100a(cuda_lib, cfg, tmp_path):
    """The CUDA source rc_params.specialize hands to NVRTC, compiled here with nvcc against the
    same headers (no GPU needed): scene constants appear as literals."""
    from conftest import scene_path
    job = harness.prepare_job(scene_path("cornell_box"), cfg, 64, 64)
    n = cuda_lib.rc_spec_source(job.scene.ptr, None, 0)
    buf = C.create_string_buffer(n + 1)
    assert cuda_lib.rc_spec_source(job.scene.ptr, buf, n + 1) == n
    src = buf.value.decode()
    assert "spec_closest_hit" in src and "#define RT_SPEC_MATS 9" in src   # lambertian + light
    # ... relative to the kernel's own origin, the centre of the box: the light's plane y = 554 is 276.5 above it
    assert "#define RT_SPEC_SHIFT mk3(277.5f, 277.5f, 277.5f)" in src and "276.5f" in src and "554.0f" not in src
    os.environ["RC_SPEC_NO_SHIFT"] = "1"
    try:
        n0 = cuda_lib.rc_spec_source(job.scene.ptr, None, 0)
        buf0 = C.create_string_buffer(n0 + 1)
        cuda_lib.rc_spec_source(job.scene.ptr, buf0, n0 + 1)
    finally:
        os.environ.pop("RC_SPEC_NO_SHIFT")
    assert "554.0f" in buf0.value.decode() and "RT_SPEC_SHIFT" not in buf0.value.decode()
    cu = tmp_path / "spec.cu"
    cu.write_text(src)
    subprocess.run(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I",
                    os.path.join(ROOT, "racer_tracer_b200", "csrc"), "-cubin", "-o", str(tmp_path / "spec.cubin"), str(cu)],
                   check=True)
    big = harness.prepare_job(scene_path("clown"), cfg, 64, 64)
    assert cuda_lib.rc_spec_source(big.scene.ptr, None, 0) > 0          # 23 spheres still fit the constant bank


def test_checker_chains_of_any_depth_and_cycles(cuda_lib, cfg):
    """Checker children are followed to any depth (checkered.rs:32-43), so a chain of six is a valid scene; a cycle of
    checker children — which YAML cannot express but a host can pass — is rejected with a message that names it.
    rc_spec_source runs the same scene validation as rc_upload_scene, without a GPU."""
    from test_gpu_shading_probes import checker_chain_job
    job = checker_chain_job(cfg, 6)
    assert cuda_lib.rc_spec_source(job.scene.ptr, None, 0) > 0, cuda_lib.rc_last_error()
    top = job.scene.c.n_textures - 1
    for leaf in (1, top):                    # c_1's leaf pointing back at the root; the root pointing at itself
        job = checker_chain_job(cfg, 6)
        tex = job.scene.c.textures
        tex[leaf].type, tex[leaf].a, tex[leaf].b = capi.RC_TEX_CHECKER, top, 0
        assert cuda_lib.rc_spec_source(job.scene.ptr, None, 0) == -1
        assert b"cycle" in cuda_lib.rc_last_error()


def _compile_like_the_library(src: str, tmp_path):
    """NVRTC with the headers and options rc_spec.cuh uses (it is stricter than nvcc about inline functions
    that are declared but never defined); nvcc when the cuda-python bindings are not importable."""
    csrc = os.path.join(ROOT, "racer_tracer_b200", "csrc")
    try:
        from cuda.bindings import nvrtc
    except ImportError:
        cu = tmp_path / "spec.cu"
        cu.write_text(src)
        subprocess.run(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I", csrc,
                        "-cubin", "-o", str(tmp_path / "spec.cubin"), str(cu)], check=True)
        return
    names = [b"rt_math.cuh", b"rt_scene.cuh", b"rt_kernels.cuh"]
    headers = [open(os.path.join(csrc, n.decode()), "rb").read() for n in names]
    err, prog = nvrtc.nvrtcCreateProgram(src.encode(), b"spec_scene.cu", len(names), headers, names)
    assert int(err) == 0
    opts = [b"--gpu-architecture=sm_100a", b"-std=c++17", b"-lineinfo", b"-default-device"]
    err, = nvrtc.nvrtcCompileProgram(prog, len(opts), opts)
    _, size = nvrtc.nvrtcGetProgramLogSize(prog)
    log = b" " * size
    nvrtc.nvrtcGetProgramLog(prog, log)
    assert int(err) == 0, log.decode(errors="replace")[:3000]
    _, size = nvrtc.nvrtcGetCUBINSize(prog)
    assert size > 0


@pytest.mark.parametrize("name,mode,needle", [
    ("sandbox", None, "rect_closest_fma"), ("sandbox_boxes", None, "aabb_hit_reference"), ("clown", None, "sphere_hit<float>"),
    ("emissive", None, "#define RT_SPEC_BG_BLACK 1"),
    # the BVH paths: kinds of primitive / material / wrapper / motion as defines, tables stay in memory
    ("random", None, "megakernel_body<RT_MODE_GLOBAL_BVH, 0, 10, true>"),
    ("sandbox_boxes", "smem", "megakernel_body<RT_MODE_SMEM_BVH, 0, 10, false>"),
    ("noise_and_textures", "global", "#define RT_SPEC_PRIMS 1\n"),
])
def test_specialised_source_of_every_scene_kind_compiles(cuda_lib, cfg, tmp_path, name, mode, needle):
    """The generator's other branches — instanced objects (cull box + ray transform + packed box faces), the
    float-index closest hit of rectangle-only scenes, spheres, textures, and the BVH paths — produce code the
    run-time compiler accepts for sm_100a."""
    from conftest import scene_path
    job = harness.prepare_job(scene_path(name), cfg, 64, 64)
    if mode:
        os.environ["RC_SCENE_MODE"] = mode
    try:
        n = cuda_lib.rc_spec_source(job.scene.ptr, None, 0)
        assert n > 0, cuda_lib.rc_last_error()
        buf = C.create_string_buffer(n + 1)
        assert cuda_lib.rc_spec_source(job.scene.ptr, buf, n + 1) == n
    finally:
        if mode:
            del os.environ["RC_SCENE_MODE"]
    src = buf.value.decode()
    assert needle in src
    _compile_like_the_library(src, tmp_path)


def _spec_source(cuda_lib, job, camera=None):
    if camera is not None:
        os.environ["RC_SPEC_CAMERA"] = ",".join(repr(float(v)) for v in camera)
    try:
        n = cuda_lib.rc_spec_source(job.scene.ptr, None, 0)
        assert n > 0, cuda_lib.rc_last_error()
        buf = C.create_string_buffer(n + 1)
        assert cuda_lib.rc_spec_source(job.scene.ptr, buf, n + 1) == n
    finally:
        os.environ.pop("RC_SPEC_CAMERA", None)
    return buf.value.decode()


def test_opposite_walls_become_one_test_only_when_every_ray_starts_between_them(cuda_lib, cfg, tmp_path):
    """Slab pairs of the specialised closest hit: two rectangles with the same bounds on parallel planes are
    tested as max(t_i, t_j) — one rectangle test for both — iff all geometry and the pinhole lie between the
    planes.  Cornell from its own camera: the side walls and floor / ceiling; from a camera left of the red wall
    only floor / ceiling; with a lens, or in a scene with spheres or instanced boxes, none."""
    from conftest import scene_path
    job = harness.prepare_job(scene_path("cornell_box"), cfg, 64, 64)
    def n_tests(src):   # rectangle tests of the closest hit, whichever form of the update each one uses
        return src.count("rect_closest_fma(") + src.count("rect_closest_fma_pair(") + src.count("rect_closest_first(")
    inside = _spec_source(cuda_lib, job, camera=job.camera.origin)
    assert inside.count("// slab pair") == 2 and n_tests(inside) == 4 and inside.count("rect_closest_fma_pair(") == 2
    assert inside.count("rect_closest_first(") == 1    # the first test selects between literals
    _compile_like_the_library(inside, tmp_path)
    left_of_the_box = _spec_source(cuda_lib, job, camera=(-100.0, 278.0, -800.0))
    assert left_of_the_box.count("// slab pair") == 1 and n_tests(left_of_the_box) == 5
    # (planes y = 0 / 555 relative to the kernel's origin, handed over as register constants)
    assert "pair_t(X.k_spec[0], X.k_spec[1], r.o.y, r.inv_d.y, t1, t2);   // planes -277.5f, 277.5f" in left_of_the_box
    assert "fmaxf(t1, t2)" in left_of_the_box
    above = _spec_source(cuda_lib, job, camera=(278.0, 900.0, 278.0))
    assert above.count("// slab pair") == 1 and "pair_t(X.k_spec[0], X.k_spec[1], r.o.x" in above
    no_camera = _spec_source(cuda_lib, job)            # origin (0, 0, 0): on the walls, not between them
    assert no_camera.count("// slab pair") == 0 and n_tests(no_camera) == 6
    for other in ("sandbox_boxes", "emissive"):
        j = harness.prepare_job(scene_path(other), cfg, 64, 64)
        assert "// slab pair" not in _spec_source(cuda_lib, j, camera=j.camera.origin)


def test_generated_kernel_variants_compile_and_agree_on_their_planes(cuda_lib, cfg, tmp_path, monkeypatch):
    """The pieces of the generated Cornell kernel that can be switched off one at a time (DESIGN §3.1 v25 / v26) all
    compile, and in every variant the plane constant the hit record snaps a point to (spec_snap_row: the staged
    table's K) is the same literal as the plane the rectangle TEST uses — if the two differed by an ulp, a ray leaving
    a wall would re-hit it at t != 0."""
    import re
    from conftest import scene_path
    job = harness.prepare_job(scene_path("cornell_box"), cfg, 64, 64)
    for env in ({}, {"RC_SPEC_NO_REG_CONSTS": "1"}, {"RC_SPEC_PACK_ALL": "1"}, {"RC_SPEC_NO_SHIFT": "1"}, {"RC_SPEC_NO_SLAB": "1"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        src = _spec_source(cuda_lib, job, camera=job.camera.origin)
        for k in env:
            monkeypatch.delenv(k)
        _compile_like_the_library(src, tmp_path)
        tested = re.findall(r"\((-?[0-9.]+f) - r\.o\.[xyz]\) \* r\.inv_d", src)           # single rectangles
        for a, b in re.findall(r"// planes (-?[0-9.]+f), (-?[0-9.]+f)", src):                 # slab pairs
            tested += [a, b]
        for a, b in re.findall(r"pair_t\((-?[0-9.]+f), (-?[0-9.]+f), r\.o", src):             # packed pairs with literal planes
            if "// planes" not in src or (a, b) not in re.findall(r"// planes (-?[0-9.]+f), (-?[0-9.]+f)", src):
                tested += [a, b]
        rows = re.findall(r"case \d+: a = make_float4\(([^)]*)\); bx = (-?[0-9.]+f); cw = [0-9.]+f;", src)
        if "RC_SPEC_NO_SHIFT" in env:
            assert not rows and "RT_SPEC_SNAP_TABLE" not in src      # world coordinates: the table keeps the uploaded k
            continue
        assert len(rows) == 6 and "#define RT_SPEC_SNAP_TABLE 1" in src
        snapped = []
        for a, bx in rows:
            mx, my, kx, ky = [t.strip() for t in a.split(",")]
            ks = [v for v, m in ((kx, mx), (ky, my)) if m == "0.0f"] or [bx]
            assert len(ks) == 1
            snapped.append(ks[0])
        assert sorted(snapped) == sorted(tested), (env, sorted(snapped), sorted(tested))
