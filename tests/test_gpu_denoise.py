"""rc_render_denoised / rc_denoise_filter: the à-trous filter against an f64 restatement of its contract, its inputs
against the renders and hits they claim to be, one quality claim, and the behaviour of the call.

Error model of the filter (GPU fp32 against `restate`, f64, on the same fp32-rounded inputs).  Every weight is a
continuous function of its inputs but for the id test, which compares integers exactly, so the two differ by rounding
only.  In fp32 a weight is off by a relative ~(3 sigma_n + 30) 2^-24: the normals' dot product is off by ~3 2^-24
and the power sigma_n multiplies that; exp, the divisions and the products add a few units each.  A level's output is a
convex combination, so it moves by at most that much times the spread of the values it mixes; levels add.  For the
synthetic images (linear values in [0.05, 3], so gamma'd values >= 0.2) that is far below 1e-4 in gamma'd units on
average, and the test allows 1e-4 at every pixel.  Real renders have values near 0, where the gamma (sqrt) magnifies a
linear difference d into sqrt(d); there the comparison is |gpu^2 - host^2| <= 1e-4 max(1, host^2), i.e. 1e-4 / (gpu +
host) in gamma'd units.
"""
import ctypes as C
import math
import threading
import time

import numpy as np
import pytest

from conftest import SCENES, scene_path
from racer_tracer_b200 import capi, harness
from test_gpu_adaptive import S_HOST, per_sample_y, upload
from test_host_cpp import CONFIG, read_png, racer_render, run  # noqa: F401  (racer_render: the fixture that builds the binary)

pytestmark = pytest.mark.gpu

W, H = 203, 117
SEED = 7
DEPTH = 10
GAMMA_TOL = 1e-4
H5 = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16])
H3 = np.array([0.25, 0.5, 0.25])


# ---------------------------------------------------------------------------
# The f64 restatement of include/racer_cuda.h's filter
# ---------------------------------------------------------------------------
def f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def shift(a, dy, dx):
    """(b, inside): b[y, x] = a[y + dy, x + dx] where that is inside the image, 0 elsewhere."""
    h, w = a.shape[:2]
    out, inside = np.zeros_like(a), np.zeros((h, w), dtype=bool)
    y0, y1, x0, x1 = max(0, -dy), min(h, h - dy), max(0, -dx), min(w, w - dx)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = a[y0 + dy:y1 + dy, x0 + dx:x1 + dx]
        inside[y0:y1, x0:x1] = True
    return out, inside


def restate(mean, var, albedo, normal, depth, ids, levels=5, sigma_l=4.0, sigma_n=128.0, sigma_z=1.0):
    """The filter in f64 on the fp32-rounded inputs -> gamma'd rgb (H, W, 3)."""
    mean, var, albedo, normal = f32(mean), f32(var), f32(albedo), f32(normal)
    with np.errstate(over="ignore"):
        depth = f32(depth)                                   # a miss's DBL_MAX becomes inf, as on the GPU
    ids = np.asarray(ids, dtype=np.uint32)
    h = var.shape[0]
    a = np.maximum(albedo, f32(1e-3))
    c, v = mean / a, var / a.mean(axis=2) ** 2
    hit = ids != 0
    for k in range(levels):
        s = 2 ** k
        gs, gw = np.zeros_like(v), np.zeros_like(v)
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                vq, inside = shift(v, dy, dx)
                gs += H3[dy + 1] * H3[dx + 1] * np.where(inside, vq, 0.0)
                gw += H3[dy + 1] * H3[dx + 1] * inside
        l_p = c.mean(axis=2)
        l_den = sigma_l * np.sqrt(gs / gw) + 1e-3
        sc, sv, sw = np.zeros_like(c), np.zeros_like(v), np.zeros_like(v)
        for j in range(-2, 3):
            for i in range(-2, 3):
                cq, inside = shift(c, j * s, i * s)
                vq = shift(v, j * s, i * s)[0]
                use = inside & (shift(ids, j * s, i * s)[0] == ids)
                w = H5[i + 2] * H5[j + 2] * np.exp(-np.abs(l_p - cq.mean(axis=2)) / l_den)
                if (i, j) != (0, 0):
                    nq, zq = shift(normal, j * s, i * s)[0], shift(depth, j * s, i * s)[0]
                    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
                        wn = np.maximum(0.0, (normal * nq).sum(axis=2)) ** sigma_n
                        wz = np.exp(-np.abs(depth - zq) / (sigma_z * depth * math.hypot(i, j) * s / h))
                    w = w * np.where(hit, wn * wz, 1.0)
                w = np.where(use, w, 0.0)
                sc += w[..., None] * np.where(use[..., None], cq, 0.0)
                sv += w * w * np.where(use, vq, 0.0)
                sw += w
        c, v = sc / sw[..., None], sv / sw ** 2
    return np.sqrt(np.maximum(0.0, a * c))


def synthetic(w, h, seed):
    """Noise over piecewise-constant ids (one region a miss), normals and depths, albedos with a channel below the
    1e-3 clamp, and a region of zero variance."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    region = (xx // 11 + 2 * (yy // 9)) % 6                            # 6 ids in blocks that recur across the image
    ids = (10 + region).astype(np.uint32)
    ids[region == 5] = 0
    base_n = rng.normal(size=(6, 3))
    normal = base_n[region] / np.linalg.norm(base_n, axis=1)[region][..., None] + 0.06 * rng.normal(size=(h, w, 3))
    normal /= np.linalg.norm(normal, axis=2, keepdims=True)
    depth = rng.uniform(2.0, 6.0, 6)[region] * (1.0 + 0.3 * xx / w) + 0.02 * rng.random((h, w))
    albedo = rng.uniform(0.1, 1.0, (6, 3))[region]
    albedo[region == 2, 0] = 0.0
    clean = albedo * (0.4 + 0.3 * np.sin(xx / 9.0) * np.cos(yy / 13.0))[..., None] + 0.05
    var = rng.uniform(0.0, 0.03, (h, w))
    var[region == 1] = 0.0                                             # zero variance: constant there
    noise = rng.normal(size=(h, w, 3)) * np.sqrt(var)[..., None] * 3.0
    mean = np.clip(clean + noise, 0.05, 3.0)
    mean[region == 1] = clean[region == 1]
    normal[ids == 0] = 0.0
    depth[ids == 0] = np.finfo(np.float64).max
    albedo[ids == 0] = 1.0
    return mean, var, albedo, normal, depth, ids


PARAM_SETS = [(4.0, 128.0, 1.0), (1.0, 32.0, 0.5), (10.0, 64.0, 4.0)]


def denoise(levels, sigma_l, sigma_n, sigma_z):
    return harness.default_denoise(levels, sigma_l, sigma_n, sigma_z)


# ---------------------------------------------------------------------------
# The filter against the restatement, on synthetic inputs
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("params", PARAM_SETS, ids=["svgf", "tight", "loose"])
@pytest.mark.parametrize("levels", range(7))
@pytest.mark.parametrize("size", [(203, 117), (64, 64)], ids=["203x117", "64x64"])
def test_filter_matches_the_restatement(renderer, size, levels, params):
    w, h = size
    inputs = synthetic(w, h, 100 + levels)
    got = renderer.denoise_filter(*inputs, denoise=denoise(levels, *params))
    st = renderer.stats()
    assert st.kernel_launches == 2 + levels and st.samples == 0 and st.gpu_ms > 0
    want = restate(*inputs, levels, *params)
    err = np.abs(got - want).max()
    assert err <= GAMMA_TOL, f"max |gpu - f64| = {err:.3g}"
    if levels > 0:   # counterfactuals: one level fewer, or sigma_n halved, are told apart by the same tolerance
        sl, sn, sz = params
        assert np.abs(got - restate(*inputs, levels - 1, *params)).max() > GAMMA_TOL
        assert np.abs(got - restate(*inputs, levels, sl, sn / 2, sz)).max() > GAMMA_TOL


def test_filter_is_bit_identical_when_repeated(renderer):
    inputs = synthetic(203, 117, 5)
    a = renderer.denoise_filter(*inputs)
    renderer.denoise_filter(*synthetic(64, 64, 6), denoise=denoise(3, 1.0, 32.0, 0.5))
    b = renderer.denoise_filter(*inputs)
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


# ---------------------------------------------------------------------------
# Composition on real scenes
# ---------------------------------------------------------------------------
def gamma_close(got, want):
    """Within the module's error model: |got^2 - want^2| <= 1e-4 max(1, want^2)."""
    return np.abs(got * got - want * want) <= GAMMA_TOL * np.maximum(1.0, want * want)


def aux_inputs(aux):
    return aux["mean"], aux["var"], aux["albedo"], aux["normal"], aux["depth"], aux["id"]


@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("name", SCENES)
def test_render_denoised_composes_on_real_scenes(renderer, cfg, name, spec):
    upload(renderer, cfg, name)
    p = harness.make_params(W, H, 16, DEPTH, seed=SEED, specialize=spec)
    rgb, aux = renderer.render_denoised(p, aux=True)
    st = renderer.stats()
    assert st.specialized == spec
    ok = gamma_close(rgb, restate(*aux_inputs(aux)))
    assert ok.all(), f"{int((~ok).sum())} values beyond the error model"
    again = renderer.denoise_filter(*aux_inputs(aux))
    assert np.array_equal(again.view(np.uint8), rgb.view(np.uint8))
    # the inputs are what they claim: the mean is rc_render's image before the gamma ...
    uni = renderer.render(p)
    close = np.isclose(np.sqrt(aux["mean"]), uni, rtol=1e-5, atol=1e-7).all(axis=2)
    np.testing.assert_allclose(np.sqrt(aux["mean"]), uni, rtol=1e-3, atol=1e-6)
    # (as in test_gpu_adaptive: one pixel of noise_and_textures' specialised moments kernel is off by 4e-5)
    assert (~close).sum() <= max(1, close.size // 2000), f"{int((~close).sum())} pixels beyond rtol 1e-5"
    # ... and the guides are rc_primary_aov's, bit for bit
    ids, t, nrm, _ = renderer.primary_aov(p, precision=32)
    assert np.array_equal(aux["id"].ravel(), ids)
    assert np.array_equal(aux["depth"].ravel().view(np.uint64), t.view(np.uint64))
    assert np.array_equal(aux["normal"].reshape(-1, 3).view(np.uint64), nrm.view(np.uint64))


@pytest.mark.parametrize("name", ["cornell_box", "three_balls", "noise_and_textures"])
def test_variance_recomputed_on_the_host(renderer, cfg, name):
    """aux.var against the f64 value from the 16 one-sample shares of a 16-spp frame; the fp32 sums behind S1 and S2
    move S2 - S1^2 / n by at most 4 (n + 4) 2^-24 S2 (test_gpu_adaptive.host_err)."""
    upload(renderer, cfg, name)
    y = per_sample_y(renderer)
    n = S_HOST
    s1, s2 = y.sum(0), (y * y).sum(0)
    want = np.maximum(0.0, (s2 - s1 * s1 / n) / (n - 1)) / n
    slack = 4.0 * (n + 4) * 2.0 ** -24 * s2 / ((n - 1) * n) + 1e-6 * want + 1e-300
    _, aux = renderer.render_denoised(harness.make_params(W, H, n, DEPTH, seed=SEED), aux=True)
    off = np.abs(aux["var"] - want) > slack
    assert not off.any(), f"{int(off.sum())} pixels: GPU {aux['var'][off][:4]} host {want[off][:4]}"
    assert (want > 0).mean() > 0.3
    wrong = np.roll(y, -1, axis=0)[: n - 1]   # counterfactual: 15 of the samples
    w1, w2 = wrong.sum(0), (wrong * wrong).sum(0)
    alt = np.maximum(0.0, (w2 - w1 * w1 / (n - 1)) / (n - 2)) / (n - 1)
    assert (np.abs(aux["var"] - alt) > slack).mean() > 0.3


def material_colour_by_id(job):
    """object id -> albedo the guide must give: texture colour for Lambertian / Metal, 1 otherwise (solid colours)."""
    fs = job.scene
    out = {}
    for pid, m in zip(fs.np["prim_id"], fs.np["prim_material"]):
        mat = fs.materials[int(m)]
        if mat.type in (capi.RC_MAT_LAMBERTIAN, capi.RC_MAT_METAL):
            tex = fs.textures[mat.texture]
            out[int(pid)] = (tuple(tex.color) if tex.type == capi.RC_TEX_SOLID else None)
        else:
            out[int(pid)] = (1.0, 1.0, 1.0)
    return out


@pytest.mark.parametrize("name", SCENES)
def test_albedo_guide(renderer, cfg, name, oracle):
    """Solid colours: the hit material's colour exactly.  Textures: oracle_texture_value at the f64 first hit, skipping
    pixels whose fp32 and f64 first hits differ.  (The albedo kernel is compiled apart from the one that gives the
    ids, so at most one pixel in 2000 may have hit another object at a silhouette.)"""
    job = upload(renderer, cfg, name)
    p = harness.make_params(W, H, 4, DEPTH, seed=SEED)
    _, aux = renderer.render_denoised(p, aux=True)
    alb = aux["albedo"].reshape(-1, 3)
    ids = aux["id"].ravel()
    colour = material_colour_by_id(job)
    solid = np.array([colour.get(int(i)) is not None for i in ids]) & (ids != 0)
    want = np.array([f32(colour[int(i)]) if s else (0.0, 0.0, 0.0) for i, s in zip(ids, solid)]).reshape(-1, 3)
    off = int((ids == 0).sum() - (alb[ids == 0] == 1.0).all(axis=1).sum()) + int((alb[solid] != want[solid]).any(axis=1).sum())
    assert off <= max(1, ids.size // 2000), f"{off} pixels off"
    textured = (ids != 0) & ~solid
    if not textured.any():
        return
    ids64, _, n64, p64 = renderer.primary_aov(p, precision=64)
    check = np.flatnonzero(textured & (ids64 == ids))
    assert len(check) > 0.9 * textured.sum()
    fs = job.scene
    tex_of = {int(pid): fs.materials[int(m)].texture for pid, m in zip(fs.np["prim_id"], fs.np["prim_material"])}
    L = oracle.lib()
    out = oracle.d3([0, 0, 0])
    bad = 0
    for k in check:
        nrm = n64[k]                                    # camera outside every sphere: the face normal is the outward one
        u = (math.atan2(-nrm[2], nrm[0]) + math.pi) / (2 * math.pi)
        v = math.acos(max(-1.0, min(1.0, -nrm[1]))) / math.pi
        L.oracle_texture_value(fs.ptr, tex_of[int(ids[k])], u, v, oracle.d3(p64[k]), out)
        bad += np.abs(alb[k] - np.array(list(out))).max() > 2e-3
    # checker edges (the sign of a product of sines) and texel edges may flip between the fp32 and the f64 hit point
    assert bad <= 0.01 * len(check), f"{bad} of {len(check)} textured pixels"


# ---------------------------------------------------------------------------
# Quality: the one statistical claim
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name,size", [("cornell_box", (480, 270)), ("three_balls", (300, 300))])
def test_denoised_beats_noisy_at_64spp(renderer, cfg, name, size):
    w, h = size
    upload(renderer, cfg, name, w, h)
    ref = renderer.render(harness.make_params(w, h, 4096, DEPTH, seed=424242))
    p = harness.make_params(w, h, 64, DEPTH, seed=SEED)
    noisy = renderer.render(p)
    den = renderer.render_denoised(p)
    rmse = lambda img: float(np.sqrt(((img - ref) ** 2).mean()))  # noqa: E731
    assert rmse(den) < rmse(noisy), (rmse(den), rmse(noisy))


# ---------------------------------------------------------------------------
# Behaviour of the call
# ---------------------------------------------------------------------------
def test_two_identical_calls_are_bit_identical_and_stats(renderer, cfg):
    upload(renderer, cfg, "noise_and_textures")
    p = harness.make_params(W, H, 32, DEPTH, seed=SEED)
    first = renderer.render_denoised(p)
    st = renderer.stats()
    assert st.samples == W * H * 32
    # one megakernel (the moments round runs unsliced), moments, two guide kernels, prepare, 5 levels, finish
    assert st.kernel_launches == 1 + 4 + 5 + 1
    assert st.gpu_ms > 0 and st.segments >= st.samples
    renderer.render(harness.make_params(64, 48, 3, DEPTH, seed=99))
    renderer.render_denoised(harness.make_params(120, 77, 8, DEPTH, seed=98), denoise=denoise(2, 1.0, 8.0, 2.0))
    again = renderer.render_denoised(p)
    assert np.array_equal(first.view(np.uint8), again.view(np.uint8))
    zero = renderer.render_denoised(p, denoise=denoise(0, 4.0, 128.0, 1.0))
    assert renderer.stats().kernel_launches == 1 + 4 + 0 + 1
    np.testing.assert_allclose(zero, renderer.render(p), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("case", ["samples_1", "levels_neg", "levels_11", "sigma_l_0", "sigma_z_neg", "sigma_n_neg",
                                  "sigma_nan", "sigma_inf", "wavefront", "rejection", "rounds_7", "world_2",
                                  "spec_fixed_jitter"])
def test_unsupported_inputs_are_rejected(renderer, cfg, case):
    upload(renderer, cfg, "cornell_box")
    kw, s, dn = {}, 8, [5, 4.0, 128.0, 1.0]
    if case == "samples_1":
        s = 1
    elif case == "levels_neg":
        dn[0] = -1
    elif case == "levels_11":
        dn[0] = 11
    elif case == "sigma_l_0":
        dn[1] = 0.0
    elif case == "sigma_z_neg":
        dn[3] = -1.0
    elif case == "sigma_n_neg":
        dn[2] = -1.0
    elif case == "sigma_nan":
        dn[1] = float("nan")
    elif case == "sigma_inf":
        dn[2] = float("inf")
    elif case == "wavefront":
        kw = {"variant": capi.RC_VARIANT_WAVEFRONT}
    elif case == "rejection":
        kw = {"sampler": capi.RC_SAMPLER_REJECTION}
    elif case == "rounds_7":
        kw = {"rng_rounds": 7}
    elif case == "world_2":
        kw = {"rank": 0, "world": 2}
    elif case == "spec_fixed_jitter":
        kw = {"specialize": 1, "fixed_jitter": 1}
    with pytest.raises(capi.RacerCudaError) as e:
        renderer.render_denoised(harness.make_params(W, H, s, DEPTH, seed=SEED, **kw), denoise=denoise(*dn))
    assert e.value.status == capi.RC_ERR_INVALID
    if case.startswith(("levels", "sigma")):   # the filter on its own checks the same parameters
        with pytest.raises(capi.RacerCudaError) as e:
            renderer.denoise_filter(*synthetic(16, 16, 0), denoise=denoise(*dn))
        assert e.value.status == capi.RC_ERR_INVALID


def test_cancel_on_entry_and_mid_render(renderer, cfg):
    upload(renderer, cfg, "cornell_box")
    p = harness.make_params(W, H, 16, DEPTH, seed=SEED)
    flag = C.c_int32(1)
    with pytest.raises(capi.RacerCudaError) as e:
        renderer.render_denoised(p, cancel=flag)
    assert e.value.status == capi.RC_ERR_CANCELLED
    flag.value = 0
    assert np.array_equal(renderer.render_denoised(p, cancel=flag), renderer.render_denoised(p))
    # raised while the render runs (as test_gpu_bench_config's rc_render case): RC_OK, and nothing is written
    w, h, spp = 1920, 1080, 8192                      # ~0.3 s of GPU time if left alone
    upload(renderer, cfg, "cornell_box", w, h)
    renderer.render_denoised(harness.make_params(w, h, 64, 20, seed=1))   # warm up
    out = np.full((h, w, 3), -1.0)
    flag = C.c_int32(0)
    t = threading.Timer(0.03, lambda: setattr(flag, "value", 1))
    t0 = time.perf_counter()
    t.start()
    dn = harness.default_denoise()
    st = renderer.lib.rc_render_denoised(renderer.ctx, C.byref(harness.make_params(w, h, spp, 20, seed=1)), C.byref(dn),
                                         out.ctypes.data_as(C.POINTER(C.c_double)), None,
                                         C.cast(C.pointer(flag), C.POINTER(C.c_int32)))
    dt = time.perf_counter() - t0
    t.join()
    assert st == capi.RC_OK
    assert float(out.min()) == -1.0 and float(out.max()) == -1.0, "a cancelled render wrote pixels"
    assert dt < 0.6 * (w * h * spp / 5.0e10), dt


def test_racer_render_denoise_png_equals_the_harness_path(racer_render, tmp_path, cfg, renderer):  # noqa: F811
    w, h, spp = 96, 64, 32
    job = harness.prepare_job(scene_path("cornell_box"), cfg, w, h)
    renderer.upload(job)
    rgb = renderer.render_denoised(harness.make_params(w, h, spp, cfg.render.max_depth, seed=5, specialize=2),
                                   denoise=denoise(3, 4.0, 128.0, 1.0))
    want = renderer.postprocess(job.tone_map, rgb)[0]
    common = ["--scene", scene_path("cornell_box"), "--width", str(w), "--height", str(h), "--samples", str(spp), "--seed", "5"]
    out = tmp_path / "flags.png"
    run(racer_render, "--config", CONFIG, *common, "--denoise", "--denoise-levels", "3", "--out", str(out))
    assert np.array_equal(read_png(out), want)
    cfg_file = tmp_path / "config.yml"
    cfg_file.write_text(open(CONFIG).read() + "gpu:\n  denoise:\n    levels: 3\n    sigma_l: 4\n")
    out = tmp_path / "block.png"
    run(racer_render, "--config", str(cfg_file), *common, "--out", str(out))
    assert np.array_equal(read_png(out), want)
