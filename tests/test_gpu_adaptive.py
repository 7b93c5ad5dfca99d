"""rc_render_adaptive: adaptive sampling, checked against renders and arithmetic that do not depend on it.

* Equivalence.  Streams are counter-based on (pixel, sample, segment), so a pixel the adaptive render gives n samples
  must equal the uniform n-spp render there, up to the order of fp32 sums (rtol 1e-5, atol 1e-7, as test_gpu_shares).
* Decisions.  The sample shares of a 16-spp frame (RC_SPLIT_SAMPLES, world 16, rank k = sample k) give every pixel's
  per-sample radiance, c_k = 16 out_k^2.  From them the host recomputes every error estimate in f64 and predicts each
  pixel's sample count; the GPU must agree wherever the estimate is not within 1e-4 (relative) of the threshold at a
  round that decides.  The same prediction from the wrong samples (rank k + 1) must not.
* Calibration, limits, state, statistics, errors, cancellation, and the C++ host's flags and config block.
"""
import math

import ctypes as C
import numpy as np
import pytest

from conftest import scene_path
from racer_tracer_b200 import capi, harness
from test_gpu_parity import job_for
from test_host_cpp import CONFIG, read_png, racer_render, run  # noqa: F401  (racer_render: the fixture that builds the binary)

pytestmark = pytest.mark.gpu

W, H = 203, 117
SEED = 7
DEPTH = 10
EQ_SCENES = ["cornell_box", "three_balls", "noise_and_textures", "random", "sandbox"]
_JOBS = {}


def upload(renderer, cfg, name, w=W, h=H):
    if (name, w, h) not in _JOBS:
        _JOBS[(name, w, h)] = job_for(name, cfg, w, h)
    renderer.upload(_JOBS[(name, w, h)])
    return _JOBS[(name, w, h)]


def doubling_set(n0, s):
    out, n = [], n0
    while n < s:
        out.append(n)
        n *= 2
    return out + [s]


def check_map(spp, err, threshold, n0, s):
    """Every n_p is one of n0, 2 n0, 4 n0, .., S; a pixel stopped before S only because its estimate passed."""
    assert np.isin(spp, doubling_set(n0, s)).all()
    assert (err[spp < s] <= threshold).all()
    assert np.isfinite(err).all() and (err >= 0).all()


def _err(mu, num, n):
    se = np.sqrt(np.maximum(0.0, num / (n - 1)) / n)
    return 0.5 * (np.sqrt(mu + se) - np.sqrt(np.maximum(mu - se, 0.0)))


def host_err(y, n):
    """(err, lo, hi): the header's estimate from the first n per-sample y (axis 0) in f64, and its range under the
    rounding of the library's fp32 sums.  S2 - S1^2 / n is what the spread rests on; the fp32 sums of n values (and the
    per-sample y and y^2) are each off by at most about (n + 4) 2^-24 of S2, so that difference is bounded by
    +-4 (n + 4) 2^-24 S2 and err (monotone in it) by the estimate at the two ends."""
    s1, s2 = y[:n].sum(0), (y[:n] ** 2).sum(0)
    mu, num = s1 / n, s2 - s1 * s1 / n
    dnum = 4.0 * (n + 4) * 2.0 ** -24 * s2
    return _err(mu, num, n), _err(mu, num - dnum, n), _err(mu, num + dnum, n)


def predict(y, threshold, n0, s, rel=1e-4):
    """(n_p, ambiguous): the host's schedule, and the pixels whose estimate (with its fp32 range) lies within `rel` of
    the threshold at a round that decides whether they go on."""
    n_p = np.full(y.shape[1:], s, dtype=np.int64)
    going = np.ones(y.shape[1:], dtype=bool)
    ambiguous = np.zeros(y.shape[1:], dtype=bool)
    for n in doubling_set(n0, s):
        if n == s:
            break
        e, lo, hi = host_err(y, n)
        ambiguous |= going & (lo - rel * threshold <= threshold) & (threshold <= hi + rel * threshold)
        stop = going & (e <= threshold)
        n_p[stop] = n
        going &= ~stop
    return n_p, ambiguous


# ---------------------------------------------------------------------------
# Equivalence with uniform renders
# ---------------------------------------------------------------------------
def _equivalence(renderer, w, h, s, n0, spec):
    # a threshold that splits the image: the median estimate after n0 samples
    rgb0, spp0, err0 = renderer.render_adaptive(harness.make_params(w, h, s, DEPTH, seed=SEED, specialize=spec), 1e30, n0)
    assert (spp0 == n0).all()
    threshold = float(np.median(err0[err0 > 0]))
    rgb, spp, err = renderer.render_adaptive(harness.make_params(w, h, s, DEPTH, seed=SEED, specialize=spec), threshold, n0)
    st = renderer.stats()
    assert st.specialized == spec
    assert st.samples == int(spp.sum())
    check_map(spp, err, threshold, n0, s)
    counts = np.unique(spp)
    assert len(counts) >= 2, counts
    off = np.zeros(spp.shape, dtype=bool)
    for n in counts:
        uni = renderer.render(harness.make_params(w, h, int(n), DEPTH, seed=SEED, specialize=spec))
        assert renderer.stats().specialized == spec
        m = spp == n
        close = np.isclose(rgb, uni, rtol=1e-5, atol=1e-7).all(axis=2)
        np.testing.assert_allclose(rgb[m], uni[m], rtol=1e-3, atol=1e-6, err_msg=f"pixels with {n} samples")
        off |= m & ~close
    # The moments kernel is compiled on its own, and on a B200 one pixel of noise_and_textures (specialised, 8415 pixels
    # at 64 samples) came out 4e-5 off, more than reordered fp32 sums of 64 non-negative terms can be (< 4e-6): one
    # sample's value differed.  At most one pixel in 2000 may do so, within 1e-3; every other pixel within 1e-5.
    assert off.sum() <= max(1, spp.size // 2000), f"{int(off.sum())} pixels beyond rtol 1e-5"
    return spp


@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("name", EQ_SCENES)
def test_adaptive_pixels_equal_uniform_renders(renderer, cfg, name, spec):
    upload(renderer, cfg, name)
    _equivalence(renderer, W, H, 64, 4, spec)


@pytest.mark.parametrize("spec", [0, 1])
def test_adaptive_equals_uniform_at_1080p(renderer, cfg, spec):
    upload(renderer, cfg, "cornell_box", 1920, 1080)
    spp = _equivalence(renderer, 1920, 1080, 1024, 16, spec)
    assert spp.max() == 1024


# ---------------------------------------------------------------------------
# Decisions recomputed on the host from the per-sample radiance
# ---------------------------------------------------------------------------
S_HOST, N0_HOST = 16, 2


def per_sample_y(renderer):
    """(16, H, W) y of every sample, from the 16 one-sample shares of a 16-spp frame."""
    ys = []
    for k in range(S_HOST):
        out = renderer.render(harness.make_params(W, H, S_HOST, DEPTH, seed=SEED, split=capi.RC_SPLIT_SAMPLES, rank=k, world=S_HOST))
        ys.append((S_HOST * out * out).mean(axis=2))
    return np.stack(ys)


@pytest.mark.parametrize("name", ["cornell_box", "three_balls", "noise_and_textures"])
def test_decisions_recomputed_on_the_host(renderer, cfg, name):
    upload(renderer, cfg, name)
    y = per_sample_y(renderer)
    e0 = host_err(y, N0_HOST)[0]
    threshold = float(np.median(e0[e0 > 0]))
    rgb, spp, err = renderer.render_adaptive(harness.make_params(W, H, S_HOST, DEPTH, seed=SEED), threshold, N0_HOST)
    check_map(spp, err, threshold, N0_HOST, S_HOST)
    pred, ambiguous = predict(y, threshold, N0_HOST, S_HOST)
    assert ambiguous.mean() < 0.01
    ok = ~ambiguous
    bad = ok & (spp != pred)
    assert not bad.any(), f"{int(bad.sum())} pixels: GPU {spp[bad][:5]} host {pred[bad][:5]}"
    assert len(np.unique(spp)) >= 3
    # the returned estimate is the host's at the GPU's n_p: within 1e-3 of it, or within its fp32 range
    e_host, lo, hi = (np.zeros_like(err) for _ in range(3))
    for n in np.unique(spp):
        m = spp == n
        for dst, src in zip((e_host, lo, hi), host_err(y, int(n))):
            dst[m] = src[m]
    off = np.abs(err - e_host) > np.maximum(1e-3 * e_host, hi - lo)
    assert not off.any(), f"{int(off.sum())} pixels: GPU {err[off][:4]} host {e_host[off][:4]} range {lo[off][:4]} {hi[off][:4]}"
    assert (np.abs(err - e_host) <= 1e-3 * e_host).mean() > 0.5
    # counterfactual: the same schedule from the wrong samples (rank k + 1) is told apart
    wrong, amb2 = predict(np.roll(y, -1, axis=0), threshold, N0_HOST, S_HOST)
    assert ((spp != wrong) & ~amb2).mean() > 0.02


@pytest.mark.parametrize("name", ["cornell_box", "three_balls", "noise_and_textures"])
def test_threshold_zero_stops_only_pixels_whose_samples_are_equal(renderer, cfg, name):
    upload(renderer, cfg, name)
    y = per_sample_y(renderer)
    rgb, spp, err = renderer.render_adaptive(harness.make_params(W, H, S_HOST, DEPTH, seed=SEED), 0.0, N0_HOST)
    check_map(spp, err, 0.0, N0_HOST, S_HOST)
    spread = np.abs(y[0] - y[1]) / np.maximum(y[0] + y[1], 1e-300)
    black = (y[0] == 0) & (y[1] == 0)
    differ = spread > 1e-2        # far above the rounding of the fp32 sums
    assert (spp[black] == N0_HOST).all() and (err[black] == 0).all()
    assert (spp[differ] == S_HOST).all()
    assert differ.any()
    if name == "cornell_box":   # black background: rays that leave the box bring back exactly 0
        assert black.any()


# ---------------------------------------------------------------------------
# Calibration: err is the spread of sqrt(mean y) over independent renders
# ---------------------------------------------------------------------------
# Measured on a B200 (1000 W): three_balls within [0.8, 1.25]; the Cornell box about 1.5: there a sample's radiance is heavy-tailed (a path that
# reaches the small light brings back 15 per channel, most bring back far less), and 64 such samples mostly
# underestimate their variance, so the estimate is optimistic by half.
CALIBRATION = {"three_balls": (0.8, 1.25), "cornell_box": (1.25, 1.75)}


@pytest.mark.parametrize("name", sorted(CALIBRATION))
def test_error_estimate_is_calibrated(renderer, cfg, name):
    upload(renderer, cfg, name)
    roots, errs = [], []
    for seed in range(16):
        rgb, spp, err = renderer.render_adaptive(harness.make_params(W, H, 64, DEPTH, seed=1000 + seed), 1e30, 64)
        assert (spp == 64).all()
        roots.append(np.sqrt((rgb * rgb).mean(axis=2)))
        errs.append(err)
    roots, errs = np.stack(roots), np.stack(errs)
    mu = (roots ** 2).mean(axis=0)
    m = (mu > 0.01) & (errs.mean(axis=0) > 0)   # (a pixel that sees only the light has no spread at all)
    ratio = roots.std(axis=0, ddof=1)[m] / errs.mean(axis=0)[m]
    med = float(np.median(ratio))
    lo, hi = CALIBRATION[name]
    assert lo <= med <= hi, med


# ---------------------------------------------------------------------------
# Limits, state and statistics
# ---------------------------------------------------------------------------
def test_huge_threshold_is_the_uniform_min_samples_render(renderer, cfg):
    upload(renderer, cfg, "three_balls")
    p = harness.make_params(W, H, 256, DEPTH, seed=SEED)
    rgb, spp, err = renderer.render_adaptive(p, 1e30, 8)
    st = renderer.stats()
    assert (spp == 8).all() and st.samples == 8 * W * H
    uni = renderer.render(harness.make_params(W, H, 8, DEPTH, seed=SEED))
    np.testing.assert_allclose(rgb, uni, rtol=1e-5, atol=1e-7)
    assert st.segments == renderer.stats().segments   # exactly the samples [0, 8) of every pixel were traced
    # one init, one megakernel + one test per round, one finalize: the rounds are launched whether or not a pixel is
    # still active (CTAs of inactive tiles leave at once), 8 .. 256 = 6 rounds
    assert st.kernel_launches == 2 + 2 * 6


def test_two_identical_calls_are_bit_identical(renderer, cfg):
    upload(renderer, cfg, "noise_and_textures")
    p = harness.make_params(W, H, 128, DEPTH, seed=SEED)
    first = renderer.render_adaptive(p, 0.02, 4)
    st = renderer.stats()
    n_rounds = int(math.log2(128 // 4)) + 1
    assert st.samples == int(first[1].sum())
    assert st.kernel_launches == 2 + 2 * n_rounds
    assert st.gpu_ms > 0 and st.segments >= st.samples
    again = renderer.render_adaptive(p, 0.02, 4)
    # another seed and size in between: nothing of it may show through
    renderer.render(harness.make_params(64, 48, 3, DEPTH, seed=99))
    renderer.render_adaptive(harness.make_params(120, 77, 32, DEPTH, seed=98), 0.01, 2)
    third = renderer.render_adaptive(p, 0.02, 4)
    for a, b, c in zip(first, again, third):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)) and np.array_equal(a.view(np.uint8), c.view(np.uint8))


def test_fixed_jitter_runs_on_the_precompiled_kernel(renderer, cfg):
    upload(renderer, cfg, "cornell_box")
    rgb, spp, err = renderer.render_adaptive(harness.make_params(W, H, 16, DEPTH, seed=SEED, fixed_jitter=1), 0.05, 4)
    uni = {n: renderer.render(harness.make_params(W, H, int(n), DEPTH, seed=SEED, fixed_jitter=1)) for n in np.unique(spp)}
    for n, img in uni.items():
        np.testing.assert_allclose(rgb[spp == n], img[spp == n], rtol=1e-5, atol=1e-7)


# ---------------------------------------------------------------------------
# Errors and cancellation
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["n0_1", "n0_above_s", "negative", "nan", "inf", "wavefront", "rejection", "rounds_7",
                                  "world_2", "spec_fixed_jitter"])
def test_unsupported_inputs_are_rejected(renderer, cfg, case):
    upload(renderer, cfg, "cornell_box")
    kw, n0, thr = {}, 4, 0.01
    if case == "n0_1":
        n0 = 1
    elif case == "n0_above_s":
        n0 = 17
    elif case == "negative":
        thr = -1e-3
    elif case == "nan":
        thr = float("nan")
    elif case == "inf":
        thr = float("inf")
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
        renderer.render_adaptive(harness.make_params(W, H, 16, DEPTH, seed=SEED, **kw), thr, n0)
    assert e.value.status == capi.RC_ERR_INVALID


def test_null_arguments_on_a_live_context(renderer, cfg):
    upload(renderer, cfg, "cornell_box")
    lib = renderer.lib
    p = harness.make_params(W, H, 8, DEPTH, seed=SEED)
    a = capi.rc_adaptive(min_samples=2, threshold=0.01)
    rgb = np.empty((H, W, 3))
    ptr = rgb.ctypes.data_as(C.POINTER(C.c_double))
    assert lib.rc_render_adaptive(renderer.ctx, None, C.byref(a), ptr, None, None, None) == capi.RC_ERR_INVALID
    assert lib.rc_render_adaptive(renderer.ctx, C.byref(p), None, ptr, None, None, None) == capi.RC_ERR_INVALID
    assert lib.rc_render_adaptive(renderer.ctx, C.byref(p), C.byref(a), None, None, None, None) == capi.RC_ERR_INVALID
    # out_spp and out_err may be NULL
    assert lib.rc_render_adaptive(renderer.ctx, C.byref(p), C.byref(a), ptr, None, None, None) == capi.RC_OK
    full = renderer.render_adaptive(p, 0.01, 2)
    assert np.array_equal(rgb, full[0])
    assert renderer.stats().samples == int(full[1].sum())


def test_cancel_flag_set_on_entry(renderer, cfg):
    upload(renderer, cfg, "cornell_box")
    flag = C.c_int32(1)
    with pytest.raises(capi.RacerCudaError) as e:
        renderer.render_adaptive(harness.make_params(W, H, 16, DEPTH, seed=SEED), 0.01, 2, cancel=flag)
    assert e.value.status == capi.RC_ERR_CANCELLED
    # a flag that stays down: the relayed rounds give the same render as a call without one
    flag.value = 0
    with_flag = renderer.render_adaptive(harness.make_params(W, H, 16, DEPTH, seed=SEED), 0.01, 2, cancel=flag)
    without = renderer.render_adaptive(harness.make_params(W, H, 16, DEPTH, seed=SEED), 0.01, 2)
    for a, b in zip(with_flag, without):
        assert np.array_equal(a, b)


# ---------------------------------------------------------------------------
# The C++ host
# ---------------------------------------------------------------------------
def test_racer_render_adaptive_png_equals_the_harness_path(racer_render, tmp_path, cfg, renderer):  # noqa: F811
    w, h, spp_max = 96, 64, 64
    job = harness.prepare_job(scene_path("cornell_box"), cfg, w, h)
    renderer.upload(job)
    rgb, spp, _ = renderer.render_adaptive(harness.make_params(w, h, spp_max, cfg.render.max_depth, seed=5, specialize=2), 0.01, 8)
    want = renderer.postprocess(job.tone_map, rgb)[0]
    assert len(np.unique(spp)) >= 2
    common = ["--scene", scene_path("cornell_box"), "--width", str(w), "--height", str(h), "--samples", str(spp_max), "--seed", "5"]
    out = tmp_path / "flags.png"
    r = run(racer_render, "--config", CONFIG, *common, "--adaptive", "0.01", "--min-samples", "8", "--out", str(out))
    assert np.array_equal(read_png(out), want)
    assert "(%d samples," % int(spp.sum()) in r.stdout
    cfg_file = tmp_path / "config.yml"
    cfg_file.write_text(open(CONFIG).read() + "gpu:\n  adaptive:\n    threshold: 0.01\n    min_samples: 8\n")
    out = tmp_path / "block.png"
    r = run(racer_render, "--config", str(cfg_file), *common, "--out", str(out))
    assert np.array_equal(read_png(out), want)
    assert "(%d samples," % int(spp.sum()) in r.stdout
