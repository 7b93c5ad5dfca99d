"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU
oracle on the same seeded inputs (SURVEY §8(c)).

Tolerances (north_star): primary-hit object ids bit-exact; hit t and normals
within 1e-5 relative; converged images PSNR >= 40 dB.  Per-sample streams are
shared with the oracle (Philox), so low-spp images must also agree almost
pixel for pixel: the only differences are paths whose branch decisions flip
under fp32 rounding.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import SCENES, SCENES_X, scene_path
from racer_tracer_b200 import capi, harness

pytestmark = pytest.mark.gpu

T_REL = 1e-5


def psnr(a, b):
    a = np.clip(a, 0.0, 1.0)
    b = np.clip(b, 0.0, 1.0)
    mse = float(((a - b) ** 2).mean())
    return 99.0 if mse == 0 else 10.0 * np.log10(1.0 / mse)


def display(oracle, job, img):
    """gamma'd image -> tone-mapped, clamped image (what the window shows)."""
    return np.clip(np.nan_to_num(oracle.tone_map(job.tone_map, img)), 0.0, 1.0)


def job_for(name, cfg, w, h, use_bvh=None):
    return harness.prepare_job(scene_path(name), cfg, w, h, seed=0, use_bvh=use_bvh)


def ambiguous_mask(oracle, job, p):
    """Pixels whose primary hit changes when every ray is translated by an
    fp32-sized amount (1e-6 of the viewing distance).  There the f64 answer is
    decided by an exact tie or a silhouette closer than fp32 can resolve (Q13:
    'exact ties are undefined'); everywhere else ids must be bit-exact."""
    import copy
    base = oracle.primary_aov(job, p)[0]
    cam = job.camera
    org = np.array(list(cam.origin))
    dist = np.linalg.norm(np.array(list(cam.horizontal))) / max(cam.viewport_width, 1e-9) if cam.viewport_width else 1.0
    delta = 1e-6 * (np.abs(org).max() + cam.focus_distance * 0 + np.linalg.norm(org) + 1.0)
    mask = np.zeros(base.shape, dtype=bool)
    right, up = np.array(list(cam.right)), np.array(list(cam.up))
    for sx, sy in ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (-1, -1)):
        j2 = copy.copy(job)
        c2 = capi.rc_camera.from_buffer_copy(cam)
        shift = delta * (sx * right + sy * up)
        c2.origin[:] = list(org + shift)
        c2.upper_left_corner[:] = list(np.array(list(cam.upper_left_corner)) + shift)
        j2.camera = c2
        mask |= oracle.primary_aov(j2, p)[0] != base
    return mask


@pytest.mark.parametrize("name", SCENES_X)
def test_primary_aov_f64_is_bit_exact(renderer, oracle, cfg, name):
    """precision=64: the reference's f64 operation order on the GPU.  ids, t and
    normals equal the CPU restatement bit for bit, ties included."""
    w, h = 600, 600
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, 1, 20, fixed_jitter=1)
    ids, t, nrm, pt = renderer.primary_aov(p, 64)
    oids, ot, onrm, opt = oracle.primary_aov(job, p)
    assert np.array_equal(ids, oids), f"{(ids != oids).sum()} primary-hit ids differ"
    assert (oids != 0).any()
    assert np.array_equal(t, ot)
    assert np.array_equal(nrm, onrm)
    assert np.array_equal(pt, opt)


@pytest.mark.parametrize("name", SCENES_X)
def test_primary_aov_fp32_matches_oracle(renderer, oracle, cfg, name):
    """precision=32: the renderer's own fp32 ray-gen + closest hit.  ids are
    bit-exact wherever the f64 answer is stable under an fp32-sized shift of the
    rays; hit t and normals are within 1e-5 relative (north_star) except for a
    handful of grazing pixels where the fp32 RAY (not the intersector) cannot
    carry that precision — bounded and counted below."""
    w, h = 600, 600
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, 1, 20, fixed_jitter=1)
    ids, t, nrm, pt = renderer.primary_aov(p, 32)
    oids, ot, onrm, opt = oracle.primary_aov(job, p)
    amb = ambiguous_mask(oracle, job, p)
    assert amb.mean() < 2e-3, f"{amb.sum()} ambiguous pixels"
    bad = (ids != oids) & ~amb
    assert not bad.any(), f"{bad.sum()} primary-hit ids differ outside the {amb.sum()} tie/silhouette pixels"
    hit = (oids != 0) & (ids == oids)
    rel = np.abs(t[hit] - ot[hit]) / np.abs(ot[hit])
    nerr = np.abs(nrm[hit] - onrm[hit]).max(axis=1)
    print(f"{name}: ambiguous {amb.sum()}, id diffs inside them {(ids != oids).sum()}, "
          f"t rel max {rel.max():.2e} frac>1e-5 {(rel > T_REL).mean():.2e}, "
          f"normal max {nerr.max():.2e} frac>1e-5 {(nerr > T_REL).mean():.2e}")
    assert (rel > T_REL).mean() < 5e-4 and rel.max() < 5e-4
    assert (nerr > T_REL).mean() < 5e-3 and nerr.max() < 5e-3
    assert np.all(t[ids == 0] == np.finfo(np.float64).max)
    scale = np.maximum(np.abs(opt[hit]).max(axis=1), 1.0)
    assert (np.abs(pt[hit] - opt[hit]).max(axis=1) / scale).max() <= 2e-4   # one fp32 ulp at |p| ~ 1000 is 6e-5


@pytest.mark.parametrize("name", SCENES_X)
@pytest.mark.parametrize("sampler", [capi.RC_SAMPLER_DIRECT, capi.RC_SAMPLER_REJECTION])
def test_same_stream_image_matches_oracle(renderer, oracle, cfg, name, sampler):
    """GPU fp32 and oracle f64 consume identical Philox streams: images agree
    except where an fp32 rounding flips a branch on some path."""
    w, h, spp = 160, 120, 8
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, spp, 20, seed=3, sampler=sampler)
    img = renderer.render(p)
    ref = oracle.render(job, p)
    assert np.isfinite(img).all()
    err = np.abs(img - ref).max(axis=2)
    frac = float((err > 2e-3).mean())
    assert frac < 0.03, f"{name}: {frac:.2%} of pixels differ (> 2e-3) from the same-stream oracle image"
    assert np.median(err) < 1e-5
    assert psnr(display(oracle, job, img), display(oracle, job, ref)) > 38.0


@pytest.mark.parametrize("name,spp", [("cornell_box", 32768), ("three_balls", 4096), ("emissive", 8192)])
def test_converged_image_psnr_independent_streams(renderer, oracle, cfg, name, spp):
    """High-spp GPU image vs high-spp oracle image drawn from an INDEPENDENT
    sequential stream with the reference's rejection samplers: >= 40 dB on the
    displayed image (north_star), with the Monte-Carlo noise floor printed."""
    w, h = 64, 48
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, spp, 20, seed=11)
    gpu = renderer.render(p)
    # Q1: u jitter is per pixel, so the oracle must share the per-pixel jitter
    # stream (Philox) to converge to the same image; all per-sample draws are
    # independent (different seed).
    po = harness.make_params(w, h, spp, 20, seed=11, sampler=capi.RC_SAMPLER_REJECTION)
    ref_a = oracle.render(job, po, sample_begin=spp, sample_count=spp)       # disjoint sample indices
    ref_b = oracle.render(job, po, sample_begin=2 * spp, sample_count=spp)
    d = lambda im: display(oracle, job, im)
    noise_floor = psnr(d(ref_a), d(ref_b))
    got = psnr(d(gpu), d(ref_a))
    print(f"{name}: PSNR(gpu, oracle) = {got:.1f} dB, PSNR(oracle, oracle') = {noise_floor:.1f} dB")
    assert got >= 40.0, "north_star: PSNR >= 40 dB against the reference's converged image"
    assert got >= noise_floor - 1.0, "the GPU image is further from the oracle than Monte-Carlo noise explains"


@pytest.mark.parametrize("name", SCENES_X)
def test_wavefront_traces_the_same_paths_as_the_megakernel(renderer, oracle, cfg, name):
    """Both variants share ray-gen, RNG streams, intersection and shading code; only the
    fp32 summation order of the per-pixel sum differs (chunks of 32 samples + atomics)."""
    w, h, spp = 150, 90, 40      # ragged tiles, spp not a multiple of the 32-sample chunk
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    a = renderer.render(harness.make_params(w, h, spp, 20, seed=5, variant=capi.RC_VARIANT_MEGAKERNEL))
    b = renderer.render(harness.make_params(w, h, spp, 20, seed=5, variant=capi.RC_VARIANT_WAVEFRONT))
    assert np.isfinite(b).all()
    # same functions, but compiled into different kernels: FMA contraction differs by an ulp here and
    # there, and a path that sits on a checker edge or a reflect/refract threshold may flip
    err = np.abs(a - b).max(axis=2)
    assert np.median(err) < 1e-6 and np.quantile(err, 0.99) < 2e-4, f"max diff {err.max():.3e}"
    assert float((err > 2e-3).mean()) < 0.005
    ref = oracle.render(job, harness.make_params(w, h, spp, 20, seed=5))
    # (Random: 484 spheres, lens and motion blur — more paths sit on an fp32 decision than in the small scenes)
    assert float((np.abs(b - ref).max(axis=2) > 2e-3).mean()) < (0.045 if name == "random" else 0.03)


def test_wavefront_partitions_and_depth_edge_cases(renderer, cfg):
    import torch
    w, h, spp = 100, 75, 33
    job = job_for("emissive", cfg, w, h)
    renderer.upload(job)
    wf = capi.RC_VARIANT_WAVEFRONT
    whole = _accumulate(renderer, harness.make_params(w, h, spp, 20, seed=2, variant=wf))
    for split in (capi.RC_SPLIT_TILES, capi.RC_SPLIT_SAMPLES):
        parts = [_accumulate(renderer, harness.make_params(w, h, spp, 20, seed=2, variant=wf, rank=r, world=3, split=split))
                 for r in range(3)]
        assert torch.allclose(torch.stack(parts).sum(dim=0), whole, rtol=1e-5, atol=1e-5)
    img0 = renderer.render(harness.make_params(w, h, 3, 0, seed=1, variant=wf))
    assert np.array_equal(img0, np.ones_like(img0))


def test_postprocess_matches_oracle_bytes(renderer, oracle, cfg):
    rng = np.random.default_rng(5)
    img = rng.random((37, 53, 3)) * 1.6
    img[0, 0] = [0.0, 0.0, 0.0]      # Reinhard 0/0 -> NaN -> 0
    img[0, 1] = [1.5, 0.5, 0.2]      # channel overflow bleeds into its neighbour (Q9)
    for node in ("None", {"Reinhard": {"default": True}}, {"Hable": {"default": True}},
                 {"Aces": {"default": True}}, {"Reinhard": {"max_white": 4.0}}):
        tm = harness.make_tone_map(harness._lower_keys(node) if isinstance(node, dict) else node)
        rgba, mapped = renderer.postprocess(tm, img)
        ref = oracle.tone_map(tm, img)
        assert np.allclose(mapped, ref, rtol=1e-12, atol=1e-14, equal_nan=True)
        ref_q = oracle.quantise_rgba(ref)
        same = (rgba == ref_q).all(axis=2)
        # a value within 1e-12 of a quantisation boundary may round differently under FMA
        assert same.mean() > 0.999
    assert tuple(oracle.quantise_rgba(np.array([[[1.5, 0.5, 0.2]]]))[0, 0]) == (0x7E, 0x7F, 0x33, 0xFF)


def _accumulate(renderer, p):
    import torch
    acc = torch.zeros(p.height * p.width * 3, dtype=torch.float32, device="cuda:0")
    renderer.set_stream(torch.cuda.current_stream().cuda_stream)
    renderer.render_accumulate(p, acc.data_ptr())
    torch.cuda.synchronize()
    return acc


def test_partitions_cover_the_image_exactly(renderer, cfg):
    """Tile split: the union over ranks equals the single-rank render bit for
    bit (every pixel is computed by exactly one rank).  Sample split: the sum
    over ranks equals the whole within fp32 summation order."""
    import torch
    w, h, spp = 333, 201, 12   # ragged: not a multiple of the 16x8 tile
    job = job_for("three_balls", cfg, w, h)
    renderer.upload(job)
    whole = _accumulate(renderer, harness.make_params(w, h, spp, 20, seed=2))
    for world in (2, 3, 8):
        parts = [_accumulate(renderer, harness.make_params(w, h, spp, 20, seed=2, rank=r, world=world))
                 for r in range(world)]
        nz = torch.stack([(q != 0).reshape(-1, 3).any(dim=1) for q in parts]).sum(dim=0)
        assert int(nz.max()) <= 1, "a pixel was traced by two ranks"
        assert torch.equal(torch.stack(parts).sum(dim=0), whole)
        parts = [_accumulate(renderer, harness.make_params(w, h, spp, 20, seed=2, rank=r, world=world,
                                                            split=capi.RC_SPLIT_SAMPLES))
                 for r in range(world)]
        s = torch.stack(parts).sum(dim=0)
        assert torch.allclose(s, whole, rtol=1e-5, atol=1e-5)


def test_sliced_tiles_equal_unsliced(renderer, cfg):
    """Few tiles per device (a multi-GPU share, or a small image): each tile's sample range is cut
    into several CTAs whose partial sums are added in slice order.  Same samples, deterministic,
    equal to the unsliced render up to fp32 summation order."""
    w, h, spp = 128, 96, 256          # 96 tiles -> sliced
    job = job_for("cornell_box", cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, spp, 20, seed=3)
    a = renderer.render(p)
    assert np.array_equal(a, renderer.render(p))
    os.environ["RC_SLICES"] = "1"
    try:
        b = renderer.render(p)
    finally:
        del os.environ["RC_SLICES"]
    assert np.allclose(a, b, rtol=1e-5, atol=1e-6)
    assert renderer.stats().kernel_launches == 1
    renderer.render(p)
    assert renderer.stats().kernel_launches == 2     # sliced megakernel + reduce_slices_kernel


def test_render_is_deterministic_and_seeded(renderer, cfg):
    w, h = 128, 96
    job = job_for("cornell_box", cfg, w, h)
    renderer.upload(job)
    a = renderer.render(harness.make_params(w, h, 8, 20, seed=1))
    b = renderer.render(harness.make_params(w, h, 8, 20, seed=1))
    c = renderer.render(harness.make_params(w, h, 8, 20, seed=2))
    assert np.array_equal(a, b)
    assert not np.array_equal(a, c)


def test_depth_zero_is_white_and_depth_one_is_emission_only(renderer, oracle, cfg):
    w, h = 64, 64
    job = job_for("cornell_box", cfg, w, h)
    renderer.upload(job)
    img0 = renderer.render(harness.make_params(w, h, 4, 0, seed=1))
    assert np.array_equal(img0, np.ones_like(img0))     # renderer.rs:48-56
    p1 = harness.make_params(w, h, 4, 1, seed=1)
    img1 = renderer.render(p1)
    assert np.allclose(img1, oracle.render(job, p1), atol=1e-6)


def test_cancel_semantics(renderer, cfg):
    w, h = 64, 64
    job = job_for("cornell_box", cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, 64, 20, seed=1)
    flag = C.c_int32(1)
    with pytest.raises(capi.RacerCudaError) as e:      # cancelled before start: TracerError::CancelEvent
        renderer.render(p, cancel=flag)
    assert e.value.status == capi.RC_ERR_CANCELLED
    flag = C.c_int32(0)
    img = renderer.render(p, cancel=flag)              # polled between 32-sample passes, flag not set
    assert np.allclose(img, renderer.render(p), rtol=1e-5, atol=1e-6)   # same samples, fp32 sum order differs


def test_errors_are_loud(renderer, cfg):
    lib = renderer.lib
    ctx = C.c_void_p()
    capi.check(lib, lib.rc_create(None, 1, C.byref(ctx)))
    p = harness.make_params(64, 64, 1, 1)
    out = np.zeros((64, 64, 3))
    st = lib.rc_render(ctx, C.byref(p), out.ctypes.data_as(C.POINTER(C.c_double)), None)
    assert st == capi.RC_ERR_STATE and b"upload" in lib.rc_last_error()
    bad = harness.make_params(1, 64, 1, 1)
    assert lib.rc_render(ctx, C.byref(bad), out.ctypes.data_as(C.POINTER(C.c_double)), None) == capi.RC_ERR_INVALID
    lib.rc_destroy(ctx)


def test_full_size_properties_cornell(renderer, cfg):
    """BASELINE size (1920x1080), size-independent properties: linearity over
    sample ranges and seed determinism of the accumulation buffer."""
    import torch
    w, h = 1920, 1080
    job = job_for("cornell_box", cfg, w, h)
    renderer.upload(job)
    a = _accumulate(renderer, harness.make_params(w, h, 16, 20, seed=9))
    p_lo = harness.make_params(w, h, 16, 20, seed=9, rank=0, world=2, split=capi.RC_SPLIT_SAMPLES)
    p_hi = harness.make_params(w, h, 16, 20, seed=9, rank=1, world=2, split=capi.RC_SPLIT_SAMPLES)
    s = _accumulate(renderer, p_lo) + _accumulate(renderer, p_hi)
    assert torch.allclose(s, a, rtol=1e-5, atol=1e-5)
    assert torch.isfinite(a).all() and float(a.min()) >= 0.0
    img = a.reshape(h, w, 3)
    # outside the box the background is black (cornell_box.yml background SolidColor 0)
    assert float(img[:, :300].abs().max()) == 0.0 and float(img[:, -300:].abs().max()) == 0.0
    st = renderer.stats()
    assert st.segments > st.samples  # more than one segment per sample inside the box


def test_two_devices_in_one_context(renderer, cfg):
    """rc_create over two devices (the single-process form the Rust host uses): tile split
    gathers disjoint tiles peer-to-peer, sample split sums partial buffers with ncclReduce."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    w, h, spp = 333, 201, 24
    job = job_for("three_balls", cfg, w, h)
    renderer.upload(job)
    one = renderer.render(harness.make_params(w, h, spp, 20, seed=4))
    r2 = harness.CudaRenderer([0, 1])
    try:
        r2.upload(job)
        two = r2.render(harness.make_params(w, h, spp, 20, seed=4, split=capi.RC_SPLIT_TILES))
        assert np.array_equal(one, two)               # x + 0 = x: the gather is exact
        assert r2.stats().n_devices == 2
        two_s = r2.render(harness.make_params(w, h, spp, 20, seed=4, split=capi.RC_SPLIT_SAMPLES))
        assert np.allclose(one, two_s, rtol=1e-5, atol=1e-6)
        # Shares that leave buffers unwritten, each right after a full render at the same size.  A 1-spp sample split:
        # sample 0 goes to device 1 and device 0's share is empty, so the reduce must add zeros, not old sums.
        from test_gpu_shares import tile_mask
        one1 = renderer.render(harness.make_params(w, h, 1, 20, seed=6))
        r2.render(harness.make_params(w, h, spp, 20, seed=5, split=capi.RC_SPLIT_SAMPLES))
        assert np.array_equal(r2.render(harness.make_params(w, h, 1, 20, seed=6, split=capi.RC_SPLIT_SAMPLES)), one1)
        # rank 1 of world 2 on the two-device context: participants 2 and 3 of 4.  Tile split: tiles k mod 4 in {2, 3}
        # and zeros elsewhere; sample split at 1 spp: participant 3 traces sample 0, participant 2 nothing.
        own = tile_mask(w, h, 2, 4) | tile_mask(w, h, 3, 4)
        r2.render(harness.make_params(w, h, spp, 20, seed=5))
        share = r2.render(harness.make_params(w, h, spp, 20, seed=4, rank=1, world=2))
        assert (share[~own] == 0.0).all() and np.array_equal(share[own], one[own])
        assert r2.stats().samples == int(own.sum()) * spp
        r2.render(harness.make_params(w, h, spp, 20, seed=5))
        share = r2.render(harness.make_params(w, h, 1, 20, seed=6, rank=1, world=2, split=capi.RC_SPLIT_SAMPLES))
        assert np.array_equal(share, one1) and r2.stats().samples == w * h
        wf = r2.render(harness.make_params(w, h, spp, 20, seed=4, variant=capi.RC_VARIANT_WAVEFRONT))
        # a different kernel: FMA contraction differs by an ulp here and there and a path on a reflect / refract
        # threshold may flip (one pixel of 66 933 did, measured) — the same criterion as the one-device comparison
        err = np.abs(one - wf).max(axis=2)
        assert np.median(err) < 1e-6 and np.quantile(err, 0.99) < 2e-4 and float((err > 2e-3).mean()) < 0.005
        # Back-to-back asynchronous frames into ONE buffer with no host synchronisation in between: the second
        # device's kernel of frame k + 1 must not store into the buffer before device 0's stream has re-zeroed it
        # and finalised frame k (the fork at the start of every frame orders the other devices' streams after
        # device 0's; the join at its end orders device 0's after theirs).
        import torch
        torch.cuda.set_device(0)
        stream = torch.cuda.current_stream()
        r2.set_stream(stream.cuda_stream)
        n = w * h * 3
        acc = torch.zeros(n, dtype=torch.float32, device="cuda:0")
        outs = [torch.empty(n, dtype=torch.float32, device="cuda:0") for _ in range(4)]
        seeds = (11, 12, 13, 14)
        for seed, out in zip(seeds, outs):
            acc.zero_()
            r2.render_accumulate(harness.make_params(w, h, spp, 20, seed=seed, split=capi.RC_SPLIT_TILES), acc.data_ptr())
            r2.finalize(acc.data_ptr(), w, h, spp, out.data_ptr())
        torch.cuda.synchronize()
        for seed, out in zip(seeds, outs):
            want = renderer.render(harness.make_params(w, h, spp, 20, seed=seed)).astype(np.float32)
            got = out.cpu().numpy().reshape(h, w, 3)
            assert np.allclose(got, want, rtol=3e-7, atol=1e-7), (seed, np.abs(got - want).max())
    finally:
        r2.close()


def test_scene_specialised_kernel_matches_the_generic_one(renderer, cfg):
    """rc_params.specialize = 1: the scene compiled into the megakernel with NVRTC (constants as
    immediates, unused material code removed) traces the same paths as the precompiled kernel."""
    w, h, spp = 200, 120, 24
    for name in ("cornell_box", "three_balls", "emissive"):
        job = job_for(name, cfg, w, h)
        renderer.upload(job)
        a = renderer.render(harness.make_params(w, h, spp, 20, seed=6))
        b = renderer.render(harness.make_params(w, h, spp, 20, seed=6, specialize=1))
        err = np.abs(a - b).max(axis=2)
        assert np.median(err) < 1e-6 and np.quantile(err, 0.99) < 2e-4, f"{name}: max diff {err.max():.3e}"
        assert float((err > 2e-3).mean()) < 0.005
    # a second upload of the same scene hits the per-scene cache (no recompilation)
    import time
    renderer.upload(job)
    t0 = time.perf_counter()
    renderer.render(harness.make_params(w, h, 1, 20, seed=6, specialize=1))
    assert time.perf_counter() - t0 < 0.5


@pytest.mark.parametrize("name,w,h", [("cornell_box", 600, 600), ("three_balls", 610, 330)])
def test_preview_renderer_matches_oracle(renderer, oracle, cfg, name, w, h):
    """rc_render_preview = CpuRendererScaled (src/renderer/cpu_scaled.rs): one colour per scale x scale
    block from config.preview's samples / depth, upscaled; same Philox streams as the oracle's restatement.
    610x330: the last tile column has a remainder, whose pixels beyond the last whole block stay 0."""
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    sw, sh = harness.preview_scales(cfg, w, h)
    assert (sw, sh) == ((4, 4) if w == 600 else (1, 3))     # 60 % 4 == 0; 61 is prime, 33 -> 3
    p = harness.make_params(w, h, cfg.preview.samples, cfg.preview.max_depth, seed=2)
    img = renderer.render_preview(p, sw, sh)
    ref = oracle.render_preview(job, p, sw, sh)
    assert img.shape == (h, w, 3) and np.isfinite(img).all()
    # constant over every block
    bw, bh = w // sw, h // sh
    blocks = img[:bh * sh, :bw * sw].reshape(bh, sh, bw, sw, 3)
    assert np.array_equal(blocks, np.broadcast_to(blocks[:, :1, :, :1], blocks.shape))
    # beyond the last whole block: zero, on both sides
    assert not img[bh * sh:].any() and not img[:, bw * sw:].any()
    assert not ref[bh * sh:].any() and not ref[:, bw * sw:].any()
    err = np.abs(img - ref).max(axis=2)
    assert float((err > 2e-3).mean()) < 0.03 and np.median(err) < 1e-5
    st = renderer.stats()
    assert st.samples == bw * bh * cfg.preview.samples
    # scale 1 == the full renderer's pixels (same u/v, same streams)
    q = harness.make_params(64, 48, 8, 10, seed=2)
    small = job_for(name, cfg, 64, 48)
    renderer.upload(small)
    assert np.allclose(renderer.render_preview(q, 1, 1), renderer.render(q), rtol=1e-6, atol=1e-7)
    with pytest.raises(capi.RacerCudaError):
        renderer.render_preview(q, 0, 1)


def check_tree(nodes, order, n_prims, aabbs):
    """Structural validity of a pre-order BVH: children follow the pre-order rule, every primitive sits in
    exactly one leaf, every box contains its children's boxes (leaves: the object's stored Aabb)."""
    assert sorted(order.tolist()) == list(range(n_prims))
    seen = np.zeros(n_prims, dtype=int)

    def visit(i):
        nd = nodes[i]
        lo, hi = np.array(list(nd.bmin)), np.array(list(nd.bmax))
        if nd.left < 0:
            first, count = ~nd.left, nd.right
            seen[first:first + count] += 1
            for q in range(first, first + count):
                assert np.array_equal(lo, aabbs[order[q], :3]) and np.array_equal(hi, aabbs[order[q], 3:])
            return lo, hi, 1
        assert nd.left == i + 1
        llo, lhi, ln = visit(nd.left)
        assert nd.right == i + 1 + ln
        rlo, rhi, rn = visit(nd.right)
        assert np.array_equal(lo, np.minimum(llo, rlo)) and np.array_equal(hi, np.maximum(lhi, rhi))   # aabb.rs:95-114
        return lo, hi, 1 + ln + rn
    import sys
    sys.setrecursionlimit(10000)
    _, _, total = visit(0)
    assert total == len(nodes) and (seen == 1).all()


@pytest.mark.parametrize("name", ["random", "sandbox_boxes", "clown", "cornell_box"])
def test_gpu_lbvh_build_and_parity(renderer, oracle, cfg, name):
    """rc_build_lbvh: the BVH built on the GPU (Morton codes + Karras topology) is a valid tree over the
    top-level objects, and tracing it gives what the oracle gets when it walks THE SAME tree (rc_get_bvh):
    f64 primary hits bit for bit, same-stream images within the fp32 tolerance.  Against the host-built
    tree the closest hit is the same wherever it is not an exact tie."""
    w, h = 320, 240
    job = job_for(name, cfg, w, h)
    renderer.upload(job)
    p = harness.make_params(w, h, 1, 20, fixed_jitter=1)
    host_ids = renderer.primary_aov(p, 64)[0]
    renderer.build_lbvh()
    nodes, order = renderer.get_bvh(job.scene.c.n_prims)
    n_obj = len(set((job.scene.np["prim_id"] >> 3).tolist()))
    assert len(nodes) == 2 * n_obj - 1
    check_tree(nodes, order, job.scene.c.n_prims, job.scene.np["prim_aabb"])
    same_tree = harness.with_bvh(job, nodes, order)
    ids, t, nrm, pt = renderer.primary_aov(p, 64)
    oids, ot, onrm, opt = oracle.primary_aov(same_tree, p)
    assert np.array_equal(ids, oids) and np.array_equal(t, ot) and np.array_equal(nrm, onrm) and np.array_equal(pt, opt)
    assert (ids != host_ids).mean() < 2e-3                       # exact ties only (cornell's 45-degree edges)
    ids32 = renderer.primary_aov(p, 32)[0]
    assert (ids32 != oids).mean() < 2e-3
    q = harness.make_params(w, h, 8, 20, seed=4)
    img = renderer.render(q)
    ref = oracle.render(same_tree, q)
    err = np.abs(img - ref).max(axis=2)
    assert float((err > 2e-3).mean()) < 0.03 and np.median(err) < 1e-5
    # building twice is idempotent (the second build sorts the already sorted objects)
    renderer.build_lbvh()
    nodes2, order2 = renderer.get_bvh(job.scene.c.n_prims)
    assert np.array_equal(order, order2) and len(nodes2) == len(nodes)
    assert np.array_equal(renderer.primary_aov(p, 64)[0], ids)


def test_library_resplits_a_median_tree_by_sah(renderer, oracle, cfg, monkeypatch):
    """A host that passes the reference's own median-split tree (Node::build, src/bvh_node.rs:31-82) — what the Rust
    shim does — gets the surface-area-heuristic tree anyway: rc_upload_scene re-splits the same leaves when that
    lowers the expected number of box tests by 10 % or more (instance-free scenes, RC_KEEP_TREE=1 keeps the tree).
    Same leaves, same primitives, another tree: the f64 primary hits are those of the oracle on the tree passed
    (ties resolve by primitive order, which the re-split keeps consistent), the image is the same image."""
    def tree_cost(nodes):
        area = lambda n: 2.0 * sum((n.bmax[a] - n.bmin[a]) * (n.bmax[(a + 1) % 3] - n.bmin[(a + 1) % 3]) for a in range(3))
        return sum(area(n) for n in nodes) / area(nodes[0])
    monkeypatch.setattr(harness, "SAH_MIN_OBJECTS", 10 ** 9)      # the harness builds the median tree, like the reference
    w, h = 320, 240
    job = job_for("random", cfg, w, h)
    p = harness.make_params(w, h, 1, 20, fixed_jitter=1)
    q = harness.make_params(w, h, 8, 20, seed=4)
    monkeypatch.setenv("RC_KEEP_TREE", "1")
    renderer.upload(job)
    kept, kept_order = renderer.get_bvh(job.scene.c.n_prims)
    ids_kept = renderer.primary_aov(p, 64)[0]
    img_kept = renderer.render(q)
    assert np.array_equal(ids_kept, oracle.primary_aov(job, p)[0])
    monkeypatch.delenv("RC_KEEP_TREE")
    renderer.upload(job)
    nodes, order = renderer.get_bvh(job.scene.c.n_prims)
    assert len(nodes) == len(kept)
    check_tree(nodes, order, job.scene.c.n_prims, job.scene.np["prim_aabb"])
    assert tree_cost(nodes) < 0.9 * tree_cost(kept), (tree_cost(nodes), tree_cost(kept))
    ids = renderer.primary_aov(p, 64)[0]
    assert (ids != ids_kept).mean() < 1e-4                      # (exact ties between different objects only)
    img = renderer.render(q)
    err = np.abs(img - img_kept).max(axis=2)
    assert float((err > 2e-3).mean()) < 1e-3 and np.median(err) == 0.0


def test_processes_store_their_tiles_into_one_shared_frame(cfg):
    """One process per GPU (the bench contract): rc_render_tiles_into stores every rank's tiles into rank 0's
    frame buffer, mapped with CUDA IPC — the tile-split gather happens inside the render kernel.  The frame is
    bit-identical to a single-GPU render."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29571", os.path.join(root, "tools", "ipc_tiles_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "IPC_TILES_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_instanced_scene_linear_path_equals_the_bvh_path(renderer, oracle, cfg):
    """The reference's default Sandbox scene (Cornell + two rotated, translated boxes) fits the linear modes:
    plain rectangles, then per instanced object the stored Aabb as cull volume (Aabb::hit verbatim, Q11/Q14)
    and its sides in the object's space.  Same primary hits and the same paths as the BVH traversal of the
    same scene, precompiled and scene-specialised."""
    w, h = 300, 300
    job = job_for("sandbox_boxes", cfg, w, h)
    p = harness.make_params(w, h, 1, 20, fixed_jitter=1)
    q = harness.make_params(w, h, 8, 20, seed=6)
    renderer.upload(job)
    ids_lin = renderer.primary_aov(p, 32)[0]
    img_lin = renderer.render(q)
    img_spec = renderer.render(harness.make_params(w, h, 8, 20, seed=6, specialize=1))
    os.environ["RC_SCENE_MODE"] = "smem"
    try:
        renderer.upload(job)
        ids_bvh = renderer.primary_aov(p, 32)[0]
        img_bvh = renderer.render(q)
        # the BVH paths' specialised kernel (kinds of primitive / material / wrapper compiled in or out)
        img_bvh_spec = renderer.render(harness.make_params(w, h, 8, 20, seed=6, specialize=1))
        assert renderer.stats().specialized == 1
    finally:
        del os.environ["RC_SCENE_MODE"]
    err = np.abs(img_bvh_spec - img_bvh).max(axis=2)
    assert np.median(err) < 1e-6 and float((err > 2e-3).mean()) < 0.01
    assert (ids_lin != ids_bvh).mean() < 1e-3          # exact ties only: the two paths order primitives differently
    for name, img in (("precompiled", img_lin), ("specialised", img_spec)):
        err = np.abs(img - img_bvh).max(axis=2)
        # different kernels: rounding differences flip a few long paths (measured: 0.01 % of the pixels)
        assert np.median(err) < 1e-6 and float((err > 2e-3).mean()) < 0.01, name
    ref = oracle.render(job, q)
    assert float((np.abs(img_spec - ref).max(axis=2) > 2e-3).mean()) < 0.01


def many_spheres_job(cfg, n, w, h, seed=5):
    """n small lambertian / metal spheres in a slab, no host BVH (n_nodes = 0), default sky."""
    rng = np.random.default_rng(seed)
    fs = harness.FlatScene()
    textures, materials, objects = [], [], {}
    for k in range(8):
        t = capi.rc_texture()
        t.type = capi.RC_TEX_SOLID
        t.color[:] = rng.uniform(0.2, 0.9, 3).tolist()
        textures.append(t)
        m = capi.rc_material()
        m.type, m.texture, m.param = (capi.RC_MAT_METAL if k == 7 else capi.RC_MAT_LAMBERTIAN), k, 0.1
        materials.append(m)
    centres = rng.uniform([-30, -8, -30], [30, 8, 30], size=(n, 3))
    radii = rng.uniform(0.15, 0.45, n)
    for i in range(n):
        c, r = centres[i].tolist(), float(radii[i])
        lo, hi = [c[a] - r for a in range(3)], [c[a] + r for a in range(3)]
        key = f"s{i:06d}"
        objects[key] = harness.TopObject(key, [harness.Prim(capi.RC_PRIM_SPHERE, c + [r, 0.0], i % 8, 0)], lo, hi, c)
    harness._flatten(fs, objects, textures, materials, [], [], use_bvh=False)
    fs.c.bg_type = capi.RC_BG_SKY
    fs.c.bg_a[:] = [1.0, 1.0, 1.0]
    fs.c.bg_b[:] = [0.5, 0.7, 1.0]
    cam = harness.make_camera({"vfov": 40.0, "aperture": 0.0, "focus_distance": 10.0, "pos": [0.0, 25.0, 70.0],
                               "look_at": [0.0, 0.0, 0.0]}, w, h)
    return harness.Job(fs, cam, harness.make_tone_map("none"), cfg, w, h)


def test_large_scene_gets_a_gpu_built_bvh(renderer, oracle, cfg):
    """9 000 spheres uploaded without nodes: too many for the linear loop, so rc_upload_scene builds the LBVH
    on the device — the multi-pass (global-memory) bitonic sort and the global-memory traversal mode, which
    the small scenes never reach.  Valid tree; f64 primary hits bit-exact against the oracle on the same tree;
    same-stream image within tolerance."""
    n, w, h = 9000, 200, 150
    job = many_spheres_job(cfg, n, w, h)
    assert job.scene.c.n_nodes == 0
    renderer.upload(job)
    nodes, order = renderer.get_bvh(n)
    assert len(nodes) == 2 * n - 1
    check_tree(nodes, order, n, job.scene.np["prim_aabb"])
    same_tree = harness.with_bvh(job, nodes, order)
    p = harness.make_params(w, h, 1, 20, fixed_jitter=1)
    ids, t, nrm, pt = renderer.primary_aov(p, 64)
    oids, ot, onrm, opt = oracle.primary_aov(same_tree, p)
    assert (oids != 0).mean() > 0.2
    assert np.array_equal(ids, oids) and np.array_equal(t, ot) and np.array_equal(nrm, onrm)
    assert (renderer.primary_aov(p, 32)[0] != oids).mean() < 2e-3
    q = harness.make_params(w, h, 4, 20, seed=2)
    img, ref = renderer.render(q), oracle.render(same_tree, q)
    err = np.abs(img - ref).max(axis=2)
    # thousands of sub-unit spheres seen from 70 units away: an fp32 rounding flips a secondary ray onto a
    # neighbouring sphere far more often than in the BASELINE scenes (7.7 % of the pixels at 4 spp, measured);
    # most pixels still agree to 1e-5 and the images agree in the mean
    assert float((err > 2e-3).mean()) < 0.12 and np.median(err) < 1e-5
    assert np.abs(img.mean(axis=(0, 1)) - ref.mean(axis=(0, 1))).max() < 2e-3


@pytest.mark.parametrize("name", ["cornell_box", "three_balls", "clown", "noise_and_textures", "sandbox_boxes"])
def test_tile_culling_changes_nothing(renderer, cfg, name):
    """Tiles whose primary rays cannot hit anything (frustum test against every primitive / object cull box)
    skip the intersection and add the background sample by sample: the image and the segment count are
    bit-identical to a render with the test switched off, precompiled and scene-specialised."""
    w, h, spp = 400, 225, 8
    job = job_for(name, cfg, w, h)
    if job.camera.lens_radius != 0.0:
        pytest.skip("culling needs a pinhole camera")
    renderer.upload(job)
    for spec in (0, 2):
        p = harness.make_params(w, h, spp, 20, seed=12, specialize=spec)
        a = renderer.render(p)
        seg_a = renderer.stats().segments
        os.environ["RC_NO_TILE_CULL"] = "1"
        try:
            b = renderer.render(p)
            seg_b = renderer.stats().segments
        finally:
            del os.environ["RC_NO_TILE_CULL"]
        assert np.array_equal(a, b) and seg_a == seg_b, (name, spec)
    # the preview renderer goes through the same test with scaled pixel coordinates
    sw, sh = harness.preview_scales(cfg, w, h)
    pv = harness.make_params(w, h, 8, 10, seed=3)
    a = renderer.render_preview(pv, sw, sh)
    os.environ["RC_NO_TILE_CULL"] = "1"
    try:
        b = renderer.render_preview(pv, sw, sh)
    finally:
        del os.environ["RC_NO_TILE_CULL"]
    assert np.array_equal(a, b)


@pytest.mark.gpu
def test_slab_pairs_trace_the_same_paths(renderer, oracle, cfg):
    """The specialised kernel tests two opposite walls as one rectangle (max of the two plane distances) when
    every ray starts between them (rc_spec.cuh).  The arithmetic of the wall that is in front of the ray is
    unchanged, so the image equals the one of the kernel generated without slab pairs bit for bit — from the
    scene's own camera (two pairs), from a camera left of the box (floor / ceiling only) and from inside it."""
    import copy
    w, h = 320, 200
    job = job_for("cornell_box", cfg, w, h)
    for pos, look_at in (((278.0, 278.0, -800.0), (278.0, 278.0, 0.0)), ((-100.0, 278.0, -800.0), (278.0, 278.0, 278.0)),
                         ((278.0, 400.0, 100.0), (100.0, 100.0, 500.0))):
        j = copy.copy(job)
        j.camera = harness.make_camera({"vfov": 40.0, "aperture": 0.0, "focus_distance": 10.0, "pos": list(pos),
                                        "look_at": list(look_at)}, w, h)
        p = harness.make_params(w, h, 16, 20, seed=3, specialize=1)
        renderer.upload(j)
        with_pairs = renderer.render(p)
        os.environ["RC_SPEC_NO_SLAB"] = "1"
        try:
            renderer.upload(j)          # the source is regenerated at the next render
            without = renderer.render(p)
        finally:
            del os.environ["RC_SPEC_NO_SLAB"]
        assert np.array_equal(with_pairs, without), pos
        ref = oracle.render(j, harness.make_params(w, h, 16, 20, seed=3))
        assert float((np.abs(with_pairs - ref).max(axis=2) > 2e-3).mean()) < 0.04, pos
