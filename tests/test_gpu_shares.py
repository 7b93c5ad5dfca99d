"""One participant's share (params.rank / params.world > 1) checked on its own, on one GPU.

A share is what every rank of a multi-GPU frame traces, and what rc_render, rc_render_preview, rc_render_accumulate and
rc_render_tiles_into hand back to a caller that passes rank / world.  The expected shares are computed here from the
rule the header documents — tile k (16 x 8 pixels, row-major over the image) goes to participant k mod world, samples
[S r / world, S (r + 1) / world) to participant r — and not from rc_partition, which is checked against that rule once.

Before every share the context renders a whole frame with another seed at the same size, so that whatever a share
leaves alone holds non-zero sums of an earlier render: a share must never show them.
"""
import numpy as np
import pytest

from racer_tracer_b200 import capi, harness
from test_gpu_parity import job_for
from test_gpu_shading_probes import SEED, W, H, check, reference, scene_job

pytestmark = pytest.mark.gpu

TILE_W, TILE_H = 16, 8
WAVE = capi.RC_VARIANT_WAVEFRONT
# kernel variants: rc_params fields on top of (width, height, spp, depth, seed, rank, world, split)
VARIANTS = {
    "mega": {},
    "spec": {"specialize": 1},
    "wave": {"variant": WAVE},
    "mega_reject": {"sampler": capi.RC_SAMPLER_REJECTION},
    "mega_r7": {"rng_rounds": 7},
}
SIZES = [(2, 2), (16, 8), (17, 9), (W, H)]      # one tile (part of one), exactly one, 4 ragged tiles, 15 x 15 tiles
WORLDS = (2, 3, 8)                                 # 8 > the tile count of the three small sizes: ranks with no tiles
SPPS = (1, 2, 3, 37, 600)                          # samples < world, uneven sample shares, >= 512 (sliced by default)
DEPTH = 6
STALE_SEED = 99
NAN_BITS = np.uint32(0x7FC0BEEF)                   # a quiet NaN whose payload says "never written"


# ---------------------------------------------------------------------------
# The share rule, restated
# ---------------------------------------------------------------------------
def tile_grid(w, h):
    return (w + TILE_W - 1) // TILE_W, (h + TILE_H - 1) // TILE_H


def tile_mask(w, h, rank, world):
    """(h, w) bool: the pixels of the tiles k with k mod world == rank."""
    tx, ty = tile_grid(w, h)
    own = (np.arange(tx * ty).reshape(ty, tx) % world) == rank
    return np.repeat(np.repeat(own, TILE_H, axis=0), TILE_W, axis=1)[:h, :w]


def sample_range(spp, rank, world):
    return spp * rank // world, spp * (rank + 1) // world


def block_mask(w, h, sw, sh, rank, world):
    """(h, w) bool: the screen pixels of a preview tile share — the tile rule over the grid of sw x sh blocks, each
    block expanded to its screen pixels; columns and rows beyond the last whole block belong to nobody."""
    gw, gh = w // sw, h // sh
    out = np.zeros((h, w), dtype=bool)
    if gw >= 1 and gh >= 1:
        out[:gh * sh, :gw * sw] = np.repeat(np.repeat(tile_mask(gw, gh, rank, world), sh, axis=0), sw, axis=1)
    return out


def share_count(w, h, spp, rank, world, split):
    """pixel-samples of a share"""
    if split == capi.RC_SPLIT_SAMPLES:
        lo, hi = sample_range(spp, rank, world)
        return w * h * (hi - lo)
    return int(tile_mask(w, h, rank, world).sum()) * spp


def params(w, h, spp, variant, seed=SEED, depth=DEPTH, **kw):
    return harness.make_params(w, h, spp, depth, seed=seed, **dict(VARIANTS[variant], **kw))


def _exact(variant, spp):
    """Both launches trace every pixel's samples in one CTA and add them once: the sums are bit-identical.  Above 31
    spp a launch may cut the samples into slices (a different number for a share than for the whole frame), and the
    wavefront adds every sample with an atomic."""
    return spp < 32 and (VARIANTS[variant].get("variant") != WAVE or spp == 1)


def _close(a, b, exact):
    return np.array_equal(a, b) if exact else np.allclose(a, b, rtol=1e-5, atol=1e-7)


def test_partition_follows_the_documented_rule(cuda_lib):
    """rc_partition against the rule above; everything else in this file uses the rule only."""
    for w, h in SIZES + [(1920, 1080)]:
        tx, ty = tile_grid(w, h)
        for world in WORLDS:
            for rank in range(world):
                for spp in SPPS:
                    for split in (capi.RC_SPLIT_TILES, capi.RC_SPLIT_SAMPLES):
                        p = harness.make_params(w, h, spp, 5, rank=rank, world=world, split=split)
                        got = harness.partition(p, rank, world)
                        assert (got["tiles_x"], got["tile_w"], got["tile_h"]) == (tx, TILE_W, TILE_H)
                        if split == capi.RC_SPLIT_TILES:
                            assert (got["tile_first"], got["tile_stride"]) == (rank, world)
                            assert got["n_tiles"] == len(range(rank, tx * ty, world))
                            assert (got["s_begin"], got["s_end"]) == (0, spp)
                        else:
                            assert (got["tile_first"], got["tile_stride"], got["n_tiles"]) == (0, 1, tx * ty)
                            assert (got["s_begin"], got["s_end"]) == sample_range(spp, rank, world)
                p = harness.make_params(w, h, 1, 5, rank=rank, world=world)
                assert np.array_equal(harness.share_mask(p, rank, world), tile_mask(w, h, rank, world))


# ---------------------------------------------------------------------------
# The edge matrix: every entry point, every rank of every world, both splits
# ---------------------------------------------------------------------------
_JOBS = {}


def _upload(renderer, cfg, w, h):
    """cornell_box at (w, h)"""
    if (w, h) not in _JOBS:
        _JOBS[(w, h)] = job_for("cornell_box", cfg, w, h)
    renderer.upload(_JOBS[(w, h)])


def _stale(renderer, w, h):
    """A whole frame with another seed: the context's buffers now hold its (non-zero) sums."""
    renderer.render(harness.make_params(w, h, 1, DEPTH, seed=STALE_SEED))


def _check_spec(renderer, variant):
    assert renderer.stats().specialized == (1 if VARIANTS[variant].get("specialize") else 0), variant


def _counts_segments(variant):
    return VARIANTS[variant].get("variant") != WAVE


@pytest.mark.parametrize("size", SIZES, ids=lambda s: "%dx%d" % s)
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_render_shares(renderer, cfg, variant, size, monkeypatch):
    """rc_render: a tile share is the whole render in its tiles and 0.0 elsewhere; a sample share's samples * out^2,
    summed over the ranks, is the whole frame's sum; an empty sample share is all zeros.  stats: the share's
    pixel-samples, and the ranks' segments add up to the whole frame's."""
    w, h = size
    _upload(renderer, cfg, w, h)
    for spp in SPPS:
        whole = renderer.render(params(w, h, spp, variant))
        _check_spec(renderer, variant)
        whole_segments = renderer.stats().segments
        whole_lin = spp * whole ** 2
        for world in WORLDS:
            tile_segments, sample_segments, lin = 0, 0, np.zeros_like(whole)
            for rank in range(world):
                label = f"{variant} {w}x{h} {spp} spp rank {rank}/{world}"
                own = tile_mask(w, h, rank, world)
                _stale(renderer, w, h)
                out = renderer.render(params(w, h, spp, variant, rank=rank, world=world))
                st = renderer.stats()
                assert (out[~own] == 0.0).all(), f"{label} tiles: {int((out[~own] != 0).any(axis=-1).sum())} pixels outside the share are not 0"
                assert _close(out[own], whole[own], _exact(variant, spp)), f"{label} tiles: {np.abs(out[own] - whole[own]).max()}"
                assert st.samples == share_count(w, h, spp, rank, world, capi.RC_SPLIT_TILES), (label, st.samples)
                tile_segments += st.segments
                if spp >= 32 and VARIANTS[variant].get("variant") != WAVE:
                    # unsliced on both sides: bit-identical again
                    monkeypatch.setenv("RC_SLICES", "1")
                    one = renderer.render(params(w, h, spp, variant))
                    _stale(renderer, w, h)
                    out1 = renderer.render(params(w, h, spp, variant, rank=rank, world=world))
                    monkeypatch.delenv("RC_SLICES")
                    assert (out1[~own] == 0.0).all() and np.array_equal(out1[own], one[own]), f"{label} tiles, RC_SLICES=1"

                _stale(renderer, w, h)
                out = renderer.render(params(w, h, spp, variant, rank=rank, world=world, split=capi.RC_SPLIT_SAMPLES))
                st = renderer.stats()
                lo, hi = sample_range(spp, rank, world)
                if hi == lo:
                    assert (out == 0.0).all(), f"{label} samples: an empty sample share is not all zeros"
                assert st.samples == share_count(w, h, spp, rank, world, capi.RC_SPLIT_SAMPLES), (label, st.samples)
                sample_segments += st.segments
                lin += spp * out ** 2
            assert np.allclose(lin, whole_lin, rtol=1e-5, atol=1e-6), f"{variant} {w}x{h} {spp} spp world {world}: {np.abs(lin - whole_lin).max()}"
            if _counts_segments(variant):
                assert tile_segments == whole_segments and sample_segments == whole_segments, \
                    (variant, w, h, spp, world, tile_segments, sample_segments, whole_segments)


@pytest.mark.parametrize("split", ["tiles", "samples"])
@pytest.mark.parametrize("variant", ["mega", "spec"])
def test_render_last_rank_of_eight_at_1080p(renderer, cfg, variant, split):
    """The benched size: rank 7 of 8 (tile 7, 15, ... of 120 x 135; or the last of 3 samples)."""
    w, h, spp, world, rank = 1920, 1080, 3, 8, 7
    _upload(renderer, cfg, w, h)
    whole = renderer.render(params(w, h, spp, variant))
    _stale(renderer, w, h)
    sp = capi.RC_SPLIT_TILES if split == "tiles" else capi.RC_SPLIT_SAMPLES
    out = renderer.render(params(w, h, spp, variant, rank=rank, world=world, split=sp))
    st = renderer.stats()
    _check_spec(renderer, variant)
    assert st.samples == share_count(w, h, spp, rank, world, sp)
    if sp == capi.RC_SPLIT_TILES:
        own = tile_mask(w, h, rank, world)
        assert (out[~own] == 0.0).all() and np.array_equal(out[own], whole[own])
    else:
        # rank 7 traces sample 2 alone; the other seven ranks' samples 0 and 1, rendered the same way, complete the sum
        rest = sum(spp * renderer.render(params(w, h, spp, variant, rank=r, world=world, split=sp)) ** 2
                   for r in range(world - 1))
        assert np.allclose(rest + spp * out ** 2, spp * whole ** 2, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("size", SIZES, ids=lambda s: "%dx%d" % s)
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_preview_shares(renderer, cfg, variant, size):
    """rc_render_preview at scale 1 x 1 and at the config's scale: the same rules over the grid of blocks."""
    w, h = size
    _upload(renderer, cfg, w, h)
    for scales in sorted({(1, 1), harness.preview_scales(cfg, w, h)}):
        for spp in SPPS:
            whole = renderer.render_preview(params(w, h, spp, variant), *scales)
            for world in WORLDS:
                lin = np.zeros_like(whole)
                for rank in range(world):
                    label = f"preview {scales} {variant} {w}x{h} {spp} spp rank {rank}/{world}"
                    own = block_mask(w, h, *scales, rank, world)
                    _stale(renderer, w, h)
                    out = renderer.render_preview(params(w, h, spp, variant, rank=rank, world=world), *scales)
                    assert (out[~own] == 0.0).all(), f"{label} tiles: {int((out[~own] != 0).any(axis=-1).sum())} pixels outside the share are not 0"
                    assert _close(out[own], whole[own], _exact(variant, spp)), f"{label} tiles: {np.abs(out[own] - whole[own]).max()}"
                    _stale(renderer, w, h)
                    out = renderer.render_preview(params(w, h, spp, variant, rank=rank, world=world, split=capi.RC_SPLIT_SAMPLES), *scales)
                    lo, hi = sample_range(spp, rank, world)
                    if hi == lo:
                        assert (out == 0.0).all(), f"{label} samples: an empty sample share is not all zeros"
                    lin += spp * out ** 2
                assert np.allclose(lin, spp * whole ** 2, rtol=1e-5, atol=1e-6), f"preview {scales} {variant} {w}x{h} {spp} spp world {world}"


def _device(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr).reshape(-1)).cuda()


@pytest.mark.parametrize("size", SIZES, ids=lambda s: "%dx%d" % s)
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_accumulate_and_tiles_into_shares(renderer, cfg, variant, size):
    """rc_render_accumulate adds its share and leaves every other float bit-identical; rc_render_tiles_into stores its
    tiles' sums and leaves every other float's bit pattern (a NaN here) as it was."""
    import torch
    w, h = size
    _upload(renderer, cfg, w, h)
    renderer.set_stream(torch.cuda.current_stream().cuda_stream)
    n = w * h * 3
    rng = np.random.default_rng(w * h)
    sentinel = rng.uniform(0.25, 4.0, n).astype(np.float32)      # finite, and a different value in every float
    nan = np.full(n, NAN_BITS, dtype=np.uint32).view(np.float32)
    wave = VARIANTS[variant].get("variant") == WAVE
    for spp in SPPS:
        for world in WORLDS:
            for rank in range(world):
                for split in (capi.RC_SPLIT_TILES, capi.RC_SPLIT_SAMPLES):
                    label = f"{variant} {w}x{h} {spp} spp rank {rank}/{world} split {split}"
                    p = params(w, h, spp, variant, rank=rank, world=world, split=split)
                    own = np.repeat(tile_mask(w, h, rank, world) if split == capi.RC_SPLIT_TILES else
                                    np.full((h, w), sample_range(spp, rank, world)[1] > sample_range(spp, rank, world)[0]), 3)
                    _stale(renderer, w, h)
                    zero = torch.zeros(n, dtype=torch.float32, device="cuda")
                    renderer.render_accumulate(p, zero.data_ptr())
                    acc = _device(sentinel)
                    _stale(renderer, w, h)
                    renderer.render_accumulate(p, acc.data_ptr())
                    torch.cuda.synchronize()
                    assert renderer.stats().samples == share_count(w, h, spp, rank, world, split), label
                    share, got = zero.cpu().numpy(), acc.cpu().numpy()
                    assert (share[~own] == 0).all(), label
                    assert np.array_equal(got[~own].view(np.uint32), sentinel[~own].view(np.uint32)), f"{label}: a float outside the share changed"
                    want = sentinel[own] + share[own]
                    assert (np.array_equal(got[own], want) if not wave else np.allclose(got[own], want, rtol=1e-5, atol=1e-6)), \
                        f"{label}: {np.abs(got[own] - want).max()}"
                    if split != capi.RC_SPLIT_TILES:
                        continue
                    img = _device(nan)
                    if wave:
                        with pytest.raises(capi.RacerCudaError) as e:
                            renderer.render_tiles_into(p, img.data_ptr())
                        assert e.value.status == capi.RC_ERR_INVALID
                        continue
                    _stale(renderer, w, h)
                    renderer.render_tiles_into(p, img.data_ptr())
                    torch.cuda.synchronize()
                    got = img.cpu().numpy()
                    assert (got[~own].view(np.uint32) == NAN_BITS).all(), f"{label}: tiles_into wrote outside its tiles"
                    assert np.isfinite(got[own]).all() and np.array_equal(got[own], share[own]), label


# ---------------------------------------------------------------------------
# Shares pixel by pixel against the oracle (the machinery of test_gpu_shading_probes)
# ---------------------------------------------------------------------------
PROBE_SCENES = ["cornell_box", "three_balls", "noise_and_textures", "random"]
MASK_SEEN = {}


def _check_share(label, gpu, ref, tol, mask, own, depth, expect_fail=False):
    """check() on the pixels of the share; outside it the oracle's own values stand in, so they cannot fail.  The mask
    bound applies to the whole image's mask, as in test_gpu_shading_probes: unstable pixels cluster (a horizon, a
    silhouette), and one rank's tiles can hold more than their share of them — 17.9 % of rank 1 of 2's preview
    blocks of noise_and_textures at depth 1.  The largest fraction within a share is recorded and printed."""
    MASK_SEEN[depth] = max(MASK_SEEN.get(depth, 0.0), float(mask[own].mean()))
    return check(label, np.where(own[..., None], gpu, ref), ref, tol, mask, depth, expect_fail)


def _ref(oracle, job, name, depth, variant, preview=None, sample=0):
    o = VARIANTS[variant]
    return reference(oracle, job, name, depth, o.get("sampler", capi.RC_SAMPLER_DIRECT), o.get("rng_rounds", 0),
                     preview, sample=sample)


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("name", PROBE_SCENES)
def test_share_probe(renderer, oracle, cfg, name, variant):
    """1 spp.  Tile split, world 2 and 3: rank r's tiles against the oracle's render (rc_render and, at the config's
    scale, rc_render_preview).  Sample split with spp = world: rank r traces sample r alone, against the oracle's
    sample r."""
    job = scene_job(cfg, name)
    renderer.upload(job)
    scales = harness.preview_scales(cfg, W, H)
    for depth in (1, 2):
        ref, tol, mask = _ref(oracle, job, name, depth, variant)
        pref, ptol, pmask = _ref(oracle, job, name, depth, variant, preview=scales)
        for world in (2, 3):
            for rank in range(world):
                label = f"{name} depth {depth} {variant} rank {rank}/{world}"
                _stale(renderer, W, H)
                out = renderer.render(params(W, H, 1, variant, depth=depth, rank=rank, world=world))
                _check_spec(renderer, variant)
                own = tile_mask(W, H, rank, world)
                assert (out[~own] == 0.0).all(), label
                _check_share(f"{label} tiles", out ** 2, ref, tol, mask, own, depth)

                _stale(renderer, W, H)
                out = renderer.render_preview(params(W, H, 1, variant, depth=depth, rank=rank, world=world), *scales)
                own = block_mask(W, H, *scales, rank, world)
                assert (out[~own] == 0.0).all(), label
                _check_share(f"{label} preview {scales} tiles", out ** 2, pref, ptol, pmask, own, depth)

                _stale(renderer, W, H)
                out = renderer.render(params(W, H, world, variant, depth=depth, rank=rank, world=world, split=capi.RC_SPLIT_SAMPLES))
                _check_spec(renderer, variant)
                sref, stol, smask = _ref(oracle, job, name, depth, variant, sample=rank)
                _check_share(f"{label} sample {rank}", world * out ** 2, sref, stol, smask, np.ones((H, W), bool), depth)

                if world == 2 and variant in ("mega", "spec", "wave"):     # (the references of the direct sampler)
                    _stale(renderer, W, H)
                    out = renderer.render_preview(params(W, H, world, variant, depth=depth, rank=rank, world=world,
                                                         split=capi.RC_SPLIT_SAMPLES), *scales)
                    sref, stol, smask = _ref(oracle, job, name, depth, variant, preview=scales, sample=rank)
                    _check_share(f"{label} preview {scales} sample {rank}", world * out ** 2, sref, stol, smask,
                                 block_mask(W, H, *scales, 0, 1), depth)
    print("largest mask fraction of a share so far, per depth:", {d: f"{v:.3%}" for d, v in sorted(MASK_SEEN.items())})


def test_share_probe_tells_sample_indices_apart(renderer, oracle, cfg):
    """Rank 1's sample share (sample 1) against the oracle's sample 0 must fail."""
    job = scene_job(cfg, "cornell_box")
    renderer.upload(job)
    out = renderer.render(params(W, H, 2, "mega", depth=2, rank=1, world=2, split=capi.RC_SPLIT_SAMPLES))
    ref, tol, mask = _ref(oracle, job, "cornell_box", 2, "mega", sample=0)
    n_bad, _ = _check_share("counterfactual: sample 1 against sample 0", 2 * out ** 2, ref, tol, mask,
                            np.ones((H, W), bool), 2, expect_fail=True)
    assert n_bad > 0, "sample 1 passes as sample 0: the comparison cannot tell sample indices apart"
