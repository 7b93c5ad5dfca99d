"""Shading checked pixel by pixel against the oracle, in every kernel variant.

At max_depth = 1 every pixel of a 1-spp render is one device operation at the primary hit — a texture value (solid,
checker, image, noise), an emission or a background value (renderer.rs:41-90); at depth 2 each pixel adds exactly one
scatter and one background or albedo lookup.  GPU and oracle consume the same Philox streams, so the only honest
difference between the GPU's fp32 and the oracle's f64 is rounding — except where the f64 answer is itself unstable
under an fp32-sized nudge (a silhouette, a texel or checker boundary, a Schlick threshold).  Those pixels are found
from the oracle alone — the scene rendered from cameras shifted by +-delta, with the rays turned by the error of the
fp32 ray direction, with the spheres' radii nudged by the error of the fp32 sphere test, and (scenes with checker or
noise textures) translated as a whole by the error of an fp32 hit point's coordinates — and masked; every other pixel
must agree within an fp32 error model.  No fraction of the image is left as slack.

Error model (2^-24 = one fp32 ulp, relative):
* solid, checker, image, emission, background: 16 ulp relative per bounce;
* every bounce after the first adds one scattered direction's error — the SFU sine / cosine of the direct sampler
  (5e-7 absolute) plus the normal from an fp32 hit point, 8 ulp of (|centre| + r + |camera|) / r for the scene's
  worst sphere, grown by up to the refraction index n per further bounce — times the slope of the sky
  (0.5 |top - bottom| per unit of direction);
* noise, at pixels whose primary hit is noise-textured: the hit point's fp32 error e_p (8 ulp of |p| + |camera|, at
  least delta, and on a sphere at least 8 ulp of |c| + r) times the slope of 0.5 (1 + sin(scale z + 10 turb)), which is 0.5 (scale + 10 depth G) with G = 2.5
  bounding |grad Perlin noise| (1.63 is the largest of 60 000 sampled points; the octave k adds 2^-k of a noise of
  p 2^k, whose argument carries 2^k e_p), plus 16 ulp of each of the `depth` octave sums, times 10; beyond depth 1
  times the brightest radiance that can come back (the largest emission, or 1).
acosf near the poles and atan2f at the seam amplify an fp32 error of the hit point by 1/sin(theta) and 1/rho; the
shifted renders amplify delta by the same factors, and for image-textured spheres the mask also takes shifts of
4 delta (the functions' own few-ulp errors of the angle).  The global tolerance is not raised for them.
"""
import copy
import ctypes as C

import numpy as np
import pytest

from conftest import SCENES_X
from racer_tracer_b200 import capi, harness
from test_gpu_parity import _accumulate, job_for, many_spheres_job

pytestmark = pytest.mark.gpu

ULP = 2.0 ** -24
W, H = 203, 117                 # ragged: neither a multiple of the 16 x 8 tile nor of a warp's 8 x 4 block
SEED = 7
NOISE_GRAD = 2.5
# Largest share of masked pixels per depth.  Measured on a B200 (1000 W) over every case of this file: depth 1
# 6.08 % (noise_and_textures, rejection sampler: the Perlin ground sphere seen up to the horizon), depth 2 9.25 %
# (random: 484 spheres, lens, motion), depth 3 1.74 % (the glass probe).
MASK_BOUND = {1: 0.12, 2: 0.15, 3: 0.025}

# kernel variants: rc_params fields on top of (width, height, 1 spp, depth, seed)
VARIANTS = {
    "mega": {},
    "mega_reject": {"sampler": capi.RC_SAMPLER_REJECTION},
    "spec": {"specialize": 1},
    "wave": {"variant": capi.RC_VARIANT_WAVEFRONT},
    "wave_reject": {"variant": capi.RC_VARIANT_WAVEFRONT, "sampler": capi.RC_SAMPLER_REJECTION},
    "mega_r7": {"rng_rounds": 7},
    "spec_r7": {"specialize": 1, "rng_rounds": 7},
    "wave_r7": {"variant": capi.RC_VARIANT_WAVEFRONT, "rng_rounds": 7},
}


# ---------------------------------------------------------------------------
# The comparison
# ---------------------------------------------------------------------------
def _with_camera_shift(job, shift, turn_only=False):
    """The job seen from a camera translated by `shift` — or, turn_only, with only the viewport moved: rays turned by
    |shift| / |upper_left_corner - origin|."""
    j = copy.copy(job)
    c = capi.rc_camera.from_buffer_copy(job.camera)
    if not turn_only:
        c.origin[:] = list(np.array(list(job.camera.origin)) + shift)
    c.upper_left_corner[:] = list(np.array(list(job.camera.upper_left_corner)) + shift)
    j.camera = c
    return j


def _delta(job):
    """1e-6 of the viewing distance scale, as ambiguous_mask (test_gpu_parity) uses for the primary hits."""
    org = np.array(list(job.camera.origin))
    return 1e-6 * (np.abs(org).max() + np.linalg.norm(org) + 1.0)


def _with_radius_nudge(job, sign):
    """The job with every sphere's radius changed by 8 ulp of |c| + r.  The fp32 sphere test solves a quadratic whose
    |o - c|^2 - r^2 cancels: its hit point moves along the ray by about that much (1e-3 on the reference's 1000-radius
    ground spheres, far more than the camera nudge), which decides the checker cells near y = 0."""
    src = job.scene
    fs = harness.FlatScene()
    fs.c = capi.rc_scene.from_buffer_copy(src.c)
    fs.keep, fs.np = list(src.keep), dict(src.np)
    data = src.np["prim_data"].copy()
    sph = np.isin(src.np["prim_type"], [capi.RC_PRIM_SPHERE, capi.RC_PRIM_MOVING_SPHERE])
    data[sph, 3] += sign * 8 * ULP * (np.linalg.norm(data[sph, :3], axis=1) + data[sph, 3])
    fs.np["prim_data"] = data
    fs.keep.append(data)
    fs.c.prim_data = data.ctypes.data_as(C.POINTER(C.c_double))
    out = copy.copy(job)
    out.scene = fs
    return out


def _texture_point_error(job):
    """fp32 error of a hit point's world coordinates, per axis: a sphere's point is formed as centre + r * normal
    (make_hit_local), whose components carry a few ulp of r, and the sum an ulp of |centre|; a rectangle's point a
    few ulp of its coordinates.  8 ulp of the largest coordinate of any primitive's box (1e-3 on the reference's
    1000-radius ground spheres: y there is -(x^2 + z^2) / 2000, so that checker cells near the top are undecided)."""
    return 8 * ULP * np.abs(job.scene.np["prim_aabb"]).max()


def _with_translation(job, shift):
    """The whole scene and the camera translated by `shift`: the same rays hit the same geometry, but checker and noise
    textures, which are functions of the world point, are evaluated at the hit point + shift — the off-surface error
    of an fp32 hit point, which no change of the geometry reproduces (a moved surface moves the hit along the ray).
    Not for scenes with RotateY / Translate instances (they rotate about the world's origin)."""
    src = job.scene
    assert src.c.n_instances == 0 or (src.np["prim_instance"] < 0).all()
    fs = harness.FlatScene()
    fs.c = capi.rc_scene.from_buffer_copy(src.c)
    fs.keep, fs.np = list(src.keep), dict(src.np)
    data, aabb, motion = src.np["prim_data"].copy(), src.np["prim_aabb"] + np.tile(shift, 2), src.np["prim_motion"].copy()
    ty = src.np["prim_type"]
    sph = np.isin(ty, [capi.RC_PRIM_SPHERE, capi.RC_PRIM_MOVING_SPHERE])
    data[sph, :3] += shift
    motion[ty == capi.RC_PRIM_MOVING_SPHERE, :3] += shift
    for kind, (a, b, k) in ((capi.RC_PRIM_XY_RECT, (0, 1, 2)), (capi.RC_PRIM_XZ_RECT, (0, 2, 1)), (capi.RC_PRIM_YZ_RECT, (1, 2, 0))):
        on = ty == kind
        data[on, 0:2] += shift[a]
        data[on, 2:4] += shift[b]
        data[on, 4] += shift[k]
    for name, arr, field, ctype in (("prim_data", data, "prim_data", C.c_double), ("prim_aabb", aabb, "prim_aabb", C.c_double),
                                    ("prim_motion", motion, "prim_motion", C.c_double)):
        arr = np.ascontiguousarray(arr)
        fs.np[name] = arr
        fs.keep.append(arr)
        if name != "prim_motion" or src.c.prim_motion:
            setattr(fs.c, field, arr.ctypes.data_as(C.POINTER(ctype)))
    nodes = []
    for nd in (src.c.nodes[i] for i in range(src.c.n_nodes)):
        n2 = capi.rc_bvh_node.from_buffer_copy(nd)
        n2.bmin[:] = list(np.array(list(nd.bmin)) + shift)
        n2.bmax[:] = list(np.array(list(nd.bmax)) + shift)
        nodes.append(n2)
    if nodes:
        arr = (capi.rc_bvh_node * len(nodes))(*nodes)
        fs.keep.append(arr)
        fs.c.nodes = arr
    fs.nodes = nodes
    for name in ("images", "textures", "materials", "instances", "object_keys", "camera_cfg", "tone_map_cfg"):
        setattr(fs, name, getattr(src, name, None))
    out = _with_camera_shift(job, shift)
    out.scene = fs
    return out


def _has_world_textures(job):
    s = job.scene
    return any(s.c.textures[i].type in (capi.RC_TEX_CHECKER, capi.RC_TEX_NOISE) for i in range(s.c.n_textures))


def _eps_dir(job):
    """Error of one scattered direction (see the module docstring)."""
    s, org = job.scene, np.linalg.norm(list(job.camera.origin))
    ratio = 1.0
    for t, d in zip(s.np["prim_type"], s.np["prim_data"]):
        if t in (capi.RC_PRIM_SPHERE, capi.RC_PRIM_MOVING_SPHERE) and d[3] > 0:
            ratio = max(ratio, (np.linalg.norm(d[:3]) + d[3] + org) / d[3])
    return 5e-7 + 8 * ULP * ratio


def _max_ior(job):
    s = job.scene
    return max([1.0] + [max(m.param, 1.0 / m.param) for m in (s.c.materials[i] for i in range(s.c.n_materials))
                        if m.type == capi.RC_MAT_DIELECTRIC and m.param > 0])


def _noise_tolerance(oracle, job, params):
    """Per-pixel bound of the noise texture's fp32 error at the primary hit (module docstring), 0 elsewhere."""
    s = job.scene
    w, h = params.width, params.height
    noise = {}
    for pid, mi, ty, d in zip(s.np["prim_id"], s.np["prim_material"], s.np["prim_type"], s.np["prim_data"]):
        m = s.c.materials[int(mi)]
        if m.type == capi.RC_MAT_DIELECTRIC:
            continue
        t = s.c.textures[m.texture]
        if t.type == capi.RC_TEX_NOISE:
            sphere_err = 8 * ULP * (np.linalg.norm(d[:3]) + d[3]) if ty in (capi.RC_PRIM_SPHERE, capi.RC_PRIM_MOVING_SPHERE) else 0.0
            noise[int(pid)] = (max(abs(v) for v in t.color), t.scale, t.b, sphere_err)
    if not noise:
        return 0.0
    # the albedo's error multiplies the radiance that comes back: at most the brightest emission (or the sky's 1)
    back = max([1.0] + [max(s.c.textures[m.texture].color) for m in (s.c.materials[i] for i in range(s.c.n_materials))
                        if m.type == capi.RC_MAT_DIFFUSE_LIGHT]) if params.max_depth > 1 else 1.0
    p = harness.make_params(w, h, 1, 1, fixed_jitter=1)
    ids, _, _, pt = oracle.primary_aov(job, p)
    ids, pt = ids.reshape(h, w), pt.reshape(h, w, 3)
    org = np.linalg.norm(list(job.camera.origin))
    e_p = np.maximum(_delta(job), 8 * ULP * (np.linalg.norm(pt, axis=2) + org))
    tol = np.zeros((h, w))
    for pid, (col, scale, depth, sphere_err) in noise.items():
        on = ids == pid
        e = np.maximum(e_p[on], sphere_err)      # a sphere's hit point: the error of its quadratic (_with_radius_nudge)
        tol[on] = back * 0.5 * col * ((abs(scale) + 10 * depth * NOISE_GRAD) * e + 10 * depth * 16 * ULP)
    # the rendered rays are jittered within the pixel: take the largest bound of the 3 x 3 neighbourhood
    pad = np.pad(tol, 1, mode="edge")
    return np.max([pad[dy:dy + h, dx:dx + w] for dy in range(3) for dx in range(3)], axis=0)[..., None]


def _tolerance(oracle, job, params, ref):
    d = max(params.max_depth, 1)
    tol = 16 * ULP * d * np.maximum(1.0, np.abs(ref))
    if d > 1 and job.scene.c.bg_type == capi.RC_BG_SKY:
        slope = 0.5 * np.abs(np.array(list(job.scene.c.bg_b)) - np.array(list(job.scene.c.bg_a))).max()
        # (a refraction turns a direction error e into up to n e: the index bounds the growth per bounce)
        tol = tol + slope * _eps_dir(job) * sum(_max_ior(job) ** k for k in range(d - 1))
    return tol + _noise_tolerance(oracle, job, params)


def _oracle_linear(oracle, job, q, preview, sample=0):
    """The linear radiance of sample `sample` alone (q.samples = 1)."""
    if preview:
        return oracle.render_preview(job, q, *preview, sample_begin=sample, sample_count=1) ** 2 * q.samples
    return oracle.render(job, q, linear_sum=True, sample_begin=sample, sample_count=1)


_REF_CACHE = {}


def reference(oracle, job, key, depth, sampler=capi.RC_SAMPLER_DIRECT, rounds=0, preview=None, widen=False, sample=0):
    """(linear radiance, per-pixel tolerance, instability mask) of the oracle's sample `sample`; cached per key."""
    ck = (key, depth, sampler, rounds, preview, widen, sample)
    if ck in _REF_CACHE:
        return _REF_CACHE[ck]
    q = harness.make_params(job.width, job.height, 1, depth, seed=SEED, sampler=sampler, rng_rounds=rounds)
    ref = _oracle_linear(oracle, job, q, preview, sample)
    tol = _tolerance(oracle, job, q, ref)
    cam = job.camera
    right, up = np.array(list(cam.right)), np.array(list(cam.up))
    mask = np.zeros(ref.shape[:2], dtype=bool)
    for scale in ((1.0, 4.0) if widen else (1.0,)):
        delta = scale * _delta(job)
        for sx, sy in ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (-1, -1), (1, -1), (-1, 1)):
            shifted = _oracle_linear(oracle, _with_camera_shift(job, delta * (sx * right + sy * up)), q, preview, sample)
            mask |= (np.abs(shifted - ref) > tol).any(axis=2)
    # the fp32 ray direction (upper_left_corner + u horizontal - v vertical - origin) carries 8 ulp of its length: at
    # the horizon of a ground plane that moves the hit point far more than the translation above
    turn = 8 * ULP * np.linalg.norm(np.array(list(cam.upper_left_corner)) - np.array(list(cam.origin)))
    nudged = [_with_camera_shift(job, turn * (sx * right + sy * up), turn_only=True) for sx, sy in ((1, 0), (-1, 0), (0, 1), (0, -1))]
    nudged += [_with_radius_nudge(job, sign) for sign in (1.0, -1.0)]
    if _has_world_textures(job):
        e = _texture_point_error(job)
        nudged += [_with_translation(job, sign * e * axis) for axis in np.eye(3) for sign in (1.0, -1.0)]
    for j in nudged:
        mask |= (np.abs(_oracle_linear(oracle, j, q, preview, sample) - ref) > tol).any(axis=2)
    _REF_CACHE[ck] = ref, tol, mask
    return _REF_CACHE[ck]


def gpu_linear(renderer, job, depth, variant, preview=None):
    """The GPU's linear radiance of the 1-spp render and whether the scene-specialised kernel ran."""
    p = harness.make_params(job.width, job.height, 1, depth, seed=SEED, **VARIANTS[variant])
    if preview:
        img = renderer.render_preview(p, *preview) ** 2
    else:
        img = _accumulate(renderer, p).reshape(job.height, job.width, 3).cpu().numpy().astype(np.float64)
    return img, renderer.stats().specialized


def check(label, gpu, ref, tol, mask, depth, expect_fail=False):
    """Every pixel outside the mask within its tolerance; the mask within its bound.  Returns the failing count."""
    err = np.abs(gpu - ref)
    bad = (err > tol).any(axis=2) & ~mask
    outside = np.where(mask[..., None], 0.0, err)
    # the image-level criterion of test_gpu_parity, on the displayed (square-rooted) images
    d = np.abs(np.sqrt(np.maximum(gpu, 0)) - np.sqrt(np.maximum(ref, 0))).max(axis=2)
    old_ok = float((d > 2e-3).mean()) < 0.03 and float(np.median(d)) < 1e-5
    print(f"{label}: mask {mask.sum()} px ({mask.mean():.3%}), max err outside {outside.max():.3e}, "
          f"max err/tol outside {(outside / tol).max():.3g}, failing {bad.sum()}, image-level criterion "
          f"{'passes' if old_ok else 'fails'}")
    assert np.isfinite(gpu).all()
    if not expect_fail:
        assert mask.mean() <= MASK_BOUND[depth], f"{label}: {mask.mean():.3%} of the pixels are unstable"
        assert not bad.any(), f"{label}: {bad.sum()} pixels outside the mask differ by more than the fp32 error model"
    return int(bad.sum()), old_ok


def probe(renderer, oracle, job, key, depth, variant, preview=None, ref_job=None, widen=False, expect_fail=False):
    opts = VARIANTS[variant]
    renderer.upload(job)
    gpu, spec = gpu_linear(renderer, job, depth, variant, preview)
    assert spec == (1 if opts.get("specialize") else 0), f"{key} {variant}: stats().specialized = {spec}"
    ref, tol, mask = reference(oracle, ref_job or job, key, depth, opts.get("sampler", capi.RC_SAMPLER_DIRECT),
                               opts.get("rng_rounds", 0), preview, widen)
    return check(f"{key} depth {depth} {variant}{' preview %dx%d' % preview if preview else ''}", gpu, ref, tol, mask,
                 depth, expect_fail)


# ---------------------------------------------------------------------------
# Probe scenes, built the way many_spheres_job builds one
# ---------------------------------------------------------------------------
def solid(rgb):
    t = capi.rc_texture()
    t.type = capi.RC_TEX_SOLID
    t.color[:] = list(rgb)
    return t


def checker(a, b, scale):
    t = capi.rc_texture()
    t.type, t.a, t.b, t.scale = capi.RC_TEX_CHECKER, a, b, scale
    return t


def material(kind, texture=0, param=0.0):
    m = capi.rc_material()
    m.type, m.texture, m.param = kind, texture, param
    return m


def sphere(key, centre, r, mat):
    lo, hi = [c - r for c in centre], [c + r for c in centre]
    return key, harness.TopObject(key, [harness.Prim(capi.RC_PRIM_SPHERE, list(centre) + [r, 0.0], mat, 0)], lo, hi, list(centre))


def xy_rect(key, x0, x1, y0, y1, k, mat):
    data, lo, hi, pos = harness._rect_prims(capi.RC_PRIM_XY_RECT, x0, x1, y0, y1, k)
    return key, harness.TopObject(key, [harness.Prim(capi.RC_PRIM_XY_RECT, data, mat, 0)], lo, hi, pos)


def build_job(cfg, textures, materials, objects, camera, images=(), perlins=(), bg=None, w=W, h=H):
    fs = harness.FlatScene()
    harness._flatten(fs, dict(objects), textures, materials, list(images), list(perlins))
    fs.c.bg_type = capi.RC_BG_SKY if bg is None else capi.RC_BG_SOLID
    fs.c.bg_a[:] = [1.0, 1.0, 1.0] if bg is None else list(bg)
    fs.c.bg_b[:] = [0.5, 0.7, 1.0]
    cam = harness.make_camera(dict({"vfov": 40.0, "aperture": 0.0, "focus_distance": 10.0}, **camera), w, h)
    return harness.Job(fs, cam, harness.make_tone_map("none"), cfg, w, h)


def checker_chain_job(cfg, depth, shared=False):
    """A ground sphere textured by a chain of `depth` checkers (c_depth -> ... -> c_1 -> solid), each level with its
    own scale and its own second child, so that every level decides some pixels and every leaf colour shows; two
    more spheres whose checkers share children (shared=True: two roots over one sub-chain, and a diamond)."""
    rng = np.random.default_rng(depth)
    textures = [solid(rng.uniform(0.1, 0.9, 3)) for _ in range(depth + 1)]
    prev = 0
    for level in range(1, depth + 1):
        textures.append(checker(prev, level, (10.0, 7.0, 4.3, 2.9, 1.7, 1.1, 0.7)[level - 1]))
        prev = len(textures) - 1
    mats = [material(capi.RC_MAT_LAMBERTIAN, prev)]
    objs = [sphere("ground", (0.0, -1000.0, 0.0), 1000.0, 0)]
    if shared:
        sub = prev
        textures.append(checker(sub, 1, 3.3))                      # a second root over the same chain
        textures.append(checker(sub, sub, 5.1))                    # a diamond: both children the same texture
        mats += [material(capi.RC_MAT_LAMBERTIAN, len(textures) - 2), material(capi.RC_MAT_LAMBERTIAN, len(textures) - 1)]
        objs += [sphere("s1", (-1.2, 1.0, 0.0), 1.0, 1), sphere("s2", (1.2, 1.0, 0.0), 1.0, 2)]
    return build_job(cfg, textures, mats, objs, {"pos": [0.5, 3.0, 9.0], "look_at": [0.0, 0.5, 0.0]})


def probe_image(shift=0):
    """37 x 23 RGBA, a different colour in every texel: a one-texel error is a gross error (6 / 255 or 11 / 255)."""
    j, i = np.mgrid[0:23, 0:37]
    px = np.stack([i * 6 + 10, j * 11 + 5, (i * 23 + j * 7) % 200 + 40, np.full_like(i, 255)], axis=2).astype(np.uint8)
    return np.ascontiguousarray(np.roll(px, shift, axis=1))


def image_job(cfg, kind, shift=0):
    px = probe_image(shift)
    textures = [checker(1, 2, 10.0), solid((0.3, 0.3, 0.3)), solid((0.6, 0.6, 0.6)), capi.rc_texture()]
    textures[3].type, textures[3].a = capi.RC_TEX_IMAGE, 0
    mats = [material(capi.RC_MAT_LAMBERTIAN, 3), material(capi.RC_MAT_DIFFUSE_LIGHT, 3)]
    if kind == "sphere":     # the seam (x < 0, z = 0) and the north pole in view
        objs = [sphere("globe", (0.0, 0.0, 0.0), 1.0, 1)]
        cam = {"pos": [-3.0, 2.2, 0.6], "look_at": [0.0, 0.2, 0.0], "vfov": 45.0}
    else:                    # all four edges in view: u, v in {0, 1}, the clamp and the fi >= fw branch
        objs = [xy_rect("panel", -1.3, 1.1, -0.7, 0.9, -1.0, 1)]
        cam = {"pos": [0.2, 0.3, 3.0], "look_at": [-0.1, 0.1, -1.0], "vfov": 60.0}
    return build_job(cfg, textures, mats, objs, cam, images=[(37, 23, px)], bg=(0.05, 0.05, 0.05))


def noise_job(cfg, where, scale=4.0):
    """Noise-textured geometry at negative coordinates: |p| ~ 1-10 ('near') and ~ 1000 ('far')."""
    textures = [capi.rc_texture()]
    textures[0].type, textures[0].a, textures[0].b, textures[0].scale = capi.RC_TEX_NOISE, 0, 7, scale
    textures[0].color[:] = [1.0, 0.9, 0.8]
    mats = [material(capi.RC_MAT_LAMBERTIAN, 0)]
    if where == "near":
        objs = [sphere("a", (-1.5, -0.5, -2.0), 1.0, 0), sphere("b", (-6.0, -3.0, -9.0), 3.0, 0),
                xy_rect("wall", -14.0, 2.0, -9.0, 3.0, -14.0, 0)]
        cam = {"pos": [1.0, 1.0, 3.0], "look_at": [-3.0, -2.0, -6.0], "vfov": 60.0}
    else:
        objs = [sphere("a", (-700.0, -300.0, -650.0), 40.0, 0), sphere("b", (-900.0, -420.0, -880.0), 120.0, 0),
                xy_rect("wall", -1300.0, -500.0, -800.0, -100.0, -1100.0, 0)]
        cam = {"pos": [-560.0, -180.0, -420.0], "look_at": [-820.0, -380.0, -900.0], "vfov": 60.0}
    return build_job(cfg, textures, mats, objs, cam, perlins=[harness.make_perlin(0, 0)])


def glass_job(cfg, ior=1.5):
    """A glass sphere under the sky over a dark ground: refraction, total internal reflection, the Schlick choice."""
    textures = [solid((0.2, 0.25, 0.3))]
    mats = [material(capi.RC_MAT_DIELECTRIC, 0, ior), material(capi.RC_MAT_LAMBERTIAN, 0)]
    objs = [sphere("glass", (0.0, 1.0, 0.0), 1.0, 0), sphere("ground", (0.0, -1000.0, 0.0), 1000.0, 1)]
    return build_job(cfg, textures, mats, objs, {"pos": [0.0, 1.6, 4.5], "look_at": [0.0, 1.0, 0.0], "vfov": 45.0})


PROBES = {
    "checker4": lambda cfg: checker_chain_job(cfg, 4),
    "checker5": lambda cfg: checker_chain_job(cfg, 5),
    "checker6": lambda cfg: checker_chain_job(cfg, 6),
    "checker_shared": lambda cfg: checker_chain_job(cfg, 3, shared=True),
    "image_sphere": lambda cfg: image_job(cfg, "sphere"),
    "image_rect": lambda cfg: image_job(cfg, "rect"),
    "noise_near": lambda cfg: noise_job(cfg, "near"),
    "noise_far": lambda cfg: noise_job(cfg, "far"),
    "glass": lambda cfg: glass_job(cfg),
}
PROBE_DEPTHS = {"glass": (2, 3)}


_JOBS = {}


def scene_job(cfg, name):
    """One job per scene for the whole session: the oracle's references are cached by scene name."""
    if name not in _JOBS:
        _JOBS[name] = job_for(name, cfg, W, H)
    return _JOBS[name]


# ---------------------------------------------------------------------------
# 1. Every BASELINE scene, every kernel variant
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("name", SCENES_X)
def test_scene_probe(renderer, oracle, cfg, name, depth, variant):
    job = scene_job(cfg, name)
    if name == "random" and variant == "wave_r7":
        renderer.upload(job)
        with pytest.raises(capi.RacerCudaError) as e:          # moving spheres: 10 rounds only in the wavefront
            gpu_linear(renderer, job, depth, variant)
        assert e.value.status == capi.RC_ERR_INVALID
        return
    probe(renderer, oracle, job, name, depth, variant)


# ---------------------------------------------------------------------------
# 2. The probe scenes, every kernel variant
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("kind", list(PROBES))
def test_probe_scene(renderer, oracle, cfg, kind, variant):
    job = PROBES[kind](cfg)
    for depth in PROBE_DEPTHS.get(kind, (1, 2)):
        probe(renderer, oracle, job, kind, depth, variant, widen=kind == "image_sphere")


def test_cyclic_checker_is_rejected(renderer, cfg):
    job = checker_chain_job(cfg, 3)
    tex = job.scene.c.textures
    top = job.scene.c.n_textures - 1
    tex[1].type, tex[1].a, tex[1].b = capi.RC_TEX_CHECKER, top, 0           # c_1's leaf becomes the chain's root
    with pytest.raises(capi.RacerCudaError) as e:
        renderer.upload(job)
    assert e.value.status == capi.RC_ERR_INVALID and "cycle" in str(e.value)


# ---------------------------------------------------------------------------
# 3. The preview renderer, the GPU-built BVH, the global-memory scene mode
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("at_scale", [False, True])
@pytest.mark.parametrize("name", ["cornell_box", "three_balls", "noise_and_textures", "random"])
def test_preview_probe(renderer, oracle, cfg, name, at_scale, spec):
    job = scene_job(cfg, name)
    scales = harness.preview_scales(cfg, W, H) if at_scale else (1, 1)
    probe(renderer, oracle, job, name, 2, "spec" if spec else "mega", preview=scales)


@pytest.mark.parametrize("name", ["random", "sandbox_boxes", "clown", "cornell_box"])
def test_lbvh_probe(renderer, oracle, cfg, name):
    job = job_for(name, cfg, W, H)
    renderer.upload(job)
    renderer.build_lbvh()
    nodes, order = renderer.get_bvh(job.scene.c.n_prims)
    same_tree = harness.with_bvh(job, nodes, order)
    for variant in ("mega", "spec"):
        p = harness.make_params(W, H, 1, 2, seed=SEED, **VARIANTS[variant])
        gpu = _accumulate(renderer, p).reshape(H, W, 3).cpu().numpy().astype(np.float64)   # (no re-upload: the LBVH)
        assert renderer.stats().specialized == (variant == "spec")
        ref, tol, mask = reference(oracle, same_tree, f"{name}+lbvh", 2)
        check(f"{name} lbvh depth 2 {variant}", gpu, ref, tol, mask, 2)


@pytest.mark.parametrize("variant", ["mega", "spec"])
def test_global_scene_mode_probe(renderer, oracle, cfg, variant, monkeypatch):
    monkeypatch.setenv("RC_SCENE_MODE", "global")
    probe(renderer, oracle, scene_job(cfg, "random"), "random", 2, variant)


@pytest.mark.parametrize("variant", ["mega", "spec"])
def test_many_spheres_probe(renderer, oracle, cfg, variant):
    job = many_spheres_job(cfg, 9000, 160, 120)
    renderer.upload(job)                          # no nodes: the library builds the LBVH, traced from global memory
    same_tree = harness.with_bvh(job, *renderer.get_bvh(9000))
    for depth in (1, 2):
        p = harness.make_params(160, 120, 1, depth, seed=SEED, **VARIANTS[variant])
        gpu = _accumulate(renderer, p).reshape(120, 160, 3).cpu().numpy().astype(np.float64)
        assert renderer.stats().specialized == (variant == "spec")
        ref, tol, mask = reference(oracle, same_tree, "many_spheres", depth)
        check(f"many_spheres depth {depth} {variant}", gpu, ref, tol, mask, depth)


# ---------------------------------------------------------------------------
# 4. The comparison can fail: the GPU render against the oracle of a slightly different scene
# ---------------------------------------------------------------------------
def _random_later_time_b(cfg):
    job = job_for("random", cfg, W, H)
    job.scene.np["prim_motion"][:, 4] = np.where(job.scene.np["prim_type"] == capi.RC_PRIM_MOVING_SPHERE, 1.01, 0.0)
    return job


COUNTERFACTUALS = {
    "image_one_texel": (lambda cfg: image_job(cfg, "rect"), lambda cfg: image_job(cfg, "rect", shift=1), 1),
    "noise_scale": (lambda cfg: noise_job(cfg, "far"), lambda cfg: noise_job(cfg, "far", scale=4.001), 1),
    "refraction_index": (glass_job, lambda cfg: glass_job(cfg, ior=1.501), 3),     # into the glass and out to the sky
    "moving_time_b": (lambda cfg: job_for("random", cfg, W, H), _random_later_time_b, 2),
}


@pytest.mark.parametrize("case", list(COUNTERFACTUALS))
def test_probe_detects_a_perturbed_scene(renderer, oracle, cfg, case):
    make, perturbed, depth = COUNTERFACTUALS[case]
    n_bad, _ = probe(renderer, oracle, make(cfg), f"counterfactual {case}", depth, "mega", ref_job=perturbed(cfg),
                     expect_fail=True)
    assert n_bad > 0, f"{case}: the perturbed scene passes the pixel comparison"


# ---------------------------------------------------------------------------
# 5. Sliced launches trace every sample exactly once
# ---------------------------------------------------------------------------
def _render_with(renderer, p, monkeypatch, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    try:
        img = renderer.render(p)
        st = renderer.stats()
    finally:
        for k in env:
            monkeypatch.delenv(k)
    return img, st


@pytest.mark.parametrize("spp", [37, 1000, 1024])
@pytest.mark.parametrize("halving", [0, 1])
@pytest.mark.parametrize("slices", [2, 3, 4, 5, 7])
def test_sliced_launch_traces_every_sample_once(renderer, cfg, slices, halving, spp, monkeypatch):
    w, h = 61, 37
    renderer.upload(job_for("cornell_box", cfg, w, h))
    p = harness.make_params(w, h, spp, 20, seed=3, specialize=2)
    one, st1 = _render_with(renderer, p, monkeypatch, RC_SLICES=1)
    img, st = _render_with(renderer, p, monkeypatch, RC_SLICES=slices, RC_SLICE_HALVING=halving)
    assert st1.kernel_launches == 1 and st.kernel_launches == 2 and st.specialized == 1
    assert st.segments == st1.segments and st.samples == st1.samples
    assert np.allclose(img, one, rtol=1e-5, atol=1e-6), np.abs(img - one).max()


def test_bench_frame_slices_trace_every_sample_once(renderer, cfg, monkeypatch):
    """cornell_box 1920 x 1080, 1024 spp, specialize = 2: the benched frame runs as two linear slices."""
    w, h = 1920, 1080
    renderer.upload(job_for("cornell_box", cfg, w, h))
    p = harness.make_params(w, h, 1024, 20, seed=1, specialize=2)
    sliced = renderer.render(p)
    st = renderer.stats()
    one, st1 = _render_with(renderer, p, monkeypatch, RC_SLICES=1)
    assert st.kernel_launches == 2 and st1.kernel_launches == 1 and st.specialized == 1
    assert st.segments == st1.segments
    assert np.allclose(sliced, one, rtol=1e-5, atol=1e-6), np.abs(sliced - one).max()
