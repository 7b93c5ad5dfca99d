"""Python stand-in for the reference's Rust host, used by tests and bench.py.

It does what the Rust side keeps doing in north_star: parse the YAML scene and
config formats, derive the camera, flatten the hittable list into
structure-of-arrays primitive buffers plus a host-built BVH, and hand the flat
structs of include/racer_cuda.h to the C ABI.  The same flat structs feed the
CPU oracle, so both sides trace the identical scene and tree.

Reference semantics followed (paths relative to /root/reference/racer-tracer/):
  scene YAML          src/scene/yml.rs:49-458
  config YAML         src/config.rs:69-225, config.yml
  camera merge        src/camera.rs:393-464, src/main.rs:95-111
  camera derivation   src/camera.rs:196-234
  tone-map selection  src/main.rs:84-86, src/tone_map.rs:18-66
  BVH                 src/bvh_node.rs:31-82 (median split; our axis choice is
                      deterministic where the reference's is random)
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field

import numpy as np
import yaml

from . import capi
from .capi import (rc_bvh_node, rc_camera, rc_image, rc_instance, rc_material, rc_params,
                   rc_perlin, rc_scene, rc_texture, rc_tone_map)

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32(ctr, key, rounds=10):
    """Philox4x32 (Salmon et al., SC'11); same stream definition as the GPU."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for r in range(rounds):
        if r:
            k0 = (k0 + W0) & MASK
            k1 = (k1 + W1) & MASK
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & MASK, p1 & MASK, ((p0 >> 32) ^ c3 ^ k1) & MASK, p0 & MASK
    return c0, c1, c2, c3


def u01(x: int) -> float:
    return (x >> 8) / 16777216.0


TAG_PERLIN = 2


def make_perlin(seed: int, index: int) -> rc_perlin:
    """Perlin::new (src/texture/noise.rs:44-55): 256 gradients = normalised
    uniform(-1,1)^3 vectors, here drawn from Philox(seed) so that host, oracle
    and GPU share them; identity permutation tables (noise.rs:122, Q17)."""
    p = rc_perlin()
    key = (seed & MASK, (seed >> 32) & MASK)
    for i in range(256):
        r = philox4x32((i, index, 0, TAG_PERLIN << 24), key)
        v = [2.0 * u01(r[k]) - 1.0 for k in range(3)]
        n = math.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
        for k in range(3):
            p.ran_vec[i][k] = v[k] / n
        p.perm_x[i] = p.perm_y[i] = p.perm_z[i] = i
    return p


class SceneLoadError(Exception):
    """TracerError::SceneLoad / UnknownMaterial / Configuration (src/error.rs)."""


def _lower_keys(node):
    # the `config` 0.13 crate lower-cases every map key on load
    if isinstance(node, dict):
        return {str(k).lower(): _lower_keys(v) for k, v in node.items()}
    if isinstance(node, list):
        return [_lower_keys(v) for v in node]
    return node


def _vec3(node, what="pos"):
    """Vec3 deserialises from {pos: [x,y,z]} with alias `color` (src/vec3.rs:12-16)."""
    if isinstance(node, dict):
        for k in ("pos", "color"):
            if k in node:
                node = node[k]
                break
        else:
            raise SceneLoadError(f"missing field `pos` in {what}")
    if not isinstance(node, (list, tuple)) or len(node) != 3:
        raise SceneLoadError(f"expected 3 numbers for {what}")
    return [float(v) for v in node]


def _enum(node, what):
    """Externally tagged serde enum: {Variant: {fields}} or a bare 'Variant'."""
    if isinstance(node, str):
        return node.lower(), {}
    if isinstance(node, dict) and len(node) == 1:
        (k, v), = node.items()
        return str(k).lower(), (v if v is not None else {})
    raise SceneLoadError(f"expected a single enum variant for {what}")


@dataclass
class Prim:
    type: int
    data: list
    material: int
    obj: int          # top-level object ordinal (1-based, canonical)
    side: int = 0
    instance: int = -1
    motion: list | None = None   # moving sphere: [pos_b x, y, z, time_a, time_b]


@dataclass
class TopObject:
    key: str
    prims: list
    aabb_min: list = field(default_factory=list)
    aabb_max: list = field(default_factory=list)
    pos: list = field(default_factory=lambda: [0.0, 0.0, 0.0])
    rotate_deg: float | None = None
    translate: list | None = None


def _aabb(a, b):
    # Aabb::new, src/aabb.rs:10-26
    return [min(a[i], b[i]) for i in range(3)], [max(a[i], b[i]) for i in range(3)]


def _rect_prims(kind, a0, a1, b0, b1, k):
    if kind == capi.RC_PRIM_XY_RECT:      # xy_rect.rs:50-55, geometry_creation.rs:41-57
        lo, hi = _aabb([a0, b0, k - 0.0001], [a1, b1, k + 0.0001]); pos = [a0, b0, k]
    elif kind == capi.RC_PRIM_XZ_RECT:    # xz_rect.rs:51-56
        lo, hi = _aabb([a0, k - 0.0001, b0], [a1, k + 0.0001, b1]); pos = [a0, k, b0]
    else:                                 # yz_rect.rs:51-56
        lo, hi = _aabb([k - 0.0001, a0, b0], [k + 0.0001, a1, b1]); pos = [k, a0, b0]
    return [a0, a1, b0, b1, k], lo, hi, pos


class FlatScene:
    """Owns the arrays an rc_scene points into."""

    def __init__(self):
        self.c = rc_scene()
        self.keep = []
        self.object_keys: list[str] = []
        self.camera_cfg: dict | None = None
        self.tone_map_cfg = None
        self.prims: list[Prim] = []

    @property
    def ptr(self):
        return C.byref(self.c)


def _flatten(fs: "FlatScene", objects: dict, textures, materials, images, perlins, use_bvh=None):
    """Top-level objects -> structure-of-arrays primitives + host BVH (what the Rust shim does before
    rc_upload_scene)."""
    # canonical ids (SURVEY §8(c)): objects numbered 1..N by sorted lower-cased
    # key; reported id = (object << 3) | box side
    instances: list[rc_instance] = []
    ordered = [objects[k] for k in sorted(objects)]
    for n, o in enumerate(ordered, start=1):
        inst = -1
        if o.rotate_deg is not None or o.translate is not None:
            ri = rc_instance()
            if o.rotate_deg is not None:
                ri.flags |= 1
                rad = o.rotate_deg * math.pi / 180.0  # util.rs:5-7
                ri.sin_theta, ri.cos_theta = math.sin(rad), math.cos(rad)
            if o.translate is not None:
                ri.flags |= 2
                ri.offset[:] = o.translate
            inst = len(instances)
            instances.append(ri)
        for p in o.prims:
            p.obj, p.instance = n, inst
    fs.object_keys = [o.key for o in ordered]

    if use_bvh is None:
        use_bvh = True
    nodes: list[rc_bvh_node] = []
    if use_bvh and ordered:
        order: list[TopObject] = []
        if len(ordered) >= SAH_MIN_OBJECTS and not instances:
            _build_bvh_sah(list(enumerate(ordered)), nodes, order)
        else:
            _build_bvh(ordered, nodes, order)
        ordered = order
        # fix leaf prim offsets now that the DFS order is known
        first = {}
        n = 0
        for o in ordered:
            first[id(o)] = n
            n += len(o.prims)
        for nd in nodes:
            if nd.left < 0:
                o = ordered[~nd.left]
                nd.left = ~first[id(o)]
                nd.right = len(o.prims)

    prims = [p for o in ordered for p in o.prims]
    aabbs = [o.aabb_min + o.aabb_max for o in ordered for _ in o.prims]
    fs.prims = prims
    n = len(prims)
    prim_type = np.array([p.type for p in prims], dtype=np.int32)
    prim_data = np.array([p.data for p in prims], dtype=np.float64).reshape(n, 5)
    prim_material = np.array([p.material for p in prims], dtype=np.int32)
    prim_id = np.array([(p.obj << 3) | p.side for p in prims], dtype=np.uint32)
    prim_instance = np.array([p.instance for p in prims], dtype=np.int32)
    prim_aabb = np.array(aabbs, dtype=np.float64).reshape(n, 6)
    prim_motion = np.array([p.motion if p.motion is not None else [0.0] * 5 for p in prims], dtype=np.float64).reshape(n, 5)

    c = fs.c
    c.n_prims = n
    c.prim_type = prim_type.ctypes.data_as(C.POINTER(C.c_int32))
    c.prim_data = prim_data.ctypes.data_as(C.POINTER(C.c_double))
    c.prim_material = prim_material.ctypes.data_as(C.POINTER(C.c_int32))
    c.prim_id = prim_id.ctypes.data_as(C.POINTER(C.c_uint32))
    c.prim_instance = prim_instance.ctypes.data_as(C.POINTER(C.c_int32))
    c.prim_aabb = prim_aabb.ctypes.data_as(C.POINTER(C.c_double))
    if any(p.motion is not None for p in prims):
        c.prim_motion = prim_motion.ctypes.data_as(C.POINTER(C.c_double))
    fs.keep += [prim_type, prim_data, prim_material, prim_id, prim_instance, prim_aabb, prim_motion]
    fs.np = dict(prim_type=prim_type, prim_data=prim_data, prim_material=prim_material, prim_id=prim_id,
                 prim_instance=prim_instance, prim_aabb=prim_aabb, prim_motion=prim_motion)

    def arr(ctype, items):
        a = (ctype * max(1, len(items)))(*items)
        fs.keep.append(a)
        return a

    c.n_instances, c.instances = len(instances), arr(rc_instance, instances)
    c.n_materials, c.materials = len(materials), arr(rc_material, materials)
    c.n_textures, c.textures = len(textures), arr(rc_texture, textures)
    c.n_perlin, c.perlin = len(perlins), arr(rc_perlin, perlins)
    c.n_nodes, c.nodes = len(nodes), arr(rc_bvh_node, nodes)
    imgs = []
    for (w, h, px) in images:
        im = rc_image()
        im.width, im.height = w, h
        im.rgba = px.ctypes.data_as(C.POINTER(C.c_uint8))
        fs.keep.append(px)
        imgs.append(im)
    c.n_images, c.images = len(imgs), arr(rc_image, imgs)
    fs.images = images
    fs.textures, fs.materials, fs.nodes, fs.instances = textures, materials, nodes, instances



def sandbox_additions(doc: dict):
    """Sandbox::load_cornell_box (src/scene/sandbox.rs:39-81) on top of the parsed cornell_box.yml: two white
    Lambertian boxes, each rotated about y and then translated (create_box / create_rotate_y / create_translate),
    black background, the Cornell camera.  Expressed as additions to the (lower-cased) YAML document, so that the
    ordinary YAML pathway (yml.rs:292-439) flattens them."""
    doc["textures"]["sandbox_white"] = {"solidcolor": {"color": {"color": [0.63, 0.63, 0.63]}}}
    doc["materials"]["sandbox_white"] = {"lambertian": {"texture": "sandbox_white"}}
    g = doc["geometry"]
    g["sandbox_box1"] = {"box": {"min": {"pos": [0.0, 0.0, 0.0]}, "max": {"pos": [165.0, 330.0, 165.0]}, "material": "sandbox_white"}}
    g["sandbox_box1_rotate"] = {"rotatey": {"key": "sandbox_box1", "degrees": 15.0}}
    g["sandbox_box1_translate"] = {"translate": {"key": "sandbox_box1", "pos": [265.0, 0.0, 295.0]}}
    g["sandbox_box2"] = {"box": {"min": {"pos": [0.0, 0.0, 0.0]}, "max": {"pos": [165.0, 165.0, 165.0]}, "material": "sandbox_white"}}
    g["sandbox_box2_rotate"] = {"rotatey": {"key": "sandbox_box2", "degrees": -18.0}}
    g["sandbox_box2_translate"] = {"translate": {"key": "sandbox_box2", "pos": [130.0, 0.0, 65.0]}}
    doc["background"] = {"solidcolor": {"pos": [0.0, 0.0, 0.0]}}
    doc["camera"] = {"vfov": 40.0, "aperture": 0.0, "focus_distance": 10000.0, "pos": {"pos": [278.0, 278.0, -800.0]},
                     "look_at": {"pos": [278.0, 278.0, 0.0]}}
    doc.pop("tone_map", None)


def load_scene(path: str, seed: int = 0, use_bvh: bool | None = None, image_dirs=(), additions=None) -> FlatScene:
    """YmlLoader::load + TryInto<SceneLoadData> (src/scene/yml.rs:43-47,173-458),
    followed by the flattening the Rust shim performs before rc_upload_scene."""
    with open(path, "r") as f:
        try:
            doc = yaml.safe_load(f)
        except yaml.YAMLError as e:
            raise SceneLoadError(f"Configuration({path}): {e}")
    if not isinstance(doc, dict):
        raise SceneLoadError(f"Configuration({path}): not a mapping")
    doc = _lower_keys(doc)
    if additions is not None:
        additions(doc)
    for req in ("textures", "materials", "geometry"):
        if req not in doc or not isinstance(doc[req], dict):
            raise SceneLoadError(f"Configuration({path}): missing field `{req}`")

    fs = FlatScene()
    textures: list[rc_texture] = []
    tex_index: dict[str, int] = {}
    images: list[tuple[int, int, np.ndarray]] = []
    perlins: list[rc_perlin] = []
    checkered = {}
    # textures: everything but Checkered first (yml.rs:177-210), in sorted key
    # order so that indices are deterministic (the reference uses a HashMap)
    for key in sorted(doc["textures"]):
        variant, f_ = _enum(doc["textures"][key], f"texture {key}")
        t = rc_texture()
        if variant == "checkered":
            checkered[key] = f_
            continue
        if variant == "solidcolor":
            t.type = capi.RC_TEX_SOLID
            t.color[:] = _vec3(f_.get("color"), f"texture {key}.color")
        elif variant == "image":
            t.type = capi.RC_TEX_IMAGE
            t.a = len(images)
            images.append(_load_image(str(f_["path"]), path, image_dirs))
        elif variant == "noise":
            t.type = capi.RC_TEX_NOISE
            t.a = len(perlins)
            t.b = int(f_["depth"])
            t.scale = float(f_["scale"])
            t.color[:] = _vec3(f_.get("color"), f"texture {key}.color")
            perlins.append(make_perlin(seed, t.a))
        else:
            raise SceneLoadError(f"Configuration({path}): unknown texture variant `{variant}`")
        tex_index[key] = len(textures)
        textures.append(t)
    for key in sorted(checkered):  # yml.rs:212-243
        f_ = checkered[key]
        ta, tb = str(f_["texture_a"]), str(f_["texture_b"])
        for name in (ta, tb):
            if name not in tex_index:
                raise SceneLoadError(f'Checkered texture "{key}" expected texture "{ta}" to exist.')
        t = rc_texture()
        t.type = capi.RC_TEX_CHECKER
        t.a, t.b = tex_index[ta], tex_index[tb]
        t.scale = 10.0  # checkered.rs:19
        tex_index[key] = len(textures)
        textures.append(t)

    materials: list[rc_material] = []
    mat_index: dict[str, int] = {}
    for key in sorted(doc["materials"]):  # yml.rs:245-286
        variant, f_ = _enum(doc["materials"][key], f"material {key}")
        m = rc_material()
        tex_key = f_.get("texture", f_.get("texture_key"))
        names = {"lambertian": (capi.RC_MAT_LAMBERTIAN, "lambertian"), "metal": (capi.RC_MAT_METAL, "metal"),
                 "diffuselight": (capi.RC_MAT_DIFFUSE_LIGHT, "diffuse light")}
        if variant in names:
            m.type = names[variant][0]
            if tex_key not in tex_index:
                raise SceneLoadError(
                    f'Failed to find texture "{tex_key}" for {names[variant][1]} material "{key}"')
            m.texture = tex_index[tex_key]
            if variant == "metal":
                m.param = float(f_["fuzz"])
        elif variant == "dialectric":
            m.type = capi.RC_MAT_DIELECTRIC
            m.param = float(f_["refraction_index"])
        else:
            raise SceneLoadError(f"Configuration({path}): unknown material variant `{variant}`")
        mat_index[key] = len(materials)
        materials.append(m)

    def mat(name):
        if name not in mat_index:
            raise SceneLoadError(f"UnknownMaterial({name})")
        return mat_index[name]

    objects: dict[str, TopObject] = {}
    rotations, translations = {}, {}
    for key in sorted(doc["geometry"]):  # yml.rs:292-399
        variant, f_ = _enum(doc["geometry"][key], f"geometry {key}")
        if variant == "sphere":
            pos, r = _vec3(f_, f"geometry {key}"), float(f_["radius"])
            lo, hi = _aabb([pos[i] - r for i in range(3)], [pos[i] + r for i in range(3)])  # sphere.rs:72-77
            objects[key] = TopObject(key, [Prim(capi.RC_PRIM_SPHERE, pos + [r, 0.0], mat(f_["material"]), 0)],
                                     lo, hi, pos)
        elif variant in ("xyrect", "xzrect", "yzrect"):
            kind = {"xyrect": capi.RC_PRIM_XY_RECT, "xzrect": capi.RC_PRIM_XZ_RECT, "yzrect": capi.RC_PRIM_YZ_RECT}[variant]
            names = {"xyrect": ("x0", "x1", "y0", "y1"), "xzrect": ("x0", "x1", "z0", "z1"),
                     "yzrect": ("y0", "y1", "z0", "z1")}[variant]
            a0, a1, b0, b1 = (float(f_[n]) for n in names)
            data, lo, hi, pos = _rect_prims(kind, a0, a1, b0, b1, float(f_["k"]))
            objects[key] = TopObject(key, [Prim(kind, data, mat(f_["material"]), 0)], lo, hi, pos)
        elif variant == "box":  # box.rs:21-77, geometry_creation.rs:98-106
            mn, mx, m = _vec3(f_["min"], "box.min"), _vec3(f_["max"], "box.max"), mat(f_["material"])
            sides = [(capi.RC_PRIM_XY_RECT, mn[0], mx[0], mn[1], mx[1], mx[2]),
                     (capi.RC_PRIM_XY_RECT, mn[0], mx[0], mn[1], mx[1], mn[2]),
                     (capi.RC_PRIM_XZ_RECT, mn[0], mx[0], mn[2], mx[2], mx[1]),
                     (capi.RC_PRIM_XZ_RECT, mn[0], mx[0], mn[2], mx[2], mn[1]),
                     (capi.RC_PRIM_YZ_RECT, mn[1], mx[1], mn[2], mx[2], mx[0]),
                     (capi.RC_PRIM_YZ_RECT, mn[1], mx[1], mn[2], mx[2], mn[0])]
            prims = [Prim(k, _rect_prims(k, a0, a1, b0, b1, kk)[0], m, 0, side=i)
                     for i, (k, a0, a1, b0, b1, kk) in enumerate(sides)]
            lo, hi = _aabb(mn, mx)
            objects[key] = TopObject(key, prims, lo, hi, mn)
        elif variant == "rotatey":
            rotations[str(f_["key"]).lower()] = float(f_["degrees"])
        elif variant == "translate":
            translations[str(f_["key"]).lower()] = _vec3(f_, f"geometry {key}")
        else:
            raise SceneLoadError(f"Configuration({path}): unknown geometry variant `{variant}`")
    # rotations first, then translations; each is keyed by its CHILD's name and
    # the wrapper takes that name (yml.rs:401-439, Q26)
    for child, deg in rotations.items():
        if child not in objects:
            raise SceneLoadError(f'Rotation_Y "{child}" did not have any child with key "{child}"')
        o = objects[child]
        o.rotate_deg = deg
        o.aabb_min, o.aabb_max = _rotate_y_aabb(o, deg)
    for child, off in translations.items():
        if child not in objects:
            raise SceneLoadError(f'Translation "{child}" did not have any child with key "{child}"')
        o = objects[child]
        o.translate = off
        o.aabb_min = [o.aabb_min[i] + off[i] for i in range(3)]  # translate.rs:44-47
        o.aabb_max = [o.aabb_max[i] + off[i] for i in range(3)]

    _flatten(fs, objects, textures, materials, images, perlins, use_bvh)
    c = fs.c

    # background, yml.rs:443-453; default Sky (background_color.rs:18-25)
    bg = doc.get("background")
    if bg is None:
        c.bg_type = capi.RC_BG_SKY
        c.bg_a[:] = [1.0, 1.0, 1.0]
        c.bg_b[:] = [0.5, 0.7, 1.0]
    else:
        variant, f_ = _enum(bg, "background")
        if variant == "sky":
            c.bg_type = capi.RC_BG_SKY
            c.bg_a[:] = _vec3(f_["top"], "sky.top")
            c.bg_b[:] = _vec3(f_["bottom"], "sky.bottom")
        elif variant == "solidcolor":
            c.bg_type = capi.RC_BG_SOLID
            c.bg_a[:] = _vec3(f_, "background")
        else:
            raise SceneLoadError(f"Configuration({path}): unknown background `{variant}`")
    fs.camera_cfg = doc.get("camera")
    fs.tone_map_cfg = doc.get("tone_map")
    return fs


TAG_SCENE = 3


class _SceneRng:
    """Sequential uniforms for procedural scenes: Philox4x32-10(counter = (n, 0, 0, TAG_SCENE << 24),
    key = seed), four 24-bit uniforms per block, consumed in order.  The reference draws from the
    OS-seeded thread_rng (src/util.rs:9-23), so its Random scene is different on every run."""

    def __init__(self, seed: int):
        self.key = (seed & MASK, (seed >> 32) & MASK)
        self.n, self.buf = 0, []

    def uniform(self) -> float:
        if not self.buf:
            self.buf = [u01(w) for w in philox4x32((self.n, 0, 0, TAG_SCENE << 24), self.key)]
            self.n += 1
        return self.buf.pop(0)

    def range(self, lo: float, hi: float) -> float:   # random_double_range, util.rs:19-23
        return lo + (hi - lo) * self.uniform()


def random_scene(seed: int = 0, use_bvh: bool | None = None) -> FlatScene:
    """Random::load (src/scene/random.rs:25-95): a checkered ground sphere, a 22 x 22 grid of small
    spheres (80 % diffuse MOVING spheres, 5 % metal, 15 % glass; skipped near (4, 0.2, 0)) and three
    large spheres; default Sky; camera vfov 20, aperture 0.1, focus 10, from (0, 2, 10) to the origin."""
    rng = _SceneRng(seed)
    fs = FlatScene()
    textures, materials, objects = [], [], {}

    def solid(rgb):
        t = rc_texture()
        t.type = capi.RC_TEX_SOLID
        t.color[:] = rgb
        textures.append(t)
        return len(textures) - 1

    def material(kind, texture=0, param=0.0):
        m = rc_material()
        m.type, m.texture, m.param = kind, texture, param
        materials.append(m)
        return len(materials) - 1

    def sphere(center, radius, mat, center_b=None):
        key = f"obj{len(objects):04d}"      # creation order == sorted key order
        lo, hi = _aabb([center[i] - radius for i in range(3)], [center[i] + radius for i in range(3)])
        prim = Prim(capi.RC_PRIM_SPHERE, list(center) + [radius, 0.0], mat, 0)
        if center_b is not None:   # create_movable_sphere, geometry_creation.rs:23-38; union box, moving_sphere.rs:90-99
            prim.type = capi.RC_PRIM_MOVING_SPHERE
            prim.motion = list(center_b) + [0.0, 1.0]
            lo2, hi2 = _aabb([center_b[i] - radius for i in range(3)], [center_b[i] + radius for i in range(3)])
            lo, hi = [min(lo[i], lo2[i]) for i in range(3)], [max(hi[i], hi2[i]) for i in range(3)]
        objects[key] = TopObject(key, [prim], lo, hi, list(center))

    even, odd = solid([0.2, 0.3, 0.1]), solid([0.9, 0.9, 0.9])
    chk = rc_texture()
    chk.type, chk.a, chk.b, chk.scale = capi.RC_TEX_CHECKER, even, odd, 10.0
    textures.append(chk)
    sphere([0.0, -1000.0, 0.0], 1000.0, material(capi.RC_MAT_LAMBERTIAN, len(textures) - 1))
    for a in range(-11, 11):
        for b in range(-11, 11):
            choose_mat = rng.uniform()
            center = [a + 0.9 * rng.uniform(), 0.2, b + 0.9 * rng.uniform()]
            if math.sqrt((center[0] - 4.0) ** 2 + (center[1] - 0.2) ** 2 + center[2] ** 2) > 0.9:
                if choose_mat < 0.8:      # diffuse, moving
                    c1 = [rng.uniform() for _ in range(3)]
                    c2 = [rng.uniform() for _ in range(3)]
                    albedo = [c1[i] * c2[i] for i in range(3)]
                    center2 = [center[0], center[1] + rng.range(0.0, 0.5), center[2]]
                    sphere(center, 0.2, material(capi.RC_MAT_LAMBERTIAN, solid(albedo)), center2)
                elif choose_mat > 0.95:   # metal
                    albedo = [rng.range(0.5, 1.0) for _ in range(3)]
                    fuzz = rng.range(0.0, 0.5)
                    sphere(center, 0.2, material(capi.RC_MAT_METAL, solid(albedo), fuzz))
                else:                     # glass
                    sphere(center, 0.2, material(capi.RC_MAT_DIELECTRIC, 0, 1.5))
    sphere([0.0, 1.0, 0.0], 1.0, material(capi.RC_MAT_DIELECTRIC, 0, 1.5))
    sphere([-4.0, 1.0, 0.0], 1.0, material(capi.RC_MAT_LAMBERTIAN, solid([0.4, 0.2, 0.1])))
    sphere([4.0, 1.0, 0.0], 1.0, material(capi.RC_MAT_METAL, solid([0.7, 0.6, 0.5]), 0.0))
    _flatten(fs, objects, textures, materials, [], [], use_bvh)
    c = fs.c
    c.bg_type = capi.RC_BG_SKY
    c.bg_a[:] = [1.0, 1.0, 1.0]
    c.bg_b[:] = [0.5, 0.7, 1.0]
    fs.camera_cfg = {"vfov": 20.0, "aperture": 0.1, "focus_distance": 10.0,
                     "pos": [0.0, 2.0, 10.0], "look_at": [0.0, 0.0, 0.0]}
    fs.tone_map_cfg = None
    return fs


def _rotate_y_aabb(o: TopObject, deg: float):
    """RotateY::create_bounding_box VERBATIM, including its two bugs
    (src/geometry/rotate_y.rs:68-90, Q14): `cos*x + sin + z`, and min/max
    shifted by pos inside the corner loop.  The result is the object's ray-cull
    volume (Q11), so it has to be reproduced, not corrected."""
    rad = deg * math.pi / 180.0
    s, c = math.sin(rad), math.cos(rad)
    fmax = 1.7976931348623157e308
    mn, mx = [fmax] * 3, [-fmax] * 3
    lo, hi, pos = o.aabb_min, o.aabb_max, o.pos
    for i in range(2):
        for j in range(2):
            for k in range(2):
                x = i * hi[0] + (1 - i) * lo[0]
                y = j * hi[1] + (1 - j) * lo[1]
                z = k * hi[2] + (1 - k) * lo[2]
                t = [c * x + s + z, y, -s * x + c * z]
                mn = [min(mn[a], t[a]) for a in range(3)]
                mx = [max(mx[a], t[a]) for a in range(3)]
                mn = [mn[a] + pos[a] for a in range(3)]
                mx = [mx[a] + pos[a] for a in range(3)]
    return _aabb(mn, mx)


def _build_bvh(objs, nodes, order):
    """Node::build (src/bvh_node.rs:31-82): sort by Aabb minimum on one axis,
    split at the median, leaves hold one object.  The reference picks the axis
    at random from {x, y} (Q10); here it is the axis with the widest spread of
    box minima (ties -> lowest axis), a stable sort keeps equal keys in
    canonical order.  Emits nodes in pre-order and objects in DFS leaf order."""
    idx = len(nodes)
    nd = rc_bvh_node()
    nodes.append(nd)
    if len(objs) == 1:
        o = objs[0]
        nd.bmin[:], nd.bmax[:] = o.aabb_min, o.aabb_max
        nd.left, nd.right = ~len(order), 1
        order.append(o)
        return idx
    spread = [max(o.aabb_min[a] for o in objs) - min(o.aabb_min[a] for o in objs) for a in range(3)]
    axis = max(range(3), key=lambda a: (spread[a], -a))
    objs = sorted(objs, key=lambda o: o.aabb_min[axis])
    mid = len(objs) // 2
    l = _build_bvh(objs[:mid], nodes, order)
    r = _build_bvh(objs[mid:], nodes, order)
    nd.left, nd.right = l, r
    for a in range(3):  # Aabb::from((&a, &b)), src/aabb.rs:95-114
        nd.bmin[a] = min(nodes[l].bmin[a], nodes[r].bmin[a])
        nd.bmax[a] = max(nodes[l].bmax[a], nodes[r].bmax[a])
    return idx


SAH_MIN_OBJECTS = 65   # smaller scenes keep the reference's median split (and with it their primitive order)


def _area(lo, hi):
    dx, dy, dz = hi[0] - lo[0], hi[1] - lo[1], hi[2] - lo[2]
    return 2.0 * (dx * dy + dy * dz + dz * dx)


def _build_bvh_sah(objs, nodes, order):
    """Surface-area-heuristic tree over the same leaves as _build_bvh (one top-level object each), for scenes
    large enough to be traced through the BVH: the closest hit does not depend on the tree (the images are
    identical), the number of boxes a ray visits does — the Random scene's ground sphere inflates every
    ancestor box of a median split.  `objs` = [(canonical index, object)].  Per node: for each axis, sort by
    box centre (ties: canonical index), sweep every split k and keep the first minimum of
    area(left) * k + area(right) * (m - k), axes in order x, y, z.  Same node / leaf-order output as
    _build_bvh; racer_host.cpp::build_bvh_sah is the same algorithm in the same arithmetic."""
    idx = len(nodes)
    nd = rc_bvh_node()
    nodes.append(nd)
    if len(objs) == 1:
        o = objs[0][1]
        nd.bmin[:], nd.bmax[:] = o.aabb_min, o.aabb_max
        nd.left, nd.right = ~len(order), 1
        order.append(o)
        return idx
    m = len(objs)
    best = None
    for axis in range(3):
        srt = sorted(objs, key=lambda e: (e[1].aabb_min[axis] + e[1].aabb_max[axis], e[0]))
        lo = np.minimum.accumulate(np.array([e[1].aabb_min for e in srt], dtype=np.float64), axis=0)
        hi = np.maximum.accumulate(np.array([e[1].aabb_max for e in srt], dtype=np.float64), axis=0)
        rlo = np.minimum.accumulate(np.array([e[1].aabb_min for e in srt[::-1]], dtype=np.float64), axis=0)[::-1]
        rhi = np.maximum.accumulate(np.array([e[1].aabb_max for e in srt[::-1]], dtype=np.float64), axis=0)[::-1]
        for k in range(1, m):
            cost = _area(lo[k - 1], hi[k - 1]) * k + _area(rlo[k], rhi[k]) * (m - k)
            if best is None or cost < best[0]:
                best = (cost, srt, k)
    _, srt, k = best
    l = _build_bvh_sah(srt[:k], nodes, order)
    r = _build_bvh_sah(srt[k:], nodes, order)
    nd.left, nd.right = l, r
    for a in range(3):
        nd.bmin[a] = min(nodes[l].bmin[a], nodes[r].bmin[a])
        nd.bmax[a] = max(nodes[l].bmax[a], nodes[r].bmax[a])
    return idx


def _load_image(rel: str, scene_path: str, image_dirs=()):
    """TextureImage::try_new (src/texture/image.rs:17-25): decode to RGBA8."""
    from PIL import Image
    cands = [rel, os.path.join(os.path.dirname(os.path.abspath(scene_path)), rel)]
    cands += [os.path.join(d, os.path.basename(rel)) for d in image_dirs]
    for p in cands:
        if os.path.exists(p):
            im = Image.open(p).convert("RGBA")
            px = np.ascontiguousarray(np.asarray(im, dtype=np.uint8))
            return im.width, im.height, px
    raise SceneLoadError(f"FailedToOpenImage({rel})")


# ---------------------------------------------------------------------------
# config.yml
# ---------------------------------------------------------------------------
@dataclass
class RenderConfig:  # src/config.rs:75-82
    samples: int = 0
    max_depth: int = 0
    num_threads_width: int = 0
    num_threads_height: int = 0
    scale: int = 0


@dataclass
class Config:  # src/config.rs:180-225
    preview: RenderConfig = field(default_factory=RenderConfig)
    render: RenderConfig = field(default_factory=RenderConfig)
    width: int = 0
    height: int = 0
    camera: dict = field(default_factory=dict)
    tone_map: object = "none"
    renderer: str = "cpu"
    gpu: dict = field(default_factory=dict)   # new optional block: seed, variant, sampler, split, devices


def load_config(path: str) -> Config:
    with open(path, "r") as f:
        doc = _lower_keys(yaml.safe_load(f) or {})
    cfg = Config()
    for name in ("preview", "render"):
        d = doc.get(name) or {}
        setattr(cfg, name, RenderConfig(**{k: int(d.get(k, 0)) for k in RenderConfig.__dataclass_fields__}))
    scr = doc.get("screen") or {}
    cfg.width, cfg.height = int(scr.get("width", 0)), int(scr.get("height", 0))
    cfg.camera = doc.get("camera") or {}
    cfg.tone_map = doc.get("tone_map", "none")
    r = doc.get("renderer", "cpu")
    cfg.renderer = _enum(r, "renderer")[0]
    cfg.gpu = doc.get("gpu") or {}
    return cfg


def default_config() -> Config:
    """The values of the reference's racer-tracer/config.yml."""
    cfg = Config()
    cfg.preview = RenderConfig(40, 10, 10, 10, 4)
    cfg.render = RenderConfig(200, 20, 10, 10, 1)
    cfg.width = cfg.height = 600
    cfg.camera = {"vfov": 40, "aperture": 0.0, "focus_distance": 10000,
                  "pos": {"pos": [278, 278, -800]}, "look_at": {"pos": [278, 278, 0]}}
    cfg.tone_map = {"aces": {"default": True}}
    return cfg


def merged_camera(scene_cam: dict | None, config_cam: dict | None) -> dict:
    """CameraData::merge (src/camera.rs:404-464): scene overrides config field
    by field; defaults vfov 20, aperture 0, focus 1000, pos 0, look_at -z."""
    a, b = scene_cam or {}, config_cam or {}

    def pick(k, default):
        v = a.get(k)
        if v is None:
            v = b.get(k)
        return default if v is None else v
    return {"vfov": float(pick("vfov", 20.0)), "aperture": float(pick("aperture", 0.0)),
            "focus_distance": float(pick("focus_distance", 1000.0)),
            "pos": _vec3(pick("pos", [0.0, 0.0, 0.0]), "camera.pos"),
            "look_at": _vec3(pick("look_at", [0.0, 0.0, -1.0]), "camera.look_at")}


def make_camera(cam: dict, width: int, height: int) -> rc_camera:
    """Camera::new (src/camera.rs:196-234) with scene_up = +y, time 0..1
    (src/main.rs:97-110)."""
    def sub(a, b): return [a[i] - b[i] for i in range(3)]
    def mul(a, s): return [a[i] * s for i in range(3)]
    def cross(a, b): return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]

    def unit(a):
        n = math.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])
        return [a[0] / n, a[1] / n, a[2] / n]
    aspect = width / height  # src/image.rs:12-16
    h = math.tan((cam["vfov"] * math.pi / 180.0) / 2.0)
    vh = 2.0 * h
    vw = aspect * vh
    frm, at, fd = cam["pos"], cam["look_at"], cam["focus_distance"]
    forward = unit(sub(frm, at))
    right = unit(cross([0.0, 1.0, 0.0], forward))
    up = cross(forward, right)
    horizontal = mul(right, fd * vw)
    vertical = mul(up, fd * vh)
    ulc = [frm[i] + vertical[i] / 2.0 - horizontal[i] / 2.0 - fd * forward[i] for i in range(3)]
    c = rc_camera()
    c.origin[:], c.upper_left_corner[:], c.forward[:], c.right[:], c.up[:] = frm, ulc, forward, right, up
    c.horizontal[:], c.vertical[:] = horizontal, vertical
    c.vfov, c.viewport_width, c.viewport_height = cam["vfov"], vw, vh
    c.lens_radius, c.focus_distance, c.time_a, c.time_b = cam["aperture"] * 0.5, fd, 0.0, 1.0
    return c


def make_tone_map(node) -> rc_tone_map:
    """From<&ToneMapConfig> for Box<dyn ToneMap> (src/tone_map.rs:18-66)."""
    tm = rc_tone_map()
    variant, f_ = _enum(node if node is not None else "none", "tone_map")
    f_ = f_ or {}
    tm.max_white = 25.0
    tm.hable[:] = [0.15, 0.5, 0.1, 0.2, 0.02, 0.3]
    tm.exposure_bias, tm.linear_white_point = 2.0, 11.2
    tm.aces_in[:] = [0.59719, 0.35458, 0.04823, 0.07600, 0.90834, 0.01566, 0.02840, 0.13383, 0.83777]
    tm.aces_out[:] = [1.60475, -0.53108, -0.07367, -0.10208, 1.10813, -0.00605, -0.00327, -0.07276, 1.07602]
    if variant == "reinhard":
        tm.type = capi.RC_TONE_REINHARD
        if f_.get("max_white") is not None:
            tm.max_white = float(f_["max_white"])
    elif variant == "hable":
        tm.type = capi.RC_TONE_HABLE
        for i, k in enumerate(("shoulder_strength", "linear_strength", "linear_angle", "toe_strength",
                               "toe_numerator", "toe_denominator")):
            if f_.get(k) is not None:
                tm.hable[i] = float(f_[k])
        if f_.get("exposure_bias") is not None:
            tm.exposure_bias = float(f_["exposure_bias"])
        if f_.get("linear_white_point") is not None:
            tm.linear_white_point = float(f_["linear_white_point"])
    elif variant == "aces":
        tm.type = capi.RC_TONE_ACES
        for name, dst in (("input_matrix", tm.aces_in), ("output_matrix", tm.aces_out)):
            m = f_.get(name)
            if m is not None:
                rows = [_vec3(r, name) for r in m["colors"]]
                dst[:] = [v for r in rows for v in r]
    elif variant == "none":
        tm.type = capi.RC_TONE_NONE
    else:
        raise SceneLoadError(f"unknown tone map `{variant}`")
    return tm


def make_params(width, height, samples, max_depth, seed=0, variant=capi.RC_VARIANT_MEGAKERNEL,
                sampler=capi.RC_SAMPLER_DIRECT, split=capi.RC_SPLIT_TILES, rank=0, world=1,
                fixed_jitter=0, tile_w=0, tile_h=0, rng_rounds=0, specialize=0) -> rc_params:
    p = rc_params()
    p.width, p.height, p.samples, p.max_depth, p.seed = width, height, samples, max_depth, seed
    p.variant, p.sampler, p.split, p.rank, p.world = variant, sampler, split, rank, world
    p.fixed_jitter, p.tile_w, p.tile_h, p.rng_rounds = fixed_jitter, tile_w, tile_h, rng_rounds
    p.specialize = specialize
    return p


def default_denoise(levels=5, sigma_l=4.0, sigma_n=128.0, sigma_z=1.0) -> capi.rc_denoise:
    """rc_denoise with SVGF's published parameters unless given."""
    return capi.rc_denoise(levels=levels, sigma_l=sigma_l, sigma_n=sigma_n, sigma_z=sigma_z)


def preview_scales(cfg: "Config", width: int, height: int) -> tuple[int, int]:
    """CpuRendererScaled::new (src/renderer/cpu_scaled.rs:17-43): the highest divisor of
    image.width / num_threads_width (height likewise) that does not exceed config.preview.scale."""
    def highest_divisible(value: int, div: int) -> int:
        while value % div != 0:
            div -= 1
        return div
    pv = cfg.preview
    return (highest_divisible(width // max(1, pv.num_threads_width), max(1, pv.scale)),
            highest_divisible(height // max(1, pv.num_threads_height), max(1, pv.scale)))


def with_bvh(job: "Job", nodes, prim_order) -> "Job":
    """A copy of `job` whose primitives are permuted by prim_order and whose BVH is `nodes` — the tree a
    GPU build (rc_build_lbvh / rc_get_bvh) produced — so the oracle traces the very same structure."""
    import copy
    fs, src = FlatScene(), job.scene
    fs.c = rc_scene.from_buffer_copy(src.c)
    fs.keep = list(src.keep)
    order = np.asarray(prim_order, dtype=np.int64)
    fs.np = {k: np.ascontiguousarray(v[order]) for k, v in src.np.items()}
    c = fs.c
    c.prim_type = fs.np["prim_type"].ctypes.data_as(C.POINTER(C.c_int32))
    c.prim_data = fs.np["prim_data"].ctypes.data_as(C.POINTER(C.c_double))
    c.prim_material = fs.np["prim_material"].ctypes.data_as(C.POINTER(C.c_int32))
    c.prim_id = fs.np["prim_id"].ctypes.data_as(C.POINTER(C.c_uint32))
    c.prim_instance = fs.np["prim_instance"].ctypes.data_as(C.POINTER(C.c_int32))
    c.prim_aabb = fs.np["prim_aabb"].ctypes.data_as(C.POINTER(C.c_double))
    if src.c.prim_motion:
        c.prim_motion = fs.np["prim_motion"].ctypes.data_as(C.POINTER(C.c_double))
    arr = (rc_bvh_node * max(1, len(nodes)))(*nodes)
    fs.keep.append(arr)
    c.n_nodes, c.nodes = len(nodes), arr
    fs.nodes = list(nodes)
    for name in ("images", "textures", "materials", "instances", "object_keys", "camera_cfg", "tone_map_cfg"):
        setattr(fs, name, getattr(src, name, None))
    out = copy.copy(job)
    out.scene = fs
    return out


def partition(params: rc_params, part: int, parts: int) -> dict:
    """rc_partition: the share of participant `part` of `parts` (host arithmetic only)."""
    lib = capi.load()
    out = (C.c_int32 * 8)()
    capi.check(lib, lib.rc_partition(C.byref(params), part, parts, out))
    keys = ("tile_first", "tile_stride", "n_tiles", "tiles_x", "tile_w", "tile_h", "s_begin", "s_end")
    return dict(zip(keys, [int(v) for v in out]))


def share_mask(params: rc_params, part: int, parts: int) -> np.ndarray:
    """Boolean (H, W) mask of the pixels participant `part` traces."""
    sh = partition(params, part, parts)
    mask = np.zeros((params.height, params.width), dtype=bool)
    for k in range(sh["n_tiles"]):
        tile = sh["tile_first"] + k * sh["tile_stride"]
        tx, ty = tile % sh["tiles_x"], tile // sh["tiles_x"]
        mask[ty * sh["tile_h"]:(ty + 1) * sh["tile_h"], tx * sh["tile_w"]:(tx + 1) * sh["tile_w"]] = True
    return mask


@dataclass
class Job:
    """Everything one Renderer::render call needs (RenderData, renderer.rs:92-99)."""
    scene: FlatScene
    camera: rc_camera
    tone_map: rc_tone_map
    config: Config
    width: int
    height: int


def prepare_job(scene_path: str, config: Config | None = None, width=None, height=None, seed=0,
                use_bvh=None, image_dirs=()) -> Job:
    """The wiring of src/main.rs:74-119 up to the point where render() is called."""
    cfg = config or default_config()
    w, h = width or cfg.width, height or cfg.height
    if scene_path == "random":      # SceneLoaderConfig::Random, config.rs:84-93
        fs = random_scene(seed=seed, use_bvh=use_bvh)
    elif scene_path.startswith("sandbox:"):   # SceneLoaderConfig::Sandbox over the given cornell_box.yml (sandbox.rs:41-42)
        fs = load_scene(scene_path[len("sandbox:"):], seed=seed, use_bvh=use_bvh, image_dirs=image_dirs, additions=sandbox_additions)
    else:
        fs = load_scene(scene_path, seed=seed, use_bvh=use_bvh, image_dirs=image_dirs)
    cam = make_camera(merged_camera(fs.camera_cfg, cfg.camera), w, h)
    tm = make_tone_map(fs.tone_map_cfg if fs.tone_map_cfg is not None else cfg.tone_map)  # main.rs:84-86
    return Job(fs, cam, tm, cfg, w, h)


# ---------------------------------------------------------------------------
# The renderer handle: a thin, loud wrapper over the C ABI
# ---------------------------------------------------------------------------
class _DevicePointer:
    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}


def device_view(ptr: int, n: int):
    """A torch view (no copy) of n floats of device memory the library owns, e.g. rc_render_frame's image."""
    import torch
    return torch.as_tensor(_DevicePointer(ptr, n), device="cuda")


class CudaRenderer:
    """Plays `impl Renderer for CudaRenderer` of the Rust shim (INTEGRATION.md):
    render(job, params) returns what CpuRenderer sends in BufferUpdate messages."""

    def __init__(self, devices=None):
        self.lib = capi.load()
        self.ctx = C.c_void_p()
        if devices is None:
            devices = [0]
        arr = (C.c_int32 * len(devices))(*devices)
        capi.check(self.lib, self.lib.rc_create(arr, len(devices), C.byref(self.ctx)))

    def close(self):
        if self.ctx:
            self.lib.rc_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int):
        capi.check(self.lib, self.lib.rc_set_stream(self.ctx, C.c_void_p(cuda_stream)))

    def upload(self, job: Job):
        capi.check(self.lib, self.lib.rc_upload_scene(self.ctx, job.scene.ptr))
        capi.check(self.lib, self.lib.rc_set_camera(self.ctx, C.byref(job.camera)))

    def build_lbvh(self):
        """rc_build_lbvh: rebuild the uploaded scene's BVH on the GPU (LBVH over Morton codes)."""
        capi.check(self.lib, self.lib.rc_build_lbvh(self.ctx))

    def get_bvh(self, n_prims: int):
        """rc_get_bvh -> (list of rc_bvh_node in pre-order, prim_order int32 array of length n_prims)."""
        n = self.lib.rc_get_bvh(self.ctx, None, 0, None, 0)
        if n < 0:
            capi.check(self.lib, n)
        nodes = (rc_bvh_node * max(1, n))()
        order = np.full(n_prims, -1, dtype=np.int32)
        got = self.lib.rc_get_bvh(self.ctx, nodes, n, order.ctypes.data_as(C.POINTER(C.c_int32)), n_prims)
        if got < 0:
            capi.check(self.lib, got)
        assert got == n and (order >= 0).all()
        return [nodes[i] for i in range(n)], order

    def render(self, params: rc_params, cancel=None, out: np.ndarray | None = None) -> np.ndarray:
        """rc_render into `out` ((H, W, 3) float64, C-contiguous; e.g. a pinned buffer) or a new array."""
        if out is None:
            out = np.empty((params.height, params.width, 3), dtype=np.float64)
        assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == params.height * params.width * 3
        cptr = C.cast(C.pointer(cancel), C.POINTER(C.c_int32)) if cancel is not None else None
        capi.check(self.lib, self.lib.rc_render(self.ctx, C.byref(params),
                                                out.ctypes.data_as(C.POINTER(C.c_double)), cptr))
        return out

    def render_adaptive(self, params: rc_params, threshold: float, min_samples: int, cancel=None):
        """rc_render_adaptive -> (rgb (H, W, 3) float64, spp (H, W) int32, err (H, W) float64): every pixel traces
        samples [0, n_p), n_p doubling from min_samples up to params.samples until its error estimate is <= threshold."""
        h, w = params.height, params.width
        rgb = np.empty((h, w, 3), dtype=np.float64)
        spp = np.empty((h, w), dtype=np.int32)
        err = np.empty((h, w), dtype=np.float64)
        a = capi.rc_adaptive()
        a.min_samples, a.threshold = min_samples, threshold
        cptr = C.cast(C.pointer(cancel), C.POINTER(C.c_int32)) if cancel is not None else None
        capi.check(self.lib, self.lib.rc_render_adaptive(self.ctx, C.byref(params), C.byref(a),
                                                         rgb.ctypes.data_as(C.POINTER(C.c_double)),
                                                         spp.ctypes.data_as(C.POINTER(C.c_int32)),
                                                         err.ctypes.data_as(C.POINTER(C.c_double)), cptr))
        return rgb, spp, err

    def render_denoised(self, params: rc_params, denoise: capi.rc_denoise | None = None, aux=False, cancel=None):
        """rc_render_denoised -> rgb (H, W, 3) float64, or (rgb, aux) with aux = the filter's inputs as the call built
        them: {"mean": (H, W, 3), "var": (H, W), "albedo": (H, W, 3), "normal": (H, W, 3), "depth": (H, W),
        "id": (H, W) uint32}.  denoise=None: SVGF's parameters (levels 5, sigma_l 4, sigma_n 128, sigma_z 1)."""
        h, w = params.height, params.width
        dn = denoise if denoise is not None else default_denoise()
        rgb = np.empty((h, w, 3), dtype=np.float64)
        arrays, aux_ptr = None, None
        if aux:
            arrays = {"mean": np.empty((h, w, 3)), "var": np.empty((h, w)), "albedo": np.empty((h, w, 3)),
                      "normal": np.empty((h, w, 3)), "depth": np.empty((h, w)), "id": np.empty((h, w), dtype=np.uint32)}
            a = capi.rc_denoise_aux()
            for k, v in arrays.items():
                setattr(a, k, v.ctypes.data_as(C.POINTER(C.c_uint32 if k == "id" else C.c_double)))
            aux_ptr = C.byref(a)
        cptr = C.cast(C.pointer(cancel), C.POINTER(C.c_int32)) if cancel is not None else None
        capi.check(self.lib, self.lib.rc_render_denoised(self.ctx, C.byref(params), C.byref(dn),
                                                         rgb.ctypes.data_as(C.POINTER(C.c_double)), aux_ptr, cptr))
        return (rgb, arrays) if aux else rgb

    def denoise_filter(self, mean, var, albedo, normal, depth, ids, denoise: capi.rc_denoise | None = None) -> np.ndarray:
        """rc_denoise_filter on host arrays shaped as render_denoised's aux -> rgb (H, W, 3) float64."""
        h, w = np.shape(var)
        dn = denoise if denoise is not None else default_denoise()
        f64 = [np.ascontiguousarray(x, dtype=np.float64) for x in (mean, var, albedo, normal, depth)]
        for x, shape in zip(f64, ((h, w, 3), (h, w), (h, w, 3), (h, w, 3), (h, w))):
            assert x.shape == shape, (x.shape, shape)
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        assert ids.shape == (h, w)
        rgb = np.empty((h, w, 3), dtype=np.float64)
        capi.check(self.lib, self.lib.rc_denoise_filter(
            self.ctx, C.byref(dn), w, h, *[x.ctypes.data_as(C.POINTER(C.c_double)) for x in f64],
            ids.ctypes.data_as(C.POINTER(C.c_uint32)), rgb.ctypes.data_as(C.POINTER(C.c_double))))
        return rgb

    def render_preview(self, params: rc_params, scale_w: int, scale_h: int, cancel=None) -> np.ndarray:
        """rc_render_preview: what CpuRendererScaled sends (cpu_scaled.rs); params = screen size + config.preview."""
        out = np.empty((params.height, params.width, 3), dtype=np.float64)
        cptr = C.cast(C.pointer(cancel), C.POINTER(C.c_int32)) if cancel is not None else None
        capi.check(self.lib, self.lib.rc_render_preview(self.ctx, C.byref(params), scale_w, scale_h,
                                                        out.ctypes.data_as(C.POINTER(C.c_double)), cptr))
        return out

    def render_accumulate(self, params: rc_params, d_accum_ptr: int):
        capi.check(self.lib, self.lib.rc_render_accumulate(self.ctx, C.byref(params),
                                                           C.c_void_p(d_accum_ptr), None))

    def render_tiles_into(self, params: rc_params, d_image_ptr: int):
        """rc_render_tiles_into: this participant's tiles STORED into a (possibly remote) frame buffer."""
        capi.check(self.lib, self.lib.rc_render_tiles_into(self.ctx, C.byref(params), C.c_void_p(d_image_ptr), None))

    def shared_alloc(self, nbytes: int):
        """rc_shared_alloc -> (device pointer, 64-byte IPC handle)."""
        ptr, handle = C.c_void_p(), (C.c_uint8 * 64)()
        capi.check(self.lib, self.lib.rc_shared_alloc(self.ctx, nbytes, C.byref(ptr), handle))
        return ptr.value, bytes(handle)

    def shared_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        capi.check(self.lib, self.lib.rc_shared_open(self.ctx, (C.c_uint8 * 64).from_buffer_copy(handle), C.byref(ptr)))
        return ptr.value

    def shared_close(self, ptr: int):
        capi.check(self.lib, self.lib.rc_shared_close(self.ctx, C.c_void_p(ptr)))

    # ---- the one-process-per-GPU tile split (rc_frame_* / rc_render_frame) ----
    def frame_create(self, width: int, height: int, world: int):
        """rank 0: -> (frame handle, 64-byte IPC handle for the other ranks)."""
        f, handle = C.c_void_p(), (C.c_uint8 * 64)()
        capi.check(self.lib, self.lib.rc_frame_create(self.ctx, width, height, world, C.byref(f), handle))
        return f.value, bytes(handle)

    def frame_open(self, handle: bytes, width: int, height: int, rank: int, world: int) -> int:
        f = C.c_void_p()
        capi.check(self.lib, self.lib.rc_frame_open(self.ctx, (C.c_uint8 * 64).from_buffer_copy(handle), width, height,
                                                    rank, world, C.byref(f)))
        return f.value

    def frame_close(self, frame: int):
        capi.check(self.lib, self.lib.rc_frame_close(self.ctx, C.c_void_p(frame)))

    def render_frame(self, params: rc_params, frame: int, want_device_ptr=False, out: np.ndarray | None = None, cancel=None):
        """rc_render_frame.  Rank 0: returns the device pointer of the finished float image (want_device_ptr) and / or
        fills `out` ((H, W, 3) float64, e.g. pinned); other ranks pass neither."""
        dptr = C.c_void_p()
        optr = None
        if out is not None:
            assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == params.height * params.width * 3
            optr = out.ctypes.data_as(C.POINTER(C.c_double))
        cptr = C.cast(C.pointer(cancel), C.POINTER(C.c_int32)) if cancel is not None else None
        capi.check(self.lib, self.lib.rc_render_frame(self.ctx, C.byref(params), C.c_void_p(frame),
                                                      C.byref(dptr) if want_device_ptr else None, optr, cptr))
        return dptr.value if want_device_ptr else None

    def finalize(self, d_accum_ptr: int, width: int, height: int, samples: int, d_rgb_ptr: int):
        capi.check(self.lib, self.lib.rc_finalize(self.ctx, C.c_void_p(d_accum_ptr), width, height,
                                                  samples, C.c_void_p(d_rgb_ptr)))

    def postprocess(self, tm: rc_tone_map, rgb: np.ndarray):
        h, w, _ = rgb.shape
        rgb = np.ascontiguousarray(rgb, dtype=np.float64)
        rgba = np.empty((h, w, 4), dtype=np.uint8)
        mapped = np.empty((h, w, 3), dtype=np.float64)
        capi.check(self.lib, self.lib.rc_postprocess(
            self.ctx, C.byref(tm), rgb.ctypes.data_as(C.POINTER(C.c_double)), w, h,
            rgba.ctypes.data_as(C.POINTER(C.c_uint8)), mapped.ctypes.data_as(C.POINTER(C.c_double))))
        return rgba, mapped

    def primary_aov(self, params: rc_params, precision=32):
        n = params.width * params.height
        ids = np.empty(n, dtype=np.uint32)
        t = np.empty(n, dtype=np.float64)
        nrm = np.empty((n, 3), dtype=np.float64)
        pt = np.empty((n, 3), dtype=np.float64)
        capi.check(self.lib, self.lib.rc_primary_aov(
            self.ctx, C.byref(params), precision, ids.ctypes.data_as(C.POINTER(C.c_uint32)),
            t.ctypes.data_as(C.POINTER(C.c_double)), nrm.ctypes.data_as(C.POINTER(C.c_double)),
            pt.ctypes.data_as(C.POINTER(C.c_double))))
        return ids, t, nrm, pt

    def fp32_peak(self):
        """(TFLOP/s, G lane-instr/s) of the FFMA micro-benchmark on device 0."""
        tf, gi = C.c_double(), C.c_double()
        capi.check(self.lib, self.lib.rc_fp32_peak(self.ctx, C.byref(tf), C.byref(gi)))
        return tf.value, gi.value

    def stats(self) -> capi.rc_stats:
        s = capi.rc_stats()
        capi.check(self.lib, self.lib.rc_get_stats(self.ctx, C.byref(s)))
        return s
