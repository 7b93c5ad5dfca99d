#!/usr/bin/env python
"""Builds racer_tracer_b200/rust_shim/patch/reference.diff: the patch a maintainer applies to the reference crate
(`cd racer-tracer && patch -p1 < reference.diff`) to get `renderer: Cuda` / `preview_renderer: CudaPreview`.

The patch = the two new source files kept under rust_shim/racer-tracer/src/ (flatten.rs, renderer/cuda.rs) + the
small edits to existing reference files listed in EDITS below (a method added to a trait, an `impl` of it per
type, two enum variants, one factory arm, one error variant).  The script copies the reference crate to a scratch
directory, applies the edits there (every anchor must occur exactly once), and writes `diff -ruN` of the two trees.
Nothing of the reference is stored in this repository except the context lines of that diff.
tests/test_rust_shim.py applies the result with `patch --dry-run` to the checkout RACER_TRACER_REFERENCE names.

No Rust toolchain exists in this image: the patch is checked to APPLY, not to compile.

    python tools/make_rust_patch.py [/root/reference/racer-tracer]
"""
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "racer_tracer_b200", "rust_shim")
NEW_FILES = ["src/flatten.rs", "src/renderer/cuda.rs"]

RECT = """    fn flatten(
        &self,
        obj: &crate::scene::SceneObject,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), crate::error::TracerError> {
        out.push_prim(
            top,
            side,
            wrap,
            racer_cuda_sys::%s,
            [self.%s, self.%s, self.%s, self.%s, self.k],
            None,
            &obj.material(),
        )
    }

"""

# (file, anchor, text, where): where = "after" (text goes after the anchor line block), "before", or "replace"
EDITS = [
    ("Cargo.toml", 'serde = { version = "1", features = ["derive"] }\n',
     'racer-cuda-sys = { path = "../racer-cuda-sys" }\n', "after"),
    ("src/main.rs", "mod error;\nmod aabb;\n", "mod flatten;\n", "after"),
    # ---- error: one new variant, exit code 23 (src/error.rs:71-97 maps variants to 1..22)
    ("src/error.rs", '    #[error("Failed to parse \\"{0}\\" into a vector: {1}")]\n    FailedToParse(String, String),\n',
     '\n    #[error("CUDA backend error {0}: {1}")]\n    CudaBackend(i32, String),\n', "after"),
    ("src/error.rs", "            TracerError::FailedToParse(_, _) => 22,\n",
     "            TracerError::CudaBackend(_, _) => 23,\n", "after"),
    # ---- config: two new renderer kinds (YAML: `renderer: Cuda`, `preview_renderer: CudaPreview`)
    ("src/config.rs", "    Cpu,\n    CpuPreview,\n", "    Cuda,\n    CudaPreview,\n", "after"),
    # ---- renderer factory
    ("src/renderer.rs", "pub mod cpu_scaled;\n", "pub mod cuda;\n", "after"),
    ("src/renderer.rs", "            RendererConfig::CpuPreview => Box::new(CpuRendererScaled::new(r.1.clone(), r.2)),\n",
     "            RendererConfig::Cuda => Box::new(cuda::CudaRenderer::new(r.1.clone())),\n"
     "            RendererConfig::CudaPreview => Box::new(cuda::CudaRendererScaled::new(r.1.clone(), r.2)),\n", "after"),
    # ---- camera: the 14 fields of CameraSharedData as the C struct (they are private to this module)
    ("src/camera.rs", "impl SharedCamera {\n",
     """impl CameraSharedData {
    /// include/racer_cuda.h `rc_camera`: the same 14 fields, Vec3 as [f64; 3]
    pub fn to_rc_camera(&self) -> racer_cuda_sys::rc_camera {
        use crate::flatten::v3;
        racer_cuda_sys::rc_camera {
            origin: v3(&self.origin),
            upper_left_corner: v3(&self.upper_left_corner),
            forward: v3(&self.forward),
            right: v3(&self.right),
            up: v3(&self.up),
            horizontal: v3(&self.horizontal),
            vertical: v3(&self.vertical),
            vfov: self.vfov,
            viewport_width: self.viewport_width,
            viewport_height: self.viewport_height,
            lens_radius: self.lens_radius,
            focus_distance: self.focus_distance,
            time_a: self.time_a,
            time_b: self.time_b,
        }
    }
}

""", "before"),
    # ---- Hittable: describe yourself + a generation counter (defaults: nothing, 0 = "always re-upload")
    ("src/geometry.rs", "    fn bounding_box(&self, time_a: f64, time_b: f64) -> &Aabb;\n",
     """
    /// Appends this hittable's primitives (and BVH nodes) to the flat scene of the CUDA backend.
    fn flatten(&self, _out: &mut crate::flatten::FlatScene) -> Result<(), crate::error::TracerError> {
        Ok(())
    }

    /// Changes whenever `flatten` would produce something else; 0 = unknown (flatten before every render).
    fn generation(&self) -> u64 {
        0
    }
""", "after"),
    # ---- scene objects
    ("src/scene.rs", "    fn update_pos(&mut self, pos_delta: &Vec3);\n}\n",
     """    fn update_pos(&mut self, pos_delta: &Vec3);
    /// Appends this geometry to the flat scene: `obj` is the SceneObject that owns it (position, material),
    /// `top` the top-level object (id, stored Aabb), `side` the face of a Boxx, `wrap` the wrappers above it.
    fn flatten(
        &self,
        obj: &SceneObject,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), TracerError>;
}
""", "replace"),
    ("src/scene.rs", "    pub fn aabb(&self) -> &Aabb {\n        &self.aabb\n    }\n}\n",
     """    pub fn aabb(&self) -> &Aabb {
        &self.aabb
    }

    /// This object as a TOP-LEVEL object of the flat scene (a leaf of the BVH).
    pub fn flatten_top(&self, out: &mut crate::flatten::FlatScene) -> Result<(), TracerError> {
        let top = crate::flatten::Top { id: self.obj_id, aabb: &self.aabb };
        self.hittable.flatten(self, &top, 0, &crate::flatten::Wrap::default(), out)
    }

    /// This object as a part of `top`: a face of a Boxx, the object inside a RotateY / Translate.
    pub fn flatten_as(
        &self,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), TracerError> {
        self.hittable.flatten(self, top, side, wrap, out)
    }
}
""", "replace"),
    # ---- the eight geometries
    ("src/geometry/sphere.rs", "impl HittableSceneObject for Sphere {\n",
     """    fn flatten(
        &self,
        obj: &SceneObject,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), crate::error::TracerError> {
        let c = obj.pos();
        out.push_prim(
            top,
            side,
            wrap,
            racer_cuda_sys::RC_PRIM_SPHERE,
            [*c.x(), *c.y(), *c.z(), self.radius, 0.0],
            None,
            &obj.material(),
        )
    }

""", "after"),
    ("src/geometry/moving_sphere.rs", "impl HittableSceneObject for MovingSphere {\n",
     """    fn flatten(
        &self,
        obj: &SceneObject,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), crate::error::TracerError> {
        if !wrap.is_none() {
            return Err(crate::flatten::unsupported("a moving sphere inside RotateY / Translate"));
        }
        let a = obj.pos();
        out.push_prim(
            top,
            side,
            wrap,
            racer_cuda_sys::RC_PRIM_MOVING_SPHERE,
            [*a.x(), *a.y(), *a.z(), self.radius, 0.0],
            Some([*self.pos_b.x(), *self.pos_b.y(), *self.pos_b.z(), self.time_a, self.time_b]),
            &obj.material(),
        )
    }

""", "after"),
    ("src/geometry/xy_rect.rs", "impl HittableSceneObject for XyRect {\n", RECT % ("RC_PRIM_XY_RECT", "x0", "x1", "y0", "y1"), "after"),
    ("src/geometry/xz_rect.rs", "impl HittableSceneObject for XzRect {\n", RECT % ("RC_PRIM_XZ_RECT", "x0", "x1", "z0", "z1"), "after"),
    ("src/geometry/yz_rect.rs", "impl HittableSceneObject for YzRect {\n", RECT % ("RC_PRIM_YZ_RECT", "y0", "y1", "z0", "z1"), "after"),
    ("src/geometry/box.rs", "impl HittableSceneObject for Boxx {\n",
     """    fn flatten(
        &self,
        _obj: &crate::scene::SceneObject,
        top: &crate::flatten::Top,
        _side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), crate::error::TracerError> {
        // six rectangles in Boxx::new order (+z, -z, +y, -y, +x, -x): the order Boxx::obj_hit tests them in
        for (i, side) in self.sides.iter().enumerate() {
            side.flatten_as(top, i as u32, wrap, out)?;
        }
        Ok(())
    }

""", "after"),
    ("src/geometry/rotate_y.rs", "impl HittableSceneObject for RotateY {\n",
     """    fn flatten(
        &self,
        _obj: &SceneObject,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), crate::error::TracerError> {
        if wrap.rotate.is_some() {
            return Err(crate::flatten::unsupported("RotateY inside RotateY"));
        }
        let mut inner = *wrap;
        inner.rotate = Some((self.sin_theta, self.cos_theta));
        self.object.flatten_as(top, side, &inner, out)
    }

""", "after"),
    ("src/geometry/translate.rs", "impl HittableSceneObject for Translate {\n",
     """    fn flatten(
        &self,
        _obj: &SceneObject,
        top: &crate::flatten::Top,
        side: u32,
        wrap: &crate::flatten::Wrap,
        out: &mut crate::flatten::FlatScene,
    ) -> Result<(), crate::error::TracerError> {
        // the C ABI takes a ray into object space as translate-then-rotate: Translate(RotateY(object))
        if !wrap.is_none() {
            return Err(crate::flatten::unsupported("Translate inside another wrapper"));
        }
        let mut inner = *wrap;
        inner.translate = Some(crate::flatten::v3(&self.offset));
        self.object.flatten_as(top, side, &inner, out)
    }

""", "after"),
    # ---- BVH: nodes in pre-order, leaves = runs of primitives; generation bumped on every rebuild
    ("src/bvh_node.rs", "impl From<&Node> for Aabb {\n",
     """impl Node {
    /// Pre-order `rc_bvh_node`s: an inner node's left child is the next node, `right` is the index of its right
    /// child; a leaf stores `!first_primitive` and the primitive count.  Returns this node's index.
    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<i32, TracerError> {
        use crate::flatten::v3;
        let index = out.nodes.len();
        out.nodes.push(racer_cuda_sys::rc_bvh_node::default());
        match self {
            Node::Leaf { obj } => {
                let first = out.n_prims();
                obj.flatten_top(out)?;
                let count = out.n_prims() - first;
                if count == 0 || count > 127 {
                    return Err(crate::flatten::unsupported("an object with no or more than 127 primitives"));
                }
                out.nodes[index] = racer_cuda_sys::rc_bvh_node {
                    bmin: v3(obj.aabb().min()),
                    bmax: v3(obj.aabb().max()),
                    left: !(first as i32),
                    right: count as i32,
                };
            }
            Node::Inner { left, right, aabb } => {
                left.flatten(out)?;
                let right_index = right.flatten(out)?;
                out.nodes[index] = racer_cuda_sys::rc_bvh_node {
                    bmin: v3(aabb.min()),
                    bmax: v3(aabb.max()),
                    left: index as i32 + 1,
                    right: right_index,
                };
            }
        }
        Ok(index as i32)
    }
}

""", "before"),
    ("src/bvh_node.rs", "    time_b: f64,\n    changed: bool,\n}\n",
     "    time_b: f64,\n    changed: bool,\n    generation: u64,\n}\n", "replace"),
    ("src/bvh_node.rs", "            time_b,\n            changed: true,\n        }\n",
     "            time_b,\n            changed: true,\n            generation: 1,\n        }\n", "replace"),
    ("src/bvh_node.rs", "        if self.changed {\n            self.node = Node::build(\n",
     "        if self.changed {\n            self.generation += 1;\n            self.node = Node::build(\n", "replace"),
    ("src/bvh_node.rs", "    fn bounding_box(&self, time_a: f64, time_b: f64) -> &Aabb {\n        self.node.bounding_box(time_a, time_b)\n    }\n",
     """
    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<(), TracerError> {
        self.node.flatten(out).map(|_| ())
    }

    fn generation(&self) -> u64 {
        self.generation
    }
""", "after"),
    # ---- materials
    ("src/material.rs", "    fn scatter(&self, ray: &Ray, hit_record: &HitRecord) -> Option<(Ray, Color)>;\n",
     "    /// This material as an `rc_material` (its texture is appended to `out` first).\n"
     "    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_material, crate::error::TracerError>;\n", "after"),
    ("src/material/lambertian.rs", "impl Material for Lambertian {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_material, crate::error::TracerError> {
        Ok(racer_cuda_sys::rc_material { type_: racer_cuda_sys::RC_MAT_LAMBERTIAN, texture: out.texture(&self.texture)?, param: 0.0 })
    }

""", "after"),
    ("src/material/metal.rs", "impl Material for Metal {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_material, crate::error::TracerError> {
        Ok(racer_cuda_sys::rc_material { type_: racer_cuda_sys::RC_MAT_METAL, texture: out.texture(&self.texture)?, param: self.fuzz })
    }

""", "after"),
    ("src/material/dialectric.rs", "impl Material for Dialectric {\n",
     """    fn flatten(&self, _out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_material, crate::error::TracerError> {
        Ok(racer_cuda_sys::rc_material { type_: racer_cuda_sys::RC_MAT_DIELECTRIC, texture: -1, param: self.refraction_index })
    }

""", "after"),
    ("src/material/diffuse_light.rs", "impl Material for DiffuseLight {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_material, crate::error::TracerError> {
        Ok(racer_cuda_sys::rc_material { type_: racer_cuda_sys::RC_MAT_DIFFUSE_LIGHT, texture: out.texture(&self.texture)?, param: 0.0 })
    }

""", "after"),
    # ---- textures
    ("src/texture.rs", "    fn value(&self, u: f64, v: f64, point: &Vec3) -> Color;\n",
     "    /// This texture as an `rc_texture` (children, image pixels and Perlin tables are appended to `out`).\n"
     "    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_texture, crate::error::TracerError>;\n", "after"),
    ("src/texture/solid_color.rs", "impl Texture for SolidColor {\n",
     """    fn flatten(&self, _out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_texture, crate::error::TracerError> {
        Ok(racer_cuda_sys::rc_texture { type_: racer_cuda_sys::RC_TEX_SOLID, color: crate::flatten::v3(&self.color), ..Default::default() })
    }

""", "after"),
    ("src/texture/checkered.rs", "impl Texture for Checkered {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_texture, crate::error::TracerError> {
        // value(): sines < 0 -> odd, else even (checkered.rs:33-42); rc_texture.a = even, .b = odd (the `sines < 0` branch)
        let (even, odd) = (out.texture(&self.even)?, out.texture(&self.odd)?);
        Ok(racer_cuda_sys::rc_texture { type_: racer_cuda_sys::RC_TEX_CHECKER, a: even, b: odd, scale: self.checker_size, ..Default::default() })
    }

""", "after"),
    ("src/texture/image.rs", "impl Texture for TextureImage {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_texture, crate::error::TracerError> {
        out.images.push((self.img.width() as i32, self.img.height() as i32, self.img.as_raw().clone()));
        Ok(racer_cuda_sys::rc_texture { type_: racer_cuda_sys::RC_TEX_IMAGE, a: (out.images.len() - 1) as i32, ..Default::default() })
    }

""", "after"),
    ("src/texture/noise.rs", "impl Texture for Noise {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) -> Result<racer_cuda_sys::rc_texture, crate::error::TracerError> {
        let mut table = racer_cuda_sys::rc_perlin { ran_vec: [[0.0; 3]; 256], perm_x: self.perlin.perm_x, perm_y: self.perlin.perm_y, perm_z: self.perlin.perm_z };
        for (dst, src) in table.ran_vec.iter_mut().zip(self.perlin.ran_vec.iter()) {
            *dst = crate::flatten::v3(src);
        }
        out.perlin.push(table);
        Ok(racer_cuda_sys::rc_texture {
            type_: racer_cuda_sys::RC_TEX_NOISE,
            a: (out.perlin.len() - 1) as i32,
            b: self.depth,
            reserved: 0,
            color: crate::flatten::v3(&self.color),
            scale: self.scale,
        })
    }

""", "after"),
    # ---- backgrounds
    ("src/background_color.rs", "    fn color(&self, ray: &Ray) -> Color;\n",
     "    /// bg_type / bg_a / bg_b of `rc_scene`.\n    fn flatten(&self, out: &mut crate::flatten::FlatScene);\n", "after"),
    ("src/background_color.rs", "impl BackgroundColor for Sky {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) {
        out.bg_type = racer_cuda_sys::RC_BG_SKY;
        out.bg_a = crate::flatten::v3(&self.top);
        out.bg_b = crate::flatten::v3(&self.bottom);
    }

""", "after"),
    ("src/background_color.rs", "impl BackgroundColor for SolidBackgroundColor {\n",
     """    fn flatten(&self, out: &mut crate::flatten::FlatScene) {
        out.bg_type = racer_cuda_sys::RC_BG_SOLID;
        out.bg_a = crate::flatten::v3(&self.color);
        out.bg_b = [0.0; 3];
    }

""", "after"),
]


def build(reference: str, out_path: str) -> str:
    tmp = tempfile.mkdtemp(prefix="rust_patch_")
    a, b = os.path.join(tmp, "a"), os.path.join(tmp, "b")
    keep = lambda d, names: [n for n in names if n in ("target", ".git", "Cargo.lock")]
    shutil.copytree(reference, a, ignore=keep)
    shutil.copytree(reference, b, ignore=keep)
    for rel, anchor, text, where in EDITS:
        path = os.path.join(b, rel)
        src = open(path).read()
        assert src.count(anchor) == 1, f"{rel}: anchor occurs {src.count(anchor)} times: {anchor!r}"
        new = {"after": anchor + text, "before": text + anchor, "replace": text}[where]
        open(path, "w").write(src.replace(anchor, new))
    for rel in NEW_FILES:
        os.makedirs(os.path.dirname(os.path.join(b, rel)), exist_ok=True)
        shutil.copy(os.path.join(SHIM, "racer-tracer", rel), os.path.join(b, rel))
    r = subprocess.run(["diff", "-ruN", "a", "b"], cwd=tmp, capture_output=True, text=True)
    assert r.returncode in (0, 1), r.stderr
    # stable header lines (no timestamps of the scratch copies)
    lines = []
    for ln in r.stdout.splitlines(keepends=True):
        if ln.startswith(("--- a/", "+++ b/", "--- /dev/null", "+++ /dev/null")):
            ln = ln.split("\t")[0].rstrip("\n") + "\n"
        lines.append(ln)
    open(out_path, "w").write("".join(lines))
    shutil.rmtree(tmp)
    return out_path


if __name__ == "__main__":
    ref = sys.argv[1] if len(sys.argv) > 1 else "/root/reference/racer-tracer"
    out = build(ref, os.path.join(SHIM, "patch", "reference.diff"))
    n = sum(1 for ln in open(out) if ln.startswith("+") and not ln.startswith("+++"))
    print(f"wrote {out}: {n} added lines over {len(EDITS)} edits + {len(NEW_FILES)} new files")
