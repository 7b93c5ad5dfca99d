// rt_scene.cuh — device-side scene layout and the per-ray building blocks:
// closest hit (linear list or threaded BVH), hit-record reconstruction,
// textures, materials and background.  Everything is templated on the scalar
// so the primary-visibility AOV can instantiate the very same intersectors in
// f64.  Reference citations are relative to /root/reference/racer-tracer/.
#pragma once
#include "rt_math.cuh"

// ---------------------------------------------------------------------------
// Layout.  A primitive is four 16-byte words (float4 / double4-as-2x):
//   a: sphere (cx, cy, cz, r)            rect (a0, a1, b0, b1)
//   b: sphere (|c|^2 - r^2, -, -, -)     rect (k, -, -, -);  b.y = material
//      parameter (fuzz / refraction index), b.z = packed kinds, b.w = texture
//      index (non-solid) or -1
//   c: (r, g, b) of a solid-colour texture (albedo or emission), c.w = bits of
//      the canonical object id
//   n: rect: the +axis unit normal (xy_rect.rs:45 etc.), so that the hit record
//      is formed with multiply-adds instead of per-type selects;  sphere: the
//      centre's velocity per unit of ray time, centre(time) = a.xyz + time * n.xyz
//      (MovingSphere::pos, moving_sphere.rs:37-39; 0 for a static sphere); n.w = material kind as a float
// packed kinds (b.z bits): [0:4) prim type, [4:8) material type, [8:12)
// texture type, [12:32) instance index + 1 (0 = none)
// ---------------------------------------------------------------------------
#define RT_PRIM_SPHERE 0
#define RT_PRIM_XY 1
#define RT_PRIM_XZ 2
#define RT_PRIM_YZ 3
#define RT_PRIM_MOVING 4        // moving sphere (moving_sphere.rs): a = centre at ray time 0, r; n = centre velocity
// spheres (static and moving) are the kinds whose low two bits are 0
#define RT_IS_SPHERE(type) (((type) & 3) == 0)
#define RT_MAT_LAMBERTIAN 0
#define RT_MAT_METAL 1
#define RT_MAT_DIELECTRIC 2
#define RT_MAT_LIGHT 3
#define RT_TEX_SOLID 0
#define RT_TEX_CHECKER 1
#define RT_TEX_IMAGE 2
#define RT_TEX_NOISE 3

// Which primitive kinds a scene contains (bit RT_PRIM_*).  A scene-specialised translation unit
// defines it; the precompiled kernels keep every kind.
#ifndef RT_SPEC_PRIMS
#define RT_SPEC_PRIMS 0xF
#endif
#ifndef RT_HAS_INSTANCES
#define RT_HAS_INSTANCES 1    /* a scene-specialised kernel sets 0 when nothing is rotated / translated */
#endif
#define RT_HAS_SPHERES (RT_SPEC_PRIMS & 1)
#define RT_HAS_RECTS (RT_SPEC_PRIMS & 0xE)

#define RT_MAX_CONST_PRIMS 40   // primitives kept in the kernel-parameter constant bank
#define RT_MAX_CONST_RECTS 8    // per axis group, fully unrolled with constant-bank operands
#define RT_MAX_CONST_OBJS 8     // instanced top-level objects (Box + RotateY / Translate) of the linear modes
#define RT_MAX_IMAGES 8
#define RT_T_MIN 0.001          // src/renderer.rs:58

struct DevPrim {      // fp32 primitive record, 64 B
    float4 a, b, c, n;
};

struct DevPrimD {     // f64 geometry of the same primitive (AOV f64 instantiation)
    double a[4];
    double k_or_cc;
    double motion[5];  // moving sphere: pos_b xyz, time_a, time_b
};

struct DevNode {      // threaded BVH node, pre-order; 32 B
    float4 lo;        // bmin.xyz, w = bits(skip index)
    float4 hi;        // bmax.xyz, w = bits(leaf: first | count << 24; inner: -1)
};

struct DevNodeD {
    double lo[3], hi[3];
    int skip, leaf;
};

struct DevTexture {   // 32 B
    int type, a, b;
    float scale;
    float4 color;
};

struct DevInstance {  // src/geometry/rotate_y.rs, translate.rs
    float sin_theta, cos_theta, ox, oy, oz;
    int flags;        // bit 0 rotate, bit 1 translate
};

struct DevInstanceD {
    double sin_theta, cos_theta, offset[3];
    int flags, pad;
};

template <typename T>
struct DevCamera {    // CameraSharedData, src/camera.rs:57-72 (the fields get_ray reads)
    Vec3T<T> origin, upper_left_corner, right, up, horizontal, vertical;
    T lens_radius, time_a, time_b;
};

// Kernel parameters: passed by value (constant bank), < 4 KB.
struct KParams {
    DevCamera<float> cam;
    float4 bg_a, bg_b;          // background colours; bg_a.w = bits(bg type)
    int width, height;          // the grid of traced pixels (preview: the grid of scaled blocks)
    float inv_wm1, inv_hm1;     // 1/(W-1), 1/(H-1) of the SCREEN (cpu.rs:35-40 divide by W-1 and H-1)
    float wm1;                  // (float)(screen width - 1)
    float4 vstep;               // cam.vertical / ((H - 1) * 65536): what one unit of the 16-bit v jitter adds to a ray direction
    int px_scale_x, px_scale_y; // screen pixels per traced pixel: 1 for a full render; the preview renderer's
                                // scale_width / scale_height (cpu_scaled.rs:31-34) otherwise
    int s_begin, s_end;         // sample range traced by this launch
    int max_depth;
    int fixed_jitter;
    uint32_t key;               // Philox2x32 key = seed_lo ^ seed_hi
    uint32_t ks[10];            // its key schedule: key + r * 0x9E3779B9
    int tile_first, tile_stride, n_tiles;   // interleaved tile partition
    int overwrite;              // 1: pixel sums are STORED (rc_render_tiles_into: a buffer shared by several GPUs,
                                // every pixel owned by one of them); 0: added to the accumulation buffer
    float final_scale;          // != 0: what is stored is sqrt(final_scale * sum), Vec3::scale_sqrt folded into the store
                                // (rc_render_frame: the pixel goes straight into the finished image); needs overwrite
    int slices;                 // > 1: every tile's sample range is cut into this many CTAs (few tiles per GPU)
    int slice_halving;          // slice lengths: 0 = linearly decreasing (S, S-1, .., 1), 1 = halving (n/2, n/4, .., last two equal)
    float* slice_buf;           // [slices][n_tiles * 128][3] partial sums, reduced in slice order afterwards
    int tiles_x, tile_w, tile_h;
    int n_prims, n_nodes;
    int lin_end[4];             // type-sorted linear table: [0,lin_end[0]) spheres, then xy, xz, yz rects
    int n_perlin;
    int checker_depth;          // checker levels of the longest texture chain (rc_upload_scene rejects cycles)
    int lens_enabled;
    int tile_cull;              // 1: a CTA first asks whether its tile's primary rays can hit anything at all (pinhole
                                // camera, nothing moves, linear modes); if not, its samples are background only
    int has_motion;             // the scene has a moving sphere: primary rays carry a time (camera.rs:335)
    int ref_aabb;               // scenes with RotateY: BVH culling uses the reference's per-axis Aabb::hit
    const DevPrim* prims;       // all primitives, BVH depth-first order (global memory)
    const DevPrim* prims_lin;   // the same primitives sorted by type (linear modes)
    const DevNode* nodes;       // threaded BVH (global memory)
    const DevTexture* textures;
    const DevInstance* instances;
    const float4* perlin;       // n_perlin x 256 gradients (xyz, w unused)
    const uint8_t* perlin_perm; // n_perlin x 3 x 256
    cudaTextureObject_t images[RT_MAX_IMAGES];
    int image_w[RT_MAX_IMAGES], image_h[RT_MAX_IMAGES];
    unsigned long long* segment_counter;
    const int* cancel_flag;     // NULL, or a word in this device's memory: every CTA reads it once before it starts and leaves
                                // at once when it is set (the host's cancel flag relayed by rc_render, renderer.rs:25-30)
    DevPrim cprims[RT_MAX_CONST_PRIMS];   // type-sorted copy for the linear constant-bank path
    // rectangles of the constant-bank path once more, split by plane axis so that the
    // unrolled tests address them with compile-time offsets (operands straight from the
    // constant bank, no load instructions): group 0 = xy, 1 = xz, 2 = yz
    float4 crect_bounds[3][RT_MAX_CONST_RECTS];   // (centre a, half extent a, centre b, half extent b)
    float crect_k[3][RT_MAX_CONST_RECTS];
    // Instanced top-level objects of the linear modes (the reference's default Sandbox scene: Cornell + two
    // rotated, translated boxes).  Their primitives follow the four type groups in the linear table.  The
    // stored Aabb is the object's cull volume (bvh_node.rs:119; RotateY's is not a bounding box, Q14), tested
    // exactly as Aabb::hit does before the ray is taken into the object's space.
    int n_cobj;
    float4 cobj_lo[RT_MAX_CONST_OBJS];   // Aabb min, w = bits(first primitive in the linear table)
    float4 cobj_hi[RT_MAX_CONST_OBJS];   // Aabb max, w = bits(primitive count | instance index << 8)
    DevInstance cinst[RT_MAX_CONST_OBJS];
};

// ---------------------------------------------------------------------------
// Scene accessors.  ConstScene reads primitives from the kernel parameters
// (uniform addresses in the linear loop -> constant-bank operands, no load
// instructions); SmemScene reads primitives and nodes staged in shared
// memory; GlobalScene reads them through the read-only path.
// ---------------------------------------------------------------------------
// 16-byte load from a 32-bit shared-memory address (computed once per kernel: the generic-to-shared
// conversion otherwise costs three uniform instructions at every use inside the path loop)
RT_D float4 lds128(unsigned addr) {
    float4 v;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

struct ConstScene {
    const KParams& P;
    unsigned sh;   // shared-memory address of the same type-sorted table, staged per CTA: per-lane (divergent) indices
    RT_D ConstScene(const KParams& p, const DevPrim* staged) : P(p), sh((unsigned)__cvta_generic_to_shared(staged)) {}
    RT_D ConstScene(const KParams& p, unsigned staged_addr) : P(p), sh(staged_addr) {}
    // uniform index (the intersection loops): constant-bank operands
    RT_D float4 ua(int i) const { return P.cprims[i].a; }
    RT_D float4 ub(int i) const { return P.cprims[i].b; }
    RT_D float4 un(int i) const { return P.cprims[i].n; }
    // per-lane index (hit record, shading): shared memory — an indexed constant load replays
    // once per distinct address in the warp
    RT_D float4 pa(int i) const { return lds128(sh + 64u * (unsigned)i); }
    RT_D float4 pb(int i) const { return lds128(sh + 64u * (unsigned)i + 16u); }
    RT_D float4 pc(int i) const { return lds128(sh + 64u * (unsigned)i + 32u); }
    RT_D float4 pn(int i) const { return lds128(sh + 64u * (unsigned)i + 48u); }
    RT_D float4 nlo(int) const { return make_float4(0.f, 0.f, 0.f, 0.f); }  // no BVH in the constant bank
    RT_D float4 nhi(int) const { return make_float4(0.f, 0.f, 0.f, 0.f); }
    RT_D const DevInstance* instances() const { return P.cinst; }           // the scene's instance table (<= RT_MAX_CONST_OBJS)
    RT_D bool reference_aabb() const { return false; }
};

struct PtrScene {  // shared or global, decided by where the pointers point
    const DevPrim* prims;
    const DevNode* nodes;
    const DevInstance* inst;   // RotateY / Translate table (global memory), may be null
    int ref_aabb;              // 1: cull with the reference's per-axis Aabb::hit (scenes with RotateY, Q11/Q14)
    RT_D const DevInstance* instances() const { return inst; }
    RT_D bool reference_aabb() const { return ref_aabb != 0; }
    RT_D float4 ua(int i) const { return prims[i].a; }
    RT_D float4 ub(int i) const { return prims[i].b; }
    RT_D float4 un(int i) const { return prims[i].n; }
    RT_D float4 pa(int i) const { return prims[i].a; }
    RT_D float4 pb(int i) const { return prims[i].b; }
    RT_D float4 pc(int i) const { return prims[i].c; }
    RT_D float4 pn(int i) const { return prims[i].n; }
    RT_D float4 nlo(int i) const { return nodes[i].lo; }
    RT_D float4 nhi(int i) const { return nodes[i].hi; }
};

RT_D int kinds_prim(float packed) { return __float_as_int(packed) & 15; }
RT_D int kinds_mat(float packed) { return (__float_as_int(packed) >> 4) & 15; }
RT_D int kinds_tex(float packed) { return (__float_as_int(packed) >> 8) & 15; }
RT_D int kinds_inst(float packed) { return (int)((unsigned)__float_as_int(packed) >> 12) - 1; }

// ---------------------------------------------------------------------------
// Primitive tests.  `self` marks the primitive the ray starts on.
//
// fp32 adaptation of the reference's f64 behaviour (DESIGN.md "fp32"): in f64
// a scattered ray re-tests the surface it leaves and finds the root t ~ 1e-13,
// which t_min = 0.001 rejects (src/renderer.rs:58).  In fp32 the origin sits
// up to ~1e-4 off the surface, so that root can exceed t_min at grazing
// angles.  We therefore give the departed primitive the limit the f64 code
// converges to: a sphere is solved with c = |oc|^2 - r^2 = 0 exactly (roots 0
// and -2b/a), and a rectangle's hit point is snapped onto its plane so that
// the re-test yields t = (k - o_n)/d_n = 0 exactly, below t_min.
// ---------------------------------------------------------------------------

// src/geometry/sphere.rs:39-58.  Returns the accepted root or -1.
//
// Two fp32-robust evaluations of the same quadratic (SURVEY H3), picked per ray:
//   far from the sphere (|oc|^2 > 2.6 r^2): the discriminant is formed from
//     l = oc - (b/a) d, the centre-to-ray vector, as a (r^2 - |l|^2) — no
//     b^2 - a c cancellation for small spheres seen from far away (clown);
//   near or inside it: c = |o|^2 - 2 o.ctr + (|ctr|^2 - r^2) with the last
//     term precomputed in f64 on the host — no |oc|^2 - r^2 cancellation for
//     the radius-1000 ground spheres seen from just above their surface.
// Both use the stable root formula q = -(b + sign(b) sqrt(disc)); t = q/a, c/q.
#define RT_SPHERE_FAR_RATIO 2.6f
template <typename T>
RT_D T sphere_hit(Vec3T<T> o, Vec3T<T> d, T a, T inv_a, Vec3T<T> ctr, T radius, T cc, bool self, T t_min, T t_max, bool use_cc = true) {
    Vec3T<T> oc = o - ctr;
    T b = dot(oc, d);  // half_b
    T oc2 = dot(oc, oc), r2 = radius * radius;
    T c, disc;
    if (oc2 > T(RT_SPHERE_FAR_RATIO) * r2) {
        T ba = b * inv_a;
        Vec3T<T> l = mk3<T>(oc.x - ba * d.x, oc.y - ba * d.y, oc.z - ba * d.z);
        disc = a * (r2 - dot(l, l));
        c = oc2 - r2;
    } else {
        // a moving sphere has no precomputed |ctr|^2 - r^2; its radius is small against its distance
        // from the origin only when oc is small too, so |oc|^2 - r^2 is the accurate form there
        Vec3T<T> o2 = mk3<T>(o.x - T(2) * ctr.x, o.y - T(2) * ctr.y, o.z - T(2) * ctr.z);
        c = self ? T(0) : (use_cc ? dot(o, o2) + cc : oc2 - r2);
        disc = b * b - a * c;
    }
    if (!(disc >= T(0))) return T(-1);
    T s = rt_sqrt(disc);
    T q = b < T(0) ? (s - b) : -(b + s);
    T r_qa = q * inv_a;
    T r_cq = c * rt_rcp(q);
    T near_root = b < T(0) ? r_cq : r_qa;
    T far_root = b < T(0) ? r_qa : r_cq;
    // "nearest root that lies in the acceptable range", sphere.rs:51-58
    if (near_root >= t_min && near_root <= t_max) return near_root;
    if (far_root >= t_min && far_root <= t_max) return far_root;
    return T(-1);
}

// Outward normal (p - ctr)/r of an accepted sphere hit (sphere.rs:61), formed
// from small-magnitude vectors so that it keeps fp32 precision for small
// spheres far from the origin: (l -+ (sqrt(disc)/a) d)/r in the far case,
// (oc + t d)/r otherwise.
RT_D vec3f sphere_normal(vec3f o, vec3f d, float a, float inv_a, vec3f ctr, float radius, float t) {
    vec3f oc = o - ctr;
    float oc2 = dot(oc, oc), r2 = radius * radius;
    float inv_r = fast_rcp(radius);
    if (oc2 > RT_SPHERE_FAR_RATIO * r2) {
        float b = dot(oc, d);
        float ba = b * inv_a;
        vec3f l = mk3(oc.x - ba * d.x, oc.y - ba * d.y, oc.z - ba * d.z);
        float h = fast_sqrt(fmaxf(0.0f, (r2 - dot(l, l)) * inv_a));   // |t - t_closest|
        float dt = (t < -ba) ? -h : h;                            // near or far root
        return mk3((l.x + dt * d.x) * inv_r, (l.y + dt * d.y) * inv_r, (l.z + dt * d.z) * inv_r);
    }
    return mk3((oc.x + t * d.x) * inv_r, (oc.y + t * d.y) * inv_r, (oc.z + t * d.z) * inv_r);
}

// src/geometry/xy_rect.rs:29-41 (and xz_rect.rs, yz_rect.rs): plane distance,
// range test, inclusive bounds test.  Returns t or -1.
template <typename T>
RT_D T rect_hit(int type, Vec3T<T> o, Vec3T<T> d, Vec3T<T> inv_d, T a0, T a1, T b0, T b1, T k, T t_min, T t_max) {
    T on, in, oa, da, ob, db;
    if (type == RT_PRIM_XY) { on = o.z; in = inv_d.z; oa = o.x; da = d.x; ob = o.y; db = d.y; }
    else if (type == RT_PRIM_XZ) { on = o.y; in = inv_d.y; oa = o.x; da = d.x; ob = o.z; db = d.z; }
    else { on = o.x; in = inv_d.x; oa = o.y; da = d.y; ob = o.z; db = d.z; }
    T t = (k - on) * in;
    if (!(t >= t_min && t <= t_max)) return T(-1);
    T pa = oa + t * da, pb = ob + t * db;
    if (pa < a0 || pa > a1 || pb < b0 || pb > b1) return T(-1);
    return t;
}

template <typename T>
struct RayT {
    Vec3T<T> o, d, inv_d;
    T time;   // Ray::time (src/ray.rs), read by moving spheres only
};

template <typename T>
RT_D RayT<T> make_ray(Vec3T<T> o, Vec3T<T> d, T time = T(0)) {
    RayT<T> r;
    r.o = o; r.d = d; r.time = time;
    r.inv_d = mk3<T>(rt_rcp(d.x), rt_rcp(d.y), rt_rcp(d.z));
    return r;
}

// Ray into the space of an instanced object: Translate is the outer wrapper (the ray moves by
// -offset, translate.rs:32), RotateY the inner one (rotate_y.rs:38-47).  t is preserved.
RT_D RayT<float> to_local(const DevInstance& in, const RayT<float>& r) {
    vec3f o = r.o, d = r.d;
    if (in.flags & 2) o = mk3(o.x - in.ox, o.y - in.oy, o.z - in.oz);
    if (in.flags & 1) {
        const float s = in.sin_theta, c = in.cos_theta;
        o = mk3(c * o.x - s * o.z, o.y, s * o.x + c * o.z);
        d = mk3(c * d.x - s * d.z, d.y, s * d.x + c * d.z);
    }
    return make_ray(o, d, r.time);
}

// centre of a (possibly moving) sphere at the ray's time
RT_D vec3f sphere_centre(float4 a, float4 n, float time) {
    return mk3(fmaf(time, n.x, a.x), fmaf(time, n.y, a.y), fmaf(time, n.z, a.z));
}

// One primitive of the fp32 tables against a ray already in the primitive's space; returns t or -1.
template <class Scene>
RT_D float prim_test_local(const Scene& S, int i, float4 a, float4 b, const RayT<float>& r, bool self, bool instanced, float t_max) {
    int type = kinds_prim(b.z);
    if (RT_HAS_SPHERES && (!RT_HAS_RECTS || RT_IS_SPHERE(type))) {
        const float aa = dot(r.d, r.d);
        const bool moving = type == RT_PRIM_MOVING;
        const vec3f ctr = moving ? sphere_centre(a, S.pn(i), r.time) : mk3(a.x, a.y, a.z);
        return sphere_hit<float>(r.o, r.d, aa, fast_rcp(aa), ctr, a.w, b.x, self, (float)RT_T_MIN, t_max, !moving);
    }
    // an instanced rectangle's hit point goes through a rotation before it becomes the next
    // origin, so it is not exactly on the plane any more: the rectangle a ray leaves is skipped
    if (self && instanced) return -1.0f;
    return rect_hit<float>(type, r.o, r.d, r.inv_d, a.x, a.y, a.z, a.w, b.x, (float)RT_T_MIN, t_max);
}

// One primitive against a world-space ray (SceneObject::hit, src/scene.rs:98-101).
template <class Scene>
RT_D float prim_test(const Scene& S, int i, const RayT<float>& r, int last_prim, float t_max) {
    float4 a = S.pa(i), b = S.pb(i);
    const int inst = kinds_inst(b.z);
    if (inst >= 0) {
        const RayT<float> lr = to_local(S.instances()[inst], r);
        return prim_test_local(S, i, a, b, lr, i == last_prim, true, t_max);
    }
    return prim_test_local(S, i, a, b, r, i == last_prim, false, t_max);
}

#define RT_NO_HIT 3.0e38f   /* closest-hit distances start here; +inf marks "no candidate" */

// Candidate distance of one axis-aligned rectangle: t when the in-plane hit point lies inside
// the rectangle and t >= t_min; +inf otherwise.  The bounds test a0 <= pa <= a1 (xy_rect.rs:36-38)
// is evaluated as |pa - ca| <= ha with ca = (a0 + a1)/2, ha = (a1 - a0)/2 formed in f64 on the
// host: one FADD (FMA pipe) + one compare with |.| per axis instead of two compares — the ALU
// pipe (compares, selects, logic) is the saturated one in this kernel (profiles/).  `xa`, `xb`
// are the hit coordinates already relative to the centre.  Three chained setp + one selp.
//
// No "is this the rectangle the ray leaves" test is needed: make_hit() snaps the hit point
// onto the plane, so for that rectangle k - o_n is exactly 0 and t = (k - o_n) * (1/d_n) is 0
// (or NaN when d_n = 0) — rejected by t >= t_min exactly as the reference's 1e-13 is.
RT_D float rect_candidate(float t, float xa, float xb, float ha, float hb) {
    asm("{\n\t.reg .pred p;\n\t"
        "setp.le.f32 p, %1, %3;\n\t"
        "setp.le.and.f32 p, %2, %4, p;\n\t"
        "setp.ge.and.f32 p, %0, 0f3A83126F, p;\n\t"   /* t >= 0.001f */
        "selp.f32 %0, %0, 0f7F800000, p;\n\t}"
        : "+f"(t) : "f"(fabsf(xa)), "f"(fabsf(xb)), "f"(ha), "f"(hb));
    return t;
}

// rect_candidate() and the closest-hit update in one predicate chain (scene-specialised kernels): if the
// rectangle is hit (bounds, t >= t_min) and t <= best_t, it becomes the best hit — `<=`: a later rectangle
// wins an exact tie (sphere.rs:53 / shared_scene.rs:37-53).  Four compares and two predicated moves per
// rectangle (ptxas turns the moves into selects: 6 instructions against 7 for rect_candidate + the select
// reduction).  Packing the index into the low mantissa bits of t would make the update one predicated FMNMX
// (5 instructions) at the price of 3 bits of t; not taken.
RT_D void rect_closest(float t, float xa, float xb, float ha, float hb, int index, float& best_t, int& best) {
    asm("{\n\t.reg .pred p;\n\t"
        "setp.le.f32 p, %2, %4;\n\t"
        "setp.le.and.f32 p, %3, %5, p;\n\t"
        "setp.ge.and.f32 p, %6, 0f3A83126F, p;\n\t"   /* t >= 0.001f */
        "setp.le.and.f32 p, %6, %0, p;\n\t"
        "@p mov.f32 %0, %6;\n\t"
        "@p mov.s32 %1, %7;\n\t}"
        : "+f"(best_t), "+r"(best) : "f"(fabsf(xa)), "f"(fabsf(xb)), "f"(ha), "f"(hb), "f"(t), "r"(index));
}

// The same update with the two conditional moves done by PREDICATED FFMAs (best = t * 1 + 0, index = index * 0 +
// i as a float): four compares on the ALU pipe and two instructions on the FMA pipe, which has room, instead of
// four compares + two selects on the ALU pipe, which is the saturated one.  `best_index` carries the index as a
// float (-1 = none).  t > 0 here, so t * 1 + 0 is t exactly.
RT_D void rect_closest_fma(float t, float xa, float xb, float ha, float hb, float index, float& best_t, float& best_index) {
    asm("{\n\t.reg .pred p;\n\t"
        "setp.le.f32 p, %2, %4;\n\t"
        "setp.le.and.f32 p, %3, %5, p;\n\t"
        "setp.ge.and.f32 p, %6, 0f3A83126F, p;\n\t"   /* t >= 0.001f */
        "setp.le.and.f32 p, %6, %0, p;\n\t"
        "@p fma.rn.f32 %0, %6, 0f3F800000, 0f00000000;\n\t"
        "@p fma.rn.f32 %1, %1, 0f00000000, %7;\n\t}"
        : "+f"(best_t), "+f"(best_index) : "f"(fabsf(xa)), "f"(fabsf(xb)), "f"(ha), "f"(hb), "f"(t), "f"(index));
}

// The FIRST test of a generated closest hit: nothing has been hit yet (best_t = RT_NO_HIT, index -1), so the two
// results are selects between literals instead of updates of running values — two instructions fewer than the
// general form, whose multiply-adds with the known start values ptxas does not fold.
// The compare t <= RT_NO_HIT is redundant: a ray parallel to the plane has t = +-inf or NaN, and then the in-plane
// coordinates t * d + o are +-inf or NaN too, which the bounds tests at the head of the chain reject.  But the
// kernel WITHOUT it measured 2.1 % slower, 33.39 against 32.71 ms on the same GPU (profiles/r02_v26_sweeps.txt):
// one instruction fewer, another ptxas schedule.  At 142 instructions the schedule's luck is worth more than an
// instruction.
RT_D void rect_closest_first(float t, float xa, float xb, float ha, float hb, float index, float& best_t, float& best_index) {
    asm("{\n\t.reg .pred p;\n\t"
        "setp.le.f32 p, %2, %4;\n\t"
        "setp.le.and.f32 p, %3, %5, p;\n\t"
        "setp.ge.and.f32 p, %6, 0f3A83126F, p;\n\t"   /* t >= 0.001f */
        "setp.le.and.f32 p, %6, 0f7F61B1E6, p;\n\t"   /* t <= RT_NO_HIT (3e38f) */
        "selp.f32 %0, %6, 0f7F61B1E6, p;\n\t"
        "selp.f32 %1, %7, 0fBF800000, p;\n\t}"
        : "=f"(best_t), "=f"(best_index) : "f"(fabsf(xa)), "f"(fabsf(xb)), "f"(ha), "f"(hb), "f"(t), "f"(index));
}

// The update for a SLAB PAIR (rc_spec.cuh): `t` = max(t_lo, t_hi) is the distance of whichever of the two parallel
// walls lies in front of the ray, and the index that goes with it is `base` (wall lo) or `base + step` (wall hi,
// when t_hi > t_lo).  The choice is one FSET (1.0 / 0.0) and the predicated move an FADD / FFMA with an immediate,
// instead of compare + select between two literals (one of which costs a register move per iteration) + move.
RT_D void rect_closest_fma_pair(float t, float xa, float xb, float ha, float hb, float t_lo, float t_hi, float base, float step,
                                float& best_t, float& best_index) {
    if (step == 1.0f)   // (a literal in generated code: neighbouring table entries, the usual case — an add needs no second literal)
    asm("{\n\t.reg .pred p;\n\t.reg .f32 w;\n\t"
        "setp.le.f32 p, %2, %4;\n\t"
        "setp.le.and.f32 p, %3, %5, p;\n\t"
        "setp.ge.and.f32 p, %6, 0f3A83126F, p;\n\t"   /* t >= 0.001f */
        "setp.le.and.f32 p, %6, %0, p;\n\t"
        "set.gt.f32.f32 w, %8, %7;\n\t"
        "@p fma.rn.f32 %0, %6, 0f3F800000, 0f00000000;\n\t"
        "@p add.f32 %1, w, %9;\n\t}"
        : "+f"(best_t), "+f"(best_index) : "f"(fabsf(xa)), "f"(fabsf(xb)), "f"(ha), "f"(hb), "f"(t), "f"(t_lo), "f"(t_hi), "f"(base));
    else
    asm("{\n\t.reg .pred p;\n\t.reg .f32 w;\n\t"
        "setp.le.f32 p, %2, %4;\n\t"
        "setp.le.and.f32 p, %3, %5, p;\n\t"
        "setp.ge.and.f32 p, %6, 0f3A83126F, p;\n\t"   /* t >= 0.001f */
        "setp.le.and.f32 p, %6, %0, p;\n\t"
        "set.gt.f32.f32 w, %8, %7;\n\t"
        "@p fma.rn.f32 %0, %6, 0f3F800000, 0f00000000;\n\t"
        "@p fma.rn.f32 %1, w, %10, %9;\n\t}"
        : "+f"(best_t), "+f"(best_index) : "f"(fabsf(xa)), "f"(fabsf(xb)), "f"(ha), "f"(hb), "f"(t), "f"(t_lo), "f"(t_hi), "f"(base), "f"(step));
}

// Packed FP32 (sm_100a FFMA2 / FADD2 / FMUL2: two fp32 lanes per instruction, one issue slot, scalar operands
// broadcast).  The pipe spends two cycles on them, so the FP32 peak is unchanged (tools/micro/ffma2_bench.cu:
// 71 vs 73 TFLOP/s) — but this kernel is bound by ISSUE slots, not by the FMA pipe (34 % busy), and two
// rectangles on the same axis need the same three operations with the same ray operands:
//   pair_t   (k1, k2) - o_n, times 1/d_n                       -> the two plane distances
//   pair_oc  o_a - (c1, c2)                                    -> origins relative to the two centres
//   pair_x   (t1, t2) * d_a + (oc1, oc2)                       -> the two in-plane coordinates
// Each is one instruction for two rectangles; the arithmetic (round-to-nearest sub, mul, fused fma) is what
// the scalar code does, so results are bit-identical.
RT_D void pair_t(float k1, float k2, float on, float inv, float& t1, float& t2) {
    asm("{\n\t.reg .b64 kk, oo, ii, tt;\n\t"
        "mov.b64 kk, {%2, %3};\n\tmov.b64 oo, {%4, %4};\n\tmov.b64 ii, {%5, %5};\n\t"
        "sub.f32x2 tt, kk, oo;\n\tmul.f32x2 tt, tt, ii;\n\t"
        "mov.b64 {%0, %1}, tt;\n\t}" : "=f"(t1), "=f"(t2) : "f"(k1), "f"(k2), "f"(on), "f"(inv));
}
RT_D void pair_oc(float oa, float c1, float c2, float& oc1, float& oc2) {
    asm("{\n\t.reg .b64 oo, cc, rr;\n\t"
        "mov.b64 oo, {%2, %2};\n\tmov.b64 cc, {%3, %4};\n\t"
        "sub.f32x2 rr, oo, cc;\n\t"
        "mov.b64 {%0, %1}, rr;\n\t}" : "=f"(oc1), "=f"(oc2) : "f"(oa), "f"(c1), "f"(c2));
}
RT_D void pair_x(float t1, float t2, float d, float oc1, float oc2, float& x1, float& x2) {
    asm("{\n\t.reg .b64 tt, dd, cc, xx;\n\t"
        "mov.b64 tt, {%2, %3};\n\tmov.b64 dd, {%4, %4};\n\tmov.b64 cc, {%5, %6};\n\t"
        "fma.rn.f32x2 xx, tt, dd, cc;\n\t"
        "mov.b64 {%0, %1}, xx;\n\t}" : "=f"(x1), "=f"(x2) : "f"(t1), "f"(t2), "f"(d), "f"(oc1), "f"(oc2));
}

// Linear closest hit over the TYPE-SORTED table (spheres, xy, xz, yz rects):
// one tight loop per primitive kind with the axes hard-wired, no per-primitive
// type decode and no early exits — every rectangle is a fixed sequence of
// 3 FFMA + predicate compares + 2 selects, with the rectangle's constants
// read through uniform (warp-wide) addresses.  Within the table a later
// primitive wins an exact tie (`t <= closest`, src/shared_scene.rs:37-53,
// sphere.rs:53); exact ties are otherwise undefined in the reference (Q13).
template <int AXIS_N, class Scene>
RT_D void rect_group(const Scene& S, int begin, int end, const RayT<float>& r, int last_prim, float& best_t, int& best) {
    // plane axis n, in-plane axes (a, b): xy -> (z; x, y), xz -> (y; x, z), yz -> (x; y, z)
    const float on = AXIS_N == 2 ? r.o.z : (AXIS_N == 1 ? r.o.y : r.o.x);
    const float in = AXIS_N == 2 ? r.inv_d.z : (AXIS_N == 1 ? r.inv_d.y : r.inv_d.x);
    const float oa = AXIS_N == 0 ? r.o.y : r.o.x, da = AXIS_N == 0 ? r.d.y : r.d.x;
    const float ob = AXIS_N == 2 ? r.o.y : r.o.z, db = AXIS_N == 2 ? r.d.y : r.d.z;
    (void)last_prim;
#pragma unroll 2
    for (int i = begin; i < end; ++i) {
        const float4 a = S.ua(i);
        const float k = S.ub(i).x;
        const float t = (k - on) * in;                   // (k - o_n) / d_n; exactly 0 on the plane the ray leaves
        const float pa = fmaf(t, da, oa), pb = fmaf(t, db, ob);
        const float tc = rect_candidate(t, pa - 0.5f * (a.x + a.y), pb - 0.5f * (a.z + a.w), 0.5f * (a.y - a.x), 0.5f * (a.w - a.z));
        const bool hit = tc <= best_t;
        best_t = hit ? tc : best_t;
        best = hit ? i : best;
    }
}

// The same test with the rectangle constants addressed at compile-time offsets
// of the kernel parameters (fully unrolled, one uniform branch per rectangle).
// Two passes so the rectangles do not serialise on `best_t`: first every
// rectangle's own candidate distance (t if the plane hit is inside the bounds
// and beyond t_min, +inf otherwise) — independent chains the scheduler can
// interleave — then a short ordered min-reduction (`<=`: a later rectangle
// wins an exact tie).

template <int AXIS_N>
RT_D void rect_group_const(const KParams& P, const RayT<float>& r, int last_prim, float& best_t, int& best) {
    constexpr int G = AXIS_N == 2 ? 0 : (AXIS_N == 1 ? 1 : 2);
    const int base = P.lin_end[G];
    const int n = P.lin_end[G + 1] - base;
    if (n <= 0) return;
    const float on = AXIS_N == 2 ? r.o.z : (AXIS_N == 1 ? r.o.y : r.o.x);
    const float in = AXIS_N == 2 ? r.inv_d.z : (AXIS_N == 1 ? r.inv_d.y : r.inv_d.x);
    const float oa = AXIS_N == 0 ? r.o.y : r.o.x, da = AXIS_N == 0 ? r.d.y : r.d.x;
    const float ob = AXIS_N == 2 ? r.o.y : r.o.z, db = AXIS_N == 2 ? r.d.y : r.d.z;
    (void)last_prim;
    float tc[RT_MAX_CONST_RECTS];
#pragma unroll
    for (int j = 0; j < RT_MAX_CONST_RECTS; ++j) {
        if (j >= n) break;  // uniform
        const float4 a = P.crect_bounds[G][j];   // (ca, ha, cb, hb)
        const float t = (P.crect_k[G][j] - on) * in;  // (k - o_n) / d_n; exactly 0 on the plane the ray leaves
        const float xa = fmaf(t, da, oa - a.x), xb = fmaf(t, db, ob - a.z);
        tc[j] = rect_candidate(t, xa, xb, a.y, a.w);
    }
#pragma unroll
    for (int j = 0; j < RT_MAX_CONST_RECTS; ++j) {
        if (j >= n) break;  // uniform
        const bool hit = tc[j] <= best_t;
        best_t = hit ? tc[j] : best_t;
        best = hit ? base + j : best;
    }
}

RT_D bool aabb_hit_reference(float4 lo, float4 hi, const RayT<float>& r, float t_max);

// The instanced objects of a linear scene, after its plain primitives: cull volume (Aabb::hit verbatim),
// then the object's primitives against the ray in the object's space — SceneObject::hit through the
// Translate / RotateY wrappers (translate.rs:23-42, rotate_y.rs:29-66), Boxx::obj_hit (box.rs:82-101).
template <class Scene>
RT_D void linear_objects(const KParams& P, const Scene& S, const RayT<float>& r, int last_prim, float& best_t, int& best) {
#pragma unroll 1
    for (int k = 0; k < P.n_cobj; ++k) {
        const float4 lo = P.cobj_lo[k], hi = P.cobj_hi[k];
        if (!aabb_hit_reference(lo, hi, r, best_t)) continue;
        const int first = __float_as_int(lo.w), meta = __float_as_int(hi.w);
        const RayT<float> lr = to_local(P.cinst[meta >> 8], r);
        for (int p = first; p < first + (meta & 255); ++p) {
            const float t = prim_test_local(S, p, S.ua(p), S.ub(p), lr, p == last_prim, true, best_t);
            if (t >= 0.0f) { best_t = t; best = p; }
        }
    }
}

template <bool CONST_RECTS, class Scene>
RT_D int closest_hit_linear(const KParams& P, const Scene& S, const RayT<float>& r, int last_prim, float& best_t) {
    int best = -1;
    best_t = RT_NO_HIT;
    const int n_sph = P.lin_end[0];
    if (n_sph > 0) {
        const float a = dot(r.d, r.d), inv_a = fast_rcp(a);
#pragma unroll 1
        for (int i = 0; i < n_sph; ++i) {
            const float4 pa = S.ua(i), pb = S.ub(i);
            const bool moving = kinds_prim(pb.z) == RT_PRIM_MOVING;   // uniform: i is
            const vec3f ctr = moving ? sphere_centre(pa, S.un(i), r.time) : mk3(pa.x, pa.y, pa.z);
            const float t = sphere_hit<float>(r.o, r.d, a, inv_a, ctr, pa.w, pb.x, i == last_prim,
                                              (float)RT_T_MIN, best_t, !moving);
            const bool hit = t >= 0.0f;
            best_t = hit ? t : best_t;
            best = hit ? i : best;
        }
    }
    if (CONST_RECTS) {
        rect_group_const<2>(P, r, last_prim, best_t, best);
        rect_group_const<1>(P, r, last_prim, best_t, best);
        rect_group_const<0>(P, r, last_prim, best_t, best);
    } else {
        rect_group<2>(S, P.lin_end[0], P.lin_end[1], r, last_prim, best_t, best);
        rect_group<1>(S, P.lin_end[1], P.lin_end[2], r, last_prim, best_t, best);
        rect_group<0>(S, P.lin_end[2], P.lin_end[3], r, last_prim, best_t, best);
    }
    linear_objects(P, S, r, last_prim, best_t, best);
    return best;
}

// Slab test against [t_min, t_max]; conservative with respect to
// src/aabb.rs:42-59 (which clips every axis against the original interval and
// so accepts a superset).  Boxes are padded at upload, see rc_api.cu.
RT_D bool aabb_hit(float4 lo, float4 hi, const RayT<float>& r, float t_max) {
    float tx0 = (lo.x - r.o.x) * r.inv_d.x, tx1 = (hi.x - r.o.x) * r.inv_d.x;
    float ty0 = (lo.y - r.o.y) * r.inv_d.y, ty1 = (hi.y - r.o.y) * r.inv_d.y;
    float tz0 = (lo.z - r.o.z) * r.inv_d.z, tz1 = (hi.z - r.o.z) * r.inv_d.z;
    float tn = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), (float)RT_T_MIN));
    float tf = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), t_max));
    return tn <= tf;
}

// The same slab test for the BVH walk, where it is most of the instructions: per ray, the reciprocal
// direction I (a zero component gives +-1e20 instead of infinity, so that no product is inf - inf) and
// N = -o * I; per box, t = bound * I + N — two packed multiply-adds for x and y of both corners (lo.xy and
// hi.xy are register pairs as loaded) and two scalar ones for z, instead of six subtractions and six
// multiplications.  Rounds differently from aabb_hit by an ulp of |o * I|: the same order as the
// rounding of (bound - o) there, and inside the pad the boxes get at upload.
struct BoxRay {
    float ix, iy, iz, nx, ny, nz;
};
RT_D BoxRay make_box_ray(const RayT<float>& r) {
    BoxRay b;
    b.ix = fminf(fmaxf(r.inv_d.x, -1e20f), 1e20f);
    b.iy = fminf(fmaxf(r.inv_d.y, -1e20f), 1e20f);
    b.iz = fminf(fmaxf(r.inv_d.z, -1e20f), 1e20f);
    b.nx = -r.o.x * b.ix; b.ny = -r.o.y * b.iy; b.nz = -r.o.z * b.iz;
    return b;
}
RT_D bool aabb_hit_packed(float4 lo, float4 hi, const BoxRay& b, float t_max) {
    float tx0, ty0, tx1, ty1;
    fma2(lo.x, lo.y, b.ix, b.iy, b.nx, b.ny, tx0, ty0);
    fma2(hi.x, hi.y, b.ix, b.iy, b.nx, b.ny, tx1, ty1);
    const float tz0 = fmaf(lo.z, b.iz, b.nz), tz1 = fmaf(hi.z, b.iz, b.nz);
    float tn = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), (float)RT_T_MIN));
    float tf = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), t_max));
    return tn <= tf;
}

// Aabb::hit exactly as the reference evaluates it (src/aabb.rs:42-59): every axis is clipped
// against the ORIGINAL [t_min, t_max] (Q12).  Needed when stored boxes are not bounding boxes —
// RotateY's (Q14) — because the box then decides which rays may see the object at all (Q11).
RT_D bool aabb_hit_reference(float4 lo, float4 hi, const RayT<float>& r, float t_max) {
    const float t_min = (float)RT_T_MIN;
    float t0 = (lo.x - r.o.x) * r.inv_d.x, t1 = (hi.x - r.o.x) * r.inv_d.x;
    if (r.inv_d.x < 0.0f) { float q = t0; t0 = t1; t1 = q; }
    if ((t1 < t_max ? t1 : t_max) <= (t0 > t_min ? t0 : t_min)) return false;
    t0 = (lo.y - r.o.y) * r.inv_d.y; t1 = (hi.y - r.o.y) * r.inv_d.y;
    if (r.inv_d.y < 0.0f) { float q = t0; t0 = t1; t1 = q; }
    if ((t1 < t_max ? t1 : t_max) <= (t0 > t_min ? t0 : t_min)) return false;
    t0 = (lo.z - r.o.z) * r.inv_d.z; t1 = (hi.z - r.o.z) * r.inv_d.z;
    if (r.inv_d.z < 0.0f) { float q = t0; t0 = t1; t1 = q; }
    if ((t1 < t_max ? t1 : t_max) <= (t0 > t_min ? t0 : t_min)) return false;
    return true;
}

// The primitives of one leaf (one top-level object: a single primitive, or the six sides of a Box
// tested in order, src/geometry/box.rs:82-101; they share the object's instance transform, applied
// to the ray once per leaf).  The walk reaches the leaves in the reference's order and a primitive
// only reports a hit within best_t, so every hit replaces the best one: a later primitive wins an
// exact tie, as with the reference's `t <= closest` (bvh_node.rs:124-129, sphere.rs:53).
template <class Scene>
RT_D void leaf_test(const Scene& S, int leaf, const RayT<float>& r, int last_prim, float& best_t, int& best) {
    const int first = leaf & 0xffffff, count = leaf >> 24;
    const int inst = RT_HAS_INSTANCES ? kinds_inst(S.pb(first).z) : -1;
    if (RT_HAS_INSTANCES && inst >= 0) {
        const RayT<float> lr = to_local(S.instances()[inst], r);
        for (int p = first; p < first + count; ++p) {
            const float t = prim_test_local(S, p, S.pa(p), S.pb(p), lr, p == last_prim, true, best_t);
            if (t >= 0.0f) { best_t = t; best = p; }
        }
    } else {
        for (int p = first; p < first + count; ++p) {
            const float t = prim_test_local(S, p, S.pa(p), S.pb(p), r, p == last_prim, false, best_t);
            if (t >= 0.0f) { best_t = t; best = p; }
        }
    }
}

// Threaded pre-order BVH: left child = i + 1, `skip` = next node when this
// subtree is done.  Visits left before right with a shrinking t_max, exactly
// the order of Node::hit (src/bvh_node.rs:112-132), over the node range
// [i, end) (the whole tree, or one subtree).
template <class Scene>
RT_D void closest_hit_threaded(const Scene& S, int i, int end, const RayT<float>& r, int last_prim, float& best_t, int& best) {
    if (S.reference_aabb()) {   // stored boxes that are not bounding boxes (Q14): the reference's own test
#pragma unroll 1
        while (i < end) {
            const float4 lo = S.nlo(i), hi = S.nhi(i);
            const int leaf = __float_as_int(hi.w);
            const bool box_hit = aabb_hit_reference(lo, hi, r, best_t);
            if (box_hit && leaf >= 0) leaf_test(S, leaf, r, last_prim, best_t, best);
            i = box_hit && leaf < 0 ? i + 1 : __float_as_int(lo.w);
        }
        return;
    }
    const BoxRay br = make_box_ray(r);
#pragma unroll 1
    while (i < end) {
        const float4 lo = S.nlo(i), hi = S.nhi(i);
        const int leaf = __float_as_int(hi.w);
        const bool box_hit = aabb_hit_packed(lo, hi, br, best_t);
        // the only divergent branch of a step is the leaf; the next node is a select
        if (box_hit && leaf >= 0) leaf_test(S, leaf, r, last_prim, best_t, best);
        i = box_hit && leaf < 0 ? i + 1 : __float_as_int(lo.w);
    }
}

template <class Scene>
RT_D int closest_hit_bvh(const Scene& S, int n_nodes, const RayT<float>& r, int last_prim, float& best_t) {
    int best = -1;
    best_t = RT_NO_HIT;
    closest_hit_threaded(S, 0, n_nodes, r, last_prim, best_t, best);
    return best;
}

// ---------------------------------------------------------------------------
// Hit record (src/geometry.rs:17-57) rebuilt from (ray, t, primitive).
// ---------------------------------------------------------------------------
struct Hit {
    vec3f p, n;        // point, face normal (world space)
    vec3f outward;     // outward normal in the primitive's own space (sphere uv, sphere.rs:61-63)
    vec3f lp;          // hit point in the primitive's own space (rectangle uv)
    bool front_face;
};

template <class Scene>
RT_D Hit make_hit_local(const Scene& S, int prim, float4 a, float4 b, const RayT<float>& r, float t, float k_two = 2.0f) {
    Hit h;
    fma2_bcast(t, r.d.x, r.d.y, r.o.x, r.o.y, h.p.x, h.p.y);   // Ray::at
    h.p.z = fmaf(t, r.d.z, r.o.z);
    if (RT_HAS_SPHERES && (!RT_HAS_RECTS || RT_IS_SPHERE(kinds_prim(b.z)))) {
        vec3f ctr = kinds_prim(b.z) == RT_PRIM_MOVING ? sphere_centre(a, S.pn(prim), r.time) : mk3(a.x, a.y, a.z);
        const float aa = dot(r.d, r.d);
        h.outward = sphere_normal(r.o, r.d, aa, fast_rcp(aa), ctr, a.w, t);  // sphere.rs:61
        h.p = ctr + a.w * h.outward;   // the point on the surface that normal belongs to
        h.front_face = dot(r.d, h.outward) < 0.0f;  // geometry.rs:49-56
        h.n = h.front_face ? h.outward : -h.outward;
    } else {
        // rectangles, branch- and select-free: N = the +axis unit normal (xy_rect.rs:45 etc.) read
        // from the table.  The point is put back on the plane — the reference's f64 ray.at(t)
        // lands on it to 1e-13 — by adding (k - p.N) N: k - p.N is exact (p.N is within rounding
        // of k) and so is the sum, so the next segment's re-test of this plane gives t = 0.
        const float4 n4 = S.pn(prim);
        const vec3f N = mk3(n4.x, n4.y, n4.z);
#ifdef RT_SPEC_SNAP_TABLE
        // the same, from the mask / offset form of the plane that the specialised kernel keeps in its staged table
        // (rc_spec.cuh, spec_snap_row): p * M + K
        fma2(h.p.x, h.p.y, a.x, a.y, a.z, a.w, h.p.x, h.p.y);
        h.p.z = fmaf(h.p.z, S.pc(prim).w, b.x);
#else
        const float e = b.x - dot(h.p, N);
        fma2_bcast(e, N.x, N.y, h.p.x, h.p.y, h.p.x, h.p.y);
        h.p.z = fmaf(e, N.z, h.p.z);
#endif
        const float dn = dot(r.d, N);
        h.front_face = dn < 0.0f;   // dot(d, axis) < 0, geometry.rs:49-56
        // +1 if dn < 0 else -1, on the FMA pipe: sat(-dn * 3e38) is 1 or 0 (|dn| below 3e-39 — an fp32 subnormal —
        // would give a fraction; a ray that parallel to the plane has no hit to shade)
        h.outward = N;
        const float sgn = fmaf(k_two, __saturatef(dn * -3.0e38f), -1.0f);
        mul2_bcast(sgn, N.x, N.y, h.n.x, h.n.y);
        h.n.z = sgn * N.z;
    }
    h.lp = h.p;
    return h;
}

// Hit record of (world ray, t, primitive), through the instance wrappers when there are any:
// RotateY turns point and normal back and re-derives the face from the ROTATED ray and the
// WORLD normal (rotate_y.rs:51-63, Q15); Translate adds the offset and runs set_face_normal
// again on the already-flipped normal (translate.rs:34-37, Q15).
template <class Scene>
RT_D Hit make_hit(const Scene& S, int prim, const RayT<float>& r, float t, float k_two = 2.0f) {
    float4 a = S.pa(prim), b = S.pb(prim);
    const int inst = kinds_inst(b.z);
    if (!RT_HAS_INSTANCES || inst < 0) return make_hit_local(S, prim, a, b, r, t, k_two);
    const DevInstance in = S.instances()[inst];
    const RayT<float> lr = to_local(in, r);
    Hit h = make_hit_local(S, prim, a, b, lr, t, k_two);
    if (in.flags & 1) {
        const float s = in.sin_theta, c = in.cos_theta;
        h.p = mk3(c * h.p.x + s * h.p.z, h.p.y, -s * h.p.x + c * h.p.z);
        const vec3f n = mk3(c * h.n.x + s * h.n.z, h.n.y, -s * h.n.x + c * h.n.z);
        h.front_face = dot(lr.d, n) < 0.0f;
        h.n = h.front_face ? n : -n;
    }
    if (in.flags & 2) {
        h.p = mk3(h.p.x + in.ox, h.p.y + in.oy, h.p.z + in.oz);
        h.front_face = dot(r.d, h.n) < 0.0f;   // the moved ray has the original direction
        h.n = h.front_face ? h.n : -h.n;
    }
    return h;
}

// uv on demand: sphere.rs:20-27, xy_rect.rs:42-43 (only image textures read it)
template <class Scene>
RT_D void hit_uv(const Scene& S, int prim, const Hit& h, float& u, float& v) {
    float4 a = S.pa(prim), b = S.pb(prim);
    int type = kinds_prim(b.z);
    const float PI_F = 3.14159265358979323846f;
    if (RT_IS_SPHERE(type)) {
        // sphere.rs:62 takes uv from the outward normal, moving_sphere.rs:76 from the POINT (Q27)
        const vec3f q = type == RT_PRIM_MOVING ? h.p : h.outward;
        float theta = acosf(fminf(fmaxf(-q.y, -1.0f), 1.0f));
        float phi = atan2f(-q.z, q.x) + PI_F;
        u = phi / (2.0f * PI_F);
        v = theta / PI_F;
    } else {
        float pa = type == RT_PRIM_YZ ? h.lp.y : h.lp.x;
        float pb = type == RT_PRIM_XY ? h.lp.y : h.lp.z;
        u = (pa - a.x) / (a.y - a.x);
        v = (pb - a.z) / (a.w - a.z);
    }
}

// ---------------------------------------------------------------------------
// Textures — src/texture/*.rs
// ---------------------------------------------------------------------------
// Perlin::noise + perlin_interp, src/texture/noise.rs:57-96.  `grad` and
// `perm` point at this texture's tables (shared memory when staged).
RT_D float perlin_noise(const float4* grad, const uint8_t* perm, vec3f p) {
    float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    float u = p.x - fx, v = p.y - fy, w = p.z - fz;
    int i = (int)fx, j = (int)fy, k = (int)fz;
    float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
    float accum = 0.0f;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                int idx = perm[(i + di) & 255] ^ perm[256 + ((j + dj) & 255)] ^ perm[512 + ((k + dk) & 255)];
                float4 g = grad[idx];
                float wx = u - (float)di, wy = v - (float)dj, wz = w - (float)dk;
                float bl = (di ? uu : 1.0f - uu) * (dj ? vv : 1.0f - vv) * (dk ? ww : 1.0f - ww);
                accum += bl * (g.x * wx + g.y * wy + g.z * wz);
            }
    return accum;
}

// Perlin::turbulence, src/texture/noise.rs:98-109
RT_D float perlin_turbulence(const float4* grad, const uint8_t* perm, vec3f p, int depth) {
    float accum = 0.0f, weight = 1.0f;
#pragma unroll 1
    for (int i = 0; i < depth; ++i) {
        accum += weight * perlin_noise(grad, perm, p);
        weight *= 0.5f;
        p = p * 2.0f;
    }
    return fabsf(accum);
}

struct TexCtx {            // where the Perlin tables live for this kernel
    const float4* perlin;  // n_perlin x 256
    const uint8_t* perm;   // n_perlin x 768
    // Two literals of the shading code that share an instruction with another literal (FFMA takes one immediate), so
    // one of the two has to sit in a register.  Left to itself ptxas re-creates that register in every iteration of
    // the path loop (a MOV / HFMA2 per use); the megakernel loads them once, from shared memory, which ptxas cannot
    // fold back into an immediate.  Same values either way.
    float k_two = 2.0f;                                   // make_hit_local: face sign
    float k_phi = 6.283185307179586f / 16777216.0f;       // sphere_direct_w: 24-bit integer -> angle
    float k_one = 1.0f;                                   // sphere_direct_w: 1 - 2u as ONE multiply-add
    // ... and literals of a GENERATED closest hit that would otherwise be re-created per iteration (the plane pair of
    // a slab pair is a packed operand: two UMOVs); which ones, the generator decides (spec_reg_consts, rc_spec.cuh)
    float k_spec[4] = {0.0f, 0.0f, 0.0f, 0.0f};
};

// Texture::value for a non-solid texture index (solid colours are folded into
// the primitive record).  Checker children are resolved iteratively, to any
// depth: the upload measures the longest chain, which bounds the loop.
template <class Scene>
RT_D vec3f texture_value(const KParams& P, const TexCtx& X, const Scene& S, int tex, int prim, const Hit& h) {
    DevTexture t = P.textures[tex];
#pragma unroll 1
    for (int level = 0; level < P.checker_depth && t.type == RT_TEX_CHECKER; ++level) {
        // checkered.rs:32-43 — world-space sines, odd if negative
        float sines = sinf(h.p.x * t.scale) * sinf(h.p.y * t.scale) * sinf(h.p.z * t.scale);
        t = P.textures[sines < 0.0f ? t.b : t.a];
    }
    if (t.type == RT_TEX_IMAGE) {  // image.rs:28-51: nearest texel, v flipped, clamped
        float u, v;
        hit_uv(S, prim, h, u, v);
        u = fminf(fmaxf(u, 0.0f), 1.0f);
        v = 1.0f - fminf(fmaxf(v, 0.0f), 1.0f);
        float fw = (float)P.image_w[t.a], fh = (float)P.image_h[t.a];
        float fi = u * fw, fj = v * fh;
        if (fi >= fw) fi = fw - 1.0f;
        if (fj >= fh) fj = fh - 1.0f;
        float4 px = tex2D<float4>(P.images[t.a], floorf(fi) + 0.5f, floorf(fj) + 0.5f);
        return mk3(px.x, px.y, px.z);
    }
    if (t.type == RT_TEX_NOISE) {  // noise.rs:26-33
        float turb = perlin_turbulence(X.perlin + 256 * t.a, X.perm + 768 * t.a, h.p, t.b);
        float s = 0.5f * (1.0f + sinf(t.scale * h.p.z + 10.0f * turb));
        return mk3(t.color.x * s, t.color.y * s, t.color.z * s);
    }
    return mk3(t.color.x, t.color.y, t.color.z);  // solid_color.rs:24-28
}

// BackgroundColor::color, src/background_color.rs:27-48
RT_D vec3f background_color(const KParams& P, vec3f d) {
    if (__float_as_int(P.bg_a.w) == 0) {  // Sky
        // explicit fused operations: this function is inlined in several places (general loop, culled tiles,
        // wavefront) and every copy has to round identically, whatever the compiler would contract around it
        const float t = 0.5f * fmaf(d.y, rsqrtf(fmaf(d.z, d.z, fmaf(d.y, d.y, d.x * d.x))), 1.0f), u = 1.0f - t;
        return mk3(fmaf(t, P.bg_b.x, u * P.bg_a.x), fmaf(t, P.bg_b.y, u * P.bg_a.y), fmaf(t, P.bg_b.z, u * P.bg_a.z));
    }
    return mk3(P.bg_a.x, P.bg_a.y, P.bg_a.z);
}

// ---------------------------------------------------------------------------
// Samplers.  DIRECT: inverse transforms of the distributions the reference's
// rejection loops produce.  REJECTION: those loops themselves, one Philox
// block per iteration (src/vec3.rs:424-444, src/util.rs:25-39).
// ---------------------------------------------------------------------------
struct RngCtx {
    const uint32_t* ks;   // Philox key schedule (kernel parameters)
    uint32_t pixel, sample;
};

// (cos, sin) of 2*pi*u for u in [0,1): the SFU sine/cosine are evaluated at
// 2*pi*u - pi (their accurate range) and negated; abs error ~5e-7.
RT_D void fast_sincos_2pi(float u, float& s, float& c) {
    const float phi = fmaf(u, 6.283185307179586f, -3.14159265358979323846f);
    s = -__sinf(phi);
    c = -__cosf(phi);
}

RT_D vec3f sphere_direct(float u1, float u2) {
    float z = 1.0f - 2.0f * u1;
    float r = fast_sqrt(fmaxf(0.0f, 1.0f - z * z));
    float s, c;
    fast_sincos_2pi(u2, s, c);
    return mk3(r * c, r * s, z);
}

// sphere_direct(u24(wx), u24(wy)) with the integer -> uniform scalings folded into the
// multiply-adds (same values: u24 is exact in fp32 and the scale factors are powers of two)
RT_D vec3f sphere_direct_w(uint32_t wx, uint32_t wy, float k_phi = 6.283185307179586f / 16777216.0f, float k_one = 1.0f) {
    // (w >> 8 as the high word of w * 2^24: an IMAD.HI on the FMA pipe instead of a shift on the ALU pipe)
    wx = __umulhi(wx, 1u << 24); wy = __umulhi(wy, 1u << 24);
    // 1 - 2 u1, in [-1 + 2^-23, 1]: one multiply-add whose second literal, 1, the caller holds in a register (TexCtx;
    // the product is exact — a power of two — so it rounds like a multiply followed by an add)
    const float z = fmaf((float)wx, -1.0f / 8388608.0f, k_one);
    const float r = fast_sqrt(fmaf(-z, z, 1.0f));                                       // |z| <= 1 exactly: never negative
    const float phi = fmaf((float)wy, k_phi, -3.14159265358979323846f);
    return mk3(-r * __cosf(phi), -r * __sinf(phi), z);
}

template <int ROUNDS>
RT_D vec3f reject_in_unit_sphere(const RngCtx& R, uint32_t bounce) {  // vec3.rs:424-430
    for (uint32_t j = 0;; ++j) {
        uint2 w = philox2x32_ks<ROUNDS>(R.pixel | (j << 24), rt_ctr1(R.sample, bounce, RT_TAG_REJECT), R.ks);
        float a, b, c;
        u21x3(w, a, b, c);
        vec3f v = mk3(2.0f * a - 1.0f, 2.0f * b - 1.0f, 2.0f * c - 1.0f);   // random_range(-1, 1)
        if (length_squared(v) >= 1.0f) continue;
        return v;
    }
}
