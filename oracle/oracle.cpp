// oracle.cpp — CPU parity oracle: an f64 restatement of racer-tracer's render
// hot path.  TEST INFRASTRUCTURE ONLY (see oracle.h): never linked, loaded or
// called by the product.  PARITY UNPINNED at the bit level by the reference (it
// has no render tests and cannot be built here); pinned by hand-derived known
// answers (tests/test_oracle_kat.py) and, statistically, by the reference's own
// published renders (tests/test_reference_renders.py).
//
// Every function cites the reference lines it follows, relative to
// /root/reference/racer-tracer/.  The code is a restatement over the flat
// structs of include/racer_cuda.h, not a translation of the Rust sources.

#include "oracle.h"

#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <thread>
#include <vector>

namespace {

const double PI = 3.14159265358979323846;  // std::f64::consts::PI

// ---------------------------------------------------------------------------
// Vec3 — src/vec3.rs (f64 triple; only the operations the hot path uses)
// ---------------------------------------------------------------------------
struct V3 {
    double x, y, z;
    double operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
};
inline V3 v3(double x, double y, double z) { return V3{x, y, z}; }
inline V3 v3(const double* p) { return V3{p[0], p[1], p[2]}; }
inline V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
inline V3 operator*(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
inline V3 operator*(double s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
inline V3 operator*(V3 a, double s) { return v3(a.x * s, a.y * s, a.z * s); }
inline V3 operator/(V3 a, double s) { return v3(a.x / s, a.y / s, a.z / s); }
inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }  // vec3.rs:171-173
inline V3 cross(V3 a, V3 b) {                                                // vec3.rs:175-181
    return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
inline double length_squared(V3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }  // vec3.rs:91-93
inline double length(V3 a) { return std::sqrt(length_squared(a)); }              // vec3.rs:87-89
inline V3 unit_vector(V3 a) {                                                    // vec3.rs:79-85
    double len = length(a);
    return v3(a.x / len, a.y / len, a.z / len);
}
inline bool near_zero(V3 a) {  // vec3.rs:127-130
    const double s = 1e-8;
    return std::fabs(a.x) < s && std::fabs(a.y) < s && std::fabs(a.z) < s;
}
inline V3 reflect(V3 v, V3 n) { return v - 2.0 * dot(v, n) * n; }  // vec3.rs:412-414
inline V3 refract(V3 uv, V3 n, double etai_over_etat) {           // vec3.rs:416-422
    double cos_theta = std::fmin(dot(-uv, n), 1.0);
    V3 r_out_perp = etai_over_etat * (uv + (cos_theta * n));
    V3 r_out_parallel = -std::sqrt(std::fabs(1.0 - length_squared(r_out_perp))) * n;
    return r_out_perp + r_out_parallel;
}

struct Ray {  // src/ray.rs
    V3 origin, direction;
    double time;
    V3 at(double t) const { return origin + t * direction; }
};

// ---------------------------------------------------------------------------
// RNG.  The reference draws from rand::thread_rng() (src/util.rs:9-23), which
// is OS-seeded and unreproducible.  Two back ends replace it:
//   Philox2x32 keyed by the seed with counter (pixel | j, sample | bounce | tag) —
//   the streams the GPU consumes (DESIGN.md "RNG streams"); Philox4x32 is kept
//   for the Perlin gradient tables the host derives from the seed;
//   xoshiro256** — an independent sequential stream drawn in call order.
// ---------------------------------------------------------------------------
inline void philox4x32(const uint32_t c_in[4], const uint32_t k_in[2], int rounds, uint32_t out[4]) {
    // Salmon et al., "Parallel random numbers: as easy as 1, 2, 3" (SC'11).
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    uint32_t c0 = c_in[0], c1 = c_in[1], c2 = c_in[2], c3 = c_in[3];
    uint32_t k0 = k_in[0], k1 = k_in[1];
    for (int r = 0; r < rounds; ++r) {
        if (r > 0) { k0 += W0; k1 += W1; }
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Philox2x32-R, same paper: 64-bit counter, 32-bit key
inline void philox2x32(uint32_t c0, uint32_t c1, uint32_t key, int rounds, uint32_t out[2]) {
    const uint32_t M = 0xD256D193u, W = 0x9E3779B9u;
    for (int r = 0; r < rounds; ++r) {
        if (r > 0) key += W;
        uint64_t p = (uint64_t)M * c0;
        uint32_t hi = (uint32_t)(p >> 32), lo = (uint32_t)p;
        c0 = hi ^ key ^ c1;
        c1 = lo;
    }
    out[0] = c0; out[1] = c1;
}

inline double u01_from_bits(uint32_t x) { return (double)(x >> 8) * (1.0 / 16777216.0); }

struct Xoshiro {
    uint64_t s[4];
    static uint64_t splitmix(uint64_t& z) {
        z += 0x9E3779B97F4A7C15ull;
        uint64_t r = z;
        r = (r ^ (r >> 30)) * 0xBF58476D1CE4E5B9ull;
        r = (r ^ (r >> 27)) * 0x94D049BB133111EBull;
        return r ^ (r >> 31);
    }
    void seed(uint64_t v) { for (auto& e : s) e = splitmix(v); }
    static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    uint64_t next() {
        uint64_t result = rotl(s[1] * 5, 7) * 9, t = s[1] << 17;
        s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45);
        return result;
    }
    double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }  // gen::<f64>()
};

// Philox2x32 counter layout — DESIGN.md "RNG streams"; the GPU
// (racer_tracer_b200/csrc/rt_math.cuh) uses the same table:
//   c0 = pixel (24 bits) | rejection iteration j << 24
//   c1 = sample (24 bits) | bounce (6 bits) << 24 | tag << 30
//   key = seed_lo ^ seed_hi
// One PATH block per path segment e (0 = primary ray): the upper 24 bits of each word feed the
// scattering event at the end of that segment (hit number b = e + 1); the low byte of each word
// is spare, and in block 0 the two spare bytes are the NEXT sample's 16-bit v jitter (sample s reads
// them from block 0 of sample (s - 1) mod 2^24), so that no sample needs its own block before its first hit.
const uint32_t TAG_PATH = 0u;    // segment e: scatter bits of hit e + 1; e = 0 also: low bytes -> v jitter of the next sample
const uint32_t TAG_PIXEL = 1u;   // x -> per-pixel u jitter
const uint32_t TAG_LENS = 2u;    // j = 0: direct lens sample, low bytes -> ray time; j >= 1: rejection iteration j
const uint32_t TAG_REJECT = 3u;  // (hit number b, iteration j): three 21-bit uniforms

inline double u21_from_bits(uint32_t x) { return (double)x * (1.0 / 2097152.0); }  // x < 2^21

// One sample's random source.  With ORACLE_RNG_PHILOX every request maps to a
// fixed counter, so the values do not depend on call order; with
// ORACLE_RNG_SEQUENTIAL each request pulls the next uniforms of the stream.
struct Draws {
    int backend;
    uint32_t key;
    int rounds;
    uint32_t pixel, sample;
    Xoshiro* seq;

    void words(uint32_t j, uint32_t smp, uint32_t bounce, uint32_t tag, uint32_t out[2]) const {
        philox2x32(pixel | (j << 24), smp | (bounce << 24) | (tag << 30), key, rounds, out);
    }
    static void split21(const uint32_t w[2], double u[3]) {
        u[0] = u21_from_bits(w[0] >> 11); u[1] = u21_from_bits(w[1] >> 11);
        u[2] = u21_from_bits(((w[0] & 0x7FFu) << 10) | (w[1] & 0x3FFu));
    }
    double pixel_jitter() const {  // cpu.rs:35-36
        if (backend != ORACLE_RNG_PHILOX) return seq->uniform();
        uint32_t w[2];
        words(0u, 0u, 0u, TAG_PIXEL, w);
        return u01_from_bits(w[0]);
    }
    static double u16_low_bytes(const uint32_t w[2]) { return (double)(((w[0] & 0xFFu) << 8) | (w[1] & 0xFFu)) * (1.0 / 65536.0); }
    static void split16(const uint32_t w[2], double u[3]) {   // three 16-bit uniforms from the upper 24 bits of each word
        u[0] = (double)(w[0] >> 16) * (1.0 / 65536.0); u[1] = (double)(w[1] >> 16) * (1.0 / 65536.0);
        u[2] = (double)((((w[0] >> 8) & 0xFFu) << 8) | ((w[1] >> 8) & 0xFFu)) * (1.0 / 65536.0);
    }
    double v_jitter() const {  // cpu.rs:39-40
        if (backend != ORACLE_RNG_PHILOX) return seq->uniform();
        uint32_t w[2];
        words(0u, (sample - 1u) & 0xFFFFFFu, 0u, TAG_PATH, w);   // the spare bytes of the PREVIOUS sample's block 0
        return u16_low_bytes(w);
    }
    // j = 0: the direct lens sample (u1, u2); j >= 1: the j-th iteration of random_in_unit_disk
    void lens(uint32_t j, double u[2]) const {
        if (backend != ORACLE_RNG_PHILOX) { u[0] = seq->uniform(); u[1] = seq->uniform(); return; }
        uint32_t w[2];
        words(j, sample, 0u, TAG_LENS, w);
        u[0] = u01_from_bits(w[0]); u[1] = u01_from_bits(w[1]);
    }
    double time_u() const {  // camera.rs:335
        if (backend != ORACLE_RNG_PHILOX) return seq->uniform();
        uint32_t w[2];
        words(0u, sample, 0u, TAG_LENS, w);
        return u16_low_bytes(w);
    }
    void two(uint32_t b, double u[2]) const {     // lambertian, direct
        if (backend != ORACLE_RNG_PHILOX) { u[0] = seq->uniform(); u[1] = seq->uniform(); return; }
        uint32_t w[2];
        words(0u, sample, b - 1u, TAG_PATH, w);   // hit number b closes segment b - 1
        u[0] = u01_from_bits(w[0]); u[1] = u01_from_bits(w[1]);
    }
    void three(uint32_t b, double u[3]) const {   // metal, direct: three 16-bit uniforms
        if (backend != ORACLE_RNG_PHILOX) { for (int i = 0; i < 3; ++i) u[i] = seq->uniform(); return; }
        uint32_t w[2];
        words(0u, sample, b - 1u, TAG_PATH, w);
        split16(w, u);
    }
    double one(uint32_t b) const {                // dielectric
        if (backend != ORACLE_RNG_PHILOX) return seq->uniform();
        uint32_t w[2];
        words(0u, sample, b - 1u, TAG_PATH, w);
        return u01_from_bits(w[0]);
    }
    void reject(uint32_t b, uint32_t j, double u[3]) const {  // iteration j of a rejection loop
        if (backend != ORACLE_RNG_PHILOX) { for (int i = 0; i < 3; ++i) u[i] = seq->uniform(); return; }
        uint32_t w[2];
        words(j, sample, b, TAG_REJECT, w);
        split21(w, u);
    }
};

// ---------------------------------------------------------------------------
// Scene access
// ---------------------------------------------------------------------------
struct Counters {
    oracle_counters c;
    Counters() { std::memset(&c, 0, sizeof(c)); }
    void add(const Counters& o) {
        const uint64_t* a = reinterpret_cast<const uint64_t*>(&o.c);
        uint64_t* b = reinterpret_cast<uint64_t*>(&c);
        for (size_t i = 0; i < sizeof(oracle_counters) / sizeof(uint64_t); ++i) b[i] += a[i];
    }
};

struct HitRecord {  // src/geometry.rs:17-26
    V3 point, normal;
    double t;
    bool front_face;
    int material;
    double u, v;
    uint32_t obj_id;
    int prim;
};

// HitRecord::set_face_normal, src/geometry.rs:49-56
inline void set_face_normal(HitRecord& rec, const Ray& ray, V3 outward_normal) {
    rec.front_face = dot(ray.direction, outward_normal) < 0.0;
    rec.normal = rec.front_face ? outward_normal : -outward_normal;
}

// Aabb::hit, src/aabb.rs:42-59.  Each axis is clipped against the ORIGINAL
// [t_min, t_max]; the interval is not carried across axes.
inline bool aabb_hit(const double* bmin, const double* bmax, const Ray& ray, double t_min, double t_max) {
    for (int a = 0; a < 3; ++a) {
        double inv_d = 1.0 / ray.direction[a];
        double t0 = (bmin[a] - ray.origin[a]) * inv_d;
        double t1 = (bmax[a] - ray.origin[a]) * inv_d;
        if (inv_d < 0.0) { double tmp = t0; t0 = t1; t1 = tmp; }
        double mn = t0 > t_min ? t0 : t_min;
        double mx = t1 < t_max ? t1 : t_max;
        if (mx <= mn) return false;
    }
    return true;
}

// Sphere::get_sphere_uv, src/geometry/sphere.rs:20-27
inline void sphere_uv(V3 p, double& u, double& v) {
    double theta = std::acos(-p.y);
    double phi = std::atan2(-p.z, p.x) + PI;
    u = phi / (2.0 * PI);
    v = theta / PI;
}

// obj_hit of the four primitive kinds in their own space.
bool prim_hit_local(const rc_scene& sc, int i, const Ray& ray, double t_min, double t_max,
                    HitRecord& rec, Counters& cnt) {
    const double* d = sc.prim_data + 5 * (size_t)i;
    int type = sc.prim_type[i];
    const bool moving = type == RC_PRIM_MOVING_SPHERE;
    if (moving) type = RC_PRIM_SPHERE;   // counted with the spheres
    cnt.c.prim_tests[type]++;
    rec.material = sc.prim_material[i];
    rec.obj_id = sc.prim_id[i];
    rec.prim = i;
    if (type == RC_PRIM_SPHERE) {
        // src/geometry/sphere.rs:31-68; moving_sphere.rs:42-88 is the same body around pos(time)
        V3 center = v3(d[0], d[1], d[2]);
        if (moving) {   // MovingSphere::pos, moving_sphere.rs:37-39
            const double* m = sc.prim_motion + 5 * (size_t)i;
            center = center + ((ray.time - m[3]) / (m[4] - m[3])) * (v3(m[0], m[1], m[2]) - center);
        }
        double radius = d[3];
        V3 oc = ray.origin - center;
        double a = length_squared(ray.direction);
        double half_b = dot(oc, ray.direction);
        double c = length_squared(oc) - radius * radius;
        double discriminant = half_b * half_b - a * c;
        if (discriminant < 0.0) return false;
        double sqrtd = std::sqrt(discriminant);
        double root = (-half_b - sqrtd) / a;
        if (root < t_min || t_max < root) {
            root = (-half_b + sqrtd) / a;
            if (root < t_min || t_max < root) return false;
        }
        rec.t = root;
        rec.point = ray.at(root);
        V3 outward_normal = (rec.point - center) / radius;
        // sphere.rs:62 takes uv from the outward normal; moving_sphere.rs:76 from the POINT (quirk, Q27)
        sphere_uv(moving ? rec.point : outward_normal, rec.u, rec.v);
        set_face_normal(rec, ray, outward_normal);
        cnt.c.prim_hits[type]++;
        return true;
    }
    // Rectangles: src/geometry/xy_rect.rs:21-48, xz_rect.rs:21-49, yz_rect.rs:21-49.
    // (a, b) are the in-plane axes, n the plane axis.
    int ax_a, ax_b, ax_n;
    if (type == RC_PRIM_XY_RECT) { ax_a = 0; ax_b = 1; ax_n = 2; }
    else if (type == RC_PRIM_XZ_RECT) { ax_a = 0; ax_b = 2; ax_n = 1; }
    else { ax_a = 1; ax_b = 2; ax_n = 0; }
    double a0 = d[0], a1 = d[1], b0 = d[2], b1 = d[3], k = d[4];
    double t = (k - ray.origin[ax_n]) / ray.direction[ax_n];
    if (t < t_min || t > t_max) return false;
    double pa = ray.origin[ax_a] + t * ray.direction[ax_a];
    double pb = ray.origin[ax_b] + t * ray.direction[ax_b];
    if (pa < a0 || pa > a1 || pb < b0 || pb > b1) return false;
    rec.u = (pa - a0) / (a1 - a0);
    rec.v = (pb - b0) / (b1 - b0);
    rec.t = t;
    rec.point = ray.at(t);
    V3 n = v3(ax_n == 0 ? 1.0 : 0.0, ax_n == 1 ? 1.0 : 0.0, ax_n == 2 ? 1.0 : 0.0);
    set_face_normal(rec, ray, n);
    cnt.c.prim_hits[type]++;
    return true;
}

// SceneObject::hit (src/scene.rs:98-101) including the RotateY / Translate
// wrappers (src/geometry/rotate_y.rs:29-66, translate.rs:23-42); YAML applies
// the rotation first, then the translation (src/scene/yml.rs:401-439), so the
// translation is the outer wrapper.
bool prim_hit(const rc_scene& sc, int i, const Ray& ray, double t_min, double t_max,
              HitRecord& rec, Counters& cnt) {
    int inst = (sc.prim_instance && sc.n_instances > 0) ? sc.prim_instance[i] : -1;
    if (inst < 0) return prim_hit_local(sc, i, ray, t_min, t_max, rec, cnt);
    const rc_instance& in = sc.instances[inst];
    Ray moved = ray;
    if (in.flags & 2) moved.origin = ray.origin - v3(in.offset);  // translate.rs:32
    Ray rotated = moved;
    if (in.flags & 1) {  // rotate_y.rs:38-47
        double s = in.sin_theta, c = in.cos_theta;
        rotated.origin.x = c * moved.origin.x - s * moved.origin.z;
        rotated.origin.z = s * moved.origin.x + c * moved.origin.z;
        rotated.direction.x = c * moved.direction.x - s * moved.direction.z;
        rotated.direction.z = s * moved.direction.x + c * moved.direction.z;
    }
    if (!prim_hit_local(sc, i, rotated, t_min, t_max, rec, cnt)) return false;
    if (in.flags & 1) {  // rotate_y.rs:51-63: point and normal back to world
        double s = in.sin_theta, c = in.cos_theta;
        V3 p = rec.point, n = rec.normal;
        p.x = c * rec.point.x + s * rec.point.z;
        p.z = -s * rec.point.x + c * rec.point.z;
        n.x = c * rec.normal.x + s * rec.normal.z;
        n.z = -s * rec.normal.x + c * rec.normal.z;
        rec.point = p;
        set_face_normal(rec, rotated, n);  // rotated ray, world normal (rotate_y.rs:62)
    }
    if (in.flags & 2) {  // translate.rs:34-37
        rec.point = rec.point + v3(in.offset);
        set_face_normal(rec, moved, rec.normal);
    }
    return true;
}

// Node::hit, src/bvh_node.rs:112-132: AABB test at every node including
// leaves, left child first, then right with t_max shrunk to the left hit.
bool node_hit(const rc_scene& sc, int n, const Ray& ray, double t_min, double t_max,
              HitRecord& rec, Counters& cnt) {
    const rc_bvh_node& node = sc.nodes[n];
    cnt.c.node_tests++;
    if (!aabb_hit(node.bmin, node.bmax, ray, t_min, t_max)) return false;
    if (node.left < 0) {
        // leaf = one top-level object: a single primitive, or the sides of a
        // Box tested in order with a shrinking t_max (src/geometry/box.rs:82-101)
        bool any = false;
        double closest = t_max;
        HitRecord tmp;
        for (int i = ~node.left; i < ~node.left + node.right; ++i)
            if (prim_hit(sc, i, ray, t_min, closest, tmp, cnt)) { closest = tmp.t; rec = tmp; any = true; }
        return any;
    }
    HitRecord l;
    if (node_hit(sc, node.left, ray, t_min, t_max, l, cnt)) {
        HitRecord r;
        if (node_hit(sc, node.right, ray, t_min, l.t, r, cnt)) rec = r; else rec = l;
        return true;
    }
    return node_hit(sc, node.right, ray, t_min, t_max, rec, cnt);
}

// scene.hit: the BVH (src/bvh_node.rs:208-216) or, without nodes, the linear
// closest-hit loop of src/shared_scene.rs:37-53.
bool scene_hit(const rc_scene& sc, const Ray& ray, double t_min, double t_max,
               HitRecord& rec, Counters& cnt) {
    if (sc.n_nodes > 0) return node_hit(sc, 0, ray, t_min, t_max, rec, cnt);
    bool any = false;
    double closest = t_max;
    HitRecord tmp;
    for (int i = 0; i < sc.n_prims; ++i) {
        if (prim_hit(sc, i, ray, t_min, closest, tmp, cnt)) {
            closest = tmp.t;
            rec = tmp;
            any = true;
        }
    }
    return any;
}

// ---------------------------------------------------------------------------
// Textures — src/texture/*.rs
// ---------------------------------------------------------------------------
// Perlin::noise + perlin_interp, src/texture/noise.rs:57-96
double perlin_noise(const rc_perlin& p, V3 pt, Counters& cnt) {
    cnt.c.noise_calls++;
    double u = pt.x - std::floor(pt.x), v = pt.y - std::floor(pt.y), w = pt.z - std::floor(pt.z);
    int i = (int)std::floor(pt.x), j = (int)std::floor(pt.y), k = (int)std::floor(pt.z);
    V3 c[2][2][2];
    for (int di = 0; di < 2; ++di)
        for (int dj = 0; dj < 2; ++dj)
            for (int dk = 0; dk < 2; ++dk) {
                int index = p.perm_x[(i + di) & 255] ^ p.perm_y[(j + dj) & 255] ^ p.perm_z[(k + dk) & 255];
                c[di][dj][dk] = v3(p.ran_vec[index]);
            }
    double uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
    double accum = 0.0;
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2; ++b)
            for (int cc = 0; cc < 2; ++cc) {
                V3 weight = v3(u - a, v - b, w - cc);
                accum += (a * uu + (1.0 - a) * (1.0 - uu)) * (b * vv + (1.0 - b) * (1.0 - vv)) *
                         (cc * ww + (1.0 - cc) * (1.0 - ww)) * dot(c[a][b][cc], weight);
            }
    return accum;
}

// Perlin::turbulence, src/texture/noise.rs:98-109
double perlin_turbulence(const rc_perlin& p, V3 pt, int depth, Counters& cnt) {
    double accum = 0.0, weight = 1.0;
    V3 temp_p = pt;
    for (int i = 0; i < depth; ++i) {
        accum += weight * perlin_noise(p, temp_p, cnt);
        weight *= 0.5;
        temp_p = temp_p * 2.0;
    }
    return std::fabs(accum);
}

V3 texture_value(const rc_scene& sc, int t, double u, double v, V3 point, Counters& cnt) {
    const rc_texture& tex = sc.textures[t];
    cnt.c.tex_evals[tex.type]++;
    switch (tex.type) {
    case RC_TEX_SOLID:  // solid_color.rs:24-28
        return v3(tex.color);
    case RC_TEX_CHECKER: {  // checkered.rs:32-43
        double sines = std::sin(point.x * tex.scale) * std::sin(point.y * tex.scale) * std::sin(point.z * tex.scale);
        return sines < 0.0 ? texture_value(sc, tex.b, u, v, point, cnt) : texture_value(sc, tex.a, u, v, point, cnt);
    }
    case RC_TEX_IMAGE: {  // image.rs:28-51
        const rc_image& img = sc.images[tex.a];
        double uc = std::fmin(std::fmax(u, 0.0), 1.0);
        double vc = 1.0 - std::fmin(std::fmax(v, 0.0), 1.0);
        double fi = uc * (double)img.width, fj = vc * (double)img.height;
        if (fi >= (double)img.width) fi = (double)img.width - 1.0;
        if (fj >= (double)img.height) fj = (double)img.height - 1.0;
        uint32_t ii = (uint32_t)fi, jj = (uint32_t)fj;
        const uint8_t* px = img.rgba + 4 * ((size_t)jj * img.width + ii);
        double color_scale = 1.0 / 255.0;
        return v3(px[0] * color_scale, px[1] * color_scale, px[2] * color_scale);
    }
    case RC_TEX_NOISE: {  // noise.rs:26-33
        const rc_perlin& p = sc.perlin[tex.a];
        return v3(tex.color) * 0.5 * (1.0 + std::sin(tex.scale * point.z + 10.0 * perlin_turbulence(p, point, tex.b, cnt)));
    }
    }
    return v3(0, 0, 0);
}

// BackgroundColor::color, src/background_color.rs:27-48
V3 background_color(const rc_scene& sc, const Ray& ray, Counters& cnt) {
    cnt.c.background++;
    if (sc.bg_type == RC_BG_SKY) {
        V3 unit_direction = unit_vector(ray.direction);
        double t = 0.5 * (unit_direction.y + 1.0);
        return (1.0 - t) * v3(sc.bg_a) + t * v3(sc.bg_b);
    }
    return v3(sc.bg_a);
}

// ---------------------------------------------------------------------------
// Samplers.  REJECTION follows src/vec3.rs:424-444 and src/util.rs:25-39 op
// for op (iteration j of a loop consumes Philox block j).  DIRECT draws the
// same distributions by inverse transform from one block, as the GPU's
// default does.
// ---------------------------------------------------------------------------
struct Sampler {
    const Draws& dr;
    int mode;
    Counters& cnt;

    // random_in_unit_sphere, vec3.rs:424-430
    V3 in_unit_sphere(uint32_t bounce) const {
        double u[3];
        if (mode == RC_SAMPLER_REJECTION) {
            for (uint32_t j = 0;; ++j) {
                dr.reject(bounce, j, u);
                cnt.c.rejection_iters++;
                V3 v = v3(2.0 * u[0] - 1.0, 2.0 * u[1] - 1.0, 2.0 * u[2] - 1.0);  // random_range(-1,1)
                if (length_squared(v) >= 1.0) continue;
                return v;
            }
        }
        dr.three(bounce, u);
        return std::cbrt(u[2]) * sphere_direct(u[0], u[1]);
    }
    // random_unit_vector, vec3.rs:442-444
    V3 unit_vec(uint32_t bounce) const {
        if (mode == RC_SAMPLER_REJECTION) return unit_vector(in_unit_sphere(bounce));
        double u[2];
        dr.two(bounce, u);
        return sphere_direct(u[0], u[1]);
    }
    static V3 sphere_direct(double u1, double u2) {
        double z = 1.0 - 2.0 * u1;
        double r = std::sqrt(std::fmax(0.0, 1.0 - z * z));
        double phi = 2.0 * PI * u2;
        return v3(r * std::cos(phi), r * std::sin(phi), z);
    }
};

// ---------------------------------------------------------------------------
// Materials — src/material/*.rs.  Returns false when the ray is absorbed.
// ---------------------------------------------------------------------------
bool scatter(const rc_scene& sc, const Ray& ray, const HitRecord& rec, uint32_t bounce,
             const Sampler& smp, Ray& scattered, V3& attenuation, Counters& cnt) {
    const rc_material& m = sc.materials[rec.material];
    cnt.c.scatters[m.type]++;
    switch (m.type) {
    case RC_MAT_LAMBERTIAN: {  // lambertian.rs:25-39
        V3 scatter_direction = rec.normal + smp.unit_vec(bounce);
        if (near_zero(scatter_direction)) scatter_direction = rec.normal;
        scattered = Ray{rec.point, scatter_direction, ray.time};
        attenuation = texture_value(sc, m.texture, rec.u, rec.v, rec.point, cnt);
        return true;
    }
    case RC_MAT_METAL: {  // metal.rs:25-44
        V3 reflected = reflect(unit_vector(ray.direction), rec.normal);
        scattered = Ray{rec.point, reflected + m.param * smp.in_unit_sphere(bounce), ray.time};
        if (dot(scattered.direction, rec.normal) < 0.0) return false;
        attenuation = texture_value(sc, m.texture, rec.u, rec.v, rec.point, cnt);
        return true;
    }
    case RC_MAT_DIELECTRIC: {  // dialectric.rs:25-56
        double refraction_ratio = rec.front_face ? 1.0 / m.param : m.param;
        V3 unit_direction = unit_vector(ray.direction);
        double cos_theta = std::fmin(dot(-unit_direction, rec.normal), 1.0);
        double sin_theta = std::sqrt(1.0 - cos_theta * cos_theta);
        bool cannot_refract = refraction_ratio * sin_theta > 1.0;
        bool do_reflect = cannot_refract;
        if (!do_reflect) {  // the RNG is drawn only if refraction is possible (short-circuit ||)
            do_reflect = oracle_reflectance(cos_theta, refraction_ratio) > smp.dr.one(bounce);
        }
        V3 direction = do_reflect ? reflect(unit_direction, rec.normal)
                                  : refract(unit_direction, rec.normal, refraction_ratio);
        scattered = Ray{rec.point, direction, ray.time};
        attenuation = v3(1.0, 1.0, 1.0);
        return true;
    }
    case RC_MAT_DIFFUSE_LIGHT:  // diffuse_light.rs:25-32
        return false;
    }
    return false;
}

// Material::color_emitted: material.rs:12-14, diffuse_light.rs:34-36
V3 color_emitted(const rc_scene& sc, const HitRecord& rec, Counters& cnt) {
    const rc_material& m = sc.materials[rec.material];
    if (m.type == RC_MAT_DIFFUSE_LIGHT) return texture_value(sc, m.texture, rec.u, rec.v, rec.point, cnt);
    return v3(0, 0, 0);
}

struct RayImageData {  // src/renderer.rs:33-39
    V3 rgb, normal, pos;
    double depth;
    uint32_t obj_id;
    double t;
};

// ray_color, src/renderer.rs:41-90 (recursive, as in the reference).
// `bounce` numbers the hit along the path (1 = primary hit) and keys the RNG.
RayImageData ray_color(const rc_scene& sc, const Ray& ray, int depth, uint32_t bounce, V3 camera_pos,
                       const Sampler& smp, Counters& cnt) {
    RayImageData out;
    out.normal = v3(0, 0, 0);
    out.pos = v3(0, 0, 0);
    out.depth = std::numeric_limits<double>::max();
    out.obj_id = 0;
    out.t = std::numeric_limits<double>::max();
    if (depth == 0) {  // renderer.rs:48-56: depth exhaustion is white
        cnt.c.depth_exhausted++;
        out.rgb = v3(1.0, 1.0, 1.0);
        return out;
    }
    HitRecord rec;
    cnt.c.segments++;
    if (scene_hit(sc, ray, 0.001, std::numeric_limits<double>::infinity(), rec, cnt)) {
        V3 emitted = color_emitted(sc, rec, cnt);
        Ray scattered;
        V3 attenuation;
        V3 color;
        if (scatter(sc, ray, rec, bounce, smp, scattered, attenuation, cnt))
            color = emitted + attenuation * ray_color(sc, scattered, depth - 1, bounce + 1, camera_pos, smp, cnt).rgb;
        else
            color = emitted;
        out.rgb = color;
        out.normal = rec.normal;
        out.pos = rec.point;
        out.depth = length(rec.point - camera_pos);
        out.obj_id = rec.obj_id;
        out.t = rec.t;
        return out;
    }
    out.rgb = background_color(sc, ray, cnt);
    return out;
}

// Camera::get_ray, src/camera.rs:326-337, with the lens sample passed in.
Ray get_ray(const rc_camera& cam, double u, double v, double dx, double dy, double time) {
    V3 rd = cam.lens_radius * v3(dx, dy, 0.0);
    V3 offset = v3(cam.right) * rd.x + v3(cam.up) * rd.y;
    Ray r;
    r.origin = v3(cam.origin) + offset;
    r.direction = v3(cam.upper_left_corner) + u * v3(cam.horizontal) - v * v3(cam.vertical) - v3(cam.origin) - offset;
    r.time = time;
    return r;
}

// One pixel-sample: src/renderer/cpu.rs:39-50 + camera.rs:326-337 RNG shape.
RayImageData trace_sample(const rc_scene& sc, const rc_camera& cam, const rc_params& p, const Draws& dr,
                          double u_pix, int x, int y, Counters& cnt) {
    (void)x;
    Sampler smp{dr, p.sampler, cnt};
    double v, dx = 0.0, dy = 0.0, time = cam.time_a;
    if (p.fixed_jitter) {
        v = ((double)y + 0.5) / (double)(p.height - 1);
    } else {
        v = ((double)y + dr.v_jitter()) / (double)(p.height - 1);  // cpu.rs:39-40
        // camera.rs:327: the reference samples the lens even when lens_radius
        // is 0; the offset is then exactly 0, so the draw is skipped here as on
        // the GPU (with counter-based streams nothing shifts).
        if (cam.lens_radius != 0.0 || dr.backend != ORACLE_RNG_PHILOX) {
            double q[2];
            if (p.sampler == RC_SAMPLER_REJECTION) {
                for (uint32_t j = 1;; ++j) {  // random_in_unit_disk, util.rs:25-39
                    dr.lens(j, q);
                    cnt.c.rejection_iters++;
                    dx = 2.0 * q[0] - 1.0; dy = 2.0 * q[1] - 1.0;
                    if (dx * dx + dy * dy >= 1.0) continue;
                    break;
                }
            } else {
                dr.lens(0, q);
                double r = std::sqrt(q[0]), phi = 2.0 * PI * q[1];
                dx = r * std::cos(phi); dy = r * std::sin(phi);
            }
        }
        time = cam.time_a + (cam.time_b - cam.time_a) * dr.time_u();  // camera.rs:335
    }
    Ray ray = get_ray(cam, u_pix, v, dx, dy, time);
    cnt.c.samples++;
    return ray_color(sc, ray, p.max_depth, 1, v3(cam.origin), smp, cnt);
}

double pixel_u(const rc_params& p, const Draws& dr, int x) {
    if (p.fixed_jitter) return ((double)x + 0.5) / (double)(p.width - 1);
    return ((double)x + dr.pixel_jitter()) / (double)(p.width - 1);  // cpu.rs:35-36, once per pixel
}

struct Tile { int x, y, w, h; };

// CpuRenderer::prepare_threads, src/renderer/cpu.rs:73-115: x-major tile
// order, remainder columns/rows on the last tile.
std::vector<Tile> prepare_tiles(int width, int height, int ntw, int nth) {
    std::vector<Tile> tiles;
    int width_step = width / ntw, height_step = height / nth;
    for (int ws = 0; ws < ntw; ++ws)
        for (int hs = 0; hs < nth; ++hs) {
            Tile t;
            t.x = width_step * ws;
            t.y = height_step * hs;
            t.w = ws == ntw - 1 ? width - width_step * ws : width_step;
            t.h = hs == nth - 1 ? height - height_step * hs : height_step;
            tiles.push_back(t);
        }
    return tiles;
}

int check(const rc_scene* sc, const rc_camera* cam, const rc_params* p) {
    if (!sc || !cam || !p) return RC_ERR_INVALID;
    if (p->width < 2 || p->height < 2 || p->samples < 1 || p->max_depth < 0) return RC_ERR_INVALID;
    return RC_OK;
}

// ToneMap implementations, src/tone_map/*.rs
V3 tone_map_one(const rc_tone_map& tm, V3 c) {
    switch (tm.type) {
    case RC_TONE_REINHARD: {  // reinhard.rs:16-42
        double max_white_pow = tm.max_white * tm.max_white;
        V3 w = v3(0.2126, 0.7152, 0.0722);
        double l_old = dot(c, w);
        double numerator = l_old * (1.0 + (l_old / max_white_pow));
        double l_new = numerator / (1.0 + l_old);
        double color_luminance = dot(c, w);
        return c * (l_new / color_luminance);
    }
    case RC_TONE_HABLE: {  // hable.rs:41-80
        double A = tm.hable[0], B = tm.hable[1], C = tm.hable[2], D = tm.hable[3], E = tm.hable[4], F = tm.hable[5];
        double toe_angle = E / F;
        auto partial = [&](double x) { return ((x * (A * x + C * B) + D * E) / (x * (A * x + B) + D * F)) - toe_angle; };
        double white_scale = 1.0 / partial(tm.linear_white_point);
        V3 e = c * tm.exposure_bias;
        return v3(partial(e.x) * white_scale, partial(e.y) * white_scale, partial(e.z) * white_scale);
    }
    case RC_TONE_ACES: {  // aces.rs:18-55
        auto mul = [](const double* m, V3 q) {
            return v3(m[0] * q.x + m[1] * q.y + m[2] * q.z, m[3] * q.x + m[4] * q.y + m[5] * q.z,
                      m[6] * q.x + m[7] * q.y + m[8] * q.z);
        };
        auto fit = [](double x) {
            double a = x * (x + 0.0245786) - 0.000090537;
            double b = x * (0.983729 * x + 0.4329510) + 0.238081;
            return a / b;
        };
        V3 i = mul(tm.aces_in, c);
        return mul(tm.aces_out, v3(fit(i.x), fit(i.y), fit(i.z)));
    }
    default:  // none.rs:14-18
        return c;
    }
}

// Rust `f64 as u32`: saturating, NaN -> 0.
inline uint32_t f64_as_u32(double v) {
    if (!(v == v)) return 0u;
    if (v <= 0.0) return 0u;
    if (v >= 4294967295.0) return 4294967295u;
    return (uint32_t)v;
}

}  // namespace

// ===========================================================================
// C API
// ===========================================================================
extern "C" {

int oracle_render(const rc_scene* scene, const rc_camera* camera, const rc_params* params,
                  const oracle_options* opt_in, double* out_rgb, oracle_counters* counters) {
    int st = check(scene, camera, params);
    if (st != RC_OK || !out_rgb) return RC_ERR_INVALID;
    oracle_options opt;
    std::memset(&opt, 0, sizeof(opt));
    if (opt_in) opt = *opt_in;
    if (opt.tiles_w <= 0) opt.tiles_w = 10;
    if (opt.tiles_h <= 0) opt.tiles_h = 10;
    if (opt.tiles_w > params->width) opt.tiles_w = params->width;
    if (opt.tiles_h > params->height) opt.tiles_h = params->height;
    int n_threads = opt.threads > 0 ? opt.threads : (int)std::thread::hardware_concurrency();
    if (n_threads < 1) n_threads = 1;
    const int s_begin = opt.sample_begin;
    const int s_count = opt.sample_count > 0 ? opt.sample_count : params->samples;
    const int rounds = params->rng_rounds > 0 ? params->rng_rounds : 10;

    std::vector<Tile> tiles = prepare_tiles(params->width, params->height, opt.tiles_w, opt.tiles_h);
    std::atomic<size_t> next(0);
    std::vector<Counters> per_thread(n_threads);

    auto worker = [&](int tid) {
        Counters& cnt = per_thread[tid];
        for (;;) {
            size_t ti = next.fetch_add(1);
            if (ti >= tiles.size()) break;
            const Tile& tile = tiles[ti];
            Xoshiro seq;
            seq.seed(params->seed * 0x9E3779B97F4A7C15ull + ti + 1);
            // CpuRenderer::raytrace, src/renderer/cpu.rs:26-71
            for (int row = 0; row < tile.h; ++row)
                for (int col = 0; col < tile.w; ++col) {
                    int x = tile.x + col, y = tile.y + row;
                    Draws dr;
                    dr.backend = opt.rng;
                    dr.key = (uint32_t)params->seed ^ (uint32_t)(params->seed >> 32);
                    dr.rounds = rounds;
                    dr.pixel = (uint32_t)(y * params->width + x);
                    dr.sample = 0;
                    dr.seq = &seq;
                    double u = pixel_u(*params, dr, x);
                    V3 color = v3(0, 0, 0);
                    for (int s = s_begin; s < s_begin + s_count; ++s) {
                        dr.sample = (uint32_t)s;
                        // COUNTERFACTUAL (not the reference): a fresh u jitter for every sample, i.e. what
                        // cpu.rs:35-36 would be if it stood inside the sample loop.  Only the Q1 signature test
                        // uses it, to show that the statistic it checks can tell the two apart.
                        if ((opt.counterfactual & ORACLE_CF_PER_SAMPLE_U) && !params->fixed_jitter)
                            u = ((double)x + seq.uniform()) / (double)(params->width - 1);
                        color = color + trace_sample(*scene, *camera, *params, dr, u, x, y, cnt).rgb;
                    }
                    double* o = out_rgb + 3 * ((size_t)y * params->width + x);
                    if (opt.linear_sum) {
                        o[0] = color.x; o[1] = color.y; o[2] = color.z;
                    } else {  // Vec3::scale_sqrt, src/vec3.rs:119-125
                        double scale = 1.0 / (double)params->samples;
                        o[0] = std::sqrt(scale * color.x);
                        o[1] = std::sqrt(scale * color.y);
                        o[2] = std::sqrt(scale * color.z);
                    }
                }
        }
    };
    if (n_threads == 1) {
        worker(0);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < n_threads; ++t) pool.emplace_back(worker, t);
        for (auto& t : pool) t.join();
    }
    if (counters) {
        Counters total;
        for (auto& c : per_thread) total.add(c);
        *counters = total.c;
    }
    return RC_OK;
}

int oracle_render_preview(const rc_scene* scene, const rc_camera* camera, const rc_params* params,
                          const oracle_options* opt_in, int32_t scale_w, int32_t scale_h, double* out_rgb) {
    int st = check(scene, camera, params);
    if (st != RC_OK || !out_rgb || scale_w < 1 || scale_h < 1) return RC_ERR_INVALID;
    oracle_options opt;
    std::memset(&opt, 0, sizeof(opt));
    if (opt_in) opt = *opt_in;
    if (opt.tiles_w <= 0) opt.tiles_w = 10;
    if (opt.tiles_h <= 0) opt.tiles_h = 10;
    const int rounds = params->rng_rounds > 0 ? params->rng_rounds : 10;
    const int s_begin = opt.sample_begin;
    const int s_count = opt.sample_count > 0 ? opt.sample_count : params->samples;
    const int W = params->width, H = params->height;
    const int grid_w = W / scale_w;   // block grid of the whole screen (Philox pixel index)
    std::memset(out_rgb, 0, sizeof(double) * 3 * (size_t)W * H);   // vec![Vec3::default(); ..], cpu_scaled.rs:53
    std::vector<Tile> tiles = prepare_tiles(W, H, opt.tiles_w, opt.tiles_h);
    Counters cnt;
    for (size_t ti = 0; ti < tiles.size(); ++ti) {
        const Tile& tile = tiles[ti];
        Xoshiro seq;
        seq.seed(params->seed * 0x9E3779B97F4A7C15ull + ti + 1);
        const int scaled_width = tile.w / scale_w, scaled_height = tile.h / scale_h;   // cpu_scaled.rs:51-52
        for (int row = 0; row < scaled_height; ++row)
            for (int column = 0; column < scaled_width; ++column) {
                const int x = tile.x + column * scale_w, y = tile.y + row * scale_h;
                Draws dr;
                dr.backend = opt.rng;
                dr.key = (uint32_t)params->seed ^ (uint32_t)(params->seed >> 32);
                dr.rounds = rounds;
                dr.pixel = (uint32_t)((y / scale_h) * grid_w + x / scale_w);
                dr.sample = 0;
                dr.seq = &seq;
                const double u = pixel_u(*params, dr, x);   // once per block, cpu_scaled.rs:55-56
                V3 color = v3(0, 0, 0);
                for (int s = s_begin; s < s_begin + s_count; ++s) {
                    dr.sample = (uint32_t)s;
                    color = color + trace_sample(*scene, *camera, *params, dr, u, x, y, cnt).rgb;   // v: cpu_scaled.rs:59-60
                }
                const double scale = 1.0 / (double)params->samples;   // scale_sqrt, cpu_scaled.rs:75
                const V3 c = v3(std::sqrt(scale * color.x), std::sqrt(scale * color.y), std::sqrt(scale * color.z));
                for (int sh = 0; sh < scale_h; ++sh)
                    for (int sw = 0; sw < scale_w; ++sw) {
                        double* o = out_rgb + 3 * ((size_t)(y + sh) * W + (x + sw));
                        o[0] = c.x; o[1] = c.y; o[2] = c.z;
                    }
            }
    }
    return RC_OK;
}

int oracle_primary_aov(const rc_scene* scene, const rc_camera* camera, const rc_params* params,
                       uint32_t* id, double* t, double* normal, double* point) {
    int st = check(scene, camera, params);
    if (st != RC_OK) return st;
    rc_params p = *params;
    p.fixed_jitter = 1;
    p.max_depth = 1;  // one scene.hit; the scattered ray returns at depth 0
    // rows are independent (fixed jitter: no random stream is consumed): spread them over the host threads
    std::atomic<int> next_row(0);
    auto worker = [&]() {
        Counters cnt;
        for (;;) {
            const int y = next_row.fetch_add(1);
            if (y >= p.height) break;
            for (int x = 0; x < p.width; ++x) {
                Draws dr;
                std::memset(&dr, 0, sizeof(dr));
                dr.backend = ORACLE_RNG_PHILOX;
                dr.rounds = 10;
                dr.pixel = (uint32_t)(y * p.width + x);
                double u = pixel_u(p, dr, x);
                RayImageData d = trace_sample(*scene, *camera, p, dr, u, x, y, cnt);
                size_t i = (size_t)y * p.width + x;
                if (id) id[i] = d.obj_id;
                if (t) t[i] = d.t;
                if (normal) { normal[3 * i] = d.normal.x; normal[3 * i + 1] = d.normal.y; normal[3 * i + 2] = d.normal.z; }
                if (point) { point[3 * i] = d.pos.x; point[3 * i + 1] = d.pos.y; point[3 * i + 2] = d.pos.z; }
            }
        }
    };
    int n_threads = (int)std::thread::hardware_concurrency();
    if (n_threads < 1 || (long long)p.width * p.height < 65536) n_threads = 1;
    if (n_threads == 1) worker();
    else {
        std::vector<std::thread> pool;
        for (int k = 0; k < n_threads; ++k) pool.emplace_back(worker);
        for (auto& th : pool) th.join();
    }
    return RC_OK;
}

int oracle_sample_radiance(const rc_scene* scene, const rc_camera* camera, const rc_params* params,
                           int32_t n, const int32_t* pixel_idx, const int32_t* sample_idx,
                           double* out, int32_t* out_segments) {
    int st = check(scene, camera, params);
    if (st != RC_OK) return st;
    const int rounds = params->rng_rounds > 0 ? params->rng_rounds : 10;
    for (int i = 0; i < n; ++i) {
        Counters cnt;
        Draws dr;
        dr.backend = ORACLE_RNG_PHILOX;
        dr.key = (uint32_t)params->seed ^ (uint32_t)(params->seed >> 32);
        dr.rounds = rounds;
        dr.pixel = (uint32_t)pixel_idx[i];
        dr.sample = 0;
        dr.seq = nullptr;
        int x = pixel_idx[i] % params->width, y = pixel_idx[i] / params->width;
        double u = pixel_u(*params, dr, x);
        dr.sample = (uint32_t)sample_idx[i];
        RayImageData d = trace_sample(*scene, *camera, *params, dr, u, x, y, cnt);
        out[3 * i] = d.rgb.x; out[3 * i + 1] = d.rgb.y; out[3 * i + 2] = d.rgb.z;
        if (out_segments) out_segments[i] = (int32_t)cnt.c.segments;
    }
    return RC_OK;
}

void oracle_camera_new(const double look_from[3], const double look_at[3], const double scene_up[3],
                       double vfov, double aperture, double focus_distance, double aspect_ratio,
                       double time_a, double time_b, rc_camera* out) {
    // Camera::new, src/camera.rs:196-234
    double h = std::tan((vfov * PI / 180.0) / 2.0);  // util.rs:5-7
    double viewport_height = 2.0 * h;
    double viewport_width = aspect_ratio * viewport_height;
    V3 from = v3(look_from), at = v3(look_at), vup = v3(scene_up);
    V3 forward = unit_vector(from - at);
    V3 right = unit_vector(cross(vup, forward));
    V3 up = cross(forward, right);
    V3 horizontal = focus_distance * viewport_width * right;
    V3 vertical = focus_distance * viewport_height * up;
    V3 ulc = from + vertical / 2.0 - horizontal / 2.0 - focus_distance * forward;
    auto put = [](double* d, V3 v) { d[0] = v.x; d[1] = v.y; d[2] = v.z; };
    put(out->origin, from); put(out->upper_left_corner, ulc); put(out->forward, forward);
    put(out->right, right); put(out->up, up); put(out->horizontal, horizontal); put(out->vertical, vertical);
    out->vfov = vfov; out->viewport_width = viewport_width; out->viewport_height = viewport_height;
    out->lens_radius = aperture * 0.5; out->focus_distance = focus_distance;
    out->time_a = time_a; out->time_b = time_b;
}

void oracle_tone_map(const rc_tone_map* tm, const double* rgb, int64_t n_pixels, double* out) {
    for (int64_t i = 0; i < n_pixels; ++i) {
        V3 c = tone_map_one(*tm, v3(rgb + 3 * i));
        out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
    }
}

void oracle_quantise_rgba(const double* rgb, int64_t n_pixels, uint8_t* rgba) {
    // src/image_action/png.rs:21-31
    for (int64_t i = 0; i < n_pixels; ++i) {
        uint32_t red = f64_as_u32(rgb[3 * i] * 255.0);
        uint32_t green = f64_as_u32(rgb[3 * i + 1] * 255.0);
        uint32_t blue = f64_as_u32(rgb[3 * i + 2] * 255.0);
        uint32_t val = (red << 24) | (green << 16) | (blue << 8) | 255u;
        rgba[4 * i] = (uint8_t)(val >> 24); rgba[4 * i + 1] = (uint8_t)(val >> 16);
        rgba[4 * i + 2] = (uint8_t)(val >> 8); rgba[4 * i + 3] = (uint8_t)val;
    }
}

void oracle_philox4x32(const uint32_t ctr[4], const uint32_t key[2], int32_t rounds, uint32_t out[4]) {
    philox4x32(ctr, key, rounds, out);
}

void oracle_philox2x32(const uint32_t ctr[2], uint32_t key, int32_t rounds, uint32_t out[2]) {
    philox2x32(ctr[0], ctr[1], key, rounds, out);
}

int oracle_aabb_hit(const double bmin[3], const double bmax[3], const double origin[3],
                    const double dir[3], double t_min, double t_max) {
    Ray r{v3(origin), v3(dir), 0.0};
    return aabb_hit(bmin, bmax, r, t_min, t_max) ? 1 : 0;
}

static void put_rec(const HitRecord& rec, double out[10]) {
    out[0] = rec.t; out[1] = rec.point.x; out[2] = rec.point.y; out[3] = rec.point.z;
    out[4] = rec.normal.x; out[5] = rec.normal.y; out[6] = rec.normal.z;
    out[7] = rec.u; out[8] = rec.v; out[9] = rec.front_face ? 1.0 : 0.0;
}

int oracle_prim_hit(const rc_scene* scene, int32_t prim, const double origin[3], const double dir[3],
                    double t_min, double t_max, double out[10]) {
    Ray r{v3(origin), v3(dir), 0.0};
    HitRecord rec;
    Counters cnt;
    if (!prim_hit(*scene, prim, r, t_min, t_max, rec, cnt)) return 0;
    put_rec(rec, out);
    return 1;
}

int oracle_scene_hit(const rc_scene* scene, const double origin[3], const double dir[3],
                     double t_min, double t_max, double out[10]) {
    Ray r{v3(origin), v3(dir), 0.0};
    HitRecord rec;
    Counters cnt;
    if (!scene_hit(*scene, r, t_min, t_max, rec, cnt)) return -1;
    put_rec(rec, out);
    return rec.prim;
}

double oracle_reflectance(double cosine, double refraction_index) {
    // Dialectric::reflectance, src/material/dialectric.rs:17-22
    double r0 = (1.0 - refraction_index) / (1.0 + refraction_index);
    r0 = r0 * r0;
    return r0 + (1.0 - r0) * std::pow(1.0 - cosine, 5.0);
}

void oracle_reflect(const double v[3], const double n[3], double out[3]) {
    V3 r = reflect(v3(v), v3(n));
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}

void oracle_refract(const double uv[3], const double n[3], double etai_over_etat, double out[3]) {
    V3 r = refract(v3(uv), v3(n), etai_over_etat);
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}

void oracle_texture_value(const rc_scene* scene, int32_t texture, double u, double v,
                          const double point[3], double out[3]) {
    Counters cnt;
    V3 c = texture_value(*scene, texture, u, v, v3(point), cnt);
    out[0] = c.x; out[1] = c.y; out[2] = c.z;
}

double oracle_perlin_noise(const rc_perlin* p, const double point[3]) {
    Counters cnt;
    return perlin_noise(*p, v3(point), cnt);
}

double oracle_perlin_turbulence(const rc_perlin* p, const double point[3], int32_t depth) {
    Counters cnt;
    return perlin_turbulence(*p, v3(point), depth, cnt);
}

void oracle_background(const rc_scene* scene, const double dir[3], double out[3]) {
    Counters cnt;
    Ray r{v3(0, 0, 0), v3(dir), 0.0};
    V3 c = background_color(*scene, r, cnt);
    out[0] = c.x; out[1] = c.y; out[2] = c.z;
}

void oracle_get_ray(const rc_camera* cam, double u, double v, double dx, double dy,
                    double origin[3], double dir[3]) {
    Ray r = get_ray(*cam, u, v, dx, dy, 0.0);
    origin[0] = r.origin.x; origin[1] = r.origin.y; origin[2] = r.origin.z;
    dir[0] = r.direction.x; dir[1] = r.direction.y; dir[2] = r.direction.z;
}

void oracle_vec3_op(int32_t op, const double a[3], const double b[3], double out[3]) {
    V3 x = v3(a), y = v3(b), r = v3(0, 0, 0);
    if (op == 0) r = x + y;
    else if (op == 1) r = x - y;
    else if (op == 2) r = x * y;
    else r = x / b[0];
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}

}  // extern "C"
