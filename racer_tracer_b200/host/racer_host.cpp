// racer_host.cpp — see racer_host.hpp.  Reference citations are relative to racer-tracer/src/.
#include "racer_host.hpp"

#include <zlib.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <mutex>
#include <sstream>

#include "jpeg_baseline.hpp"
#include "yaml_lite.hpp"

namespace racer {

using yaml_lite::Node;

namespace {

const double PI = 3.14159265358979323846;

std::string read_file(const std::string& path, bool& ok) {
    std::ifstream f(path.c_str(), std::ios::binary);
    ok = (bool)f;
    std::stringstream ss;
    if (ok) ss << f.rdbuf();
    return ss.str();
}

bool file_exists(const std::string& p) { std::ifstream f(p.c_str()); return (bool)f; }
std::string dir_of(const std::string& p) { size_t s = p.find_last_of('/'); return s == std::string::npos ? std::string(".") : p.substr(0, s); }
std::string base_of(const std::string& p) { size_t s = p.find_last_of('/'); return s == std::string::npos ? p : p.substr(s + 1); }

// Vec3 deserialises from {pos: [x,y,z]} with alias `color` (vec3.rs:12-16); a bare [x,y,z] is accepted too
Vec3 vec3_of(const Node& n, const std::string& what) {
    const Node* v = &n;
    if (n.is_map()) {
        v = n.find("pos");
        if (!v) v = n.find("color");
        if (!v) throw yaml_lite::ParseError("missing field `pos` in " + what);
    }
    if (!v->is_seq() || v->seq.size() != 3) throw yaml_lite::ParseError("expected 3 numbers for " + what);
    return Vec3{v->seq[0].as_double(), v->seq[1].as_double(), v->seq[2].as_double()};
}

// externally tagged serde enum: {Variant: {fields}} or a bare 'Variant'
std::pair<std::string, Node> enum_of(const Node& n, const std::string& what) {
    if (n.is_scalar()) return {yaml_lite::to_lower(n.scalar), Node()};
    if (n.is_map() && n.map.size() == 1) return {yaml_lite::to_lower(n.map[0].first), n.map[0].second};
    throw yaml_lite::ParseError("expected a single enum variant for " + what);
}

// ---- Philox4x32-10 for the Perlin gradient tables (the same streams as the Python harness) -------
void philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += W0; k1 += W1; }
        const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Perlin::new (texture/noise.rs:44-55): 256 normalised uniform(-1,1)^3 gradients, drawn from Philox(seed)
// so that host, oracle and GPU share them; identity permutation tables (noise.rs:122, SURVEY Q17)
rc_perlin make_perlin(uint64_t seed, int index) {
    rc_perlin p;
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    for (int i = 0; i < 256; ++i) {
        const uint32_t ctr[4] = {(uint32_t)i, (uint32_t)index, 0u, 2u << 24};
        uint32_t r[4];
        philox4x32(ctr, key, r);
        double v[3];
        for (int k = 0; k < 3; ++k) v[k] = 2.0 * ((double)(r[k] >> 8) / 16777216.0) - 1.0;
        const double n = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
        for (int k = 0; k < 3; ++k) p.ran_vec[i][k] = v[k] / n;
        p.perm_x[i] = p.perm_y[i] = p.perm_z[i] = i;
    }
    return p;
}

struct Prim {
    int type;
    double data[5];
    int material, obj, side, instance;
    bool moving = false;
    double motion[5] = {0, 0, 0, 0, 0};   // pos_b xyz, time_a, time_b
    Prim(int t, std::initializer_list<double> d, int m, int o, int s, int i) : type(t), material(m), obj(o), side(s), instance(i) {
        int k = 0;
        for (double v : d) data[k++] = v;
    }
};

struct TopObject {
    std::string key;
    std::vector<Prim> prims;
    double lo[3], hi[3], pos[3];
    bool has_rotate = false, has_translate = false;
    double rotate_deg = 0, translate[3] = {0, 0, 0};
};

void aabb_of(const double a[3], const double b[3], double lo[3], double hi[3]) {   // Aabb::new, aabb.rs:10-26
    for (int i = 0; i < 3; ++i) { lo[i] = std::min(a[i], b[i]); hi[i] = std::max(a[i], b[i]); }
}

// a rectangle's data, padded Aabb and position (xy_rect.rs:50-55, xz_rect.rs:51-56, yz_rect.rs:51-56,
// geometry_creation.rs:41-96)
Prim rect_prim(int kind, double a0, double a1, double b0, double b1, double k, int material, double lo[3], double hi[3], double pos[3]) {
    Prim p(kind, {a0, a1, b0, b1, k}, material, 0, 0, -1);
    double a[3], b[3];
    if (kind == RC_PRIM_XY_RECT) { a[0] = a0; a[1] = b0; a[2] = k - 0.0001; b[0] = a1; b[1] = b1; b[2] = k + 0.0001; pos[0] = a0; pos[1] = b0; pos[2] = k; }
    else if (kind == RC_PRIM_XZ_RECT) { a[0] = a0; a[1] = k - 0.0001; a[2] = b0; b[0] = a1; b[1] = k + 0.0001; b[2] = b1; pos[0] = a0; pos[1] = k; pos[2] = b0; }
    else { a[0] = k - 0.0001; a[1] = a0; a[2] = b0; b[0] = k + 0.0001; b[1] = a1; b[2] = b1; pos[0] = k; pos[1] = a0; pos[2] = b0; }
    aabb_of(a, b, lo, hi);
    return p;
}

// RotateY::create_bounding_box VERBATIM, including its two bugs (geometry/rotate_y.rs:68-90, SURVEY Q14):
// `cos*x + sin + z`, and min/max shifted by pos inside the corner loop.  The result is the object's
// ray-cull volume (Q11), so it has to be reproduced, not corrected.
void rotate_y_aabb(TopObject& o, double deg) {
    const double rad = deg * PI / 180.0, s = std::sin(rad), c = std::cos(rad);
    const double fmax = 1.7976931348623157e308;
    double mn[3] = {fmax, fmax, fmax}, mx[3] = {-fmax, -fmax, -fmax};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j)
            for (int k = 0; k < 2; ++k) {
                const double x = i * o.hi[0] + (1 - i) * o.lo[0];
                const double y = j * o.hi[1] + (1 - j) * o.lo[1];
                const double z = k * o.hi[2] + (1 - k) * o.lo[2];
                const double t[3] = {c * x + s + z, y, -s * x + c * z};
                for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], t[a]); mx[a] = std::max(mx[a], t[a]); }
                for (int a = 0; a < 3; ++a) { mn[a] += o.pos[a]; mx[a] += o.pos[a]; }
            }
    aabb_of(mn, mx, o.lo, o.hi);
}

// Node::build (bvh_node.rs:31-82): sort by Aabb minimum on one axis, split at the median, leaves hold
// one object.  The reference picks the axis at random from {x, y} (Q10); here it is the axis with the
// widest spread of box minima (ties -> lowest axis); a stable sort keeps equal keys in canonical order.
// Emits nodes in pre-order and objects in depth-first leaf order.
int build_bvh(std::vector<TopObject*> objs, std::vector<rc_bvh_node>& nodes, std::vector<TopObject*>& order) {
    const int idx = (int)nodes.size();
    nodes.push_back(rc_bvh_node());
    if (objs.size() == 1) {
        TopObject* o = objs[0];
        for (int a = 0; a < 3; ++a) { nodes[idx].bmin[a] = o->lo[a]; nodes[idx].bmax[a] = o->hi[a]; }
        nodes[idx].left = ~(int)order.size();
        nodes[idx].right = 1;
        order.push_back(o);
        return idx;
    }
    int axis = 0;
    double best = -1.0;
    for (int a = 0; a < 3; ++a) {
        double lo = objs[0]->lo[a], hi = objs[0]->lo[a];
        for (auto* o : objs) { lo = std::min(lo, o->lo[a]); hi = std::max(hi, o->lo[a]); }
        if (hi - lo > best) { best = hi - lo; axis = a; }
    }
    std::stable_sort(objs.begin(), objs.end(), [axis](const TopObject* x, const TopObject* y) { return x->lo[axis] < y->lo[axis]; });
    const size_t mid = objs.size() / 2;
    const int l = build_bvh(std::vector<TopObject*>(objs.begin(), objs.begin() + mid), nodes, order);
    const int r = build_bvh(std::vector<TopObject*>(objs.begin() + mid, objs.end()), nodes, order);
    nodes[idx].left = l; nodes[idx].right = r;
    for (int a = 0; a < 3; ++a) {   // Aabb::from((&a, &b)), aabb.rs:95-114
        nodes[idx].bmin[a] = std::min(nodes[l].bmin[a], nodes[r].bmin[a]);
        nodes[idx].bmax[a] = std::max(nodes[l].bmax[a], nodes[r].bmax[a]);
    }
    return idx;
}

// Surface-area-heuristic tree over the same leaves (one top-level object each), for scenes large enough to be
// traced through the BVH: the closest hit does not depend on the tree, the number of boxes a ray visits
// does.  Per node: for each axis, sort by box centre (ties: canonical index), sweep every split k, keep the
// first minimum of area(left) * k + area(right) * (m - k).  The same algorithm in the same f64 arithmetic as
// harness.py::_build_bvh_sah (tests/test_host_cpp.py compares the trees).
const size_t SAH_MIN_OBJECTS = 65;

double box_area(const double lo[3], const double hi[3]) {
    const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return 2.0 * (dx * dy + dy * dz + dz * dx);
}

int build_bvh_sah(const std::vector<std::pair<int, TopObject*>>& objs, std::vector<rc_bvh_node>& nodes, std::vector<TopObject*>& order) {
    const int idx = (int)nodes.size();
    nodes.push_back(rc_bvh_node());
    if (objs.size() == 1) {
        TopObject* o = objs[0].second;
        for (int a = 0; a < 3; ++a) { nodes[idx].bmin[a] = o->lo[a]; nodes[idx].bmax[a] = o->hi[a]; }
        nodes[idx].left = ~(int)order.size();
        nodes[idx].right = 1;
        order.push_back(o);
        return idx;
    }
    const size_t m = objs.size();
    bool have = false;
    double best_cost = 0.0;
    size_t best_k = 0;
    std::vector<std::pair<int, TopObject*>> best_sorted;
    std::vector<double> llo(3 * m), lhi(3 * m), rlo(3 * m), rhi(3 * m);
    for (int axis = 0; axis < 3; ++axis) {
        std::vector<std::pair<int, TopObject*>> srt(objs);
        std::sort(srt.begin(), srt.end(), [axis](const std::pair<int, TopObject*>& x, const std::pair<int, TopObject*>& y) {
            const double kx = x.second->lo[axis] + x.second->hi[axis], ky = y.second->lo[axis] + y.second->hi[axis];
            return kx < ky || (kx == ky && x.first < y.first);
        });
        for (size_t i = 0; i < m; ++i)
            for (int a = 0; a < 3; ++a) {
                llo[3 * i + a] = i ? std::min(llo[3 * (i - 1) + a], srt[i].second->lo[a]) : srt[i].second->lo[a];
                lhi[3 * i + a] = i ? std::max(lhi[3 * (i - 1) + a], srt[i].second->hi[a]) : srt[i].second->hi[a];
            }
        for (size_t i = m; i-- > 0;)
            for (int a = 0; a < 3; ++a) {
                rlo[3 * i + a] = i + 1 < m ? std::min(rlo[3 * (i + 1) + a], srt[i].second->lo[a]) : srt[i].second->lo[a];
                rhi[3 * i + a] = i + 1 < m ? std::max(rhi[3 * (i + 1) + a], srt[i].second->hi[a]) : srt[i].second->hi[a];
            }
        for (size_t k = 1; k < m; ++k) {
            const double left = box_area(&llo[3 * (k - 1)], &lhi[3 * (k - 1)]) * (double)k;
            const double right = box_area(&rlo[3 * k], &rhi[3 * k]) * (double)(m - k);
            const double cost = left + right;
            if (!have || cost < best_cost) { have = true; best_cost = cost; best_k = k; best_sorted = srt; }
        }
    }
    const std::vector<std::pair<int, TopObject*>> lhs(best_sorted.begin(), best_sorted.begin() + best_k), rhs(best_sorted.begin() + best_k, best_sorted.end());
    const int l = build_bvh_sah(lhs, nodes, order);
    const int r = build_bvh_sah(rhs, nodes, order);
    nodes[idx].left = l; nodes[idx].right = r;
    for (int a = 0; a < 3; ++a) {
        nodes[idx].bmin[a] = std::min(nodes[l].bmin[a], nodes[r].bmin[a]);
        nodes[idx].bmax[a] = std::max(nodes[l].bmax[a], nodes[r].bmax[a]);
    }
    return idx;
}

// Top-level objects (canonical order) -> structure-of-arrays primitives + host BVH: what the Rust shim
// does before rc_upload_scene.
void flatten_objects(SceneData& sd, std::vector<TopObject*> ordered) {
    // ---- canonical ids (SURVEY §8(c)): objects numbered 1..N by sorted lower-cased key; id = (object << 3) | side
    int n = 0;
    for (TopObject* o : ordered) {
        ++n;
        int inst = -1;
        if (o->has_rotate || o->has_translate) {
            rc_instance ri;
            std::memset(&ri, 0, sizeof(ri));
            if (o->has_rotate) {
                ri.flags |= 1;
                const double rad = o->rotate_deg * PI / 180.0;   // util.rs:5-7
                ri.sin_theta = std::sin(rad); ri.cos_theta = std::cos(rad);
            }
            if (o->has_translate) { ri.flags |= 2; std::memcpy(ri.offset, o->translate, sizeof(ri.offset)); }
            inst = (int)sd.instances.size();
            sd.instances.push_back(ri);
        }
        for (Prim& p : o->prims) { p.obj = n; p.instance = inst; }
        sd.object_keys.push_back(o->key);
    }
    // ---- BVH over the top-level objects; primitives stored in its depth-first leaf order
    if (!ordered.empty()) {
        std::vector<TopObject*> order;
        if (ordered.size() >= SAH_MIN_OBJECTS && sd.instances.empty()) {
            std::vector<std::pair<int, TopObject*>> indexed;
            for (size_t i = 0; i < ordered.size(); ++i) indexed.emplace_back((int)i, ordered[i]);
            build_bvh_sah(indexed, sd.nodes, order);
        } else {
            build_bvh(ordered, sd.nodes, order);
        }
        ordered = order;
        std::vector<int> first(ordered.size());
        int count = 0;
        for (size_t i = 0; i < ordered.size(); ++i) { first[i] = count; count += (int)ordered[i]->prims.size(); }
        for (auto& nd : sd.nodes)
            if (nd.left < 0) {
                const int oi = ~nd.left;
                nd.left = ~first[oi];
                nd.right = (int)ordered[oi]->prims.size();
            }
    }
    for (TopObject* o : ordered)
        for (const Prim& p : o->prims) {
            sd.prim_type.push_back(p.type);
            for (int k = 0; k < 5; ++k) sd.prim_data.push_back(p.data[k]);
            sd.prim_material.push_back(p.material);
            sd.prim_id.push_back(((uint32_t)p.obj << 3) | (uint32_t)p.side);
            sd.prim_instance.push_back(p.instance);
            for (int a = 0; a < 3; ++a) sd.prim_aabb.push_back(o->lo[a]);
            for (int a = 0; a < 3; ++a) sd.prim_aabb.push_back(o->hi[a]);
            for (int k = 0; k < 5; ++k) sd.prim_motion.push_back(p.motion[k]);
            if (p.moving) sd.has_motion = true;
        }
}

CameraConfig camera_config_of(const Node* n) {
    CameraConfig c;
    if (!n || !n->is_map()) return c;
    if (n->has("vfov")) { c.has_vfov = true; c.vfov = n->at("vfov").as_double(); }
    if (n->has("aperture")) { c.has_aperture = true; c.aperture = n->at("aperture").as_double(); }
    if (n->has("focus_distance")) { c.has_focus_distance = true; c.focus_distance = n->at("focus_distance").as_double(); }
    if (n->has("pos")) { c.has_pos = true; c.pos = vec3_of(n->at("pos"), "camera.pos"); }
    if (n->has("look_at")) { c.has_look_at = true; c.look_at = vec3_of(n->at("look_at"), "camera.look_at"); }
    return c;
}

// From<&ToneMapConfig> for Box<dyn ToneMap>, tone_map.rs:18-66
rc_tone_map tone_map_of(const Node* node) {
    rc_tone_map tm = make_tone_map_default();
    if (!node || node->is_null()) return tm;
    auto e = enum_of(*node, "tone_map");
    const Node& f = e.second;
    auto opt = [&](const char* k, double& dst) { if (f.has(k)) dst = f.at(k).as_double(); };
    if (e.first == "reinhard") { tm.type = RC_TONE_REINHARD; opt("max_white", tm.max_white); }
    else if (e.first == "hable") {
        tm.type = RC_TONE_HABLE;
        const char* names[6] = {"shoulder_strength", "linear_strength", "linear_angle", "toe_strength", "toe_numerator", "toe_denominator"};
        for (int i = 0; i < 6; ++i) opt(names[i], tm.hable[i]);
        opt("exposure_bias", tm.exposure_bias);
        opt("linear_white_point", tm.linear_white_point);
    } else if (e.first == "aces") {
        tm.type = RC_TONE_ACES;
        const char* names[2] = {"input_matrix", "output_matrix"};
        double* dst[2] = {tm.aces_in, tm.aces_out};
        for (int m = 0; m < 2; ++m)
            if (f.has(names[m])) {
                const Node& rows = f.at(names[m]).at("colors");
                if (!rows.is_seq() || rows.seq.size() != 3) throw yaml_lite::ParseError(std::string(names[m]) + ".colors needs 3 rows");
                for (int r = 0; r < 3; ++r) { Vec3 v = vec3_of(rows.seq[r], names[m]); dst[m][3 * r] = v.x; dst[m][3 * r + 1] = v.y; dst[m][3 * r + 2] = v.z; }
            }
    } else if (e.first == "none") tm.type = RC_TONE_NONE;
    else throw yaml_lite::ParseError("unknown tone map `" + e.first + "`");
    return tm;
}

RendererConfig renderer_of(const Node& n) {
    const std::string v = enum_of(n, "renderer").first;
    if (v == "cpu") return RendererConfig::Cpu;
    if (v == "cpupreview") return RendererConfig::CpuPreview;
    if (v == "cuda") return RendererConfig::Cuda;
    if (v == "cudapreview") return RendererConfig::CudaPreview;
    throw yaml_lite::ParseError("unknown variant `" + v + "`, expected one of `Cpu`, `CpuPreview`, `Cuda`, `CudaPreview`");
}

RenderConfig render_config_of(const Node* n) {
    RenderConfig r;
    if (!n || !n->is_map()) return r;
    auto get = [&](const char* k) { return n->has(k) ? (size_t)n->at(k).as_int() : (size_t)0; };
    r.samples = get("samples"); r.max_depth = get("max_depth"); r.num_threads_width = get("num_threads_width");
    r.num_threads_height = get("num_threads_height"); r.scale = get("scale");
    return r;
}

void json_doubles(std::ostringstream& o, const double* p, size_t n) {
    o << "[";
    char buf[40];
    for (size_t i = 0; i < n; ++i) { std::snprintf(buf, sizeof(buf), "%.17g", p[i]); o << (i ? "," : "") << buf; }
    o << "]";
}
template <typename T>
void json_ints(std::ostringstream& o, const T* p, size_t n) {
    o << "[";
    for (size_t i = 0; i < n; ++i) o << (i ? "," : "") << (long long)p[i];
    o << "]";
}

}  // namespace

// =================================================================================================
rc_tone_map make_tone_map_default() {
    rc_tone_map tm;
    std::memset(&tm, 0, sizeof(tm));
    tm.type = RC_TONE_NONE;
    tm.max_white = 25.0;                                              // tone_map.rs:21-23
    const double hable[6] = {0.15, 0.5, 0.1, 0.2, 0.02, 0.3};         // tone_map.rs:24-44
    std::memcpy(tm.hable, hable, sizeof(hable));
    tm.exposure_bias = 2.0; tm.linear_white_point = 11.2;
    const double in[9] = {0.59719, 0.35458, 0.04823, 0.07600, 0.90834, 0.01566, 0.02840, 0.13383, 0.83777};      // tone_map.rs:45-60
    const double out[9] = {1.60475, -0.53108, -0.07367, -0.10208, 1.10813, -0.00605, -0.00327, -0.07276, 1.07602};
    std::memcpy(tm.aces_in, in, sizeof(in));
    std::memcpy(tm.aces_out, out, sizeof(out));
    return tm;
}

Config::Config() { tone_map = make_tone_map_default(); }

Config Config::from_file(const std::string& file) {
    bool ok = false;
    const std::string text = read_file(file, ok);
    if (!ok) throw TracerError(TracerError::Configuration, "Config Error (" + file + "): configuration file \"" + file + "\" not found");
    Config cfg;
    try {
        Node doc = yaml_lite::parse(text);
        yaml_lite::lower_keys(doc);
        cfg.preview = render_config_of(doc.find("preview"));
        cfg.render = render_config_of(doc.find("render"));
        if (const Node* s = doc.find("screen")) {
            if (s->has("width")) cfg.screen.width = (size_t)s->at("width").as_int();
            if (s->has("height")) cfg.screen.height = (size_t)s->at("height").as_int();
        }
        if (doc.has("loader")) {
            auto e = enum_of(doc.at("loader"), "loader");
            if (e.first == "none") cfg.loader.kind = SceneLoaderConfig::None;
            else if (e.first == "yml") { cfg.loader.kind = SceneLoaderConfig::Yml; cfg.loader.path = e.second.at("path").as_string(); }
            else if (e.first == "random") cfg.loader.kind = SceneLoaderConfig::Random;
            else if (e.first == "sandbox") cfg.loader.kind = SceneLoaderConfig::Sandbox;
            else throw yaml_lite::ParseError("unknown loader `" + e.first + "`");
        }
        if (doc.has("image_action")) {
            const std::string v = enum_of(doc.at("image_action"), "image_action").first;
            if (v == "savepng") cfg.image_action = ImageActionConfig::SavePng;
            else if (v == "none") cfg.image_action = ImageActionConfig::None;
            else throw yaml_lite::ParseError("unknown image_action `" + v + "`");
        }
        if (doc.has("image_output_dir")) { cfg.has_image_output_dir = true; cfg.image_output_dir = doc.at("image_output_dir").as_string(); }
        if (doc.has("renderer")) cfg.renderer = renderer_of(doc.at("renderer"));
        if (doc.has("preview_renderer")) cfg.preview_renderer = renderer_of(doc.at("preview_renderer"));
        cfg.camera = camera_config_of(doc.find("camera"));
        cfg.tone_map = tone_map_of(doc.find("tone_map"));
        if (const Node* g = doc.find("gpu")) {
            if (g->has("seed")) cfg.gpu.seed = (uint64_t)g->at("seed").as_int();
            if (g->has("variant")) cfg.gpu.variant = yaml_lite::to_lower(g->at("variant").as_string()) == "wavefront" ? RC_VARIANT_WAVEFRONT : RC_VARIANT_MEGAKERNEL;
            if (g->has("sampler")) cfg.gpu.sampler = yaml_lite::to_lower(g->at("sampler").as_string()) == "rejection" ? RC_SAMPLER_REJECTION : RC_SAMPLER_DIRECT;
            if (g->has("split")) cfg.gpu.split = yaml_lite::to_lower(g->at("split").as_string()) == "samples" ? RC_SPLIT_SAMPLES : RC_SPLIT_TILES;
            if (g->has("specialize")) cfg.gpu.specialize = (int)g->at("specialize").as_int();
            if (g->has("devices") && g->at("devices").is_seq())
                for (auto& d : g->at("devices").seq) cfg.gpu.devices.push_back((int32_t)d.as_int());
            if (const Node* a = g->find("adaptive")) {
                cfg.gpu.adaptive = true;
                if (a->has("threshold")) cfg.gpu.adaptive_threshold = a->at("threshold").as_double();
                if (a->has("min_samples")) cfg.gpu.adaptive_min_samples = (int32_t)a->at("min_samples").as_int();
            }
            if (const Node* dn = g->find("denoise")) {
                cfg.gpu.denoise = true;
                if (dn->has("levels")) cfg.gpu.denoise_levels = (int32_t)dn->at("levels").as_int();
                if (dn->has("sigma_l")) cfg.gpu.denoise_sigma_l = dn->at("sigma_l").as_double();
                if (dn->has("sigma_n")) cfg.gpu.denoise_sigma_n = dn->at("sigma_n").as_double();
                if (dn->has("sigma_z")) cfg.gpu.denoise_sigma_z = dn->at("sigma_z").as_double();
            }
            if (cfg.gpu.adaptive && cfg.gpu.denoise) throw TracerError(TracerError::Configuration, "Config Error (" + file + "): gpu.adaptive and gpu.denoise exclude each other");
        }
    } catch (const yaml_lite::ParseError& e) {
        throw TracerError(TracerError::Configuration, "Config Error (" + file + "): " + e.what());
    }
    return cfg;
}

CameraData merge_camera(const CameraConfig& a, const CameraConfig& b) {   // camera.rs:404-464: scene over config, then defaults
    CameraData c;
    if (a.has_vfov) c.vfov = a.vfov; else if (b.has_vfov) c.vfov = b.vfov;
    if (a.has_aperture) c.aperture = a.aperture; else if (b.has_aperture) c.aperture = b.aperture;
    if (a.has_focus_distance) c.focus_distance = a.focus_distance; else if (b.has_focus_distance) c.focus_distance = b.focus_distance;
    if (a.has_pos) c.pos = a.pos; else if (b.has_pos) c.pos = b.pos;
    if (a.has_look_at) c.look_at = a.look_at; else if (b.has_look_at) c.look_at = b.look_at;
    return c;
}

rc_camera make_camera(const CameraData& cam, const Image& image) {
    auto sub = [](Vec3 a, Vec3 b) { return Vec3{a.x - b.x, a.y - b.y, a.z - b.z}; };
    auto mul = [](Vec3 a, double s) { return Vec3{a.x * s, a.y * s, a.z * s}; };
    auto cross = [](Vec3 a, Vec3 b) { return Vec3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; };
    auto unit = [](Vec3 a) { const double n = std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); return Vec3{a.x / n, a.y / n, a.z / n}; };
    const double aspect = (double)image.width / (double)image.height;   // image.rs:12-16
    const double h = std::tan((cam.vfov * PI / 180.0) / 2.0);
    const double vh = 2.0 * h, vw = aspect * vh, fd = cam.focus_distance;
    const Vec3 forward = unit(sub(cam.pos, cam.look_at));
    const Vec3 right = unit(cross(Vec3{0.0, 1.0, 0.0}, forward));
    const Vec3 up = cross(forward, right);
    const Vec3 horizontal = mul(right, fd * vw), vertical = mul(up, fd * vh);
    const Vec3 ulc{cam.pos.x + vertical.x / 2.0 - horizontal.x / 2.0 - fd * forward.x,
                   cam.pos.y + vertical.y / 2.0 - horizontal.y / 2.0 - fd * forward.y,
                   cam.pos.z + vertical.z / 2.0 - horizontal.z / 2.0 - fd * forward.z};
    rc_camera c;
    std::memset(&c, 0, sizeof(c));
    auto put = [](double* d, Vec3 v) { d[0] = v.x; d[1] = v.y; d[2] = v.z; };
    put(c.origin, cam.pos); put(c.upper_left_corner, ulc); put(c.forward, forward); put(c.right, right); put(c.up, up);
    put(c.horizontal, horizontal); put(c.vertical, vertical);
    c.vfov = cam.vfov; c.viewport_width = vw; c.viewport_height = vh;
    c.lens_radius = cam.aperture * 0.5; c.focus_distance = fd; c.time_a = 0.0; c.time_b = 1.0;
    return c;
}

// =================================================================================================
SceneData::SceneData() {
    std::memset(&scene, 0, sizeof(scene));
    tone_map = make_tone_map_default();
}

namespace {
// Sandbox::load_cornell_box (scene/sandbox.rs:39-81) as additions to the parsed, lower-cased cornell_box.yml: two
// white Lambertian boxes, each rotated about y and then translated, black background, the Cornell camera.
void sandbox_additions(Node& doc) {
    const Node extra = yaml_lite::parse(
        "textures:\n"
        "  sandbox_white: {solidcolor: {color: {color: [0.63, 0.63, 0.63]}}}\n"
        "materials:\n"
        "  sandbox_white: {lambertian: {texture: sandbox_white}}\n"
        "geometry:\n"
        "  sandbox_box1: {box: {min: {pos: [0.0, 0.0, 0.0]}, max: {pos: [165.0, 330.0, 165.0]}, material: sandbox_white}}\n"
        "  sandbox_box1_rotate: {rotatey: {key: sandbox_box1, degrees: 15.0}}\n"
        "  sandbox_box1_translate: {translate: {key: sandbox_box1, pos: [265.0, 0.0, 295.0]}}\n"
        "  sandbox_box2: {box: {min: {pos: [0.0, 0.0, 0.0]}, max: {pos: [165.0, 165.0, 165.0]}, material: sandbox_white}}\n"
        "  sandbox_box2_rotate: {rotatey: {key: sandbox_box2, degrees: -18.0}}\n"
        "  sandbox_box2_translate: {translate: {key: sandbox_box2, pos: [130.0, 0.0, 65.0]}}\n"
        "background: {solidcolor: {pos: [0.0, 0.0, 0.0]}}\n"
        "camera: {vfov: 40.0, aperture: 0.0, focus_distance: 10000.0, pos: {pos: [278.0, 278.0, -800.0]}, look_at: {pos: [278.0, 278.0, 0.0]}}\n");
    auto section = [&](const std::string& name) -> Node& {
        for (auto& kv : doc.map) if (kv.first == name) return kv.second;
        doc.map.emplace_back(name, Node());
        doc.map.back().second.kind = Node::Map;
        return doc.map.back().second;
    };
    for (const char* name : {"textures", "materials", "geometry"})
        for (auto& kv : extra.at(name).map) section(name).map.push_back(kv);
    section("background") = extra.at("background");
    section("camera") = extra.at("camera");
    for (size_t i = 0; i < doc.map.size(); ++i)
        if (doc.map[i].first == "tone_map") { doc.map.erase(doc.map.begin() + i); break; }
}
}  // namespace

std::unique_ptr<SceneData> SceneData::load_sandbox(const std::string& cornell_box_yml, uint64_t seed) {
    return load_yml(cornell_box_yml, seed, {}, true);
}

std::unique_ptr<SceneData> SceneData::load_yml(const std::string& path, uint64_t seed, const std::vector<std::string>& image_dirs, bool sandbox) {
    bool ok = false;
    const std::string text = read_file(path, ok);
    auto cfg_err = [&](const std::string& m) { return TracerError(TracerError::Configuration, "Config Error (" + path + "): " + m); };
    if (!ok) throw cfg_err("configuration file \"" + path + "\" not found");
    std::unique_ptr<SceneData> sd(new SceneData());
    Node doc;
    try {
        doc = yaml_lite::parse(text);
    } catch (const yaml_lite::ParseError& e) { throw cfg_err(e.what()); }
    if (!doc.is_map()) throw cfg_err("not a mapping");
    yaml_lite::lower_keys(doc);
    if (sandbox) sandbox_additions(doc);
    for (const char* req : {"textures", "materials", "geometry"})
        if (!doc.find(req) || !doc.at(req).is_map()) throw cfg_err(std::string("missing field `") + req + "`");
    try {
        // ---- textures: everything but Checkered first (yml.rs:177-210), in sorted key order so that indices
        // are deterministic (the reference iterates a HashMap), then Checkered (yml.rs:212-243)
        std::map<std::string, int> tex_index;
        std::vector<std::pair<std::string, Node>> checkered;
        const Node& tnode = doc.at("textures");
        for (const std::string& key : tnode.sorted_keys()) {
            auto e = enum_of(tnode.at(key), "texture " + key);
            const Node& f = e.second;
            rc_texture t;
            std::memset(&t, 0, sizeof(t));
            if (e.first == "checkered") { checkered.emplace_back(key, f); continue; }
            if (e.first == "solidcolor") {
                t.type = RC_TEX_SOLID;
                Vec3 c = vec3_of(f.at("color"), "texture " + key + ".color");
                t.color[0] = c.x; t.color[1] = c.y; t.color[2] = c.z;
            } else if (e.first == "image") {   // TextureImage::try_new, texture/image.rs:17-25
                t.type = RC_TEX_IMAGE;
                t.a = (int32_t)sd->image_pixels.size();
                const std::string rel = f.at("path").as_string();
                std::vector<std::string> cands = {rel, dir_of(path) + "/" + rel};
                for (auto& d : image_dirs) cands.push_back(d + "/" + base_of(rel));
                std::string found;
                for (auto& c : cands) if (file_exists(c)) { found = c; break; }
                if (found.empty()) throw TracerError(TracerError::FailedToOpenImage, "Failed to open image " + rel + ": No such file or directory");
                bool iok = false;
                const std::string bytes = read_file(found, iok);
                try {
                    jpeg_baseline::Image im = jpeg_baseline::decode((const uint8_t*)bytes.data(), bytes.size());
                    rc_image ri;
                    ri.width = im.width; ri.height = im.height; ri.rgba = nullptr;
                    sd->image_pixels.push_back(std::move(im.rgba));
                    sd->images.push_back(ri);
                } catch (const jpeg_baseline::Error& je) {
                    throw TracerError(TracerError::FailedToOpenImage, "Failed to open image " + rel + ": " + je.what());
                }
            } else if (e.first == "noise") {
                t.type = RC_TEX_NOISE;
                t.a = (int32_t)sd->perlin.size();
                t.b = (int32_t)f.at("depth").as_int();
                t.scale = f.at("scale").as_double();
                Vec3 c = vec3_of(f.at("color"), "texture " + key + ".color");
                t.color[0] = c.x; t.color[1] = c.y; t.color[2] = c.z;
                sd->perlin.push_back(make_perlin(seed, t.a));
            } else throw yaml_lite::ParseError("unknown texture variant `" + e.first + "`");
            tex_index[key] = (int)sd->textures.size();
            sd->textures.push_back(t);
        }
        std::sort(checkered.begin(), checkered.end(), [](const std::pair<std::string, Node>& a, const std::pair<std::string, Node>& b) { return a.first < b.first; });
        for (auto& kv : checkered) {
            const std::string ta = kv.second.at("texture_a").as_string(), tb = kv.second.at("texture_b").as_string();
            for (const std::string& name : {ta, tb})
                if (!tex_index.count(name))
                    throw TracerError(TracerError::SceneLoad, "Scene failed to load: Checkered texture \"" + kv.first + "\" expected texture \"" + ta + "\" to exist.");
            rc_texture t;
            std::memset(&t, 0, sizeof(t));
            t.type = RC_TEX_CHECKER; t.a = tex_index[ta]; t.b = tex_index[tb]; t.scale = 10.0;   // checkered.rs:19
            tex_index[kv.first] = (int)sd->textures.size();
            sd->textures.push_back(t);
        }
        // ---- materials, yml.rs:245-286
        std::map<std::string, int> mat_index;
        const Node& mnode = doc.at("materials");
        for (const std::string& key : mnode.sorted_keys()) {
            auto e = enum_of(mnode.at(key), "material " + key);
            const Node& f = e.second;
            rc_material m;
            std::memset(&m, 0, sizeof(m));
            const char* label = nullptr;
            if (e.first == "lambertian") { m.type = RC_MAT_LAMBERTIAN; label = "lambertian"; }
            else if (e.first == "metal") { m.type = RC_MAT_METAL; label = "metal"; }
            else if (e.first == "diffuselight") { m.type = RC_MAT_DIFFUSE_LIGHT; label = "diffuse light"; }
            else if (e.first == "dialectric") { m.type = RC_MAT_DIELECTRIC; m.param = f.at("refraction_index").as_double(); }
            else throw yaml_lite::ParseError("unknown material variant `" + e.first + "`");
            if (label) {
                const Node* tk = f.find("texture");
                if (!tk) tk = f.find("texture_key");
                const std::string tex_key = tk && tk->is_scalar() ? tk->scalar : std::string("None");
                if (!tex_index.count(tex_key))
                    throw TracerError(TracerError::SceneLoad, "Scene failed to load: Failed to find texture \"" + tex_key + "\" for " + label + " material \"" + key + "\"");
                m.texture = tex_index[tex_key];
                if (m.type == RC_MAT_METAL) m.param = f.at("fuzz").as_double();
            }
            mat_index[key] = (int)sd->materials.size();
            sd->materials.push_back(m);
        }
        auto mat = [&](const Node& f) {
            const std::string name = f.at("material").as_string();
            if (!mat_index.count(name)) throw TracerError(TracerError::UnknownMaterial, "Unknown Material " + name + ".");
            return mat_index[name];
        };
        // ---- geometry, yml.rs:292-399
        std::map<std::string, TopObject> objects;
        std::vector<std::pair<std::string, double>> rotations;
        std::vector<std::pair<std::string, Vec3>> translations;
        const Node& gnode = doc.at("geometry");
        for (const std::string& key : gnode.sorted_keys()) {
            auto e = enum_of(gnode.at(key), "geometry " + key);
            const Node& f = e.second;
            const std::string& v = e.first;
            if (v == "sphere") {
                const Vec3 p = vec3_of(f, "geometry " + key);
                const double r = f.at("radius").as_double();
                TopObject o;
                o.key = key;
                o.prims.push_back(Prim(RC_PRIM_SPHERE, {p.x, p.y, p.z, r, 0.0}, mat(f), 0, 0, -1));
                const double a[3] = {p.x - r, p.y - r, p.z - r}, b[3] = {p.x + r, p.y + r, p.z + r};   // sphere.rs:72-77
                aabb_of(a, b, o.lo, o.hi);
                o.pos[0] = p.x; o.pos[1] = p.y; o.pos[2] = p.z;
                objects[key] = o;
            } else if (v == "xyrect" || v == "xzrect" || v == "yzrect") {
                const int kind = v == "xyrect" ? RC_PRIM_XY_RECT : (v == "xzrect" ? RC_PRIM_XZ_RECT : RC_PRIM_YZ_RECT);
                const char* names[3][4] = {{"x0", "x1", "y0", "y1"}, {"x0", "x1", "z0", "z1"}, {"y0", "y1", "z0", "z1"}};
                const char* const* n = names[kind - 1];
                TopObject o;
                o.key = key;
                o.prims.push_back(rect_prim(kind, f.at(n[0]).as_double(), f.at(n[1]).as_double(), f.at(n[2]).as_double(),
                                            f.at(n[3]).as_double(), f.at("k").as_double(), mat(f), o.lo, o.hi, o.pos));
                objects[key] = o;
            } else if (v == "box") {   // box.rs:21-77, geometry_creation.rs:98-106
                const Vec3 mn = vec3_of(f.at("min"), "box.min"), mx = vec3_of(f.at("max"), "box.max");
                const int m = mat(f);
                const double s[6][6] = {{(double)RC_PRIM_XY_RECT, mn.x, mx.x, mn.y, mx.y, mx.z}, {(double)RC_PRIM_XY_RECT, mn.x, mx.x, mn.y, mx.y, mn.z},
                                        {(double)RC_PRIM_XZ_RECT, mn.x, mx.x, mn.z, mx.z, mx.y}, {(double)RC_PRIM_XZ_RECT, mn.x, mx.x, mn.z, mx.z, mn.y},
                                        {(double)RC_PRIM_YZ_RECT, mn.y, mx.y, mn.z, mx.z, mx.x}, {(double)RC_PRIM_YZ_RECT, mn.y, mx.y, mn.z, mx.z, mn.x}};
                TopObject o;
                o.key = key;
                for (int i = 0; i < 6; ++i) {
                    double lo[3], hi[3], pos[3];
                    Prim p = rect_prim((int)s[i][0], s[i][1], s[i][2], s[i][3], s[i][4], s[i][5], m, lo, hi, pos);
                    p.side = i;
                    o.prims.push_back(p);
                }
                const double a[3] = {mn.x, mn.y, mn.z}, b[3] = {mx.x, mx.y, mx.z};
                aabb_of(a, b, o.lo, o.hi);
                o.pos[0] = mn.x; o.pos[1] = mn.y; o.pos[2] = mn.z;
                objects[key] = o;
            } else if (v == "rotatey") rotations.emplace_back(yaml_lite::to_lower(f.at("key").as_string()), f.at("degrees").as_double());
            else if (v == "translate") translations.emplace_back(yaml_lite::to_lower(f.at("key").as_string()), vec3_of(f, "geometry " + key));
            else throw yaml_lite::ParseError("unknown geometry variant `" + v + "`");
        }
        // rotations first, then translations; each is keyed by its CHILD's name and the wrapper takes that
        // name (yml.rs:401-439, SURVEY Q26)
        for (auto& r : rotations) {
            if (!objects.count(r.first))
                throw TracerError(TracerError::SceneLoad, "Scene failed to load: Rotation_Y \"" + r.first + "\" did not have any child with key \"" + r.first + "\"");
            TopObject& o = objects[r.first];
            o.has_rotate = true; o.rotate_deg = r.second;
            rotate_y_aabb(o, r.second);
        }
        for (auto& t : translations) {
            if (!objects.count(t.first))
                throw TracerError(TracerError::SceneLoad, "Scene failed to load: Translation \"" + t.first + "\" did not have any child with key \"" + t.first + "\"");
            TopObject& o = objects[t.first];
            o.has_translate = true;
            o.translate[0] = t.second.x; o.translate[1] = t.second.y; o.translate[2] = t.second.z;
            for (int a = 0; a < 3; ++a) { o.lo[a] += o.translate[a]; o.hi[a] += o.translate[a]; }   // translate.rs:44-47
        }
        std::vector<TopObject*> ordered;
        for (auto& kv : objects) ordered.push_back(&kv.second);   // std::map iterates in sorted key order
        flatten_objects(*sd, ordered);
        // ---- background, yml.rs:443-453; default Sky (background_color.rs:18-25)
        rc_scene& c = sd->scene;
        const Node* bg = doc.find("background");
        if (!bg || bg->is_null()) {
            c.bg_type = RC_BG_SKY;
            c.bg_a[0] = c.bg_a[1] = c.bg_a[2] = 1.0;
            c.bg_b[0] = 0.5; c.bg_b[1] = 0.7; c.bg_b[2] = 1.0;
        } else {
            auto e = enum_of(*bg, "background");
            if (e.first == "sky") {
                c.bg_type = RC_BG_SKY;
                Vec3 t = vec3_of(e.second.at("top"), "sky.top"), b = vec3_of(e.second.at("bottom"), "sky.bottom");
                c.bg_a[0] = t.x; c.bg_a[1] = t.y; c.bg_a[2] = t.z; c.bg_b[0] = b.x; c.bg_b[1] = b.y; c.bg_b[2] = b.z;
            } else if (e.first == "solidcolor") {
                c.bg_type = RC_BG_SOLID;
                Vec3 t = vec3_of(e.second, "background");
                c.bg_a[0] = t.x; c.bg_a[1] = t.y; c.bg_a[2] = t.z;
            } else throw yaml_lite::ParseError("unknown background `" + e.first + "`");
        }
        sd->camera = camera_config_of(doc.find("camera"));
        if (doc.has("tone_map")) { sd->has_tone_map = true; sd->tone_map = tone_map_of(doc.find("tone_map")); }
    } catch (const yaml_lite::ParseError& e) { throw cfg_err(e.what()); }

    sd->wire();
    return sd;
}

namespace {
// Sequential uniforms for procedural scenes: Philox4x32-10(counter = (n, 0, 0, 3 << 24), key = seed), four
// 24-bit uniforms per block, consumed in order (the same stream as the Python harness's _SceneRng).  The
// reference draws from the OS-seeded thread_rng (util.rs:9-23): its Random scene differs on every run.
struct SceneRng {
    uint32_t key[2];
    uint32_t n = 0;
    double buf[4];
    int left = 0;
    explicit SceneRng(uint64_t seed) { key[0] = (uint32_t)seed; key[1] = (uint32_t)(seed >> 32); }
    double uniform() {
        if (left == 0) {
            const uint32_t ctr[4] = {n++, 0u, 0u, 3u << 24};
            uint32_t r[4];
            philox4x32(ctr, key, r);
            for (int k = 0; k < 4; ++k) buf[k] = (double)(r[k] >> 8) / 16777216.0;
            left = 4;
        }
        return buf[4 - left--];
    }
    double range(double lo, double hi) { return lo + (hi - lo) * uniform(); }   // random_double_range, util.rs:19-23
};
}  // namespace

// Random::load, scene/random.rs:25-95
std::unique_ptr<SceneData> SceneData::load_random(uint64_t seed) {
    std::unique_ptr<SceneData> sd(new SceneData());
    SceneRng rng(seed);
    std::vector<TopObject> objects;
    objects.reserve(512);
    auto solid = [&](double r, double g, double b) {
        rc_texture t;
        std::memset(&t, 0, sizeof(t));
        t.type = RC_TEX_SOLID; t.color[0] = r; t.color[1] = g; t.color[2] = b;
        sd->textures.push_back(t);
        return (int)sd->textures.size() - 1;
    };
    auto material = [&](int kind, int texture, double param) {
        rc_material m;
        std::memset(&m, 0, sizeof(m));
        m.type = kind; m.texture = texture; m.param = param;
        sd->materials.push_back(m);
        return (int)sd->materials.size() - 1;
    };
    auto sphere = [&](const double c[3], double radius, int mat, const double* c2) {
        TopObject o;
        char key[16];
        std::snprintf(key, sizeof(key), "obj%04d", (int)objects.size());
        o.key = key;
        Prim p(RC_PRIM_SPHERE, {c[0], c[1], c[2], radius, 0.0}, mat, 0, 0, -1);
        const double a[3] = {c[0] - radius, c[1] - radius, c[2] - radius}, b[3] = {c[0] + radius, c[1] + radius, c[2] + radius};
        aabb_of(a, b, o.lo, o.hi);
        if (c2) {   // create_movable_sphere, geometry_creation.rs:23-38; box = union of both ends, moving_sphere.rs:90-99
            p.type = RC_PRIM_MOVING_SPHERE; p.moving = true;
            p.motion[0] = c2[0]; p.motion[1] = c2[1]; p.motion[2] = c2[2]; p.motion[3] = 0.0; p.motion[4] = 1.0;
            for (int k = 0; k < 3; ++k) { o.lo[k] = std::min(o.lo[k], c2[k] - radius); o.hi[k] = std::max(o.hi[k], c2[k] + radius); }
        }
        o.prims.push_back(p);
        o.pos[0] = c[0]; o.pos[1] = c[1]; o.pos[2] = c[2];
        objects.push_back(o);
    };
    const int even = solid(0.2, 0.3, 0.1), odd = solid(0.9, 0.9, 0.9);
    rc_texture chk;
    std::memset(&chk, 0, sizeof(chk));
    chk.type = RC_TEX_CHECKER; chk.a = even; chk.b = odd; chk.scale = 10.0;
    sd->textures.push_back(chk);
    const double ground[3] = {0.0, -1000.0, 0.0};
    sphere(ground, 1000.0, material(RC_MAT_LAMBERTIAN, (int)sd->textures.size() - 1, 0.0), nullptr);
    for (int a = -11; a < 11; ++a)
        for (int b = -11; b < 11; ++b) {
            const double choose_mat = rng.uniform();
            const double cx = a + 0.9 * rng.uniform();
            const double cz = b + 0.9 * rng.uniform();
            const double center[3] = {cx, 0.2, cz};
            if (std::sqrt((cx - 4.0) * (cx - 4.0) + (0.2 - 0.2) * (0.2 - 0.2) + cz * cz) > 0.9) {
                if (choose_mat < 0.8) {   // diffuse, moving
                    double c1[3], c2[3];
                    for (double& v : c1) v = rng.uniform();
                    for (double& v : c2) v = rng.uniform();
                    const double dy = rng.range(0.0, 0.5);
                    const double center2[3] = {cx, 0.2 + dy, cz};
                    sphere(center, 0.2, material(RC_MAT_LAMBERTIAN, solid(c1[0] * c2[0], c1[1] * c2[1], c1[2] * c2[2]), 0.0), center2);
                } else if (choose_mat > 0.95) {   // metal
                    double al[3];
                    for (double& v : al) v = rng.range(0.5, 1.0);
                    const double fuzz = rng.range(0.0, 0.5);
                    sphere(center, 0.2, material(RC_MAT_METAL, solid(al[0], al[1], al[2]), fuzz), nullptr);
                } else sphere(center, 0.2, material(RC_MAT_DIELECTRIC, 0, 1.5), nullptr);   // glass
            }
        }
    const double b1[3] = {0.0, 1.0, 0.0}, b2[3] = {-4.0, 1.0, 0.0}, b3[3] = {4.0, 1.0, 0.0};
    sphere(b1, 1.0, material(RC_MAT_DIELECTRIC, 0, 1.5), nullptr);
    sphere(b2, 1.0, material(RC_MAT_LAMBERTIAN, solid(0.4, 0.2, 0.1), 0.0), nullptr);
    sphere(b3, 1.0, material(RC_MAT_METAL, solid(0.7, 0.6, 0.5), 0.0), nullptr);
    std::vector<TopObject*> ordered;
    for (auto& o : objects) ordered.push_back(&o);
    flatten_objects(*sd, ordered);
    rc_scene& c = sd->scene;
    c.bg_type = RC_BG_SKY;
    c.bg_a[0] = c.bg_a[1] = c.bg_a[2] = 1.0;
    c.bg_b[0] = 0.5; c.bg_b[1] = 0.7; c.bg_b[2] = 1.0;
    CameraConfig& cam = sd->camera;
    cam.has_vfov = cam.has_aperture = cam.has_focus_distance = cam.has_pos = cam.has_look_at = true;
    cam.vfov = 20.0; cam.aperture = 0.1; cam.focus_distance = 10.0;
    cam.pos = Vec3{0.0, 2.0, 10.0}; cam.look_at = Vec3{0.0, 0.0, 0.0};
    sd->wire();
    return sd;
}

void SceneData::wire() {
    // ---- wire the rc_scene to the owned arrays
    rc_scene& c = scene;
    c.n_prims = (int32_t)prim_type.size();
    c.prim_type = prim_type.data(); c.prim_data = prim_data.data(); c.prim_material = prim_material.data();
    c.prim_id = prim_id.data(); c.prim_instance = prim_instance.data(); c.prim_aabb = prim_aabb.data();
    c.n_instances = (int32_t)instances.size(); c.instances = instances.data();
    c.n_materials = (int32_t)materials.size(); c.materials = materials.data();
    c.n_textures = (int32_t)textures.size(); c.textures = textures.data();
    for (size_t i = 0; i < images.size(); ++i) images[i].rgba = image_pixels[i].data();
    c.n_images = (int32_t)images.size(); c.images = images.data();
    c.n_perlin = (int32_t)perlin.size(); c.perlin = perlin.data();
    c.n_nodes = (int32_t)nodes.size(); c.nodes = nodes.data();
    c.prim_motion = has_motion ? prim_motion.data() : nullptr;
}

std::string SceneData::to_json() const {
    std::ostringstream o;
    o << "{\"prim_type\":"; json_ints(o, prim_type.data(), prim_type.size());
    o << ",\"prim_data\":"; json_doubles(o, prim_data.data(), prim_data.size());
    o << ",\"prim_material\":"; json_ints(o, prim_material.data(), prim_material.size());
    o << ",\"prim_id\":"; json_ints(o, prim_id.data(), prim_id.size());
    o << ",\"prim_instance\":"; json_ints(o, prim_instance.data(), prim_instance.size());
    o << ",\"prim_aabb\":"; json_doubles(o, prim_aabb.data(), prim_aabb.size());
    o << ",\"prim_motion\":"; json_doubles(o, prim_motion.data(), prim_motion.size());
    o << ",\"instances\":[";
    for (size_t i = 0; i < instances.size(); ++i) {
        const double v[5] = {instances[i].sin_theta, instances[i].cos_theta, instances[i].offset[0], instances[i].offset[1], instances[i].offset[2]};
        o << (i ? "," : "") << "{\"flags\":" << instances[i].flags << ",\"v\":"; json_doubles(o, v, 5); o << "}";
    }
    o << "],\"materials\":[";
    for (size_t i = 0; i < materials.size(); ++i) {
        o << (i ? "," : "") << "{\"type\":" << materials[i].type << ",\"texture\":" << materials[i].texture << ",\"param\":";
        json_doubles(o, &materials[i].param, 1); o << "}";
    }
    o << "],\"textures\":[";
    for (size_t i = 0; i < textures.size(); ++i) {
        const double v[4] = {textures[i].color[0], textures[i].color[1], textures[i].color[2], textures[i].scale};
        o << (i ? "," : "") << "{\"type\":" << textures[i].type << ",\"a\":" << textures[i].a << ",\"b\":" << textures[i].b << ",\"v\":";
        json_doubles(o, v, 4); o << "}";
    }
    o << "],\"nodes\":[";
    for (size_t i = 0; i < nodes.size(); ++i) {
        o << (i ? "," : "") << "{\"left\":" << nodes[i].left << ",\"right\":" << nodes[i].right << ",\"bmin\":";
        json_doubles(o, nodes[i].bmin, 3); o << ",\"bmax\":"; json_doubles(o, nodes[i].bmax, 3); o << "}";
    }
    o << "],\"perlin0\":";
    if (!perlin.empty()) json_doubles(o, &perlin[0].ran_vec[0][0], 768); else o << "[]";
    o << ",\"images\":[";
    for (size_t i = 0; i < images.size(); ++i) {
        unsigned long long sum = 0;
        for (uint8_t b : image_pixels[i]) sum += b;
        o << (i ? "," : "") << "{\"width\":" << images[i].width << ",\"height\":" << images[i].height << ",\"byte_sum\":" << sum << "}";
    }
    o << "],\"bg_type\":" << scene.bg_type << ",\"bg_a\":"; json_doubles(o, scene.bg_a, 3);
    o << ",\"bg_b\":"; json_doubles(o, scene.bg_b, 3);
    o << ",\"object_keys\":[";
    for (size_t i = 0; i < object_keys.size(); ++i) o << (i ? "," : "") << "\"" << object_keys[i] << "\"";
    o << "]}";
    return o.str();
}

// =================================================================================================
namespace {
void check(int status, const char* what) {
    if (status == RC_OK) return;
    const std::string text = std::string(what) + ": " + rc_last_error();
    if (status == RC_ERR_CANCELLED) throw TracerError(TracerError::CancelEvent, "Cancel event");
    throw TracerError(TracerError::Cuda, "CUDA renderer error (" + std::to_string(status) + "): " + text);
}

size_t get_highest_divdable(size_t value, size_t div) {   // cpu_scaled.rs:17-23
    if (div < 1) div = 1;
    while ((value % div) != 0) div -= 1;
    return div;
}
}  // namespace

namespace {
// ONE rc_ctx per process and device list, shared by the full and the preview renderer (both are made by
// make_renderer, main.rs:127-129, and never render at the same time): the scene is uploaded once, whichever of the
// two renders first after a change.  Destroyed with its last renderer.
std::shared_ptr<rc_ctx> acquire_context(const GpuConfig& gpu) {
    static std::mutex mutex;
    static std::map<std::vector<int32_t>, std::weak_ptr<rc_ctx>> live;
    std::lock_guard<std::mutex> lock(mutex);
    std::weak_ptr<rc_ctx>& slot = live[gpu.devices];
    if (std::shared_ptr<rc_ctx> alive = slot.lock()) return alive;
    rc_ctx* raw = nullptr;
    const int32_t* devs = gpu.devices.empty() ? nullptr : gpu.devices.data();
    check(rc_create(devs, gpu.devices.empty() ? 1 : (int32_t)gpu.devices.size(), &raw), "rc_create");
    std::shared_ptr<rc_ctx> fresh(raw, [](rc_ctx* c) { rc_destroy(c); });
    slot = fresh;
    return fresh;
}
}  // namespace

CudaRenderer::CudaRenderer(const RenderConfig& config, const GpuConfig& gpu)
    : config_(config), gpu_(gpu), shared_(acquire_context(gpu)), ctx_(shared_.get()) {}

CudaRenderer::~CudaRenderer() {}

rc_stats CudaRenderer::stats() const {
    rc_stats s;
    check(rc_get_stats(ctx_, &s), "rc_get_stats");
    return s;
}

void CudaRenderer::sync_scene(const RenderData& rd) {
    if (!rd.scene || !rd.camera_data || !rd.image) throw TracerError(TracerError::Cuda, "RenderData is incomplete");
    if (rd.scene->changed) {   // re-upload when bvh.changed(), main.rs:178-183
        check(rc_upload_scene(ctx_, &rd.scene->scene), "rc_upload_scene");
        rd.scene->changed = false;
    }
    check(rc_set_camera(ctx_, rd.camera_data), "rc_set_camera");
}

rc_params CudaRenderer::params(const RenderData& rd) const {
    rc_params p;
    std::memset(&p, 0, sizeof(p));
    p.width = (int32_t)rd.image->width; p.height = (int32_t)rd.image->height;
    p.samples = (int32_t)config_.samples; p.max_depth = (int32_t)config_.max_depth;
    p.seed = gpu_.seed; p.variant = gpu_.variant; p.sampler = gpu_.sampler; p.split = gpu_.split;
    p.rank = 0; p.world = 1;
    p.specialize = (gpu_.variant == RC_VARIANT_MEGAKERNEL && gpu_.sampler == RC_SAMPLER_DIRECT) ? gpu_.specialize : 0;
    return p;
}

void CudaRenderer::render(const RenderData& rd, const DataWriter<ImageBufferEvent>& writer) {
    if (rd.cancel_event && *rd.cancel_event) throw TracerError(TracerError::CancelEvent, "Cancel event");   // cpu.rs:79-83
    sync_scene(rd);
    const rc_params p = params(rd);
    const size_t n = rd.image->width * rd.image->height;
    ImageBufferEvent ev;
    ev.rgb.resize(n);
    static_assert(sizeof(Color) == 3 * sizeof(double), "Color is three packed doubles");
    if (gpu_.adaptive) {
        rc_adaptive a;
        std::memset(&a, 0, sizeof(a));
        a.min_samples = gpu_.adaptive_min_samples;
        a.threshold = gpu_.adaptive_threshold;
        check(rc_render_adaptive(ctx_, &p, &a, reinterpret_cast<double*>(ev.rgb.data()), nullptr, nullptr, rd.cancel_event),
              "rc_render_adaptive");
    } else if (gpu_.denoise) {
        rc_denoise dn;
        std::memset(&dn, 0, sizeof(dn));
        dn.levels = gpu_.denoise_levels;
        dn.sigma_l = gpu_.denoise_sigma_l; dn.sigma_n = gpu_.denoise_sigma_n; dn.sigma_z = gpu_.denoise_sigma_z;
        check(rc_render_denoised(ctx_, &p, &dn, reinterpret_cast<double*>(ev.rgb.data()), nullptr, rd.cancel_event), "rc_render_denoised");
    } else {
        check(rc_render(ctx_, &p, reinterpret_cast<double*>(ev.rgb.data()), rd.cancel_event), "rc_render");
    }
    if (rd.cancel_event && *rd.cancel_event) return;   // cancelled midway: nothing is written, cpu.rs:55-62
    ev.r = 0; ev.c = 0; ev.width = rd.image->width; ev.height = rd.image->height;   // one message for the whole image
    writer.write(std::move(ev));
}

CudaPreviewRenderer::CudaPreviewRenderer(const RenderConfig& config, const GpuConfig& gpu, const Image& image)
    : CudaRenderer(config, gpu),
      scale_width_(get_highest_divdable(image.width / std::max<size_t>(1, config.num_threads_width), config.scale)),      // cpu_scaled.rs:31-34
      scale_height_(get_highest_divdable(image.height / std::max<size_t>(1, config.num_threads_height), config.scale)) {}

void CudaPreviewRenderer::render(const RenderData& rd, const DataWriter<ImageBufferEvent>& writer) {
    if (rd.cancel_event && *rd.cancel_event) throw TracerError(TracerError::CancelEvent, "Cancel event");
    sync_scene(rd);
    rc_params p = params(rd);
    p.specialize = 0;   // interactive latency: no run-time compilation on the preview path
    ImageBufferEvent ev;
    ev.rgb.resize(rd.image->width * rd.image->height);
    check(rc_render_preview(ctx_, &p, (int32_t)scale_width_, (int32_t)scale_height_, reinterpret_cast<double*>(ev.rgb.data()), rd.cancel_event),
          "rc_render_preview");
    if (rd.cancel_event && *rd.cancel_event) return;
    ev.r = 0; ev.c = 0; ev.width = rd.image->width; ev.height = rd.image->height;
    writer.write(std::move(ev));
}

std::unique_ptr<Renderer> make_renderer(RendererConfig which, const RenderConfig& config, const GpuConfig& gpu, const Image& image) {
    switch (which) {
    case RendererConfig::Cuda: return std::unique_ptr<Renderer>(new CudaRenderer(config, gpu));
    case RendererConfig::CudaPreview: return std::unique_ptr<Renderer>(new CudaPreviewRenderer(config, gpu, image));
    default:
        throw TracerError(TracerError::Configuration, "Config Error (renderer): `Cpu` / `CpuPreview` are the reference's own renderers; "
                                                      "this host only provides `Cuda` and `CudaPreview` (no CPU fallback)");
    }
}

void ScreenBuffer::update(const ImageBufferEvent& ev, CudaRenderer& gpu) {
    // image_buffer.rs:147-153: tone map every colour of the update, store it at (r, c); then the packer of
    // image_action/png.rs:21-31 over the whole screen.  Both run in rc_postprocess.
    std::vector<Color> mapped(ev.rgb.size());
    std::vector<uint8_t> bytes(ev.rgb.size() * 4);
    check(rc_postprocess(gpu.context(), &tone_map_, reinterpret_cast<const double*>(ev.rgb.data()), (int32_t)ev.width, (int32_t)ev.height,
                         bytes.data(), reinterpret_cast<double*>(mapped.data())), "rc_postprocess");
    rgba_.resize(image_.width * image_.height * 4);
    for (size_t row = 0; row < ev.height; ++row) {
        std::copy(mapped.begin() + row * ev.width, mapped.begin() + (row + 1) * ev.width, rgb_.begin() + (ev.r + row) * image_.width + ev.c);
        std::copy(bytes.begin() + 4 * row * ev.width, bytes.begin() + 4 * (row + 1) * ev.width, rgba_.begin() + 4 * ((ev.r + row) * image_.width + ev.c));
    }
}

// =================================================================================================
// SHA-256 (FIPS 180-4) for SavePng's file name
std::string sha256_hex_upper(const uint8_t* data, size_t n) {
    static const uint32_t K[64] = {
        0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
        0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
        0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
        0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
        0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
        0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
    uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    std::vector<uint8_t> msg(data, data + n);
    msg.push_back(0x80);
    while (msg.size() % 64 != 56) msg.push_back(0);
    const uint64_t bits = (uint64_t)n * 8;
    for (int i = 7; i >= 0; --i) msg.push_back((uint8_t)(bits >> (8 * i)));
    auto rotr = [](uint32_t x, int k) { return (x >> k) | (x << (32 - k)); };
    for (size_t off = 0; off < msg.size(); off += 64) {
        uint32_t w[64];
        for (int i = 0; i < 16; ++i) w[i] = ((uint32_t)msg[off + 4 * i] << 24) | ((uint32_t)msg[off + 4 * i + 1] << 16) | ((uint32_t)msg[off + 4 * i + 2] << 8) | msg[off + 4 * i + 3];
        for (int i = 16; i < 64; ++i) {
            const uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3), s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
            w[i] = w[i - 16] + s0 + w[i - 7] + s1;
        }
        uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
        for (int i = 0; i < 64; ++i) {
            const uint32_t S1 = rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25), ch = (e & f) ^ (~e & g), t1 = hh + S1 + ch + K[i] + w[i];
            const uint32_t S0 = rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22), mj = (a & b) ^ (a & c) ^ (b & c), t2 = S0 + mj;
            hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
    }
    char buf[65];
    for (int i = 0; i < 8; ++i) std::snprintf(buf + 8 * i, 9, "%08X", h[i]);
    return std::string(buf, 64);
}

std::string save_png(const std::vector<uint8_t>& rgba, size_t width, size_t height, const std::string& image_output_dir,
                     const std::string& explicit_path) {
    if (rgba.size() != width * height * 4) throw TracerError(TracerError::ImageSave, "Image save error: buffer size does not match the image");
    std::string path = explicit_path;
    if (path.empty()) path = image_output_dir + (image_output_dir.empty() || image_output_dir.back() == '/' ? "" : "/") + sha256_hex_upper(rgba.data(), rgba.size()) + ".png";
    // scanlines with filter type 0
    std::vector<uint8_t> raw;
    raw.reserve((width * 4 + 1) * height);
    for (size_t y = 0; y < height; ++y) {
        raw.push_back(0);
        raw.insert(raw.end(), rgba.begin() + y * width * 4, rgba.begin() + (y + 1) * width * 4);
    }
    uLongf zlen = compressBound((uLong)raw.size());
    std::vector<uint8_t> z(zlen);
    if (compress2(z.data(), &zlen, raw.data(), (uLong)raw.size(), 6) != Z_OK) throw TracerError(TracerError::ImageSave, "Image save error: deflate failed");
    z.resize(zlen);
    std::vector<uint8_t> out = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    auto be32 = [](std::vector<uint8_t>& v, uint32_t x) { for (int i = 3; i >= 0; --i) v.push_back((uint8_t)(x >> (8 * i))); };
    auto chunk = [&](const char type[4], const std::vector<uint8_t>& body) {
        be32(out, (uint32_t)body.size());
        std::vector<uint8_t> tb(type, type + 4);
        tb.insert(tb.end(), body.begin(), body.end());
        out.insert(out.end(), tb.begin(), tb.end());
        be32(out, (uint32_t)crc32(0L, tb.data(), (uInt)tb.size()));
    };
    std::vector<uint8_t> ihdr;
    be32(ihdr, (uint32_t)width); be32(ihdr, (uint32_t)height);
    ihdr.push_back(8); ihdr.push_back(6); ihdr.push_back(0); ihdr.push_back(0); ihdr.push_back(0);   // 8-bit RGBA (ColorType::Rgba8)
    chunk("IHDR", ihdr);
    chunk("IDAT", z);
    chunk("IEND", std::vector<uint8_t>());
    std::ofstream f(path.c_str(), std::ios::binary);
    if (!f) throw TracerError(TracerError::ImageSave, "Image save error: cannot open " + path);
    f.write((const char*)out.data(), (std::streamsize)out.size());
    if (!f) throw TracerError(TracerError::ImageSave, "Image save error: write to " + path + " failed");
    return path;
}

}  // namespace racer
