// rc_spec.cuh — scene-specialised megakernel, compiled at run time with NVRTC.
//
// The precompiled megakernel reads the primitive tables from the constant bank with uniform
// loads and loops whose trip counts it learns at run time.  For a final render of one scene it
// pays to compile the scene INTO the kernel: every rectangle / sphere constant becomes an
// immediate operand, the loops unroll exactly, and material kinds / background / lens that the
// scene does not use disappear from the code.  The source is generated here (a closest-hit
// function with the constants spelled out + a few #defines), compiled for sm_100a against the
// same rt_*.cuh headers the precompiled kernels use (read from csrc/ next to the library), loaded
// with the driver API and cached per scene.  libnvrtc and libcuda are dlopen'ed, so the library
// has no link-time dependency on either; when rc_params.specialize == 1 and anything here fails
// the render call fails loudly (rc_params.specialize == 2 falls back to the precompiled CUDA
// kernel instead).
//
// Beyond immediates, the generator decides things only it can know (DESIGN.md §3.1, v22 - v26): which opposite walls
// are one rectangle test (slab pairs), the origin the kernel traces relative to (RT_SPEC_SHIFT: the most common
// rectangle centre per axis), which literals are handed over as register constants (spec_reg_consts), the layout of
// the staged table's rows for the hit record's plane snap (spec_snap_row), and where packed two-lane arithmetic pays
// (operands already in register pairs).  Each was measured against the form it replaced (DESIGN.md §3.1).  Slab pairs
// alone keep a switch that turns them off (RC_SPEC_NO_SLAB), because the tests trace the kernel without them as the
// reference the slab pairs must match.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "rt_kernels.cuh"

struct SpecKernel {
    void* module = nullptr;     // CUmodule
    void* function = nullptr;   // CUfunction
    std::string source;
    std::string error;          // non-empty: this source failed to compile / load (remembered, not retried per render)
    uint64_t last_use = 0;      // LRU stamp
};

// A scene edit or a camera move into / out of a wall pair's slab is a new source text, hence a new module: the cache
// keeps the most recently used few and unloads the rest (an interactive host re-uploads on every edit).
#define RC_SPEC_CACHE_MAX 8

struct SpecApi {
    bool tried = false, ok = false;
    std::string err;
    void* nvrtc = nullptr;
    void* cuda = nullptr;
    int (*CreateProgram)(void**, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*CompileProgram)(void*, int, const char* const*) = nullptr;
    int (*GetCUBINSize)(void*, size_t*) = nullptr;
    int (*GetCUBIN)(void*, char*) = nullptr;
    int (*GetProgramLogSize)(void*, size_t*) = nullptr;
    int (*GetProgramLog)(void*, char*) = nullptr;
    int (*DestroyProgram)(void**) = nullptr;
    int (*cuModuleLoadData)(void**, const void*) = nullptr;
    int (*cuModuleGetFunction)(void**, void*, const char*) = nullptr;
    int (*cuModuleUnload)(void*) = nullptr;
    int (*cuLaunchKernel)(void*, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void*, void**, void**) = nullptr;
    std::string header_dir;
};

inline SpecApi& spec_api() {
    static SpecApi api;
    return api;
}

inline bool spec_load_api(const void* anchor_symbol) {
    SpecApi& a = spec_api();
    if (a.tried) return a.ok;
    a.tried = true;
    const char* nvrtc_names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"};
    for (const char* n : nvrtc_names) { a.nvrtc = dlopen(n, RTLD_NOW); if (a.nvrtc) break; }
    if (!a.nvrtc) { a.err = "libnvrtc.so.12 not found"; return false; }
    a.cuda = dlopen("libcuda.so.1", RTLD_NOW);
    if (!a.cuda) { a.err = "libcuda.so.1 not found"; return false; }
#define RC_SYM(lib, field, name)                                                        \
    *(void**)(&a.field) = dlsym(a.lib, name);                                           \
    if (!a.field) { a.err = std::string("missing symbol ") + name; return false; }
    RC_SYM(nvrtc, CreateProgram, "nvrtcCreateProgram");
    RC_SYM(nvrtc, CompileProgram, "nvrtcCompileProgram");
    RC_SYM(nvrtc, GetCUBINSize, "nvrtcGetCUBINSize");
    RC_SYM(nvrtc, GetCUBIN, "nvrtcGetCUBIN");
    RC_SYM(nvrtc, GetProgramLogSize, "nvrtcGetProgramLogSize");
    RC_SYM(nvrtc, GetProgramLog, "nvrtcGetProgramLog");
    RC_SYM(nvrtc, DestroyProgram, "nvrtcDestroyProgram");
    RC_SYM(cuda, cuModuleLoadData, "cuModuleLoadData");
    RC_SYM(cuda, cuModuleGetFunction, "cuModuleGetFunction");
    RC_SYM(cuda, cuModuleUnload, "cuModuleUnload");
    RC_SYM(cuda, cuLaunchKernel, "cuLaunchKernel");
#undef RC_SYM
    Dl_info info;
    if (!dladdr(anchor_symbol, &info) || !info.dli_fname) { a.err = "cannot locate the library on disk"; return false; }
    std::string path(info.dli_fname);
    size_t slash = path.find_last_of('/');
    a.header_dir = (slash == std::string::npos ? std::string(".") : path.substr(0, slash)) + "/csrc/";
    a.ok = true;
    return true;
}

inline int __float_as_int_host(float f) { int i; std::memcpy(&i, &f, sizeof(i)); return i; }

inline std::string spec_float(float v) {
    char buf[64];
    std::snprintf(buf, sizeof(buf), "%.9g", (double)v);
    std::string s(buf);
    if (s.find_first_of(".eEn") == std::string::npos) s += ".0";
    return s + "f";
}

// Entry point of a specialised translation unit: the plain megakernel, or (moments) the one of the adaptive rounds.
// The two are separate sources, hence separate modules in the cache; the plain text is what it always was.
inline std::string spec_entry(const char* mode, int rounds, bool tex, bool moments) {
    std::ostringstream o;
    o << "extern \"C\" __global__ void __launch_bounds__(RT_BLOCK, RT_MIN_BLOCKS)\n"
         "spec_megakernel(const __grid_constant__ KParams P, float* __restrict__ accum"
      << (moments ? ", const uint8_t* __restrict__ active, float* __restrict__ round_m2" : "") << ") {\n"
         "    extern __shared__ __align__(16) unsigned char smem[];\n"
         "    megakernel_body<" << mode << ", 0, " << rounds << ", " << (tex ? "true" : "false") << (moments ? ", true" : "")
      << ">(P, accum, smem" << (moments ? ", active, round_m2" : "") << ");\n}\n";
    return o.str();
}

// Source of the specialised translation unit for a scene already laid out in KParams
// (type-sorted constant-bank table).
inline std::string spec_generate(const KParams& kp, bool tex, int mats_mask, int mode = RT_MODE_CONST_LINEAR, int prims_mask_all = 0xF,
                                 bool instanced = false, int rounds = 10, bool moments = false) {
    std::ostringstream o;
    if (mode != RT_MODE_CONST_LINEAR) {
        // BVH paths: the tables stay in memory; what is compiled in is which kinds of primitive, material, wrapper,
        // lens and motion the scene has — the leaf test and the shading lose the branches of everything absent.
        const bool black = __float_as_int_host(kp.bg_a.w) != 0 && kp.bg_a.x == 0.f && kp.bg_a.y == 0.f && kp.bg_a.z == 0.f;
        o << "#define RT_SPEC_PRIMS " << prims_mask_all << "\n";
        o << "#define RT_SPEC_BG_BLACK " << (black ? 1 : 0) << "\n";
        o << "#define RT_HAS_INSTANCES " << (instanced ? 1 : 0) << "\n";
        o << "#define RT_HAS_LENS " << (kp.lens_enabled ? 1 : 0) << "\n";
        o << "#define RT_HAS_MOTION " << (kp.has_motion ? 1 : 0) << "\n";
        if (mode == RT_MODE_GLOBAL_BVH) o << "#define RT_MIN_BLOCKS RT_MIN_BLOCKS_GLOBAL_BVH\n";   // see rt_kernels.cuh
        o << "#include \"rt_scene.cuh\"\n";
        o << "RT_D int spec_closest_hit(const RayT<float>&, int, float&, const TexCtx&) { return -1; }   // constant-table scenes only\n";
        o << "#define RT_SPEC_REG_CONSTS 0\nRT_D void spec_reg_consts(float*) {}\n";
        o << "#define RT_SPECIALIZED 1\n";
        o << "#define RT_SPEC_MATS " << mats_mask << "\n";
        o << "#define RT_FIXED_JITTER(P) 0\n";
        o << "#include \"rt_kernels.cuh\"\n";
        o << spec_entry(mode == RT_MODE_SMEM_BVH ? "RT_MODE_SMEM_BVH" : "RT_MODE_GLOBAL_BVH", rounds, tex, moments);
        return o.str();
    }
    // primitive kinds present, background: known before the headers are read
    int prims_mask = 0;   // bit RT_PRIM_* (moving spheres count as spheres), instanced primitives included
    for (int i = 0; i < kp.n_prims && i < RT_MAX_CONST_PRIMS; ++i) {
        const int type = __float_as_int_host(kp.cprims[i].b.z) & 15;
        prims_mask |= 1 << (type == RT_PRIM_MOVING ? RT_PRIM_SPHERE : type);
    }
    o << "#define RT_SPEC_PRIMS " << prims_mask << "\n";
    const bool black = __float_as_int_host(kp.bg_a.w) != 0 && kp.bg_a.x == 0.f && kp.bg_a.y == 0.f && kp.bg_a.z == 0.f;
    o << "#define RT_SPEC_BG_BLACK " << (black ? 1 : 0) << "\n";
    o << "#define RT_HAS_INSTANCES " << (kp.n_cobj > 0 ? 1 : 0) << "\n";
    o << "#define RT_HAS_LENS " << (kp.lens_enabled ? 1 : 0) << "\n";   // part of the source, hence of the cache key
    // Scene origin of the kernel.  In a rectangle-only scene without textures nothing but the closest hit and the
    // hit record ever looks at a POSITION, and both only at differences to rectangle centres and planes.  The kernel
    // therefore traces in coordinates relative to the most common rectangle centre of each axis (Cornell: the centre
    // of the box): for every rectangle centred there `origin - centre` is the origin itself — one FADD less per axis
    // and ray.  Camera origin, plane constants (tests and the staged table's, from the same literal) and centres are
    // shifted; directions, distances and colours are what they were up to fp32 rounding.
    double shift[3] = {0.0, 0.0, 0.0};
    const bool shift_ok = (prims_mask & 1) == 0 && kp.n_cobj == 0 && !tex;
    if (shift_ok) o << "#define RT_SPEC_SNAP_TABLE 1\n";    // (see spec_snap_row below)
    if (shift_ok) {
        std::map<float, int> votes[3];
        for (int g = 0; g < 3; ++g)
            for (int i = kp.lin_end[g]; i < kp.lin_end[g + 1]; ++i) {
                const float4 c = kp.crect_bounds[g][i - kp.lin_end[g]];
                ++votes[g == 2 ? 1 : 0][c.x];    // in-plane axis a: x for the xy and xz groups, y for the yz group
                ++votes[g == 0 ? 1 : 2][c.z];    // in-plane axis b: y for the xy group, z for the others
            }
        for (int ax = 0; ax < 3; ++ax) {
            int best = 0;
            for (auto& kv : votes[ax])
                if (kv.second > best) { best = kv.second; shift[ax] = (double)kv.first; }
        }
        if (shift[0] != 0.0 || shift[1] != 0.0 || shift[2] != 0.0)
            o << "#define RT_SPEC_SHIFT mk3(" << spec_float((float)shift[0]) << ", " << spec_float((float)shift[1]) << ", " << spec_float((float)shift[2]) << ")\n";
    }
    // plane constant / centre of a rectangle in the kernel's coordinates (same literal wherever it is used)
    auto plane = [&](int i, int g) { return (float)((double)kp.cprims[i].b.x - shift[2 - g]); };
    auto centre_a = [&](float c, int g) { return (float)((double)c - shift[g == 2 ? 1 : 0]); };
    auto centre_b = [&](float c, int g) { return (float)((double)c - shift[g == 0 ? 1 : 2]); };
    if (const char* e = std::getenv("RC_STEAL")) o << "#define RT_STEAL " << std::atoi(e) << "\n";
    o << "#include \"rt_scene.cuh\"\n";
    // rectangle-only scenes keep the index of the best hit as a FLOAT, so that both conditional moves of the
    // closest-hit update are predicated FFMAs on the FMA pipe (rect_closest_fma); with spheres around, the
    // index stays an integer (rect_closest)
    const bool fidx = (prims_mask & 1) == 0;
    o << "RT_D int spec_closest_hit(const RayT<float>& r, int last_prim, float& best_t, const TexCtx& X) {\n";
    o << "    (void)X;\n";
    // literals handed to the kernel as register constants (TexCtx::k_spec): the plane pairs of slab pairs
    std::vector<float> reg_consts;
    auto reg_pair = [&](float k1, float k2) {   // -> the two operand expressions
        for (size_t j = 0; j + 1 < reg_consts.size(); j += 2)
            if (reg_consts[j] == k1 && reg_consts[j + 1] == k2) return std::make_pair("X.k_spec[" + std::to_string(j) + "]", "X.k_spec[" + std::to_string(j + 1) + "]");
        if (reg_consts.size() + 2 > 4) return std::make_pair(spec_float(k1), spec_float(k2));
        reg_consts.push_back(k1); reg_consts.push_back(k2);
        const size_t j = reg_consts.size() - 2;
        return std::make_pair("X.k_spec[" + std::to_string(j) + "]", "X.k_spec[" + std::to_string(j + 1) + "]");
    };
    o << "    int best = -1;\n    best_t = RT_NO_HIT;\n    (void)last_prim;\n";
    if (fidx) o << "    float bestf = -1.0f;\n";
    const int n_sph = kp.lin_end[0];
    bool any_motion = false;
    if (n_sph > 0) {
        o << "    {\n        const float a = dot(r.d, r.d), inv_a = fast_rcp(a);\n        float t;\n";
        for (int i = 0; i < n_sph; ++i) {
            const DevPrim& p = kp.cprims[i];
            const bool moving = (__float_as_int_host(p.b.z) & 15) == RT_PRIM_MOVING;
            if (moving) {
                any_motion = true;
                o << "        t = sphere_hit<float>(r.o, r.d, a, inv_a, mk3(fmaf(r.time, " << spec_float(p.n.x) << ", " << spec_float(p.a.x)
                  << "), fmaf(r.time, " << spec_float(p.n.y) << ", " << spec_float(p.a.y) << "), fmaf(r.time, " << spec_float(p.n.z) << ", "
                  << spec_float(p.a.z) << ")), " << spec_float(p.a.w) << ", 0.0f, last_prim == " << i << ", (float)RT_T_MIN, best_t, false);\n";
            } else
            o << "        t = sphere_hit<float>(r.o, r.d, a, inv_a, mk3(" << spec_float(p.a.x) << ", " << spec_float(p.a.y) << ", "
              << spec_float(p.a.z) << "), " << spec_float(p.a.w) << ", " << spec_float(p.b.x) << ", last_prim == " << i
              << ", (float)RT_T_MIN, best_t);\n";
            o << "        if (t >= 0.0f) { best_t = t; best = " << i << "; }\n";
        }
        o << "    }\n";
    }
    // rectangles: per axis group, all candidates first (independent), then the ordered min-reduction.
    // Origins relative to each distinct rectangle centre are formed once per ray and shared.
    const char* on[3] = {"r.o.z", "r.o.y", "r.o.x"};
    const char* in[3] = {"r.inv_d.z", "r.inv_d.y", "r.inv_d.x"};
    const char* oa[3] = {"r.o.x", "r.o.x", "r.o.y"};
    const char* da[3] = {"r.d.x", "r.d.x", "r.d.y"};
    const char* ob[3] = {"r.o.y", "r.o.z", "r.o.z"};
    const char* db[3] = {"r.d.y", "r.d.z", "r.d.z"};
    std::map<std::string, std::string> rel;   // "r.o.x - 277.5f" -> variable name
    auto rel_origin = [&](const char* axis, float centre) {
        if (centre == 0.0f) return std::string(axis);    // (the kernel's origin is this rectangle's centre on that axis)
        std::string key = std::string(axis) + " - " + spec_float(centre);
        auto it = rel.find(key);
        if (it != rel.end()) return it->second;
        std::string name = "oc" + std::to_string(rel.size());
        o << "    const float " << name << " = " << key << ";\n";
        rel[key] = name;
        return name;
    };
    // The two in-plane coordinates of ONE rectangle, t * (d_a, d_b) + (oc_a, oc_b): one packed multiply-add when the
    // operands already sit in register pairs — the ray direction is held as (x, y), z, so that is the xy group —
    // and two scalar ones otherwise: building a pair costs a MOV per operand on the ALU pipe, which made the packed
    // form of the xz / yz groups 2.5 - 3 instructions against 2.
    auto coords = [&](const std::string& t, int g, const std::string& oca, const std::string& ocb, const std::string& xa, const std::string& xb) {
        if (g == 0)
            o << "        fma2_bcast(" << t << ", " << da[g] << ", " << db[g] << ", " << oca << ", " << ocb << ", " << xa << ", " << xb << ");\n";
        else
            o << "        " << xa << " = fmaf(" << t << ", " << da[g] << ", " << oca << "); " << xb << " = fmaf(" << t << ", " << db[g] << ", " << ocb << ");\n";
    };
    // slab pairs (below) need every ray origin inside the slab: rectangles only, nothing instanced, a pinhole
    bool nothing_yet = n_sph == 0;   // no test emitted so far: best_t / bestf still hold their start values
    const bool slab_scene_ok = kp.n_cobj == 0 && !kp.lens_enabled && std::getenv("RC_SPEC_NO_SLAB") == nullptr;
    for (int g = 0; g < 3; ++g) {
        const int begin = kp.lin_end[g], end = kp.lin_end[g + 1];
        if (end <= begin) continue;
        std::vector<std::string> va(end - begin), vb(end - begin);
        for (int i = begin; i < end; ++i) {
            const float4 c = kp.crect_bounds[g][i - begin];
            va[i - begin] = rel_origin(oa[g], centre_a(c.x, g));
            vb[i - begin] = rel_origin(ob[g], centre_b(c.z, g));
        }
        o << "    {\n";
        // Slab pair: two rectangles of this group with the same bounds (opposite walls) between which every ray of
        // the scene starts — all geometry and the pinhole lie inside the slab.  Exactly one of the two planes is
        // then in front of a ray, max(t_i, t_j), and ONE rectangle test serves both walls.
        int s0 = -1, s1 = -1;
        if (fidx && slab_scene_ok) {
            const int n_axis = 2 - g;   // plane axis of the group: xy -> z, xz -> y, yz -> x
            for (int i = begin; i < end && s0 < 0; ++i)
                for (int j = i + 1; j < end && s0 < 0; ++j) {
                    const float4 c = kp.crect_bounds[g][i - begin], c2 = kp.crect_bounds[g][j - begin];
                    if (c.x != c2.x || c.y != c2.y || c.z != c2.z || c.w != c2.w) continue;
                    const float k_lo = std::fmin(kp.cprims[i].b.x, kp.cprims[j].b.x), k_hi = std::fmax(kp.cprims[i].b.x, kp.cprims[j].b.x);
                    if (!(k_lo < k_hi)) continue;
                    const float cam_n = n_axis == 0 ? kp.cam.origin.x : (n_axis == 1 ? kp.cam.origin.y : kp.cam.origin.z);
                    bool inside = cam_n > k_lo && cam_n < k_hi;
                    for (int gg = 0; gg < 3 && inside; ++gg)
                        for (int r = kp.lin_end[gg]; r < kp.lin_end[gg + 1] && inside; ++r) {
                            const float4 b = kp.crect_bounds[gg][r - kp.lin_end[gg]];
                            const int rn = 2 - gg, ra = gg == 2 ? 1 : 0, rb = gg == 0 ? 1 : 2;   // plane axis, in-plane axes
                            float lo, hi;
                            if (n_axis == rn) lo = hi = kp.cprims[r].b.x;
                            else if (n_axis == ra) { lo = b.x - b.y; hi = b.x + b.y; }
                            else { (void)rb; lo = b.z - b.w; hi = b.z + b.w; }
                            inside = lo >= k_lo && hi <= k_hi;
                        }
                    if (inside) { s0 = kp.cprims[i].b.x < kp.cprims[j].b.x ? i : j; s1 = s0 == i ? j : i; }
                }
        }
        std::vector<int> rest;
        for (int i = begin; i < end; ++i)
            if (i != s0 && i != s1) rest.push_back(i);
        if (s0 >= 0) {
            o << "        float t" << s0 << ", t" << s1 << ", xa" << s0 << ", xb" << s0 << ";\n";
            const auto kk = reg_pair(plane(s0, g), plane(s1, g));
            o << "        pair_t(" << kk.first << ", " << kk.second << ", " << on[g] << ", " << in[g] << ", t" << s0 << ", t" << s1 << ");   // planes "
              << spec_float(plane(s0, g)) << ", " << spec_float(plane(s1, g)) << "\n";
            o << "        const float ts" << s0 << " = fmaxf(t" << s0 << ", t" << s1 << ");   // slab pair " << s0 << " / " << s1 << "\n";
            coords("ts" + std::to_string(s0), g, va[s0 - begin], vb[s0 - begin], "xa" + std::to_string(s0), "xb" + std::to_string(s0));
        }
        for (size_t u = 0; u < rest.size(); ++u) {
            const int i = rest[u];
            if (u + 1 < rest.size()) {   // two rectangles of this axis group per packed instruction
                const int j = rest[u + 1];
                const float4 c = kp.crect_bounds[g][i - begin], c2 = kp.crect_bounds[g][j - begin];
                o << "        float t" << i << ", t" << j << ", xa" << i << ", xa" << j << ", xb" << i << ", xb" << j << ";\n";
                o << "        pair_t(" << spec_float(plane(i, g)) << ", " << spec_float(plane(j, g)) << ", " << on[g] << ", " << in[g] << ", t" << i << ", t" << j << ");\n";
                auto centres = [&](const char* axis, float ca1, float ca2, const std::string& v1, const std::string& v2, const char* tag) {
                    if (ca1 == ca2) return std::make_pair(v1, v2);      // one shared scalar, broadcast
                    const std::string n1 = std::string(tag) + std::to_string(i), n2 = std::string(tag) + std::to_string(j);
                    o << "        float " << n1 << ", " << n2 << ";\n";
                    o << "        pair_oc(" << axis << ", " << spec_float(ca1) << ", " << spec_float(ca2) << ", " << n1 << ", " << n2 << ");\n";
                    return std::make_pair(n1, n2);
                };
                const auto pa = centres(oa[g], centre_a(c.x, g), centre_a(c2.x, g), va[i - begin], va[j - begin], "pa");
                const auto pb = centres(ob[g], centre_b(c.z, g), centre_b(c2.z, g), vb[i - begin], vb[j - begin], "pb");
                o << "        pair_x(t" << i << ", t" << j << ", " << da[g] << ", " << pa.first << ", " << pa.second << ", xa" << i << ", xa" << j << ");\n";
                o << "        pair_x(t" << i << ", t" << j << ", " << db[g] << ", " << pb.first << ", " << pb.second << ", xb" << i << ", xb" << j << ");\n";
                ++u;
                continue;
            }
            // one rectangle: its two in-plane coordinates are the two lanes
            o << "        const float t" << i << " = (" << spec_float(plane(i, g)) << " - " << on[g] << ") * " << in[g] << ";\n";
            o << "        float xa" << i << ", xb" << i << ";\n";
            coords("t" + std::to_string(i), g, va[i - begin], vb[i - begin], "xa" + std::to_string(i), "xb" + std::to_string(i));
        }
        if (s0 >= 0) {
            const float4 c = kp.crect_bounds[g][s0 - begin];
            o << "        rect_closest_fma_pair(ts" << s0 << ", xa" << s0 << ", xb" << s0 << ", " << spec_float(c.y) << ", " << spec_float(c.w) << ", t" << s0
              << ", t" << s1 << ", " << spec_float((float)s0) << ", " << spec_float((float)(s1 - s0)) << ", best_t, bestf);\n";
        }
        if (s0 >= 0) nothing_yet = false;
        for (int i : rest) {
            const float4 c = kp.crect_bounds[g][i - begin];
            if (fidx && nothing_yet) {   // the first test of the function: selects between literals
                o << "        rect_closest_first(t" << i << ", xa" << i << ", xb" << i << ", " << spec_float(c.y) << ", " << spec_float(c.w) << ", "
                  << spec_float((float)i) << ", best_t, bestf);\n";
                nothing_yet = false;
                continue;
            }
            nothing_yet = false;
            if (fidx)
                o << "        rect_closest_fma(t" << i << ", xa" << i << ", xb" << i << ", " << spec_float(c.y) << ", " << spec_float(c.w) << ", "
                  << spec_float((float)i) << ", best_t, bestf);\n";
            else
                o << "        rect_closest(t" << i << ", xa" << i << ", xb" << i << ", " << spec_float(c.y) << ", " << spec_float(c.w) << ", " << i
                  << ", best_t, best);\n";
        }
        o << "    }\n";
    }
    // instanced objects: cull volume, ray into the object's space (constants spelled out), then its rectangles
    for (int k = 0; k < kp.n_cobj; ++k) {
        const float4 lo = kp.cobj_lo[k], hi = kp.cobj_hi[k];
        const int first = __float_as_int_host(lo.w), meta = __float_as_int_host(hi.w), count = meta & 255;
        const DevInstance& in = kp.cinst[meta >> 8];
        o << "    if (aabb_hit_reference(make_float4(" << spec_float(lo.x) << ", " << spec_float(lo.y) << ", " << spec_float(lo.z)
          << ", 0.0f), make_float4(" << spec_float(hi.x) << ", " << spec_float(hi.y) << ", " << spec_float(hi.z) << ", 0.0f), r, best_t)) {\n";
        o << "        vec3f lo_ = r.o, ld_ = r.d;\n";
        if (in.flags & 2) o << "        lo_ = mk3(lo_.x - " << spec_float(in.ox) << ", lo_.y - " << spec_float(in.oy) << ", lo_.z - " << spec_float(in.oz) << ");\n";
        if (in.flags & 1) {
            const std::string c = spec_float(in.cos_theta), sn = spec_float(in.sin_theta);
            o << "        lo_ = mk3(" << c << " * lo_.x - " << sn << " * lo_.z, lo_.y, " << sn << " * lo_.x + " << c << " * lo_.z);\n";
            o << "        ld_ = mk3(" << c << " * ld_.x - " << sn << " * ld_.z, ld_.y, " << sn << " * ld_.x + " << c << " * ld_.z);\n";
        }
        o << "        const RayT<float> lr = make_ray(lo_, ld_, r.time);\n";
        // the object's primitives in order (Boxx::obj_hit, box.rs:82-101): rectangle candidates first
        // (independent), spheres solved in place, then the ordered reduction.  The rectangle the ray leaves is
        // skipped (its hit point went through a rotation and is not exactly on the plane any more).
        const char* ln[3] = {"lr.o.z", "lr.o.y", "lr.o.x"};
        const char* li[3] = {"lr.inv_d.z", "lr.inv_d.y", "lr.inv_d.x"};
        const char* la[3] = {"lr.o.x", "lr.o.x", "lr.o.y"};
        const char* lda[3] = {"lr.d.x", "lr.d.x", "lr.d.y"};
        const char* lb[3] = {"lr.o.y", "lr.o.z", "lr.o.z"};
        const char* ldb[3] = {"lr.d.y", "lr.d.z", "lr.d.z"};
        for (int i = first; i < first + count; ++i) {
            const DevPrim& p = kp.cprims[i];
            const int type = __float_as_int_host(p.b.z) & 15;
            if (type == RT_PRIM_SPHERE || type == RT_PRIM_MOVING) continue;
            const int g = type - 1;
            const double ca = 0.5 * ((double)p.a.x + p.a.y), ha = 0.5 * ((double)p.a.y - p.a.x);
            const double cb = 0.5 * ((double)p.a.z + p.a.w), hb = 0.5 * ((double)p.a.w - p.a.z);
            // two consecutive sides on the same axis (a Box's opposite faces): packed arithmetic, as for the plain groups
            if (i + 1 < first + count && (__float_as_int_host(kp.cprims[i + 1].b.z) & 15) == type) {
                const DevPrim& q = kp.cprims[i + 1];
                const int j = i + 1;
                const double ca2 = 0.5 * ((double)q.a.x + q.a.y), cb2 = 0.5 * ((double)q.a.z + q.a.w);
                o << "        float u" << i << ", u" << j << ", ea" << i << ", ea" << j << ", eb" << i << ", eb" << j << ", ca" << i << ", ca" << j
                  << ", cb" << i << ", cb" << j << ";\n";
                o << "        pair_t(" << spec_float(p.b.x) << ", " << spec_float(q.b.x) << ", " << ln[g] << ", " << li[g] << ", u" << i << ", u" << j << ");\n";
                if ((float)ca == (float)ca2) o << "        ca" << i << " = ca" << j << " = " << la[g] << " - " << spec_float((float)ca) << ";\n";
                else o << "        pair_oc(" << la[g] << ", " << spec_float((float)ca) << ", " << spec_float((float)ca2) << ", ca" << i << ", ca" << j << ");\n";
                if ((float)cb == (float)cb2) o << "        cb" << i << " = cb" << j << " = " << lb[g] << " - " << spec_float((float)cb) << ";\n";
                else o << "        pair_oc(" << lb[g] << ", " << spec_float((float)cb) << ", " << spec_float((float)cb2) << ", cb" << i << ", cb" << j << ");\n";
                o << "        pair_x(u" << i << ", u" << j << ", " << lda[g] << ", ca" << i << ", ca" << j << ", ea" << i << ", ea" << j << ");\n";
                o << "        pair_x(u" << i << ", u" << j << ", " << ldb[g] << ", cb" << i << ", cb" << j << ", eb" << i << ", eb" << j << ");\n";
                // the rectangle the ray leaves gets t = -1, which fails t >= t_min
                o << "        u" << i << " = last_prim == " << i << " ? -1.0f : u" << i << "; u" << j << " = last_prim == " << j << " ? -1.0f : u" << j << ";\n";
                ++i;
                continue;
            }
            // the rectangle the ray leaves gets t = -1, which fails t >= t_min
            o << "        const float u" << i << " = last_prim == " << i << " ? -1.0f : (" << spec_float(p.b.x) << " - " << ln[g] << ") * " << li[g] << ";\n";
            o << "        const float ea" << i << " = fmaf(u" << i << ", " << lda[g] << ", " << la[g] << " - " << spec_float((float)ca) << "), eb" << i
              << " = fmaf(u" << i << ", " << ldb[g] << ", " << lb[g] << " - " << spec_float((float)cb) << ");\n";
        }
        for (int i = first; i < first + count; ++i) {
            const DevPrim& p = kp.cprims[i];
            const int type = __float_as_int_host(p.b.z) & 15;
            if (type == RT_PRIM_SPHERE) {
                o << "        { const float a_ = dot(lr.d, lr.d); const float t_ = sphere_hit<float>(lr.o, lr.d, a_, fast_rcp(a_), mk3(" << spec_float(p.a.x)
                  << ", " << spec_float(p.a.y) << ", " << spec_float(p.a.z) << "), " << spec_float(p.a.w) << ", " << spec_float(p.b.x) << ", last_prim == " << i
                  << ", (float)RT_T_MIN, best_t); if (t_ >= 0.0f) { best_t = t_; best = " << i << "; } }\n";
            } else if (type == RT_PRIM_MOVING) {
                o << "#error \"instanced moving spheres are rejected at upload\"\n";
            } else {
                const double ha = 0.5 * ((double)p.a.y - p.a.x), hb = 0.5 * ((double)p.a.w - p.a.z);
                if (fidx)
                    o << "        rect_closest_fma(u" << i << ", ea" << i << ", eb" << i << ", " << spec_float((float)ha) << ", " << spec_float((float)hb) << ", "
                      << spec_float((float)i) << ", best_t, bestf);\n";
                else
                o << "        rect_closest(u" << i << ", ea" << i << ", eb" << i << ", " << spec_float((float)ha) << ", " << spec_float((float)hb) << ", " << i
                  << ", best_t, best);\n";
            }
        }
        o << "    }\n";
    }
    if (fidx) o << "    best = __float2int_rn(bestf);\n";
    o << "    return best;\n}\n";
    o << "#define RT_SPEC_REG_CONSTS " << reg_consts.size() << "\n";
    o << "RT_D void spec_reg_consts(float* out) {\n    (void)out;\n";
    for (size_t j = 0; j < reg_consts.size(); ++j) o << "    out[" << j << "] = " << spec_float(reg_consts[j]) << ";\n";
    o << "}\n";
    if (shift_ok) {
        // Rectangle-only scenes: the hit record puts the hit point back onto the plane the TEST used (rt_scene.cuh
        // make_hit_local) as p * M + K with M = 1 - N (0 on the plane's axis, 1 on the others) and K = k N, k the
        // plane constant in the kernel's coordinates from the same literal as the test's: a packed and a scalar
        // multiply-add instead of a dot product, a subtraction and three multiply-adds, same bits (p_axis * 0 + k = k,
        // p * 1 + 0 = p).  The CTA patches its staged table once: row a = (M.x, M.y, K.x, K.y), b.x = K.z, c.w = M.z
        // (bounds, plane constant and object id, which a rectangle's hit record and shading do not read).
        o << "RT_D void spec_snap_row(int i, float4& a, float& bx, float& cw) {\n    switch (i) {\n";
        for (int g = 0; g < 3; ++g)
            for (int i = kp.lin_end[g]; i < kp.lin_end[g + 1]; ++i) {
                const int ax = 2 - g;   // plane axis
                const std::string k = spec_float(plane(i, g));
                o << "        case " << i << ": a = make_float4(" << (ax == 0 ? "0.0f" : "1.0f") << ", " << (ax == 1 ? "0.0f" : "1.0f") << ", "
                  << (ax == 0 ? k : std::string("0.0f")) << ", " << (ax == 1 ? k : std::string("0.0f")) << "); bx = " << (ax == 2 ? k : std::string("0.0f"))
                  << "; cw = " << (ax == 2 ? "0.0f" : "1.0f") << "; break;\n";
            }
        o << "    }\n}\n";
    }
    o << "#define RT_SPECIALIZED 1\n";
    o << "#define RT_SPEC_MATS " << mats_mask << "\n";
    o << "#define RT_HAS_MOTION " << (any_motion ? 1 : 0) << "\n";
    o << "#define RT_FIXED_JITTER(P) 0\n";   // renders with fixed jitter (parity checks) use the precompiled kernels
    o << "#include \"rt_kernels.cuh\"\n";
    o << spec_entry("RT_MODE_CONST_LINEAR", rounds, tex, moments);
    return o.str();
}

inline bool spec_read(const std::string& path, std::string& out) {
    std::ifstream f(path.c_str());
    if (!f) return false;
    std::stringstream ss;
    ss << f.rdbuf();
    out = ss.str();
    return true;
}

// Compile + load; returns nullptr and sets err on failure.
inline SpecKernel* spec_build(std::map<std::string, SpecKernel>& cache, const std::string& source, std::string& err, uint64_t now = 0) {
    auto it = cache.find(source);
    if (it != cache.end()) {
        it->second.last_use = now;
        if (!it->second.error.empty()) { err = it->second.error; return nullptr; }
        return &it->second;
    }
    while (cache.size() >= RC_SPEC_CACHE_MAX) {   // evict the least recently used entry
        auto victim = cache.begin();
        for (auto j = cache.begin(); j != cache.end(); ++j)
            if (j->second.last_use < victim->second.last_use) victim = j;
        if (victim->second.module && spec_api().cuModuleUnload) spec_api().cuModuleUnload(victim->second.module);
        cache.erase(victim);
    }
    auto remember_failure = [&]() {
        SpecKernel bad;
        bad.error = err;
        bad.last_use = now;
        cache.emplace(source, bad);
        return (SpecKernel*)nullptr;
    };
    SpecApi& a = spec_api();
    std::string h_math, h_scene, h_kernels;
    if (!spec_read(a.header_dir + "rt_math.cuh", h_math) || !spec_read(a.header_dir + "rt_scene.cuh", h_scene) ||
        !spec_read(a.header_dir + "rt_kernels.cuh", h_kernels)) {
        err = "kernel headers not found in " + a.header_dir;
        return nullptr;
    }
    const char* headers[3] = {h_math.c_str(), h_scene.c_str(), h_kernels.c_str()};
    const char* names[3] = {"rt_math.cuh", "rt_scene.cuh", "rt_kernels.cuh"};
    void* prog = nullptr;
    if (a.CreateProgram(&prog, source.c_str(), "spec_scene.cu", 3, headers, names) != 0) { err = "nvrtcCreateProgram failed"; return nullptr; }
    const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-default-device"};
    int rc = a.CompileProgram(prog, 4, opts);
    if (rc != 0) {
        size_t n = 0;
        a.GetProgramLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) a.GetProgramLog(prog, &log[0]);
        err = "nvrtc compile failed: " + log.substr(0, 1500);
        a.DestroyProgram(&prog);
        return remember_failure();
    }
    size_t n = 0;
    a.GetCUBINSize(prog, &n);
    std::vector<char> cubin(n);
    a.GetCUBIN(prog, cubin.data());
    a.DestroyProgram(&prog);
    SpecKernel k;
    k.source = source;
    k.last_use = now;
    if (a.cuModuleLoadData(&k.module, cubin.data()) != 0) { err = "cuModuleLoadData failed"; return remember_failure(); }
    if (a.cuModuleGetFunction(&k.function, k.module, "spec_megakernel") != 0) { err = "spec_megakernel not found in module"; return remember_failure(); }
    auto res = cache.emplace(source, k);
    return &res.first->second;
}

inline void spec_release(std::map<std::string, SpecKernel>& cache) {
    SpecApi& a = spec_api();
    for (auto& kv : cache)
        if (kv.second.module && a.cuModuleUnload) a.cuModuleUnload(kv.second.module);
    cache.clear();
}

// `active` / `round_m2`: the two extra arguments of a moments entry point (spec_entry), NULL for the plain one
inline int spec_launch(SpecKernel* k, const KParams& kp, float* accum, int blocks, size_t smem, cudaStream_t st,
                       const uint8_t* active = nullptr, float* round_m2 = nullptr) {
    SpecApi& a = spec_api();
    KParams p = kp;
    void* args[4] = {&p, &accum, &active, &round_m2};
    return a.cuLaunchKernel(k->function, (unsigned)blocks, 1, 1, RT_BLOCK, 1, 1, (unsigned)smem, (void*)st, args, nullptr);
}
