// rc_api.cu — implementation of the C ABI declared in include/racer_cuda.h.
// Host-side orchestration only: table conversion (f64 -> fp32), uploads,
// kernel launches, multi-device partitioning.  No CPU rendering path exists.
#include "../../include/racer_cuda.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "rt_kernels.cuh"
#include "rt_wavefront.cuh"
#include <algorithm>

#include "rc_multi.cuh"
#include "rc_lbvh.cuh"
#include "rc_spec.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int status, const std::string& msg) {
    g_last_error = msg;
    return status;
}

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(RC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));     \
    } while (0)

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    size_t cap = 0;   // elements allocated (>= n): a re-upload of a scene of the same or a smaller size allocates nothing
    // host -> device on `st` (asynchronous with respect to the host only for pinned memory; the caller synchronises
    // the stream before `h` goes away)
    cudaError_t assign(const std::vector<T>& h, cudaStream_t st = nullptr) {
        if (h.size() > cap || !p) {
            release();
            if (h.empty()) return cudaSuccess;
            cudaError_t e = cudaMalloc(&p, h.size() * sizeof(T));
            if (e != cudaSuccess) return e;
            cap = h.size();
        }
        n = h.size();
        if (n == 0) return cudaSuccess;
        return cudaMemcpyAsync(p, h.data(), n * sizeof(T), cudaMemcpyHostToDevice, st);
    }
    cudaError_t resize(size_t count) {
        if (count == n && p) return cudaSuccess;
        if (count <= cap && p && count > 0) { n = count; return cudaSuccess; }
        release();
        n = count;
        if (n == 0) return cudaSuccess;
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    // scratch buffers that are reused call after call: grow, never shrink
    cudaError_t reserve(size_t count) { return (p && n >= count) ? cudaSuccess : resize(count); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cap = 0;
    }
};

struct DeviceState {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_traced = nullptr;   // this device's share of the current render has been traced (cancel relay, fork)
    DevBuf<int> cancel_word;           // the word this device's kernels watch during a cancellable render (KParams::cancel_flag)
    cudaStream_t cancel_stream = nullptr;   // carries the 4-byte copy that raises it while the render kernel runs
    DevBuf<DevPrim> prims;
    DevBuf<DevPrim> prims_lin;
    DevBuf<DevNode> nodes;
    DevBuf<DevTexture> textures;
    DevBuf<DevInstance> instances;
    DevBuf<float4> perlin;
    DevBuf<uint8_t> perm;
    DevBuf<DevPrimD> prims_d;
    DevBuf<int> prim_kind;
    DevBuf<uint32_t> prim_id;
    DevBuf<DevNodeD> nodes_d;
    DevBuf<int> prim_inst;
    DevBuf<DevInstanceD> instances_d;
    std::vector<cudaArray_t> arrays;
    std::vector<std::pair<int, int>> array_dims;   // width, height of arrays[i]: a re-upload with the same image sizes reuses array and texture object
    std::vector<cudaTextureObject_t> tex;
    DevBuf<float> accum;
    DevBuf<float> slice_buf;
    DevBuf<double> out64;
    DevBuf<double> pp_in, pp_mapped;   // rc_postprocess scratch (kept between calls)
    DevBuf<uint8_t> pp_rgba;
    DevBuf<unsigned long long> counter;
    // rc_render_adaptive, per pixel: still tracing, samples traced, the last round's sum of y^2, running sum of y^2, error
    DevBuf<uint8_t> ad_active;
    DevBuf<int> ad_spp;
    DevBuf<float> ad_m2;
    DevBuf<double> ad_s2, ad_err;
    WavefrontState wf;
    std::map<std::string, SpecKernel> spec_cache;   // scene-specialised kernels loaded on this device
    int sm_count = 0, clock_khz = 0;
};

}  // namespace

// One image shared by the ranks of a box (rc_frame_create / rc_frame_open): [image 0][image 1][progress words],
// all in one allocation on rank 0's device.  Word 32 * r: the last frame rank r has stored completely (r >= 1);
// word 0: the last frame whose image rank 0 has released for writing.
struct rc_frame {
    float* base = nullptr;
    size_t image_floats = 0;
    int* words = nullptr;
    int width = 0, height = 0, rank = 0, world = 1;
    int frame_no = 0;                  // frames rendered through this handle so far
    bool owner = false;
    int* timed_out = nullptr;          // mapped host word raised by a wait that gave up
    DevBuf<double> out64;
};

struct rc_ctx {
    std::vector<DeviceState> devs;
    KParams kp;             // scene part filled at upload (device pointers of device 0 patched per launch)
    AovParamsD aov;
    int mode = RT_MODE_CONST_LINEAR;
    size_t smem_bytes = 0;
    bool has_scene = false, has_camera = false;
    bool has_textures = false;   // any primitive whose texture is not a solid colour
    int mats_mask = 0xF;         // material kinds the scene uses
    int prims_mask = 0xF;        // primitive kinds the scene uses (bit RT_PRIM_*; moving spheres count as spheres)
    std::string spec_source;     // generated source of the scene-specialised kernel ("" = not generated yet)
    std::string spec_source_moments;   // the same kernel with second moments, for adaptive rounds ("" = not generated yet)
    int spec_rounds = 10;        // Philox rounds spec_source and spec_source_moments were generated for
    std::vector<LbvhObject> objects, objects_next;   // top-level objects of the uploaded scene (rc_build_lbvh)
    std::vector<int> prim_order;       // device primitive i = uploaded primitive prim_order[i] (empty: identity)
    bool lbvh = false;
    std::vector<rc_frame*> frames;     // rc_frame_create / rc_frame_open
    bool stats_pending = false;        // the last render's time / counters have not been read back yet
    std::vector<void*> shared_owned, shared_opened;   // rc_shared_alloc / rc_shared_open
    int n_prims = 0, n_perlin = 0;
    bool instanced = false;
    rc_camera camera;
    rc_stats stats;
    MultiState multi;
    int* cancel_relay = nullptr;       // one page-locked word holding 1: the source of the copy that raises a device's cancel word
    uint64_t spec_clock = 0;           // use counter of the scene-specialised kernel caches (LRU)
};

namespace {

void free_scene(DeviceState& d) {
    cudaSetDevice(d.device);
    for (auto t : d.tex) cudaDestroyTextureObject(t);
    for (auto a : d.arrays) cudaFreeArray(a);
    d.tex.clear();
    d.arrays.clear();
    d.array_dims.clear();
}

void free_tables(DeviceState& d) {
    d.prims.release(); d.prims_lin.release(); d.nodes.release(); d.textures.release(); d.instances.release();
    d.perlin.release(); d.perm.release(); d.prims_d.release(); d.prim_kind.release();
    d.prim_id.release(); d.nodes_d.release(); d.prim_inst.release(); d.instances_d.release();
}

// Checker levels of the longest chain of checker textures (checkered.rs:32-43 follows children without a limit), or -1
// when a chain runs into a cycle; then *cycle_at is a texture on it.  The children must already be in range.
int checker_chain_depth(const rc_scene* s, int* cycle_at) {
    std::vector<int> depth(s->n_textures, -1);   // -1: not measured yet, -2: on the path being followed
    int longest = 0;
    for (int root = 0; root < s->n_textures; ++root) {
        // iterative depth-first walk: (texture, children visited so far)
        std::vector<std::pair<int, int>> stack{{root, 0}};
        while (!stack.empty()) {
            auto& top = stack.back();
            const rc_texture& t = s->textures[top.first];
            if (t.type != RC_TEX_CHECKER) { depth[top.first] = 0; stack.pop_back(); continue; }
            if (top.second == 0) {
                if (depth[top.first] >= 0) { stack.pop_back(); continue; }
                depth[top.first] = -2;
            }
            if (top.second < 2) {
                const int child = top.second++ == 0 ? t.a : t.b;
                if (depth[child] == -2) { *cycle_at = child; return -1; }
                if (depth[child] == -1) stack.push_back({child, 0});
                continue;
            }
            depth[top.first] = 1 + std::max(depth[t.a], depth[t.b]);
            longest = std::max(longest, depth[top.first]);
            stack.pop_back();
        }
    }
    return longest;
}

int validate_scene(const rc_scene* s) {
    if (!s) return fail(RC_ERR_INVALID, "scene is NULL");
    if (s->n_prims < 0 || s->n_materials < 0 || s->n_textures < 0 || s->n_images < 0 || s->n_perlin < 0 || s->n_nodes < 0)
        return fail(RC_ERR_INVALID, "negative table size");
    if (s->n_prims > 0 && (!s->prim_type || !s->prim_data || !s->prim_material || !s->prim_id))
        return fail(RC_ERR_INVALID, "primitive arrays missing");
    if (s->n_images > RT_MAX_IMAGES) return fail(RC_ERR_INVALID, "more than 8 image textures");
    if ((s->n_materials > 0 && !s->materials) || (s->n_textures > 0 && !s->textures) || (s->n_nodes > 0 && !s->nodes) ||
        (s->n_images > 0 && !s->images) || (s->n_perlin > 0 && !s->perlin))
        return fail(RC_ERR_INVALID, "a table with a non-zero count is NULL");
    for (int i = 0; i < s->n_images; ++i)
        if (s->images[i].width <= 0 || s->images[i].height <= 0 || !s->images[i].rgba) return fail(RC_ERR_INVALID, "empty image texture");
    if (s->n_prims >= (1 << 24)) return fail(RC_ERR_INVALID, "too many primitives");
    for (int i = 0; i < s->n_prims; ++i) {
        if (s->prim_type[i] < 0 || s->prim_type[i] > RC_PRIM_MOVING_SPHERE) return fail(RC_ERR_INVALID, "unknown primitive type");
        if (s->prim_type[i] == RC_PRIM_MOVING_SPHERE) {
            if (!s->prim_motion) return fail(RC_ERR_INVALID, "moving sphere without prim_motion");
            if (s->prim_motion[5 * (size_t)i + 4] == s->prim_motion[5 * (size_t)i + 3]) return fail(RC_ERR_INVALID, "moving sphere with time_a == time_b");
            if (s->prim_instance && s->n_instances > 0 && s->prim_instance[i] >= 0) return fail(RC_ERR_INVALID, "instanced moving spheres are not supported");
        }
        int m = s->prim_material[i];
        if (m < 0 || m >= s->n_materials) return fail(RC_ERR_INVALID, "primitive material index out of range");
        if (s->prim_id[i] == 0) return fail(RC_ERR_INVALID, "object id 0 is reserved for a miss");
        if (s->prim_instance && s->n_instances > 0 && (s->prim_instance[i] >= s->n_instances || s->prim_instance[i] < -1))
            return fail(RC_ERR_INVALID, "primitive instance index out of range");
    }
    for (int i = 0; i < s->n_materials; ++i) {
        const rc_material& m = s->materials[i];
        if (m.type < 0 || m.type > 3) return fail(RC_ERR_INVALID, "unknown material type");
        if (m.type != RC_MAT_DIELECTRIC && (m.texture < 0 || m.texture >= s->n_textures))
            return fail(RC_ERR_INVALID, "material texture index out of range");
    }
    for (int i = 0; i < s->n_textures; ++i) {
        const rc_texture& t = s->textures[i];
        if (t.type < 0 || t.type > 3) return fail(RC_ERR_INVALID, "unknown texture type");
        if (t.type == RC_TEX_CHECKER && (t.a < 0 || t.a >= s->n_textures || t.b < 0 || t.b >= s->n_textures))
            return fail(RC_ERR_INVALID, "checker child texture out of range");
        if (t.type == RC_TEX_IMAGE && (t.a < 0 || t.a >= s->n_images)) return fail(RC_ERR_INVALID, "image index out of range");
        if (t.type == RC_TEX_NOISE && (t.a < 0 || t.a >= s->n_perlin)) return fail(RC_ERR_INVALID, "perlin index out of range");
    }
    int cycle_at = -1;
    if (checker_chain_depth(s, &cycle_at) < 0)
        return fail(RC_ERR_INVALID, "checker texture " + std::to_string(cycle_at) + " is its own descendant (a cycle of checker children)");
    for (int i = 0; i < s->n_nodes; ++i) {
        const rc_bvh_node& n = s->nodes[i];
        if (n.left >= 0) {
            if (n.left != i + 1 || n.right <= n.left || n.right >= s->n_nodes)
                return fail(RC_ERR_INVALID, "BVH nodes must be stored in pre-order (left child = index + 1)");
        } else {
            int first = ~n.left;
            if (first < 0 || n.right < 1 || n.right > 127 || first + n.right > s->n_prims)
                return fail(RC_ERR_INVALID, "BVH leaf range out of bounds");
        }
    }
    if (s->n_instances > 0 && s->prim_instance) {
        if (!s->instances) return fail(RC_ERR_INVALID, "instance table missing");
        for (int i = 0; i < s->n_prims; ++i)
            if (s->prim_instance[i] >= 0 && s->n_nodes == 0)
                return fail(RC_ERR_INVALID, "scenes with RotateY / Translate instances need the BVH (n_nodes > 0)");
    }
    return RC_OK;
}

inline float4 f4(double x, double y, double z, float w) { return make_float4((float)x, (float)y, (float)z, w); }
inline float bits(int v) { float f; std::memcpy(&f, &v, 4); return f; }
inline float ubits(uint32_t v) { float f; std::memcpy(&f, &v, 4); return f; }
inline int ibits(float f) { int v; std::memcpy(&v, &f, 4); return v; }

// next float toward -inf / +inf, then a relative pad: the fp32 boxes must
// contain the f64 boxes and tolerate fp32 slab arithmetic
inline float pad_lo(double v, double ext) { return (float)(v - (1e-6 * ext + 1e-6 * std::fabs(v) + 1e-30)); }
inline float pad_hi(double v, double ext) { return (float)(v + (1e-6 * ext + 1e-6 * std::fabs(v) + 1e-30)); }

void set_skip(const rc_scene* s, int i, int skip, std::vector<int>& out) {
    out[i] = skip;
    const rc_bvh_node& n = s->nodes[i];
    if (n.left >= 0) {
        set_skip(s, n.left, n.right, out);
        set_skip(s, n.right, skip, out);
    }
}

#define RC_SMEM_STAGE_LIMIT (36 * 1024)
int pick_mode(const rc_scene* s, bool rects_fit, bool instanced, size_t& smem_bytes) {
    const char* force = std::getenv("RC_SCENE_MODE");  // experiments: const | smem | global | smemlin
    size_t perlin_bytes = (size_t)s->n_perlin * (256 * 16 + 768);
    size_t bvh_bytes = (size_t)s->n_nodes * sizeof(DevNode) + (size_t)s->n_prims * sizeof(DevPrim);
    int mode;
    // instanced scenes always traverse the BVH: its (possibly non-bounding, Q14) boxes are part of the semantics
    if (!instanced && s->n_prims <= RT_MAX_CONST_PRIMS && rects_fit) mode = RT_MODE_CONST_LINEAR;
    // shared-memory staging pays only while it does not cost occupancy (profiles/r01_random_bvh_v1_ncu.md:
    // 62 KB per CTA left 12 warps per SM and 44 % issue utilisation; the same tables read through L1 ran 1.5x
    // faster): keep the per-CTA copy below a sixth of the SM's 227 KB, larger tables are read through L1/L2
    else if (s->n_nodes > 0 && bvh_bytes + perlin_bytes <= RC_SMEM_STAGE_LIMIT) mode = RT_MODE_SMEM_BVH;
    else if (s->n_nodes > 0) mode = RT_MODE_GLOBAL_BVH;
    else mode = RT_MODE_SMEM_LINEAR;
    if (force && !instanced) {
        std::string f(force);
        if (f == "const" && s->n_prims <= RT_MAX_CONST_PRIMS && rects_fit) mode = RT_MODE_CONST_LINEAR;
        else if (f == "smem" && s->n_nodes > 0) mode = RT_MODE_SMEM_BVH;
        else if (f == "global" && s->n_nodes > 0) mode = RT_MODE_GLOBAL_BVH;
        else if (f == "smemlin") mode = RT_MODE_SMEM_LINEAR;
    }
    smem_bytes = perlin_bytes;
    if (mode == RT_MODE_SMEM_BVH) smem_bytes += bvh_bytes;
    // the linear modes stage the type-sorted table (the constant-bank mode too: its hit records
    // and shading index it per lane)
    if (mode == RT_MODE_SMEM_LINEAR || mode == RT_MODE_CONST_LINEAR) smem_bytes += (size_t)s->n_prims * sizeof(DevPrim);
    return mode;
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return RC_OK;
}

template <int MODE, bool TEX>
int launch_mega_mode(const KParams& kp, float* accum, int sampler, int rounds, int blocks, size_t smem, cudaStream_t st) {
#define RC_LAUNCH(S, R)                                                                         \
    do {                                                                                        \
        int rc__ = set_smem(megakernel_render<MODE, S, R, TEX>, smem);                          \
        if (rc__ != RC_OK) return rc__;                                                         \
        megakernel_render<MODE, S, R, TEX><<<blocks, RT_BLOCK, smem, st>>>(kp, accum);          \
    } while (0)
    if (rounds == 7) { if (sampler == RC_SAMPLER_REJECTION) RC_LAUNCH(1, 7); else RC_LAUNCH(0, 7); }
    else { if (sampler == RC_SAMPLER_REJECTION) RC_LAUNCH(1, 10); else RC_LAUNCH(0, 10); }
#undef RC_LAUNCH
    CUDA_TRY(cudaGetLastError());
    return RC_OK;
}

// one adaptive round: the direct sampler and 10 Philox rounds only
template <int MODE, bool TEX>
int launch_moments_mode(const KParams& kp, float* accum, int blocks, size_t smem, cudaStream_t st, const uint8_t* active, float* round_m2) {
    int rc = set_smem(megakernel_moments<MODE, TEX>, smem);
    if (rc != RC_OK) return rc;
    megakernel_moments<MODE, TEX><<<blocks, RT_BLOCK, smem, st>>>(kp, accum, active, round_m2);
    CUDA_TRY(cudaGetLastError());
    return RC_OK;
}

// active != NULL: an adaptive round (megakernel_moments)
int launch_mega(int mode, bool tex, const KParams& kp, float* accum, int sampler, int rounds, int blocks, size_t smem, cudaStream_t st,
                const uint8_t* active = nullptr, float* round_m2 = nullptr) {
#define RC_MODE(M) (!active ? (tex ? launch_mega_mode<M, true>(kp, accum, sampler, rounds, blocks, smem, st)          \
                                   : launch_mega_mode<M, false>(kp, accum, sampler, rounds, blocks, smem, st))        \
                             : (tex ? launch_moments_mode<M, true>(kp, accum, blocks, smem, st, active, round_m2)     \
                                    : launch_moments_mode<M, false>(kp, accum, blocks, smem, st, active, round_m2)))
    switch (mode) {
    case RT_MODE_CONST_LINEAR: return RC_MODE(RT_MODE_CONST_LINEAR);
    case RT_MODE_SMEM_BVH: return RC_MODE(RT_MODE_SMEM_BVH);
    case RT_MODE_GLOBAL_BVH: return RC_MODE(RT_MODE_GLOBAL_BVH);
    default: return RC_MODE(RT_MODE_SMEM_LINEAR);
    }
#undef RC_MODE
}

int check_params(const rc_params* p) {
    if (!p) return fail(RC_ERR_INVALID, "params is NULL");
    if (p->width < 2 || p->height < 2) return fail(RC_ERR_INVALID, "width and height must be >= 2 (u = x/(W-1), cpu.rs:35-40)");
    if (p->samples < 1) return fail(RC_ERR_INVALID, "samples must be >= 1");
    if (p->max_depth < 0) return fail(RC_ERR_INVALID, "max_depth must be >= 0");
    if (p->world < 0 || p->rank < 0 || (p->world > 0 && p->rank >= p->world)) return fail(RC_ERR_INVALID, "bad rank/world");
    if (p->rng_rounds != 0 && p->rng_rounds != 7 && p->rng_rounds != 10) return fail(RC_ERR_INVALID, "rng_rounds must be 0, 7 or 10");
    if ((long long)p->width * p->height > (1 << 24)) return fail(RC_ERR_INVALID, "more than 2^24 pixels (RNG counter layout)");
    if (p->samples > (1 << 24)) return fail(RC_ERR_INVALID, "more than 2^24 samples per pixel (RNG counter layout)");
    if (p->max_depth > 63) return fail(RC_ERR_INVALID, "max_depth > 63 (RNG counter layout)");
    if (p->variant != RC_VARIANT_MEGAKERNEL && p->variant != RC_VARIANT_WAVEFRONT) return fail(RC_ERR_INVALID, "unknown variant");
    if (p->sampler != RC_SAMPLER_DIRECT && p->sampler != RC_SAMPLER_REJECTION) return fail(RC_ERR_INVALID, "unknown sampler");
    if (p->split != RC_SPLIT_TILES && p->split != RC_SPLIT_SAMPLES) return fail(RC_ERR_INVALID, "unknown split");
    if (p->specialize < 0 || p->specialize > 2) return fail(RC_ERR_INVALID, "specialize must be 0, 1 or 2");
    if (!(p->tile_w == 0 && p->tile_h == 0) && !(p->tile_w == RT_TILE_W && p->tile_h == RT_TILE_H))
        return fail(RC_ERR_INVALID, "tile_w x tile_h must be 0 x 0 or 16 x 8 (the kernels' tile is fixed)");
    return RC_OK;
}

// KParams::vstep from the camera and the (screen) height behind inv_hm1: vertical / ((H - 1) * 65536), in f64
void set_vstep(KParams& kp, int screen_height) {
    const double s = 1.0 / ((double)(screen_height - 1) * 65536.0);
    kp.vstep = make_float4((float)(kp.cam.vertical.x * s), (float)(kp.cam.vertical.y * s), (float)(kp.cam.vertical.z * s), 0.0f);
}

// Fill the per-launch part of KParams for participant `part` of `parts`.
void partition(KParams& kp, const rc_params* p, int part, int parts) {
    kp.width = p->width; kp.height = p->height;
    kp.max_depth = p->max_depth;
    kp.fixed_jitter = p->fixed_jitter;
    kp.key = (uint32_t)p->seed ^ (uint32_t)(p->seed >> 32);
    for (int r = 0; r < 10; ++r) kp.ks[r] = kp.key + (uint32_t)r * PHILOX2_W;
    kp.inv_wm1 = 1.0f / (float)(p->width - 1); kp.inv_hm1 = 1.0f / (float)(p->height - 1);
    kp.wm1 = (float)(p->width - 1);
    set_vstep(kp, p->height);
    kp.px_scale_x = kp.px_scale_y = 1;
    kp.tile_w = RT_TILE_W; kp.tile_h = RT_TILE_H;
    kp.slices = 1; kp.slice_buf = nullptr;
    kp.overwrite = 0;
    kp.final_scale = 0.0f;
    kp.tiles_x = (p->width + RT_TILE_W - 1) / RT_TILE_W;
    int tiles_y = (p->height + RT_TILE_H - 1) / RT_TILE_H;
    int total = kp.tiles_x * tiles_y;
    if (p->split == RC_SPLIT_SAMPLES) {
        // contiguous sample slices; every participant traces all tiles
        kp.tile_first = 0; kp.tile_stride = 1; kp.n_tiles = total;
        long long lo = (long long)p->samples * part / parts, hi = (long long)p->samples * (part + 1) / parts;
        kp.s_begin = (int)lo; kp.s_end = (int)hi;
    } else {
        // interleaved tiles: tile k -> participant k mod parts
        kp.tile_first = part; kp.tile_stride = parts;
        kp.n_tiles = part < total ? (total - part + parts - 1) / parts : 0;
        kp.s_begin = 0; kp.s_end = p->samples;
    }
}

bool cancelled(const volatile int32_t* cancel) { return cancel && *cancel != 0; }

// tile split over the devices of one context with peer stores into device 0's buffer (rc_multi.cuh)
bool direct_tiles(const rc_ctx* ctx, const rc_params* p) {
    return ctx->devs.size() > 1 && p->split == RC_SPLIT_TILES && ctx->multi.peer_write_ok && p->variant == RC_VARIANT_MEGAKERNEL;
}

// One round of rc_render_adaptive: the samples [s_begin, s_end) of the pixels flagged in `active`
struct AdaptiveRound {
    const uint8_t* active;
    float* round_m2;
    int s_begin, s_end;
};

// What one render call asks of trace_share besides its rc_params
struct ShareCall {
    float* accum0;                       // device 0's destination buffer
    const volatile int32_t* cancel;      // the caller's cancel flag (may be null)
    bool store = false;                  // KParams::overwrite: store the pixel sums instead of adding them
    float final_scale = 0.0f;            // KParams::final_scale
    bool spread_stores = false;          // a sample-split rc_render_frame of several ranks: no forced tail slicing
    int preview_sw = 0, preview_sh = 0, preview_w = 0, preview_h = 0;   // preview scale and screen size (0: no preview)
    const AdaptiveRound* round = nullptr;   // a round of rc_render_adaptive, which owns the call's start event and
                                            // segment counter
};

// Trace this context's share into each device's own accumulation buffer (device 0 uses `call.accum0`), then,
// unless the render was cancelled, join or gather the other devices' pixels onto device 0.
int trace_share(rc_ctx* ctx, const rc_params* p, const ShareCall& call, bool& was_cancelled) {
    was_cancelled = false;
    const int n_dev = (int)ctx->devs.size();
    const int world = p->world > 0 ? p->world : 1;
    const int parts = world * n_dev;
    const int rounds = p->rng_rounds ? p->rng_rounds : 10;
    // direct tile split: every device stores its pixels into device 0's buffer (peer memory) itself
    const bool direct = direct_tiles(ctx, p);
    uint64_t launches = 0;
    bool used_spec = false;
    for (int k = 0; k < n_dev; ++k) {
        DeviceState& d = ctx->devs[k];
        CUDA_TRY(cudaSetDevice(d.device));
        if (k == 0) {
            if (!call.round) CUDA_TRY(cudaEventRecord(d.ev0, d.stream));
            // fork: whatever device 0's stream holds so far — the zero-fill of the buffer the other devices are about
            // to store into, the previous frame's finalize that still reads it — happens before any of them starts
            if (n_dev > 1) CUDA_TRY(cudaEventRecord(d.ev_traced, d.stream));
        } else {
            CUDA_TRY(cudaStreamWaitEvent(d.stream, ctx->devs[0].ev_traced, 0));
        }
        if (!call.round) CUDA_TRY(cudaMemsetAsync(d.counter.p, 0, sizeof(unsigned long long), d.stream));
    }
    // A cancel flag does not change how the frame is launched (one launch per device, sliced if need be): every CTA
    // reads a word in its device's memory before it starts, and this call relays the caller's flag to that word — a
    // 4-byte copy on a second stream — while it waits (do_cancel per row, src/renderer/cpu.rs:55-62).  (The word used to
    // be mapped HOST memory: ten thousand CTAs per GPU then each read it over PCIe, which cost 0.7 ms per frame on one
    // GPU and 7 ms with eight processes on one host.)  The wavefront variant is not interruptible.
    const bool relay = call.cancel != nullptr && p->variant == RC_VARIANT_MEGAKERNEL;
    if (relay)
        for (int k = 0; k < n_dev; ++k) {
            DeviceState& d = ctx->devs[k];
            CUDA_TRY(cudaSetDevice(d.device));
            CUDA_TRY(d.cancel_word.resize(1));
            CUDA_TRY(cudaMemsetAsync(d.cancel_word.p, 0, sizeof(int), d.stream));
        }
    for (int k = 0; k < n_dev; ++k) {
        DeviceState& d = ctx->devs[k];
        CUDA_TRY(cudaSetDevice(d.device));
        KParams kp = ctx->kp;
        kp.prims = d.prims.p; kp.prims_lin = d.prims_lin.p; kp.nodes = d.nodes.p; kp.textures = d.textures.p;
        kp.instances = d.instances.p;
        kp.perlin = d.perlin.p; kp.perlin_perm = d.perm.p;
        for (size_t i = 0; i < d.tex.size(); ++i) kp.images[i] = d.tex[i];
        kp.segment_counter = d.counter.p;
        kp.cancel_flag = relay ? d.cancel_word.p : nullptr;
        partition(kp, p, p->rank * n_dev + k, parts);
        // tile culling needs one ray origin per tile (no lens), primitives that stay where they are, and a linear mode
        kp.tile_cull = (!kp.lens_enabled && !kp.has_motion && !p->fixed_jitter && std::getenv("RC_NO_TILE_CULL") == nullptr) ? 1 : 0;
        if (call.preview_sw > 0) {   // scaled preview: p->width/height is the block grid, u and v refer to the screen
            kp.px_scale_x = call.preview_sw; kp.px_scale_y = call.preview_sh;
            kp.wm1 = (float)(call.preview_w - 1);
            kp.inv_wm1 = 1.0f / (float)(call.preview_w - 1); kp.inv_hm1 = 1.0f / (float)(call.preview_h - 1);
            set_vstep(kp, call.preview_h);
        }
        float* accum = (k == 0 || direct) ? call.accum0 : d.accum.p;
        kp.overwrite = call.store ? 1 : 0;
        kp.final_scale = call.final_scale;
        const uint8_t* active = nullptr;
        float* round_m2 = nullptr;
        if (call.round) {
            kp.s_begin = call.round->s_begin; kp.s_end = call.round->s_end;
            active = call.round->active; round_m2 = call.round->round_m2;
        }
        if (kp.n_tiles == 0 || kp.s_end <= kp.s_begin) { if (relay) CUDA_TRY(cudaEventRecord(d.ev_traced, d.stream)); continue; }
        if (p->variant == RC_VARIANT_WAVEFRONT) {
            if (kp.has_motion && rounds != 10) return fail(RC_ERR_INVALID, "the wavefront variant traces moving spheres with 10 Philox rounds only");
            int rc = wavefront_render(d.wf, ctx->mode, kp, accum, p->sampler, rounds, ctx->smem_bytes, d.stream, d.sm_count, launches);
            if (rc != RC_OK) return fail(rc, "wavefront launch failed: " + std::string(cudaGetErrorString(cudaGetLastError())));
            continue;
        }
        // scene-specialised kernel (NVRTC), cached per scene and device
        SpecKernel* spec = nullptr;
        // (the constant-table path gets its primitives as immediates; the BVH paths get the scene's kinds of
        // primitive, material and wrapper compiled in or out — 48 KB of dynamic shared memory without opt-in)
        const bool spec_mode_ok = ctx->smem_bytes <= 48 * 1024 &&
                                  (ctx->mode == RT_MODE_CONST_LINEAR ||
                                   ctx->mode == RT_MODE_SMEM_BVH || ctx->mode == RT_MODE_GLOBAL_BVH);
        if (p->specialize && spec_mode_ok && p->sampler == RC_SAMPLER_DIRECT && !p->fixed_jitter) {
            std::string err;
            if (!spec_load_api((const void*)&rc_abi_version)) err = spec_api().err;
            else {
                if (ctx->spec_rounds != rounds) { ctx->spec_source.clear(); ctx->spec_source_moments.clear(); }
                std::string& source = call.round ? ctx->spec_source_moments : ctx->spec_source;
                if (source.empty()) {
                    source = spec_generate(ctx->kp, ctx->has_textures, ctx->mats_mask, ctx->mode, ctx->prims_mask, ctx->instanced, rounds,
                                           call.round != nullptr);
                    ctx->spec_rounds = rounds;
                }
                spec = spec_build(d.spec_cache, source, err, ++ctx->spec_clock);
            }
            if (!spec && p->specialize == 1) return fail(RC_ERR_STATE, "scene specialisation failed: " + err);
        } else if (p->specialize == 1) {
            return fail(RC_ERR_INVALID, "specialize = 1 needs the megakernel, the direct sampler and no fixed jitter");
        }
        const int s0 = kp.s_begin, s1 = kp.s_end;
        // few tiles on this device (its share of a multi-GPU render): cut every tile's sample range
        // into slices so that the grid is still >= 8 full machine loads of CTAs
        kp.slices = 1;
        kp.slice_buf = nullptr;
        kp.slice_halving = 0;
        if (!call.round) {   // (adaptive rounds run unsliced: the round's moments are stored per pixel by the kernel)
            const long long want = 8LL * d.sm_count * 10;
            long long sl = (want + kp.n_tiles - 1) / kp.n_tiles;
            if (sl > (s1 - s0) / 16) sl = (s1 - s0) / 16;
            // A frame with plenty of tiles still ends in a tail: a CTA of the bench frame (128 pixels x 1024 samples)
            // runs for 4 ms, and while the last ones finish the machine drains.  Two slices (2/3 and 1/3 of the samples)
            // halve that: 32.37 against 32.63 ms for the whole frame on one GPU (tools/time_share.py 1); three or more
            // cost more in per-CTA set-up than they save.
            // (not for a sample-split frame of several ranks: there the kernel's own stores go to rank 0 over NVLink and
            // should be spread over the frame, not issued by reduce_slices_kernel in one burst at its end)
            if (sl < 2 && s1 - s0 >= 512 && !call.spread_stores) sl = 2;
            if (const char* e = std::getenv("RC_SLICES")) sl = std::atoll(e);
            // Slice lengths: halving (n/2, n/4, .., the last two equal) from five slices on, linearly decreasing below —
            // with two or three slices the halving scheme's last slice is too long a tail.  One rank's share of the
            // bench frame alone on one GPU (tools/time_share.py): 8-way split, six slices: 4.17 ms halving / 4.21 linear
            // (4.08 = an eighth of the frame); 2-way split, two slices: 16.54 halving / 16.39 linear (16.32 = half).
            kp.slice_halving = sl >= 5 ? 1 : 0;
            if (const char* e = std::getenv("RC_SLICE_HALVING")) kp.slice_halving = std::atoi(e);
            while (kp.slice_halving && sl > 1 && ((s1 - s0) >> (sl - 1)) < 8) --sl;   // the last two slices keep >= 8 samples
            if (sl > 1) {
                CUDA_TRY(d.slice_buf.resize((size_t)sl * kp.n_tiles * RT_BLOCK * 3));
                kp.slices = (int)sl;
                kp.slice_buf = d.slice_buf.p;
            }
        }
        {
            int rc = RC_ERR_CUDA;
            if (spec) {
                rc = spec_launch(spec, kp, accum, kp.n_tiles * kp.slices, ctx->smem_bytes, d.stream, active, round_m2) == 0 ? RC_OK : RC_ERR_CUDA;
                if (rc == RC_OK) used_spec = true;
                else if (p->specialize == 1) return fail(rc, "launch of the scene-specialised kernel failed");
            }
            if (rc != RC_OK)   // no specialised kernel, or (specialize == 2) it could not be launched: the precompiled one
                rc = launch_mega(ctx->mode, ctx->has_textures, kp, accum, p->sampler, rounds, kp.n_tiles * kp.slices, ctx->smem_bytes, d.stream,
                                 active, round_m2);
            if (rc != RC_OK) return rc;
            ++launches;
            if (kp.slices > 1) {
                reduce_slices_kernel<<<(kp.n_tiles * RT_BLOCK + 255) / 256, 256, 0, d.stream>>>(kp, accum);
                CUDA_TRY(cudaGetLastError());
                ++launches;
            }
        }
        if (relay) CUDA_TRY(cudaEventRecord(d.ev_traced, d.stream));
    }
    ctx->stats.kernel_launches = launches;
    ctx->stats.specialized = used_spec ? 1 : 0;
    if (relay) {
        // wait for the frame while relaying the caller's flag; a raised flag empties the rest of the grid at once
        for (;;) {
            bool done = true;
            for (int k = 0; k < n_dev && done; ++k) {
                const cudaError_t e = cudaEventQuery(ctx->devs[k].ev_traced);
                if (e == cudaErrorNotReady) done = false;
                else if (e != cudaSuccess) return fail(RC_ERR_CUDA, std::string("cudaEventQuery: ") + cudaGetErrorString(e));
            }
            if (!was_cancelled && cancelled(call.cancel)) {
                was_cancelled = true;
                for (int k = 0; k < n_dev; ++k) {
                    DeviceState& d = ctx->devs[k];
                    CUDA_TRY(cudaSetDevice(d.device));
                    CUDA_TRY(cudaMemcpyAsync(d.cancel_word.p, ctx->cancel_relay, sizeof(int), cudaMemcpyHostToDevice, d.cancel_stream));
                }
                // (the copy has landed before this call returns, so it can never hit the word of a later frame)
                for (int k = 0; k < n_dev; ++k) CUDA_TRY(cudaStreamSynchronize(ctx->devs[k].cancel_stream));
            }
            if (done) break;
            std::this_thread::sleep_for(std::chrono::microseconds(20));
        }
        CUDA_TRY(cudaSetDevice(ctx->devs[0].device));
    }
    if (was_cancelled || n_dev == 1) return RC_OK;
    auto stream_of = [&](size_t k) { return ctx->devs[k].stream; };
    auto device_of = [&](size_t k) { return ctx->devs[k].device; };
    if (direct) {
        if (multi_join(ctx->multi, stream_of, device_of) != 0)
            return fail(RC_ERR_CUDA, std::string("multi-device join failed: ") + multi_error(ctx->multi));
        return RC_OK;
    }
    const int rc = multi_gather(ctx->multi, p->split, (size_t)p->width * p->height * 3, call.accum0,
                                [&](size_t k) { return ctx->devs[k].accum.p; }, stream_of, device_of);
    if (rc != RC_OK) return fail(rc, std::string("multi-device gather failed: ") + multi_error(ctx->multi));
    return RC_OK;
}

int ensure_accum(rc_ctx* ctx, const rc_params* p, bool device0_too, bool zero = true) {
    size_t n = (size_t)p->width * p->height * 3;
    for (size_t k = device0_too ? 0 : 1; k < ctx->devs.size(); ++k) {
        DeviceState& d = ctx->devs[k];
        CUDA_TRY(cudaSetDevice(d.device));
        CUDA_TRY(d.accum.resize(n));
        if (zero) CUDA_TRY(cudaMemsetAsync(d.accum.p, 0, n * sizeof(float), d.stream));
    }
    return RC_OK;
}

// rc_render / rc_render_preview own their accumulation buffers and trace every pixel's samples in ONE launch, so the
// megakernel can STORE the sums instead of adding them to a zero-filled buffer (no memset, no read of the frame) —
// but only when this call's launches write every pixel of every buffer read afterwards: a tile split with a single
// participant overall (one device, or peer stores of all devices into device 0's buffer, and world = 1), or a sample
// split in which every device of the context has samples to trace (each writes all pixels of its own buffer,
// ncclReduce adds them).  Otherwise a pixel nobody writes would keep the previous render's sums.
bool can_store(const rc_ctx* ctx, const rc_params* p) {
    if (p->variant != RC_VARIANT_MEGAKERNEL) return false;
    const int n_dev = (int)ctx->devs.size();
    const int world = p->world > 0 ? p->world : 1;
    if (p->split == RC_SPLIT_TILES) return world == 1 && (n_dev == 1 || direct_tiles(ctx, p));
    const int parts = world * n_dev;
    for (int k = 0; k < n_dev; ++k) {
        const int part = p->rank * n_dev + k;
        if ((long long)p->samples * (part + 1) / parts <= (long long)p->samples * part / parts) return false;
    }
    return true;
}

// pixel-samples of participant `part`'s share: its tiles clipped to the image, times its samples
uint64_t share_samples(const rc_params* p, int part, int parts) {
    KParams kp;
    std::memset(&kp, 0, sizeof(kp));
    partition(kp, p, part, parts);
    uint64_t pixels = 0;
    for (int i = 0; i < kp.n_tiles; ++i) {
        const int tile = kp.tile_first + i * kp.tile_stride;
        const int tx = tile % kp.tiles_x, ty = tile / kp.tiles_x;
        pixels += (uint64_t)std::min(RT_TILE_W, p->width - tx * RT_TILE_W) * std::min(RT_TILE_H, p->height - ty * RT_TILE_H);
    }
    return pixels * (uint64_t)(kp.s_end - kp.s_begin);
}

// End of a render call: the stop event is recorded, nothing is waited for.  Time and segment counters are
// resolved when somebody asks (rc_get_stats), so that a caller who only enqueues work — bench.py's timed
// loop, a multi-rank job — never has its stream drained by the library.
int finish_stats(rc_ctx* ctx, const rc_params* p) {
    DeviceState& d0 = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d0.device));
    CUDA_TRY(cudaEventRecord(d0.ev1, d0.stream));
    const int n_dev = (int)ctx->devs.size();
    const int parts = (p->world > 0 ? p->world : 1) * n_dev;
    ctx->stats.samples = 0;
    for (int k = 0; k < n_dev; ++k) ctx->stats.samples += share_samples(p, p->rank * n_dev + k, parts);
    ctx->stats_pending = true;
    return RC_OK;
}

int resolve_stats(rc_ctx* ctx) {
    if (!ctx->stats_pending) return RC_OK;
    DeviceState& d0 = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d0.device));
    CUDA_TRY(cudaEventSynchronize(d0.ev1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, d0.ev0, d0.ev1));
    ctx->stats.gpu_ms = ms;
    uint64_t segs = 0;
    for (auto& d : ctx->devs) {
        unsigned long long v = 0;
        CUDA_TRY(cudaSetDevice(d.device));
        CUDA_TRY(cudaStreamSynchronize(d.stream));
        CUDA_TRY(cudaMemcpy(&v, d.counter.p, sizeof(v), cudaMemcpyDeviceToHost));
        segs += v;
    }
    ctx->stats.segments = segs;
    ctx->stats_pending = false;
    CUDA_TRY(cudaSetDevice(d0.device));
    return RC_OK;
}

}  // namespace

// ---------------------------------------------------------------------------
// Tree quality.  A host hands over the tree it has; the reference's is a median split along a RANDOM axis
// (src/bvh_node.rs:31-82), and one huge object — the Random scene's radius-1000 ground sphere — then inflates every
// ancestor box.  The closest hit does not depend on the tree (exact ties aside, Q13), the number of boxes a ray
// visits does: for instance-free scenes of RC_SAH_MIN_LEAVES leaves and more the library re-splits THE SAME LEAVES by
// the surface-area heuristic (full sweep over three axes per node; same algorithm as harness._build_bvh_sah and
// racer_host.cpp::build_bvh_sah) and keeps the result when its expected number of box tests per ray is at least
// 10 % below the given tree's — so a tree that is already SAH-quality is walked exactly as passed.
// Scenes with instances keep their tree: there the stored boxes decide visibility (Q14).  RC_KEEP_TREE=1: never.
// ---------------------------------------------------------------------------
#define RC_SAH_MIN_LEAVES 65
struct ResplitScene {   // a re-ordered copy of the primitive arrays + the new nodes; `scene` points into it
    rc_scene scene;
    std::vector<int32_t> type, material, instance, order;
    std::vector<double> data, aabb, motion;
    std::vector<uint32_t> id;
    std::vector<rc_bvh_node> nodes;
};

namespace {
struct SahLeaf { double lo[3], hi[3]; int first, count; };

double sah_area(const double* lo, const double* hi) {
    const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return 2.0 * (dx * dy + dy * dz + dz * dx);
}

// expected box tests per ray ~ sum over nodes of area(node) / area(root)
double sah_tree_cost(const rc_bvh_node* nodes, int n) {
    const double root = sah_area(nodes[0].bmin, nodes[0].bmax);
    double c = 0.0;
    for (int i = 0; i < n; ++i) c += sah_area(nodes[i].bmin, nodes[i].bmax);
    return root > 0.0 ? c / root : (double)n;
}

int sah_build(const std::vector<SahLeaf>& leaves, std::vector<int>& idx, int begin, int end, std::vector<rc_bvh_node>& nodes, std::vector<int>& leaf_order) {
    const int me = (int)nodes.size();
    nodes.push_back(rc_bvh_node());
    const int m = end - begin;
    if (m == 1) {
        const SahLeaf& l = leaves[idx[begin]];
        for (int a = 0; a < 3; ++a) { nodes[me].bmin[a] = l.lo[a]; nodes[me].bmax[a] = l.hi[a]; }
        nodes[me].left = ~(int)leaf_order.size();   // patched to the primitive range afterwards
        nodes[me].right = 1;
        leaf_order.push_back(idx[begin]);
        return me;
    }
    int best_axis = 0, best_k = 1;
    double best_cost = 0.0;
    bool have = false;
    std::vector<int> srt(idx.begin() + begin, idx.begin() + end);
    std::vector<double> rarea((size_t)m);
    for (int axis = 0; axis < 3; ++axis) {
        std::sort(srt.begin(), srt.end(), [&](int x, int y) {
            const double kx = leaves[x].lo[axis] + leaves[x].hi[axis], ky = leaves[y].lo[axis] + leaves[y].hi[axis];
            return kx < ky || (kx == ky && x < y);
        });
        double lo[3], hi[3];
        for (int i = m - 1; i >= 1; --i) {      // area of the box of srt[i..m)
            const SahLeaf& l = leaves[srt[i]];
            for (int a = 0; a < 3; ++a) {
                lo[a] = i == m - 1 ? l.lo[a] : std::min(lo[a], l.lo[a]);
                hi[a] = i == m - 1 ? l.hi[a] : std::max(hi[a], l.hi[a]);
            }
            rarea[i] = sah_area(lo, hi);
        }
        for (int k = 1; k < m; ++k) {           // left = srt[0..k)
            const SahLeaf& l = leaves[srt[k - 1]];
            for (int a = 0; a < 3; ++a) {
                lo[a] = k == 1 ? l.lo[a] : std::min(lo[a], l.lo[a]);
                hi[a] = k == 1 ? l.hi[a] : std::max(hi[a], l.hi[a]);
            }
            const double cost = sah_area(lo, hi) * (double)k + rarea[k] * (double)(m - k);
            if (!have || cost < best_cost) { have = true; best_cost = cost; best_axis = axis; best_k = k; }
        }
    }
    std::sort(idx.begin() + begin, idx.begin() + end, [&](int x, int y) {
        const double kx = leaves[x].lo[best_axis] + leaves[x].hi[best_axis], ky = leaves[y].lo[best_axis] + leaves[y].hi[best_axis];
        return kx < ky || (kx == ky && x < y);
    });
    const int l = sah_build(leaves, idx, begin, begin + best_k, nodes, leaf_order);
    const int r = sah_build(leaves, idx, begin + best_k, end, nodes, leaf_order);
    nodes[me].left = l; nodes[me].right = r;
    for (int a = 0; a < 3; ++a) {
        nodes[me].bmin[a] = std::min(nodes[l].bmin[a], nodes[r].bmin[a]);
        nodes[me].bmax[a] = std::max(nodes[l].bmax[a], nodes[r].bmax[a]);
    }
    return me;
}
}  // namespace

// Returns true and fills `out` (out.scene = the scene to upload instead of *s) when the tree was replaced.
static bool resplit_sah(const rc_scene* s, ResplitScene& out) {
    if (s->n_nodes < 2 * RC_SAH_MIN_LEAVES - 1 || std::getenv("RC_KEEP_TREE") != nullptr) return false;
    if (s->prim_instance && s->n_instances > 0)
        for (int i = 0; i < s->n_prims; ++i) if (s->prim_instance[i] >= 0) return false;
    std::vector<SahLeaf> leaves;
    for (int i = 0; i < s->n_nodes; ++i) {
        const rc_bvh_node& n = s->nodes[i];
        if (n.left >= 0) continue;
        SahLeaf l;
        for (int a = 0; a < 3; ++a) { l.lo[a] = n.bmin[a]; l.hi[a] = n.bmax[a]; }
        l.first = ~n.left; l.count = n.right;
        leaves.push_back(l);
    }
    if ((int)leaves.size() < RC_SAH_MIN_LEAVES || leaves.size() > 200000) return false;
    std::vector<int> idx(leaves.size()), leaf_order;
    for (size_t i = 0; i < idx.size(); ++i) idx[i] = (int)i;
    out.nodes.clear();
    out.nodes.reserve((size_t)s->n_nodes);
    sah_build(leaves, idx, 0, (int)leaves.size(), out.nodes, leaf_order);
    if (sah_tree_cost(out.nodes.data(), (int)out.nodes.size()) > 0.9 * sah_tree_cost(s->nodes, s->n_nodes)) return false;
    // primitives into the new tree's depth-first leaf order
    std::vector<int> first_new(leaf_order.size());
    out.order.clear();
    for (size_t k = 0; k < leaf_order.size(); ++k) {
        const SahLeaf& l = leaves[leaf_order[k]];
        first_new[k] = (int)out.order.size();
        for (int j = 0; j < l.count; ++j) out.order.push_back(l.first + j);
    }
    if ((int)out.order.size() != s->n_prims) return false;   // a primitive outside every leaf: leave the scene alone
    for (rc_bvh_node& n : out.nodes)
        if (n.left < 0) { const int k = ~n.left; n.left = ~first_new[k]; n.right = leaves[leaf_order[k]].count; }
    const int np = s->n_prims;
    out.type.resize(np); out.material.resize(np); out.id.resize(np); out.data.resize(5 * (size_t)np);
    out.instance.assign(np, -1);
    if (s->prim_aabb) out.aabb.resize(6 * (size_t)np);
    if (s->prim_motion) out.motion.resize(5 * (size_t)np);
    for (int i = 0; i < np; ++i) {
        const int src = out.order[i];
        out.type[i] = s->prim_type[src]; out.material[i] = s->prim_material[src]; out.id[i] = s->prim_id[src];
        std::memcpy(&out.data[5 * (size_t)i], s->prim_data + 5 * (size_t)src, 5 * sizeof(double));
        if (s->prim_aabb) std::memcpy(&out.aabb[6 * (size_t)i], s->prim_aabb + 6 * (size_t)src, 6 * sizeof(double));
        if (s->prim_motion) std::memcpy(&out.motion[5 * (size_t)i], s->prim_motion + 5 * (size_t)src, 5 * sizeof(double));
    }
    out.scene = *s;
    out.scene.prim_type = out.type.data(); out.scene.prim_material = out.material.data(); out.scene.prim_id = out.id.data();
    out.scene.prim_data = out.data.data();
    out.scene.prim_instance = s->prim_instance ? out.instance.data() : nullptr;
    out.scene.prim_aabb = s->prim_aabb ? out.aabb.data() : nullptr;
    out.scene.prim_motion = s->prim_motion ? out.motion.data() : nullptr;
    out.scene.nodes = out.nodes.data();
    out.scene.n_nodes = (int32_t)out.nodes.size();
    return true;
}

struct HostTables {   // everything rc_upload_scene derives from an rc_scene, before any device call
    std::vector<DevPrim> prims, prims_lin;
    std::vector<DevPrimD> prims_d;
    std::vector<int> kinds;
    std::vector<uint32_t> ids;
    std::vector<DevNode> nodes;
    std::vector<DevNodeD> nodes_d;
    std::vector<DevTexture> textures;
    std::vector<float4> perlin;
    std::vector<uint8_t> perm;
    std::vector<DevInstance> instances;
    std::vector<DevInstanceD> instances_d;
    std::vector<int> prim_inst;
    KParams kp;
    int mode = RT_MODE_CONST_LINEAR;
    size_t smem_bytes = 0;
    bool has_textures = false;
    int mats_mask = 0xF;
    int prims_mask = 0xF;
};

// f64 host scene -> fp32 device tables (pure host arithmetic)
static void build_tables(const rc_scene* s, HostTables& t) {
    std::memset(&t.kp, 0, sizeof(t.kp));
    // ---- fp32 + f64 primitive tables ----
    std::vector<DevPrim>& prims = t.prims; prims.assign(s->n_prims, DevPrim());
    std::vector<DevPrimD>& prims_d = t.prims_d; prims_d.assign(s->n_prims, DevPrimD());
    std::vector<int>& kinds = t.kinds; kinds.assign(s->n_prims, 0);
    std::vector<uint32_t>& ids = t.ids; ids.assign(s->n_prims, 0u);
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    bool any_textured = false, any_motion = false;
    for (int i = 0; i < s->n_prims; ++i) {
        const double* d = s->prim_data + 5 * (size_t)i;
        const rc_material& m = s->materials[s->prim_material[i]];
        int type = s->prim_type[i];
        DevPrim& p = prims[i];
        DevPrimD& q = prims_d[i];
        for (int k = 0; k < 4; ++k) q.a[k] = d[k];
        for (int k = 0; k < 5; ++k) q.motion[k] = 0.0;
        double vel[3] = {0.0, 0.0, 0.0};
        if (type == RC_PRIM_SPHERE) {
            double cc = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] - d[3] * d[3];
            p.a = make_float4((float)d[0], (float)d[1], (float)d[2], (float)d[3]);
            p.b.x = (float)cc;
            q.k_or_cc = cc;
        } else if (type == RC_PRIM_MOVING_SPHERE) {
            // MovingSphere::pos (moving_sphere.rs:37-39) = pos + (time - ta)/(tb - ta) (pos_b - pos)
            //                                            = (pos - ta v) + time v,  v = (pos_b - pos)/(tb - ta)
            const double* m = s->prim_motion + 5 * (size_t)i;
            for (int k = 0; k < 5; ++k) q.motion[k] = m[k];
            double c0[3];
            for (int k = 0; k < 3; ++k) { vel[k] = (m[k] - d[k]) / (m[4] - m[3]); c0[k] = d[k] - m[3] * vel[k]; }
            p.a = make_float4((float)c0[0], (float)c0[1], (float)c0[2], (float)d[3]);
            p.b.x = 0.f;
            q.k_or_cc = 0.0;
            any_motion = true;
        } else {
            p.a = make_float4((float)d[0], (float)d[1], (float)d[2], (float)d[3]);
            p.b.x = (float)d[4];
            q.k_or_cc = d[4];
        }
        p.b.y = (float)m.param;
        int tex_type = RT_TEX_SOLID, tex_index = -1;
        double col[3] = {1.0, 1.0, 1.0};
        if (m.type != RC_MAT_DIELECTRIC) {
            const rc_texture& t = s->textures[m.texture];
            tex_type = t.type;
            tex_index = m.texture;
            if (t.type == RC_TEX_SOLID) { col[0] = t.color[0]; col[1] = t.color[1]; col[2] = t.color[2]; tex_index = -1; }
        }
        int inst = (s->prim_instance && s->n_instances > 0) ? s->prim_instance[i] : -1;
        if (tex_type != RT_TEX_SOLID) any_textured = true;
        int packed = type | (m.type << 4) | (tex_type << 8) | ((inst + 1) << 12);
        p.b.z = bits(packed);
        p.b.w = bits(tex_index);
        p.c = f4(col[0], col[1], col[2], ubits(s->prim_id[i]));
        // +axis unit normal of a rectangle (xy_rect.rs:45, xz_rect.rs:46, yz_rect.rs:46); 0 for a sphere
        // a sphere: the centre's velocity per unit of ray time (0 when it does not move)
        p.n = make_float4(type == RC_PRIM_YZ_RECT ? 1.f : 0.f, type == RC_PRIM_XZ_RECT ? 1.f : 0.f, type == RC_PRIM_XY_RECT ? 1.f : 0.f, 0.f);
        if (type == RC_PRIM_MOVING_SPHERE) p.n = make_float4((float)vel[0], (float)vel[1], (float)vel[2], 0.f);
        p.n.w = (float)m.type;   // RT_MAT_* as a float: shade_hit tests it with one float compare
        kinds[i] = type;
        ids[i] = s->prim_id[i];
        if (s->prim_aabb)
            for (int a = 0; a < 3; ++a) {
                lo[a] = std::fmin(lo[a], s->prim_aabb[6 * i + a]);
                hi[a] = std::fmax(hi[a], s->prim_aabb[6 * i + 3 + a]);
            }
    }
    // ---- threaded BVH ----
    std::vector<DevNode>& nodes = t.nodes; nodes.assign(s->n_nodes, DevNode());
    std::vector<DevNodeD>& nodes_d = t.nodes_d; nodes_d.assign(s->n_nodes, DevNodeD());
    if (s->n_nodes > 0) {
        std::vector<int> skip(s->n_nodes, s->n_nodes);
        set_skip(s, 0, s->n_nodes, skip);
        for (int i = 0; i < s->n_nodes; ++i) {
            const rc_bvh_node& n = s->nodes[i];
            int leaf = n.left < 0 ? ((~n.left) | (n.right << 24)) : -1;
            double ext = 0;
            for (int a = 0; a < 3; ++a) ext = std::fmax(ext, n.bmax[a] - n.bmin[a]);
            nodes[i].lo = make_float4(pad_lo(n.bmin[0], ext), pad_lo(n.bmin[1], ext), pad_lo(n.bmin[2], ext), bits(skip[i]));
            nodes[i].hi = make_float4(pad_hi(n.bmax[0], ext), pad_hi(n.bmax[1], ext), pad_hi(n.bmax[2], ext), bits(leaf));
            for (int a = 0; a < 3; ++a) { nodes_d[i].lo[a] = n.bmin[a]; nodes_d[i].hi[a] = n.bmax[a]; }
            nodes_d[i].skip = skip[i];
            nodes_d[i].leaf = leaf;
        }
    }
    std::vector<DevTexture>& textures = t.textures; textures.assign(s->n_textures, DevTexture());
    for (int i = 0; i < s->n_textures; ++i) {
        const rc_texture& t = s->textures[i];
        textures[i].type = t.type; textures[i].a = t.a; textures[i].b = t.b;
        textures[i].scale = (float)t.scale;
        textures[i].color = f4(t.color[0], t.color[1], t.color[2], 0.f);
    }
    std::vector<float4>& perlin = t.perlin; perlin.assign((size_t)s->n_perlin * 256, make_float4(0.f, 0.f, 0.f, 0.f));
    std::vector<uint8_t>& perm = t.perm; perm.assign((size_t)s->n_perlin * 768, 0);
    for (int k = 0; k < s->n_perlin; ++k)
        for (int i = 0; i < 256; ++i) {
            const rc_perlin& pl = s->perlin[k];
            perlin[(size_t)k * 256 + i] = f4(pl.ran_vec[i][0], pl.ran_vec[i][1], pl.ran_vec[i][2], 0.f);
            perm[(size_t)k * 768 + i] = (uint8_t)(pl.perm_x[i] & 255);
            perm[(size_t)k * 768 + 256 + i] = (uint8_t)(pl.perm_y[i] & 255);
            perm[(size_t)k * 768 + 512 + i] = (uint8_t)(pl.perm_z[i] & 255);
        }

    t.instances.assign(s->n_instances, DevInstance());
    t.instances_d.assign(s->n_instances, DevInstanceD());
    bool any_rotate = false, any_instance = false;
    for (int i = 0; i < s->n_instances; ++i) {
        const rc_instance& in = s->instances[i];
        DevInstance& d = t.instances[i];
        d.sin_theta = (float)in.sin_theta; d.cos_theta = (float)in.cos_theta;
        d.ox = (float)in.offset[0]; d.oy = (float)in.offset[1]; d.oz = (float)in.offset[2];
        d.flags = in.flags;
        DevInstanceD& q = t.instances_d[i];
        q.sin_theta = in.sin_theta; q.cos_theta = in.cos_theta;
        q.offset[0] = in.offset[0]; q.offset[1] = in.offset[1]; q.offset[2] = in.offset[2];
        q.flags = in.flags;
    }
    t.prim_inst.assign(s->n_prims, -1);
    for (int i = 0; i < s->n_prims; ++i) {
        int inst = (s->prim_instance && s->n_instances > 0) ? s->prim_instance[i] : -1;
        t.prim_inst[i] = inst;
        if (inst >= 0) { any_instance = true; if (s->instances[inst].flags & 1) any_rotate = true; }
    }
    KParams& kp = t.kp;
    kp.ref_aabb = any_rotate ? 1 : 0;
    kp.has_motion = any_motion ? 1 : 0;
    kp.n_prims = s->n_prims; kp.n_nodes = s->n_nodes; kp.n_perlin = s->n_perlin;
    int cycle_at = -1;
    kp.checker_depth = checker_chain_depth(s, &cycle_at);   // validate_scene has ruled out cycles
    kp.bg_a = f4(s->bg_a[0], s->bg_a[1], s->bg_a[2], bits(s->bg_type));
    kp.bg_b = f4(s->bg_b[0], s->bg_b[1], s->bg_b[2], 0.f);
    // type-sorted table for the linear modes (stable: canonical order within a kind)
    std::vector<DevPrim>& prims_lin = t.prims_lin;
    prims_lin.clear();
    prims_lin.reserve(s->n_prims);
    for (int type = 0; type < 4; ++type) {
        for (int i = 0; i < s->n_prims; ++i)   // moving spheres (kind 4) share group 0 with the static ones
            if (t.prim_inst[i] < 0 && (kinds[i] == RC_PRIM_MOVING_SPHERE ? 0 : kinds[i]) == type) prims_lin.push_back(prims[i]);
        kp.lin_end[type] = (int)prims_lin.size();
    }
    // instanced top-level objects follow, each a run of primitives sharing object id, instance and stored Aabb
    kp.n_cobj = 0;
    bool objs_fit = s->n_instances <= RT_MAX_CONST_OBJS && (!any_instance || s->prim_aabb != nullptr);
    for (int i = 0; i < s->n_instances && i < RT_MAX_CONST_OBJS; ++i) kp.cinst[i] = t.instances[i];
    for (int i = 0; i < s->n_prims && objs_fit; ++i) {
        if (t.prim_inst[i] < 0) continue;
        const double* b = s->prim_aabb + 6 * (size_t)i;
        bool same = false;
        if (kp.n_cobj > 0 && i > 0 && t.prim_inst[i - 1] == t.prim_inst[i] && (s->prim_id[i - 1] >> 3) == (s->prim_id[i] >> 3) &&
            std::memcmp(s->prim_aabb + 6 * (size_t)(i - 1), b, 6 * sizeof(double)) == 0) {
            const int meta = ibits(kp.cobj_hi[kp.n_cobj - 1].w);
            if ((meta & 255) < 255) { kp.cobj_hi[kp.n_cobj - 1].w = bits(meta + 1); same = true; }
        }
        if (!same) {
            if (kp.n_cobj == RT_MAX_CONST_OBJS) { objs_fit = false; break; }
            // the cull volume in fp32: rounded OUTWARD by one ulp-scale pad so it contains the f64 box
            double ext = 0;
            for (int a = 0; a < 3; ++a) ext = std::fmax(ext, b[3 + a] - b[a]);
            kp.cobj_lo[kp.n_cobj] = make_float4(pad_lo(b[0], ext), pad_lo(b[1], ext), pad_lo(b[2], ext), bits((int)prims_lin.size()));
            kp.cobj_hi[kp.n_cobj] = make_float4(pad_hi(b[3], ext), pad_hi(b[4], ext), pad_hi(b[5], ext), bits(1 | (t.prim_inst[i] << 8)));
            ++kp.n_cobj;
        }
        prims_lin.push_back(prims[i]);
    }
    if (!objs_fit) {   // too many instanced objects for the linear modes: they traverse the BVH
        kp.n_cobj = 0;
        for (int i = 0; i < s->n_prims; ++i) if (t.prim_inst[i] >= 0 && (int)prims_lin.size() < s->n_prims) prims_lin.push_back(prims[i]);
    }
    for (int i = 0; i < RT_MAX_CONST_PRIMS; ++i)
        if (i < s->n_prims) kp.cprims[i] = prims_lin[i]; else std::memset(&kp.cprims[i], 0, sizeof(DevPrim));
    std::memset(kp.crect_bounds, 0, sizeof(kp.crect_bounds));
    std::memset(kp.crect_k, 0, sizeof(kp.crect_k));
    bool rects_fit = true;
    for (int g = 0; g < 3; ++g) {
        int begin = kp.lin_end[g], n = kp.lin_end[g + 1] - begin;
        if (n > RT_MAX_CONST_RECTS) { rects_fit = false; continue; }
        for (int j = 0; j < n; ++j) {
            const float4 r4 = prims_lin[begin + j].a;   // (a0, a1, b0, b1) -> (ca, ha, cb, hb), formed in f64
            kp.crect_bounds[g][j] = make_float4((float)(0.5 * ((double)r4.x + r4.y)), (float)(0.5 * ((double)r4.y - r4.x)),
                                                (float)(0.5 * ((double)r4.z + r4.w)), (float)(0.5 * ((double)r4.w - r4.z)));
            kp.crect_k[g][j] = prims_lin[begin + j].b.x;
        }
    }
    for (int i = 0; i < RT_MAX_IMAGES; ++i) {
        kp.image_w[i] = i < s->n_images ? s->images[i].width : 0;
        kp.image_h[i] = i < s->n_images ? s->images[i].height : 0;
    }
    t.mode = pick_mode(s, rects_fit && objs_fit, any_instance && !objs_fit, t.smem_bytes);
    t.has_textures = any_textured;
    t.mats_mask = 0;
    t.prims_mask = 0;
    for (int i = 0; i < s->n_prims; ++i) {
        t.mats_mask |= 1 << s->materials[s->prim_material[i]].type;
        t.prims_mask |= 1 << (s->prim_type[i] == RC_PRIM_MOVING_SPHERE ? RC_PRIM_SPHERE : s->prim_type[i]);
    }

}

// ===========================================================================
#pragma GCC visibility push(default)
extern "C" {

const char* rc_last_error(void) { return g_last_error.c_str(); }
int rc_destroy(rc_ctx* ctx);
int rc_frame_close(rc_ctx* ctx, rc_frame* frame);
int rc_abi_version(void) { return RC_ABI_VERSION; }

int rc_create(const int32_t* devices, int32_t n, rc_ctx** out) {
    if (!out) return fail(RC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(RC_ERR_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                          " (there is no CPU fallback for the render path)");
    if (n <= 0) n = 1;
    rc_ctx* ctx = new rc_ctx();
    std::memset(&ctx->kp, 0, sizeof(ctx->kp));
    std::memset(&ctx->aov, 0, sizeof(ctx->aov));
    std::memset(&ctx->stats, 0, sizeof(ctx->stats));
    ctx->devs.resize(n);
    for (int k = 0; k < n; ++k) {
        DeviceState& d = ctx->devs[k];
        d.device = devices ? devices[k] : k;
        if (d.device < 0 || d.device >= count) {
            delete ctx;
            return fail(RC_ERR_NO_DEVICE, "device ordinal out of range");
        }
        cudaError_t err = cudaSetDevice(d.device);
        if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking);
        if (err == cudaSuccess) err = cudaEventCreate(&d.ev0);
        if (err == cudaSuccess) err = cudaEventCreate(&d.ev1);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&d.ev_traced, cudaEventDisableTiming);
        if (err == cudaSuccess) err = d.counter.resize(1);
        cudaDeviceProp prop;
        if (err == cudaSuccess) err = cudaGetDeviceProperties(&prop, d.device);
        if (err != cudaSuccess) {
            delete ctx;
            return fail(RC_ERR_CUDA, std::string("device setup failed: ") + cudaGetErrorString(err));
        }
        d.sm_count = prop.multiProcessorCount;
        d.clock_khz = prop.clockRate;
        // The small kernels every render path ends in are loaded now, not inside the first frame that needs them: with
        // lazy module loading the first launch of reduce_slices_kernel cost 0.6 s in the middle of a render.
        {
            cudaFuncAttributes fa;
            cudaFuncGetAttributes(&fa, reduce_slices_kernel);
            cudaFuncGetAttributes(&fa, finalize_kernel);
            cudaFuncGetAttributes(&fa, finalize_to_f64_kernel);
            cudaFuncGetAttributes(&fa, widen_kernel);
            cudaFuncGetAttributes(&fa, frame_wait_kernel);
            cudaFuncGetAttributes(&fa, frame_publish_kernel);
            cudaFuncGetAttributes(&fa, sum_slots_kernel);
            cudaGetLastError();
        }
    }
    ctx->stats.n_devices = n;
    ctx->stats.sm_count = ctx->devs[0].sm_count;
    ctx->stats.sm_clock_khz = ctx->devs[0].clock_khz;
    int rc = multi_init(ctx->multi, ctx->devs.size(), [&](size_t k) { return ctx->devs[k].device; });
    if (rc != RC_OK) {
        delete ctx;
        return fail(rc, "peer access setup failed");
    }
    cudaSetDevice(ctx->devs[0].device);
    // the source of the copies that raise the devices' cancel words: one page-locked word holding 1
    if (cudaHostAlloc((void**)&ctx->cancel_relay, sizeof(int), cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        rc_destroy(ctx);
        return fail(RC_ERR_CUDA, "cudaHostAlloc of the cancel relay failed");
    }
    *ctx->cancel_relay = 1;
    for (auto& d : ctx->devs) {
        cudaSetDevice(d.device);
        if (cudaStreamCreateWithFlags(&d.cancel_stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError();
            rc_destroy(ctx);
            return fail(RC_ERR_CUDA, "cudaStreamCreate of the cancel stream failed");
        }
    }
    cudaSetDevice(ctx->devs[0].device);
    *out = ctx;
    return RC_OK;
}

int rc_destroy(rc_ctx* ctx) {
    if (!ctx) return RC_OK;
    cudaSetDevice(ctx->devs.empty() ? 0 : ctx->devs[0].device);
    while (!ctx->frames.empty()) rc_frame_close(ctx, ctx->frames.back());
    for (void* q : ctx->shared_opened) cudaIpcCloseMemHandle(q);
    for (void* q : ctx->shared_owned) cudaFree(q);
    if (ctx->cancel_relay) cudaFreeHost(ctx->cancel_relay);
    multi_destroy(ctx->multi);
    for (auto& d : ctx->devs) {
        cudaSetDevice(d.device);
        cudaDeviceSynchronize();
        free_scene(d);
        free_tables(d);
        d.accum.release(); d.slice_buf.release(); d.out64.release(); d.counter.release(); d.cancel_word.release();
        d.ad_active.release(); d.ad_spp.release(); d.ad_m2.release(); d.ad_s2.release(); d.ad_err.release();
        if (d.cancel_stream) cudaStreamDestroy(d.cancel_stream);
        d.pp_in.release(); d.pp_mapped.release(); d.pp_rgba.release();
        if (d.ev_traced) cudaEventDestroy(d.ev_traced);
        wavefront_release(d.wf);
        spec_release(d.spec_cache);
        if (d.ev0) cudaEventDestroy(d.ev0);
        if (d.ev1) cudaEventDestroy(d.ev1);
        if (d.own_stream && d.stream) cudaStreamDestroy(d.stream);
    }
    delete ctx;
    return RC_OK;
}

int rc_set_stream(rc_ctx* ctx, void* cuda_stream) {
    if (!ctx) return fail(RC_ERR_INVALID, "ctx is NULL");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    if (d.own_stream && d.stream) CUDA_TRY(cudaStreamDestroy(d.stream));
    d.stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    d.own_stream = false;
    return RC_OK;
}

int rc_upload_scene(rc_ctx* ctx, const rc_scene* s) {
    if (!ctx) return fail(RC_ERR_INVALID, "ctx is NULL");
    int rc = validate_scene(s);
    if (rc != RC_OK) return rc;
    ResplitScene resplit;
    const bool resplit_done = resplit_sah(s, resplit);
    if (resplit_done) s = &resplit.scene;   // same leaves, better tree; rc_get_bvh reports it and the permutation
    HostTables t;
    build_tables(s, t);
    if (!t.instances.empty() && t.kp.n_cobj == 0 && s->n_nodes == 0)
        return fail(RC_ERR_INVALID, "a scene with more than 8 instanced objects (or without prim_aabb) needs BVH nodes");
    // everything above is validation on host memory; from here on the context changes.  It holds no scene until
    // every device has all of its tables: a failed upload leaves has_scene == false, never a half-uploaded scene.
    ctx->has_scene = false;
    {   // keep the camera / launch fields already stored in ctx->kp
        DevCamera<float> cam = ctx->kp.cam;
        int lens = ctx->kp.lens_enabled;
        ctx->kp = t.kp;
        ctx->kp.cam = cam;
        ctx->kp.lens_enabled = lens;
    }
    ctx->mode = t.mode;
    ctx->smem_bytes = t.smem_bytes;
    ctx->has_textures = t.has_textures;
    ctx->mats_mask = t.mats_mask;
    ctx->prims_mask = t.prims_mask;
    ctx->spec_source.clear();
    ctx->spec_source_moments.clear();
    ctx->aov.n_prims = s->n_prims; ctx->aov.n_nodes = s->n_nodes;
    // top-level objects = runs of primitives that share an object id (id >> 3; a Box's six sides) and a stored Aabb
    ctx->objects.clear();
    ctx->prim_order.clear();
    if (resplit_done) ctx->prim_order = resplit.order;
    ctx->lbvh = false;
    ctx->n_prims = s->n_prims; ctx->n_perlin = s->n_perlin;
    ctx->instanced = !t.instances.empty();
    if (s->prim_aabb)
        for (int i = 0; i < s->n_prims; ++i) {
            const double* b = s->prim_aabb + 6 * (size_t)i;
            if (!ctx->objects.empty()) {
                LbvhObject& o = ctx->objects.back();
                if ((s->prim_id[i] >> 3) == (s->prim_id[o.first] >> 3) && o.count < 127 && std::memcmp(o.lo, b, 3 * sizeof(double)) == 0 &&
                    std::memcmp(o.hi, b + 3, 3 * sizeof(double)) == 0) { ++o.count; continue; }
            }
            LbvhObject o;
            std::memcpy(o.lo, b, 3 * sizeof(double)); std::memcpy(o.hi, b + 3, 3 * sizeof(double));
            o.first = i; o.count = 1;
            ctx->objects.push_back(o);
        }
    std::vector<DevPrim>& prims = t.prims; std::vector<DevPrim>& prims_lin = t.prims_lin;
    std::vector<DevPrimD>& prims_d = t.prims_d; std::vector<int>& kinds = t.kinds; std::vector<uint32_t>& ids = t.ids;
    std::vector<DevNode>& nodes = t.nodes; std::vector<DevNodeD>& nodes_d = t.nodes_d;
    std::vector<DevTexture>& textures = t.textures; std::vector<float4>& perlin = t.perlin; std::vector<uint8_t>& perm = t.perm;

    for (auto& d : ctx->devs) {
        // An interactive host re-uploads after every scene edit (main.rs:178-183): the table allocations are kept
        // and refilled with stream-ordered copies — the stream also orders them after any render still reading the
        // old tables — and the stream is drained once at the end instead of once per table.
        CUDA_TRY(cudaSetDevice(d.device));
        CUDA_TRY(cudaStreamSynchronize(d.stream));
        {   // image textures are kept when the new scene's images have the same sizes (an edit re-uploads the scene:
            // src/main.rs:178-183), only their pixels are copied again; otherwise they are rebuilt
            bool same = (int)d.arrays.size() == s->n_images;
            for (int i = 0; same && i < s->n_images; ++i)
                same = d.array_dims[i].first == s->images[i].width && d.array_dims[i].second == s->images[i].height;
            if (!same) free_scene(d);
        }
        CUDA_TRY(d.prims.assign(prims, d.stream));
        CUDA_TRY(d.prims_lin.assign(prims_lin, d.stream));
        CUDA_TRY(d.nodes.assign(nodes, d.stream));
        CUDA_TRY(d.textures.assign(textures, d.stream));
        CUDA_TRY(d.perlin.assign(perlin, d.stream));
        CUDA_TRY(d.perm.assign(perm, d.stream));
        CUDA_TRY(d.prims_d.assign(prims_d, d.stream));
        CUDA_TRY(d.prim_kind.assign(kinds, d.stream));
        CUDA_TRY(d.prim_id.assign(ids, d.stream));
        CUDA_TRY(d.nodes_d.assign(nodes_d, d.stream));
        CUDA_TRY(d.instances.assign(t.instances, d.stream));
        CUDA_TRY(d.instances_d.assign(t.instances_d, d.stream));
        CUDA_TRY(d.prim_inst.assign(t.prim_inst, d.stream));
        for (int i = 0; i < s->n_images; ++i) {
            // image textures as CUDA texture objects: point filter, clamp, u8 -> float/255
            // (src/texture/image.rs:28-51, Q21)
            const rc_image& im = s->images[i];
            if (i < (int)d.arrays.size()) {   // kept from the previous upload: same size, new pixels
                CUDA_TRY(cudaMemcpy2DToArrayAsync(d.arrays[i], 0, 0, im.rgba, (size_t)im.width * 4, (size_t)im.width * 4, im.height,
                                                  cudaMemcpyHostToDevice, d.stream));
                continue;
            }
            cudaChannelFormatDesc desc = cudaCreateChannelDesc<uchar4>();
            cudaArray_t arr;
            CUDA_TRY(cudaMallocArray(&arr, &desc, im.width, im.height));
            d.arrays.push_back(arr);
            d.array_dims.push_back(std::make_pair((int)im.width, (int)im.height));
            CUDA_TRY(cudaMemcpy2DToArray(arr, 0, 0, im.rgba, (size_t)im.width * 4, (size_t)im.width * 4, im.height, cudaMemcpyHostToDevice));
            cudaResourceDesc res;
            std::memset(&res, 0, sizeof(res));
            res.resType = cudaResourceTypeArray;
            res.res.array.array = arr;
            cudaTextureDesc td;
            std::memset(&td, 0, sizeof(td));
            td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
            td.filterMode = cudaFilterModePoint;
            td.readMode = cudaReadModeNormalizedFloat;
            td.normalizedCoords = 0;
            cudaTextureObject_t tex;
            CUDA_TRY(cudaCreateTextureObject(&tex, &res, &td, nullptr));
            d.tex.push_back(tex);
        }
        CUDA_TRY(cudaStreamSynchronize(d.stream));   // the host tables above go out of scope with this call
    }
    CUDA_TRY(cudaSetDevice(ctx->devs[0].device));
    ctx->has_scene = true;
    // A scene uploaded WITHOUT a BVH whose linear table would not fit the shared-memory staging budget gets one
    // built on the device (the linear loop stays what small scenes use; a large one would be O(N) per ray and
    // its table would not fit a CTA).  Results differ from the linear order only on exact ties (Q13).
    if (s->n_nodes == 0 && ctx->mode == RT_MODE_SMEM_LINEAR && (size_t)s->n_prims * sizeof(DevPrim) > RC_SMEM_STAGE_LIMIT) {
        if (ctx->objects.empty()) {
            if ((size_t)s->n_prims * sizeof(DevPrim) > 200 * 1024)
                return fail(RC_ERR_INVALID, "a scene this large needs BVH nodes, or prim_aabb so that rc_upload_scene can build them on the GPU");
        } else {
            int rc2 = rc_build_lbvh(ctx);
            if (rc2 != RC_OK) return rc2;
        }
    }
    return RC_OK;
}

int rc_set_camera(rc_ctx* ctx, const rc_camera* c) {
    if (!ctx || !c) return fail(RC_ERR_INVALID, "ctx or camera is NULL");
    ctx->camera = *c;
    auto v3f = [](const double* p) { return mk3<float>((float)p[0], (float)p[1], (float)p[2]); };
    auto v3d = [](const double* p) { return mk3<double>(p[0], p[1], p[2]); };
    // (upper_left_corner - origin) is formed in f64 here so the fp32 kernels
    // never subtract two large, nearly equal coordinates
    double rel[3] = {c->upper_left_corner[0] - c->origin[0], c->upper_left_corner[1] - c->origin[1],
                     c->upper_left_corner[2] - c->origin[2]};
    DevCamera<float>& f = ctx->kp.cam;
    f.origin = v3f(c->origin); f.upper_left_corner = v3f(rel); f.right = v3f(c->right); f.up = v3f(c->up);
    f.horizontal = v3f(c->horizontal); f.vertical = v3f(c->vertical);
    f.lens_radius = (float)c->lens_radius; f.time_a = (float)c->time_a; f.time_b = (float)c->time_b;
    // the specialised source depends on the camera (lens or pinhole; which pairs of opposite walls enclose it):
    // regenerate it — the text is the cache key, so an unchanged text costs no recompilation
    ctx->spec_source.clear();
    ctx->spec_source_moments.clear();
    ctx->kp.lens_enabled = c->lens_radius != 0.0;
    DevCamera<double>& g = ctx->aov.cam;
    g.origin = v3d(c->origin); g.upper_left_corner = v3d(c->upper_left_corner); g.right = v3d(c->right); g.up = v3d(c->up);
    g.horizontal = v3d(c->horizontal); g.vertical = v3d(c->vertical);
    g.lens_radius = c->lens_radius; g.time_a = c->time_a; g.time_b = c->time_b;
    ctx->has_camera = true;
    return RC_OK;
}

// rc_render_accumulate (store = false) and rc_render_tiles_into (store = true) once their arguments are checked
static int render_into(rc_ctx* ctx, const rc_params* p, float* dst, const volatile int32_t* cancel, bool store) {
    if (!ctx->has_scene || !ctx->has_camera) return fail(RC_ERR_STATE, "upload a scene and set a camera first");
    if (cancelled(cancel)) return fail(RC_ERR_CANCELLED, "cancel flag set before the render started");
    int rc = ensure_accum(ctx, p, false);
    if (rc != RC_OK) return rc;
    bool was_cancelled = false;
    rc = trace_share(ctx, p, ShareCall{dst, cancel, store}, was_cancelled);
    if (rc != RC_OK) return rc;
    return finish_stats(ctx, p);
}

int rc_render_accumulate(rc_ctx* ctx, const rc_params* p, float* d_accum, const volatile int32_t* cancel) {
    if (!ctx || !d_accum) return fail(RC_ERR_INVALID, "ctx or d_accum is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    return render_into(ctx, p, d_accum, cancel, false);
}

int rc_render_tiles_into(rc_ctx* ctx, const rc_params* p, float* d_image, const volatile int32_t* cancel) {
    if (!ctx || !d_image) return fail(RC_ERR_INVALID, "ctx or d_image is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (p->split != RC_SPLIT_TILES || p->variant != RC_VARIANT_MEGAKERNEL)
        return fail(RC_ERR_INVALID, "rc_render_tiles_into needs the tile split and the megakernel (pixels are stored, not added)");
    if (ctx->devs.size() > 1 && !ctx->multi.peer_write_ok) return fail(RC_ERR_INVALID, "rc_render_tiles_into over several devices needs peer access");
    return render_into(ctx, p, d_image, cancel, true);
}

// ---- a device buffer shared by the processes of one box (CUDA IPC over NVLink / PCIe peer mappings) ----
int rc_shared_alloc(rc_ctx* ctx, uint64_t bytes, void** d_ptr, uint8_t handle[64]) {
    if (!ctx || !d_ptr || !handle || bytes == 0) return fail(RC_ERR_INVALID, "bad rc_shared_alloc arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CUDA_TRY(cudaSetDevice(ctx->devs[0].device));
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, (size_t)bytes));
    CUDA_TRY(cudaMemset(p, 0, (size_t)bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(RC_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
    std::memcpy(handle, &h, 64);
    ctx->shared_owned.push_back(p);
    *d_ptr = p;
    return RC_OK;
}

int rc_shared_open(rc_ctx* ctx, const uint8_t handle[64], void** d_ptr) {
    if (!ctx || !d_ptr || !handle) return fail(RC_ERR_INVALID, "bad rc_shared_open arguments");
    CUDA_TRY(cudaSetDevice(ctx->devs[0].device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    ctx->shared_opened.push_back(p);
    *d_ptr = p;
    return RC_OK;
}

int rc_shared_close(rc_ctx* ctx, void* d_ptr) {
    if (!ctx || !d_ptr) return fail(RC_ERR_INVALID, "bad rc_shared_close arguments");
    CUDA_TRY(cudaSetDevice(ctx->devs[0].device));
    for (size_t i = 0; i < ctx->shared_owned.size(); ++i)
        if (ctx->shared_owned[i] == d_ptr) { ctx->shared_owned.erase(ctx->shared_owned.begin() + i); CUDA_TRY(cudaFree(d_ptr)); return RC_OK; }
    for (size_t i = 0; i < ctx->shared_opened.size(); ++i)
        if (ctx->shared_opened[i] == d_ptr) { ctx->shared_opened.erase(ctx->shared_opened.begin() + i); CUDA_TRY(cudaIpcCloseMemHandle(d_ptr)); return RC_OK; }
    return fail(RC_ERR_INVALID, "pointer was not returned by rc_shared_alloc / rc_shared_open on this context");
}

// ---- the one-process-per-GPU tile split, whole (header: rc_render_frame) ----
static size_t frame_bytes(int width, int height, int world, size_t* image_floats) {
    size_t n = (size_t)width * height * 3;
    n = (n + 63) & ~(size_t)63;                       // images start on 256-byte boundaries
    *image_floats = n;
    // two images (they alternate), each with one slot per rank: the tile split stores finished pixels into slot 0;
    // the sample split stores every rank's partial sums into its own slot, and rank 0 adds the slots up
    return 2 * (size_t)world * n * sizeof(float) + (size_t)(world + 1) * 32 * sizeof(int);
}

static int frame_init(rc_ctx* ctx, rc_frame* f, void* base, int width, int height, int rank, int world, bool owner) {
    size_t nf = 0;
    frame_bytes(width, height, world, &nf);
    f->base = (float*)base; f->image_floats = nf; f->words = (int*)(f->base + 2 * (size_t)world * nf);
    f->width = width; f->height = height; f->rank = rank; f->world = world; f->owner = owner;
    if (cudaHostAlloc((void**)&f->timed_out, sizeof(int), cudaHostAllocMapped) != cudaSuccess) return fail(RC_ERR_CUDA, "cudaHostAlloc failed");
    *f->timed_out = 0;
    ctx->frames.push_back(f);
    return RC_OK;
}

int rc_frame_create(rc_ctx* ctx, int32_t width, int32_t height, int32_t world, rc_frame** out, uint8_t handle[64]) {
    if (!ctx || !out || !handle || width < 2 || height < 2 || world < 1 || world > 30) return fail(RC_ERR_INVALID, "bad rc_frame_create arguments");
    size_t nf = 0;
    void* base = nullptr;
    int rc = rc_shared_alloc(ctx, frame_bytes(width, height, world, &nf), &base, handle);   // zero-filled: frame 0 is "done" everywhere
    if (rc != RC_OK) return rc;
    rc_frame* f = new rc_frame();
    rc = frame_init(ctx, f, base, width, height, 0, world, true);
    if (rc != RC_OK) { delete f; return rc; }
    *out = f;
    return RC_OK;
}

int rc_frame_open(rc_ctx* ctx, const uint8_t handle[64], int32_t width, int32_t height, int32_t rank, int32_t world, rc_frame** out) {
    if (!ctx || !out || !handle || width < 2 || height < 2 || world < 2 || rank < 1 || rank >= world) return fail(RC_ERR_INVALID, "bad rc_frame_open arguments");
    void* base = nullptr;
    int rc = rc_shared_open(ctx, handle, &base);
    if (rc != RC_OK) return rc;
    rc_frame* f = new rc_frame();
    rc = frame_init(ctx, f, base, width, height, rank, world, false);
    if (rc != RC_OK) { delete f; return rc; }
    *out = f;
    return RC_OK;
}

int rc_frame_close(rc_ctx* ctx, rc_frame* f) {
    if (!ctx || !f) return fail(RC_ERR_INVALID, "bad rc_frame_close arguments");
    auto it = std::find(ctx->frames.begin(), ctx->frames.end(), f);
    if (it == ctx->frames.end()) return fail(RC_ERR_INVALID, "frame does not belong to this context");
    ctx->frames.erase(it);
    cudaSetDevice(ctx->devs[0].device);
    cudaStreamSynchronize(ctx->devs[0].stream);
    int rc = rc_shared_close(ctx, f->base);
    if (f->timed_out) cudaFreeHost(f->timed_out);
    f->out64.release();
    delete f;
    return rc;
}

int rc_render_frame(rc_ctx* ctx, const rc_params* p, rc_frame* f, const float** d_rgb, double* out_rgb, const volatile int32_t* cancel) {
    if (!ctx || !f) return fail(RC_ERR_INVALID, "ctx or frame is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (std::find(ctx->frames.begin(), ctx->frames.end(), f) == ctx->frames.end()) return fail(RC_ERR_INVALID, "frame does not belong to this context");
    if (p->variant != RC_VARIANT_MEGAKERNEL) return fail(RC_ERR_INVALID, "rc_render_frame needs the megakernel");
    const bool by_samples = p->split == RC_SPLIT_SAMPLES;
    if (p->width != f->width || p->height != f->height) return fail(RC_ERR_INVALID, "params and frame sizes differ");
    const int world = p->world > 0 ? p->world : 1;
    if (world != f->world || p->rank != f->rank) return fail(RC_ERR_INVALID, "params and frame rank / world differ");
    if (f->rank != 0 && (d_rgb || out_rgb)) return fail(RC_ERR_INVALID, "only rank 0 receives the image");
    if (ctx->devs.size() != 1) return fail(RC_ERR_INVALID, "rc_render_frame is the one-process-per-GPU form: the context must hold one device");
    if (!ctx->has_scene || !ctx->has_camera) return fail(RC_ERR_STATE, "upload a scene and set a camera first");
    if (cancelled(cancel)) return fail(RC_ERR_CANCELLED, "cancel flag set before the render started");
    if (*f->timed_out) return fail(RC_ERR_STATE, "an earlier frame never completed (a rank stopped publishing progress)");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    const int frame_no = ++f->frame_no;
    // slot 0 of this frame's image: where the finished pixels are (tile split: stored there by every rank's render
    // kernel; sample split: summed there by rank 0 from the ranks' slots)
    float* image = f->base + (size_t)(frame_no & 1) * f->world * f->image_floats;
    // where THIS rank's kernel stores: finished pixels of its tiles into slot 0, or its partial sums into its own slot
    float* target = by_samples ? image + (size_t)f->rank * f->image_floats : image;
    // The image of frame n was last used by frame n - 2: the others wait for rank 0 to release it.  When rank 0's
    // stream gets HERE, everything enqueued on it before this call has run: the wait for every rank's frame n - 1 and
    // whatever read the images of frames n - 1 and n - 2.  So both images are free — this frame's and the NEXT one's
    // (frame n + 1 goes into the image of n - 1) — and rank 0 releases up to n + 1: the other ranks may run one frame
    // ahead of the slowest one instead of meeting it at every frame (a per-frame barrier in all but name, which is
    // what releasing only n amounted to: rank 0 gets here only after every rank's n - 1).
    if (world > 1) {
        if (f->rank == 0) frame_publish_kernel<<<1, 1, 0, d.stream>>>(f->words, frame_no + 1);
        else frame_wait_kernel<<<1, 32, 0, d.stream>>>(f->words, 0, 1, frame_no, f->timed_out);
        CUDA_TRY(cudaGetLastError());
    }
    bool was_cancelled = false;
    ShareCall call{target, cancel, true};
    call.final_scale = by_samples ? 0.0f : 1.0f / (float)p->samples;   // sample split: raw sums, the square root comes after the slots are added
    call.spread_stores = by_samples && world > 1;
    rc = trace_share(ctx, p, call, was_cancelled);
    if (rc != RC_OK) return rc;
    if (by_samples && (long long)p->samples * (f->rank + 1) / world <= (long long)p->samples * f->rank / world) {
        // fewer samples than ranks and none for this one: its slot still holds frame n - 2's sums, and rank 0 adds it
        CUDA_TRY(cudaMemsetAsync(target, 0, f->image_floats * sizeof(float), d.stream));
    }
    uint64_t extra = 0;
    if (world > 1) {
        if (f->rank != 0) { frame_publish_kernel<<<1, 1, 0, d.stream>>>(f->words + 32 * f->rank, frame_no); extra = 2; }
        else { frame_wait_kernel<<<1, 32, 0, d.stream>>>(f->words, 1, world - 1, frame_no, f->timed_out); extra = 2; }
        CUDA_TRY(cudaGetLastError());
    }
    if (by_samples && f->rank == 0) {
        // the reduce of the sample split: every rank's kernel has stored its partial sums into its slot of this image
        // over NVLink; rank 0 adds the slots in rank order (deterministic) and takes sqrt(sum / samples) into slot 0
        const size_t n = (size_t)p->width * p->height * 3;
        sum_slots_kernel<<<(unsigned)((n + 255) / 256), 256, 0, d.stream>>>(image, f->image_floats, world, n, 1.0f / (float)p->samples);
        CUDA_TRY(cudaGetLastError());
        extra += 1;
    }
    rc = finish_stats(ctx, p);
    if (rc != RC_OK) return rc;
    ctx->stats.kernel_launches += extra;
    if (d_rgb) *d_rgb = image;
    if (out_rgb && !was_cancelled) {
        const size_t n = (size_t)p->width * p->height * 3;
        CUDA_TRY(f->out64.reserve(n));
        widen_kernel<<<(unsigned)((n + 255) / 256), 256, 0, d.stream>>>(image, f->out64.p, n);
        CUDA_TRY(cudaGetLastError());
        ctx->stats.kernel_launches += 1;
        CUDA_TRY(cudaMemcpyAsync(out_rgb, f->out64.p, n * sizeof(double), cudaMemcpyDeviceToHost, d.stream));
        CUDA_TRY(cudaStreamSynchronize(d.stream));
        if (*f->timed_out) return fail(RC_ERR_STATE, "the frame never completed (a rank stopped publishing progress)");
    }
    return RC_OK;
}

int rc_finalize(rc_ctx* ctx, const float* d_accum, int32_t width, int32_t height, int32_t samples, float* d_rgb) {
    if (!ctx || !d_accum || !d_rgb || samples < 1) return fail(RC_ERR_INVALID, "bad finalize arguments");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    size_t n = (size_t)width * height * 3;
    finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, d.stream>>>(d_accum, d_rgb, n, 1.0f / (float)samples);
    CUDA_TRY(cudaGetLastError());
    return RC_OK;
}

int rc_render(rc_ctx* ctx, const rc_params* p, double* out_rgb, const volatile int32_t* cancel) {
    if (!ctx || !out_rgb) return fail(RC_ERR_INVALID, "ctx or out_rgb is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (!ctx->has_scene || !ctx->has_camera) return fail(RC_ERR_STATE, "upload a scene and set a camera first");
    if (cancelled(cancel)) return fail(RC_ERR_CANCELLED, "cancel flag set before the render started");
    DeviceState& d0 = ctx->devs[0];
    size_t n = (size_t)p->width * p->height * 3;
    const bool store = can_store(ctx, p);
    rc = ensure_accum(ctx, p, true, !store);
    if (rc != RC_OK) return rc;
    bool was_cancelled = false;
    rc = trace_share(ctx, p, ShareCall{d0.accum.p, cancel, store}, was_cancelled);
    if (rc != RC_OK) return rc;
    if (was_cancelled) return RC_OK;  // a cancelled render writes nothing, cpu.rs:55-62
    CUDA_TRY(cudaSetDevice(d0.device));
    CUDA_TRY(d0.out64.resize(n));
    finalize_to_f64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, d0.stream>>>(d0.accum.p, d0.out64.p, n, 1.0 / (double)p->samples);
    CUDA_TRY(cudaGetLastError());
    rc = finish_stats(ctx, p);
    if (rc != RC_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_rgb, d0.out64.p, n * sizeof(double), cudaMemcpyDeviceToHost, d0.stream));
    CUDA_TRY(cudaStreamSynchronize(d0.stream));
    return RC_OK;
}

int rc_render_adaptive(rc_ctx* ctx, const rc_params* p, const rc_adaptive* a, double* out_rgb, int32_t* out_spp, double* out_err,
                       const volatile int32_t* cancel) {
    if (!ctx || !a || !out_rgb) return fail(RC_ERR_INVALID, "ctx, adaptive or out_rgb is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (ctx->devs.size() != 1 || p->world > 1) return fail(RC_ERR_INVALID, "adaptive rendering needs a one-device context and world <= 1");
    if (p->variant != RC_VARIANT_MEGAKERNEL || p->sampler != RC_SAMPLER_DIRECT || (p->rng_rounds != 0 && p->rng_rounds != 10))
        return fail(RC_ERR_INVALID, "adaptive rendering needs the megakernel, the direct sampler and 10 Philox rounds");
    if (p->specialize == 1 && p->fixed_jitter) return fail(RC_ERR_INVALID, "specialize = 1 needs fixed_jitter = 0");
    if (a->min_samples < 2 || a->min_samples > p->samples) return fail(RC_ERR_INVALID, "min_samples must be >= 2 and <= samples");
    if (!(a->threshold >= 0.0) || !std::isfinite(a->threshold)) return fail(RC_ERR_INVALID, "threshold must be finite and >= 0");
    if (!ctx->has_scene || !ctx->has_camera) return fail(RC_ERR_STATE, "upload a scene and set a camera first");
    if (cancelled(cancel)) return fail(RC_ERR_CANCELLED, "cancel flag set before the render started");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    const size_t n_pix = (size_t)p->width * p->height, n = n_pix * 3;
    CUDA_TRY(d.ad_active.reserve(n_pix));
    CUDA_TRY(d.ad_spp.reserve(n_pix));
    CUDA_TRY(d.ad_m2.reserve(n_pix));
    CUDA_TRY(d.ad_s2.reserve(n_pix));
    CUDA_TRY(d.ad_err.reserve(n_pix));
    CUDA_TRY(d.out64.resize(n));
    // the call's start: the rounds add to one segment counter and are timed together (trace_share leaves both alone)
    CUDA_TRY(cudaEventRecord(d.ev0, d.stream));
    CUDA_TRY(cudaMemsetAsync(d.counter.p, 0, sizeof(unsigned long long), d.stream));
    rc = ensure_accum(ctx, p, true);
    if (rc != RC_OK) return rc;
    const unsigned grid = (unsigned)((n_pix + 255) / 256);
    adaptive_init_kernel<<<grid, 256, 0, d.stream>>>(d.ad_active.p, d.ad_spp.p, d.ad_s2.p, d.ad_err.p, n_pix, a->min_samples);
    CUDA_TRY(cudaGetLastError());
    uint64_t launches = 1;
    int specialized = 0;
    // every pixel still active after round r has traced the same samples, so a round is one sample range for all
    for (int lo = 0, hi = a->min_samples;; lo = hi, hi = (int)std::min(2LL * hi, (long long)p->samples)) {
        const AdaptiveRound round{d.ad_active.p, d.ad_m2.p, lo, hi};
        ShareCall call{d.accum.p, cancel};
        call.round = &round;
        bool was_cancelled = false;
        rc = trace_share(ctx, p, call, was_cancelled);
        if (rc != RC_OK) return rc;
        if (was_cancelled) return RC_OK;   // a cancelled render writes nothing, cpu.rs:55-62
        launches += ctx->stats.kernel_launches;
        specialized = ctx->stats.specialized;
        adaptive_test_kernel<<<grid, 256, 0, d.stream>>>(d.accum.p, d.ad_m2.p, d.ad_s2.p, d.ad_active.p, d.ad_spp.p, d.ad_err.p, n_pix,
                                                         p->samples, a->threshold);
        CUDA_TRY(cudaGetLastError());
        ++launches;
        if (hi == p->samples) break;
        if (cancelled(cancel)) return RC_OK;
    }
    finalize_spp_to_f64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, d.stream>>>(d.accum.p, d.ad_spp.p, d.out64.p, n);
    CUDA_TRY(cudaGetLastError());
    ++launches;
    rc = finish_stats(ctx, p);
    if (rc != RC_OK) return rc;
    std::vector<int32_t> spp_host;
    int32_t* spp = out_spp;
    if (!spp) { spp_host.resize(n_pix); spp = spp_host.data(); }
    CUDA_TRY(cudaMemcpyAsync(out_rgb, d.out64.p, n * sizeof(double), cudaMemcpyDeviceToHost, d.stream));
    CUDA_TRY(cudaMemcpyAsync(spp, d.ad_spp.p, n_pix * sizeof(int32_t), cudaMemcpyDeviceToHost, d.stream));
    if (out_err) CUDA_TRY(cudaMemcpyAsync(out_err, d.ad_err.p, n_pix * sizeof(double), cudaMemcpyDeviceToHost, d.stream));
    CUDA_TRY(cudaStreamSynchronize(d.stream));
    uint64_t samples = 0;
    for (size_t i = 0; i < n_pix; ++i) samples += (uint64_t)spp[i];
    ctx->stats.samples = samples;
    ctx->stats.kernel_launches = launches;
    ctx->stats.specialized = specialized;
    return RC_OK;
}

int rc_render_preview(rc_ctx* ctx, const rc_params* p, int32_t scale_w, int32_t scale_h, double* out_rgb,
                      const volatile int32_t* cancel) {
    if (!ctx || !out_rgb) return fail(RC_ERR_INVALID, "ctx or out_rgb is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (scale_w < 1 || scale_h < 1) return fail(RC_ERR_INVALID, "scale_w and scale_h must be >= 1");
    if (!ctx->has_scene || !ctx->has_camera) return fail(RC_ERR_STATE, "upload a scene and set a camera first");
    if (cancelled(cancel)) return fail(RC_ERR_CANCELLED, "cancel flag set before the render started");
    // the grid of scaled blocks: image.width / scale_width per tile (cpu_scaled.rs:51-52); tiles start at
    // multiples of the scale, so over the whole screen that is width / scale_w whole blocks
    rc_params q = *p;
    q.width = p->width / scale_w; q.height = p->height / scale_h;
    DeviceState& d0 = ctx->devs[0];
    const size_t n_out = (size_t)p->width * p->height;
    CUDA_TRY(cudaSetDevice(d0.device));
    CUDA_TRY(d0.out64.resize(n_out * 3));
    if (q.width < 1 || q.height < 1) {   // no whole block fits: the reference's buffer stays zero
        std::memset(out_rgb, 0, n_out * 3 * sizeof(double));
        return RC_OK;
    }
    // single traced row/column: check_params wants >= 2 only because u divides by W-1, which is the screen's here
    const bool store = can_store(ctx, &q);
    rc = ensure_accum(ctx, &q, true, !store);
    if (rc != RC_OK) return rc;
    ShareCall call{d0.accum.p, cancel, store};
    call.preview_sw = scale_w; call.preview_sh = scale_h; call.preview_w = p->width; call.preview_h = p->height;
    bool was_cancelled = false;
    rc = trace_share(ctx, &q, call, was_cancelled);
    if (rc != RC_OK) return rc;
    if (was_cancelled) return RC_OK;
    CUDA_TRY(cudaSetDevice(d0.device));
    preview_expand_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, d0.stream>>>(
        d0.accum.p, d0.out64.p, p->width, p->height, q.width, q.height, scale_w, scale_h, 1.0 / (double)p->samples);
    CUDA_TRY(cudaGetLastError());
    rc = finish_stats(ctx, &q);
    if (rc != RC_OK) return rc;
    ctx->stats.kernel_launches += 1;
    CUDA_TRY(cudaMemcpyAsync(out_rgb, d0.out64.p, n_out * 3 * sizeof(double), cudaMemcpyDeviceToHost, d0.stream));
    CUDA_TRY(cudaStreamSynchronize(d0.stream));
    return RC_OK;
}

int rc_build_lbvh(rc_ctx* ctx) {
    if (!ctx) return fail(RC_ERR_INVALID, "ctx is NULL");
    if (!ctx->has_scene) return fail(RC_ERR_STATE, "upload a scene first");
    const int n = (int)ctx->objects.size();
    if (n < 1) return fail(RC_ERR_INVALID, "the uploaded scene has no prim_aabb: nothing to build a BVH over");
    int padded = 1;
    while (padded < n) padded <<= 1;
    const int n_nodes = 2 * n - 1, np = ctx->n_prims;
    const unsigned B = 256;
    auto grid = [&](int count) { return (unsigned)((count + (int)B - 1) / (int)B); };
    for (auto& d : ctx->devs) {
        CUDA_TRY(cudaSetDevice(d.device));
        DevBuf<LbvhObject> obj;
        DevBuf<unsigned long long> keys;
        DevBuf<long long> bounds;
        DevBuf<LbvhNode> tree;
        DevBuf<int> leaf_parent, arrived, first_new, order, preorder;
        CUDA_TRY(obj.assign(ctx->objects));
        CUDA_TRY(keys.resize((size_t)padded));
        CUDA_TRY(bounds.resize(6));
        CUDA_TRY(tree.resize((size_t)(n > 1 ? n - 1 : 1)));
        CUDA_TRY(leaf_parent.resize((size_t)n));
        CUDA_TRY(arrived.resize((size_t)n));
        CUDA_TRY(first_new.resize((size_t)n));
        CUDA_TRY(order.resize((size_t)np));
        CUDA_TRY(preorder.resize((size_t)n_nodes));
        const long long init[6] = {0x7fffffffffffffffLL, 0x7fffffffffffffffLL, 0x7fffffffffffffffLL,
                                   (long long)0x8000000000000000ULL, (long long)0x8000000000000000ULL, (long long)0x8000000000000000ULL};
        CUDA_TRY(cudaMemcpyAsync(bounds.p, init, sizeof(init), cudaMemcpyHostToDevice, d.stream));
        CUDA_TRY(cudaMemsetAsync(arrived.p, 0, (size_t)n * sizeof(int), d.stream));
        lbvh_bounds<<<grid(n), B, 0, d.stream>>>(obj.p, n, bounds.p);
        lbvh_morton<<<grid(padded), B, 0, d.stream>>>(obj.p, n, padded, bounds.p, keys.p);
        if (padded <= LBVH_SMEM_KEYS) {
            const size_t smem = (size_t)padded * sizeof(unsigned long long);
            if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(lbvh_sort_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            lbvh_sort_smem<<<1, 1024, smem, d.stream>>>(keys.p, padded);
        } else {
            for (int k = 2; k <= padded; k <<= 1)
                for (int j = k >> 1; j > 0; j >>= 1) lbvh_sort_step<<<grid(padded), B, 0, d.stream>>>(keys.p, padded, j, k);
        }
        if (n > 1) {
            lbvh_topology<<<grid(n - 1), B, 0, d.stream>>>(keys.p, n, tree.p, leaf_parent.p);
            lbvh_fit<<<grid(n), B, 0, d.stream>>>(keys.p, obj.p, n, tree.p, leaf_parent.p, arrived.p);
        }
        lbvh_prim_offsets<<<1, 1024, 0, d.stream>>>(keys.p, obj.p, n, first_new.p);
        lbvh_prim_order<<<grid(n), B, 0, d.stream>>>(keys.p, obj.p, n, first_new.p, order.p);
        DevBuf<DevNode> nodes;
        DevBuf<DevNodeD> nodes_d;
        CUDA_TRY(nodes.resize((size_t)n_nodes));
        CUDA_TRY(nodes_d.resize((size_t)n_nodes));
        lbvh_emit<<<grid(n_nodes), B, 0, d.stream>>>(keys.p, obj.p, n, tree.p, leaf_parent.p, first_new.p, nodes.p, nodes_d.p, preorder.p);
        // primitive tables into the tree's depth-first leaf order
        DevBuf<DevPrim> prims;
        DevBuf<DevPrimD> prims_d;
        DevBuf<int> kind, inst;
        DevBuf<uint32_t> id;
        CUDA_TRY(prims.resize((size_t)np)); CUDA_TRY(prims_d.resize((size_t)np)); CUDA_TRY(kind.resize((size_t)np));
        CUDA_TRY(inst.resize((size_t)np)); CUDA_TRY(id.resize((size_t)np));
        lbvh_gather<<<grid(np), B, 0, d.stream>>>(d.prims.p, prims.p, order.p, np);
        lbvh_gather<<<grid(np), B, 0, d.stream>>>(d.prims_d.p, prims_d.p, order.p, np);
        lbvh_gather<<<grid(np), B, 0, d.stream>>>(d.prim_kind.p, kind.p, order.p, np);
        lbvh_gather<<<grid(np), B, 0, d.stream>>>(d.prim_inst.p, inst.p, order.p, np);
        lbvh_gather<<<grid(np), B, 0, d.stream>>>(d.prim_id.p, id.p, order.p, np);
        CUDA_TRY(cudaGetLastError());
        if (&d == &ctx->devs[0]) {   // the composed permutation and the object table follow the primitives
            std::vector<int> ord((size_t)np);
            CUDA_TRY(cudaMemcpyAsync(ord.data(), order.p, (size_t)np * sizeof(int), cudaMemcpyDeviceToHost, d.stream));
            CUDA_TRY(cudaStreamSynchronize(d.stream));
            if (ctx->prim_order.empty()) ctx->prim_order = ord;
            else { std::vector<int> c((size_t)np); for (int i = 0; i < np; ++i) c[i] = ctx->prim_order[ord[i]]; ctx->prim_order = c; }
            std::vector<LbvhObject> moved;
            std::vector<int> seen((size_t)np, -1);
            for (int i = 0; i < np; ++i) seen[ord[i]] = i;
            for (const LbvhObject& o : ctx->objects) { LbvhObject q = o; q.first = seen[o.first]; moved.push_back(q); }
            std::sort(moved.begin(), moved.end(), [](const LbvhObject& a, const LbvhObject& b) { return a.first < b.first; });
            ctx->objects_next = moved;
        }
        CUDA_TRY(cudaStreamSynchronize(d.stream));
        std::swap(d.prims, prims); std::swap(d.prims_d, prims_d); std::swap(d.prim_kind, kind); std::swap(d.prim_inst, inst); std::swap(d.prim_id, id);
        std::swap(d.nodes, nodes); std::swap(d.nodes_d, nodes_d);
        prims.release(); prims_d.release(); kind.release(); inst.release(); id.release(); nodes.release(); nodes_d.release();
        obj.release(); keys.release(); bounds.release(); tree.release(); leaf_parent.release(); arrived.release(); first_new.release();
        order.release(); preorder.release();
    }
    ctx->objects = ctx->objects_next;
    ctx->kp.n_nodes = n_nodes;
    ctx->aov.n_nodes = n_nodes;
    // the traversal modes: shared memory when nodes + primitives (+ Perlin tables) fit, global memory otherwise
    const size_t perlin_bytes = (size_t)ctx->n_perlin * (256 * 16 + 768);
    const size_t bvh_bytes = (size_t)n_nodes * sizeof(DevNode) + (size_t)np * sizeof(DevPrim);
    ctx->mode = bvh_bytes + perlin_bytes <= RC_SMEM_STAGE_LIMIT ? RT_MODE_SMEM_BVH : RT_MODE_GLOBAL_BVH;
    ctx->smem_bytes = perlin_bytes + (ctx->mode == RT_MODE_SMEM_BVH ? bvh_bytes : 0);
    ctx->spec_source.clear();
    ctx->spec_source_moments.clear();
    ctx->lbvh = true;
    CUDA_TRY(cudaSetDevice(ctx->devs[0].device));
    return RC_OK;
}

int rc_get_bvh(rc_ctx* ctx, rc_bvh_node* nodes, int32_t node_capacity, int32_t* prim_order, int32_t prim_capacity) {
    if (!ctx) return fail(RC_ERR_INVALID, "ctx is NULL");
    if (!ctx->has_scene) return fail(RC_ERR_STATE, "upload a scene first");
    const int n_nodes = ctx->kp.n_nodes, np = ctx->n_prims;
    if (nodes && node_capacity >= n_nodes && n_nodes > 0) {
        DeviceState& d = ctx->devs[0];
        CUDA_TRY(cudaSetDevice(d.device));
        std::vector<DevNodeD> h((size_t)n_nodes);
        CUDA_TRY(cudaMemcpy(h.data(), d.nodes_d.p, (size_t)n_nodes * sizeof(DevNodeD), cudaMemcpyDeviceToHost));
        for (int i = 0; i < n_nodes; ++i) {
            for (int a = 0; a < 3; ++a) { nodes[i].bmin[a] = h[i].lo[a]; nodes[i].bmax[a] = h[i].hi[a]; }
            if (h[i].leaf >= 0) { nodes[i].left = ~(h[i].leaf & 0xffffff); nodes[i].right = h[i].leaf >> 24; }
            else { nodes[i].left = i + 1; nodes[i].right = h[i + 1].skip; }   // right child = first node after the left subtree
        }
    }
    if (prim_order && prim_capacity >= np)
        for (int i = 0; i < np; ++i) prim_order[i] = ctx->prim_order.empty() ? i : ctx->prim_order[i];
    return n_nodes;
}

int rc_postprocess(rc_ctx* ctx, const rc_tone_map* tm, const double* rgb, int32_t width, int32_t height,
                   uint8_t* rgba, double* rgb_out) {
    if (!ctx || !tm || !rgb || width < 1 || height < 1) return fail(RC_ERR_INVALID, "bad postprocess arguments");
    if (tm->type < 0 || tm->type > 3) return fail(RC_ERR_INVALID, "unknown tone map");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    size_t np = (size_t)width * height;
    DevBuf<double>& in = d.pp_in;          // scratch kept between calls (one tone-mapped frame per render)
    DevBuf<double>& mapped = d.pp_mapped;
    DevBuf<uint8_t>& q = d.pp_rgba;
    CUDA_TRY(in.reserve(np * 3));
    CUDA_TRY(mapped.reserve(np * 3));
    CUDA_TRY(q.reserve(np * 4));
    ToneParams tp;
    std::memset(&tp, 0, sizeof(tp));
    tp.type = tm->type;
    tp.max_white_pow = tm->max_white * tm->max_white;  // reinhard.rs:10-14
    tp.A = tm->hable[0]; tp.B = tm->hable[1]; tp.C = tm->hable[2]; tp.D = tm->hable[3]; tp.E = tm->hable[4]; tp.F = tm->hable[5];
    tp.toe_angle = tp.E / tp.F;  // hable.rs:43-50
    tp.exposure_bias = tm->exposure_bias;
    {
        double x = tm->linear_white_point;
        tp.white_scale = 1.0 / (((x * (tp.A * x + tp.C * tp.B) + tp.D * tp.E) / (x * (tp.A * x + tp.B) + tp.D * tp.F)) - tp.toe_angle);
    }
    for (int i = 0; i < 9; ++i) { tp.aces_in[i] = tm->aces_in[i]; tp.aces_out[i] = tm->aces_out[i]; }
    cudaError_t e = cudaMemcpyAsync(in.p, rgb, np * 3 * sizeof(double), cudaMemcpyHostToDevice, d.stream);
    if (e == cudaSuccess) {
        postprocess_kernel<<<(unsigned)((np + 255) / 256), 256, 0, d.stream>>>(tp, in.p, np, q.p, mapped.p);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && rgba) e = cudaMemcpyAsync(rgba, q.p, np * 4, cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess && rgb_out) e = cudaMemcpyAsync(rgb_out, mapped.p, np * 3 * sizeof(double), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, std::string("postprocess: ") + cudaGetErrorString(e));
    return RC_OK;
}

int rc_primary_aov(rc_ctx* ctx, const rc_params* p, int32_t precision, uint32_t* id, double* t, double* normal, double* point) {
    if (!ctx) return fail(RC_ERR_INVALID, "ctx is NULL");
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (precision != 32 && precision != 64) return fail(RC_ERR_INVALID, "precision must be 32 or 64");
    if (!ctx->has_scene || !ctx->has_camera) return fail(RC_ERR_STATE, "upload a scene and set a camera first");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    size_t np = (size_t)p->width * p->height;
    DevBuf<uint32_t> d_id;
    DevBuf<double> d_t, d_n, d_p;
    CUDA_TRY(d_id.resize(np)); CUDA_TRY(d_t.resize(np)); CUDA_TRY(d_n.resize(np * 3)); CUDA_TRY(d_p.resize(np * 3));
    if (precision == 32) {
        KParams kp = ctx->kp;
        kp.prims = d.prims.p; kp.prims_lin = d.prims_lin.p; kp.nodes = d.nodes.p; kp.textures = d.textures.p;
        kp.instances = d.instances.p;
        kp.perlin = d.perlin.p; kp.perlin_perm = d.perm.p;
        kp.segment_counter = nullptr;
        rc_params q = *p;
        q.fixed_jitter = 1; q.split = RC_SPLIT_TILES;
        partition(kp, &q, 0, 1);
        kp.n_perlin = 0;  // no texture work in the AOV: skip the Perlin staging
        size_t smem = ctx->smem_bytes - (size_t)ctx->kp.n_perlin * (256 * 16 + 768);
        switch (ctx->mode) {
        case RT_MODE_CONST_LINEAR:
            primary_aov_kernel<RT_MODE_CONST_LINEAR><<<kp.n_tiles, RT_BLOCK, smem, d.stream>>>(kp, d_id.p, d_t.p, d_n.p, d_p.p);
            break;
        case RT_MODE_SMEM_BVH:
            rc = set_smem(primary_aov_kernel<RT_MODE_SMEM_BVH>, smem);
            if (rc != RC_OK) return rc;
            primary_aov_kernel<RT_MODE_SMEM_BVH><<<kp.n_tiles, RT_BLOCK, smem, d.stream>>>(kp, d_id.p, d_t.p, d_n.p, d_p.p);
            break;
        case RT_MODE_GLOBAL_BVH:
            primary_aov_kernel<RT_MODE_GLOBAL_BVH><<<kp.n_tiles, RT_BLOCK, smem, d.stream>>>(kp, d_id.p, d_t.p, d_n.p, d_p.p);
            break;
        default:
            rc = set_smem(primary_aov_kernel<RT_MODE_SMEM_LINEAR>, smem);
            if (rc != RC_OK) return rc;
            primary_aov_kernel<RT_MODE_SMEM_LINEAR><<<kp.n_tiles, RT_BLOCK, smem, d.stream>>>(kp, d_id.p, d_t.p, d_n.p, d_p.p);
        }
    } else {
        AovParamsD ap = ctx->aov;
        ap.width = p->width; ap.height = p->height;
        ap.prims = d.prims_d.p; ap.prim_kind = d.prim_kind.p; ap.prim_id = d.prim_id.p; ap.nodes = d.nodes_d.p;
        ap.prim_inst = d.prim_inst.p; ap.instances = d.instances_d.p;
        dim3 block(16, 8), grid((p->width + 15) / 16, (p->height + 7) / 8);
        primary_aov_kernel_f64<<<grid, block, 0, d.stream>>>(ap, d_id.p, d_t.p, d_n.p, d_p.p);
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && id) e = cudaMemcpyAsync(id, d_id.p, np * sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess && t) e = cudaMemcpyAsync(t, d_t.p, np * sizeof(double), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess && normal) e = cudaMemcpyAsync(normal, d_n.p, np * 3 * sizeof(double), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess && point) e = cudaMemcpyAsync(point, d_p.p, np * 3 * sizeof(double), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
    d_id.release(); d_t.release(); d_n.release(); d_p.release();
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, std::string("primary_aov: ") + cudaGetErrorString(e));
    return RC_OK;
}

int rc_partition(const rc_params* p, int32_t part, int32_t parts, int32_t out[8]) {
    int rc = check_params(p);
    if (rc != RC_OK) return rc;
    if (!out || parts < 1 || part < 0 || part >= parts) return fail(RC_ERR_INVALID, "bad partition arguments");
    KParams kp;
    std::memset(&kp, 0, sizeof(kp));
    partition(kp, p, part, parts);
    out[0] = kp.tile_first; out[1] = kp.tile_stride; out[2] = kp.n_tiles; out[3] = kp.tiles_x;
    out[4] = kp.tile_w; out[5] = kp.tile_h; out[6] = kp.s_begin; out[7] = kp.s_end;
    return RC_OK;
}

int rc_fp32_peak(rc_ctx* ctx, double* tflops, double* lane_ginstr_per_s) {
    if (!ctx) return fail(RC_ERR_INVALID, "ctx is NULL");
    DeviceState& d = ctx->devs[0];
    CUDA_TRY(cudaSetDevice(d.device));
    DevBuf<float> out;
    const int blocks = d.sm_count * 8, threads = 256, iters = 4096;
    CUDA_TRY(out.resize((size_t)blocks * threads));
    double best_ms = 1e30;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_TRY(cudaEventRecord(d.ev0, d.stream));
        fma_peak_kernel<<<blocks, threads, 0, d.stream>>>(out.p, iters, 0.999f, 0.001f);
        CUDA_TRY(cudaEventRecord(d.ev1, d.stream));
        CUDA_TRY(cudaEventSynchronize(d.ev1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, d.ev0, d.ev1));
        if (rep > 0 && ms < best_ms) best_ms = ms;
    }
    out.release();
    double fmas = (double)blocks * threads * (double)iters * 64.0;
    if (lane_ginstr_per_s) *lane_ginstr_per_s = fmas / (best_ms * 1e-3) / 1e9;
    if (tflops) *tflops = 2.0 * fmas / (best_ms * 1e-3) / 1e12;
    return RC_OK;
}

int64_t rc_spec_source(const rc_scene* scene, char* out, int64_t capacity) {
    if (validate_scene(scene) != RC_OK) return -1;
    HostTables t;
    build_tables(scene, t);
    if (t.mode == RT_MODE_SMEM_LINEAR) return fail(RC_ERR_INVALID, "a node-less scene beyond the constant table has no specialised kernel (it gets a BVH at upload)");
    // host-only tooling: no camera has been set here, RC_SPEC_CAMERA="x,y,z" supplies the pinhole position
    // the generator checks wall pairs against (tools/spec_sass.py passes the scene's camera)
    if (const char* e = std::getenv("RC_SPEC_CAMERA")) {
        float x = 0.f, y = 0.f, z = 0.f;
        if (std::sscanf(e, "%f,%f,%f", &x, &y, &z) == 3) { t.kp.cam.origin.x = x; t.kp.cam.origin.y = y; t.kp.cam.origin.z = z; }
    }
    std::string src = spec_generate(t.kp, t.has_textures, t.mats_mask, t.mode, t.prims_mask, !t.instances.empty());
    if (out && capacity > 0) {
        size_t n = src.size() < (size_t)capacity - 1 ? src.size() : (size_t)capacity - 1;
        std::memcpy(out, src.data(), n);
        out[n] = '\0';
    }
    return (int64_t)src.size();
}

int rc_get_stats(rc_ctx* ctx, rc_stats* out) {
    if (!ctx || !out) return fail(RC_ERR_INVALID, "ctx or out is NULL");
    int rc = resolve_stats(ctx);
    if (rc != RC_OK) return rc;
    *out = ctx->stats;
    return RC_OK;
}

}  // extern "C"
#pragma GCC visibility pop
