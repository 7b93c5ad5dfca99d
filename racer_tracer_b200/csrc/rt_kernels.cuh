// rt_kernels.cuh — the kernels of the render path.
//
//   megakernel_render   one thread per pixel, loops over that pixel's samples
//                       with path regeneration; path state lives in registers
//   primary_aov_kernel  one ray per pixel, same ray-gen and closest hit
//   finalize_kernel     Vec3::scale_sqrt (src/vec3.rs:119-125)
//   postprocess_kernel  tone map + RGBA quantise (src/tone_map/*.rs,
//                       src/image_action/png.rs:21-31)
//
// The wavefront kernels live in rt_wavefront.cuh.
#pragma once
#include "rt_scene.cuh"

#define RT_TILE_W 16
#define RT_TILE_H 8
#define RT_BLOCK 128

#define RT_MODE_CONST_LINEAR 0   // primitives in the constant bank, linear loop
#define RT_MODE_SMEM_BVH 1       // nodes + primitives staged in shared memory
#define RT_MODE_GLOBAL_BVH 2     // nodes + primitives read from global memory
#define RT_MODE_SMEM_LINEAR 3    // primitives staged in shared memory, linear loop

// ---------------------------------------------------------------------------
// Shared-memory staging of the scene tables (coalesced 16-byte copies).
// Layout of the dynamic shared segment: [nodes][prims][perlin grads][perms]; scene_staging (rc_api.cu) sizes it
// ---------------------------------------------------------------------------
struct SmemLayout {
    const DevNode* nodes;
    const DevPrim* prims;
    const float4* perlin;
    const uint8_t* perm;
};

template <int MODE>
RT_D SmemLayout stage_scene(const KParams& P, unsigned char* smem) {
    SmemLayout L;
    L.nodes = P.nodes; L.prims = P.prims; L.perlin = P.perlin; L.perm = P.perlin_perm;
    float4* dst = reinterpret_cast<float4*>(smem);
    if (MODE == RT_MODE_SMEM_BVH) {
        const float4* src = reinterpret_cast<const float4*>(P.nodes);
        for (int i = threadIdx.x; i < P.n_nodes * 2; i += blockDim.x) dst[i] = __ldg(src + i);
        L.nodes = reinterpret_cast<const DevNode*>(dst);
        dst += P.n_nodes * 2;
    }
    if (MODE != RT_MODE_GLOBAL_BVH) {
        // the constant-bank mode stages the (type-sorted) table too: its intersection loops read
        // the kernel parameters through uniform indices, the hit record and the shading read
        // this copy through per-lane indices
        const float4* src = reinterpret_cast<const float4*>(MODE == RT_MODE_SMEM_BVH ? P.prims : P.prims_lin);
        for (int i = threadIdx.x; i < P.n_prims * 4; i += blockDim.x) dst[i] = __ldg(src + i);
        L.prims = reinterpret_cast<const DevPrim*>(dst);
        dst += P.n_prims * 4;
    }
    if (P.n_perlin > 0) {
        for (int i = threadIdx.x; i < P.n_perlin * 256; i += blockDim.x) dst[i] = __ldg(P.perlin + i);
        L.perlin = dst;
        dst += P.n_perlin * 256;
        const uint32_t* ps = reinterpret_cast<const uint32_t*>(P.perlin_perm);
        uint32_t* pd = reinterpret_cast<uint32_t*>(dst);
        for (int i = threadIdx.x; i < P.n_perlin * 192; i += blockDim.x) pd[i] = __ldg(ps + i);
        L.perm = reinterpret_cast<const uint8_t*>(pd);
    }
    __syncthreads();
    return L;
}

// Compile-time knowledge about the scene.  The precompiled kernels know nothing (all material
// kinds possible, background and lens decided at run time); a scene-specialised translation
// unit (rc_spec.cuh, NVRTC) defines these before including this header, together with
// spec_closest_hit(), the closest-hit with every primitive constant compiled in.
#ifndef RT_SPEC_MATS
#define RT_SPEC_MATS 0xF      /* bit m set: material kind m occurs in the scene */
#endif
#define RT_HAS_MAT(m) ((RT_SPEC_MATS >> (m)) & 1)
#ifndef RT_HAS_MOTION
#define RT_HAS_MOTION 1     /* a scene-specialised kernel sets 0 when no sphere moves */
#endif
#ifndef RT_FIXED_JITTER
#define RT_FIXED_JITTER(P) ((P).fixed_jitter)   /* a scene-specialised kernel is never launched with fixed jitter: 0 there */
#endif
#ifndef RT_HAS_LENS
#define RT_HAS_LENS 1       /* ... and 0 when the camera it was compiled for is a pinhole (lens_radius == 0) */
#endif

template <int MODE, class Scene>
RT_D int closest_hit(const KParams& P, const Scene& S, const RayT<float>& r, int last_prim, float& t, const TexCtx& X = TexCtx()) {
#ifdef RT_SPECIALIZED
    if constexpr (MODE == RT_MODE_CONST_LINEAR) return spec_closest_hit(r, last_prim, t, X);
#else
    if constexpr (MODE == RT_MODE_CONST_LINEAR) return closest_hit_linear<true>(P, S, r, last_prim, t);
#endif
    else if constexpr (MODE == RT_MODE_SMEM_LINEAR) return closest_hit_linear<false>(P, S, r, last_prim, t);
    else return closest_hit_bvh(S, P.n_nodes, r, last_prim, t);
}

// ---------------------------------------------------------------------------
// Ray generation: src/renderer/cpu.rs:35-40 + Camera::get_ray (camera.rs:326-337)
// ---------------------------------------------------------------------------
struct PixelCtx {
    vec3f dir0;        // upper_left_corner + u*horizontal - origin (fixed per pixel, Q1) - (row / (H-1)) * vertical:
                       // the direction of the pixel's ray with v jitter 0
    uint32_t pixel;
    int px, py;
};

template <int ROUNDS>
RT_D PixelCtx pixel_setup(const KParams& P, int px, int py) {
    PixelCtx c;
    c.px = px; c.py = py;
    c.pixel = (uint32_t)(py * P.width + px);
    float ujit = 0.5f;
    if (!RT_FIXED_JITTER(P)) ujit = u24(philox2x32_ks<ROUNDS>(c.pixel, rt_ctr1(0u, 0u, RT_TAG_PIXEL), P.ks).x);
    float u = ((float)(px * P.px_scale_x) + ujit) / P.wm1;  // once per pixel, cpu.rs:35-36 (cpu_scaled.rs:55-56)
    // cam.upper_left_corner holds (upper_left_corner - origin), formed in f64 on the host
    c.dir0 = P.cam.upper_left_corner + u * P.cam.horizontal;
    c.dir0 = c.dir0 - ((float)(py * P.px_scale_y) * P.inv_hm1) * P.cam.vertical;   // the row term of v (cpu.rs:39-40)
    return c;
}

// Primary ray of one sample.  `w` = the sample's start block (x -> v jitter).
template <int SAMPLER, int ROUNDS>
RT_D void camera_ray(const KParams& P, const PixelCtx& c, uint32_t sample, float vjit16, vec3f& o, vec3f& d, float& time) {
    // cpu.rs:39-40 (cpu_scaled.rs:59-60): v = (row + jitter) / (H - 1), direction = .. - v * vertical.  The row's share
    // is in c.dir0 (once per pixel); the sample's share is vjit16 — the v jitter times 65536, an integer — times
    // P.vstep = vertical / ((H - 1) * 65536), formed in f64 on the host: three multiply-adds per primary ray.
    d = mk3(fmaf(-vjit16, P.vstep.x, c.dir0.x), fmaf(-vjit16, P.vstep.y, c.dir0.y), fmaf(-vjit16, P.vstep.z, c.dir0.z));
    o = P.cam.origin;
#ifdef RT_SPEC_SHIFT
    o = o - RT_SPEC_SHIFT;   // scene-specialised kernels may trace relative to another origin (rc_spec.cuh)
#endif
    time = P.cam.time_a;
    if (RT_HAS_MOTION && P.has_motion && !RT_FIXED_JITTER(P)) {
        // camera.rs:335: random_double_range(time_a, time_b); the draw is the spare 16 bits of LENS block 0
        const uint2 w = philox2x32_ks<ROUNDS>(c.pixel, rt_ctr1(sample, 0u, RT_TAG_LENS), P.ks);
        time = fmaf(P.cam.time_b - P.cam.time_a, u16lo(w), P.cam.time_a);
    }
    if (RT_HAS_LENS && P.lens_enabled && !RT_FIXED_JITTER(P)) {  // camera.rs:327-328; skipped when lens_radius == 0 (offset = 0)
        float dx, dy;
        if (SAMPLER == 1) {  // random_in_unit_disk, util.rs:25-39
            for (uint32_t j = 1;; ++j) {
                uint2 w = philox2x32_ks<ROUNDS>(c.pixel | (j << 24), rt_ctr1(sample, 0u, RT_TAG_LENS), P.ks);
                dx = 2.0f * u24(w.x) - 1.0f; dy = 2.0f * u24(w.y) - 1.0f;
                if (dx * dx + dy * dy >= 1.0f) continue;
                break;
            }
        } else {
            uint2 w = philox2x32_ks<ROUNDS>(c.pixel, rt_ctr1(sample, 0u, RT_TAG_LENS), P.ks);   // the same block as the time's: CSE
            float r = fast_sqrt(u24(w.x)), s, cs;
            fast_sincos_2pi(u24(w.y), s, cs);
            dx = r * cs; dy = r * s;
        }
        vec3f offset = (P.cam.lens_radius * dx) * P.cam.right + (P.cam.lens_radius * dy) * P.cam.up;
        o = o + offset;
        d = d - offset;
    }
}

// ---------------------------------------------------------------------------
// Tile culling.  With a pinhole camera every primary ray of a tile leaves the same point inside the frustum
// spanned by the tile's corner rays (jitter included).  A primitive (or an instanced object's cull box) that
// lies entirely outside one of the four side planes cannot be hit by any of them; if that holds for EVERY
// primitive, each sample of the tile is one segment that ends in the background, and the CTA adds the
// background radiance sample by sample (same order, same values as the general loop: bit-identical sums)
// without intersecting anything.  Conservative by construction (bounding spheres / corner tests with a
// margin); half of the Cornell frame and most of the clown frame are such tiles.
// Returns true if something may be hit.  All threads of the CTA must call it.
// ---------------------------------------------------------------------------
RT_D bool tile_may_hit(const KParams& P, const DevPrim* prims, int tx, int ty) {
    // corner directions: u in [x0, x1 + 1) / (W - 1), v in [y0, y1 + 1) / (H - 1), padded by a hundredth of a pixel
    const float u0 = ((float)(tx * RT_TILE_W * P.px_scale_x) - 0.01f) / P.wm1;
    const float u1 = ((float)((tx * RT_TILE_W + RT_TILE_W - 1) * P.px_scale_x) + 1.01f) / P.wm1;
    const float v0 = ((float)(ty * RT_TILE_H * P.px_scale_y) - 0.01f) * P.inv_hm1;
    const float v1 = ((float)((ty * RT_TILE_H + RT_TILE_H - 1) * P.px_scale_y) + 1.01f) * P.inv_hm1;
    const vec3f c = P.cam.upper_left_corner, hx = P.cam.horizontal, vy = P.cam.vertical;
    const vec3f d00 = c + u0 * hx - v0 * vy, d10 = c + u1 * hx - v0 * vy, d01 = c + u0 * hx - v1 * vy, d11 = c + u1 * hx - v1 * vy;
    const vec3f dc = c + (0.5f * (u0 + u1)) * hx - (0.5f * (v0 + v1)) * vy;
    auto cross3 = [](vec3f a, vec3f b) { return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); };
    vec3f n[4] = {cross3(d00, d01), cross3(d10, d11), cross3(d00, d10), cross3(d01, d11)};   // left, right, top, bottom
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        n[k] = unit_vector(n[k]);
        if (dot(n[k], dc) < 0.0f) n[k] = -n[k];   // inward
    }
    const vec3f o = P.cam.origin;
    // is the point set {q_j} (+ radius) entirely outside one side plane?
    auto outside = [&](const vec3f* q, int nq, float radius) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            bool all_out = true;
            for (int j = 0; j < nq; ++j) {
                const vec3f rel = q[j] - o;
                const float margin = radius + 1e-5f * (fabsf(rel.x) + fabsf(rel.y) + fabsf(rel.z)) + 1e-6f;
                if (dot(n[k], rel) >= -margin) all_out = false;
            }
            if (all_out) return true;
        }
        return false;
    };
    bool may = false;
    for (int i = threadIdx.x; i < P.n_prims; i += blockDim.x) {
        const float4 a = prims[i].a, b = prims[i].b;
        if (kinds_inst(b.z) >= 0) continue;               // instanced: decided by the object's cull box below
        const int type = kinds_prim(b.z);
        if (RT_IS_SPHERE(type)) {
            const vec3f ctr = mk3(a.x, a.y, a.z);
            if (!outside(&ctr, 1, fabsf(a.w))) may = true;
        } else {
            vec3f q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float pa = (j & 1) ? a.y : a.x, pb = (j & 2) ? a.w : a.z;
                q[j] = type == RT_PRIM_XY ? mk3(pa, pb, b.x) : (type == RT_PRIM_XZ ? mk3(pa, b.x, pb) : mk3(b.x, pa, pb));
            }
            if (!outside(q, 4, 0.0f)) may = true;
        }
    }
    for (int k = threadIdx.x; k < P.n_cobj; k += blockDim.x) {
        const float4 lo = P.cobj_lo[k], hi = P.cobj_hi[k];
        vec3f q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) q[j] = mk3((j & 1) ? hi.x : lo.x, (j & 2) ? hi.y : lo.y, (j & 4) ? hi.z : lo.z);
        if (!outside(q, 8, 0.0f)) may = true;
    }
    return __syncthreads_or(may ? 1 : 0) != 0;
}

// ---------------------------------------------------------------------------
// Shade one hit: emission + scatter (src/renderer.rs:59-69, src/material/*.rs).
// Returns true if the path continues with (o, d) and throughput T updated;
// `emit` receives the emitted radiance.
// ---------------------------------------------------------------------------
template <int SAMPLER, int ROUNDS, bool TEX, class Scene>
RT_D bool shade_hit(const KParams& P, const TexCtx& X, const Scene& S, const RngCtx& R, int prim,
                    const RayT<float>& r, float t, uint32_t bounce, uint2 rnd, vec3f& o, vec3f& d,
                    vec3f& T, vec3f& emit) {
    Hit h = make_hit(S, prim, r, t, X.k_two);
    // The next segment starts at the hit point.  Assigned here, unconditionally: a path that ends below never reads
    // its origin again, and this way the point is formed in the origin's registers instead of being copied into them
    // by the surviving lanes (`r` holds its own copy of the old origin).
    o = h.p;
    float4 pb = S.pb(prim), pc = S.pc(prim);
    // the material kind as a float (n.w of the table): one float compare instead of mask + integer compare
    const float mat = S.pn(prim).w;
    vec3f col = mk3(pc.x, pc.y, pc.z);
    if (TEX) {  // compiled out for scenes whose textures are all solid colours
        if (kinds_tex(pb.z) != RT_TEX_SOLID) col = texture_value(P, X, S, __float_as_int(pb.w), prim, h);
    }
    emit = mk3(0.0f, 0.0f, 0.0f);
    if (RT_HAS_MAT(RT_MAT_LIGHT) && mat == (float)RT_MAT_LIGHT) {  // diffuse_light.rs:25-36
        emit = col;
        return false;
    }
    vec3f nd;
    if (RT_HAS_MAT(RT_MAT_LAMBERTIAN) && (mat == (float)RT_MAT_LAMBERTIAN || !(RT_HAS_MAT(RT_MAT_METAL) || RT_HAS_MAT(RT_MAT_DIELECTRIC)))) {  // lambertian.rs:25-39
        vec3f rv;
        if (SAMPLER == 1) rv = unit_vector(reject_in_unit_sphere<ROUNDS>(R, bounce));
        else rv = sphere_direct_w(rnd.x, rnd.y, X.k_phi, X.k_one);
        nd = h.n + rv;
        // near_zero, vec3.rs:127-130: all three components below 1e-8 (rv = -n; one draw in 2^24) -> the normal.
        // As arithmetic (nd + k n, k = 1 in that case: what is left of nd vanishes against the unit normal)
        // instead of three selects: the ALU pipe is the saturated one.
        const float k0 = fmaxf(fmaxf(fabsf(nd.x), fabsf(nd.y)), fabsf(nd.z)) < 1e-8f ? 1.0f : 0.0f;
        fma2_bcast(k0, h.n.x, h.n.y, nd.x, nd.y, nd.x, nd.y);
        nd.z = fmaf(k0, h.n.z, nd.z);
    } else if (RT_HAS_MAT(RT_MAT_METAL) && (mat == (float)RT_MAT_METAL || !RT_HAS_MAT(RT_MAT_DIELECTRIC))) {  // metal.rs:25-44
        vec3f rv;
        if (SAMPLER == 1) rv = reject_in_unit_sphere<ROUNDS>(R, bounce);
        else {
            float u1, u2, u3;
            u16x3(rnd, u1, u2, u3);
            rv = cbrtf(u3) * sphere_direct(u1, u2);
        }
        vec3f refl = reflect(unit_vector(r.d), h.n);
        nd = refl + pb.y * rv;
        if (dot(nd, h.n) < 0.0f) return false;
    } else {  // dialectric.rs:25-56
        float ratio = h.front_face ? fast_rcp(pb.y) : pb.y;
        vec3f ud = unit_vector(r.d);
        float cos_theta = fminf(-dot(ud, h.n), 1.0f);
        float sin_theta = fast_sqrt(fmaxf(0.0f, 1.0f - cos_theta * cos_theta));
        bool do_reflect = ratio * sin_theta > 1.0f;
        if (!do_reflect) {
            float r0 = (1.0f - ratio) * fast_rcp(1.0f + ratio);
            r0 = r0 * r0;
            float m = 1.0f - cos_theta, m2 = m * m;
            float refl = r0 + (1.0f - r0) * (m2 * m2 * m);  // powf(5), dialectric.rs:17-22
            do_reflect = refl > u24(rnd.x);
        }
        if (do_reflect) nd = reflect(ud, h.n);
        else {  // refract, vec3.rs:416-422
            vec3f perp = ratio * (ud + cos_theta * h.n);
            vec3f par = (-fast_sqrt(fabsf(1.0f - length_squared(perp)))) * h.n;
            nd = perp + par;
        }
        col = mk3(1.0f, 1.0f, 1.0f);
    }
    mul2(T.x, T.y, col.x, col.y, T.x, T.y);
    T.z = T.z * col.z;
    d = nd;
    return true;
}

// ---------------------------------------------------------------------------
// Megakernel.  Block = 128 threads = one 16x8 pixel tile; each warp owns an
// 8x4 sub-tile so its lanes trace neighbouring pixels.  A lane runs all the
// samples [s_begin, s_end) of its pixel: when a path ends the lane starts the
// next sample in the same loop iteration (path regeneration), so lanes idle
// only at the very end of the tile.  Radiance sums stay in registers and are
// added to the accumulation buffer once.
// ---------------------------------------------------------------------------
#ifndef RT_MIN_BLOCKS
#define RT_MIN_BLOCKS 6
#endif
// The global-memory BVH walk waits on loads, not on registers: 9 CTAs of 56 registers (a few spilled
// values) run the Random scene 7 % faster than 6 CTAs of 80 (measured, tools/bvh_trees.py).
#ifndef RT_MIN_BLOCKS_GLOBAL_BVH
#define RT_MIN_BLOCKS_GLOBAL_BVH 9
#endif
// Background known at compile time (scene-specialised kernels): 0 unknown, 1 solid black
#ifndef RT_SPEC_BG_BLACK
#define RT_SPEC_BG_BLACK 0
#endif

// Sample stealing inside a warp (RT_STEAL).  A lane owns a pixel and its samples; paths differ in length, and
// pixels differ systematically (a pixel that looks at the light or past the geometry ends its paths after one
// segment), so the lanes of a warp run out of samples at different times — at the BENCH configuration 1.7 of
// 32 lanes idled on average (profiles/r02_megakernel_v22_1024spp_ncu.md).  A lane with nothing left takes the
// upper half of the unstarted samples of the lane that has most.  Streams are counter-based (pixel, sample,
// segment), so the samples traced are exactly the same ones; what changes is which lane adds them up: the thief
// parks what it had summed for its previous pixel in shared memory (one lane at a time, in a fixed order), and
// every pixel's total is its owner's own sum plus what was parked for it.  No pixel without a steal changes by
// a bit; the schedule is a function of the inputs only, so renders stay reproducible.
#ifndef RT_STEAL
#define RT_STEAL 1
#endif

// channel mean of the radiance a * b that a path adds where it ends
RT_D float radiance_y(const vec3f& a, const vec3f& b) { return (a.x * b.x + a.y * b.y + a.z * b.z) * (1.0f / 3.0f); }

// MOMENTS (adaptive rounds, rc_render_adaptive): only the pixels flagged in `active` trace [s_begin, s_end); every lane
// also sums y^2 of each sample it traces (y = channel mean of the sample's radiance) and the pixel's total goes to
// round_m2.  The launch is unsliced.  Without MOMENTS the kernel is exactly the plain one.  (The two per-pixel buffers
// are kernel arguments of their own, not KParams fields: a larger KParams would move every kernel argument behind it.)
template <int MODE, int SAMPLER, int ROUNDS, bool TEX, bool MOMENTS = false>
RT_D void megakernel_body(const KParams& P, float* __restrict__ accum, unsigned char* smem,
                          const uint8_t* __restrict__ active_px = nullptr, float* __restrict__ round_m2 = nullptr) {
    constexpr int PARKED = MOMENTS ? 4 : 3;   // floats parked per lane: the three sums (and the second moment)
    __shared__ float steal_parked[RT_STEAL ? PARKED * RT_BLOCK : 1];   // per lane of the CTA: sums other lanes traced for its pixel
    // A render the host may cancel (interactive.rs:236-251 always passes a cancel event): CTAs that have not started
    // when the flag is raised do nothing, so a cancelled frame drains in the time of the CTAs already running.
    if (P.cancel_flag != nullptr &&
        __syncthreads_or(threadIdx.x == 0 && *reinterpret_cast<const volatile int*>(P.cancel_flag) != 0)) return;
    bool active = true;   // (MOMENTS) this lane's pixel traces samples in this round
    if constexpr (MOMENTS) {
        // a tile without an active pixel leaves before it stages the scene: later rounds keep the ordinary tile grid
        const int tile = P.tile_first + (int)blockIdx.x * P.tile_stride;
        const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
        const int x = (tile % P.tiles_x) * RT_TILE_W + (w & 1) * 8 + (l & 7);
        const int y = (tile / P.tiles_x) * RT_TILE_H + (w >> 1) * 4 + (l >> 3);
        active = x < P.width && y < P.height && active_px[y * P.width + x] != 0;
        if (!__syncthreads_or(active ? 1 : 0)) return;
    }
    __shared__ float reg_consts[7];
    if (threadIdx.x == 0) {
        reg_consts[0] = 2.0f; reg_consts[1] = 6.283185307179586f / 16777216.0f; reg_consts[2] = 1.0f;
#ifdef RT_SPECIALIZED
        spec_reg_consts(reg_consts + 3);
#endif
    }
    SmemLayout L = stage_scene<MODE>(P, smem);    // (ends with the barrier that publishes reg_consts)
    TexCtx X; X.perlin = L.perlin; X.perm = L.perm;
    {   // volatile: a plain load would be folded back into the literal (the only value ever stored there)
        const volatile float* rc = reg_consts;
        // held in registers across the path loop, see TexCtx
        X.k_two = rc[0];
        X.k_phi = rc[1];
        X.k_one = rc[2];
#ifdef RT_SPECIALIZED
#pragma unroll
        for (int j = 0; j < RT_SPEC_REG_CONSTS; ++j) X.k_spec[j] = rc[3 + j];
#endif
    }

    // CTA -> (tile, slice of the sample range).  With one GPU there are thousands of tiles and
    // slices == 1; when the tiles are shared out over several GPUs each tile's samples are cut
    // into `slices` CTAs so the grid still fills the machine many times over.
    // Slice-major order with DECREASING slice lengths — halving (n/2, n/4, .., the last two equal: five slices and
    // more) or linear (weights S, S-1, .., 1): the CTAs scheduled last — the ones that form the tail of the grid — are the
    // short ones, and most of the work sits in few long CTAs.
    const int slice = P.slices > 1 ? (int)blockIdx.x / P.n_tiles : 0;
    const int tile_k = P.slices > 1 ? (int)blockIdx.x - slice * P.n_tiles : (int)blockIdx.x;
    const int tile = P.tile_first + tile_k * P.tile_stride;
    const int tx = tile % P.tiles_x, ty = tile / P.tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tx * RT_TILE_W + (warp & 1) * 8 + (lane & 7);
    const int py = ty * RT_TILE_H + (warp >> 1) * 4 + (lane >> 3);
    const bool valid = px < P.width && py < P.height;
    int s_first = P.s_begin, s_last = P.s_end;
    if (P.slices > 1 && P.slice_halving) {
        // halving lengths: n/2, n/4, ..., and the last two slices equal — boundaries n - (n >> j)
        const int n = P.s_end - P.s_begin;
        s_first = P.s_begin + (n - (n >> slice));
        s_last = slice + 1 == P.slices ? P.s_end : P.s_begin + (n - (n >> (slice + 1)));
    } else if (P.slices > 1) {
        const long long n = P.s_end - P.s_begin, S = P.slices, total = S * (S + 1) / 2;
        const long long c0 = (long long)slice * S - (long long)slice * (slice - 1) / 2;       // weights of the slices before this one
        const long long c1 = c0 + (S - slice);
        s_first = P.s_begin + (int)(n * c0 / total);
        s_last = P.s_begin + (int)(n * c1 / total);
    }

    PixelCtx pc = pixel_setup<ROUNDS>(P, valid ? px : 0, valid ? py : 0);
    RngCtx R; R.ks = P.ks; R.pixel = pc.pixel; R.sample = 0;
    const uint32_t own_pixel = pc.pixel;
    PhiloxPre ppre = philox2x32_pre(pc.pixel, P.ks);   // round 0 of every PATH block of this pixel, but for the xor with c1
    // 16-bit v jitter of the next sample this lane starts: the spare bytes of the previous sample's block 0
    uint32_t vj_bits = __byte_perm(0u, 0u, 0);
    {
        const uint2 w = philox2x32_from<ROUNDS>(ppre, rt_ctr1(rt_vjit_sample((uint32_t)s_first), 0u, RT_TAG_PATH), P.ks);
        vj_bits = __byte_perm(w.y, w.x, 0x0040);
    }
    int owner = lane;          // the lane of this warp whose pixel `sum` is being traced for
    float* const parked = steal_parked + 32 * PARKED * warp;
    if (RT_STEAL) {
        parked[lane] = 0.0f; parked[lane + 32] = 0.0f; parked[lane + 64] = 0.0f;
        if constexpr (MOMENTS) parked[lane + 96] = 0.0f;
        __syncwarp();
    }

    // Path state.  Radiance is only ever picked up where a path ENDS (escape, light, depth
    // exhaustion): lights do not scatter and nothing else emits (src/material/*.rs), so
    // ray_color's `emitted + attenuation * recurse` collapses to throughput x terminal radiance.
    vec3f sum = mk3(0.0f, 0.0f, 0.0f);
    float m2 = 0.0f;           // (MOMENTS) sum of y^2 over the samples in `sum`: one path adds radiance once, where it ends
    vec3f o = mk3(0.0f, 0.0f, 0.0f), d = o, T = o;
    const vec3f T_ONE = mk3(1.0f, 1.0f, 1.0f);
    float time = 0.0f;         // Ray::time of the path (scattered rays inherit it, lambertian.rs:36 etc.)
    int s = valid && active ? s_first : s_last;   // a pixel with nothing to trace starts idle (and may steal)
    // > 0: this lane is on a path that may still trace that many segments; 0: no path.  A float (max_depth <= 63
    // is exact): counting down and the "budget spent" weight are then FADD / FADD.SAT on the FMA pipe instead
    // of integer add + compare + select on the ALU pipe, which is the saturated one in this kernel.
    float depth_left = 0.0f;
    int last_prim = -1;
    uint32_t seg = 0;          // index of the segment about to be traced (0 = primary ray)
    uint32_t ctr1 = 0;         // Philox counter word of that segment's block: sample | seg << 24 (tag PATH = 0), kept incrementally
    unsigned sh_prims = (unsigned)__cvta_generic_to_shared(L.prims);   // (meaningful in the staged modes only)
    asm volatile("" : "+r"(sh_prims));   // opaque: kept in a register instead of being rebuilt (S2UR + 2 uniform ops) at every use
    unsigned nseg = 0;
    if (P.max_depth <= 0) {    // renderer.rs:48-56: depth 0 is white, for every sample
        const float n = (float)(s_last - s);
        sum = mk3(n, n, n);
        if constexpr (MOMENTS) m2 = n;   // y = 1
        s = s_last;
    }

    if (P.tile_cull && (MODE == RT_MODE_CONST_LINEAR || MODE == RT_MODE_SMEM_LINEAR) && P.max_depth > 0) {
        if (!tile_may_hit(P, L.prims, tx, ty)) {
            // every sample of this tile is one segment into the background (renderer.rs:78-88), T = 1
            if (valid) {
                nseg += (unsigned)(s_last - s);
#pragma unroll 1
                for (; s < s_last; ++s) {
                    if (RT_SPEC_BG_BLACK) { s = s_last; break; }
                    vec3f bg;
                    if (__float_as_int(P.bg_a.w) == 0) {   // Sky: depends on the sample's direction
                        const uint2 rnd = philox2x32_ks<ROUNDS>(pc.pixel, rt_ctr1(rt_vjit_sample((uint32_t)s), 0u, RT_TAG_PATH), P.ks);
                        const float vjit = RT_FIXED_JITTER(P) ? 32768.0f : u16lo_int(rnd);
                        camera_ray<SAMPLER, ROUNDS>(P, pc, (uint32_t)s, vjit, o, d, time);
                        bg = background_color(P, d);
                    } else bg = mk3(P.bg_a.x, P.bg_a.y, P.bg_a.z);
                    sum = mk3(fmaf(T_ONE.x, bg.x, sum.x), fmaf(T_ONE.y, bg.y, sum.y), fmaf(T_ONE.z, bg.z, sum.z));
                    if constexpr (MOMENTS) { const float y = radiance_y(T_ONE, bg); m2 = fmaf(y, y, m2); }
                }
            }
            s = s_last;
        }
    }

#ifdef RT_SPEC_SNAP_TABLE
    // The path loop of a rectangle-only scene reads the staged table's rows in another layout (and, with
    // RT_SPEC_SHIFT, in the kernel's own coordinates): rc_spec.cuh, spec_snap_row.  The tile test above read the
    // table as uploaded; every thread of the CTA passes both barriers.
    __syncthreads();
    if ((int)threadIdx.x < P.n_prims) {
        float* row = const_cast<float*>(reinterpret_cast<const float*>(L.prims + threadIdx.x));
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        float bx = 0.f, cw = 0.f;
        spec_snap_row((int)threadIdx.x, a, bx, cw);
        row[0] = a.x; row[1] = a.y; row[2] = a.z; row[3] = a.w; row[4] = bx; row[11] = cw;
    }
    __syncthreads();
#endif

    // One iteration of the path loop, for a lane that has a path or a sample to start (RT_LANE_BUSY: every loop below
    // only lets such lanes in): a lane whose path ended takes the next sample of its pixel (bookkeeping only), then
    // every lane draws its segment's block and traces one segment.  ONE body for all loops: what a sample
    // contributes must not depend on which loop traced it (ptxas contracts multiply-adds per code copy).
    auto iteration = [&]() {
        const bool fresh = depth_left == 0.0f;      // no path: then there is a sample (the lane is busy)
        if (fresh) {
            R.sample = (uint32_t)s;
            ctr1 = R.sample;
            seg = 0; last_prim = -1;
            T = mk3(1.0f, 1.0f, 1.0f);
            depth_left = (float)P.max_depth;
        }
        // (a predicated add: `s += fresh ? 1 : 0` compiled to a zeroed register, a predicated move and an add)
        asm("{\n\t.reg .pred pf;\n\tsetp.ne.s32 pf, %1, 0;\n\t@pf add.s32 %0, %0, 1;\n\t}" : "+r"(s) : "r"((int)fresh));
        if (fresh) {   // primary ray: cpu.rs:39-40, camera.rs:326-337; its v jitter came with the PREVIOUS sample's block 0
            const float vjit = RT_FIXED_JITTER(P) ? 32768.0f : (float)(unsigned short)vj_bits;
            camera_ray<SAMPLER, ROUNDS>(P, pc, R.sample, vjit, o, d, time);
        }
        // ---- the segment's random block: drawn here, by all lanes together.  Nothing before the hit record needs
        // it (the spare bytes of a sample's block 0 are the NEXT sample's v jitter, DESIGN §4), so its ten dependent
        // multiply-xor rounds are scheduled between the instructions of the closest hit instead of in front of them.
        const uint2 rnd = philox2x32_from<ROUNDS>(ppre, ctr1, P.ks);   // == philox2x32_ks(pc.pixel, rt_ctr1(R.sample, seg, RT_TAG_PATH))
        if (fresh) vj_bits = __byte_perm(rnd.y, rnd.x, 0x0040);
        RayT<float> r = make_ray(o, d, time);
        float t;
        int prim;
        if (MODE == RT_MODE_CONST_LINEAR) { ConstScene S(P, sh_prims); prim = closest_hit<MODE>(P, S, r, last_prim, t, X); }
        else { PtrScene S; S.prims = L.prims; S.nodes = L.nodes; S.inst = P.instances; S.ref_aabb = P.ref_aabb; prim = closest_hit<MODE>(P, S, r, last_prim, t, X); }
        ++nseg;
        if (prim < 0) {  // renderer.rs:78-88
            if (!RT_SPEC_BG_BLACK) {
                const vec3f bg = background_color(P, d);
                sum = mk3(fmaf(T.x, bg.x, sum.x), fmaf(T.y, bg.y, sum.y), fmaf(T.z, bg.z, sum.z));
                if constexpr (MOMENTS) { const float y = radiance_y(T, bg); m2 = fmaf(y, y, m2); }
            }
            depth_left = 0.0f;
        } else {
            ++seg;   // hit number along the path (1 = primary hit)
            ctr1 += 1u << 24;
            vec3f X_end;   // radiance that ends the path
            bool cont;
            if (MODE == RT_MODE_CONST_LINEAR) { ConstScene S(P, sh_prims); cont = shade_hit<SAMPLER, ROUNDS, TEX>(P, X, S, R, prim, r, t, seg, rnd, o, d, T, X_end); }
            else { PtrScene S; S.prims = L.prims; S.nodes = L.nodes; S.inst = P.instances; S.ref_aabb = P.ref_aabb; cont = shade_hit<SAMPLER, ROUNDS, TEX>(P, X, S, R, prim, r, t, seg, rnd, o, d, T, X_end); }
            if (!cont) {                 // absorbed (X_end = 0) or a light (X_end = emission)
                sum = sum + T * X_end;
                if constexpr (MOMENTS) { const float y = radiance_y(T, X_end); m2 = fmaf(y, y, m2); }
                depth_left = 0.0f;
            } else {
                last_prim = prim;
                // white at depth 0 (renderer.rs:48-56): sum += w T with w = 1 when the budget is spent, as arithmetic
                depth_left -= 1.0f;
                const float w = __saturatef(1.0f - depth_left);   // 1 when the budget is spent (depth_left == 0), else 0
                fma2_bcast(w, T.x, T.y, sum.x, sum.y, sum.x, sum.y);
                sum.z = fmaf(w, T.z, sum.z);
                if constexpr (MOMENTS) { const float y = radiance_y(T_ONE, T); m2 = fmaf(w, y * y, m2); }   // w is 0 or 1
            }
        }
        };
#define RT_LANE_BUSY ((depth_left != 0.0f) | (s < s_last))
    // The loops of one warp over the lanes in `m` (all of them converged here).  Hot loop: while EVERY lane is busy,
    // one iteration each — no per-lane test inside.  When some lane has run out (the warp's tail) it takes over half
    // of the unstarted samples of the lane that has most, and the hot loop resumes; when nothing is worth taking any
    // more, each lane finishes what it has and leaves (a lane that is idle then stays idle).
    auto warp_loops = [&](const unsigned m) {
        for (;;) {
            if (__all_sync(m, RT_LANE_BUSY)) {
#pragma unroll 1
                do iteration(); while (__all_sync(m, RT_LANE_BUSY));
            }
            bool stolen = false;
            if (RT_STEAL) {
                if (!__any_sync(m, RT_LANE_BUSY)) break;
                for (;;) {
                    const int rem = s_last - s;
                    const unsigned idle = __ballot_sync(m, !(RT_LANE_BUSY));
                    if (idle == 0u) break;
                    const int most = __reduce_max_sync(m, rem);
                    // a victim keeps at least half of >= 4 unstarted samples; below that the tail is left alone.  Unstarted
                    // samples only ever shrink: nothing worth taking, now or later
                    if (most < 4) break;
                    const int victim = __ffs(__ballot_sync(m, rem == most)) - 1, thief = __ffs(idle) - 1;
                    const int take = most >> 1;
                    const int v_last = __shfl_sync(m, s_last, victim), v_owner = __shfl_sync(m, owner, victim);
                    const uint32_t v_pixel = __shfl_sync(m, pc.pixel, victim);
                    const float vx = __shfl_sync(m, pc.dir0.x, victim), vy = __shfl_sync(m, pc.dir0.y, victim),
                                vz = __shfl_sync(m, pc.dir0.z, victim);
                    if (lane == victim) s_last -= take;
                    if (lane == thief) {
                        // what this lane has summed belongs to `owner`'s pixel: park it (only this lane is active here)
                        parked[owner] += sum.x; parked[owner + 32] += sum.y; parked[owner + 64] += sum.z;
                        sum = mk3(0.0f, 0.0f, 0.0f);
                        if constexpr (MOMENTS) { parked[owner + 96] += m2; m2 = 0.0f; }
                        owner = v_owner;
                        pc.pixel = v_pixel; pc.dir0 = mk3(vx, vy, vz);
                        R.pixel = v_pixel;
                        ppre = philox2x32_pre(v_pixel, P.ks);
                        s = v_last - take; s_last = v_last;
                        const uint2 w = philox2x32_from<ROUNDS>(ppre, rt_ctr1(rt_vjit_sample((uint32_t)s), 0u, RT_TAG_PATH), P.ks);
                        vj_bits = __byte_perm(w.y, w.x, 0x0040);
                    }
                    __syncwarp(m);
                    stolen = true;
                }
            }
            if (!stolen) {
                // nothing (more) to take over: every lane finishes what it has and leaves
#pragma unroll 1
                while (RT_LANE_BUSY) iteration();
                break;
            }
        }
    };
    {
        // lanes outside the image (right / bottom edge tiles of an image that is not a multiple of the tile) have no
        // pixel and take no part; a full warp — the rule — votes with the constant mask
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        if (vmask == 0xffffffffu) warp_loops(0xffffffffu);
        else if (valid) warp_loops(vmask);
        __syncwarp();
    }
#undef RT_LANE_BUSY
    if (RT_STEAL) {
        // sums still held for another lane's pixel are parked one lane at a time, in lane order; then every pixel's
        // total = what its owner summed itself (if it still owns it) + what was parked.  x + 0 = x: nothing changes
        // for a pixel nobody helped with.
        unsigned pending = __ballot_sync(0xffffffffu, owner != lane);
        while (pending) {
            const int l = __ffs(pending) - 1;
            pending &= pending - 1;
            if (lane == l) {
                parked[owner] += sum.x; parked[owner + 32] += sum.y; parked[owner + 64] += sum.z;
                if constexpr (MOMENTS) parked[owner + 96] += m2;
            }
            __syncwarp();
        }
        if (owner != lane) { sum = mk3(0.0f, 0.0f, 0.0f); m2 = 0.0f; }
        sum = mk3(sum.x + parked[lane], sum.y + parked[lane + 32], sum.z + parked[lane + 64]);
        if constexpr (MOMENTS) m2 += parked[lane + 96];
    }
    if constexpr (MOMENTS) {
        // unsliced, added to the running sums; nothing to write for a pixel outside this round
        if (valid && active) {
            float* a = accum + 3 * (size_t)own_pixel;
            a[0] += sum.x; a[1] += sum.y; a[2] += sum.z;
            round_m2[own_pixel] = m2;
        }
    } else if (P.slices > 1) {
        // partial sum of this slice; reduce_slices_kernel adds the slices in order (deterministic)
        float* a = P.slice_buf + 3 * ((size_t)slice * ((size_t)P.n_tiles * RT_BLOCK) + (size_t)tile_k * RT_BLOCK + threadIdx.x);
        a[0] = sum.x; a[1] = sum.y; a[2] = sum.z;
    } else if (valid) {
        // (possibly a peer GPU's memory: the gather of a multi-GPU tile split happens here, over NVLink)
        float* a = accum + 3 * (size_t)own_pixel;
        if (P.final_scale != 0.0f) sum = mk3(sqrtf(P.final_scale * sum.x), sqrtf(P.final_scale * sum.y), sqrtf(P.final_scale * sum.z));
        if (P.overwrite) { a[0] = sum.x; a[1] = sum.y; a[2] = sum.z; }
        else { a[0] += sum.x; a[1] += sum.y; a[2] += sum.z; }
    }
    // segment statistics: one atomic per warp
    for (int off = 16; off > 0; off >>= 1) nseg += __shfl_xor_sync(0xffffffffu, nseg, off);
    if (lane == 0 && P.segment_counter) atomicAdd(P.segment_counter, (unsigned long long)nseg);
}

#ifndef RT_SPECIALIZED
// accum[pixel] += sum over slices (in slice order) of the partial sums the sliced megakernel left
__global__ void reduce_slices_kernel(const __grid_constant__ KParams P, float* __restrict__ accum) {
    const int rank = blockIdx.x * blockDim.x + threadIdx.x;     // tile_k * 128 + thread
    if (rank >= P.n_tiles * RT_BLOCK) return;
    const int tile_k = rank / RT_BLOCK, within = rank % RT_BLOCK;
    const int tile = P.tile_first + tile_k * P.tile_stride;
    const int tx = tile % P.tiles_x, ty = tile / P.tiles_x;
    const int warp = within >> 5, lane = within & 31;
    const int px = tx * RT_TILE_W + (warp & 1) * 8 + (lane & 7);
    const int py = ty * RT_TILE_H + (warp >> 1) * 4 + (lane >> 3);
    if (px >= P.width || py >= P.height) return;
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int j = 0; j < P.slices; ++j) {
        const float* a = P.slice_buf + 3 * ((size_t)j * ((size_t)P.n_tiles * RT_BLOCK) + rank);
        sx += a[0]; sy += a[1]; sz += a[2];
    }
    float* dst = accum + 3 * ((size_t)py * P.width + px);
    if (P.final_scale != 0.0f) { sx = sqrtf(P.final_scale * sx); sy = sqrtf(P.final_scale * sy); sz = sqrtf(P.final_scale * sz); }
    if (P.overwrite) { dst[0] = sx; dst[1] = sy; dst[2] = sz; }
    else { dst[0] += sx; dst[1] += sy; dst[2] += sz; }
}

template <int MODE, int SAMPLER, int ROUNDS, bool TEX>
__global__ void __launch_bounds__(RT_BLOCK, MODE == RT_MODE_GLOBAL_BVH ? RT_MIN_BLOCKS_GLOBAL_BVH : RT_MIN_BLOCKS)
megakernel_render(const __grid_constant__ KParams P, float* __restrict__ accum) {
    extern __shared__ __align__(16) unsigned char smem[];
    megakernel_body<MODE, SAMPLER, ROUNDS, TEX>(P, accum, smem);
}

// One adaptive round (rc_render_adaptive): the megakernel with second moments, over the active pixels only
template <int MODE, bool TEX>
__global__ void __launch_bounds__(RT_BLOCK, MODE == RT_MODE_GLOBAL_BVH ? RT_MIN_BLOCKS_GLOBAL_BVH : RT_MIN_BLOCKS)
megakernel_moments(const __grid_constant__ KParams P, float* __restrict__ accum, const uint8_t* __restrict__ active,
                   float* __restrict__ round_m2) {
    extern __shared__ __align__(16) unsigned char smem[];
    megakernel_body<MODE, 0, 10, TEX, true>(P, accum, smem, active, round_m2);
}

// After an adaptive round, for every pixel that traced it: S2 += the round's sum of y^2; S1 = the channel mean of the
// radiance sums; the error estimate of sqrt(mean) (include/racer_cuda.h, rc_adaptive) decides whether the pixel stops
// or doubles its sample count, up to `max_spp`.  spp holds the samples traced so far.
__global__ void adaptive_test_kernel(const float* __restrict__ accum, const float* __restrict__ round_m2, double* __restrict__ s2,
                                     uint8_t* __restrict__ active, int* __restrict__ spp, double* __restrict__ err,
                                     size_t n_pixels, int max_spp, double threshold) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels || !active[i]) return;
    const int n = spp[i];
    const double S2 = s2[i] + (double)round_m2[i];
    const double S1 = ((double)accum[3 * i] + (double)accum[3 * i + 1] + (double)accum[3 * i + 2]) / 3.0;
    const double mu = S1 / n, se = sqrt(fmax(0.0, (S2 - S1 * S1 / n) / (n - 1)) / n);
    const double e = 0.5 * (sqrt(mu + se) - sqrt(fmax(mu - se, 0.0)));
    s2[i] = S2;
    err[i] = e;
    if (e <= threshold || n >= max_spp) active[i] = 0;
    else spp[i] = min(2 * n, max_spp);
}

__global__ void adaptive_init_kernel(uint8_t* __restrict__ active, int* __restrict__ spp, double* __restrict__ s2,
                                     double* __restrict__ err, size_t n_pixels, int n0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    active[i] = 1; spp[i] = n0; s2[i] = 0.0; err[i] = 0.0;
}


// The albedo shade_hit multiplies a path's throughput by at this hit: the texture colour for Lambertian and Metal,
// (1, 1, 1) for dielectrics and lights (rc_render_denoised's albedo guide)
template <class Scene>
RT_D vec3f hit_albedo(const KParams& P, const SmemLayout& L, const Scene& S, int prim, const Hit& h) {
    const float mat = S.pn(prim).w;
    if (mat != (float)RT_MAT_LAMBERTIAN && mat != (float)RT_MAT_METAL) return mk3(1.0f, 1.0f, 1.0f);
    const float4 pb = S.pb(prim), pc = S.pc(prim);
    if (kinds_tex(pb.z) == RT_TEX_SOLID) return mk3(pc.x, pc.y, pc.z);
    TexCtx X; X.perlin = L.perlin; X.perm = L.perm;
    return texture_value(P, X, S, __float_as_int(pb.w), prim, h);
}

// ---------------------------------------------------------------------------
// Primary-visibility AOV (RayImageData, src/renderer.rs:33-39): fixed jitter,
// one closest hit per pixel through the renderer's fp32 code.
// GUIDE: also the hit's albedo (hit_albedo; (1, 1, 1) for a miss) into `albedo`.
// ---------------------------------------------------------------------------
template <int MODE, bool GUIDE = false>
__global__ void __launch_bounds__(RT_BLOCK)
primary_aov_kernel(const __grid_constant__ KParams P, uint32_t* __restrict__ id, double* __restrict__ t_out,
                   double* __restrict__ normal, double* __restrict__ point, double* __restrict__ albedo = nullptr) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmemLayout L = stage_scene<MODE>(P, smem);
    const int tile = P.tile_first + blockIdx.x * P.tile_stride;
    const int tx = tile % P.tiles_x, ty = tile / P.tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tx * RT_TILE_W + (warp & 1) * 8 + (lane & 7);
    const int py = ty * RT_TILE_H + (warp >> 1) * 4 + (lane >> 3);
    if (px >= P.width || py >= P.height) return;
    PixelCtx pc = pixel_setup<10>(P, px, py);
    vec3f o, d;
    float time;
    camera_ray<0, 10>(P, pc, 0u, 32768.0f, o, d, time);   // fixed jitter: time = time_a
    RayT<float> r = make_ray(o, d, time);
    float t;
    int prim;
    Hit h;
    uint32_t oid = 0;
    vec3f alb = mk3(1.0f, 1.0f, 1.0f);
    if (MODE == RT_MODE_CONST_LINEAR) {
        ConstScene S(P, L.prims);
        prim = closest_hit<MODE>(P, S, r, -1, t);
        if (prim >= 0) { h = make_hit(S, prim, r, t); oid = (uint32_t)__float_as_int(S.pc(prim).w); }
        if constexpr (GUIDE) { if (prim >= 0) alb = hit_albedo(P, L, S, prim, h); }
    } else {
        PtrScene S; S.prims = L.prims; S.nodes = L.nodes; S.inst = P.instances; S.ref_aabb = P.ref_aabb;
        prim = closest_hit<MODE>(P, S, r, -1, t);
        if (prim >= 0) { h = make_hit(S, prim, r, t); oid = (uint32_t)__float_as_int(S.pc(prim).w); }
        if constexpr (GUIDE) { if (prim >= 0) alb = hit_albedo(P, L, S, prim, h); }
    }
    size_t i = pc.pixel;
    if constexpr (GUIDE) { albedo[3 * i] = alb.x; albedo[3 * i + 1] = alb.y; albedo[3 * i + 2] = alb.z; }
    if (prim < 0) {
        if (id) id[i] = 0;
        if (t_out) t_out[i] = 1.7976931348623157e308;
        if (normal) { normal[3 * i] = 0; normal[3 * i + 1] = 0; normal[3 * i + 2] = 0; }
        if (point) { point[3 * i] = 0; point[3 * i + 1] = 0; point[3 * i + 2] = 0; }
        return;
    }
    if (id) id[i] = oid;
    if (t_out) t_out[i] = (double)t;
    if (normal) { normal[3 * i] = h.n.x; normal[3 * i + 1] = h.n.y; normal[3 * i + 2] = h.n.z; }
    if (point) { point[3 * i] = h.p.x; point[3 * i + 1] = h.p.y; point[3 * i + 2] = h.p.z; }
}

// f64 primary visibility in the REFERENCE's operation order: round-to-nearest
// f64 adds / multiplies / divides with no FMA contraction, the direct sphere
// quadratic of sphere.rs:39-58, the per-axis Aabb::hit of aabb.rs:42-59 and
// the left-to-right direction sum of camera.rs:329-334.  It exists to show
// that ids (and t, normals) are bit-identical to the CPU restatement when the
// arithmetic is the reference's; the renderer itself runs the fp32 code above.
struct AovParamsD {
    DevCamera<double> cam;   // upper_left_corner is the real corner here
    int width, height, n_prims, n_nodes;
    const DevPrimD* prims;
    const int* prim_kind;    // RT_PRIM_*
    const uint32_t* prim_id;
    const DevNodeD* nodes;
    const int* prim_inst;             // -1 or index into instances
    const DevInstanceD* instances;
};

RT_D double sd_add(double a, double b) { return __dadd_rn(a, b); }
RT_D double sd_sub(double a, double b) { return __dsub_rn(a, b); }
RT_D double sd_mul(double a, double b) { return __dmul_rn(a, b); }
RT_D double sd_div(double a, double b) { return __ddiv_rn(a, b); }
RT_D double sd_dot(Vec3T<double> a, Vec3T<double> b) { return sd_add(sd_add(sd_mul(a.x, b.x), sd_mul(a.y, b.y)), sd_mul(a.z, b.z)); }
RT_D Vec3T<double> sd_sub3(Vec3T<double> a, Vec3T<double> b) { return mk3(sd_sub(a.x, b.x), sd_sub(a.y, b.y), sd_sub(a.z, b.z)); }
RT_D Vec3T<double> sd_add3(Vec3T<double> a, Vec3T<double> b) { return mk3(sd_add(a.x, b.x), sd_add(a.y, b.y), sd_add(a.z, b.z)); }
RT_D Vec3T<double> sd_scale(double s, Vec3T<double> a) { return mk3(sd_mul(s, a.x), sd_mul(s, a.y), sd_mul(s, a.z)); }

// MovingSphere::pos in reference order (moving_sphere.rs:37-39) at the fixed-jitter ray time
RT_D Vec3T<double> sphere_centre_d(const DevPrimD& p, int type, double time) {
    Vec3T<double> c = mk3(p.a[0], p.a[1], p.a[2]);
    if (type != RT_PRIM_MOVING) return c;
    const double f = sd_div(sd_sub(time, p.motion[3]), sd_sub(p.motion[4], p.motion[3]));
    return sd_add3(c, sd_scale(f, sd_sub3(mk3(p.motion[0], p.motion[1], p.motion[2]), c)));
}

// ray into an instance's space, reference order: translate.rs:32, rotate_y.rs:38-47
RT_D void to_local_d(const DevInstanceD& in, Vec3T<double>& o, Vec3T<double>& d) {
    if (in.flags & 2) o = sd_sub3(o, mk3(in.offset[0], in.offset[1], in.offset[2]));
    if (in.flags & 1) {
        const double s = in.sin_theta, c = in.cos_theta;
        const double ox = sd_sub(sd_mul(c, o.x), sd_mul(s, o.z)), oz = sd_add(sd_mul(s, o.x), sd_mul(c, o.z));
        const double dx = sd_sub(sd_mul(c, d.x), sd_mul(s, d.z)), dz = sd_add(sd_mul(s, d.x), sd_mul(c, d.z));
        o.x = ox; o.z = oz; d.x = dx; d.z = dz;
    }
}

// obj_hit in reference order; returns t or -1
RT_D double prim_test_d(const AovParamsD& P, int i, Vec3T<double> o, Vec3T<double> d, double t_min, double t_max) {
    const DevPrimD& p = P.prims[i];
    int type = P.prim_kind[i];
    const int inst = P.prim_inst[i];
    if (inst >= 0) to_local_d(P.instances[inst], o, d);
    if (RT_IS_SPHERE(type)) {  // sphere.rs:39-58, moving_sphere.rs:50-66
        Vec3T<double> oc = sd_sub3(o, sphere_centre_d(p, type, P.cam.time_a));
        double a = sd_dot(d, d), half_b = sd_dot(oc, d);
        double c = sd_sub(sd_dot(oc, oc), sd_mul(p.a[3], p.a[3]));
        double disc = sd_sub(sd_mul(half_b, half_b), sd_mul(a, c));
        if (disc < 0.0) return -1.0;
        double sqrtd = __dsqrt_rn(disc);
        double root = sd_div(sd_sub(-half_b, sqrtd), a);
        if (root < t_min || t_max < root) {
            root = sd_div(sd_add(-half_b, sqrtd), a);
            if (root < t_min || t_max < root) return -1.0;
        }
        return root;
    }
    double on, dn, oa, da, ob, db;  // xy_rect.rs:29-41 etc.
    if (type == RT_PRIM_XY) { on = o.z; dn = d.z; oa = o.x; da = d.x; ob = o.y; db = d.y; }
    else if (type == RT_PRIM_XZ) { on = o.y; dn = d.y; oa = o.x; da = d.x; ob = o.z; db = d.z; }
    else { on = o.x; dn = d.x; oa = o.y; da = d.y; ob = o.z; db = d.z; }
    double t = sd_div(sd_sub(p.k_or_cc, on), dn);
    if (t < t_min || t > t_max) return -1.0;
    double pa = sd_add(oa, sd_mul(t, da)), pb = sd_add(ob, sd_mul(t, db));
    if (pa < p.a[0] || pa > p.a[1] || pb < p.a[2] || pb > p.a[3]) return -1.0;
    return t;
}

// Aabb::hit, aabb.rs:42-59
RT_D bool aabb_hit_d(const DevNodeD& n, Vec3T<double> o, Vec3T<double> d, double t_min, double t_max) {
    for (int a = 0; a < 3; ++a) {
        double inv_d = sd_div(1.0, axis_of(d, a));
        double t0 = sd_mul(sd_sub(n.lo[a], axis_of(o, a)), inv_d);
        double t1 = sd_mul(sd_sub(n.hi[a], axis_of(o, a)), inv_d);
        if (inv_d < 0.0) { double tmp = t0; t0 = t1; t1 = tmp; }
        double mn = t0 > t_min ? t0 : t_min;
        double mx = t1 < t_max ? t1 : t_max;
        if (mx <= mn) return false;
    }
    return true;
}

__global__ void primary_aov_kernel_f64(const __grid_constant__ AovParamsD P, uint32_t* __restrict__ id,
                                       double* __restrict__ t_out, double* __restrict__ normal,
                                       double* __restrict__ point) {
    int px = blockIdx.x * blockDim.x + threadIdx.x, py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= P.width || py >= P.height) return;
    double u = sd_div(sd_add((double)px, 0.5), (double)(P.width - 1));
    double v = sd_div(sd_add((double)py, 0.5), (double)(P.height - 1));
    // upper_left_corner + u*horizontal - v*vertical - origin - offset (offset = 0), camera.rs:329-334
    Vec3T<double> d = sd_sub3(sd_sub3(sd_add3(P.cam.upper_left_corner, sd_scale(u, P.cam.horizontal)),
                                      sd_scale(v, P.cam.vertical)), P.cam.origin);
    Vec3T<double> o = P.cam.origin;
    const double t_min = RT_T_MIN;
    double best_t = __longlong_as_double(0x7ff0000000000000LL);
    int best = -1;
    if (P.n_nodes == 0) {
        for (int i = 0; i < P.n_prims; ++i) {
            double t = prim_test_d(P, i, o, d, t_min, best_t);
            if (t >= 0.0) { best_t = t; best = i; }
        }
    } else {
        int i = 0;
        while (i < P.n_nodes) {
            const DevNodeD& n = P.nodes[i];
            if (aabb_hit_d(n, o, d, t_min, best_t)) {
                if (n.leaf >= 0) {
                    int first = n.leaf & 0xffffff, count = n.leaf >> 24;
                    for (int p = first; p < first + count; ++p) {
                        double t = prim_test_d(P, p, o, d, t_min, best_t);
                        if (t >= 0.0) { best_t = t; best = p; }
                    }
                    i = n.skip;
                } else i = i + 1;
            } else i = n.skip;
        }
    }
    size_t i = (size_t)py * P.width + px;
    if (best < 0) {
        if (id) id[i] = 0;
        if (t_out) t_out[i] = 1.7976931348623157e308;
        if (normal) { normal[3 * i] = 0; normal[3 * i + 1] = 0; normal[3 * i + 2] = 0; }
        if (point) { point[3 * i] = 0; point[3 * i + 1] = 0; point[3 * i + 2] = 0; }
        return;
    }
    const DevPrimD& p = P.prims[best];
    int type = P.prim_kind[best];
    const int inst = P.prim_inst[best];
    Vec3T<double> lo = o, ld = d;           // ray in the primitive's space
    if (inst >= 0) to_local_d(P.instances[inst], lo, ld);
    Vec3T<double> hp = sd_add3(lo, sd_scale(best_t, ld)), on;   // Ray::at
    if (RT_IS_SPHERE(type)) {
        Vec3T<double> pc = sd_sub3(hp, sphere_centre_d(p, type, P.cam.time_a));
        on = mk3(sd_div(pc.x, p.a[3]), sd_div(pc.y, p.a[3]), sd_div(pc.z, p.a[3]));  // sphere.rs:61
    } else on = mk3(type == RT_PRIM_YZ ? 1.0 : 0.0, type == RT_PRIM_XZ ? 1.0 : 0.0, type == RT_PRIM_XY ? 1.0 : 0.0);
    bool front = sd_dot(ld, on) < 0.0;
    Vec3T<double> n = front ? on : -on;
    if (inst >= 0) {
        const DevInstanceD& in = P.instances[inst];
        if (in.flags & 1) {  // rotate_y.rs:51-63
            const double s = in.sin_theta, c = in.cos_theta;
            Vec3T<double> q = hp, m = n;
            q.x = sd_add(sd_mul(c, hp.x), sd_mul(s, hp.z)); q.z = sd_add(sd_mul(-s, hp.x), sd_mul(c, hp.z));
            m.x = sd_add(sd_mul(c, n.x), sd_mul(s, n.z)); m.z = sd_add(sd_mul(-s, n.x), sd_mul(c, n.z));
            hp = q;
            n = sd_dot(ld, m) < 0.0 ? m : -m;
        }
        if (in.flags & 2) {  // translate.rs:34-37
            hp = sd_add3(hp, mk3(in.offset[0], in.offset[1], in.offset[2]));
            n = sd_dot(d, n) < 0.0 ? n : -n;
        }
    }
    if (id) id[i] = P.prim_id[best];
    if (t_out) t_out[i] = best_t;
    if (normal) { normal[3 * i] = n.x; normal[3 * i + 1] = n.y; normal[3 * i + 2] = n.z; }
    if (point) { point[3 * i] = hp.x; point[3 * i + 1] = hp.y; point[3 * i + 2] = hp.z; }
}

// ---------------------------------------------------------------------------
// Vec3::scale_sqrt, src/vec3.rs:119-125
// ---------------------------------------------------------------------------
__global__ void finalize_kernel(const float* __restrict__ accum, float* __restrict__ rgb, size_t n, float scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rgb[i] = sqrtf(scale * accum[i]);
}

// CpuRendererScaled's upscale (cpu_scaled.rs:75-86): every traced block colour, after scale_sqrt,
// fills its scale_w x scale_h screen pixels; screen pixels beyond the last whole block stay 0
// (the reference's buffer starts as Vec3::default()).
__global__ void preview_expand_kernel(const float* __restrict__ accum, double* __restrict__ rgb, int width, int height,
                                      int bw, int bh, int scale_w, int scale_h, double scale) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)width * height) return;
    const int x = (int)(i % width), y = (int)(i / width);
    const int bx = x / scale_w, by = y / scale_h;
    double r = 0.0, g = 0.0, b = 0.0;
    if (bx < bw && by < bh) {
        const float* a = accum + 3 * ((size_t)by * bw + bx);
        r = sqrt(scale * (double)a[0]); g = sqrt(scale * (double)a[1]); b = sqrt(scale * (double)a[2]);
    }
    rgb[3 * i] = r; rgb[3 * i + 1] = g; rgb[3 * i + 2] = b;
}

// ---- progress words of a frame shared by several processes (rc_render_frame) ----
// publish: everything this stream did before (the render kernel's stores into the peer's image) is visible
// system-wide before the word changes
__global__ void frame_publish_kernel(int* word, int value) {
    __threadfence_system();
    *reinterpret_cast<volatile int*>(word) = value;
    __threadfence_system();
}
// wait until words[32 * i] >= target for i in [first, first + n); gives up after ~30 s of GPU time (a rank died:
// the frame would never complete — ranks that are merely late, e.g. still compiling their kernel, are waited
// for) and raises *timed_out instead of hanging the device
__global__ void frame_wait_kernel(const int* words, int first, int n, int target, int* timed_out) {
    if ((int)threadIdx.x >= n) return;
    const volatile int* w = reinterpret_cast<const volatile int*>(words + 32 * (first + (int)threadIdx.x));
    const long long t0 = clock64();
    while (*w < target) {
        __nanosleep(200);
        if (clock64() - t0 > 60000000000LL) { *timed_out = 1; break; }
    }
    __threadfence_system();
}
// slot 0 <- sqrt(scale * (slot 0 + slot 1 + ... + slot world-1)), element by element, slots added in rank order
__global__ void sum_slots_kernel(float* __restrict__ image, size_t slot_floats, int world, size_t n, float scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = image[i];
    for (int r = 1; r < world; ++r) s += image[(size_t)r * slot_floats + i];
    image[i] = sqrtf(scale * s);
}
__global__ void widen_kernel(const float* __restrict__ in, double* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

__global__ void finalize_to_f64_kernel(const float* __restrict__ accum, double* __restrict__ rgb, size_t n, double scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rgb[i] = sqrt(scale * (double)accum[i]);
}

// finalize_to_f64_kernel with each pixel's own sample count (rc_render_adaptive); n = width * height * 3
__global__ void finalize_spp_to_f64_kernel(const float* __restrict__ accum, const int* __restrict__ spp, double* __restrict__ rgb, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rgb[i] = sqrt(1.0 / (double)spp[i / 3] * (double)accum[i]);
}

// ---------------------------------------------------------------------------
// Tone map + quantise.  f64, like the reference's ScreenBuffer thread
// (src/image_buffer.rs:147-153) — it runs once per pixel, not per sample.
// ---------------------------------------------------------------------------
struct ToneParams {
    int type;
    double max_white_pow;
    double A, B, C, D, E, F, toe_angle, exposure_bias, white_scale;
    double aces_in[9], aces_out[9];
};

RT_D double hable_partial(const ToneParams& t, double x) {  // hable.rs:52-62
    return ((x * (t.A * x + t.C * t.B) + t.D * t.E) / (x * (t.A * x + t.B) + t.D * t.F)) - t.toe_angle;
}

RT_D double aces_fit(double x) {  // aces.rs:26-30
    double a = x * (x + 0.0245786) - 0.000090537;
    double b = x * (0.983729 * x + 0.4329510) + 0.238081;
    return a / b;
}

// Rust `f64 as u32`: saturating, NaN -> 0 (png.rs:24-26)
RT_D uint32_t f64_as_u32(double v) {
    if (!(v == v) || v <= 0.0) return 0u;
    if (v >= 4294967295.0) return 4294967295u;
    return (uint32_t)v;
}

__global__ void postprocess_kernel(const __grid_constant__ ToneParams tp, const double* __restrict__ rgb,
                                   size_t n_pixels, uint8_t* __restrict__ rgba, double* __restrict__ mapped) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    double r = rgb[3 * i], g = rgb[3 * i + 1], b = rgb[3 * i + 2];
    if (tp.type == 1) {  // reinhard.rs:16-42
        double l_old = r * 0.2126 + g * 0.7152 + b * 0.0722;
        double numerator = l_old * (1.0 + (l_old / tp.max_white_pow));
        double l_new = numerator / (1.0 + l_old);
        double s = l_new / l_old;
        r *= s; g *= s; b *= s;
    } else if (tp.type == 2) {  // hable.rs:64-80
        r = hable_partial(tp, r * tp.exposure_bias) * tp.white_scale;
        g = hable_partial(tp, g * tp.exposure_bias) * tp.white_scale;
        b = hable_partial(tp, b * tp.exposure_bias) * tp.white_scale;
    } else if (tp.type == 3) {  // aces.rs:18-55
        const double* m = tp.aces_in;
        double x = aces_fit(m[0] * r + m[1] * g + m[2] * b);
        double y = aces_fit(m[3] * r + m[4] * g + m[5] * b);
        double z = aces_fit(m[6] * r + m[7] * g + m[8] * b);
        const double* q = tp.aces_out;
        r = q[0] * x + q[1] * y + q[2] * z;
        g = q[3] * x + q[4] * y + q[5] * z;
        b = q[6] * x + q[7] * y + q[8] * z;
    }
    if (mapped) { mapped[3 * i] = r; mapped[3 * i + 1] = g; mapped[3 * i + 2] = b; }
    if (rgba) {
        uint32_t val = (f64_as_u32(r * 255.0) << 24) | (f64_as_u32(g * 255.0) << 16) | (f64_as_u32(b * 255.0) << 8) | 255u;
        rgba[4 * i] = (uint8_t)(val >> 24); rgba[4 * i + 1] = (uint8_t)(val >> 16);
        rgba[4 * i + 2] = (uint8_t)(val >> 8); rgba[4 * i + 3] = (uint8_t)val;
    }
}

// ---------------------------------------------------------------------------
// FP32 FMA micro-benchmark: 16 independent FFMA chains per thread, register
// only.  Gives the measured non-tensor FP32 issue peak used as the roofline
// denominator (SURVEY §8(d)).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fma_peak_kernel(float* __restrict__ out, int iters, float a, float b) {
    float x[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) x[k] = (float)(threadIdx.x + k) * 1e-3f;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int k = 0; k < 16; ++k) x[k] = fmaf(x[k], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += x[k];
    if (s == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
#endif  // !RT_SPECIALIZED (a scene-specialised translation unit only needs megakernel_body)
