// rt_wavefront.cuh — the wavefront variant of the render path.
//
// A pool of N path slots lives in device memory (sized to stay in the 126 MB
// L2: 1 Mi slots x 80 B = 80 MB).  One pass over the pool is four kinds of
// kernels, each full-width and free of the megakernel's regenerate / miss /
// material divergence:
//
//   wf_generate   ray-gen: every dead slot starts the next sample of its work
//                 item (a chunk of RT_WF_CHUNK samples of one pixel), or flushes
//                 the chunk's radiance sum and pulls the next item with a
//                 warp-aggregated atomic
//   wf_intersect  closest hit (same code as the megakernel); escapes are
//                 terminated here; hits are appended to one of three queues by
//                 material class with a warp-ballot compaction
//   wf_shade      one launch over the three compacted queues, laid end to end:
//                 class 0 solid-colour lambertian, 1 other solid-colour
//                 materials, 2 anything whose texture needs evaluating (checker
//                 / image / Perlin) — a warp never mixes Perlin turbulence with
//                 a one-multiply albedo (except the two boundary warps)
//   wf_flush      at the end: radiance sums still held by slots
//
// Accumulation into the image is atomic but only once per chunk and channel
// (3 atomics per RT_WF_CHUNK samples).  RNG streams, ray-gen, intersection and
// shading are the megakernel's own functions, so both variants trace exactly
// the same paths; only the fp32 summation order differs.
#pragma once
#include <type_traits>
#include "rt_kernels.cuh"

#define RT_WF_CHUNK 32
#define RT_WF_BLOCK 128
#define RT_WF_QUEUES 3

struct WfPool {
    float4* o_t;      // origin.xyz, w = hit t
    float4* d_prim;   // direction.xyz, w = bits(hit primitive)
    float4* thr;      // throughput.xyz, w = bits(last primitive)
    float4* acc;      // radiance sum of the current chunk, w unused
    uint4* info;      // x = pixel, y = next sample of the chunk, z = chunk end, w = bounce | depth_left << 8 | alive << 16
    int* queue[RT_WF_QUEUES];
    // counters: [0..2] queue sizes, [3] alive paths after generate, [4..5] next work item (64-bit), [6] slots holding an unflushed chunk
    unsigned int* counters;
    const float* pixel_u;   // per-pixel u = (x + jitter)/(W-1), cpu.rs:35-36 (computed once per render)
    int n_slots;
    unsigned long long total_work;   // work items = pixels of this share x chunks
    int n_pix_share;                 // 128 x n_tiles (including the out-of-frame pixels of edge tiles)
};

struct WavefrontState {
    WfPool pool;
    size_t capacity = 0;        // slots allocated
    size_t pixel_u_capacity = 0;
    float* pixel_u = nullptr;
    unsigned int* host_counters = nullptr;  // pinned
    cudaEvent_t ev = nullptr;
    WavefrontState() { memset(&pool, 0, sizeof(pool)); }
};

inline void wavefront_release(WavefrontState& w) {
    if (w.pool.o_t) cudaFree(w.pool.o_t);
    if (w.pool.d_prim) cudaFree(w.pool.d_prim);
    if (w.pool.thr) cudaFree(w.pool.thr);
    if (w.pool.acc) cudaFree(w.pool.acc);
    if (w.pool.info) cudaFree(w.pool.info);
    for (int q = 0; q < RT_WF_QUEUES; ++q) if (w.pool.queue[q]) cudaFree(w.pool.queue[q]);
    if (w.pool.counters) cudaFree(w.pool.counters);
    if (w.pixel_u) cudaFree(w.pixel_u);
    if (w.host_counters) cudaFreeHost(w.host_counters);
    if (w.ev) cudaEventDestroy(w.ev);
    memset(&w.pool, 0, sizeof(w.pool));
    w.capacity = 0; w.pixel_u_capacity = 0; w.pixel_u = nullptr; w.host_counters = nullptr; w.ev = nullptr;
}

RT_D uint32_t wf_pack(uint32_t bounce, uint32_t depth_left, uint32_t alive) { return bounce | (depth_left << 8) | (alive << 16); }

// pixel of rank r in this share's tile list (same 16x8 tile / 8x4 warp layout as the megakernel)
RT_D bool wf_pixel_of(const KParams& P, int rank, int& px, int& py) {
    const int k = rank >> 7, within = rank & 127;
    const int tile = P.tile_first + k * P.tile_stride;
    const int tx = tile % P.tiles_x, ty = tile / P.tiles_x;
    const int warp = within >> 5, lane = within & 31;
    px = tx * RT_TILE_W + (warp & 1) * 8 + (lane & 7);
    py = ty * RT_TILE_H + (warp >> 1) * 4 + (lane >> 3);
    return px < P.width && py < P.height;
}

template <int ROUNDS>
__global__ void wf_pixel_u_kernel(const __grid_constant__ KParams P, float* __restrict__ pixel_u, int n_pix_share) {
    int rank = blockIdx.x * blockDim.x + threadIdx.x;
    if (rank >= n_pix_share) return;
    int px, py;
    if (!wf_pixel_of(P, rank, px, py)) return;
    uint32_t pixel = (uint32_t)(py * P.width + px);
    float ujit = 0.5f;
    if (!P.fixed_jitter) ujit = u24(philox2x32_ks<ROUNDS>(pixel, rt_ctr1(0u, 0u, RT_TAG_PIXEL), P.ks).x);
    pixel_u[pixel] = ((float)(px * P.px_scale_x) + ujit) / P.wm1;
}

__global__ void wf_reset_kernel(WfPool W) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 8) W.counters[i] = 0u;
    if (i >= W.n_slots) return;
    W.info[i] = make_uint4(0u, 0u, 0u, 0u);
    W.acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// Ray::time of the path of (pixel, sample): the same draw camera_ray() makes (10-round Philox: the
// wavefront kernels that need it are not templated on the round count; rounds != 10 with a moving
// sphere is rejected at launch)
RT_D float wf_path_time(const KParams& P, uint32_t pixel, uint32_t sample) {
    if (!P.has_motion || P.fixed_jitter) return P.cam.time_a;
    const uint2 w = philox2x32_ks<10>(pixel, rt_ctr1(sample, 0u, RT_TAG_LENS), P.ks);
    return fmaf(P.cam.time_b - P.cam.time_a, u16lo(w), P.cam.time_a);
}

// warp-aggregated fetch of `want` consecutive work items
RT_D unsigned long long wf_take_work(unsigned int* counters, bool want) {
    const unsigned mask = __ballot_sync(0xffffffffu, want);
    if (mask == 0u) return 0ull;
    const int leader = __ffs(mask) - 1;
    unsigned long long base = 0ull;
    if ((threadIdx.x & 31) == leader)
        base = atomicAdd(reinterpret_cast<unsigned long long*>(counters + 4), (unsigned long long)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (unsigned long long)__popc(mask & ((1u << (threadIdx.x & 31)) - 1u));
}

template <int SAMPLER, int ROUNDS>
__global__ void __launch_bounds__(RT_WF_BLOCK)
wf_generate(const __grid_constant__ KParams P, WfPool W, float* __restrict__ accum) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { W.counters[0] = 0u; W.counters[1] = 0u; W.counters[2] = 0u; }
    const bool in_pool = i < W.n_slots;
    uint4 info = in_pool ? W.info[i] : make_uint4(0u, 0u, 0u, 0u);
    bool alive = in_pool && ((info.w >> 16) & 1u);
    bool need_sample = in_pool && !alive;
    // chunk finished: flush its radiance sum (3 atomics per chunk) and take the next work item
    bool chunk_done = need_sample && info.y >= info.z;
    if (chunk_done && info.z != 0u) {
        float4 a = W.acc[i];
        float* dst = accum + 3 * (size_t)info.x;
        atomicAdd(dst, a.x); atomicAdd(dst + 1, a.y); atomicAdd(dst + 2, a.z);
        W.acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        info.z = 0u; info.y = 0u;
    }
    unsigned long long item = wf_take_work(W.counters, chunk_done);
    if (chunk_done) {
        need_sample = false;
        if (item < W.total_work) {
            const int rank = (int)(item % (unsigned long long)W.n_pix_share);
            const int chunk = (int)(item / (unsigned long long)W.n_pix_share);
            int px, py;
            if (wf_pixel_of(P, rank, px, py)) {
                info.x = (uint32_t)(py * P.width + px);
                info.y = (uint32_t)(P.s_begin + chunk * RT_WF_CHUNK);
                uint32_t end = info.y + RT_WF_CHUNK;
                info.z = end < (uint32_t)P.s_end ? end : (uint32_t)P.s_end;
                need_sample = true;
            }
        }
        if (!need_sample) W.info[i] = info;   // idle (no work left, or an out-of-frame pixel of an edge tile)
    }
    if (need_sample) {
        PixelCtx pc;
        pc.pixel = info.x;
        pc.py = (int)(info.x / (uint32_t)P.width);
        pc.px = (int)(info.x - (uint32_t)pc.py * (uint32_t)P.width);
        pc.dir0 = P.cam.upper_left_corner + W.pixel_u[info.x] * P.cam.horizontal;
        pc.dir0 = pc.dir0 - ((float)(pc.py * P.px_scale_y) * P.inv_hm1) * P.cam.vertical;   // as pixel_setup()
        const uint32_t sample = info.y;
        float vjit = 32768.0f;   // the v jitter times 65536 (camera_ray)
        if (!P.fixed_jitter) vjit = u16lo_int(philox2x32_ks<ROUNDS>(pc.pixel, rt_ctr1(rt_vjit_sample(sample), 0u, RT_TAG_PATH), P.ks));
        vec3f o, d;
        float time;   // not stored in the pool: wf_path_time() recomputes it from (pixel, sample)
        camera_ray<SAMPLER, ROUNDS>(P, pc, sample, vjit, o, d, time);
        info.y = sample + 1u;
        if (P.max_depth > 0) {
            W.o_t[i] = make_float4(o.x, o.y, o.z, 0.f);
            W.d_prim[i] = make_float4(d.x, d.y, d.z, __int_as_float(-1));
            W.thr[i] = make_float4(1.f, 1.f, 1.f, __int_as_float(-1));
            info.w = wf_pack(0u, (uint32_t)P.max_depth, 1u);
            alive = true;
        } else {  // renderer.rs:48-56: depth 0 is white
            float4 a = W.acc[i];
            W.acc[i] = make_float4(a.x + 1.f, a.y + 1.f, a.z + 1.f, 0.f);
            info.w = 0u;
        }
        W.info[i] = info;
    }
    // statistics for the host's termination test
    const unsigned alive_mask = __ballot_sync(0xffffffffu, alive);
    const unsigned pending_mask = __ballot_sync(0xffffffffu, in_pool && info.z != 0u);
    if ((threadIdx.x & 31) == 0) {
        if (alive_mask) atomicAdd(W.counters + 3, (unsigned)__popc(alive_mask));
        if (pending_mask) atomicAdd(W.counters + 6, (unsigned)__popc(pending_mask));
    }
}

template <int MODE>
__global__ void __launch_bounds__(RT_WF_BLOCK)
wf_intersect(const __grid_constant__ KParams P, WfPool W) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmemLayout L = stage_scene<MODE>(P, smem);   // launched with n_perlin = 0: geometry only
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_pool = i < W.n_slots;
    uint4 info = in_pool ? W.info[i] : make_uint4(0u, 0u, 0u, 0u);
    const bool alive = in_pool && ((info.w >> 16) & 1u);
    int cls = -1;
    if (alive) {
        float4 ot = W.o_t[i], dp = W.d_prim[i], th = W.thr[i];
        RayT<float> r = make_ray(mk3(ot.x, ot.y, ot.z), mk3(dp.x, dp.y, dp.z), wf_path_time(P, info.x, info.y - 1u));
        const int last_prim = __float_as_int(th.w);
        float t;
        int prim;
        float packed;
        if (MODE == RT_MODE_CONST_LINEAR) { ConstScene S(P, L.prims); prim = closest_hit<MODE>(P, S, r, last_prim, t); packed = prim >= 0 ? S.pb(prim).z : 0.f; }
        else { PtrScene S; S.prims = L.prims; S.nodes = L.nodes; S.inst = P.instances; S.ref_aabb = P.ref_aabb; prim = closest_hit<MODE>(P, S, r, last_prim, t); packed = prim >= 0 ? S.pb(prim).z : 0.f; }
        if (prim < 0) {  // renderer.rs:78-88
            vec3f bg = background_color(P, r.d);
            float4 a = W.acc[i];
            W.acc[i] = make_float4(a.x + th.x * bg.x, a.y + th.y * bg.y, a.z + th.z * bg.z, 0.f);
            info.w &= ~(1u << 16);
            W.info[i] = info;
        } else {
            W.o_t[i] = make_float4(ot.x, ot.y, ot.z, t);
            W.d_prim[i] = make_float4(dp.x, dp.y, dp.z, __int_as_float(prim));
            const int mat = kinds_mat(packed);
            cls = kinds_tex(packed) != RT_TEX_SOLID ? 2 : (mat == RT_MAT_LAMBERTIAN ? 0 : 1);
        }
    }
    {   // segment statistics
        const unsigned am = __ballot_sync(0xffffffffu, alive);
        if ((threadIdx.x & 31) == 0 && am && P.segment_counter) atomicAdd(P.segment_counter, (unsigned long long)__popc(am));
    }
    // warp-ballot compaction into the material-class queues
#pragma unroll
    for (int q = 0; q < RT_WF_QUEUES; ++q) {
        const unsigned mask = __ballot_sync(0xffffffffu, cls == q);
        if (mask == 0u) continue;
        const int leader = __ffs(mask) - 1;
        unsigned base = 0u;
        if ((threadIdx.x & 31) == leader) base = atomicAdd(W.counters + q, (unsigned)__popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (cls == q) W.queue[q][base + __popc(mask & ((1u << (threadIdx.x & 31)) - 1u))] = i;
    }
}

// One launch shades all three queues: entry q belongs to class 0 below counters[0], class 1
// below counters[0] + counters[1], class 2 above.  Only the (at most two) warps that straddle a
// class boundary execute more than one class's code.
template <int SAMPLER, int ROUNDS, bool TEX, class Scene>
RT_D void wf_shade_one(const KParams& P, const WfPool& W, const TexCtx& X, const Scene& S, int i) {
    float4 ot = W.o_t[i], dp = W.d_prim[i], th = W.thr[i];
    uint4 info = W.info[i];
    vec3f o = mk3(ot.x, ot.y, ot.z), d = mk3(dp.x, dp.y, dp.z), T = mk3(th.x, th.y, th.z);
    const RayT<float> r = make_ray(o, d, wf_path_time(P, info.x, info.y - 1u));
    const int prim = __float_as_int(dp.w);
    uint32_t bounce = (info.w & 0xffu) + 1u, depth_left = (info.w >> 8) & 0xffu;
    RngCtx R; R.ks = P.ks; R.pixel = info.x; R.sample = info.y - 1u;
    // the block of the segment that ended in this hit (hit number `bounce` closes segment bounce - 1)
    const uint2 rnd = philox2x32_ks<ROUNDS>(R.pixel, rt_ctr1(R.sample, bounce - 1u, RT_TAG_PATH), P.ks);
    vec3f X_end;
    bool alive = shade_hit<SAMPLER, ROUNDS, TEX>(P, X, S, R, prim, r, ot.w, bounce, rnd, o, d, T, X_end);
    if (alive) {
        if (--depth_left == 0u) { X_end = mk3(1.0f, 1.0f, 1.0f); alive = false; }  // white at depth 0
    }
    if (alive) {
        W.o_t[i] = make_float4(o.x, o.y, o.z, 0.f);
        W.d_prim[i] = make_float4(d.x, d.y, d.z, __int_as_float(-1));
        W.thr[i] = make_float4(T.x, T.y, T.z, __int_as_float(prim));
    } else {
        float4 a = W.acc[i];
        W.acc[i] = make_float4(a.x + T.x * X_end.x, a.y + T.y * X_end.y, a.z + T.z * X_end.z, 0.f);
    }
    info.w = wf_pack(bounce, depth_left, alive ? 1u : 0u);
    W.info[i] = info;
}

template <int MODE, int SAMPLER, int ROUNDS>
__global__ void __launch_bounds__(RT_WF_BLOCK)
wf_shade(const __grid_constant__ KParams P, WfPool W) {
    extern __shared__ __align__(16) unsigned char smem[];
    const unsigned n0 = W.counters[0], n1 = n0 + W.counters[1], n2 = n1 + W.counters[2];
    if (blockIdx.x * blockDim.x >= n2) return;   // whole block beyond the queues
    SmemLayout L = stage_scene<MODE>(P, smem);
    TexCtx X; X.perlin = L.perlin; X.perm = L.perm;
    const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n2) return;
    const int cls = q < n0 ? 0 : (q < n1 ? 1 : 2);
    const int i = cls == 0 ? W.queue[0][q] : (cls == 1 ? W.queue[1][q - n0] : W.queue[2][q - n1]);
    if (MODE == RT_MODE_CONST_LINEAR) {
        ConstScene S(P, L.prims);
        if (cls == 2) wf_shade_one<SAMPLER, ROUNDS, true>(P, W, X, S, i); else wf_shade_one<SAMPLER, ROUNDS, false>(P, W, X, S, i);
    } else {
        PtrScene S; S.prims = L.prims; S.nodes = L.nodes; S.inst = P.instances; S.ref_aabb = P.ref_aabb;
        if (cls == 2) wf_shade_one<SAMPLER, ROUNDS, true>(P, W, X, S, i); else wf_shade_one<SAMPLER, ROUNDS, false>(P, W, X, S, i);
    }
}

__global__ void wf_flush(WfPool W, float* __restrict__ accum) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W.n_slots) return;
    uint4 info = W.info[i];
    if (info.z == 0u) return;
    float4 a = W.acc[i];
    float* dst = accum + 3 * (size_t)info.x;
    atomicAdd(dst, a.x); atomicAdd(dst + 1, a.y); atomicAdd(dst + 2, a.z);
    W.acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    info.z = 0u;
    W.info[i] = info;
}

// ---------------------------------------------------------------------------
// Host driver
// ---------------------------------------------------------------------------
// f(std::integral_constant<int, M>()) for the runtime scene mode M (RT_MODE_*): where the host picks the kernels of a mode
template <class F>
auto with_mode(int mode, F&& f) {
    switch (mode) {
    case RT_MODE_CONST_LINEAR: return f(std::integral_constant<int, RT_MODE_CONST_LINEAR>());
    case RT_MODE_SMEM_BVH: return f(std::integral_constant<int, RT_MODE_SMEM_BVH>());
    case RT_MODE_GLOBAL_BVH: return f(std::integral_constant<int, RT_MODE_GLOBAL_BVH>());
    default: return f(std::integral_constant<int, RT_MODE_SMEM_LINEAR>());
    }
}

// smem: the scene staged per CTA; smem_perlin: its Perlin part, which wf_intersect does without
template <int MODE, int SAMPLER, int ROUNDS>
int wavefront_run(WavefrontState& w, const KParams& kp, float* accum, size_t smem, size_t smem_perlin, cudaStream_t st,
                  uint64_t& launches) {
    WfPool& W = w.pool;
    const int blocks = (W.n_slots + RT_WF_BLOCK - 1) / RT_WF_BLOCK;
    const size_t smem_int = smem - smem_perlin;   // geometry only
    KParams kp_int = kp;
    kp_int.n_perlin = 0;
    if (smem > 48 * 1024) {
        cudaFuncSetAttribute(wf_intersect<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_int);
        cudaFuncSetAttribute(wf_shade<MODE, SAMPLER, ROUNDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    wf_pixel_u_kernel<ROUNDS><<<(W.n_pix_share + 255) / 256, 256, 0, st>>>(kp, w.pixel_u, W.n_pix_share);
    wf_reset_kernel<<<blocks, RT_WF_BLOCK, 0, st>>>(W);
    launches += 2;
    const int check_every = 16;
    for (int iter = 0;; ++iter) {
        const bool check = (iter % check_every) == check_every - 1;
        if (check) cudaMemsetAsync(W.counters + 3, 0, sizeof(unsigned), st), cudaMemsetAsync(W.counters + 6, 0, sizeof(unsigned), st);
        wf_generate<SAMPLER, ROUNDS><<<blocks, RT_WF_BLOCK, 0, st>>>(kp, W, accum);
        if (check) {
            cudaMemcpyAsync(w.host_counters, W.counters, 8 * sizeof(unsigned), cudaMemcpyDeviceToHost, st);
            cudaEventRecord(w.ev, st);
        }
        wf_intersect<MODE><<<blocks, RT_WF_BLOCK, smem_int, st>>>(kp_int, W);
        wf_shade<MODE, SAMPLER, ROUNDS><<<blocks, RT_WF_BLOCK, smem, st>>>(kp, W);
        launches += 3;
        if (check) {
            if (cudaEventSynchronize(w.ev) != cudaSuccess) return RC_ERR_CUDA;
            // after this generate: nobody alive, and nobody holds an unflushed chunk -> all work is done
            if (w.host_counters[3] == 0u && w.host_counters[6] == 0u) break;
        }
        if (cudaPeekAtLastError() != cudaSuccess) return RC_ERR_CUDA;
    }
    wf_flush<<<blocks, RT_WF_BLOCK, 0, st>>>(W, accum);
    launches += 1;
    return cudaGetLastError() == cudaSuccess ? RC_OK : RC_ERR_CUDA;
}

inline int wavefront_prepare(WavefrontState& w, const KParams& kp) {
    size_t slots = (size_t)1024 * 1024;
    const size_t n_pix_share = (size_t)kp.n_tiles * 128;
    const int spp = kp.s_end - kp.s_begin;
    const size_t chunks = (size_t)(spp + RT_WF_CHUNK - 1) / RT_WF_CHUNK;
    if (slots > n_pix_share * chunks) slots = n_pix_share * chunks;     // never more slots than work items
    if (slots < 1024) slots = 1024;
    if (slots > w.capacity) {
        size_t keep_u = w.pixel_u_capacity;
        float* keep_p = w.pixel_u;
        unsigned* keep_h = w.host_counters;
        cudaEvent_t keep_e = w.ev;
        w.pixel_u = nullptr; w.host_counters = nullptr; w.ev = nullptr;
        wavefront_release(w);
        w.pixel_u = keep_p; w.pixel_u_capacity = keep_u; w.host_counters = keep_h; w.ev = keep_e;
        WfPool& W = w.pool;
        bool ok = cudaMalloc(&W.o_t, slots * sizeof(float4)) == cudaSuccess &&
                  cudaMalloc(&W.d_prim, slots * sizeof(float4)) == cudaSuccess &&
                  cudaMalloc(&W.thr, slots * sizeof(float4)) == cudaSuccess &&
                  cudaMalloc(&W.acc, slots * sizeof(float4)) == cudaSuccess &&
                  cudaMalloc(&W.info, slots * sizeof(uint4)) == cudaSuccess &&
                  cudaMalloc(&W.counters, 8 * sizeof(unsigned)) == cudaSuccess;
        for (int q = 0; q < RT_WF_QUEUES && ok; ++q) ok = cudaMalloc(&W.queue[q], slots * sizeof(int)) == cudaSuccess;
        if (!ok) return RC_ERR_CUDA;
        w.capacity = slots;
    }
    const size_t n_pixels = (size_t)kp.width * kp.height;
    if (n_pixels > w.pixel_u_capacity) {
        if (w.pixel_u) cudaFree(w.pixel_u);
        if (cudaMalloc(&w.pixel_u, n_pixels * sizeof(float)) != cudaSuccess) return RC_ERR_CUDA;
        w.pixel_u_capacity = n_pixels;
    }
    if (!w.host_counters && cudaMallocHost(&w.host_counters, 8 * sizeof(unsigned)) != cudaSuccess) return RC_ERR_CUDA;
    if (!w.ev && cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming) != cudaSuccess) return RC_ERR_CUDA;
    w.pool.n_slots = (int)slots;
    w.pool.pixel_u = w.pixel_u;
    w.pool.n_pix_share = (int)n_pix_share;
    w.pool.total_work = (unsigned long long)n_pix_share * chunks;
    return RC_OK;
}

inline int wavefront_render(WavefrontState& w, int mode, const KParams& kp, float* accum, int sampler, int rounds,
                            size_t smem, size_t smem_perlin, cudaStream_t st, uint64_t& launches) {
    int rc = wavefront_prepare(w, kp);
    if (rc != RC_OK) return rc;
    return with_mode(mode, [&](auto m) {
        constexpr int M = decltype(m)::value;
        if (rounds == 7) {
            if (sampler == RC_SAMPLER_REJECTION) return wavefront_run<M, 1, 7>(w, kp, accum, smem, smem_perlin, st, launches);
            return wavefront_run<M, 0, 7>(w, kp, accum, smem, smem_perlin, st, launches);
        }
        if (sampler == RC_SAMPLER_REJECTION) return wavefront_run<M, 1, 10>(w, kp, accum, smem, smem_perlin, st, launches);
        return wavefront_run<M, 0, 10>(w, kp, accum, smem, smem_perlin, st, launches);
    });
}
