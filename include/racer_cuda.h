/*
 * racer_cuda.h — C ABI of libracer_cuda.so, the B200 (sm_100a) path-tracing
 * backend that drops in behind racer-tracer's `Renderer::render`.
 *
 * All reference citations are relative to /root/reference/racer-tracer/.
 *
 * What this boundary replaces (SURVEY.md §8(b)):
 *   trait Renderer { fn render(&self, RenderData, &DataWriter<ImageBufferEvent>) }
 *                                                  src/renderer.rs:101-107
 *   RenderData { camera_data, image, scene, background, config, cancel_event }
 *                                                  src/renderer.rs:92-99
 *   CpuRenderer::render / raytrace / prepare_threads   src/renderer/cpu.rs:26-131
 *   ray_color                                      src/renderer.rs:41-90
 *
 * The reference passes opaque trait objects (`&dyn Hittable`, `&dyn
 * BackgroundColor`); the host shim flattens them into the plain structs below
 * (structure-of-arrays primitive buffers, small material / texture tables, a
 * host-built BVH) before calling in.  Everything on the host side is f64, as
 * in the reference; the library converts to fp32 on upload.
 *
 * Conventions: every entry point returns RC_OK (0) or a negative rc_status;
 * rc_last_error() returns the text of the last failure on the calling thread.
 * The library never keeps a host pointer after a call returns.  There is no
 * CPU fallback: without a usable CUDA device rc_create fails with
 * RC_ERR_NO_DEVICE.
 */
#ifndef RACER_CUDA_H
#define RACER_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RC_ABI_VERSION 2

/* ---- status ------------------------------------------------------------ */
typedef enum rc_status {
    RC_OK = 0,
    RC_ERR_INVALID = -1,    /* bad argument / inconsistent scene            */
    RC_ERR_NO_DEVICE = -2,  /* no CUDA device; maps to a new TracerError
                               variant (src/error.rs:71-97, ordinal 23)     */
    RC_ERR_CUDA = -3,       /* a CUDA runtime call failed                   */
    RC_ERR_STATE = -4,      /* scene / camera not uploaded yet              */
    RC_ERR_CANCELLED = -5,  /* cancel flag was already set on entry:
                               TracerError::CancelEvent, cpu.rs:79-83       */
    RC_ERR_NCCL = -6        /* NCCL unavailable / failed (sample split)     */
} rc_status;

/* ---- primitives (SoA) -------------------------------------------------- */
/* src/geometry/sphere.rs:31-68, xy_rect.rs:21-48, xz_rect.rs:21-49,
 * yz_rect.rs:21-49 */
enum { RC_PRIM_SPHERE = 0, RC_PRIM_XY_RECT = 1, RC_PRIM_XZ_RECT = 2, RC_PRIM_YZ_RECT = 3,
       /* src/geometry/moving_sphere.rs:19-100: a sphere whose centre moves linearly from
        * pos (ray time time_a) to pos_b (ray time time_b); prim_data = pos, radius and
        * prim_motion = pos_b, time_a, time_b.  Only the Random loader creates it
        * (src/scene/random.rs:53-56). */
       RC_PRIM_MOVING_SPHERE = 4 };

/* src/material/lambertian.rs, metal.rs, dialectric.rs, diffuse_light.rs */
enum { RC_MAT_LAMBERTIAN = 0, RC_MAT_METAL = 1, RC_MAT_DIELECTRIC = 2, RC_MAT_DIFFUSE_LIGHT = 3 };

/* src/texture/solid_color.rs, checkered.rs, image.rs, noise.rs */
enum { RC_TEX_SOLID = 0, RC_TEX_CHECKER = 1, RC_TEX_IMAGE = 2, RC_TEX_NOISE = 3 };

/* src/background_color.rs:27-48 */
enum { RC_BG_SKY = 0, RC_BG_SOLID = 1 };

/* src/tone_map.rs:18-66 */
enum { RC_TONE_NONE = 0, RC_TONE_REINHARD = 1, RC_TONE_HABLE = 2, RC_TONE_ACES = 3 };

typedef struct rc_material {
    int32_t type;     /* RC_MAT_*                                           */
    int32_t texture;  /* index into rc_scene.textures (unused: dielectric)  */
    double  param;    /* metal: fuzz; dielectric: refraction_index          */
} rc_material;

typedef struct rc_texture {
    int32_t type;      /* RC_TEX_*                                          */
    int32_t a;         /* checker: even texture (texture_a); image: image
                          index; noise: perlin table index                  */
    int32_t b;         /* checker: odd texture (texture_b); noise: depth    */
    int32_t reserved;
    double  color[3];  /* solid: colour; noise: colour                      */
    double  scale;     /* noise: scale; checker: checker_size (10.0,
                          src/texture/checkered.rs:19)                      */
} rc_texture;

typedef struct rc_image {
    int32_t width, height;
    const uint8_t* rgba;  /* width*height*4, row 0 = top, as image::RgbaImage
                             (src/texture/image.rs:18-24)                   */
} rc_image;

/* One Perlin instance (src/texture/noise.rs:36-55).  The reference's
 * permutation tables are the identity (noise.rs:122 iterates an empty range);
 * they are still passed explicitly. */
typedef struct rc_perlin {
    double  ran_vec[256][3];
    int32_t perm_x[256], perm_y[256], perm_z[256];
} rc_perlin;

/* Instance transform of a top-level object (next scope, SURVEY §8(f)-1):
 * RotateY then Translate, src/geometry/rotate_y.rs:29-66, translate.rs:23-42,
 * src/scene/yml.rs:401-439.  flags bit0 = rotate, bit1 = translate. */
typedef struct rc_instance {
    int32_t flags;
    int32_t reserved;
    double  sin_theta, cos_theta;
    double  offset[3];
} rc_instance;

/* Flat binary BVH (src/bvh_node.rs:31-140).  Leaves hold one primitive, as in
 * the reference.  left >= 0: inner node, children = nodes[left], nodes[right].
 * left < 0: leaf over one top-level object, first primitive = ~left, `right`
 * = number of consecutive primitives (1, or 6 for the sides of a Box, tested
 * in order like Boxx::obj_hit, src/geometry/box.rs:82-101).  Node 0 is the
 * root.  n_nodes == 0 selects the linear closest-hit loop over all primitives
 * in index order (the reference's src/shared_scene.rs:37-53 semantics) — for
 * scenes whose table fits a CTA's staging budget (a few hundred primitives);
 * larger ones get a BVH built on the GPU from prim_aabb (rc_build_lbvh).
 * Primitives must be stored in the tree's depth-first (left-to-right) leaf
 * order so that "later visited wins an exact tie" (bvh_node.rs:124-129,
 * sphere.rs:53) reduces to "higher index wins". */
typedef struct rc_bvh_node {
    double  bmin[3], bmax[3];
    int32_t left, right;
} rc_bvh_node;

typedef struct rc_scene {
    /* primitives, structure of arrays, n_prims entries each */
    int32_t         n_prims;
    const int32_t*  prim_type;      /* RC_PRIM_*                            */
    const double*   prim_data;      /* 5 per prim: sphere cx,cy,cz,r,0;
                                       xy: x0,x1,y0,y1,k; xz: x0,x1,z0,z1,k;
                                       yz: y0,y1,z0,z1,k                    */
    const int32_t*  prim_material;  /* index into materials                 */
    const uint32_t* prim_id;        /* canonical object id, >= 1; 0 = miss
                                       (src/renderer.rs:81-87)              */
    const int32_t*  prim_instance;  /* -1 or index into instances; may be
                                       NULL when n_instances == 0           */
    const double*   prim_aabb;      /* 6 per prim: min xyz, max xyz — the
                                       top-level object's stored Aabb, a
                                       ray-cull volume (bvh_node.rs:119)    */
    int32_t            n_instances;
    const rc_instance* instances;
    int32_t            n_materials;
    const rc_material* materials;
    int32_t            n_textures;
    const rc_texture*  textures;
    int32_t            n_images;
    const rc_image*    images;
    int32_t            n_perlin;
    const rc_perlin*   perlin;
    int32_t            n_nodes;
    const rc_bvh_node* nodes;
    /* background */
    int32_t bg_type;      /* RC_BG_*                                        */
    int32_t reserved;
    double  bg_a[3];      /* sky: top; solid: colour                        */
    double  bg_b[3];      /* sky: bottom                                    */
    /* ABI 2 */
    const double* prim_motion;  /* 5 per prim (pos_b xyz, time_a, time_b), read
                                   for RC_PRIM_MOVING_SPHERE only; may be NULL
                                   when the scene has no moving sphere       */
} rc_scene;

/* The 14 fields of CameraSharedData, src/camera.rs:57-72. */
typedef struct rc_camera {
    double origin[3];
    double upper_left_corner[3];
    double forward[3];
    double right[3];
    double up[3];
    double horizontal[3];
    double vertical[3];
    double vfov;
    double viewport_width;
    double viewport_height;
    double lens_radius;
    double focus_distance;
    double time_a;
    double time_b;
} rc_camera;

/* ---- render parameters -------------------------------------------------- */
enum { RC_VARIANT_MEGAKERNEL = 0, RC_VARIANT_WAVEFRONT = 1 };
/* RC_SAMPLER_DIRECT: inverse-transform sampling of the same distributions
 * (uniform on the sphere / in the ball / in the disk), one Philox block per
 * event.  RC_SAMPLER_REJECTION: the reference's rejection loops op for op
 * (src/vec3.rs:424-444, src/util.rs:25-39), one Philox block per iteration. */
enum { RC_SAMPLER_DIRECT = 0, RC_SAMPLER_REJECTION = 1 };
/* How the image is partitioned over `world` participants (devices of one
 * context, or ranks of a multi-process job): interleaved tiles (tile k ->
 * participant k mod world), or contiguous sample slices. */
enum { RC_SPLIT_TILES = 0, RC_SPLIT_SAMPLES = 1 };

typedef struct rc_params {
    int32_t  width, height;   /* config.screen, src/config.rs:70-73         */
    int32_t  samples;         /* config.render.samples, src/config.rs:75-82 */
    int32_t  max_depth;       /* config.render.max_depth                    */
    uint64_t seed;            /* Philox key; the reference is unseeded
                                 (src/util.rs:9-23)                         */
    int32_t  variant;         /* RC_VARIANT_*                               */
    int32_t  sampler;         /* RC_SAMPLER_*                               */
    int32_t  split;           /* RC_SPLIT_*                                 */
    int32_t  tile_w, tile_h;  /* interleaved tile size: 0 x 0 or 16 x 8, the
                                 kernels' fixed tile; anything else is
                                 RC_ERR_INVALID                             */
    int32_t  rank, world;     /* this participant's slot when the caller
                                 drives several processes; 0,1 otherwise    */
    int32_t  fixed_jitter;    /* 1: pixel-centre, lens-centre rays
                                 (primary-hit parity, SURVEY §8(c))         */
    int32_t  rng_rounds;      /* Philox rounds; 0 = 10                      */
    int32_t  specialize;      /* 0: precompiled kernels.  1: compile the scene
                                 into the megakernel at run time (NVRTC, cached
                                 per scene: primitives as immediates for scenes
                                 on the constant-table path, the kinds of
                                 primitive / material / wrapper present for BVH
                                 scenes) and fail if that is impossible.  2: the
                                 same, but fall back to the precompiled kernel.
                                 Needs the megakernel, the direct sampler and
                                 fixed_jitter = 0                            */
} rc_params;

typedef struct rc_tone_map {
    int32_t type;             /* RC_TONE_*                                  */
    int32_t reserved;
    double  max_white;        /* Reinhard, default 25.0 (tone_map.rs:21-23) */
    double  hable[6];         /* shoulder_strength, linear_strength,
                                 linear_angle, toe_strength, toe_numerator,
                                 toe_denominator (tone_map.rs:24-44)        */
    double  exposure_bias;    /* 2.0                                        */
    double  linear_white_point; /* 11.2                                     */
    double  aces_in[9];       /* row-major 3x3 (tone_map.rs:45-60)          */
    double  aces_out[9];
} rc_tone_map;

/* Counters of the last render on this context (device work only). */
typedef struct rc_stats {
    double   gpu_ms;          /* CUDA-event time of the last render call    */
    uint64_t samples;         /* pixel-samples traced by this context's
                                 participants (their shares only)           */
    uint64_t segments;        /* ray segments traced (0 if not counted)     */
    uint64_t kernel_launches; /* kernels launched by the last render call   */
    int32_t  n_devices;
    int32_t  sm_count;        /* of device 0                                */
    int32_t  sm_clock_khz;    /* max SM clock of device 0                   */
    int32_t  specialized;     /* 1: the last render ran the scene-specialised
                                 (NVRTC) megakernel, 0: a precompiled kernel */
} rc_stats;

typedef struct rc_ctx rc_ctx;

/* ---- entry points ------------------------------------------------------- */

/* Create a context over `n` CUDA devices (device ordinals in `devices`; NULL
 * = 0..n-1).  Replaces the construction of Box<dyn Renderer> at
 * src/renderer.rs:109-116 / src/main.rs:127-129. */
int rc_create(const int32_t* devices, int32_t n, rc_ctx** out);
int rc_destroy(rc_ctx* ctx);

/* Launch on a caller-owned CUDA stream (a cudaStream_t cast to void*) on
 * device 0 of the context instead of the context's own stream. */
int rc_set_stream(rc_ctx* ctx, void* cuda_stream);

/* Upload the flattened scene to every device of the context.  Replaces the
 * `scene: &dyn Hittable` + `background: &dyn BackgroundColor` members of
 * RenderData (src/renderer.rs:92-99); called again whenever the BVH changed
 * (src/main.rs:178-183, src/bvh_node.rs:176-205). */
int rc_upload_scene(rc_ctx* ctx, const rc_scene* scene);

/* Build the acceleration structure of the uploaded scene ON THE GPU: a linear BVH over the
 * Morton codes of the top-level objects' Aabb centres (prim_aabb must have been supplied), in
 * the traversal layout the kernels read.  Replaces BoundingVolumeHirearchy::new / Node::build
 * (src/bvh_node.rs:31-82,142-170) and the host rebuild after an edit (bvh_node.rs:176-205); the
 * nodes passed to rc_upload_scene, if any, are superseded.  Leaves keep the reference's semantics:
 * one top-level object each, its stored Aabb is its cull volume (bvh_node.rs:119). */
int rc_build_lbvh(rc_ctx* ctx);

/* The acceleration structure currently on the device, as rc_bvh_node records in pre-order, and
 * prim_order[i] = index (in the uploaded arrays) of the primitive now stored at position i — so
 * that a host (or the parity oracle) can trace the very same tree.  Returns the node count (0 for
 * the linear modes); fills only the arrays whose capacity suffices. */
int rc_get_bvh(rc_ctx* ctx, rc_bvh_node* nodes, int32_t node_capacity, int32_t* prim_order, int32_t prim_capacity);

/* Replaces `camera_data: &CameraSharedData` (src/renderer.rs:93). */
int rc_set_camera(rc_ctx* ctx, const rc_camera* camera);

/* The whole of CpuRenderer::render (src/renderer/cpu.rs:118-131) for one
 * image: every pixel x sample through ray_color (src/renderer.rs:41-90), then
 * Vec3::scale_sqrt (src/vec3.rs:119-125).  out_rgb receives width*height*3
 * doubles, row 0 = top, gamma'd (sqrt of the mean) and NOT tone-mapped —
 * exactly what CpuRenderer puts in ImageBufferEvent::BufferUpdate
 * (src/renderer/cpu.rs:64-70).  `cancel` (may be NULL) is polled between
 * passes like do_cancel (src/renderer.rs:25-30); a cancelled render returns
 * RC_OK without touching out_rgb (cpu.rs:55-62).  With several devices in
 * the context the image is partitioned as params->split says and gathered /
 * reduced onto device 0 before the download.
 * With params->world > 1 the call renders only this participant's share
 * (params->rank): a tile share gives sqrt(sum / samples) in its tiles and
 * 0.0 in every other pixel; a sample share gives sqrt(share_sum / samples)
 * in every pixel, where share_sum is the sum over its samples only (so
 * samples * out^2, summed over the ranks, is the whole frame's sum), and
 * all zeros when the share holds no sample (samples < world).  Nothing of
 * an earlier render shows through.  rc_get_stats' `samples` is the share's
 * pixel-samples. */
int rc_render(rc_ctx* ctx, const rc_params* params, double* out_rgb,
              const volatile int32_t* cancel);

/* Adaptive sampling: every pixel gets as many samples as its noise needs, up to params->samples (S).
 * Round 0 traces samples [0, min_samples) of every pixel.  After each round every pixel still active is tested; one
 * that passes stops, the others go from n to min(2n, S) samples.  So each pixel ends with n_p in {n0, 2 n0, 4 n0, ..,
 * S} (n0 = min_samples), traced as samples [0, n_p) of its own stream with rc_render's seed, jitter and depth: the
 * pixel equals rc_render's with samples = n_p, up to the order of fp32 sums.
 * The test, on y = (r + g + b) / 3 of each sample's linear radiance, with S1 = sum y and S2 = sum y^2 over the
 * pixel's n samples: mu = S1 / n, s^2 = max(0, (S2 - S1^2 / n) / (n - 1)), se = sqrt(s^2 / n), and
 * err = (sqrt(mu + se) - sqrt(max(mu - se, 0))) / 2 — the half-width of the one-sigma interval of the returned
 * (gamma'd) value.  The pixel passes when err <= threshold.  S1 comes from the fp32 radiance sums and S2 from fp32
 * sums of y^2 per round, so err carries their rounding: threshold = 0 stops the pixels whose samples are all equal
 * where that rounding cancels (samples that are all 0, or exactly representable), and no pixel that has a spread.
 * out_rgb: width*height*3 doubles, sqrt(sum_p / n_p) as rc_render finalises them with n_p for samples.
 * out_spp (may be NULL): width*height n_p.  out_err (may be NULL): width*height err at n_p.
 * rc_get_stats: samples = sum of n_p, segments and kernel_launches of all rounds, gpu_ms of the whole call.
 * `cancel`: as for rc_render (checked at entry, relayed inside each round, checked between rounds; a cancelled call
 * writes nothing).  Supported: a one-device context, world <= 1, the megakernel, the direct sampler, 10 Philox rounds;
 * specialize as for rc_render.  Anything else is RC_ERR_INVALID. */
typedef struct rc_adaptive {
    int32_t min_samples;   /* n0 >= 2: samples every pixel gets before its first test            */
    int32_t reserved;
    double  threshold;     /* >= 0, finite: stop a pixel once its error estimate is <= threshold   */
} rc_adaptive;

int rc_render_adaptive(rc_ctx* ctx, const rc_params* params, const rc_adaptive* a,
                       double* out_rgb, int32_t* out_spp, double* out_err,
                       const volatile int32_t* cancel);

/* Denoised rendering: a render of params->samples (S >= 2) samples per pixel, filtered on the GPU by an edge-avoiding
 * à-trous wavelet filter guided by per-pixel variance and first-hit features (SVGF's spatial filter, without its
 * temporal part).
 * Inputs of the filter, per pixel p of the W x H image (what rc_denoise_aux returns):
 *   m_p    linear mean radiance (rgb): sum / S of the same samples rc_render traces (up to the order of fp32 sums);
 *   v_p    variance of the mean of y = (r + g + b) / 3: s^2 / S with s^2 = max(0, (S2 - S1^2 / S) / (S - 1)), S1 = sum y,
 *          S2 = sum y^2 over the pixel's samples (S2 from fp32 sums of y^2, as rc_render_adaptive's test);
 *   alb_p  the first hit's albedo: the texture colour for Lambertian and Metal, (1, 1, 1) for dielectrics, lights and
 *          misses;
 *   n_p, z_p, id_p   the first hit's normal, t (the primary direction is not normalised, so t is proportional to
 *          depth along the view axis) and object id (0 = miss): rc_primary_aov's precision-32 values, from the centre ray
 *          of the pixel (fixed jitter).
 * Every input is rounded to fp32; the filter runs in fp32.
 *   Demodulate: a_p = max(alb_p, 1e-3) per channel, c_p = m_p / a_p, abar_p = mean(a_p), var_p = v_p / abar_p^2;
 *     l = (c.r + c.g + c.b) / 3.
 *   Level k = 0 .. levels-1, step s = 2^k: taps q = p + s (i, j), i, j in -2..2; taps outside the image are skipped.
 *     g_p = 3x3 blur of var with weights [1/4, 1/2, 1/4]^2 over the in-image pixels around p (unit spacing),
 *       renormalised by the weights used, no id test; recomputed from each level's input var.
 *     w(p, q) = h(i) h(j) [id_p == id_q] w_l w_n w_z, h = [1/16, 1/4, 3/8, 1/4, 1/16],
 *       w_l = exp(-|l_p - l_q| / (sigma_l sqrt(g_p) + 1e-3)), w_n = max(0, n_p . n_q)^sigma_n,
 *       w_z = exp(-|z_p - z_q| / (sigma_z z_p |(i, j)| s / H)); w_n = w_z = 1 for q = p and where id_p = 0.
 *     c'_p = sum w c_q / sum w, var'_p = sum w^2 var_q / (sum w)^2 (the centre tap keeps sum w >= (3/8)^2).
 *   Remodulate and gamma: out_p = sqrt(max(0, a_p c_p)) per channel — rc_render's units.  levels = 0 gives the noisy
 *   image up to rounding.
 * out_rgb: width*height*3 doubles.  aux (may be NULL; each of its pointers may be NULL): the filter's inputs in f64 as
 * this call built them — mean (W*H*3), var (W*H), albedo (W*H*3), normal (W*H*3), depth (W*H; DBL_MAX for a miss),
 * id (W*H) — so rc_denoise_filter on them gives the same out_rgb bit for bit.
 * rc_get_stats: samples = W*H*S; segments, gpu_ms and kernel_launches of the whole call (render, guides, filter);
 * specialized as for rc_render.  `cancel`: as for rc_render (checked at entry and relayed during the render; a
 * cancelled call writes nothing).  Supported: a one-device context, world <= 1, the megakernel, the direct sampler,
 * 10 Philox rounds, samples >= 2; specialize as for rc_render.  Anything else is RC_ERR_INVALID, and so are levels
 * outside 0..10, sigma_l <= 0, sigma_z <= 0, sigma_n < 0 and any sigma that is not finite. */
typedef struct rc_denoise {
    int32_t levels;        /* à-trous levels, 0..10 (SVGF: 5)                                          */
    int32_t reserved;
    double  sigma_l;       /* luminance edge stop, > 0 (SVGF: 4)                                        */
    double  sigma_n;       /* normal edge stop exponent, >= 0 (SVGF: 128)                               */
    double  sigma_z;       /* depth edge stop, > 0 (SVGF: 1)                                            */
} rc_denoise;

typedef struct rc_denoise_aux {   /* optional outputs of rc_render_denoised; any may be NULL */
    double*   mean;
    double*   var;
    double*   albedo;
    double*   normal;
    double*   depth;
    uint32_t* id;
} rc_denoise_aux;

int rc_render_denoised(rc_ctx* ctx, const rc_params* params, const rc_denoise* denoise, double* out_rgb,
                       const rc_denoise_aux* aux, const volatile int32_t* cancel);

/* The filter of rc_render_denoised on the caller's inputs (layouts as rc_denoise_aux; depth must be finite and > 0
 * where id != 0), on device 0 of the context; needs no scene.  rc_get_stats: gpu_ms of the filter's kernels (not the
 * copies), kernel_launches = 2 + levels, samples = 0.  Same parameter checks as rc_render_denoised. */
int rc_denoise_filter(rc_ctx* ctx, const rc_denoise* denoise, int32_t width, int32_t height, const double* mean,
                      const double* var, const double* albedo, const double* normal, const double* depth,
                      const uint32_t* id, double* out_rgb);

/* The whole of CpuRendererScaled::render (src/renderer/cpu_scaled.rs:37-121), the preview renderer
 * (`preview_renderer`, src/config.rs:203-207, used while the camera moves, src/main.rs:174-190).
 * params->width/height are the screen; params->samples / max_depth come from config.preview
 * (src/config.rs:75-82).  One colour is traced per scale_w x scale_h block of screen pixels — u from
 * the block's left column with one jitter per block, v from its top row with one jitter per sample
 * (cpu_scaled.rs:55-60) — and, after scale_sqrt, fills the block (cpu_scaled.rs:75-86).  scale_w and
 * scale_h are what CpuRendererScaled::new derives (cpu_scaled.rs:31-34: the highest divisor of
 * image.width / num_threads_width not above config.preview.scale); columns / rows beyond the last
 * whole block stay 0 as in the reference.  out_rgb: width*height*3 doubles.  Cancel semantics and the
 * share of params->rank / params->world (over the grid of blocks) as rc_render. */
int rc_render_preview(rc_ctx* ctx, const rc_params* params, int32_t scale_w, int32_t scale_h,
                      double* out_rgb, const volatile int32_t* cancel);

/* Device-resident form for callers that own device memory (bench, multi-
 * process jobs): traces this participant's share (params->rank/world) and
 * ADDS linear radiance sums into d_accum (width*height*3 floats on device 0;
 * pixels outside the share are left untouched).  No host transfer. */
int rc_render_accumulate(rc_ctx* ctx, const rc_params* params, float* d_accum,
                         const volatile int32_t* cancel);

/* Tile split across the GPUs of one box without an exchange step: this participant's tiles
 * (params->rank / params->world, RC_SPLIT_TILES, megakernel) are traced and their radiance sums
 * STORED into d_image (width*height*3 floats), which may live on ANOTHER GPU — a buffer opened
 * with rc_shared_open, or device 0's buffer when the context spans several devices.  Every pixel is
 * owned by exactly one participant, so after all of them have finished (the caller's barrier)
 * d_image holds the whole frame: the gather of SURVEY §8(e) ("tiles are gathered peer-to-peer")
 * happens inside the render kernel, over NVLink, as each tile completes. */
int rc_render_tiles_into(rc_ctx* ctx, const rc_params* params, float* d_image,
                         const volatile int32_t* cancel);

/* A device buffer on device 0 of `ctx` that the other processes of the box can map (CUDA IPC):
 * rc_shared_alloc creates it (zero-filled) and returns the 64-byte handle to pass on (any byte
 * channel: a file, a pipe, a broadcast); rc_shared_open maps it into the calling process with peer
 * access to its GPU; rc_shared_close unmaps / frees.  The one-process-per-GPU form of the tile-split
 * gather (the reference itself is a single process, so this has no counterpart there). */
int rc_shared_alloc(rc_ctx* ctx, uint64_t bytes, void** d_ptr, uint8_t handle[64]);
int rc_shared_open(rc_ctx* ctx, const uint8_t handle[64], void** d_ptr);
int rc_shared_close(rc_ctx* ctx, void* d_ptr);

/* ---- the tile-split render of one box with one process per GPU, whole, behind the ABI ------------------------
 * (SURVEY §8(e): "tile k -> GPU k mod N ... gather disjoint tiles to rank 0 ... direct remote stores into rank 0's
 * buffer".  The reference is one process — CpuRenderer::render, src/renderer/cpu.rs:118-131, hands its tiles to a
 * rayon pool and every tile is written into one ScreenBuffer (src/image_buffer.rs:147-170); this is that, with GPUs
 * for pool threads and rank 0's frame for the ScreenBuffer.)
 *
 * rank 0 creates the frame: ONE allocation on its device 0 holding two width*height*3 float images (they
 * alternate, so a rank already tracing the next frame never stores into the one being read) and a line of
 * progress words per rank, and gets the 64-byte handle to pass to the other ranks (any byte channel); they map it
 * with rc_frame_open (CUDA IPC: peer access over NVLink).  rc_frame_close unmaps / frees.
 *
 * rc_render_frame(params with rank / world, megakernel), called by EVERY rank once per frame.  With RC_SPLIT_TILES:
 *   - waits on the device until rank 0 has released the image this frame goes into (rank 0 releases the images of
 *     frames n and n + 1 when its stream reaches its own call n: the other ranks may run one frame ahead of the
 *     slowest rank instead of meeting it at every frame),
 *   - traces this rank's tiles and stores sqrt(sum / samples) — Vec3::scale_sqrt (src/vec3.rs:119-125) folded into
 *     the store — straight into rank 0's image as each tile finishes: the gather happens inside the render kernel,
 *   - publishes "frame f done" in its progress word; rank 0's stream then waits for every rank's word.
 * With RC_SPLIT_SAMPLES (every rank traces its samples of every pixel) the same protocol carries the REDUCE: a rank's
 * kernel stores its partial sums into its own slot of the image (the frame holds one slot per rank and image:
 * 2 * world * width * height * 12 bytes on rank 0), and rank 0, after the wait, adds the slots in rank order and takes
 * sqrt(sum / samples) — deterministic, no ncclReduce.
 * Nothing but kernels and stream-ordered waits is enqueued: no collective library, no host synchronisation.
 * On rank 0, *d_rgb (if not NULL) receives the device pointer of the finished float image (stream-ordered: valid for
 * work enqueued on the context's stream BEFORE the next rc_render_frame — that call hands the image to the ranks for
 * the frame after it); if out_rgb is not NULL the image is
 * widened to f64, copied into it (width*height*3 doubles, like rc_render) and the call returns when it is there.
 * On other ranks both must be NULL.  cancel: as for rc_render (every rank must pass a flag or none). */
typedef struct rc_frame rc_frame;
int rc_frame_create(rc_ctx* ctx, int32_t width, int32_t height, int32_t world, rc_frame** out, uint8_t handle[64]);
int rc_frame_open(rc_ctx* ctx, const uint8_t handle[64], int32_t width, int32_t height, int32_t rank, int32_t world,
                  rc_frame** out);
int rc_frame_close(rc_ctx* ctx, rc_frame* frame);
int rc_render_frame(rc_ctx* ctx, const rc_params* params, rc_frame* frame, const float** d_rgb, double* out_rgb,
                    const volatile int32_t* cancel);

/* scale_sqrt on a device accumulation buffer: d_rgb[i] = sqrt(d_accum[i] /
 * samples) (src/vec3.rs:119-125).  d_rgb may alias d_accum. */
int rc_finalize(rc_ctx* ctx, const float* d_accum, int32_t width, int32_t height,
                int32_t samples, float* d_rgb);

/* Tone map + quantise a gamma'd image: ScreenBuffer::update
 * (src/image_buffer.rs:147-153) followed by the RGBA packer of
 * src/image_action/png.rs:21-31 — `(v*255.0) as u32` per channel, no clamp,
 * (r<<24)|(g<<16)|(b<<8)|255 written big-endian.  rgb is host memory
 * (width*height*3 doubles); rgba receives width*height*4 bytes.  rgb_out
 * (optional) receives the tone-mapped doubles. */
int rc_postprocess(rc_ctx* ctx, const rc_tone_map* tm, const double* rgb,
                   int32_t width, int32_t height, uint8_t* rgba, double* rgb_out);

/* Primary-visibility AOV: one ray per pixel through the same ray-gen and
 * closest-hit code as the renderer, with the fixed jitter (pixel centre,
 * lens centre).  Mirrors the RayImageData fields of src/renderer.rs:33-39.
 * precision: 32 = the renderer's fp32 intersectors, 64 = the same code
 * instantiated in f64.  Outputs (any may be NULL): id[w*h] canonical object
 * id (0 = miss), t[w*h] (f64::MAX on a miss, as renderer.rs:85),
 * normal[w*h*3], point[w*h*3]. */
int rc_primary_aov(rc_ctx* ctx, const rc_params* params, int32_t precision,
                   uint32_t* id, double* t, double* normal, double* point);

int rc_get_stats(rc_ctx* ctx, rc_stats* out);

/* The CUDA source rc_params.specialize compiles for this scene (host only; for
 * inspection and tests).  Returns its length, writes at most capacity-1 bytes
 * and a terminator to `out` (may be NULL). */
int64_t rc_spec_source(const rc_scene* scene, char* out, int64_t capacity);

/* The share of participant `part` of `parts` under params->split, as the
 * kernels will trace it (pure host arithmetic, no device needed): interleaved
 * 16x8-pixel tiles `tile_first + k * tile_stride`, k < n_tiles, of a
 * tiles_x-wide tile grid, and the sample range [s_begin, s_end).  The tile
 * grid plays the role of CpuRenderer::prepare_threads (src/renderer/cpu.rs:
 * 73-115); out = {tile_first, tile_stride, n_tiles, tiles_x, tile_w, tile_h,
 * s_begin, s_end}. */
int rc_partition(const rc_params* params, int32_t part, int32_t parts, int32_t out[8]);

/* FP32 (non-tensor) FMA micro-benchmark on device 0: the roofline denominator
 * of SURVEY §8(d).  Returns achieved TFLOP/s (FMA = 2 flop) of a register-only
 * FFMA loop filling every SM, and the SM clock implied by it. */
int rc_fp32_peak(rc_ctx* ctx, double* tflops, double* lane_ginstr_per_s);

/* Text of the last error raised on the calling thread ("" if none). */
const char* rc_last_error(void);

/* RC_ABI_VERSION the library was built with. */
int rc_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RACER_CUDA_H */
