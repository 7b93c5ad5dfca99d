//! Raw bindings to `include/racer_cuda.h` (RC_ABI_VERSION 2).  Field order and types follow the
//! header exactly; `tests/test_abi.py::test_struct_layouts_match_the_header` pins the sizes the
//! C compiler sees.  NOT COMPILED in this repository's CI: the build image has no Rust toolchain.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const RC_OK: c_int = 0;
pub const RC_ERR_INVALID: c_int = -1;
pub const RC_ERR_NO_DEVICE: c_int = -2;
pub const RC_ERR_CUDA: c_int = -3;
pub const RC_ERR_STATE: c_int = -4;
pub const RC_ERR_CANCELLED: c_int = -5;
pub const RC_ERR_NCCL: c_int = -6;

pub const RC_PRIM_SPHERE: i32 = 0;
pub const RC_PRIM_XY_RECT: i32 = 1;
pub const RC_PRIM_XZ_RECT: i32 = 2;
pub const RC_PRIM_YZ_RECT: i32 = 3;
pub const RC_PRIM_MOVING_SPHERE: i32 = 4;
pub const RC_MAT_LAMBERTIAN: i32 = 0;
pub const RC_MAT_METAL: i32 = 1;
pub const RC_MAT_DIELECTRIC: i32 = 2;
pub const RC_MAT_DIFFUSE_LIGHT: i32 = 3;
pub const RC_TEX_SOLID: i32 = 0;
pub const RC_TEX_CHECKER: i32 = 1;
pub const RC_TEX_IMAGE: i32 = 2;
pub const RC_TEX_NOISE: i32 = 3;
pub const RC_BG_SKY: i32 = 0;
pub const RC_BG_SOLID: i32 = 1;
pub const RC_VARIANT_MEGAKERNEL: i32 = 0;
pub const RC_VARIANT_WAVEFRONT: i32 = 1;
pub const RC_SAMPLER_DIRECT: i32 = 0;
pub const RC_SAMPLER_REJECTION: i32 = 1;
pub const RC_SPLIT_TILES: i32 = 0;
pub const RC_SPLIT_SAMPLES: i32 = 1;

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_material { pub type_: i32, pub texture: i32, pub param: f64 }

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_texture { pub type_: i32, pub a: i32, pub b: i32, pub reserved: i32, pub color: [f64; 3], pub scale: f64 }

#[repr(C)] #[derive(Clone, Copy)]
pub struct rc_image { pub width: i32, pub height: i32, pub rgba: *const u8 }

#[repr(C)] #[derive(Clone, Copy)]
pub struct rc_perlin { pub ran_vec: [[f64; 3]; 256], pub perm_x: [i32; 256], pub perm_y: [i32; 256], pub perm_z: [i32; 256] }

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_instance { pub flags: i32, pub reserved: i32, pub sin_theta: f64, pub cos_theta: f64, pub offset: [f64; 3] }

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_bvh_node { pub bmin: [f64; 3], pub bmax: [f64; 3], pub left: i32, pub right: i32 }

#[repr(C)]
pub struct rc_scene {
    pub n_prims: i32,
    pub prim_type: *const i32,
    pub prim_data: *const f64,
    pub prim_material: *const i32,
    pub prim_id: *const u32,
    pub prim_instance: *const i32,
    pub prim_aabb: *const f64,
    pub n_instances: i32, pub instances: *const rc_instance,
    pub n_materials: i32, pub materials: *const rc_material,
    pub n_textures: i32, pub textures: *const rc_texture,
    pub n_images: i32, pub images: *const rc_image,
    pub n_perlin: i32, pub perlin: *const rc_perlin,
    pub n_nodes: i32, pub nodes: *const rc_bvh_node,
    pub bg_type: i32, pub reserved: i32,
    pub bg_a: [f64; 3], pub bg_b: [f64; 3],
    pub prim_motion: *const f64,   // ABI 2: 5 per prim (pos_b, time_a, time_b) for RC_PRIM_MOVING_SPHERE; may be null
}

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_camera {
    pub origin: [f64; 3], pub upper_left_corner: [f64; 3], pub forward: [f64; 3], pub right: [f64; 3],
    pub up: [f64; 3], pub horizontal: [f64; 3], pub vertical: [f64; 3],
    pub vfov: f64, pub viewport_width: f64, pub viewport_height: f64, pub lens_radius: f64,
    pub focus_distance: f64, pub time_a: f64, pub time_b: f64,
}

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_params {
    pub width: i32, pub height: i32, pub samples: i32, pub max_depth: i32, pub seed: u64,
    pub variant: i32, pub sampler: i32, pub split: i32, pub tile_w: i32, pub tile_h: i32,
    pub rank: i32, pub world: i32, pub fixed_jitter: i32, pub rng_rounds: i32, pub specialize: i32,
}

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rc_stats {
    pub gpu_ms: f64, pub samples: u64, pub segments: u64, pub kernel_launches: u64,
    pub n_devices: i32, pub sm_count: i32, pub sm_clock_khz: i32, pub specialized: i32,
}

/// rc_render_adaptive: samples every pixel gets before its first test, and the error estimate that stops it.
#[repr(C)] #[derive(Clone, Copy)]
pub struct rc_adaptive {
    pub min_samples: i32, pub reserved: i32, pub threshold: f64,
}

/// rc_render_denoised / rc_denoise_filter: the à-trous filter's levels and edge-stopping parameters.
#[repr(C)] #[derive(Clone, Copy)]
pub struct rc_denoise {
    pub levels: i32, pub reserved: i32, pub sigma_l: f64, pub sigma_n: f64, pub sigma_z: f64,
}

/// rc_render_denoised: optional outputs, the filter's inputs as the call built them (any pointer may be null).
#[repr(C)] #[derive(Clone, Copy)]
pub struct rc_denoise_aux {
    pub mean: *mut f64, pub var: *mut f64, pub albedo: *mut f64, pub normal: *mut f64, pub depth: *mut f64, pub id: *mut u32,
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct rc_tone_map {
    pub type_: i32, pub reserved: i32, pub max_white: f64, pub hable: [f64; 6], pub exposure_bias: f64,
    pub linear_white_point: f64, pub aces_in: [f64; 9], pub aces_out: [f64; 9],
}
pub const RC_TONE_NONE: i32 = 0;
pub const RC_TONE_REINHARD: i32 = 1;
pub const RC_TONE_HABLE: i32 = 2;
pub const RC_TONE_ACES: i32 = 3;

#[repr(C)] pub struct rc_ctx { _private: [u8; 0] }
#[repr(C)] pub struct rc_frame { _private: [u8; 0] }

extern "C" {
    pub fn rc_create(devices: *const i32, n: i32, out: *mut *mut rc_ctx) -> c_int;
    pub fn rc_destroy(ctx: *mut rc_ctx) -> c_int;
    pub fn rc_set_stream(ctx: *mut rc_ctx, cuda_stream: *mut c_void) -> c_int;
    pub fn rc_upload_scene(ctx: *mut rc_ctx, scene: *const rc_scene) -> c_int;
    pub fn rc_set_camera(ctx: *mut rc_ctx, camera: *const rc_camera) -> c_int;
    pub fn rc_build_lbvh(ctx: *mut rc_ctx) -> c_int;
    pub fn rc_get_bvh(ctx: *mut rc_ctx, nodes: *mut rc_bvh_node, node_capacity: i32, prim_order: *mut i32, prim_capacity: i32) -> c_int;
    pub fn rc_render(ctx: *mut rc_ctx, params: *const rc_params, out_rgb: *mut f64, cancel: *const i32) -> c_int;
    pub fn rc_render_adaptive(ctx: *mut rc_ctx, params: *const rc_params, a: *const rc_adaptive, out_rgb: *mut f64, out_spp: *mut i32,
                              out_err: *mut f64, cancel: *const i32) -> c_int;
    pub fn rc_render_denoised(ctx: *mut rc_ctx, params: *const rc_params, denoise: *const rc_denoise, out_rgb: *mut f64,
                              aux: *const rc_denoise_aux, cancel: *const i32) -> c_int;
    pub fn rc_denoise_filter(ctx: *mut rc_ctx, denoise: *const rc_denoise, width: i32, height: i32, mean: *const f64, var: *const f64,
                             albedo: *const f64, normal: *const f64, depth: *const f64, id: *const u32, out_rgb: *mut f64) -> c_int;
    pub fn rc_render_preview(ctx: *mut rc_ctx, params: *const rc_params, scale_w: i32, scale_h: i32, out_rgb: *mut f64,
                             cancel: *const i32) -> c_int;
    pub fn rc_render_tiles_into(ctx: *mut rc_ctx, params: *const rc_params, d_image: *mut f32, cancel: *const i32) -> c_int;
    pub fn rc_shared_alloc(ctx: *mut rc_ctx, bytes: u64, d_ptr: *mut *mut c_void, handle: *mut u8) -> c_int;
    pub fn rc_shared_open(ctx: *mut rc_ctx, handle: *const u8, d_ptr: *mut *mut c_void) -> c_int;
    pub fn rc_shared_close(ctx: *mut rc_ctx, d_ptr: *mut c_void) -> c_int;
    pub fn rc_render_accumulate(ctx: *mut rc_ctx, params: *const rc_params, d_accum: *mut f32, cancel: *const i32) -> c_int;
    pub fn rc_finalize(ctx: *mut rc_ctx, d_accum: *const f32, width: i32, height: i32, samples: i32, d_rgb: *mut f32) -> c_int;
    pub fn rc_postprocess(ctx: *mut rc_ctx, tone_map: *const rc_tone_map, rgb: *const f64, width: i32, height: i32,
                          rgba: *mut u8, rgb_out: *mut f64) -> c_int;
    pub fn rc_frame_create(ctx: *mut rc_ctx, width: i32, height: i32, world: i32, out: *mut *mut rc_frame, handle: *mut u8) -> c_int;
    pub fn rc_frame_open(ctx: *mut rc_ctx, handle: *const u8, width: i32, height: i32, rank: i32, world: i32,
                         out: *mut *mut rc_frame) -> c_int;
    pub fn rc_frame_close(ctx: *mut rc_ctx, frame: *mut rc_frame) -> c_int;
    pub fn rc_render_frame(ctx: *mut rc_ctx, params: *const rc_params, frame: *mut rc_frame, d_rgb: *mut *const f32,
                           out_rgb: *mut f64, cancel: *const i32) -> c_int;
    pub fn rc_primary_aov(ctx: *mut rc_ctx, params: *const rc_params, precision: i32, id: *mut u32, t: *mut f64,
                          normal: *mut f64, point: *mut f64) -> c_int;
    pub fn rc_partition(params: *const rc_params, part: i32, parts: i32, out: *mut i32) -> c_int;
    pub fn rc_get_stats(ctx: *mut rc_ctx, out: *mut rc_stats) -> c_int;
    pub fn rc_spec_source(scene: *const rc_scene, out: *mut c_char, capacity: i64) -> i64;
    pub fn rc_fp32_peak(ctx: *mut rc_ctx, tflops: *mut f64, lane_ginstr_per_s: *mut f64) -> c_int;
    pub fn rc_last_error() -> *const c_char;
    pub fn rc_abi_version() -> c_int;
}
