"""ctypes mirror of include/racer_cuda.h and loader of libracer_cuda.so.

The structs below follow the header field for field; `load()` opens the CUDA
library that csrc/build.sh puts next to this file.  There is no fallback: if
the library is missing, or no CUDA device is usable, the calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# RC_CUDA_LIB points at an alternative build of the same library (tuning experiments)
LIB_PATH = os.environ.get("RC_CUDA_LIB", os.path.join(HERE, "libracer_cuda.so"))

RC_OK = 0
RC_ERR_INVALID, RC_ERR_NO_DEVICE, RC_ERR_CUDA, RC_ERR_STATE, RC_ERR_CANCELLED, RC_ERR_NCCL = -1, -2, -3, -4, -5, -6

RC_PRIM_SPHERE, RC_PRIM_XY_RECT, RC_PRIM_XZ_RECT, RC_PRIM_YZ_RECT, RC_PRIM_MOVING_SPHERE = 0, 1, 2, 3, 4
RC_MAT_LAMBERTIAN, RC_MAT_METAL, RC_MAT_DIELECTRIC, RC_MAT_DIFFUSE_LIGHT = 0, 1, 2, 3
RC_TEX_SOLID, RC_TEX_CHECKER, RC_TEX_IMAGE, RC_TEX_NOISE = 0, 1, 2, 3
RC_BG_SKY, RC_BG_SOLID = 0, 1
RC_TONE_NONE, RC_TONE_REINHARD, RC_TONE_HABLE, RC_TONE_ACES = 0, 1, 2, 3
RC_VARIANT_MEGAKERNEL, RC_VARIANT_WAVEFRONT = 0, 1
RC_SAMPLER_DIRECT, RC_SAMPLER_REJECTION = 0, 1
RC_SPLIT_TILES, RC_SPLIT_SAMPLES = 0, 1

c_double3 = C.c_double * 3


class rc_material(C.Structure):
    _fields_ = [("type", C.c_int32), ("texture", C.c_int32), ("param", C.c_double)]


class rc_texture(C.Structure):
    _fields_ = [("type", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("reserved", C.c_int32),
                ("color", c_double3), ("scale", C.c_double)]


class rc_image(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgba", C.POINTER(C.c_uint8))]


class rc_perlin(C.Structure):
    _fields_ = [("ran_vec", (C.c_double * 3) * 256), ("perm_x", C.c_int32 * 256),
                ("perm_y", C.c_int32 * 256), ("perm_z", C.c_int32 * 256)]


class rc_instance(C.Structure):
    _fields_ = [("flags", C.c_int32), ("reserved", C.c_int32), ("sin_theta", C.c_double),
                ("cos_theta", C.c_double), ("offset", c_double3)]


class rc_bvh_node(C.Structure):
    _fields_ = [("bmin", c_double3), ("bmax", c_double3), ("left", C.c_int32), ("right", C.c_int32)]


class rc_scene(C.Structure):
    _fields_ = [
        ("n_prims", C.c_int32),
        ("prim_type", C.POINTER(C.c_int32)),
        ("prim_data", C.POINTER(C.c_double)),
        ("prim_material", C.POINTER(C.c_int32)),
        ("prim_id", C.POINTER(C.c_uint32)),
        ("prim_instance", C.POINTER(C.c_int32)),
        ("prim_aabb", C.POINTER(C.c_double)),
        ("n_instances", C.c_int32), ("instances", C.POINTER(rc_instance)),
        ("n_materials", C.c_int32), ("materials", C.POINTER(rc_material)),
        ("n_textures", C.c_int32), ("textures", C.POINTER(rc_texture)),
        ("n_images", C.c_int32), ("images", C.POINTER(rc_image)),
        ("n_perlin", C.c_int32), ("perlin", C.POINTER(rc_perlin)),
        ("n_nodes", C.c_int32), ("nodes", C.POINTER(rc_bvh_node)),
        ("bg_type", C.c_int32), ("reserved", C.c_int32),
        ("bg_a", c_double3), ("bg_b", c_double3),
        ("prim_motion", C.POINTER(C.c_double)),
    ]


class rc_camera(C.Structure):
    _fields_ = [(n, c_double3) for n in ("origin", "upper_left_corner", "forward", "right", "up",
                                         "horizontal", "vertical")] + \
               [(n, C.c_double) for n in ("vfov", "viewport_width", "viewport_height", "lens_radius",
                                          "focus_distance", "time_a", "time_b")]


class rc_params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("samples", C.c_int32),
                ("max_depth", C.c_int32), ("seed", C.c_uint64), ("variant", C.c_int32),
                ("sampler", C.c_int32), ("split", C.c_int32), ("tile_w", C.c_int32),
                ("tile_h", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32),
                ("fixed_jitter", C.c_int32), ("rng_rounds", C.c_int32), ("specialize", C.c_int32)]


class rc_adaptive(C.Structure):
    _fields_ = [("min_samples", C.c_int32), ("reserved", C.c_int32), ("threshold", C.c_double)]


class rc_tone_map(C.Structure):
    _fields_ = [("type", C.c_int32), ("reserved", C.c_int32), ("max_white", C.c_double),
                ("hable", C.c_double * 6), ("exposure_bias", C.c_double),
                ("linear_white_point", C.c_double), ("aces_in", C.c_double * 9),
                ("aces_out", C.c_double * 9)]


class rc_stats(C.Structure):
    _fields_ = [("gpu_ms", C.c_double), ("samples", C.c_uint64), ("segments", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("n_devices", C.c_int32), ("sm_count", C.c_int32),
                ("sm_clock_khz", C.c_int32), ("specialized", C.c_int32)]


# every symbol include/racer_cuda.h declares
ABI_SYMBOLS = [
    "rc_create", "rc_destroy", "rc_set_stream", "rc_upload_scene", "rc_set_camera", "rc_render",
    "rc_render_preview", "rc_build_lbvh", "rc_get_bvh", "rc_render_tiles_into", "rc_shared_alloc", "rc_shared_open",
    "rc_shared_close", "rc_frame_create", "rc_frame_open", "rc_frame_close", "rc_render_frame",
    "rc_render_accumulate", "rc_finalize", "rc_postprocess", "rc_primary_aov", "rc_get_stats",
    "rc_last_error", "rc_abi_version", "rc_fp32_peak", "rc_partition", "rc_spec_source", "rc_render_adaptive",
]


class RacerCudaError(RuntimeError):
    def __init__(self, status: int, text: str):
        super().__init__(f"libracer_cuda status {status}: {text}")
        self.status = status


_lib = None


def load(path: str | None = None) -> C.CDLL:
    """dlopen libracer_cuda.so and declare the prototypes.  Raises if absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} not found: build it with racer_tracer_b200/csrc/build.sh "
            "(there is no CPU fallback for the render path)")
    lib = C.CDLL(p)
    vp = C.c_void_p
    lib.rc_create.argtypes = [C.POINTER(C.c_int32), C.c_int32, C.POINTER(vp)]
    lib.rc_destroy.argtypes = [vp]
    lib.rc_set_stream.argtypes = [vp, vp]
    lib.rc_upload_scene.argtypes = [vp, C.POINTER(rc_scene)]
    lib.rc_set_camera.argtypes = [vp, C.POINTER(rc_camera)]
    lib.rc_render.argtypes = [vp, C.POINTER(rc_params), C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    lib.rc_render_adaptive.argtypes = [vp, C.POINTER(rc_params), C.POINTER(rc_adaptive), C.POINTER(C.c_double),
                                       C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    lib.rc_render_tiles_into.argtypes = [vp, C.POINTER(rc_params), vp, C.POINTER(C.c_int32)]
    lib.rc_shared_alloc.argtypes = [vp, C.c_uint64, C.POINTER(vp), C.POINTER(C.c_uint8)]
    lib.rc_shared_open.argtypes = [vp, C.POINTER(C.c_uint8), C.POINTER(vp)]
    lib.rc_shared_close.argtypes = [vp, vp]
    lib.rc_frame_create.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp), C.POINTER(C.c_uint8)]
    lib.rc_frame_open.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp)]
    lib.rc_frame_close.argtypes = [vp, vp]
    lib.rc_render_frame.argtypes = [vp, C.POINTER(rc_params), vp, C.POINTER(vp), C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    lib.rc_build_lbvh.argtypes = [vp]
    lib.rc_get_bvh.argtypes = [vp, C.POINTER(rc_bvh_node), C.c_int32, C.POINTER(C.c_int32), C.c_int32]
    lib.rc_render_preview.argtypes = [vp, C.POINTER(rc_params), C.c_int32, C.c_int32, C.POINTER(C.c_double),
                                      C.POINTER(C.c_int32)]
    lib.rc_render_accumulate.argtypes = [vp, C.POINTER(rc_params), vp, C.POINTER(C.c_int32)]
    lib.rc_finalize.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, vp]
    lib.rc_postprocess.argtypes = [vp, C.POINTER(rc_tone_map), C.POINTER(C.c_double), C.c_int32,
                                   C.c_int32, C.POINTER(C.c_uint8), C.POINTER(C.c_double)]
    lib.rc_primary_aov.argtypes = [vp, C.POINTER(rc_params), C.c_int32, C.POINTER(C.c_uint32),
                                   C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.rc_get_stats.argtypes = [vp, C.POINTER(rc_stats)]
    lib.rc_fp32_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.rc_partition.argtypes = [C.POINTER(rc_params), C.c_int32, C.c_int32, C.c_int32 * 8]
    lib.rc_spec_source.argtypes = [C.POINTER(rc_scene), C.c_char_p, C.c_int64]
    lib.rc_last_error.restype = C.c_char_p
    lib.rc_last_error.argtypes = []
    lib.rc_abi_version.argtypes = []
    for name in ABI_SYMBOLS:
        if name != "rc_last_error":
            getattr(lib, name).restype = C.c_int
    lib.rc_spec_source.restype = C.c_int64
    if path is None:
        _lib = lib
    return lib


def check(lib: C.CDLL, status: int) -> None:
    if status != RC_OK:
        raise RacerCudaError(status, lib.rc_last_error().decode("utf-8", "replace"))
