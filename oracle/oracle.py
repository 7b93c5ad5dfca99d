"""ctypes binding of liboracle.so — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs import this module (see oracle/oracle.h).  The product
package never does.  Parity is UNPINNED at the bit level by the reference (no
render tests exist there, and it cannot be built here); tests/test_oracle_kat.py
pins the oracle with hand-derived known-answer vectors, and
tests/test_reference_renders.py statistically with the reference's published
renders.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from racer_tracer_b200.capi import rc_camera, rc_params, rc_perlin, rc_scene, rc_tone_map

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liboracle.so")

RNG_PHILOX, RNG_SEQUENTIAL = 0, 1
CF_PER_SAMPLE_U = 1   # oracle.h ORACLE_CF_PER_SAMPLE_U: NOT the reference (Q1 counterfactual)


class oracle_counters(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("segments", C.c_uint64), ("node_tests", C.c_uint64),
                ("prim_tests", C.c_uint64 * 4), ("prim_hits", C.c_uint64 * 4),
                ("scatters", C.c_uint64 * 4), ("tex_evals", C.c_uint64 * 4),
                ("background", C.c_uint64), ("depth_exhausted", C.c_uint64),
                ("rejection_iters", C.c_uint64), ("noise_calls", C.c_uint64)]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else int(v)
        return d


class oracle_options(C.Structure):
    _fields_ = [("rng", C.c_int32), ("threads", C.c_int32), ("tiles_w", C.c_int32),
                ("tiles_h", C.c_int32), ("sample_begin", C.c_int32), ("sample_count", C.c_int32),
                ("linear_sum", C.c_int32), ("counterfactual", C.c_int32)]


def build(force: bool = False) -> str:
    """Compile liboracle.so with oracle/Makefile if it is missing or stale."""
    src = [os.path.join(HERE, f) for f in ("oracle.cpp", "oracle.h")] + \
          [os.path.join(HERE, "..", "include", "racer_cuda.h")]
    stale = force or not os.path.exists(LIB_PATH) or \
        any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in src)
    if stale:
        subprocess.run(["make", "-C", HERE, "-B", "liboracle.so"], check=True, capture_output=True)
    return LIB_PATH


_lib = None
_d3 = C.c_double * 3
_pd = C.POINTER(C.c_double)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.oracle_render.argtypes = [C.POINTER(rc_scene), C.POINTER(rc_camera), C.POINTER(rc_params),
                                    C.POINTER(oracle_options), _pd, C.POINTER(oracle_counters)]
        L.oracle_render_preview.argtypes = [C.POINTER(rc_scene), C.POINTER(rc_camera), C.POINTER(rc_params),
                                            C.POINTER(oracle_options), C.c_int32, C.c_int32, _pd]
        L.oracle_primary_aov.argtypes = [C.POINTER(rc_scene), C.POINTER(rc_camera), C.POINTER(rc_params),
                                         C.POINTER(C.c_uint32), _pd, _pd, _pd]
        L.oracle_sample_radiance.argtypes = [C.POINTER(rc_scene), C.POINTER(rc_camera), C.POINTER(rc_params),
                                             C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), _pd,
                                             C.POINTER(C.c_int32)]
        L.oracle_camera_new.argtypes = [_d3, _d3, _d3] + [C.c_double] * 6 + [C.POINTER(rc_camera)]
        L.oracle_camera_new.restype = None
        L.oracle_tone_map.argtypes = [C.POINTER(rc_tone_map), _pd, C.c_int64, _pd]
        L.oracle_tone_map.restype = None
        L.oracle_quantise_rgba.argtypes = [_pd, C.c_int64, C.POINTER(C.c_uint8)]
        L.oracle_quantise_rgba.restype = None
        L.oracle_philox4x32.argtypes = [C.c_uint32 * 4, C.c_uint32 * 2, C.c_int32, C.c_uint32 * 4]
        L.oracle_philox4x32.restype = None
        L.oracle_philox2x32.argtypes = [C.c_uint32 * 2, C.c_uint32, C.c_int32, C.c_uint32 * 2]
        L.oracle_philox2x32.restype = None
        L.oracle_aabb_hit.argtypes = [_d3, _d3, _d3, _d3, C.c_double, C.c_double]
        L.oracle_prim_hit.argtypes = [C.POINTER(rc_scene), C.c_int32, _d3, _d3, C.c_double, C.c_double,
                                      C.c_double * 10]
        L.oracle_scene_hit.argtypes = [C.POINTER(rc_scene), _d3, _d3, C.c_double, C.c_double, C.c_double * 10]
        L.oracle_reflectance.argtypes = [C.c_double, C.c_double]
        L.oracle_reflectance.restype = C.c_double
        L.oracle_reflect.argtypes = [_d3, _d3, _d3]
        L.oracle_reflect.restype = None
        L.oracle_refract.argtypes = [_d3, _d3, C.c_double, _d3]
        L.oracle_refract.restype = None
        L.oracle_texture_value.argtypes = [C.POINTER(rc_scene), C.c_int32, C.c_double, C.c_double, _d3, _d3]
        L.oracle_texture_value.restype = None
        L.oracle_perlin_noise.argtypes = [C.POINTER(rc_perlin), _d3]
        L.oracle_perlin_noise.restype = C.c_double
        L.oracle_perlin_turbulence.argtypes = [C.POINTER(rc_perlin), _d3, C.c_int32]
        L.oracle_perlin_turbulence.restype = C.c_double
        L.oracle_background.argtypes = [C.POINTER(rc_scene), _d3, _d3]
        L.oracle_background.restype = None
        L.oracle_get_ray.argtypes = [C.POINTER(rc_camera)] + [C.c_double] * 4 + [_d3, _d3]
        L.oracle_get_ray.restype = None
        L.oracle_vec3_op.argtypes = [C.c_int32, _d3, _d3, _d3]
        L.oracle_vec3_op.restype = None
        _lib = L
    return _lib


def d3(v):
    return _d3(*[float(x) for x in v])


def render(job, params: rc_params, rng=RNG_PHILOX, threads=0, tiles=(10, 10), sample_begin=0,
           sample_count=0, linear_sum=False, want_counters=False, counterfactual=0):
    """oracle_render over a harness.Job; returns (H,W,3) float64 [and counters].
    counterfactual: CF_* bits, deliberate departures from the reference (tests that must be able to fail)."""
    opt = oracle_options(rng, threads, tiles[0], tiles[1], sample_begin, sample_count, int(linear_sum), int(counterfactual))
    out = np.empty((params.height, params.width, 3), dtype=np.float64)
    cnt = oracle_counters()
    st = lib().oracle_render(job.scene.ptr, C.byref(job.camera), C.byref(params), C.byref(opt),
                             out.ctypes.data_as(_pd), C.byref(cnt))
    if st != 0:
        raise RuntimeError(f"oracle_render failed: {st}")
    return (out, cnt) if want_counters else out


def render_preview(job, params: rc_params, scale_w: int, scale_h: int, rng=RNG_PHILOX, tiles=(10, 10), sample_begin=0,
                   sample_count=0):
    """oracle_render_preview (CpuRendererScaled, cpu_scaled.rs); returns (H,W,3) float64.  sample_begin / sample_count:
    only those samples are traced (a sample share), still scaled by 1 / params.samples."""
    opt = oracle_options(rng, 1, tiles[0], tiles[1], sample_begin, sample_count, 0, 0)
    out = np.empty((params.height, params.width, 3), dtype=np.float64)
    st = lib().oracle_render_preview(job.scene.ptr, C.byref(job.camera), C.byref(params), C.byref(opt),
                                     scale_w, scale_h, out.ctypes.data_as(_pd))
    if st != 0:
        raise RuntimeError(f"oracle_render_preview failed: {st}")
    return out


def primary_aov(job, params: rc_params):
    n = params.width * params.height
    ids = np.empty(n, dtype=np.uint32)
    t = np.empty(n, dtype=np.float64)
    nrm = np.empty((n, 3), dtype=np.float64)
    pt = np.empty((n, 3), dtype=np.float64)
    st = lib().oracle_primary_aov(job.scene.ptr, C.byref(job.camera), C.byref(params),
                                  ids.ctypes.data_as(C.POINTER(C.c_uint32)), t.ctypes.data_as(_pd),
                                  nrm.ctypes.data_as(_pd), pt.ctypes.data_as(_pd))
    if st != 0:
        raise RuntimeError(f"oracle_primary_aov failed: {st}")
    return ids, t, nrm, pt


def sample_radiance(job, params: rc_params, pixel_idx, sample_idx):
    pixel_idx = np.ascontiguousarray(pixel_idx, dtype=np.int32)
    sample_idx = np.ascontiguousarray(sample_idx, dtype=np.int32)
    n = len(pixel_idx)
    out = np.empty((n, 3), dtype=np.float64)
    seg = np.empty(n, dtype=np.int32)
    st = lib().oracle_sample_radiance(job.scene.ptr, C.byref(job.camera), C.byref(params), n,
                                      pixel_idx.ctypes.data_as(C.POINTER(C.c_int32)),
                                      sample_idx.ctypes.data_as(C.POINTER(C.c_int32)),
                                      out.ctypes.data_as(_pd), seg.ctypes.data_as(C.POINTER(C.c_int32)))
    if st != 0:
        raise RuntimeError(f"oracle_sample_radiance failed: {st}")
    return out, seg


def tone_map(tm: rc_tone_map, rgb: np.ndarray) -> np.ndarray:
    rgb = np.ascontiguousarray(rgb, dtype=np.float64)
    out = np.empty_like(rgb)
    lib().oracle_tone_map(C.byref(tm), rgb.ctypes.data_as(_pd), rgb.size // 3, out.ctypes.data_as(_pd))
    return out


def quantise_rgba(rgb: np.ndarray) -> np.ndarray:
    rgb = np.ascontiguousarray(rgb, dtype=np.float64)
    out = np.empty(rgb.shape[:-1] + (4,), dtype=np.uint8)
    lib().oracle_quantise_rgba(rgb.ctypes.data_as(_pd), rgb.size // 3, out.ctypes.data_as(C.POINTER(C.c_uint8)))
    return out
