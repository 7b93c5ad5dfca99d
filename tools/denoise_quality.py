#!/usr/bin/env python
"""Image quality per GPU-millisecond: uniform renders against denoised renders (rc_render_denoised).

For each scene a reference is rendered uniformly at 8192 spp with a seed of its own.  Against it, uniform renders at
64 .. 1024 spp and denoised renders at 16, 64 and 256 spp (SVGF's parameters: levels 5, sigma_l 4, sigma_n 128,
sigma_z 1) report: pixel-samples traced, GPU ms of the call (CUDA events, median of alternating runs after a warm-up),
RMSE and 99.9th-percentile error of the gamma'd image, and the share of RGBA bytes that differ after tone map and
quantisation.  Then the filter alone (rc_denoise_filter) at 1920x1080 with 5 levels: its kernel time (CUDA events
around the kernels, median of 20 calls), per-kernel times from torch.profiler in a separate run, and the HBM floor of
each kernel (the bytes its buffers force it to move, over 7.7 TB/s).  The card's name and power limit are read in the
same run.

    python tools/denoise_quality.py [--out profiles/r03_denoise_quality.json] [--reps 3] [--quick]

--quick: tiny images and sample counts, for a rehearsal of the script itself (numbers meaningless).
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from adaptive_quality import SCENES, UNIFORM, REF_SPP, REF_SEED, SEED, card, quality  # noqa: E402
from conftest import scene_path  # noqa: E402
from racer_tracer_b200 import harness  # noqa: E402

DENOISED = [16, 64, 256]
HBM_BYTES_PER_S = 7.7e12
# bytes per pixel each kernel must move at least: its inputs read once, its outputs written once
FILTER_BYTES = {"prepare": 11 * 8 + 3 * 16,           # mean, var, albedo, normal, depth (f64) -> three float4
                "level": 16 + 16 + 4 + 16,            # (c, var) and (n, z) float4, the id; (c', var') out
                "finish": 2 * 16 + 3 * 8}             # (c, var), albedo -> rgb f64


def filter_timing(r, w, h, levels, calls):
    rng = np.random.default_rng(0)
    mean = rng.uniform(0.05, 2.0, (h, w, 3))
    var = rng.uniform(0.0, 0.02, (h, w))
    albedo = rng.uniform(0.1, 1.0, (h, w, 3))
    normal = rng.normal(size=(h, w, 3))
    normal /= np.linalg.norm(normal, axis=2, keepdims=True)
    depth = rng.uniform(1.0, 5.0, (h, w))
    ids = (1 + (np.arange(w)[None, :] // 64 + 7 * (np.arange(h)[:, None] // 64))).astype(np.uint32)
    dn = harness.default_denoise(levels)
    args = (mean, var, albedo, normal, depth, ids)
    for _ in range(3):
        r.denoise_filter(*args, denoise=dn)
    ms = []
    for _ in range(calls):
        r.denoise_filter(*args, denoise=dn)
        ms.append(r.stats().gpu_ms)
    n = w * h
    floor_ms = {k: v * n / HBM_BYTES_PER_S * 1e3 for k, v in FILTER_BYTES.items()}
    floor_total = floor_ms["prepare"] + levels * floor_ms["level"] + floor_ms["finish"]
    out = {"width": w, "height": h, "levels": levels, "gpu_ms": float(np.median(ms)), "gpu_ms_runs": [round(x, 4) for x in ms],
           "bytes_per_pixel": FILTER_BYTES, "hbm_floor_ms": {k: round(v, 5) for k, v in floor_ms.items()},
           "hbm_floor_total_ms": round(floor_total, 5)}
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r.denoise_filter(*args, denoise=dn)
        evs = [e for e in prof.events() if e.device_type.name == "CUDA" and "memset" not in e.name.lower()
               and "memcpy" not in e.name.lower()]
        evs.sort(key=lambda e: e.time_range.start)
        out["kernels"] = [[e.name[:40], round((e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total) / 1000.0, 4)]
                          for e in evs]
    except Exception as e:   # the event timing above stands without the per-kernel split
        out["kernels"] = f"not measured: {e!r}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_denoise_quality.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    scenes, uniform, denoised, ref_spp, fw, fh = SCENES, UNIFORM, DENOISED, REF_SPP, 1920, 1080
    if a.quick:
        scenes = [(n, 64, 48) for n, _, _ in SCENES]
        uniform, denoised, ref_spp, fw, fh = [16, 32], [4, 16], 256, 64, 48
    cfg = harness.load_config(os.path.join(ROOT, "tests", "golden", "config.yml"))
    depth = cfg.render.max_depth
    r = harness.CudaRenderer([0])
    dn = harness.default_denoise()
    out = {"card": card(), "depth": depth, "reference_spp": ref_spp,
           "denoise": {"levels": dn.levels, "sigma_l": dn.sigma_l, "sigma_n": dn.sigma_n, "sigma_z": dn.sigma_z}, "scenes": {}}
    print(out["card"], flush=True)
    for name, w, h in scenes:
        job = harness.prepare_job(scene_path(name), cfg, w, h)
        r.upload(job)
        t0 = time.time()
        ref = r.render(harness.make_params(w, h, ref_spp, depth, seed=REF_SEED, specialize=2))
        rgba_ref = r.postprocess(job.tone_map, ref)[0]
        runs = [("uniform", n) for n in uniform] + [("denoised", n) for n in denoised]

        def run(kind, n):
            p = harness.make_params(w, h, n, depth, seed=SEED, specialize=2)
            img = r.render(p) if kind == "uniform" else r.render_denoised(p, dn)
            return img, r.stats()

        for spec in runs:   # warm-up: kernels compiled and loaded, buffers allocated
            run(*spec)
        ms = {spec: [] for spec in runs}
        last = {}
        for _ in range(a.reps):   # alternating: every configuration once per pass
            for spec in runs:
                img, st = run(*spec)
                ms[spec].append(st.gpu_ms)
                last[spec] = (img, st)
        rows = []
        for spec in runs:
            kind, n = spec
            img, st = last[spec]
            row = {"kind": kind, "spp": n, "samples": int(st.samples), "specialized": int(st.specialized),
                   "gpu_ms": float(np.median(ms[spec])), "gpu_ms_runs": [round(x, 3) for x in ms[spec]]}
            row.update(quality(img, ref, r.postprocess(job.tone_map, img)[0], rgba_ref))
            rows.append(row)
            print(f"{name} {kind:8s} spp={n:5d} samples={row['samples']:.3e} ms={row['gpu_ms']:.2f} "
                  f"rmse={row['rmse']:.5f} p999={row['p999']:.4f} rgba={row['rgba_bytes_differ']:.4f}", flush=True)
        out["scenes"][name] = {"width": w, "height": h, "rows": rows, "wall_s": round(time.time() - t0, 1)}
    out["filter"] = filter_timing(r, fw, fh, dn.levels, 20)
    f = out["filter"]
    print(f"filter {fw}x{fh} levels={dn.levels}: {f['gpu_ms']:.4f} ms, HBM floor {f['hbm_floor_total_ms']:.4f} ms; "
          f"kernels {f['kernels']}", flush=True)
    r.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fo:
        json.dump(out, fo, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
