#!/usr/bin/env python
"""Image quality per GPU-millisecond: uniform renders against adaptive sampling (rc_render_adaptive).

For each scene a reference is rendered uniformly at 8192 spp with a seed of its own.  Against it, uniform renders at
64 .. 1024 spp and adaptive renders (S = 4096, n0 = 16, four thresholds) report: pixel-samples traced, GPU ms of the
call (CUDA events, median of alternating runs after a warm-up), RMSE and 99.9th-percentile error of the gamma'd image,
the share of RGBA bytes that differ after tone map and quantisation, and (adaptive) the kernel times of each round
from torch.profiler in a separate run.  The card's name and power limit are read in the same run.

    python tools/adaptive_quality.py [--out profiles/r03_adaptive_quality.json] [--reps 3] [--quick]

--quick: tiny images and sample counts, for a rehearsal of the script itself (numbers meaningless).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from conftest import scene_path  # noqa: E402
from racer_tracer_b200 import harness  # noqa: E402

SCENES = [("cornell_box", 1920, 1080), ("three_balls", 600, 600), ("noise_and_textures", 600, 600), ("random", 1920, 1080)]
UNIFORM = [64, 128, 256, 512, 1024]
THRESHOLDS = [0.02, 0.01, 0.005, 0.0025]
S_MAX, N0 = 4096, 16
REF_SPP, REF_SEED, SEED = 8192, 424242, 7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def quality(img, ref, rgba, rgba_ref):
    d = np.abs(img - ref)
    return {"rmse": float(np.sqrt((d * d).mean())), "p999": float(np.quantile(d, 0.999)),
            "rgba_bytes_differ": float((rgba != rgba_ref).mean())}


def round_kernels(r, p, threshold):
    """Kernel names and times (ms) of one adaptive call, in launch order, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r.render_adaptive(p, threshold, N0)
    evs = [e for e in prof.events() if e.device_type.name == "CUDA" and "memset" not in e.name.lower() and "memcpy" not in e.name.lower()]
    evs.sort(key=lambda e: e.time_range.start)
    return [[e.name[:60], round(e.device_time_total / 1000.0 if hasattr(e, "device_time_total") else e.cuda_time_total / 1000.0, 4)] for e in evs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_adaptive_quality.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    scenes, uniform, s_max, ref_spp = SCENES, UNIFORM, S_MAX, REF_SPP
    if a.quick:
        scenes = [(n, 64, 48) for n, _, _ in SCENES]
        uniform, s_max, ref_spp = [16, 32], 64, 256
    cfg = harness.load_config(os.path.join(ROOT, "tests", "golden", "config.yml"))
    depth = cfg.render.max_depth
    r = harness.CudaRenderer([0])
    out = {"card": card(), "depth": depth, "reference_spp": ref_spp, "s_max": s_max, "n0": N0, "scenes": {}}
    print(out["card"], flush=True)
    for name, w, h in scenes:
        job = harness.prepare_job(scene_path(name), cfg, w, h)
        r.upload(job)
        t0 = time.time()
        ref = r.render(harness.make_params(w, h, ref_spp, depth, seed=REF_SEED, specialize=2))
        rgba_ref = r.postprocess(job.tone_map, ref)[0]
        runs = [("uniform", n, None) for n in uniform] + [("adaptive", s_max, t) for t in THRESHOLDS]

        def run(kind, n, t):
            p = harness.make_params(w, h, n, depth, seed=SEED, specialize=2)
            if kind == "uniform":
                return r.render(p), None, r.stats()
            rgb, spp, _ = r.render_adaptive(p, t, N0)
            return rgb, spp, r.stats()

        for spec in runs:   # warm-up: kernels compiled and loaded, buffers allocated
            run(*spec)
        ms = {spec: [] for spec in runs}
        last = {}
        for _ in range(a.reps):   # alternating: every configuration once per pass
            for spec in runs:
                img, spp, st = run(*spec)
                ms[spec].append(st.gpu_ms)
                last[spec] = (img, spp, st)
        rows = []
        for spec in runs:
            kind, n, t = spec
            img, spp, st = last[spec]
            row = {"kind": kind, "spp": n, "threshold": t, "samples": int(st.samples), "specialized": int(st.specialized),
                   "gpu_ms": float(np.median(ms[spec])), "gpu_ms_runs": [round(x, 3) for x in ms[spec]]}
            row.update(quality(img, ref, r.postprocess(job.tone_map, img)[0], rgba_ref))
            if kind == "adaptive":
                row["spp_hist"] = {int(k): int(v) for k, v in zip(*np.unique(spp, return_counts=True))}
                try:
                    row["kernels"] = round_kernels(r, harness.make_params(w, h, n, depth, seed=SEED, specialize=2), t)
                except Exception as e:   # the measurement above stands without the per-round split
                    row["kernels"] = f"not measured: {e!r}"
            rows.append(row)
            print(f"{name} {kind:8s} spp={n:5d} thr={t} samples={row['samples']:.3e} ms={row['gpu_ms']:.2f} "
                  f"rmse={row['rmse']:.5f} p999={row['p999']:.4f} rgba={row['rgba_bytes_differ']:.4f}", flush=True)
        out["scenes"][name] = {"width": w, "height": h, "rows": rows, "wall_s": round(time.time() - t0, 1)}
    r.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
