#!/usr/bin/env python
"""bench.py — samples/sec of the render hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          # our CUDA path
    python bench.py --impl reference --gpus N ...          # the CPU oracle (restated reference)
    python bench.py ... --dump-outputs DIR                 # + the image of the last timed step as DIR/*.npy

A "step" is one full render of the workload: every pixel x sample of
cornell_box.yml at 1920x1080, 1024 spp, max_depth 20 (BASELINE configs[3], the
configuration the metric is quoted on; it fits one GPU).  With N > 1 (one
process per GPU under torchrun) the image is split into interleaved 16x8 tiles
(tile k -> rank k mod N); every rank renders all samples of its tiles and its
render kernel STORES the finished pixels straight into rank 0's frame buffer
over NVLink (a CUDA-IPC mapping): the gather happens inside the kernel, what is
left of the exchange step is a per-rank "done" word rank 0's stream waits for.
The sample-split workload (clown) sums partial buffers with an NCCL reduce
instead.  Total work is fixed => "strong" scaling.

`value` is timed with CUDA events on the launching stream with the scene and
camera already resident on the device; `e2e` runs the same step through the
public host call (scene + camera upload, render, download of the gamma'd f64
image into host memory); `e2e_cancel` is the same call the way the reference's
host makes it, with a cancel flag that is never raised (interactive.rs:236-251).
The roofline is the FP32 issue roofline of SURVEY §8(d): algorithmic flops per
sample (cost table x oracle counters) x samples/s over the FFMA micro-benchmark
measured in this run; `roofline.ncu` carries the counters of the committed ncu
capture of the same kernel and configuration (profiles/r02_ncu_bench_kernel.json).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (scene, width, height, spp, max_depth, split)
    "cornell_box_1080p_1024spp": ("cornell_box", 1920, 1080, 1024, 20, "tiles"),
    "clown_4k_4096spp": ("clown", 3840, 2160, 4096, 20, "samples"),
    "three_balls_600_200spp": ("three_balls", 600, 600, 200, 20, "tiles"),
    "emissive_600_200spp": ("emissive", 600, 600, 200, 20, "tiles"),
    "noise_and_textures_600_200spp": ("noise_and_textures", 600, 600, 200, 20, "tiles"),
    # the reference's Random loader (scene/random.rs): ~480 spheres, moving spheres, lens; BVH traversal
    "random_1080p_256spp": ("random", 1920, 1080, 256, 20, "tiles"),
}


def ncu_capture(workload):
    """Counters of the committed `ncu --set full` capture of the dominant kernel at this workload
    (profiles/r02_ncu_bench_kernel.json, written by tools/ncu_bench_json.py from the .ncu-rep): HBM bytes per
    launch, issue-slot and pipe utilisation, active lanes.  None when no capture of that workload is committed."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_bench_kernel.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        return json.load(f).get(workload)


def scene_file(scene):
    return scene if scene == "random" else os.path.join(ROOT, "tests", "golden", "scenes", scene + ".yml")

# Algorithmic FP32 flop cost table, SURVEY.md §8(d) (FMA = 2, SFU = 1)
COST = {
    "raygen_accumulate": 40, "node_test": 27, "sphere_test": 23, "sphere_hit_extra": 30,
    "rect_test": 12, "rect_hit_extra": 20, "lambertian": 50, "metal": 60, "dielectric": 60,
    "emit_terminate": 6, "tex_checker": 9, "tex_image": 8, "tex_noise": 1650, "sky": 21,
}


def flops_per_sample(cnt: dict, bg_is_sky: bool, linear_prims=None) -> float:
    """A = 40 + sum over segments [nodes*27 + prims tested + hit extra + scatter + texture] + terminal.
    linear_prims = (n_spheres, n_rects): brute force over all primitives, N_node = 0 (SURVEY §8(d))."""
    s = cnt["samples"]
    f = COST["raygen_accumulate"] * s
    if linear_prims is None:
        f += COST["node_test"] * cnt["node_tests"]
        f += COST["sphere_test"] * cnt["prim_tests"][0] + COST["rect_test"] * sum(cnt["prim_tests"][1:])
    else:
        f += cnt["segments"] * (COST["sphere_test"] * linear_prims[0] + COST["rect_test"] * linear_prims[1])
    f += COST["sphere_hit_extra"] * cnt["prim_hits"][0] + COST["rect_hit_extra"] * sum(cnt["prim_hits"][1:])
    f += COST["lambertian"] * cnt["scatters"][0] + COST["metal"] * cnt["scatters"][1]
    f += COST["dielectric"] * cnt["scatters"][2] + COST["emit_terminate"] * cnt["scatters"][3]
    f += COST["tex_checker"] * cnt["tex_evals"][1] + COST["tex_image"] * cnt["tex_evals"][2]
    f += COST["tex_noise"] * cnt["tex_evals"][3]
    if bg_is_sky:
        f += COST["sky"] * cnt["background"]
    return f / s


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run_nvml(self):
        """In-process NVML: a sample every 10 ms (nvidia-smi as a subprocess manages one per ~0.3 s, and a timed region
        of a few steps lasts 0.1 - 0.2 s).  Same fields as the nvidia-smi query."""
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        while not self.stop_flag.is_set():
            r = get_reasons(h)
            self.rows.append([str(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)), str(mx), str(N.nvmlDeviceGetPowerUsage(h) / 1000.0)] +
                             ["Active" if r & b else "Not Active" for _, b in bits])
            self.stop_flag.wait(0.01)
        N.nvmlShutdown()

    def run(self):
        try:
            self.run_nvml()
            return
        except Exception:
            pass
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "reasons": reasons, "samples": len(self.rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


DUMP_BYTES = 64 * 10**6 - 4096     # everything --dump-outputs writes, .npy headers included


def dump_outputs(out_dir, image):
    """Write the (H, W, 3) image of the last timed step as out_dir/image.npy.  An image larger than DUMP_BYTES is
    written as a fixed, seeded sample of its pixels instead: image_sample.npy (K, 3) and the sampled pixels' flat
    indices y * W + x, ascending, in image_sample_pixels.npy (float64, exact)."""
    os.makedirs(out_dir, exist_ok=True)
    h, w, c = image.shape
    if image.nbytes <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "image.npy"), image)
        return
    k = DUMP_BYTES // (c * image.itemsize + 8)
    pixels = np.sort(np.random.default_rng(0).choice(h * w, size=k, replace=False))
    np.save(os.path.join(out_dir, "image_sample.npy"), image.reshape(h * w, c)[pixels])
    np.save(os.path.join(out_dir, "image_sample_pixels.npy"), pixels.astype(np.float64))


def device_image(ptr, shape):
    """A float32 CUDA tensor over device memory the library owns (no copy; valid while that memory is)."""
    import torch

    class View:
        __cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "data": (ptr, False), "strides": None,
                                    "version": 2}
    return torch.as_tensor(View(), device="cuda")


def oracle_slice(job, params, spp, threads=0):
    """Time the oracle (restated reference, f64, all host threads) on an spp-slice."""
    from oracle import oracle as O
    t0 = time.perf_counter()
    _, cnt = O.render(job, params, rng=O.RNG_SEQUENTIAL, threads=threads, sample_begin=0, sample_count=spp,
                      linear_sum=True, want_counters=True)
    dt = time.perf_counter() - t0
    return params.width * params.height * spp / dt, dt, cnt.as_dict()


def run_reference(args, wl_name):
    """--impl reference: the reference's CPU algorithm (oracle restatement; the Rust
    reference cannot be built: no cargo/rustc in the image) on all host cores."""
    from racer_tracer_b200 import capi, harness
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    scene, w, h, spp, depth, split = WORKLOADS[wl_name]
    cfg = harness.load_config(os.path.join(ROOT, "tests", "golden", "config.yml"))
    job = harness.prepare_job(scene_file(scene), cfg, w, h)
    params = harness.make_params(w, h, spp, depth, seed=0, sampler=capi.RC_SAMPLER_REJECTION)
    cores = os.cpu_count() or 1
    # bounded sample per step: ~4 s of CPU work, sized from a 2-spp probe of the same frame
    probe, _, _ = oracle_slice(job, params, 2)
    slice_spp = max(2, min(spp, int(round(probe * 4.0 / (w * h)))))
    for _ in range(args.warmup):
        oracle_slice(job, params, 1)
    t = []
    for _ in range(args.steps):
        sps, dt, _ = oracle_slice(job, params, slice_spp)
        t.append(dt)
    total = sum(t)
    value = w * h * slice_spp * args.steps / total
    line = {
        "impl": "reference", "metric": "samples/sec", "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl_name, "scene": scene + ".yml", "width": w, "height": h, "spp": spp,
                   "max_depth": depth},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{slice_spp}-spp slice of the {w}x{h} frame per step, sequential RNG, "
                                   "rejection samplers, 10x10 tile grid (restated reference, f64)"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cornell_box_1080p_1024spp", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default=os.environ.get("RC_VARIANT", "megakernel"), choices=["megakernel", "wavefront"])
    ap.add_argument("--sampler", default="direct", choices=["direct", "rejection"])
    ap.add_argument("--rng-rounds", type=int, default=10)
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (profiling runs only)")
    ap.add_argument("--specialize", type=int, default=int(os.environ.get("RC_SPECIALIZE", "2")), choices=[0, 1, 2],
                    help="2 (default): scene compiled into the megakernel with NVRTC, precompiled kernel if that is impossible "
                         "(which one ran is reported in config.kernel); 1: the same but fail instead; 0: precompiled kernels")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lbvh", action="store_true", help="rebuild the BVH on the GPU (rc_build_lbvh) after the upload")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the image the last timed step computed as DIR/*.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # its sample slice is sized from a timing probe, so two runs need not render the same samples
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        return run_reference(args, args.workload)

    import torch
    import torch.distributed as dist
    from racer_tracer_b200 import capi, harness

    if args.warmup < 3:
        print(f"note: warmup {args.warmup} < 3; numbers from this run are not valid bench values", file=sys.stderr)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the render path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    scene, w, h, spp, depth, split_name = WORKLOADS[args.workload]
    if args.spp > 0:
        spp = args.spp
    split = capi.RC_SPLIT_TILES if split_name == "tiles" else capi.RC_SPLIT_SAMPLES
    cfg = harness.load_config(os.path.join(ROOT, "tests", "golden", "config.yml"))
    job = harness.prepare_job(scene_file(scene), cfg, w, h)
    variant = capi.RC_VARIANT_MEGAKERNEL if args.variant == "megakernel" else capi.RC_VARIANT_WAVEFRONT
    sampler = capi.RC_SAMPLER_DIRECT if args.sampler == "direct" else capi.RC_SAMPLER_REJECTION
    spec = args.specialize if (args.variant == "megakernel" and args.sampler == "direct") else 0

    params = harness.make_params(w, h, spp, depth, seed=0, variant=variant, sampler=sampler, split=split,
                                 rank=rank, world=world, rng_rounds=args.rng_rounds, specialize=spec)

    r = harness.CudaRenderer([local_rank])
    stream = torch.cuda.current_stream()
    r.set_stream(stream.cuda_stream)
    r.upload(job)
    if args.lbvh:
        r.build_lbvh()
    n = w * h * 3
    accum = torch.zeros(n, dtype=torch.float32, device="cuda")
    rgb = torch.empty(n, dtype=torch.float32, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # 256 MiB > 126 MB L2

    launches = [0]

    # Tile split (every N, also 1): the whole exchange lives behind the ABI — rc_frame_create / rc_frame_open /
    # rc_render_frame.  Rank 0 owns the frame (two images, alternating, one slot per rank each) and every rank maps it
    # (CUDA IPC); the render kernel of every rank STORES sqrt(sum / spp) for its tiles into slot 0 over NVLink as they
    # finish, then publishes a progress word that rank 0's stream waits for; no collective library.  bench.py only
    # carries the 64-byte handle to the other ranks.  (RC_BENCH_NCCL_GATHER=1: local buffers + an NCCL reduce instead.)
    # Sample split: the same frame can carry the reduce (every rank stores its partial sums into its own slot, rank 0
    # adds the slots up: RC_BENCH_FRAME_SAMPLES=1); the default is local buffers summed with an NCCL reduce.
    frame = None
    # (the sample split takes the frame with RC_BENCH_FRAME_SAMPLES=1; by default it sums local buffers with an NCCL
    # reduce, which measured 3 % faster on eight GPUs: 56.6 against 58.3 ms per clown frame, DESIGN §8)
    use_frame = (split == capi.RC_SPLIT_TILES and not os.environ.get("RC_BENCH_NCCL_GATHER")) or \
                (split == capi.RC_SPLIT_SAMPLES and bool(os.environ.get("RC_BENCH_FRAME_SAMPLES")))
    if variant == capi.RC_VARIANT_MEGAKERNEL and use_frame:
        if rank == 0:
            frame, handle = r.frame_create(w, h, world)
            hbuf = torch.tensor(list(handle), dtype=torch.uint8, device="cuda")
        else:
            hbuf = torch.empty(64, dtype=torch.uint8, device="cuda")
        if world > 1:
            dist.broadcast(hbuf, 0)
        if rank != 0:
            frame = r.frame_open(bytes(hbuf.cpu().tolist()), w, h, rank, world)

    def step(p=None, want_image=False):
        """One render; with want_image (rank 0) returns the device pointer of its finished (H, W, 3) float image."""
        p = params if p is None else p
        if frame is not None:
            # enqueues only: kernels and stream-ordered waits, no host sync, no collective
            return r.render_frame(p, frame, want_device_ptr=want_image)
        accum.zero_()
        r.render_accumulate(p, accum.data_ptr())
        if world > 1:
            # exchange step: partial sample sums (or, with RC_BENCH_NCCL_GATHER, disjoint tiles) summed onto rank 0
            dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            r.finalize(accum.data_ptr(), w, h, spp, rgb.data_ptr())
        return rgb.data_ptr()

    def launches_per_step():
        """Our kernels per step: the render call's own launches (read back after a step), + the zero-fill of the
        accumulation buffer when there is one, + finalize on rank 0."""
        if frame is not None:
            return int(r.stats().kernel_launches)
        return int(r.stats().kernel_launches) + 1 + (1 if rank == 0 else 0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 1)):     # (W = 0 still runs one: the launch count is read after a step)
        step()
    barrier()
    sampler_thread = ClockSampler(local_rank) if rank == 0 else None
    if sampler_thread:
        sampler_thread.start()
    per_step = launches_per_step()      # after the warm-up steps; the timed loop itself never reads statistics back
    used_specialised = bool(r.stats().specialized)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []
    barrier()
    wall0 = time.perf_counter()
    dump = bool(args.dump_outputs) and rank == 0
    for i in range(args.steps):
        flush.fill_(float(i))          # L2 flush between timed iterations (outside the events)
        ev[i][0].record(stream)
        image_ptr = step(want_image=dump and i == args.steps - 1)
        ev[i][1].record(stream)
    barrier()
    kernel_ms.append(r.stats().gpu_ms)   # of the last step
    launches[0] = per_step * args.steps
    wall = time.perf_counter() - wall0
    if sampler_thread:
        sampler_thread.stop_flag.set()
        sampler_thread.join()
    if dump:
        # copied now: the e2e passes below render into the same frame images
        dump_outputs(args.dump_outputs, device_image(image_ptr, (h, w, 3)).cpu().numpy())
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    total_samples = w * h * spp
    value = total_samples / (ms_per_step * 1e-3)
    segs = torch.tensor([float(r.stats().segments)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(segs, op=dist.ReduceOp.SUM)

    # ---- end to end through the public host call (rank-local share; N GPUs run concurrently) ----
    e2e_steps = max(1, min(args.steps, 10))
    # the host-side result buffer: page-locked, allocated once (the Rust host reuses its Vec likewise)
    host_out = torch.empty((h, w, 3), dtype=torch.float64, pin_memory=True).numpy()
    scene_bytes = (job.scene.c.n_prims * (4 + 40 + 4 + 4 + 4 + 48) + job.scene.c.n_materials * 16 +
                   job.scene.c.n_textures * 48 + job.scene.c.n_nodes * 56 + job.scene.c.n_perlin * C.sizeof(capi.rc_perlin) +
                   sum(im[0] * im[1] * 4 for im in job.scene.images) + C.sizeof(capi.rc_camera) + C.sizeof(capi.rc_params))
    host32 = torch.empty(n, dtype=torch.float32, pin_memory=True)
    e2e_params = harness.make_params(w, h, spp, depth, seed=0, variant=variant, sampler=sampler, split=split,
                                     rank=rank, world=world, rng_rounds=args.rng_rounds, specialize=spec)

    def e2e_pass(cancel_flag=None):
        """The step through the host-facing call, host buffers on both sides: scene tables + camera host -> device,
        render, the gamma'd f64 image device -> host on rank 0.  Same call, unit and dtype at every N."""
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r.upload(job)                       # host -> device: scene tables + camera
            if args.lbvh:
                r.build_lbvh()
            if frame is not None:
                r.render_frame(e2e_params, frame, out=host_out if rank == 0 else None, cancel=cancel_flag)
            elif world == 1:
                r.render(e2e_params, out=host_out, cancel=cancel_flag)
            else:
                step(e2e_params)
                if rank == 0:
                    host32.copy_(rgb, non_blocking=True)
            torch.cuda.synchronize()
        barrier()
        dt = (time.perf_counter() - t0) / e2e_steps
        te = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return total_samples / float(te.item())

    e2e_value = e2e_pass()
    # the way the reference's host calls a full render: always with a cancel event (interactive.rs:236-251), here never raised
    e2e_cancel_value = e2e_pass(C.c_int32(0)) if (frame is not None or world == 1) else None
    d2h = n * (8 if (frame is not None or world == 1) else 4)

    if rank == 0:
        peaks, peaks_kind = measured_peaks()
        fp32_tflops, lane_ginstr = r.fp32_peak()
        st = r.stats()
        line = {
            "metric": "samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "scene": scene + ".yml", "width": w, "height": h, "spp": spp,
                       "max_depth": depth, "variant": args.variant, "sampler": args.sampler,
                       "rng": f"philox2x32-{args.rng_rounds}", "split": split_name,
                       "kernel": "scene-specialised (NVRTC)" if used_specialised else "precompiled",
                       "bvh": "gpu-lbvh" if args.lbvh else ("host" if job.scene.c.n_nodes else "none"),
                       "tile_culling": "off" if os.environ.get("RC_NO_TILE_CULL") or job.camera.lens_radius != 0.0 else "on (bit-identical images)",
                       "l2": "256 MiB buffer written between timed iterations (flush)",
                       "parallelism": f"tiles{world}" if split_name == "tiles" else f"samples{world}",
                       "exchange": ("none" if world == 1 else (
                           ("in-kernel peer stores into rank 0's frame (CUDA IPC, NVLink) + per-rank progress words (rc_render_frame; no collective)"
                            if split_name == "tiles" else
                            "in-kernel peer stores of every rank's partial sums into its slot of rank 0's frame (CUDA IPC, NVLink) + per-rank "
                            "progress words, slots added in rank order on rank 0 (rc_render_frame; no collective)")
                           if frame is not None else "NCCL reduce of the accumulation buffer to rank 0"))},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(scene_bytes),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "call": "rc_render_frame" if frame is not None else ("rc_render" if world == 1 else "rc_render_accumulate + torch reduce")},
            "e2e_cancel": {"value": e2e_cancel_value, "unit": "samples/s",
                           "what": "the e2e call with a cancel flag that is never raised, as the reference's host always passes one"},
            "gpu_launches": launches[0],
            "clocks": sampler_thread.summary() if sampler_thread else None,
            "wall_s": wall,
            "segments_per_sample": float(segs.item()) / total_samples,
            "kernel_ms_rank0": sum(kernel_ms) / len(kernel_ms),
        }
        # ---- roofline: FP32 issue (SURVEY §8(d)) + cpu baseline (oracle counters give A) ----
        cpu = None
        A = None
        if not args.no_cpu_baseline:
            from oracle import oracle as O  # noqa: F401  (checker / baseline only)
            pr = harness.make_params(w, h, spp, depth, seed=0, sampler=capi.RC_SAMPLER_REJECTION)
            probe, _, _ = oracle_slice(job, pr, 2)
            slice_spp = max(2, min(spp, int(round(probe * 15.0 / (w * h)))))
            sps, dt, cnt = oracle_slice(job, pr, slice_spp)
            types = job.scene.np["prim_type"]
            n_sph = int((types == capi.RC_PRIM_SPHERE).sum())
            A = flops_per_sample(cnt, job.scene.c.bg_type == capi.RC_BG_SKY)
            A_lin = flops_per_sample(cnt, job.scene.c.bg_type == capi.RC_BG_SKY, (n_sph, len(types) - n_sph))
            cpu = {"value": sps, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"{slice_spp}-spp slice of the full {w}x{h} frame ({dt:.1f} s), restated reference "
                             "(f64, rejection samplers, sequential RNG, 10x10 tiles, all host threads)",
                   "segments_per_sample": cnt["segments"] / cnt["samples"],
                   "flops_per_sample_bvh": A, "flops_per_sample_linear": A_lin}
        cap = ncu_capture(args.workload)
        if A is not None:
            # SURVEY §8(d): brute force (N_node = 0) when the scene has <= 8 primitives, else the
            # oracle's BVH counters
            A_used = A_lin if job.scene.c.n_prims <= 8 else A
            achieved = value / world * A_used / 1e12
            line["roofline"] = {"bound": "fp32", "achieved": achieved, "peak": fp32_tflops, "unit": "TFLOP/s",
                                "frac": achieved / fp32_tflops, "traffic": cap.get("dram_bytes_per_launch") if cap else None,
                                "traffic_source": (cap.get("source") if cap else None),
                                "ncu": cap,
                                # what was actually ISSUED (ncu, same kernel and configuration) next to what is credited
                                "frac_executed": (cap["fp32_tflops_executed"] / fp32_tflops) if cap and cap.get("fp32_tflops_executed") else None,
                                "note": ("achieved = ALGORITHMIC flops (SURVEY §8(d): the reference algorithm's work per sample, oracle counters "
                                         "x cost table) / time.  This path does not execute all of them: tiles whose frustum contains no "
                                         "primitive trace nothing, opposite walls share one test, and BVH scenes walk a SAH tree instead of the "
                                         "reference's median-split tree whose node tests the oracle counts — so the fraction can exceed what the "
                                         "FP32 pipes issued (frac_executed) and, for scenes that are mostly culled, even 1.  "
                                         "traffic = DRAM bytes ncu counted for the one launch: the kernel's only global write is the "
                                         "frame (width x height x 12 B, the algorithmic traffic), which is still in the 126 MB L2 when the "
                                         "kernel ends, so the counter sees next to nothing; the bound is instruction issue, not HBM."),
                                "algorithmic_bytes_per_launch": int(w * h * 12),
                                "peak_source": "FFMA micro-benchmark in this run (rc_fp32_peak), per GPU",
                                "flops_per_sample": A_used, "lane_ginstr_per_s_peak": lane_ginstr,
                                "hbm_peak_gbs": peaks.get("hbm_gbs"), "hbm_peak_source": peaks_kind,
                                "sm_count": st.sm_count}
        line["cpu_baseline"] = cpu
        print(json.dumps(line))
    barrier()
    if frame is not None:
        r.frame_close(frame)
    r.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
