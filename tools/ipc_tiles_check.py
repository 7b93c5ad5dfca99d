#!/usr/bin/env python
"""Two (or more) processes, one GPU each, one frame: every rank stores its tiles into rank 0's frame buffer
(rc_shared_alloc / rc_shared_open / rc_render_tiles_into, then the whole exchange behind the ABI:
rc_frame_create / rc_frame_open / rc_render_frame) and rank 0 compares the frames with its own single-GPU renders.  Run under torchrun; prints IPC_TILES_OK on success.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/ipc_tiles_check.py
"""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from racer_tracer_b200 import capi, harness  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
w, h, spp = 333, 201, 64
cfg = harness.load_config(os.path.join(ROOT, "tests", "golden", "config.yml"))
job = harness.prepare_job(os.path.join(ROOT, "tests", "golden", "scenes", "cornell_box.yml"), cfg, w, h)
r = harness.CudaRenderer([local])
r.set_stream(torch.cuda.current_stream().cuda_stream)
r.upload(job)
n = w * h * 3
if rank == 0:
    ptr, handle = r.shared_alloc(n * 4)
    hbuf = torch.tensor(list(handle), dtype=torch.uint8, device="cuda")
else:
    hbuf = torch.empty(64, dtype=torch.uint8, device="cuda")
dist.broadcast(hbuf, 0)
if rank != 0:
    ptr = r.shared_open(bytes(hbuf.cpu().tolist()))
join = torch.zeros(1, device="cuda")
for spec in (0, 2):
    p = harness.make_params(w, h, spp, 20, seed=9, rank=rank, world=world, specialize=spec)
    r.render_tiles_into(p, ptr)
    dist.all_reduce(join)
    torch.cuda.synchronize()
    if rank == 0:
        rgb = torch.empty(n, dtype=torch.float32, device="cuda")
        r.finalize(ptr, w, h, spp, rgb.data_ptr())
        got = rgb.cpu().numpy().reshape(h, w, 3)
        want = r.render(harness.make_params(w, h, spp, 20, seed=9, specialize=spec)).astype(np.float32)
        assert np.array_equal(got, want), f"specialize={spec}: {np.abs(got - want).max()}"
    dist.barrier()
r.shared_close(ptr)

# ---- the same split behind the ABI: rc_frame_* + rc_render_frame.  Several frames are enqueued back to back with
# no host synchronisation in between (the two images of the frame alternate; the progress words order the ranks),
# each with another seed; rank 0 keeps a device copy of every finished image and checks them all at the end.
if rank == 0:
    frame, handle = r.frame_create(w, h, world)
    hbuf = torch.tensor(list(handle), dtype=torch.uint8, device="cuda")
else:
    hbuf = torch.empty(64, dtype=torch.uint8, device="cuda")
dist.broadcast(hbuf, 0)
if rank != 0:
    frame = r.frame_open(bytes(hbuf.cpu().tolist()), w, h, rank, world)
seeds = [3, 4, 5, 6, 7]
kept = []
for seed in seeds:
    p = harness.make_params(w, h, spp, 20, seed=seed, rank=rank, world=world, specialize=2)
    dptr = r.render_frame(p, frame, want_device_ptr=(rank == 0))
    if rank == 0:   # a stream-ordered copy of the finished image (enqueued before the next call, which hands the image on to the ranks)
        keep = torch.empty(n, dtype=torch.float32, device="cuda")
        keep.copy_(harness.device_view(dptr, n), non_blocking=True)
        kept.append(keep)
torch.cuda.synchronize()
dist.barrier()
if rank == 0:
    for seed, keep in zip(seeds, kept):
        got = keep.cpu().numpy().reshape(h, w, 3)
        want = r.render(harness.make_params(w, h, spp, 20, seed=seed, specialize=2))
        # sqrtf(sum / n) in the kernel's store vs sqrt in f64 of the same float sum: two roundings apart at most
        assert np.allclose(got, want, rtol=3e-7, atol=1e-7), f"frame seed {seed}: {np.abs(got - want).max()}"
    # the host-buffer form (what `e2e` times): f64 out, synchronous on rank 0
out = np.empty((h, w, 3), dtype=np.float64) if rank == 0 else None
p = harness.make_params(w, h, spp, 20, seed=11, rank=rank, world=world, specialize=2)
r.render_frame(p, frame, out=out)
torch.cuda.synchronize()
dist.barrier()
if rank == 0:
    want = r.render(harness.make_params(w, h, spp, 20, seed=11, specialize=2))
    assert np.allclose(out, want, rtol=3e-7, atol=1e-7), np.abs(out - want).max()
# ---- the sample split through the same frame: every rank traces ITS samples of every pixel and stores the partial
# sums into its slot of rank 0's frame; rank 0 adds the slots in rank order.  Equal to the single-GPU render up to the
# order of the fp32 additions.
for seed in (21, 22, 23):
    out = np.empty((h, w, 3), dtype=np.float64) if rank == 0 else None
    p = harness.make_params(w, h, spp, 20, seed=seed, rank=rank, world=world, specialize=2, split=capi.RC_SPLIT_SAMPLES)
    r.render_frame(p, frame, out=out)
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        want = r.render(harness.make_params(w, h, spp, 20, seed=seed, specialize=2))
        assert np.allclose(out, want, rtol=2e-6, atol=1e-6), f"sample-split frame seed {seed}: {np.abs(out - want).max()}"
# ---- fewer samples than ranks: at 1 spp only the last rank has a sample, and every other rank must publish a zeroed
# slot — not the sums it stored there two frames ago (the frames above left both images' slots non-zero).  Three frames
# back to back, so that both alternating images are reused.
kept, seeds = [], (31, 32, 33)
for seed in seeds:
    p = harness.make_params(w, h, 1, 20, seed=seed, rank=rank, world=world, specialize=2, split=capi.RC_SPLIT_SAMPLES)
    dptr = r.render_frame(p, frame, want_device_ptr=(rank == 0))
    if rank == 0:
        keep = torch.empty(n, dtype=torch.float32, device="cuda")
        keep.copy_(harness.device_view(dptr, n), non_blocking=True)
        kept.append(keep)
torch.cuda.synchronize()
dist.barrier()
if rank == 0:
    for seed, keep in zip(seeds, kept):
        got = keep.cpu().numpy().reshape(h, w, 3)
        want = r.render(harness.make_params(w, h, 1, 20, seed=seed, specialize=2))
        assert np.allclose(got, want, rtol=3e-7, atol=1e-7), f"1-spp sample-split frame seed {seed}: {np.abs(got - want).max()}"
r.frame_close(frame)
r.close()
if rank == 0:
    print("IPC_TILES_OK")
dist.destroy_process_group()
