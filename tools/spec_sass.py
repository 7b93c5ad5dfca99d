#!/usr/bin/env python
"""Compiles the scene-specialised megakernel source (rc_spec_source) with nvcc for sm_100a — no GPU
needed — and prints registers, the static SASS opcode mix of the main loop and, with --dump, the SASS.

    python tools/spec_sass.py cornell_box [--dump out.sass] [-D RT_STEAL=0]
"""
import argparse
import collections
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from racer_tracer_b200 import capi, harness  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("scene")
ap.add_argument("--dump")
ap.add_argument("-D", action="append", default=[])
ap.add_argument("--csrc", help="directory with the rt_*.cuh headers to compile against (default: the tree's csrc/)")
args = ap.parse_args()

lib = capi.load()
cfg = harness.load_config(os.path.join(ROOT, "tests", "golden", "config.yml"))
job = harness.prepare_job(os.path.join(ROOT, "tests", "golden", "scenes", args.scene + ".yml"), cfg, 64, 64)
os.environ["RC_SPEC_CAMERA"] = ",".join(repr(float(v)) for v in job.camera.origin)   # rc_spec_source has no camera of its own
n = lib.rc_spec_source(job.scene.ptr, None, 0)
buf = C.create_string_buffer(n + 1)
lib.rc_spec_source(job.scene.ptr, buf, n + 1)
src = buf.value.decode()
tmp = tempfile.mkdtemp()
cu = os.path.join(tmp, "spec.cu")
open(cu, "w").write(src)
cubin = os.path.join(tmp, "spec.cubin")
cmd = ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-lineinfo", "-Xptxas", "-v",
       "-I", args.csrc or os.path.join(ROOT, "racer_tracer_b200", "csrc"), "-cubin", "-o", cubin, cu] + ["-D" + d for d in args.D]
r = subprocess.run(cmd, capture_output=True, text=True)
if r.returncode:
    print(r.stderr)
    sys.exit(1)
print("\n".join(l for l in r.stderr.splitlines() if "registers" in l or "spill" in l))
sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", cubin], capture_output=True, text=True).stdout
lines = [l for l in sass.splitlines() if re.match(r"\s+/\*[0-9a-f]{4}\*/", l)]
ops = []
for l in lines:
    m = re.match(r"\s+/\*([0-9a-f]{4})\*/\s+(@!?U?P\d\s+)?([A-Z0-9_.]+)", l)
    if m:
        ops.append((int(m.group(1), 16), m.group(3), l))
print(f"{len(ops)} static instructions")
mix = collections.Counter(o[1].split(".")[0] for o in ops)
print(", ".join(f"{k} {v}" for k, v in mix.most_common(24)))
# the path loop: from the target of the last backward branch after a VOTE.ANY to that branch
ALU = {"FSETP", "LOP3", "FSEL", "SEL", "ISETP", "SHF", "I2FP", "PRMT", "FMNMX", "FMNMX3", "IADD3", "VOTE", "PLOP3", "LEA", "VIADD", "MOV",
       "IABS", "FSET"}
for i, o in enumerate(ops[:-1]):
    if o[1].startswith("VOTE") and "BRA" in ops[i + 1][1]:
        m = re.search(r"BRA 0x([0-9a-f]+)", ops[i + 1][2])
        if m and int(m.group(1), 16) < o[0]:
            body = [q for q in ops if int(m.group(1), 16) <= q[0] <= ops[i + 1][0]]
            n_alu = sum(1 for q in body if q[1].split(".")[0] in ALU)
            print(f"path loop: {len(body)} static instructions, {n_alu} on the ALU pipe (compares, selects, logic, moves, conversions)")
if args.dump:
    open(args.dump, "w").write("\n".join(o[2] for o in ops))
    print("SASS ->", args.dump)
