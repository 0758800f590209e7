"""Build an experiment variant of libmugd with extra -D defines into mug_diffusion_b200/libmugd_<name>.so
usage: python tools/build_variant.py timeline -DMUGD_TC_TIMELINE ; then MUGD_LIB=<path> python tools/gemm_timeline.py"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mug_diffusion_b200 import build as B  # noqa: E402

name, defs = sys.argv[1], sys.argv[2:]
out = os.path.join(B.HERE, f"libmugd_{name}.so")
objdir = os.path.join(B.HERE, "build", name)
os.makedirs(objdir, exist_ok=True)
flags = [f for f in B.NVCC_FLAGS if f != "--use_fast_math=false"] + defs
procs, objs = [], []
for src in B.SOURCES:
    obj = os.path.join(objdir, src.replace(".cu", ".o"))
    objs.append(obj)
    procs.append(subprocess.Popen([B._nvcc(), *flags, "-c", os.path.join(B.CSRC, src), "-o", obj]))
assert all(p.wait() == 0 for p in procs)
subprocess.check_call([B._nvcc(), "-shared", "-o", out, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"])
print(out)
