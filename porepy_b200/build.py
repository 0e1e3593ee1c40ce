"""Build libporeb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libporeb200.so")
SOURCES = ["api.cu", "spmv.cu", "mpfa_launch.cu", "mpsa2d.cu", "mpsa3d.cu", "face.cu", "peaks.cu", "krylov.cu", "sparse_ops.cu", "plan_device.cu", "shard.cu", "geometry.cu", "local_blocks.cu", "gmres.cu", "solver_check.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "-Xcompiler", "-fopenmp"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "poreb200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, extra_flags=(), lib: str = LIB) -> str:
    """``extra_flags`` / ``lib``: developer knobs for A/B variants (e.g. ``-DPB_EXP_ONEBAR`` into
    ``libporeb200_onebar.so``, selected at run time with ``POREB200_LIB``)."""
    if not force and not needs_build() and lib == LIB:
        return LIB
    # one nvcc process per translation unit, in parallel (the kernel instantiations dominate)
    jobs = []
    objdir = os.path.join(HERE, "_obj", os.path.basename(lib))
    os.makedirs(objdir, exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, *extra_flags, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        jobs.append((obj, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for obj, cmd, proc in jobs:
        out, _ = proc.communicate()
        if verbose or proc.returncode:
            sys.stderr.write(out)
        if proc.returncode:
            raise subprocess.CalledProcessError(proc.returncode, cmd)
        objs.append(obj)
    subprocess.check_call([_nvcc(), "-shared", "-o", lib, *objs, "-gencode",
                           "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fopenmp", "-lgomp"])
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
