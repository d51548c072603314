"""Build libdaisy_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m recommend_lib_b200.build [--force] [--verbose]

The library has no Python or torch dependency: it is a plain C-ABI shared object
(include/daisy_b200.h) that the Python host code loads with ctypes and that a C/C++
driver can link directly.
"""
from __future__ import annotations

import glob
import os
import shlex
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libdaisy_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
    "-I", INCLUDE,
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libdaisy_b200.so cannot be built")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every csrc/*.cu to an object (only the stale ones) and link the shared library.

    Experiments (DESIGN.md section 11): DAISY_NVCC_EXTRA="-maxrregcount=64" with DAISY_LIB_VARIANT=r64 builds
    libdaisy_b200_r64.so from objects under csrc/_obj_r64/ next to the default library, which is left alone; a process
    started with DAISY_LIB_VARIANT=r64 loads that one (_lib.py), so both travel to the GPU box in one snapshot and one
    call can measure them side by side."""
    nvcc = _nvcc()
    extra = shlex.split(os.environ.get("DAISY_NVCC_EXTRA", ""))
    variant = os.environ.get("DAISY_LIB_VARIANT", "")
    if extra and not variant:
        raise RuntimeError("DAISY_NVCC_EXTRA needs DAISY_LIB_VARIANT=<name>: the default library is never built with "
                           "experimental flags")
    obj_dir = OBJ + ("_" + variant if variant else "")
    lib = LIB[:-3] + ("_" + variant if variant else "") + ".so"
    os.makedirs(obj_dir, exist_ok=True)
    headers = glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(INCLUDE, "*.h"))
    objs, procs = [], []
    for src in sources():
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src, *headers]):
            cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", src, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            procs.append((src, subprocess.Popen(cmd)))
    failed = [src for src, p in procs if p.wait() != 0]
    if failed:
        raise RuntimeError("nvcc failed for: " + ", ".join(failed))
    if force or procs or _stale(lib, objs):
        # shared cudart: inside a PyTorch process the library binds to the libcudart.so.12 torch already loaded, so
        # both see ONE runtime (same current-device state, streams and events interoperate by construction)
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "shared", "-o", lib, *objs]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
