"""Build libvvdsp_b200.so in-tree: C99 host sources with gcc, CUDA sources with nvcc for sm_100a only.

    python -m vv_dsp_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.  nvcc
cross-compiles without a GPU, so this also is the driver's "does it build" check
(__graft_entry__.build()).
"""
from __future__ import annotations

import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
INC = os.path.join(ROOT, "include")
LIB = os.path.join(PKG, "lib", "libvvdsp_b200.so")
OBJ = os.path.join(PKG, "lib", "obj")
HOST_DIR = os.path.join(PKG, "csrc", "host")
# the one list of C99 host units (the emulator build of tests/emu imports it) and the headers they share
HOST_SRCS = sorted(os.path.join(HOST_DIR, f) for f in os.listdir(HOST_DIR) if f.endswith(".c"))
HOST_DEPS = sorted(os.path.join(HOST_DIR, f) for f in os.listdir(HOST_DIR) if f.endswith(".h"))
CUDA_DIR = os.path.join(PKG, "csrc", "cuda")
# one kernel family per translation unit (vvb_tu_*.cu) + the C-ABI / runtime unit: compiled in parallel
CUDA_SRCS = sorted(os.path.join(CUDA_DIR, f) for f in os.listdir(CUDA_DIR) if f.endswith(".cu"))
CUDA_DEPS = sorted(os.path.join(CUDA_DIR, f) for f in os.listdir(CUDA_DIR) if f.endswith(".cuh"))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _headers():
    out = []
    for d, _, fs in os.walk(INC):
        out += [os.path.join(d, f) for f in fs]
    return out


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd[:3]) + " ...")
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr)
    elif "warning" in (r.stdout + r.stderr).lower():       # e.g. ptxas -warn-spills
        sys.stderr.write(f"[{os.path.basename(cmd[-3])}]\n" + r.stdout + r.stderr)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = _headers()
    objs = []
    for src in HOST_SRCS:
        o = os.path.join(OBJ, os.path.basename(src) + ".o")
        if force or _stale(o, [src] + HOST_DEPS + hdrs):
            _run(["gcc", "-std=c99", "-O2", "-fPIC", "-Wall", "-Wextra", "-I" + INC, "-c", src, "-o", o], verbose)
        objs.append(o)
    # VVB_NVCC_EXTRA: extra nvcc flags for A/B builds (e.g. "-DVVB_INV_BASETW=0")
    extra = os.environ.get("VVB_NVCC_EXTRA", "").split()
    jobs = []
    for src in CUDA_SRCS:
        o = os.path.join(OBJ, os.path.basename(src) + ".o")
        if force or _stale(o, [src] + CUDA_DEPS + hdrs):
            jobs.append([NVCC, *ARCH, "-std=c++17", "-O3", "-lineinfo", *extra, "-Xptxas", "-v" if verbose else "-warn-spills",
                         "-Xcompiler", "-fPIC", "-I" + INC, "-c", src, "-o", o])
        objs.append(o)
    if jobs:
        from concurrent.futures import ThreadPoolExecutor
        workers = int(os.environ.get("VVB_BUILD_JOBS", str(min(len(jobs), os.cpu_count() or 4))))
        with ThreadPoolExecutor(max_workers=max(1, workers)) as pool:
            list(pool.map(lambda c: _run(c, verbose), jobs))
    if force or _stale(LIB, objs):
        _run([NVCC, *ARCH, "-shared", "-cudart", "static", "-o", LIB, *objs, "-lm"], verbose)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
