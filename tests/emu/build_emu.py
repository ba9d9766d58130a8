"""TEST-ONLY: compile the kernel sources for the CPU execution emulator (tests/emu/cuda_emu.h).

Produces tests/emu/libvvdsp_b200_emu.so with the same exported C-ABI as the product
library, so the CPU test-suite can drive the very same host code and kernel code.
The product package never loads this file.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from vv_dsp_b200.build import HOST_DEPS, HOST_SRCS  # noqa: E402

PKG = os.path.join(ROOT, "vv_dsp_b200")
INC = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libvvdsp_b200_emu.so")
OBJ = os.path.join(HERE, "obj")


def build(force=False):
    os.makedirs(OBJ, exist_ok=True)
    host = HOST_SRCS
    cudir = os.path.join(PKG, "csrc", "cuda")
    cus = sorted(os.path.join(cudir, f) for f in os.listdir(cudir) if f.endswith(".cu"))
    deps = host + HOST_DEPS + cus + [os.path.join(HERE, "cuda_emu.h")]
    for d, _, fs in list(os.walk(INC)) + list(os.walk(os.path.join(PKG, "csrc", "cuda"))):
        deps += [os.path.join(d, f) for f in fs]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return LIB
    objs = []
    for src in host:
        o = os.path.join(OBJ, os.path.basename(src) + ".o")
        subprocess.run(["gcc", "-std=c99", "-O1", "-fPIC", "-I" + INC, "-c", src, "-o", o], check=True)
        objs.append(o)
    procs = []
    for cu in cus:                                    # one kernel family per unit: compile them side by side
        o = os.path.join(OBJ, os.path.basename(cu)[:-3] + "_emu.o")
        procs.append(subprocess.Popen(["g++", "-std=c++17", "-O1", "-fPIC", "-DVVB_EMU", *os.environ.get("VVB_EMU_EXTRA", "").split(),
                                       "-Wno-unknown-pragmas", "-I" + HERE,
                                       "-I" + INC, "-x", "c++", "-c", cu, "-o", o]))
        objs.append(o)
    for p in procs:
        if p.wait() != 0:
            raise RuntimeError("emulator build failed")
    subprocess.run(["g++", "-shared", "-o", LIB, *objs, "-lm"], check=True)
    return LIB


if __name__ == "__main__":
    print(build(force=True))
