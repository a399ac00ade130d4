"""In-tree build of libdmesh_b200.so (sm_100a only).

    python -m dmesh_renderer_b200.build [--force]

Plain nvcc, no torch headers (the native library has no torch dependency; the
reference's 3.5-minute build is almost all ATen header parsing).  The .so is
written next to this file so that it travels to the GPU box with the snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdmesh_b200.so")
OBJ = os.path.join(HERE, "csrc", "_obj")

SOURCES = ["capi.cu", "capi_tet.cu", "preprocess.cu", "binning.cu", "radix_sort.cu", "tri_render.cu", "tet_kernels.cu", "collective.cu", "inverse.cu", "image.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    # nvcc defaults for float semantics (fmad=true, IEEE div/sqrt, no fast-math):
    # the integer outputs of the binning stages depend on it (SURVEY App. A.10).
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _newer(a, b):
    return (not os.path.exists(b)) or os.path.getmtime(a) > os.path.getmtime(b)


def build(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    hdrs = [os.path.join(CSRC, h) for h in os.listdir(CSRC) if h.endswith(".cuh")]
    hdrs.append(os.path.join(HERE, "..", "include", "dmesh_b200.h"))
    os.makedirs(OBJ, exist_ok=True)
    jobs = []
    objs = []
    for s in srcs:
        o = os.path.join(OBJ, os.path.basename(s) + ".o")
        objs.append(o)
        if force or _newer(s, o) or any(_newer(h, o) for h in hdrs):
            jobs.append(["nvcc", "-c", s, "-o", o, *NVCC_FLAGS])
    log = []

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append((cmd[2], r.stderr))
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (cmd[2], r.stderr[-6000:]))

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
            list(ex.map(run, jobs))
    if jobs or not os.path.exists(LIB):
        cmd = ["nvcc", "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stderr[-4000:])
    if verbose:
        for name, err in log:
            print("==", os.path.basename(name))
            print(err)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv or "--verbose" in sys.argv))
