#!/usr/bin/env python3
"""Build opencv_b200/lib/libb200cv.so (sm_100a only) in-tree with nvcc + g++.

    python -m opencv_b200.build [-j N] [--force] [--verbose-ptxas]

Every .cu under csrc/ is compiled with
    nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17
host-only sources (host_tables.cpp) with g++ -ffp-contract=off (their arithmetic must round exactly like
the reference's softfloat code), and everything is linked into one shared library with a static cudart.
"""
import argparse
import concurrent.futures as cf
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "lib", "obj")
LIB = os.path.join(HERE, "lib", "libb200cv.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off", "--expt-relaxed-constexpr",
              "-I" + os.path.join(HERE, "..", "include")]
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-ffp-contract=off",
             "-I" + os.path.join(HERE, "..", "include"), "-I/usr/local/cuda/include"]


def newer(src, obj, extra=()):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    deps = [src] + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h")) + \
        glob.glob(os.path.join(HERE, "..", "include", "*.h")) + list(extra)
    return any(os.path.getmtime(d) > t for d in deps)


def compile_one(src, force, verbose):
    obj = os.path.join(OBJ, os.path.basename(src) + ".o")
    if not force and not newer(src, obj):
        return obj, 0, ""
    if src.endswith(".cu"):
        cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    else:
        cmd = ["g++"] + CXX_FLAGS + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return obj, r.returncode, (r.stdout + r.stderr)


def build(jobs=None, force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cpp")))
    objs, failed = [], False
    with cf.ThreadPoolExecutor(max_workers=jobs or os.cpu_count() or 4) as ex:
        for obj, rc, out in ex.map(lambda s: compile_one(s, force, verbose), srcs):
            objs.append(obj)
            if out.strip() and (rc != 0 or verbose):
                sys.stderr.write(out)
            if rc != 0:
                failed = True
    if failed:
        raise RuntimeError("b200cv: compilation failed")
    if force or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs + [os.path.abspath(__file__)]):
        # the soname lets a library that needs libb200cv.so (the reference built with the HAL header) use the copy already loaded,
        # wherever that library was built or moved
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-cudart", "static", "-Xlinker", "--no-undefined", "-Xlinker", "-soname=libb200cv.so",
                                                     "-lpthread", "-ldl", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("b200cv: link failed")
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("-j", type=int, default=None)
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose-ptxas", action="store_true")
    a = ap.parse_args()
    print(build(a.j, a.force, a.verbose_ptxas))
