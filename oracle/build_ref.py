#!/usr/bin/env python3
"""Build the UNMODIFIED reference CPU implementation of the hot path into oracle/_ref/.

TEST INFRASTRUCTURE ONLY.  Nothing under opencv_b200/ may import, link or execute
anything produced here; only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs use it, and only as the checker / baseline.

What it does
------------
* compiles the reference's own `modules/core/src` and `modules/imgproc/src`
  translation units *where they lie* under /root/reference (nothing is copied into
  the repo) with g++ directly -- the reference's CMake build system is NOT run;
* the handful of headers CMake would have generated (cvconfig.h, cv_cpu_config.h,
  custom_hal.hpp, opencv_modules.hpp, *.simd_declarations.hpp, empty OpenCL kernel
  tables, version string) are written by this script into oracle/_ref/gen/
  (they are configuration stubs authored here, not reference sources);
* CPU features mirror the reference's stock x86-64 configuration: baseline SSE3, run-time
  dispatched SSE4_1 / SSE4_2 / AVX / FP16 / AVX2 / AVX512_SKX variants of every
  `*.simd.hpp` listed by `ocv_add_dispatched_file` in the modules' CMakeLists.txt (those
  lines are only *read* with a regex), plus the hand-named `*.sse4_1.cpp / *.avx.cpp /
  *.avx2.cpp` units; IPP / OpenCL / ITT / OpenVX / TBB are off, threads = the reference's
  own pthreads `parallel_for_` pool;
* links them with oracle/ref_shim.cpp (our extern "C" wrapper around the public
  cv:: calls) into oracle/_ref/libocvref.so.

Outputs go ONLY to oracle/_ref/ (git-ignored, shipped to the GPU box by gpurun).
Usage: python oracle/build_ref.py [-j N] [--reference /root/reference]
"""
import argparse
import glob
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
GEN = os.path.join(OUT, "gen")

CORE_EXCLUDE = {
    # alternative parallel back-ends / GPU interop that need external SDKs
    "parallel_openmp.cpp", "parallel_tbb.cpp",
}
IMGPROC_EXCLUDE = {"imgwarp.lasx.cpp", "resize.lasx.cpp"}

CXXFLAGS = [
    "-std=c++11", "-O3", "-DNDEBUG", "-fPIC", "-fsigned-char", "-pthread",
    "-fomit-frame-pointer", "-ffunction-sections", "-fdata-sections",
    "-fvisibility=hidden", "-fvisibility-inlines-hidden", "-w",
    "-msse3",
    "-DCVAPI_EXPORTS", "-D_USE_MATH_DEFINES", "-D__OPENCV_BUILD=1",
    "-D__STDC_CONSTANT_MACROS", "-D__STDC_FORMAT_MACROS", "-D__STDC_LIMIT_MACROS",
]

BASELINE = ["SSE", "SSE2", "SSE3"]
# dispatched modes in increasing order: (name, extra flags, implied CV_CPU_COMPILE_* defines) -- cumulative
MODES = [
    ("SSE4_1", ["-mssse3", "-msse4.1"], ["SSSE3", "SSE4_1"]),
    ("SSE4_2", ["-mpopcnt", "-msse4.2"], ["POPCNT", "SSE4_2"]),
    ("AVX", ["-mavx"], ["AVX"]),
    ("FP16", ["-mf16c"], ["FP16"]),
    ("AVX2", ["-mavx2", "-mfma"], ["AVX2", "FMA3"]),
    ("AVX512_SKX", ["-mavx512f", "-mavx512cd", "-mavx512vl", "-mavx512bw", "-mavx512dq"],
     ["AVX_512F", "AVX512_COMMON", "AVX512_SKX"]),
]
MODE_NAMES = [m[0] for m in MODES]


def mode_flags(mode):
    flags, defs = [], []
    for name, f, d in MODES:
        flags += f
        defs += d
        if name == mode:
            break
    return flags + ["-DCV_CPU_COMPILE_%s=1" % x for x in defs] + ["-DCV_CPU_DISPATCH_MODE=%s" % mode]


def dispatched_files(ref, mod):
    """{name: [modes best-first]} from the module's ocv_add_dispatched_file() lines (read only)."""
    out = {}
    txt = open(os.path.join(ref, "modules", mod, "CMakeLists.txt")).read()
    for m in re.finditer(r"ocv_add_dispatched_file\(\s*(\w+)([^)]*)\)", txt):
        modes = [x for x in m.group(2).split() if x in MODE_NAMES]
        out[m.group(1)] = sorted(modes, key=MODE_NAMES.index, reverse=True)
    return out


def w(path, text):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    if os.path.exists(path) and open(path).read() == text:
        return
    with open(path, "w") as f:
        f.write(text)


def gen_headers(ref):
    w(os.path.join(GEN, "cvconfig.h"),
      "#ifndef OPENCV_CVCONFIG_H_INCLUDED\n#define OPENCV_CVCONFIG_H_INCLUDED\n"
      "#define BUILD_SHARED_LIBS\n#define CV_ENABLE_INTRINSICS\n"
      "#define CUDA_ARCH_BIN \"\"\n#define CUDA_ARCH_FEATURES \"\"\n#define CUDA_ARCH_PTX \"\"\n"
      "#define HAVE_PTHREAD\n#define HAVE_PTHREADS_PF\n#endif\n")
    cfg = "// baseline = SSE3; dispatched = SSE4_1 SSE4_2 AVX FP16 AVX2 AVX512_SKX (stock x86-64 configuration)\n"
    for f in BASELINE:
        cfg += "#define CV_CPU_COMPILE_%s 1\n#define CV_CPU_BASELINE_COMPILE_%s 1\n" % (f, f)
    cfg += "#define CV_CPU_BASELINE_FEATURES 0 \\\n" + "".join("    , CV_CPU_%s \\\n" % f for f in BASELINE) + "\n\n"
    for m in MODE_NAMES:
        cfg += "#define CV_CPU_DISPATCH_COMPILE_%s 1\n" % m
    cfg += "#define CV_CPU_DISPATCH_FEATURES 0 \\\n" + "".join("    , CV_CPU_%s \\\n" % m for m in MODE_NAMES) + "\n\n"
    w(os.path.join(GEN, "cv_cpu_config.h"), cfg)
    w(os.path.join(GEN, "custom_hal.hpp"), "#ifndef _CUSTOM_HAL_INCLUDED_\n#define _CUSTOM_HAL_INCLUDED_\n#endif\n")
    w(os.path.join(GEN, "opencv2", "opencv_modules.hpp"),
      "#define HAVE_OPENCV_CORE\n#define HAVE_OPENCV_IMGPROC\n#define HAVE_OPENCV_FEATURES2D\n#define HAVE_OPENCV_FLANN\n")
    w(os.path.join(GEN, "opencv2", "cvconfig.h"), '#include "../cvconfig.h"\n')
    w(os.path.join(GEN, "opencv_data_config.hpp"),
      '#define OPENCV_INSTALL_PREFIX "/nonexistent"\n#define OPENCV_DATA_INSTALL_PATH "share/opencv4"\n'
      '#define OPENCV_BUILD_DIR "/nonexistent"\n#define OPENCV_DATA_BUILD_DIR_SEARCH_PATHS ""\n'
      '#define OPENCV_INSTALL_DATA_DIR_RELATIVE "../share/opencv4"\n')
    w(os.path.join(GEN, "version_string.inc"),
      '"\\nOpenCV reference built by oracle/build_ref.py: core+imgproc(+sift pyramid), baseline SSE3 + dispatch SSE4_1..AVX512_SKX, '
      'IPP/OpenCL/ITT off, pthreads parallel_for_\\n"\n')
    ocl_stub = ('#include "opencv2/core/ocl.hpp"\n#include "opencv2/core/ocl_genbase.hpp"\n'
                '#include "opencv2/core/opencl/ocl_defs.hpp"\n')
    for mod in ("core", "imgproc", "features2d"):
        w(os.path.join(GEN, mod, "opencl_kernels_%s.hpp" % mod), ocl_stub)
        disp = dispatched_files(ref, mod)
        for simd in glob.glob(os.path.join(ref, "modules", mod, "src", "*.simd.hpp")):
            name = os.path.basename(simd)[:-len(".simd.hpp")]
            modes = disp.get(name, [])
            txt = '#define CV_CPU_SIMD_FILENAME "%s"\n' % simd
            for m in reversed(modes):
                txt += '#define CV_CPU_DISPATCH_MODE %s\n#include "opencv2/core/private/cv_cpu_include_simd_declarations.hpp"\n\n' % m
                w(os.path.join(GEN, mod, "%s.%s.cpp" % (name, m.lower())),
                  '#include "%s"\n#include "%s"\n' % (os.path.join(ref, "modules", mod, "src", "precomp.hpp"), simd))
            txt += "#define CV_CPU_DISPATCH_MODES_ALL %s\n#undef CV_CPU_SIMD_FILENAME\n" % ", ".join(modes + ["BASELINE"])
            w(os.path.join(GEN, mod, name + ".simd_declarations.hpp"), txt)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    ap.add_argument("-j", type=int, default=os.cpu_count() or 4)
    ap.add_argument("--hal", action="store_true",
                    help="also build libocvref_hal.so: the same reference with hal/b200cv_hal_replacement.hpp registered as its imgproc HAL "
                         "(what -DOpenCV_HAL_DIR=<repo>/hal does in a CMake build) and linked against libb200cv.so -- integration proof")
    args = ap.parse_args()
    ref = args.reference
    if not os.path.isdir(os.path.join(ref, "modules", "imgproc", "src")):
        print("reference tree not found at %s -- nothing to build (prebuilt oracle/_ref is used if present)" % ref)
        return 0
    gen_headers(ref)

    units = []  # (src, obj, module)
    def add(mod, pattern, exclude=()):
        for src in sorted(glob.glob(os.path.join(ref, "modules", mod, "src", pattern))):
            if os.path.basename(src) in exclude:
                continue
            rel = os.path.relpath(src, os.path.join(ref, "modules"))
            units.append((src, os.path.join(OUT, "obj", rel.replace("/", "__") + ".o"), mod))
    add("core", "*.cpp", CORE_EXCLUDE)
    add("core", "utils/*.cpp")
    add("core", "parallel/*.cpp", CORE_EXCLUDE)
    add("imgproc", "*.cpp", IMGPROC_EXCLUDE)
    add("features2d", "feature2d.cpp")
    add("features2d", "keypoint.cpp")
    for mod in ("core", "imgproc", "features2d"):
        for name, modes in dispatched_files(ref, mod).items():
            if mod == "features2d" and name != "sift":
                continue
            for m in modes:
                src = os.path.join(GEN, mod, "%s.%s.cpp" % (name, m.lower()))
                units.append((src, os.path.join(OUT, "obj", "%s__disp__%s.%s.o" % (mod, name, m.lower())), mod))
    # our shim (includes the reference's sift.dispatch.cpp by path to reach its pyramid builders)
    units.append((os.path.join(HERE, "ref_shim.cpp"), os.path.join(OUT, "obj", "ref_shim.o"), "features2d"))

    def incs(mod):
        i = ["-I" + GEN, "-I" + os.path.join(GEN, mod)]
        for m in ("core", "imgproc", "flann", "features2d"):
            i.append("-I" + os.path.join(ref, "modules", m, "include"))
        i.append("-I" + os.path.join(ref, "modules", mod, "src"))
        return i

    ninja = ["rule cxx\n  command = g++ $flags -MMD -MF $out.d -c $in -o $out\n  depfile = $out.d\n  deps = gcc\n  description = CXX $in\n",
             "rule link\n  command = g++ -shared -o $out $in -pthread -ldl -lm -Wl,--gc-sections\n  description = LINK $out\n"]
    objs = []
    for src, obj, mod in units:
        flags = CXXFLAGS + incs(mod)
        sfx = os.path.basename(src).split(".")
        if len(sfx) == 3 and sfx[1].upper() in MODE_NAMES:      # X.avx2.cpp etc: built for that ISA
            flags = flags + mode_flags(sfx[1].upper())
        if src.endswith("ref_shim.cpp"):
            flags = flags + ["-fno-access-control", '-DREF_SIFT_DISPATCH_CPP=\\"%s\\"' % os.path.join(ref, "modules/features2d/src/sift.dispatch.cpp"),
                             "-fvisibility=default"]
        ninja.append("build %s: cxx %s\n  flags = %s\n" % (obj, src, " ".join(flags)))
        objs.append(obj)
    lib = os.path.join(OUT, "libocvref.so")
    ninja.append("build %s: link %s\n" % (lib, " ".join(objs)))
    defaults = [lib]
    if args.hal:
        repo = os.path.dirname(HERE)
        w(os.path.join(GEN, "hal_on", "custom_hal.hpp"),
          '#ifndef _CUSTOM_HAL_INCLUDED_\n#define _CUSTOM_HAL_INCLUDED_\n#include "b200cv_hal_replacement.hpp"\n#endif\n')
        hal_objs = []
        for src, obj, mod in units:
            if mod != "imgproc":
                hal_objs.append(obj)
                continue
            hobj = obj[:-2] + ".hal.o"
            flags = CXXFLAGS + ["-I" + os.path.join(GEN, "hal_on"), "-I" + os.path.join(repo, "hal"), "-I" + os.path.join(repo, "include")] + incs(mod)
            sfx = os.path.basename(src).split(".")
            if len(sfx) == 3 and sfx[1].upper() in MODE_NAMES:
                flags = flags + mode_flags(sfx[1].upper())
            ninja.append("build %s: cxx %s\n  flags = %s\n" % (hobj, src, " ".join(flags)))
            hal_objs.append(hobj)
        hlib = os.path.join(OUT, "libocvref_hal.so")
        b200 = os.path.join(repo, "opencv_b200", "lib")
        # ninja hands the command to /bin/sh: the quotes keep $ORIGIN literal, so the library finds libb200cv.so relative to itself
        # wherever the tree is moved to
        ninja.insert(2, "rule linkhal\n  command = g++ -shared -o $out $in -pthread -ldl -lm -Wl,--gc-sections -L%s -lb200cv '-Wl,-rpath,$$ORIGIN/../../opencv_b200/lib'\n  description = LINK $out\n" % b200)
        ninja.append("build %s: linkhal %s\n" % (hlib, " ".join(hal_objs)))
        defaults.append(hlib)
    ninja.append("default %s\n" % " ".join(defaults))
    os.makedirs(os.path.join(OUT, "obj"), exist_ok=True)
    w(os.path.join(OUT, "build.ninja"), "\n".join(ninja))
    r = subprocess.call(["ninja", "-C", OUT, "-j", str(args.j)])
    return r


if __name__ == "__main__":
    sys.exit(main())
