#!/usr/bin/env python3
"""Compile tests/cpp/test_cv_surface.cpp against the REAL OpenCV headers of the reference and link it with the reference's own core + imgproc
(oracle/_ref/libocvref.so) and libb200cv.so.  Needs the reference's sources, so the binary is built next to the reference library, under
oracle/_ref/, and runs wherever that directory is copied."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = "/root/reference"
EXE = os.path.join(ROOT, "oracle", "_ref", "test_cv_surface")


def build():
    if not os.path.isdir(os.path.join(REF, "modules", "core", "include")):
        return None
    gen = os.path.join(ROOT, "oracle", "_ref", "gen")
    ocv = os.path.join(ROOT, "oracle", "_ref")
    lib = os.path.join(ROOT, "opencv_b200", "lib")
    cmd = ["g++", "-std=c++17", "-O1", "-o", EXE, os.path.join(ROOT, "tests", "cpp", "test_cv_surface.cpp"),
           "-I" + gen, "-I" + os.path.join(REF, "modules", "core", "include"), "-I" + os.path.join(REF, "modules", "imgproc", "include"),
           "-L" + ocv, "-locvref", "-L" + lib, "-lb200cv", "-Wl,-rpath,$ORIGIN/../../opencv_b200/lib", "-Wl,-rpath,$ORIGIN", "-lpthread", "-lz"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("test_cv_surface: compilation against the OpenCV headers failed")
    return EXE


if __name__ == "__main__":
    print(build())
