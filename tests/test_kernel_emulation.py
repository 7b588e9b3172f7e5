"""CPU check of kernel LOGIC: simple kernels (no shared memory / warp intrinsics / barriers) are compiled for the host against
tests/emu/cuda_emu.h, their <<<grid, block, 0, st>>> launches run as plain loops over every thread, and the result is compared with the
oracle.  This exercises index arithmetic, plane layouts, tails and the aligned / unaligned access branches without a GPU.  It is not a
parity claim for the CUDA build -- that is what the -m gpu tests are for -- but it catches logic errors before GPU time is spent."""
import ctypes
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

from reference_replay import with_twin

ROOT =os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "opencv_b200", "csrc")
OUT = os.path.join(ROOT, "tests", "emu", "_build")
GOLD = os.path.join(ROOT, "tests", "golden")

LAUNCH = re.compile(r"(\b[\w:]+(?:<[^<>;]*>)?)<<<\s*grid\s*,\s*block\s*,\s*0\s*,\s*st\s*>>>\(([^;]*)\);")

STUBS = r"""
namespace b200cv {
void set_error(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap); fputc('\n', stderr); }
int cuda_fail(cudaError_t, const char*, const char*, int) { return -1; }
void count_launch(int) {}
int check_mat(const b200cvMat* m, const char*) { return m && m->data && m->cols > 0 && m->rows > 0 ? 0 : B200CV_ERR_BAD_ARG; }
}
"""


def build_emulation(cu_name, entry_decl, entry_body):
    os.makedirs(OUT, exist_ok=True)
    src = open(os.path.join(CSRC, cu_name)).read()
    translated, n = LAUNCH.subn(r"EMU_LAUNCH(grid, block, \1(\2));", src)
    assert n > 0 and "<<<" not in translated, "untranslated kernel launch left in %s" % cu_name
    tag = re.search(r"(\w+)\(", entry_decl).group(1)            # one library per entry point: a loaded .so is never overwritten
    cpp = os.path.join(OUT, tag + ".cpp")
    so = os.path.join(OUT, tag + ".so")
    with open(cpp, "w") as f:
        f.write("#define B200CV_HOST_EMULATION 1\n" + translated + STUBS + 'extern "C" ' + entry_decl + "\n{\n" + entry_body + "\n}\n")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-w", "-I", CSRC, "-I", os.path.join(ROOT, "tests", "emu"), cpp, "-o", so])
    return ctypes.CDLL(so)


def build_emulation_raw(cu_name, entry_decl, entry_body):
    """like build_emulation for sources whose __global__ kernels are compiled out on the host (TMA / shared memory): only their
    __device__ arithmetic cores are built"""
    os.makedirs(OUT, exist_ok=True)
    src = open(os.path.join(CSRC, cu_name)).read()
    tag = re.search(r"(\w+)\(", entry_decl).group(1)
    cpp = os.path.join(OUT, tag + ".cpp")
    so = os.path.join(OUT, tag + ".so")
    with open(cpp, "w") as f:
        f.write("#define B200CV_HOST_EMULATION 1\n" + src + STUBS + 'extern "C" ' + entry_decl + "\n{\n" + entry_body + "\n}\n")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-w", "-I", CSRC, "-I", os.path.join(ROOT, "tests", "emu"), cpp, "-o", so])
    return ctypes.CDLL(so)


class Mat(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("step", ctypes.c_size_t), ("cols", ctypes.c_int), ("rows", ctypes.c_int), ("type", ctypes.c_int),
                ("frames", ctypes.c_int), ("frame_step", ctypes.c_size_t)]


def mat_of(a):
    """(H,W) / (H,W,C) / (N,H,W,C) uint8 array (rows may be strided) -> b200cvMat"""
    if a.ndim == 4:
        n, h, w, c = a.shape
        return Mat(a.ctypes.data, a.strides[1], w, h, (c - 1) << 3, n, a.strides[0])
    h, w = a.shape[:2]
    c = 1 if a.ndim == 2 else a.shape[2]
    return Mat(a.ctypes.data, a.strides[0], w, h, (c - 1) << 3, 1, 0)


@pytest.fixture(scope="module")
def yuv_emu():
    lib = build_emulation("cvtcolor_yuv.cu", "int emu_cvt_color_yuv(const b200cvMat* s, const b200cvMat* d, int code)",
                          "    return b200cv::cvt_color_yuv(s, d, code, nullptr);")
    lib.emu_cvt_color_yuv.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat), ctypes.c_int]

    def run(src, code, dst=None):
        from oracle.api import yuv_dst_shape
        if src.ndim == 4:
            n, sh, sw = src.shape[:3]
            dw, dh, dcn = yuv_dst_shape(sw, sh, code)
            dst = np.full((n, dh, dw, dcn), 0xCD, np.uint8) if dst is None else dst
        else:
            sh, sw = src.shape[:2]
            dw, dh, dcn = yuv_dst_shape(sw, sh, code)
            dst = np.full((dh, dw) if dcn == 1 else (dh, dw, dcn), 0xCD, np.uint8) if dst is None else dst
        ms, md = mat_of(src), mat_of(dst)
        rc = lib.emu_cvt_color_yuv(ctypes.byref(ms), ctypes.byref(md), int(code))
        assert rc == 0, "emulated cvt_color_yuv(code %d) returned %d" % (code, rc)
        return dst
    return run


@pytest.fixture(scope="module")
def two_plane_emu():
    lib = build_emulation("cvtcolor_yuv.cu", "int emu_two_plane(const b200cvMat* y, const b200cvMat* uv, const b200cvMat* d, int code)",
                          "    return b200cv::cvt_color_two_plane(y, uv, d, code, nullptr);")
    lib.emu_two_plane.argtypes = [ctypes.POINTER(Mat)] * 3 + [ctypes.c_int]

    def run(y, uv, code):
        h, w = y.shape[:2]
        dst = np.zeros((h, w, 4 if code >= 94 else 3), np.uint8)
        my, muv, md = mat_of(y), mat_of(uv), mat_of(dst)
        rc = lib.emu_two_plane(ctypes.byref(my), ctypes.byref(muv), ctypes.byref(md), int(code))
        assert rc == 0, "emulated cvt_color_two_plane(code %d) returned %d" % (code, rc)
        return dst
    return run


def test_emulated_two_plane_vs_port(two_plane_emu, port, rng):
    for (h, w) in [(2, 2), (18, 34), (66, 130), (250, 322)]:
        y = rng.integers(0, 256, (h, w), dtype=np.uint8)
        wide = rng.integers(0, 256, (h // 2, w // 2 + 3, 2), dtype=np.uint8)
        uv = wide[:, 1:1 + w // 2]                                  # a pitch of its own, base address off by 2 bytes
        for code in range(90, 98):
            assert np.array_equal(two_plane_emu(y, uv, code), port.cvtColorTwoPlane(y, np.ascontiguousarray(uv), code)), "two-plane code %d %dx%d" % (code, w, h)


KAT_YUV = {90: 0x46a1bb76, 91: 0x3843bb76, 92: 0xf3fdf2ea, 93: 0x6e84f2ea, 94: 0xb6a16bd3, 95: 0xa8436bd3, 96: 0x1c7fa347, 97: 0x96f7a347,
           98: 0xc5da1651, 99: 0x12161651, 100: 0xb4e62ea5, 101: 0xfa632ea5, 102: 0x0db4c69f, 103: 0x59e1c69f, 104: 0xfe09def3, 105: 0x4395def3,
           106: 0xf672b440,
           107: 0x69bea2c1, 108: 0xdc51a2c1, 111: 0x851eab45, 112: 0xf7b1ab45, 115: 0x607e8889, 116: 0xfb148889, 117: 0x239b13d4, 118: 0x402b13d4,
           119: 0xf6af910d, 120: 0x9154910d, 121: 0x14481c58, 122: 0x30d81c58, 123: 0x228e669c, 124: 0x125c62fd,
           127: 0x44bb076a, 128: 0xf908ff52, 129: 0x44bb076a, 130: 0xf908ff52, 131: 0x1b0d076a, 132: 0xda8aff52, 133: 0x1b0d076a, 134: 0xda8aff52}


@pytest.mark.parametrize("code", sorted(KAT_YUV))
def test_emulated_yuv_kernels_reproduce_the_reference_hashes(yuv_emu, code):
    name = "cvtcolor_kat_yuv420_input.npy" if code <= 106 else "cvtcolor_kat_yuv422_input.npy" if code <= 124 else "cvtcolor_kat_bgr_262x254_input.npy"
    out = yuv_emu(np.load(os.path.join(GOLD, name)), code)
    assert zlib.adler32(np.ascontiguousarray(out).tobytes()) == KAT_YUV[code]


def test_emulated_yuv_kernels_vs_port(yuv_emu, port, rng):
    for (h, w) in [(2, 2), (4, 6), (18, 34), (36, 66), (66, 130), (250, 322)]:
        yuv = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
        for code in range(90, 107):
            assert np.array_equal(yuv_emu(yuv, code), port.cvtColorYUV(yuv, code)), "4:2:0 code %d %dx%d" % (code, w, h)
        y2 = rng.integers(0, 256, (h, w, 2), dtype=np.uint8)
        for code in (107, 108, 111, 112, 115, 116, 117, 118, 119, 120, 121, 122, 123, 124):
            assert np.array_equal(yuv_emu(y2, code), port.cvtColorYUV(y2, code)), "4:2:2 code %d %dx%d" % (code, w, h)
        for code in range(127, 135):
            img = rng.integers(0, 256, (h, w, 4 if (code - 127) & 2 else 3), dtype=np.uint8)
            assert np.array_equal(yuv_emu(img, code), port.cvtColorYUV(img, code)), "to 4:2:0 code %d %dx%d" % (code, w, h)


def test_emulated_bgr_to_yuv422_vs_port(yuv_emu, port, rng):
    for (h, w) in [(2, 2), (5, 6), (18, 34), (37, 130), (250, 322)]:
        for code in range(143, 155):
            for scn in (3, 4):
                img = rng.integers(0, 256, (h, w, scn), dtype=np.uint8)
                assert np.array_equal(yuv_emu(img, code), port.cvtColorYUV(img, code)), "to 4:2:2 code %d scn %d %dx%d" % (code, scn, w, h)
    # round trip through the emulated kernels: BGR -> YUY2 -> BGR stays within the 4:2:2 quantisation on a smooth image
    yy, xx = np.mgrid[0:64, 0:96]
    img = np.stack([(xx * 2) % 256, (yy * 3) % 256, (xx + yy) % 256], axis=-1).astype(np.uint8)
    back = yuv_emu(yuv_emu(img, 148), 116).astype(np.int32)
    assert np.percentile(np.abs(back - img.astype(np.int32)), 90) <= 8


def test_emulated_yuv_kernels_unaligned_pitches_and_batches(yuv_emu, port, rng):
    """odd base offsets / pitches force the byte paths; padded destinations must keep their padding; batches walk frame_step"""
    h, w = 34, 90
    wide = rng.integers(0, 256, (h * 3 // 2, w + 7), dtype=np.uint8)
    for off in (0, 1, 3, 4):
        src = wide[:, off:off + w]
        for code in (91, 96, 99, 104, 106):
            from oracle.api import yuv_dst_shape
            dw, dh, dcn = yuv_dst_shape(w, h * 3 // 2, code)
            big = np.full((dh, dw * dcn + 13), 0xEE, np.uint8)
            view = big[:, 5:5 + dw * dcn].reshape(dh, dw, dcn) if dcn > 1 else big[:, 5:5 + dw]
            yuv_emu(src, code, dst=view)
            assert np.array_equal(view, port.cvtColorYUV(np.ascontiguousarray(src), code)), "offset %d code %d" % (off, code)
            assert (big[:, :5] == 0xEE).all() and (big[:, 5 + dw * dcn:] == 0xEE).all(), "destination padding overwritten (offset %d code %d)" % (off, code)
    batch = rng.integers(0, 256, (3, 36, 40, 1), dtype=np.uint8)
    out = yuv_emu(batch, 91)
    for f in range(3):
        assert np.array_equal(out[f], port.cvtColorYUV(batch[f, :, :, 0], 91)), "batch frame %d" % f
    bgr = rng.integers(0, 256, (2, 26, 38, 3), dtype=np.uint8)
    out = yuv_emu(bgr, 132)
    for f in range(2):
        assert np.array_equal(out[f, :, :, 0], port.cvtColorYUV(bgr[f], 132)), "YV12 batch frame %d" % f


# ---- INTER_AREA (resize_area.cu) ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def area_emu():
    lib = build_emulation("resize_area.cu", "int emu_resize_area(const b200cvMat* s, const b200cvMat* d)",
                          "    return b200cv::resize_area_impl(b200cv::make_img(s), b200cv::make_img(d), B200CV_DEPTH(s->type), B200CV_CN(s->type), nullptr);")
    lib.emu_resize_area.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat)]

    def run(src, dsize):
        dw, dh = dsize
        dst = np.zeros((dh, dw) + src.shape[2:], src.dtype)
        ms, md = mat_of(src), mat_of(dst)
        if src.dtype == np.float32:
            ms.type |= 5; md.type |= 5
        rc = lib.emu_resize_area(ctypes.byref(ms), ctypes.byref(md))
        assert rc == 0, "emulated resize_area_impl returned %d" % rc
        return dst
    return run


def test_emulated_area_resize_vs_port(area_emu, port, rng):
    """integer factors (window sums) and fractional factors (DecimateAlpha weights derived per thread in double): bit-exact against the
    port, which tests/test_oracle.py pins to the reference"""
    cases = [((120, 180), (40, 60)), ((120, 180), (30, 90)), ((121, 183), (40, 61)), ((100, 150), (37, 41)), ((97, 131), (96, 130)),
             ((64, 64), (16, 16)), ((90, 120), (30, 24)), ((50, 70), (49, 23)), ((33, 47), (1, 1)), ((300, 400), (7, 399)), ((240, 320), (150, 200))]
    for (sh, sw), (dh, dw) in cases:
        for cn in (1, 3, 4):
            shape = (sh, sw) if cn == 1 else (sh, sw, cn)
            u8 = rng.integers(0, 256, shape, dtype=np.uint8)
            f32 = (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)
            for img in (u8, f32):
                if sh == 2 * dh and sw == 2 * dw:
                    continue                                   # 2 x 2: resize.cu's own path
                got, want = area_emu(img, (dw, dh)), port.resize(img, (dw, dh), 3)
                assert np.array_equal(got, want), "INTER_AREA %s %s -> %s cn=%d" % (img.dtype, (sh, sw), (dh, dw), cn)


# ---- INTER_NEAREST_EXACT / INTER_LINEAR_EXACT (resize_exact.cu) -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def exact_emu():
    lib = build_emulation("resize_exact.cu", "int emu_resize_exact(const b200cvMat* s, const b200cvMat* d, int interp)",
                          "    return b200cv::resize_exact_impl(b200cv::make_img(s), b200cv::make_img(d), B200CV_DEPTH(s->type), B200CV_CN(s->type), interp, nullptr);")
    lib.emu_resize_exact.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat), ctypes.c_int]

    def run(src, dsize, interp):
        dw, dh = dsize
        dst = np.zeros((dh, dw) + src.shape[2:], src.dtype)
        ms, md = mat_of(src), mat_of(dst)
        if src.dtype == np.float32:
            ms.type |= 5; md.type |= 5
        rc = lib.emu_resize_exact(ctypes.byref(ms), ctypes.byref(md), interp)
        assert rc == 0, "emulated resize_exact_impl returned %d" % rc
        return dst
    return run


EXACT_CASES = [((120, 180), (40, 60)), ((121, 183), (40, 61)), ((100, 150), (237, 341)), ((97, 131), (96, 130)), ((64, 64), (160, 160)),
               ((1, 47), (5, 90)), ((50, 1), (49, 23)), ((33, 47), (1, 1)), ((300, 400), (7, 399)), ((2, 2), (9, 9)), ((3, 5), (30, 50))]


def test_emulated_resizers_reproduce_the_reference_goldens(exact_emu, area_emu):
    """Resize_Bitexact.Nearest8U and the Imgproc_resize_area rounding regressions (the reference's own expected outputs), through the kernels"""
    from test_oracle import resize_golden_cases
    for src, dsize, interp, want, tol in resize_golden_cases():
        if interp == 6:
            got = exact_emu(src, dsize, 6)
        elif src.shape[0] == 2 * dsize[1]:
            continue                                        # exact 2 x 2: resize.cu's verified path, not in this file
        else:
            got = area_emu(src, dsize)
        assert np.abs(got.astype(int) - want.astype(int)).max() <= tol, "interp %d %s -> %s" % (interp, src.shape, dsize)


def test_emulated_exact_resizers_vs_port(exact_emu, port, rng):
    for (sh, sw), (dh, dw) in EXACT_CASES:
        for cn in (1, 3, 4):
            shape = (sh, sw) if cn == 1 else (sh, sw, cn)
            u8 = rng.integers(0, 256, shape, dtype=np.uint8)
            f32 = (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)
            assert np.array_equal(exact_emu(u8, (dw, dh), 5), port.resize(u8, (dw, dh), 5)), "LINEAR_EXACT %s -> %s cn=%d" % ((sh, sw), (dh, dw), cn)
            for img in (u8, f32):
                assert np.array_equal(exact_emu(img, (dw, dh), 6), port.resize(img, (dw, dh), 6)), "NEAREST_EXACT %s %s -> %s cn=%d" % (img.dtype, (sh, sw), (dh, dw), cn)


# ---- INTER_LANCZOS4 (resize_lanczos.cu): host-built weight tables + the per-element kernel ------------------------------------------------
@pytest.fixture(scope="module")
def lanczos_emu():
    lib = build_emulation("resize_lanczos.cu", "int emu_resize_lanczos(const b200cvMat* s, const b200cvMat* d)",
                          "    return b200cv::resize_lanczos_impl(b200cv::make_img(s), b200cv::make_img(d), B200CV_DEPTH(s->type), B200CV_CN(s->type), nullptr);")
    lib.emu_resize_lanczos.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat)]

    def run(src, dsize):
        dw, dh = dsize
        dst = np.zeros((dh, dw) + src.shape[2:], src.dtype)
        ms, md = mat_of(src), mat_of(dst)
        if src.dtype == np.float32:
            ms.type |= 5; md.type |= 5
        rc = lib.emu_resize_lanczos(ctypes.byref(ms), ctypes.byref(md))
        assert rc == 0, "emulated resize_lanczos_impl returned %d" % rc
        return dst
    return run


def test_emulated_lanczos4_resize_vs_port(lanczos_emu, port, rng):
    cases = [((40, 60), (120, 180)), ((40, 60), (97, 131)), ((100, 150), (237, 341)), ((97, 131), (98, 132)), ((64, 64), (160, 32)), ((120, 180), (40, 61)),
             ((1, 47), (5, 90)), ((50, 1), (75, 23)), ((3, 5), (30, 50)), ((120, 160), (121, 100)), ((240, 320), (150, 201))]
    for (sh, sw), (dh, dw) in cases:
        for cn in (1, 3, 4):
            shape = (sh, sw) if cn == 1 else (sh, sw, cn)
            for img in (rng.integers(0, 256, shape, dtype=np.uint8), (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)):
                assert np.array_equal(lanczos_emu(img, (dw, dh)), port.resize(img, (dw, dh), 4)), "LANCZOS4 %s %s -> %s cn=%d" % (img.dtype, (sh, sw), (dh, dw), cn)


# ---- Bayer mosaics, bilinear (demosaic.cu) --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bayer_emu():
    lib = build_emulation("demosaic.cu", "int emu_demosaic(const b200cvMat* s, const b200cvMat* d, int code)",
                          "    return b200cv::demosaic_bilinear(s, d, code, nullptr);")
    lib.emu_demosaic.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat), ctypes.c_int]

    def run(src, code):
        dcn = 4 if code >= 139 else 3
        dst = np.full(src.shape[:-1] + (dcn,) if src.ndim == 4 else src.shape + (dcn,), 0xCD, np.uint8)
        ms, md = mat_of(src), mat_of(dst)
        rc = lib.emu_demosaic(ctypes.byref(ms), ctypes.byref(md), int(code))
        assert rc == 0, "emulated demosaic_bilinear(code %d) returned %d" % (code, rc)
        return dst
    return run


def test_emulated_bayer_demosaic_vs_port(bayer_emu, port, rng):
    for (h, w) in [(3, 3), (4, 5), (5, 4), (17, 33), (18, 34), (64, 96), (241, 323)]:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        for code in (46, 47, 48, 49, 139, 140, 141, 142):
            assert np.array_equal(bayer_emu(img, code), port.cvtColorYUV(img, code)), "Bayer code %d %dx%d" % (code, w, h)
    batch = rng.integers(0, 256, (3, 20, 26, 1), dtype=np.uint8)
    out = bayer_emu(batch, 48)
    for f in range(3):
        assert np.array_equal(out[f], port.cvtColorYUV(batch[f, :, :, 0], 48)), "Bayer batch frame %d" % f


# ---- cvtColor on 16-bit / float images (cvtcolor_depth.cu) and the edge-aware / 16-bit Bayer codes (demosaic.cu) against the compiled reference ----
@pytest.fixture(scope="module")
def depth_emu():
    lib = build_emulation("cvtcolor_depth.cu", "int emu_cvt_depth(const b200cvMat* s, const b200cvMat* d, int code)",
                          "    return b200cv::cvt_color_depth(s, d, code, nullptr);")
    lib.emu_cvt_depth.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat), ctypes.c_int]

    def run(src, code, dcn):
        dst = np.zeros(src.shape[:2] if dcn == 1 else src.shape[:2] + (dcn,), src.dtype)
        depth = {np.dtype(np.uint16): 2, np.dtype(np.float32): 5}[src.dtype]
        ms, md = mat_of(src), mat_of(dst)
        ms.type = depth | (((1 if src.ndim == 2 else src.shape[2]) - 1) << 3)
        md.type = depth | ((dcn - 1) << 3)
        rc = lib.emu_cvt_depth(ctypes.byref(ms), ctypes.byref(md), int(code))
        assert rc == 0, "emulated cvt_color_depth(code %d) returned %d" % (code, rc)
        return dst
    return run


def test_emulated_depth_cvtcolor_vs_reference(depth_emu, ref, rng):
    """the kernel source of cvtcolor_depth.cu compiled for the host == the compiled reference, bit for bit (vector bodies and scalar tails)"""
    ref = with_twin(ref, cvtColor=depth_emu)
    for (h, w) in [(9, 29), (5, 64), (3, 7)]:
        f3 = (rng.random((h, w, 3), dtype=np.float32) * 1.5 - 0.25).astype(np.float32)
        w3 = rng.integers(0, 65536, (h, w, 3), dtype=np.uint16)
        for src in (f3, w3):
            for code, dcn in ((0, 4), (4, 3), (6, 1), (7, 1), (36, 3), (37, 3), (82, 3), (83, 3), (38, 3), (39, 4), (84, 3), (85, 3), (32, 3), (33, 3), (34, 3), (35, 4)):
                assert np.array_equal(depth_emu(src, code, dcn), ref.cvtColor(src, code, dcn)), "%s code %d %dx%d" % (src.dtype, code, w, h)
        hsv = np.stack([rng.random((h, w), dtype=np.float32) * np.float32(420) - np.float32(30), rng.random((h, w), dtype=np.float32),
                        rng.random((h, w), dtype=np.float32)], -1).astype(np.float32)
        hsv[0, :, 1] = 0
        for code, dcn in ((40, 3), (41, 3), (66, 3), (67, 3)):
            assert np.array_equal(depth_emu(f3, code, dcn), ref.cvtColor(f3, code, dcn)), "f32 to HSV code %d %dx%d" % (code, w, h)
        for code, dcn in ((54, 3), (55, 3), (70, 4), (71, 3)):
            assert np.array_equal(depth_emu(hsv, code, dcn), ref.cvtColor(hsv, code, dcn)), "f32 from HSV code %d %dx%d" % (code, w, h)
        g = rng.integers(0, 65536, (h, w), dtype=np.uint16)
        assert np.array_equal(depth_emu(g, 8, 3), ref.cvtColor(g, 8, 3)) and np.array_equal(depth_emu(g.astype(np.float32), 9, 4), ref.cvtColor(g.astype(np.float32), 9, 4))


def test_emulated_bayer_edge_aware_and_16bit_vs_reference(ref, rng):
    lib = build_emulation("demosaic.cu", "int emu_demosaic_any(const b200cvMat* s, const b200cvMat* d, int code)",
                          "    return b200cv::demosaic_bilinear(s, d, code, nullptr);")
    lib.emu_demosaic_any.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat), ctypes.c_int]

    def emu(img, code, dcn):
        depth = 0 if img.dtype == np.uint8 else 2
        dst = np.zeros(img.shape + (dcn,), img.dtype)
        ms, md = mat_of(img), mat_of(dst)
        ms.type = depth; md.type = depth | ((dcn - 1) << 3)
        assert lib.emu_demosaic_any(ctypes.byref(ms), ctypes.byref(md), code) == 0
        return dst
    ref = with_twin(ref, cvtColor=emu)
    for dtype, depth in ((np.uint8, 0), (np.uint16, 2)):
        for (h, w) in [(3, 3), (4, 5), (17, 33), (18, 34)]:
            img = rng.integers(0, 256 if depth == 0 else 65536, (h, w)).astype(dtype)
            for code, dcn in ((135, 3), (136, 3), (137, 3), (138, 3)) + (((46, 3), (49, 3), (140, 4)) if depth else ()):
                assert np.array_equal(emu(img, code, dcn), ref.cvtColor(img, code, dcn)), "Bayer %s code %d %dx%d" % (np.dtype(dtype).name, code, w, h)


# ---- cv::integral (integral.cu): six map-only kernels ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def integral_emu():
    lib = build_emulation("integral.cu", "int emu_integral(const b200cvMat* s, const b200cvMat* sum, const b200cvMat* sq)",
                          "    return b200cv::integral_impl(s, sum, sq, nullptr);")
    lib.emu_integral.argtypes = [ctypes.POINTER(Mat)] * 3

    def run(src, with_sq):
        lead = src.shape[:1] if src.ndim == 4 else ()
        h, w = src.shape[-3:-1] if src.ndim == 4 else src.shape
        tail = (1,) if src.ndim == 4 else ()
        s = np.full(lead + (h + 1, w + 1) + tail, -7, np.int32)
        q = np.full(lead + (h + 1, w + 1) + tail, -7.0, np.float64)
        ms, md, mq = mat_of(src), mat_of(s), mat_of(q)
        md.type = 4; mq.type = 6
        rc = lib.emu_integral(ctypes.byref(ms), ctypes.byref(md), ctypes.byref(mq) if with_sq else None)
        assert rc == 0, "emulated integral_impl returned %d" % rc
        return (s, q) if with_sq else s
    return run


def test_emulated_integral_vs_port(integral_emu, port, rng):
    for (h, w) in [(1, 1), (5, 7), (16, 16), (17, 15), (33, 65), (100, 257), (240, 321)]:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        ws, wq = port.integral(img, True)
        gs, gq = integral_emu(img, True)
        assert np.array_equal(gs, ws) and np.array_equal(gq, wq), "integral %dx%d" % (w, h)
        assert np.array_equal(integral_emu(img, False), ws)
    batch = rng.integers(0, 256, (3, 40, 50, 1), dtype=np.uint8)
    gs = integral_emu(batch, False)
    for f in range(3):
        assert np.array_equal(gs[f, :, :, 0], port.integral(batch[f, :, :, 0])), "integral batch frame %d" % f


# ---- SIFT extrema / refinement / orientation / descriptors (sift_detect.cu) -----------------------------------------------------------------
@pytest.fixture(scope="module")
def sift_emu():
    lib = build_emulation("sift_detect.cu", "int emu_sift(const float* g, const float* d, const int* dims, int no, int nl, double ct, double et, double sigma, "
                          "int first_octave, int nfeatures, const unsigned char* mask, size_t mstep, int mw, int mh, int max_kp, float* kp, float* desc, int* n)",
                          "    return b200cv::sift_detect_impl(g, d, dims, no, nl, ct, et, sigma, first_octave, nfeatures, mask, mstep, mw, mh, max_kp, kp, desc, n, nullptr);")

    def run(gauss, dog, nl=3, ct=0.04, et=10.0, sigma=1.6, max_kp=100000, nfeatures=0, mask=None):
        no = len(gauss)
        dims = np.array([[g[0].shape[1], g[0].shape[0]] for g in gauss], np.int32).reshape(-1)
        G = np.concatenate([np.ascontiguousarray(l, np.float32).reshape(-1) for g in gauss for l in g])
        D = np.concatenate([np.ascontiguousarray(l, np.float32).reshape(-1) for d in dog for l in d])
        kp = np.zeros((max_kp, 6), np.float32); desc = np.zeros((max_kp, 128), np.float32); n = ctypes.c_int(0)
        fp = ctypes.POINTER(ctypes.c_float)
        rc = lib.emu_sift(G.ctypes.data_as(fp), D.ctypes.data_as(fp), dims.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), no, nl, ctypes.c_double(ct),
                          ctypes.c_double(et), ctypes.c_double(sigma), -1, nfeatures,
                          mask.ctypes.data_as(ctypes.c_void_p) if mask is not None else None, ctypes.c_size_t(mask.strides[0] if mask is not None else 0),
                          mask.shape[1] if mask is not None else 0, mask.shape[0] if mask is not None else 0,
                          max_kp, kp.ctypes.data_as(fp), desc.ctypes.data_as(fp), ctypes.byref(n))
        assert rc == 0, "emulated sift_detect_impl returned %d" % rc
        return kp[:n.value, :5].copy(), kp[:n.value, 5].copy().view(np.int32), desc[:n.value].copy()
    return run


def test_emulated_sift_front_end_vs_port(sift_emu, port, rng):
    """the three kernels + the host-side sort / duplicate removal, run on the host, against the port on the same (port-built) pyramids:
    same float expressions, same libm -> identical keypoints and descriptors"""
    small = rng.random((22, 30)).astype(np.float32)
    img = np.kron(small, np.ones((8, 8), np.float32))[:160, :220] + 0.15 * rng.random((160, 220)).astype(np.float32)
    img = ((img - img.min()) / (img.max() - img.min()) * 255).astype(np.uint8)
    G, D = port.sift_pyramid(img)
    kp, octv = port.sift_detect_from_pyramid(G, D)
    gk, go, gd = sift_emu(G, D)
    assert len(gk) == len(kp) and len(kp) > 100
    assert np.array_equal(gk, kp) and np.array_equal(go, octv), "keypoints"
    assert np.array_equal(gd, port.sift_descriptors_from_pyramid(G, kp, octv)), "descriptors"
    # nfeatures: the strongest responses, ties included -- the same SET as the port's (the order after nth_element / partition is the library's)
    bk, bo, bd = sift_emu(G, D, nfeatures=50)
    pk, po = port.sift_detect_from_pyramid(G, D, nfeatures=50)
    assert 50 <= len(bk) == len(pk) and sorted(map(tuple, bk.tolist())) == sorted(map(tuple, pk.tolist()))
    assert bk[:, 4].min() >= np.sort(kp[:, 4])[-50]
    # mask (KeyPointsFilter::runByPixelsMask): keypoints whose rounded position has a zero mask byte disappear, with their descriptors
    mask = np.zeros(img.shape, np.uint8); mask[40:120, 60:180] = 255
    mk, mo, md = sift_emu(G, D, mask=mask)
    keep = mask[(kp[:, 1] + 0.5).astype(np.int32), (kp[:, 0] + 0.5).astype(np.int32)] != 0
    assert 0 < keep.sum() < len(kp) and np.array_equal(mk, kp[keep]) and np.array_equal(md, gd[keep])


# ---- BGR / RGB <-> Lab, 8-bit (cvtcolor_lab.cu): host-built tables + per-pixel kernels ----------------------------------------------------
@pytest.fixture(scope="module")
def lab_emu():
    lib = build_emulation("cvtcolor_lab.cu", "int emu_lab(const b200cvMat* s, const b200cvMat* d, int code)",
                          "    return code >= 32 && code <= 35 ? b200cv::cvt_color_xyz(s, d, code, nullptr) : b200cv::cvt_color_lab(s, d, code, nullptr);")
    lib.emu_lab.argtypes = [ctypes.POINTER(Mat), ctypes.POINTER(Mat), ctypes.c_int]

    def run(src, code, dcn=3):
        dst = np.zeros(src.shape[:-1] + (dcn,), np.uint8)
        ms, md = mat_of(src), mat_of(dst)
        rc = lib.emu_lab(ctypes.byref(ms), ctypes.byref(md), int(code))
        assert rc == 0, "emulated cvt_color_lab(code %d) returned %d" % (code, rc)
        return dst
    return run


def test_emulated_lab_kernels_vs_port(lab_emu, port, rng):
    """a 1/64 sample of the colour cube (every 4th level of each channel, 262 144 colours, all table regions) plus random data, both directions,
    sRGB and linear; the port itself equals the reference on all 2^24 colours (tests/test_oracle.py)"""
    v = np.arange(0, 256, 4, dtype=np.uint8)
    cube = np.stack(np.meshgrid(v, v, v, indexing="ij"), axis=-1).reshape(512, 512, 3)
    rnd = rng.integers(0, 256, (97, 131, 3), dtype=np.uint8)
    for img in (cube, rnd):
        for code in (44, 45, 74, 75, 56, 57, 78, 79, 32, 33, 34, 35):
            assert np.array_equal(lab_emu(img, code), port.cvtColorLab(img, code)), "Lab / XYZ code %d" % code
    bgra = rng.integers(0, 256, (40, 50, 4), dtype=np.uint8)
    assert np.array_equal(lab_emu(bgra, 44), port.cvtColorLab(np.ascontiguousarray(bgra[:, :, :3]), 44)), "4-channel source"
    out4 = lab_emu(rnd, 56, dcn=4)
    assert np.array_equal(out4[:, :, :3], port.cvtColorLab(rnd, 56)) and (out4[:, :, 3] == 255).all()


# ---- the one piece of the INTER_AREA enlargement that lives in resize.cu (not emulated as a whole: it uses IDP2A / PRMT): linear_coef() ----------
def test_emulated_area_mode_weights_in_resize_cu():
    """extract the device function linear_coef from resize.cu, compile it for the host and compare its area-mode branch with the reference's
    expressions (resize.cpp:4104-4109, :4158-4163) evaluated in numpy: s = floor(d * scale), f = float((d + 1) - (s + 1) * inv_scale), f <= 0 -> 0,
    else f - floor(f); and its default branch with f = float((d + 0.5) * scale - 0.5), s = floor(f), f -= s"""
    os.makedirs(OUT, exist_ok=True)
    src = open(os.path.join(CSRC, "resize.cuh")).read()
    m = re.search(r"__device__ __forceinline__ void linear_coef\(.*?\n}\n", src, re.S)
    assert m, "linear_coef not found in resize.cuh"
    fn = m.group(0).replace("bool area_mode = false, double inv_scale = 0.", "bool area_mode, double inv_scale")
    cpp = os.path.join(OUT, "emu_linear_coef.cpp")
    so = os.path.join(OUT, "emu_linear_coef.so")
    with open(cpp, "w") as f:
        f.write('#include "cuda_emu.h"\n' + fn +
                'extern "C" void emu_linear_coef(int n, double scale, int ssize, int clamp, int area, double inv, int* s, float* fr)\n'
                "{ for (int d = 0; d < n; d++) linear_coef(d, scale, ssize, s[d], fr[d], clamp != 0, area != 0, inv); }\n")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-w", "-I", os.path.join(ROOT, "tests", "emu"), cpp, "-o", so])
    lib = ctypes.CDLL(so)
    for ssize, dsize in [(60, 180), (131, 997), (47, 90), (1, 23), (640, 641), (5, 50)]:
        inv = dsize / ssize
        scale = 1.0 / inv
        s = np.zeros(dsize, np.int32); fr = np.zeros(dsize, np.float32)
        for clamp in (0, 1):
            lib.emu_linear_coef(dsize, ctypes.c_double(scale), ssize, clamp, 1, ctypes.c_double(inv), s.ctypes.data_as(ctypes.c_void_p), fr.ctypes.data_as(ctypes.c_void_p))
            d = np.arange(dsize, dtype=np.float64)
            ws = np.floor(d * scale).astype(np.int32)
            wf = ((d + 1) - (ws + 1).astype(np.float64) * inv).astype(np.float32)
            wf = np.where(wf <= 0, np.float32(0), wf - np.floor(wf)).astype(np.float32)
            if clamp:
                lo, hi = ws < 0, ws >= ssize - 1
                wf = np.where(lo | hi, np.float32(0), wf); ws = np.where(lo, 0, np.where(hi, ssize - 1, ws))
            assert np.array_equal(s, ws) and np.array_equal(fr, wf), "area-mode weights %d -> %d clamp=%d" % (ssize, dsize, clamp)
        lib.emu_linear_coef(dsize, ctypes.c_double(scale), ssize, 0, 0, ctypes.c_double(inv), s.ctypes.data_as(ctypes.c_void_p), fr.ctypes.data_as(ctypes.c_void_p))
        f0 = ((np.arange(dsize, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
        s0 = np.floor(f0).astype(np.int32)
        assert np.array_equal(s, s0) and np.array_equal(fr, (f0 - s0.astype(np.float32)).astype(np.float32)), "default weights %d -> %d" % (ssize, dsize)


# ---- cv::matchTemplate with a mask (matchtemplate_mask.cu): preparation kernel + one thread per result element -----------------------------
@pytest.fixture(scope="module")
def mtmask_emu():
    lib = build_emulation("matchtemplate_mask.cu", "int emu_mt_mask(const b200cvMat* i, const b200cvMat* t, const b200cvMat* m, const b200cvMat* r, int method)",
                          "    return b200cv::match_template_masked(i, t, m, r, method, nullptr);")
    lib.emu_mt_mask.argtypes = [ctypes.POINTER(Mat)] * 4 + [ctypes.c_int]

    def run(img, templ, mask, method):
        res = np.zeros((img.shape[0] - templ.shape[0] + 1, img.shape[1] - templ.shape[1] + 1), np.float32)
        mats = [mat_of(a) for a in (img, templ, mask, res)]
        for a, m in zip((img, templ, mask, res), mats):
            if a.dtype == np.float32:
                m.type |= 5
        rc = lib.emu_mt_mask(*[ctypes.byref(m) for m in mats], int(method))
        assert rc == 0, "emulated match_template_masked returned %d" % rc
        return res
    return run


def test_emulated_masked_match_template_vs_port(mtmask_emu, port, rng):
    img = rng.integers(0, 256, (60, 80), dtype=np.uint8)
    templ = img[20:33, 30:51].copy()
    m8 = (rng.random(templ.shape) > 0.3).astype(np.uint8) * 255
    mf = rng.random(templ.shape).astype(np.float32)
    for im, tt in ((img, templ), (img.astype(np.float32), templ.astype(np.float32))):
        for mk in (m8, mf):
            for method in range(6):
                got, want = mtmask_emu(im, tt, mk, method), port.matchTemplateMasked(im, tt, method, mk)
                assert np.array_equal(got, want), "masked matchTemplate %s mask %s method %d" % (im.dtype, mk.dtype, method)


# ---- GaussianBlur CV_16U, 16.16 fixed point (gauss_u16.cu) ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gauss16_emu(port):
    lib = build_emulation("gauss_u16.cu", "int emu_gauss_u16(const b200cvMat* s, const b200cvMat* d, const long long* fx, int kw, const long long* fy, int kh, int border)",
                          "    return b200cv::gauss_u16_impl(b200cv::make_img(s), b200cv::make_img(d), B200CV_CN(s->type), fx, kw, fy, kh, border, nullptr);")

    def run(img, k, sigma, border):
        fx = np.zeros(k, np.int64)
        port.lib.port_gaussian_taps_fixed(k, ctypes.c_double(sigma), 16, fx.ctypes.data_as(ctypes.c_void_p))
        dst = np.zeros_like(img)
        ms, md = mat_of(img), mat_of(dst)
        ms.type |= 2; md.type |= 2
        lp = ctypes.POINTER(ctypes.c_longlong)
        rc = lib.emu_gauss_u16(ctypes.byref(ms), ctypes.byref(md), fx.ctypes.data_as(lp), k, fx.ctypes.data_as(lp), k, border)
        assert rc == 0, "emulated gauss_u16_impl returned %d" % rc
        return dst
    return run


def test_emulated_gaussian_u16_vs_port(gauss16_emu, port, rng):
    import opencv_b200 as C
    for shape in [(37, 53), (40, 66, 3), (20, 31, 4), (1, 40), (33, 1)]:
        img = rng.integers(0, 65536, shape, dtype=np.uint16)
        ext = np.where(rng.random(shape) < 0.5, 0, 65535).astype(np.uint16)
        for im in (img, ext):
            for k, s in [(3, 0), (5, 0), (7, 1.5), (15, 3.0), (31, 0)]:
                if (shape[0] == 1 or shape[1] == 1):
                    continue                              # 1-pixel dimensions shrink the kernel in the dispatcher (smooth.dispatch.cpp:624-631), not in this file
                for border in (4, 1, 0, 2, 3):
                    assert np.array_equal(gauss16_emu(im, k, s, border), port.GaussianBlur(im, (k, k), s, s, border)), "u16 %s k=%d s=%g border=%d" % (shape, k, s, border)
    # the product's own 16-bit taps (host_tables.cpp, softdouble exp) are the port's
    for k, s in [(3, 0), (5, 0), (7, 1.5), (9, 0), (15, 3.0), (31, 0), (5, 0.3), (13, 2.2)]:
        want = np.zeros(k, np.int64)
        port.lib.port_gaussian_taps_fixed(k, ctypes.c_double(s), 16, want.ctypes.data_as(ctypes.c_void_p))
        assert list(C.getGaussianKernelFixed(k, s, 16)) == list(want) and int(want.sum()) == 65536, "16-bit taps k=%d sigma=%g" % (k, s)


# ---- GaussianBlur / 8.8 sepFilter2D CV_8UC1, K <= 9: the warp-streaming kernel (gauss_u8_march.cu) ------------------------------------------
# TMA and mbarriers cannot run on the host; everything a lane does with a staged chunk can.  The test walks the kernel's own work
# decomposition (items -> chunks), stages every 256 x CH chunk with cv::borderInterpolate (what the TMA zero fill, the row-wise mirrored
# loads and the apron patch produce together) and runs gm_lane_chunk for the 32 lanes, each with its register window carried across chunks.
@pytest.fixture(scope="module")
def gauss_march_emu(port):
    body = r"""
    using namespace b200cv;
    Img si = make_img(s), di = make_img(d);
    GMParams p; gm_fill_params(p, KB, tx, ty);
    p.W = si.cols; p.H = si.rows; p.border = border; p.sep_mode = sep_mode; p.even_limit = even_limit;
    const int H = KB / 2, CH = KB == 3 ? GMCfg<3>::CH : KB == 5 ? GMCfg<5>::CH : KB == 7 ? GMCfg<7>::CH : GMCfg<9>::CH;
    p.tiles_x = (p.W + GM_OW - 1) / GM_OW;
    p.seg_rows = ((seg_rows + CH - 1) / CH) * CH; p.nseg = (p.H + p.seg_rows - 1) / p.seg_rows; p.nitems = p.tiles_x * p.nseg * si.frames;
    unsigned char* buf = (unsigned char*)malloc((size_t)GM_IW * CH);
#define RUN(K, SEP) do { for (int item = 0; item < p.nitems; item++) { const GMItem g = gm_item<K>(p, item); \
        for (int lane = 0; lane < 32; lane++) { uint32_t win[GMCfg<K>::NP][8]; memset(win, 0x5A, sizeof(win)); \
            for (int chunk = 0; chunk < g.nchunks; chunk++) { \
                for (int r = 0; r < CH; r++) for (int c = 0; c < GM_IW; c++) { \
                    const int gy = g.ys - H + chunk * CH + r, gx = g.x0 - GM_RA + c; \
                    const int sy = border_interpolate(gy, p.H, border), sx = border_interpolate(gx, p.W, border); \
                    buf[r * GM_IW + c] = (sy < 0 || sx < 0) ? 0 : si.row<unsigned char>(g.f, sy)[sx]; } \
                gm_lane_chunk<K, SEP>(buf, lane, p, di, g, chunk, win); } } } } while (0)
    if (sep_mode) { if (KB == 3) RUN(3, true); else if (KB == 5) RUN(5, true); else if (KB == 7) RUN(7, true); else RUN(9, true); }
    else { if (KB == 3) RUN(3, false); else if (KB == 5) RUN(5, false); else if (KB == 7) RUN(7, false); else RUN(9, false); }
    free(buf);
    return 0;"""
    lib = build_emulation_raw("gauss_u8_march.cu", "int emu_gauss_march(const b200cvMat* s, const b200cvMat* d, int KB, const unsigned char* tx, const unsigned char* ty, int border, int sep_mode, int even_limit, int seg_rows)", body)

    def run(img, k, sigma, border, sep=False, seg_rows=64):
        fx = np.zeros(k, np.int64)
        port.lib.port_gaussian_taps_fixed(k, ctypes.c_double(sigma), 8, fx.ctypes.data_as(ctypes.c_void_p))
        assert fx.sum() == 256 and fx.max() <= 255
        t = fx.astype(np.uint8)
        dst = np.full_like(img, 0xCD)
        ms, md = mat_of(img), mat_of(dst)
        even_limit = (img.shape[-1] // 16) * 16 if sep else 0           # sepfilter.cu: ((cols * cn) / 16) * 16
        rc = lib.emu_gauss_march(ctypes.byref(ms), ctypes.byref(md), k, t.ctypes.data_as(ctypes.c_void_p), t.ctypes.data_as(ctypes.c_void_p), border, int(sep), even_limit, seg_rows)
        assert rc == 0
        return (dst, (t / 256.0).astype(np.float32)) if sep else dst
    return run


def test_emulated_gaussian_march_vs_port(gauss_march_emu, port, rng):
    for shape in [(37, 53), (150, 250), (131, 224), (300, 449), (200, 448), (2, 40, 230, 1)]:
        img = rng.integers(0, 256, shape, dtype=np.uint8)
        ext = np.where(rng.random(shape) < 0.5, 0, 255).astype(np.uint8)
        for im in (img, ext):
            for k, s in [(3, 0), (5, 0), (7, 0), (9, 0), (5, 1.7), (9, 2.5)]:
                for border in (4, 1, 0, 2):
                    got = gauss_march_emu(im, k, s, border, seg_rows=(64 if border != 1 else 1000))
                    if im.ndim == 4:
                        want = np.stack([port.GaussianBlur(im[i, :, :, 0], (k, k), s, s, border) for i in range(im.shape[0])])[..., None]
                    else:
                        want = port.GaussianBlur(im, (k, k), s, s, border)
                    assert np.array_equal(got, want), "u8 march %s k=%d s=%g border=%d" % (shape, k, s, border)


def test_emulated_sepfilter_8p8_march_vs_port(gauss_march_emu, port, rng):
    """sepFilter2D's 8.8 fixed-point mode on the same kernel: half-to-even in the reference's vector body, half-up in its tail"""
    for shape in [(37, 53), (150, 250), (64, 241)]:
        img = rng.integers(0, 256, shape, dtype=np.uint8)
        for k, s in [(3, 0), (5, 0), (7, 0), (9, 0)]:
            for border in (4, 1, 0, 2):
                got, taps = gauss_march_emu(img, k, s, border, sep=True)
                want = port.sepFilter2D(img, -1, taps, taps, borderType=border)
                assert np.array_equal(got, want), "u8 8.8 sepFilter2D march %s k=%d border=%d" % (shape, k, border)


# ---- cv::resize INTER_LINEAR / INTER_CUBIC, 8-bit, tiled separable kernels (resize_sep.cu) ----------------------------------------------------
# The kernel's shared-memory tile becomes a plain array; the H pass runs for all 256 threads, then the V pass (what the barrier separates).
@pytest.fixture(scope="module")
def resize_sep_emu():
    body = r"""
    using namespace b200cv;
    Img si = make_img(s), di = make_img(d);
    ResizeParams p;
    p.sw = si.cols; p.sh = si.rows; p.dw = di.cols; p.dh = di.rows;
    const double inv_x = (double)p.dw / p.sw, inv_y = (double)p.dh / p.sh;
    p.ifx = 1. / inv_x; p.ify = 1. / inv_y; p.scale_x = 1. / inv_x; p.scale_y = 1. / inv_y; p.inv_x = inv_x; p.inv_y = inv_y; p.area_mode = area_mode;
    ResTab* xt = (ResTab*)malloc(sizeof(ResTab) * (p.dw + p.dh)); ResTab* yt = xt + p.dw;
    for (int i = 0; i < p.dw + p.dh; i++) {
        const bool is_y = i >= p.dw; const int dd = is_y ? i - p.dw : i;
        (is_y ? yt : xt)[dd] = cubic ? res_tab_entry<true, true>(dd, is_y, p) : res_tab_entry<false, true>(dd, is_y, p);
    }
    const int RMAX = rs_host_rmax(p, cubic != 0, DH);
    int rc = 0;
#define RUN(CN, CUBIC) do { typedef RSCfg<CN, CUBIC> C; \
        unsigned char* mid = (unsigned char*)malloc((size_t)RMAX * C::E * C::MIDB); RSRow* yrow = (RSRow*)malloc(sizeof(RSRow) * DH); \
        for (int f = 0; f < si.frames; f++) for (int y0 = 0; y0 < p.dh; y0 += DH) for (int x0 = 0; x0 < p.dw; x0 += C::DW) { \
            const int nrows_out = min(DH, p.dh - y0), ncols_out = min((int)C::DW, p.dw - x0); int row_lo, R; \
            rs_tile_rows<CUBIC>(yt, y0, nrows_out, p.sh, row_lo, R); if (R > RMAX) { rc = 77; R = RMAX; } \
            memset(mid, 0xEE, (size_t)RMAX * C::E * C::MIDB); \
            for (int tid = 0; tid < 256; tid++) { if (tid < nrows_out) rs_fill_row<CUBIC>(yrow[tid], yt[y0 + tid], row_lo, p.sh); \
                const int col = tid % C::DW, rpar = tid / C::DW; \
                if (col < ncols_out) rs_hpass_thread<CN, CUBIC>(si, f, p, xt[x0 + col], row_lo, R, rpar, 256 / C::DW, mid + (size_t)col * CN * C::MIDB); } \
            for (int tid = 0; tid < 256; tid++) rs_vpass_thread<CN, CUBIC>(tid, 256, mid, yrow, di, f, p, x0, y0, nrows_out, ncols_out); } \
        free(mid); free(yrow); } while (0)
    const int cn = B200CV_CN(s->type);
    if (cubic) { if (cn == 1) RUN(1, true); else if (cn == 3) RUN(3, true); else RUN(4, true); }
    else { if (cn == 1) RUN(1, false); else if (cn == 3) RUN(3, false); else RUN(4, false); }
    free(xt);
    return rc;"""
    lib = build_emulation_raw("resize_sep.cu", "int emu_resize_sep(const b200cvMat* s, const b200cvMat* d, int cubic, int area_mode, int DH)", body)

    def run(src, dsize, cubic, DH=16, area_mode=0, pad=0):
        dw, dh = dsize
        shape = (dh, dw) if src.ndim == 2 else (dh, dw, src.shape[2])
        if pad:        # odd pitch / base alignment: the byte paths
            buf = np.full((shape[0], shape[1] * (1 if src.ndim == 2 else src.shape[2]) + pad), 0xCD, np.uint8)
            dst = buf[:, :shape[1] * (1 if src.ndim == 2 else src.shape[2])].reshape(shape)
        else:
            dst = np.full(shape, 0xCD, np.uint8)
        ms, md = mat_of(src), mat_of(dst)
        rc = lib.emu_resize_sep(ctypes.byref(ms), ctypes.byref(md), int(cubic), int(area_mode), DH)
        assert rc == 0, "emulated resize_sep returned %d" % rc
        return dst
    return run


def test_emulated_tiled_resize_vs_port(resize_sep_emu, port, rng):
    cases = [((64, 97), (61, 40)), ((48, 300), (517, 100)), ((33, 70), (140, 66)), ((120, 131), (87, 80)), ((20, 24), (300, 37)), ((301, 260), (173, 201))]
    for cn in (1, 3, 4):
        for (sh, sw), (dw, dh) in cases:
            src = rng.integers(0, 256, (sh, sw) if cn == 1 else (sh, sw, cn), dtype=np.uint8)
            for cubic in (0, 1):
                for DH in (8, 16):
                    got = resize_sep_emu(src, (dw, dh), cubic, DH)
                    want = port.resize(src, (dw, dh), 2 if cubic else 1)
                    assert np.array_equal(got, want), "tiled resize cn=%d %dx%d -> %dx%d cubic=%d DH=%d" % (cn, sw, sh, dw, dh, cubic, DH)
    # unaligned source / destination pitches (byte paths)
    base = rng.integers(0, 256, (50, 3 * 77 + 1), dtype=np.uint8)
    src = base[:, 1:].reshape(50, 77, 3)
    for cubic in (0, 1):
        got = resize_sep_emu(src, (113, 41), cubic, 16, pad=3)
        assert np.array_equal(got, port.resize(np.ascontiguousarray(src), (113, 41), 2 if cubic else 1)), "tiled resize, unaligned pitches, cubic=%d" % cubic
