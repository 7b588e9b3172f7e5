"""CPU: pin the oracle.
  * the C port (oracle/port) against the reference's own golden vectors / known-answer hashes;
  * the C port against the unmodified reference (oracle/_ref) where that library is present;
  * the product's host-side coefficient tables against both.
"""
import os
import sys
import zlib

import numpy as np
import pytest

import opencv_b200 as C
from util import assert_close, assert_exact, rand_u8

GOLD = os.path.join(os.path.dirname(__file__), "golden")

# modules/imgproc/test/test_smooth_bitexact.cpp:14-30 (8.8 fixed point)
GOLD_U8_KERNELS = {
    (1, 0): [256], (3, 0): [64, 128, 64], (5, 0): [16, 64, 96, 64, 16], (7, 0): [8, 28, 56, 72, 56, 28, 8],
    (9, 0): [4, 13, 30, 51, 60, 51, 30, 13, 4], (3, 1.75): [81, 94, 81], (3, 0.875): [65, 126, 65], (5, 0.375): [0, 7, 242, 7, 0],
    (5, 0.75): [4, 56, 136, 56, 4],
}
# modules/imgproc/test/test_color.cpp:2847-2855
KAT = {C.COLOR_RGB2GRAY: 0x416bd44a, C.COLOR_BGR2GRAY: 0x3008c6b8, C.COLOR_BGR2YUV: 0xc2cbcfda, C.COLOR_RGB2YUV: 0x4e98e757,
       C.COLOR_YUV2BGR: 0xb2c62a3f, C.COLOR_YUV2RGB: 0x6d242a3f}


@pytest.mark.parametrize("key", sorted(GOLD_U8_KERNELS))
def test_product_fixed_point_taps_match_reference_goldens(key):
    n, s = key
    assert list(C.getGaussianKernelFixed8(n, s)) == GOLD_U8_KERNELS[key]


def bitexact_eval(img, kx, ky, border, port):
    """the reference test's evaluator (test_smooth_bitexact.cpp:40-53) in numpy: sat((sum ky*(sum kx*src) + 2^15) >> 16)"""
    from oracle.api import Oracle  # noqa: F401
    h, w = img.shape
    rx, ry = len(kx) // 2, len(ky) // 2

    def bi(p, n):
        if 0 <= p < n:
            return p
        if border == 0:
            return -1
        if border == 1:
            return 0 if p < 0 else n - 1
        if border == 3:
            return p % n
        d = 1 if border == 4 else 0
        if n == 1:
            return 0
        while not 0 <= p < n:
            p = -p - 1 + d if p < 0 else n - 1 - (p - n) - d
        return p
    xs = [[bi(x + i - rx, w) for i in range(len(kx))] for x in range(w)]
    ys = [[bi(y + j - ry, h) for j in range(len(ky))] for y in range(h)]
    src = img.astype(np.int64)
    rows = np.zeros((h, w), np.int64)
    for x in range(w):
        for i, sx in enumerate(xs[x]):
            if sx >= 0:
                rows[:, x] += kx[i] * src[:, sx]
    out = np.zeros((h, w), np.int64)
    for y in range(h):
        for j, sy in enumerate(ys[y]):
            if sy >= 0:
                out[y] += ky[j] * rows[sy]
    return np.clip((out + 32768) >> 16, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("key", sorted(GOLD_U8_KERNELS))
def test_port_gaussian_u8_matches_bitexact_model(port, rng, key):
    n, s = key
    img = rand_u8(rng, 23, 31)
    k = GOLD_U8_KERNELS[key]
    for border in (0, 1, 2, 3, 4):
        assert_exact(port.GaussianBlur(img, (n, n), s, s, border), bitexact_eval(img, k, k, border, port), "port GaussianBlur %s border %d" % (key, border))


@pytest.mark.parametrize("code", sorted(KAT))
def test_port_cvtcolor_known_answer_hashes(port, code):
    img = np.load(os.path.join(GOLD, "cvtcolor_kat_input.npy"))
    dcn = 1 if code in (C.COLOR_RGB2GRAY, C.COLOR_BGR2GRAY) else 3
    assert zlib.adler32(np.ascontiguousarray(port.cvtColor(img, code, dcn)).tobytes()) == KAT[code]


# modules/imgproc/test/test_color.cpp:2857-2900 (Imgproc_cvtColor_BE, "packed input"): code -> (adler32, input fixture)
KAT_YUV = {90: 0x46a1bb76, 91: 0x3843bb76, 92: 0xf3fdf2ea, 93: 0x6e84f2ea, 94: 0xb6a16bd3, 95: 0xa8436bd3, 96: 0x1c7fa347, 97: 0x96f7a347,
           98: 0xc5da1651, 99: 0x12161651, 100: 0xb4e62ea5, 101: 0xfa632ea5, 102: 0x0db4c69f, 103: 0x59e1c69f, 104: 0xfe09def3, 105: 0x4395def3,
           106: 0xf672b440,
           107: 0x69bea2c1, 108: 0xdc51a2c1, 111: 0x851eab45, 112: 0xf7b1ab45, 115: 0x607e8889, 116: 0xfb148889, 117: 0x239b13d4, 118: 0x402b13d4,
           119: 0xf6af910d, 120: 0x9154910d, 121: 0x14481c58, 122: 0x30d81c58, 123: 0x228e669c, 124: 0x125c62fd,
           127: 0x44bb076a, 128: 0xf908ff52, 129: 0x44bb076a, 130: 0xf908ff52, 131: 0x1b0d076a, 132: 0xda8aff52, 133: 0x1b0d076a, 134: 0xda8aff52}


def kat_yuv_input(code):
    name = "cvtcolor_kat_yuv420_input.npy" if code <= 106 else "cvtcolor_kat_yuv422_input.npy" if code <= 124 else "cvtcolor_kat_bgr_262x254_input.npy"
    return np.load(os.path.join(GOLD, name))


@pytest.mark.parametrize("code", sorted(KAT_YUV))
def test_port_yuv_wire_formats_known_answer_hashes(port, code):
    """NV12 / NV21 / YV12 / IYUV / UYVY / YUY2 / YVYU -> BGR family, Y extraction, BGR family -> I420 / YV12: the port reproduces the
    reference's own known-answer hashes (the RGBA codes are fed the 3-channel image, as the reference's test does)"""
    assert zlib.adler32(np.ascontiguousarray(port.cvtColorYUV(kat_yuv_input(code), code)).tobytes()) == KAT_YUV[code]


def test_port_vs_reference_yuv_wire_formats(ref, port, rng):
    for (h, w) in [(4, 6), (18, 34), (36, 66), (250, 320), (480, 642)]:        # h % 4 == 2: the V plane starts in the middle of a row
        yuv = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
        for code in range(90, 107):
            assert np.array_equal(ref.cvtColorYUV(yuv, code), port.cvtColorYUV(yuv, code)), "4:2:0 code %d %dx%d" % (code, w, h)
        y2 = rng.integers(0, 256, (h, w, 2), dtype=np.uint8)
        for code in (107, 108, 111, 112, 115, 116, 117, 118, 119, 120, 121, 122, 123, 124):
            assert np.array_equal(ref.cvtColorYUV(y2, code), port.cvtColorYUV(y2, code)), "4:2:2 code %d %dx%d" % (code, w, h)
        for code in range(127, 135):
            img = rng.integers(0, 256, (h, w, 4 if (code - 127) & 2 else 3), dtype=np.uint8)
            assert np.array_equal(ref.cvtColorYUV(img, code), port.cvtColorYUV(img, code)), "to 4:2:0 code %d %dx%d" % (code, w, h)
        for code in range(143, 155):                  # BGR family -> UYVY / YUY2 / YVYU; the channel count is the source's, whatever the code says
            for scn in (3, 4):
                img = rng.integers(0, 256, (h, w, scn), dtype=np.uint8)
                assert np.array_equal(ref.cvtColorYUV(img, code), port.cvtColorYUV(img, code)), "to 4:2:2 code %d scn %d %dx%d" % (code, scn, w, h)


def test_port_vs_reference_bayer_demosaic(ref, port, rng):
    """Bayer BG / GB / RG / GR -> BGR and BGRA, bilinear (demosaicing.cpp:806-1056), including the copied border columns / rows"""
    for (h, w) in [(3, 3), (4, 5), (5, 4), (17, 33), (18, 34), (64, 96), (241, 323), (480, 640)]:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        for code in (46, 47, 48, 49, 139, 140, 141, 142):
            assert np.array_equal(ref.cvtColorYUV(img, code), port.cvtColorYUV(img, code)), "Bayer code %d %dx%d" % (code, w, h)


def test_port_vs_reference_integral(ref, port, rng):
    """cv::integral 8UC1 -> 32S sum and 64F sum of squares"""
    for (h, w) in [(1, 1), (5, 7), (33, 65), (240, 321), (1080, 1920)]:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        a, aq = ref.integral(img, True)
        b, bq = port.integral(img, True)
        assert np.array_equal(a, b) and np.array_equal(aq, bq), "integral %dx%d" % (w, h)
        assert a[-1, -1] == int(img.sum(dtype=np.int64)) and aq[-1, -1] == float((img.astype(np.int64) ** 2).sum())


def test_port_lab_on_the_whole_colour_cube(ref, port):
    """8-bit BGR / RGB <-> Lab, sRGB and linear: the port (libm pow, softfloat's cbrt restated bit for bit, the reference's integer formulas)
    equals the reference on ALL 2^24 colours, in both directions"""
    v = np.arange(1 << 24, dtype=np.uint32)
    cube = np.stack([v & 255, (v >> 8) & 255, (v >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    for code in (44, 45, 74, 75, 56, 57, 78, 79, 32, 33, 34, 35):          # and CIE XYZ, both directions
        assert np.array_equal(ref.cvtColor(cube, code, 3), port.cvtColorLab(cube, code)), "Lab / XYZ code %d" % code


def test_wrapper_destination_geometry_matches_the_reference(ref):
    """the Python wrappers size cv::cvtColor's destination themselves (opencv_b200._cvt_dst_geometry): it must be the reference's own
    destination size and channel count for every code whose geometry changes, and the C++ mirror's table (host/b200cv.hpp) must agree"""
    from oracle.api import yuv_dst_shape
    for code in list(range(90, 109)) + [111, 112] + list(range(115, 125)) + list(range(127, 135)) + list(range(143, 155)) + [46, 47, 48, 49, 139, 140, 141, 142]:
        if 90 <= code <= 106:
            src = np.zeros((36, 48), np.uint8)
        elif 107 <= code <= 124:
            src = np.zeros((24, 48, 2), np.uint8)
        elif code in (46, 47, 48, 49, 139, 140, 141, 142):
            src = np.zeros((24, 48), np.uint8)
        else:
            src = np.zeros((24, 48, 3), np.uint8)
        want = ref.cvtColorYUV(src, code)                     # cv::cvtColor with dcn = 0 would size it the same; the shim passes our dims and asserts
        sh, sw = src.shape[:2]
        w, h, cn = C._cvt_dst_geometry(code, sw, sh, 0)
        assert (w, h, cn) == yuv_dst_shape(sw, sh, code)
        assert want.shape[:2] == (h, w) and (want.shape[2] if want.ndim == 3 else 1) == cn, "code %d" % code
    hpp = open(os.path.join(os.path.dirname(GOLD), "..", "opencv_b200", "host", "b200cv.hpp")).read()
    assert "code >= 143 && code <= 154" in hpp and "code >= 127 && code <= 134" in hpp and "code >= 90 && code <= 105" in hpp


def test_port_vs_reference_masked_match_template(ref, port, rng):
    """cv::matchTemplate with a mask, all six methods, 8-bit (binarised) and float (weight) masks: the port's direct double sums against the
    reference's float DFT path, 1e-3 of the result range (the reference's own bar for matchTemplate, test_templmatch.cpp:333); measured ~2e-7"""
    img = rng.integers(0, 256, (90, 120), dtype=np.uint8)
    templ = img[20:41, 30:63].copy()
    m8 = (rng.random(templ.shape) > 0.3).astype(np.uint8) * 255
    mf = rng.random(templ.shape).astype(np.float32)
    for im, tt in ((img, templ), (img.astype(np.float32), templ.astype(np.float32))):
        for mk in (m8, mf):
            for method in range(6):
                a, b = ref.matchTemplateMasked(im, tt, method, mk), port.matchTemplateMasked(im, tt, method, mk)
                assert_close(b, a, atol=1e-3 * max(1.0, float(np.abs(a).max())), what="masked matchTemplate %s %s method %d" % (im.dtype, mk.dtype, method))
    big = rng.integers(0, 256, (300, 400), dtype=np.uint8)       # large enough for the reference's block DFT
    tb = big[100:164, 150:214].copy(); mb = np.zeros(tb.shape, np.uint8); mb[8:56, 8:56] = 1
    for method in (1, 3, 5):
        a, b = ref.matchTemplateMasked(big, tb, method, mb), port.matchTemplateMasked(big, tb, method, mb)
        assert_close(b, a, atol=1e-3 * max(1.0, float(np.abs(a).max())), what="masked matchTemplate 64x64 method %d" % method)
        assert np.unravel_index(b.argmin() if method == 1 else b.argmax(), b.shape) == (100, 150)


def test_port_vs_reference_gaussian_u16(ref, port, rng):
    """GaussianBlur CV_16U: 16.16 fixed-point taps, 32-bit rows, 64-bit columns (fixedSmoothInvoker<uint16_t, ufixedpoint32>): bit-exact"""
    for shape in [(37, 53), (64, 96, 3), (20, 31, 4), (1, 40), (33, 1)]:
        img = rng.integers(0, 65536, shape, dtype=np.uint16)
        ext = np.where(rng.random(shape) < 0.5, 0, 65535).astype(np.uint16)
        for im in (img, ext):
            for k, s in [(3, 0), (5, 0), (7, 1.5), (9, 0), (15, 3.0), (0, 1.2), (31, 0), (5, 0.3)]:
                for border in (4, 1, 0, 2, 3):
                    assert np.array_equal(ref.GaussianBlur(im, (k, k), s, s, border), port.GaussianBlur(im, (k, k), s, s, border)), \
                        "u16 %s k=%d s=%g border=%d" % (shape, k, s, border)


def test_port_vs_reference_two_plane(ref, port, rng):
    """cv::cvtColorTwoPlane: the same arithmetic with separate luma / chroma buffers; also equal to cvtColor on the concatenated planes"""
    for (h, w) in [(4, 6), (18, 34), (250, 322)]:
        y = rng.integers(0, 256, (h, w), dtype=np.uint8); uv = rng.integers(0, 256, (h // 2, w // 2, 2), dtype=np.uint8)
        one = np.concatenate([y, uv.reshape(h // 2, w)], axis=0)
        for code in range(90, 98):
            a = ref.cvtColorTwoPlane(y, uv, code)
            assert np.array_equal(a, port.cvtColorTwoPlane(y, uv, code)), "two-plane code %d" % code
            assert np.array_equal(a, ref.cvtColorYUV(one, code)), "two-plane == one buffer, code %d" % code


@pytest.mark.reference_library
def test_kat_input_is_the_reference_rng_stream(ref):
    """tests/golden/cvtcolor_kat_input.npy was generated by cv::RNG(0).fill(263x255 8UC3, UNIFORM, 0, 255) -- regenerate and compare"""
    img = np.load(os.path.join(GOLD, "cvtcolor_kat_input.npy"))
    assert_exact(ref.rng_fill((255, 263, 3), np.uint8, 0, 0, 255), img, "KAT input")
    sys.path.insert(0, os.path.join(os.path.dirname(GOLD), "..", "tools"))
    import make_golden
    for name, shape in make_golden.FIXTURES.items():
        assert_exact(ref.rng_fill(shape, np.uint8, 0, 0, 255), np.load(os.path.join(GOLD, name)), name)


def test_product_and_port_gaussian_kernels_match_reference(ref, port):
    for n in list(range(1, 34, 2)) + [4, 6, 20]:
        for s in (0, 0.3, 0.5, 0.8, 1.0, 1.2263, 1.5, 1.75, 2.3, 3.09, 5.1, 10.0):
            want = ref.getGaussianKernel(n, s)
            assert np.array_equal(port.getGaussianKernel(n, s).view(np.uint64), want.view(np.uint64)), (n, s)
            assert np.array_equal(C.getGaussianKernel(n, s).view(np.uint64), want.view(np.uint64)), (n, s)


def test_port_vs_reference_filters(ref, port, rng):
    img1 = rand_u8(rng, 97, 131); img3 = rand_u8(rng, 61, 77, 3); f1 = img1.astype(np.float32)
    for img in (img1, img3):
        for k, s in ((3, 0), (5, 0), (9, 0), (5, 1.1), (15, 0), (31, 5.0), (0, 1.3)):
            for b in (0, 1, 2, 3, 4):
                assert_exact(port.GaussianBlur(img, (k, k), s, s, b), ref.GaussianBlur(img, (k, k), s, s, b), "GaussianBlur u8")
    for k, s in ((3, 0), (7, 1.5), (31, 5.0)):
        assert_close(port.GaussianBlur(f1, (k, k), s), ref.GaussianBlur(f1, (k, k), s), atol=1e-4, what="GaussianBlur f32")
    for delta in (0, 3):
        assert_exact(port.sepFilter2D(img3, -1, [.25, .5, .25], [.125, .75, .125], delta=delta), ref.sepFilter2D(img3, -1, [.25, .5, .25], [.125, .75, .125], delta=delta), "sep bit-exact mode")
    for ks in (1, 3, 5, 7):
        assert_exact(port.Sobel(img1, 3, 1, 0, ks), ref.Sobel(img1, 3, 1, 0, ks), "Sobel s16")
    from util import assert_exact_body
    for k in (3, 5, 9):      # below 130 taps the reference evaluates the direct sum: the port follows its operation order
        ker = rng.random((k, k)).astype(np.float32); ker /= ker.sum()
        assert_exact(port.filter2D(img1, -1, ker, delta=2.5), ref.filter2D(img1, -1, ker, delta=2.5), "filter2D u8 k=%d" % k)
        assert_exact(port.filter2D(img3, -1, ker), ref.filter2D(img3, -1, ker), "filter2D 8UC3 k=%d" % k)
        assert_exact(port.filter2D(img1, 3, ker * 64), ref.filter2D(img1, 3, ker * 64), "filter2D u8->s16 k=%d" % k)
        assert_exact_body(port.filter2D(f1, -1, ker, delta=0.3), ref.filter2D(f1, -1, ker, delta=0.3), 8, atol=5e-4, rtol=1e-5, what="filter2D f32 k=%d" % k)
        if k * k < 50:
            assert_exact(port.filter2D(img1, 5, ker, delta=0.3), ref.filter2D(img1, 5, ker, delta=0.3), "filter2D u8->f32 k=%d" % k)


def test_port_float_separable_filters_follow_the_reference_operation_order(ref, port, rng):
    """The port (and the CUDA kernels that mirror it) run float separable filters in the operation order of the reference's SIMD
    loops -- centre-out 3/5-tap rows, tap-order FMA rows, mirrored-pair FMA columns, un-fused products when the column kernel has
    no symmetry -- so every element the reference computes in a full vector is bit-identical.  Remainder columns: tolerance."""
    from util import assert_exact_body
    for shape in ((97, 131), (64, 648), (33, 77)):
        f = (rng.random(shape) * 255).astype(np.float32)
        u = rand_u8(rng, *shape)
        for k in (3, 5, 7, 13, 31):
            sig = 0.3 * ((k - 1) * 0.5 - 1) + 0.87
            g = ref.getGaussianKernel(k, sig).astype(np.float32)
            d = np.arange(k, dtype=np.float32) - k // 2; d /= np.abs(d).sum() * 1.01
            rk = rng.random(k).astype(np.float32)
            for b in (0, 1, 4):
                assert_exact_body(port.GaussianBlur(f, (k, k), sig, sig, b), ref.GaussianBlur(f, (k, k), sig, sig, b), 8, atol=1e-4, rtol=1e-5, what="GaussianBlur f32 k=%d" % k)
            assert_exact_body(port.GaussianBlur(f, (k, 3), 2.2), ref.GaussianBlur(f, (k, 3), 2.2), 8, atol=1e-4, rtol=1e-5, what="GaussianBlur f32 %dx3" % k)
            assert_exact_body(port.sepFilter2D(f, -1, d, g, delta=0.25), ref.sepFilter2D(f, -1, d, g, delta=0.25), 8, atol=1e-3, rtol=1e-5, what="antisymmetric rows")
            assert_exact_body(port.sepFilter2D(f, -1, g, d), ref.sepFilter2D(f, -1, g, d), 8, atol=1e-3, rtol=1e-5, what="antisymmetric columns")
            assert_exact_body(port.sepFilter2D(f, -1, rk, rk, delta=1.5), ref.sepFilter2D(f, -1, rk, rk, delta=1.5), 8, atol=1e-2, rtol=1e-5, what="no symmetry")
            assert_exact_body(port.sepFilter2D(u, 5, g, g, delta=0.5), ref.sepFilter2D(u, 5, g, g, delta=0.5), 32, atol=1e-3, rtol=1e-5, what="u8 -> f32")
            assert_exact_body(port.sepFilter2D(u, -1, g, g), ref.sepFilter2D(u, -1, g, g), 32, atol=1, what="u8 through float")
            assert_exact_body(port.sepFilter2D(u, 5, rk, rk, delta=1.5), ref.sepFilter2D(u, 5, rk, rk, delta=1.5), 32, atol=1e-2, rtol=1e-5, what="u8 -> f32, no symmetry")


def test_port_vs_reference_color(ref, port):
    bgr = np.load(os.path.join(GOLD, "cvtcolor_kat_input.npy"))
    for code, dcn in ((6, 1), (7, 1), (82, 3), (83, 3), (36, 3), (37, 3), (40, 3), (41, 3), (66, 3), (67, 3), (4, 3), (0, 4), (2, 4),
                      (84, 3), (85, 3), (38, 3), (39, 4), (54, 3), (55, 4), (70, 3), (71, 3)):
        assert_exact(port.cvtColor(bgr, code, dcn), ref.cvtColor(bgr, code, dcn), "cvtColor %d" % code)


def test_port_vs_reference_geometry(ref, port, rng):
    for (ssz, dsz) in (((97, 131), (61, 77)), ((64, 48), (128, 96)), ((120, 160), (60, 80)), ((7, 9), (31, 45))):
        for cn in (1, 3):
            img = rand_u8(rng, ssz[0], ssz[1], cn)
            for it in (0, 1, 2):
                assert_exact(port.resize(img, (dsz[1], dsz[0]), it), ref.resize(img, (dsz[1], dsz[0]), it), "resize u8 %s %s %d" % (ssz, dsz, it))
                f = img.astype(np.float32)
                assert_close(port.resize(f, (dsz[1], dsz[0]), it), ref.resize(f, (dsz[1], dsz[0]), it), atol=1e-4, what="resize f32")
    img = rand_u8(rng, 131, 157, 3)
    M = ref.getRotationMatrix2D((78, 65), 7, 0.9)
    H = np.array([[0.95, 0.02, 5.0], [-0.015, 0.97, 3.0], [1e-5, 2e-5, 1.0]])
    for it in (0, 1, 2):
        for b in (0, 1, 2, 3, 4):
            for fl in (it, it | 16):
                assert_exact(port.warpAffine(img, M, (170, 140), fl, b, (10, 20, 30, 40)), ref.warpAffine(img, M, (170, 140), fl, b, (10, 20, 30, 40)), "warpAffine")
            assert_exact(port.warpPerspective(img, H, (170, 140), it, b, (10, 20, 30, 40)), ref.warpPerspective(img, H, (170, 140), it, b, (10, 20, 30, 40)), "warpPerspective")


def _smooth(rng, h, w):
    small = rng.random((h // 8 + 2, w // 8 + 2)).astype(np.float32)
    img = np.kron(small, np.ones((8, 8), np.float32))[:h, :w] + 0.15 * rng.random((h, w)).astype(np.float32)
    img = (img - img.min()) / (img.max() - img.min())
    return (img * 255).astype(np.uint8)


def test_port_vs_reference_area_resize(ref, port, rng):
    """INTER_AREA, true area mode: integer factors (window sums; float sums in groups of four) and fractional factors (DecimateAlpha)"""
    cases = [((120, 180), (40, 60)), ((120, 180), (30, 90)), ((121, 183), (40, 61)), ((100, 150), (37, 41)), ((480, 640), (300, 400)),
             ((97, 131), (96, 130)), ((64, 64), (16, 16)), ((90, 120), (30, 24)), ((50, 70), (49, 23)), ((33, 47), (1, 1)), ((300, 400), (7, 399)),
             # an enlarging axis: bilinear with area-mode weights
             ((40, 60), (120, 180)), ((40, 60), (97, 131)), ((100, 150), (237, 341)), ((64, 64), (160, 32)), ((64, 64), (32, 160)), ((1, 47), (5, 90)),
             ((50, 1), (75, 23)), ((120, 160), (121, 100))]
    for (sh, sw), (dh, dw) in cases:
        for cn in (1, 3, 4):
            shape = (sh, sw) if cn == 1 else (sh, sw, cn)
            for img in (rng.integers(0, 256, shape, dtype=np.uint8), (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)):
                assert np.array_equal(ref.resize(img, (dw, dh), 3), port.resize(img, (dw, dh), 3)), "INTER_AREA %s %s -> %s cn=%d" % (img.dtype, (sh, sw), (dh, dw), cn)


# the reference's own golden vectors for the exact / area resizers (modules/imgproc/test/test_resize_bitexact.cpp:190-241, Resize_Bitexact.Nearest8U;
# test_imgwarp.cpp:1285-1317, Imgproc_resize_area.regression_half_round / regression_quarter_round)
NEAREST_EXACT_GOLDENS = [
    ([[0, 1, 2, 3, 4, 5]], [[1, 3, 5]]),
    ([[0, 1, 2, 3, 4]], [[2]]),
    ([[0, 1, 2, 3, 4]], [[0, 2, 4]]),
    ([[0, 1, 2, 3, 4]], [[1, 3]]),
    ([[0, 1, 2, 3, 4], [5, 6, 7, 8, 9], [10, 11, 12, 13, 14]],
     [[0, 1, 1, 2, 3, 3, 4], [0, 1, 1, 2, 3, 3, 4], [5, 6, 6, 7, 8, 8, 9], [10, 11, 11, 12, 13, 13, 14], [10, 11, 11, 12, 13, 13, 14]]),
    ([[0, 1, 2], [3, 4, 5]], [[0, 0, 1, 1, 2, 2], [0, 0, 1, 1, 2, 2], [3, 3, 4, 4, 5, 5], [3, 3, 4, 4, 5, 5]]),
]


def resize_golden_cases():
    """(src, dsize, interpolation, want, max |difference|) -- the goldens above, both orientations, plus the INTER_AREA rounding regressions"""
    cases = []
    for s, d in NEAREST_EXACT_GOLDENS:
        s, d = np.array(s, np.uint8), np.array(d, np.uint8)
        cases.append((s, (d.shape[1], d.shape[0]), 6, d, 0))
        cases.append((np.ascontiguousarray(s.T), (d.shape[0], d.shape[1]), 6, np.ascontiguousarray(d.T), 0))
    i = np.arange(32 * 32)
    src = (i % 2 + 253 + i // (16 * 32)).astype(np.uint8).reshape(32, 32)
    j = np.arange(16 * 16)
    cases.append((src, (16, 16), 3, (254 + j // (16 * 8)).astype(np.uint8).reshape(16, 16), 0))     # check_resize_area(..., 0.5): exact for integers
    cases.append((src, (8, 8), 3, np.full((8, 8), 254, np.uint8), 0))
    return cases


def test_port_reproduces_the_reference_resize_goldens(port, ref):
    for src, dsize, interp, want, tol in resize_golden_cases():
        for o in (port, ref):
            got = o.resize(src, dsize, interp)
            assert np.abs(got.astype(int) - want.astype(int)).max() <= tol, "%s interp %d %s -> %s" % (o.kind, interp, src.shape, dsize)


def test_port_vs_reference_exact_resizers(ref, port, rng):
    """INTER_LINEAR_EXACT (8.8 fixed point; float data falls back to INTER_LINEAR, 2 x 2 decimation to the INTER_AREA fast path) and
    INTER_NEAREST_EXACT (16.16 pixel-centre coordinates)"""
    cases = [((120, 180), (40, 60)), ((120, 180), (60, 90)), ((121, 183), (40, 61)), ((100, 150), (237, 341)), ((480, 640), (300, 400)),
             ((97, 131), (96, 130)), ((64, 64), (160, 160)), ((1, 47), (5, 90)), ((50, 1), (49, 23)), ((33, 47), (1, 1)), ((300, 400), (7, 399)),
             ((2, 2), (9, 9)), ((3, 5), (30, 50)), ((120, 178), (60, 89)), ((120, 182), (60, 91))]
    for (sh, sw), (dh, dw) in cases:
        for cn in (1, 3, 4):
            shape = (sh, sw) if cn == 1 else (sh, sw, cn)
            for img in (rng.integers(0, 256, shape, dtype=np.uint8), (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)):
                for interp in (5, 6):
                    assert np.array_equal(ref.resize(img, (dw, dh), interp), port.resize(img, (dw, dh), interp)), \
                        "interp %d %s %s -> %s cn=%d" % (interp, img.dtype, (sh, sw), (dh, dw), cn)


def test_port_vs_reference_lanczos4_resize(ref, port, rng):
    """INTER_LANCZOS4: 8 x 8 taps, weights from double sin / cos (the same libm as the reference's), 8-bit fixed point and float with the
    reference's body / remainder summation orders"""
    cases = [((40, 60), (120, 180)), ((40, 60), (97, 131)), ((100, 150), (237, 341)), ((97, 131), (98, 132)), ((64, 64), (160, 32)), ((120, 180), (40, 61)),
             ((1, 47), (5, 90)), ((50, 1), (75, 23)), ((3, 5), (30, 50)), ((120, 160), (121, 100)), ((240, 320), (150, 201)), ((480, 640), (300, 402))]
    for (sh, sw), (dh, dw) in cases:
        for cn in (1, 3, 4):
            shape = (sh, sw) if cn == 1 else (sh, sw, cn)
            for img in (rng.integers(0, 256, shape, dtype=np.uint8), (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)):
                assert np.array_equal(ref.resize(img, (dw, dh), 4), port.resize(img, (dw, dh), 4)), "LANCZOS4 %s %s -> %s cn=%d" % (img.dtype, (sh, sw), (dh, dw), cn)


@pytest.mark.reference_library
def test_reference_sift_front_end_is_reachable(ref, rng):
    """the oracle for SURVEY 8(f) rank 1: cv::SIFT::detectAndCompute of the unmodified reference (keypoints + 128-float descriptors)"""
    small = rng.random((30, 40)).astype(np.float32)
    img = (np.kron(small, np.ones((8, 8), np.float32)) * 255).astype(np.uint8)
    kp, octv, desc = ref.sift_detect_and_compute(img)
    kp2, octv2, desc2 = ref.sift_detect_and_compute(img)
    assert len(kp) > 20 and desc.shape == (len(kp), 128)
    assert np.array_equal(kp, kp2) and np.array_equal(desc, desc2) and np.array_equal(octv, octv2), "the reference's SIFT is deterministic"
    mask = np.zeros(img.shape, np.uint8); mask[50:150, 80:240] = 1
    km, om, dm = ref.sift_detect_and_compute(img, mask=mask)
    keep = mask[(kp[:, 1] + 0.5).astype(np.int32), (kp[:, 0] + 0.5).astype(np.int32)] != 0
    assert 0 < len(km) < len(kp) and np.array_equal(km, kp[keep]) and np.array_equal(dm, desc[keep]), "mask = runByPixelsMask on the rounded positions"
    assert (kp[:, 0] >= 0).all() and (kp[:, 0] < img.shape[1]).all() and (kp[:, 1] >= 0).all() and (kp[:, 1] < img.shape[0]).all()
    assert np.all(desc >= 0) and np.all(desc <= 255) and np.all(desc == np.round(desc)), "descriptors are 8-bit-valued floats (sift.simd.hpp:1018-1034)"


def _sift_test_image(rng, h, w):
    small = rng.random((h // 8 + 2, w // 8 + 2)).astype(np.float32)
    img = np.kron(small, np.ones((8, 8), np.float32))[:h, :w] + 0.15 * rng.random((h, w)).astype(np.float32)
    img = (img - img.min()) / (img.max() - img.min())
    return (img * 255).astype(np.uint8)


def match_keypoints(a, b, tol_xy=1e-3, tol_angle=1e-2):
    """greedy one-to-one match of two (n,5) keypoint arrays on (x, y, size, angle): returns the number of matched pairs"""
    used = np.zeros(len(b), bool)
    hit = 0
    order = np.lexsort((b[:, 1], b[:, 0]))
    bx = b[order, 0]
    for k in a:
        lo, hi = np.searchsorted(bx, k[0] - tol_xy), np.searchsorted(bx, k[0] + tol_xy)
        for j in order[lo:hi]:
            if not used[j] and abs(b[j, 1] - k[1]) <= tol_xy and abs(b[j, 2] - k[2]) <= tol_xy and \
                    min(abs(b[j, 3] - k[3]), 360 - abs(b[j, 3] - k[3])) <= tol_angle:
                used[j] = True; hit += 1
                break
    return hit


def test_port_sift_pyramid_default_first_octave(ref, port, rng):
    """upscale = 2: the first octave of SIFT::create's default (enable_precise_upscale = false: cv::resize LINEAR instead of warpAffine)"""
    img = _sift_test_image(rng, 120, 160)
    rg, rd = ref.sift_pyramid(img, 3, 1.6, 2)
    pg, pd = port.sift_pyramid(img, 3, 1.6, 2)
    assert len(rg) == len(pg)
    for o in range(len(rg)):
        for a, b in zip(rg[o], pg[o]):
            assert_close(b, a, atol=1e-4, what="gauss octave %d" % o)
    assert not np.array_equal(rg[0][0], ref.sift_pyramid(img, 3, 1.6, 1)[0][0][0]), "the two first octaves differ"
    # and the reference's default detector sits on exactly this pyramid
    kr, octr, _ = ref.sift_detect_and_compute(img, precise_upscale=False)
    kp, octp = port.sift_detect_from_pyramid(rg, rd)
    assert abs(len(kp) - len(kr)) <= max(3, len(kr) // 100) and match_keypoints(kr, kp) >= 0.99 * len(kr)


def test_port_sift_detector_and_descriptors_vs_reference(ref, port, rng):
    """SURVEY 8(f) rank 1: scale-space extrema + refinement + orientation + descriptors, restated; fed the reference's own pyramids so that only
    this stage is compared.  The reference's SIFT objects are FMA-contracted AVX2 / AVX-512 builds with OpenCV's approximate exp / atan2: the
    agreement is by tolerance.  Measured: >= 99% of the keypoints agree to 1e-3 px / 1e-2 deg (typically all but a handful of borderline
    accept / reject decisions, differences ~3e-5 px); descriptors of identical keypoints differ in < 1e-4 of their entries, by 1."""
    for (h, w) in [(240, 320), (300, 400)]:
        img = _sift_test_image(rng, h, w)
        kr, octr, dr = ref.sift_detect_and_compute(img)
        G, D = ref.sift_pyramid(img)
        kp, octp = port.sift_detect_from_pyramid(G, D)
        assert abs(len(kp) - len(kr)) <= max(3, len(kr) // 100), "keypoint count %d vs %d" % (len(kp), len(kr))
        assert match_keypoints(kr, kp) >= 0.99 * len(kr)
        dp = port.sift_descriptors_from_pyramid(G, kr, octr)
        diff = np.abs(dp - dr)
        assert diff.max() <= 1 and (diff > 0).mean() < 1e-4, "descriptor entries differing: %d of %d, max %g" % ((diff > 0).sum(), diff.size, diff.max())


def test_port_vs_reference_remap(ref, port, rng):
    """cv::remap restated in the port: float planes, packed float pairs, fixed-point maps (incl. the NNDeltaTab_i quirk), NaN and
    out-of-range coordinates -- bit-exact against the reference for u8 and f32."""
    yy, xx = np.mgrid[0:80, 0:111].astype(np.float32)
    mx = (xx * 1.3 - 7.25).astype(np.float32); my = (yy * 0.7 + 3.5 + 4 * np.sin(xx / 9)).astype(np.float32)
    mx[0, 0] = np.nan; mx[0, 1] = 1e20; my[0, 2] = -1e20; mx[1, 0] = 40000.4; my[1, 1] = -40000.6; mx[2, :5] = [0.5, 1.5, 2.5, -0.5, -1.5]
    rx = (rng.random((80, 111)) * 171 - 20).astype(np.float32); ry = (rng.random((80, 111)) * 137 - 20).astype(np.float32)
    for dt in (np.uint8, np.float32):
        for cn in (1, 3):
            src = (rng.random((97, 131, cn) if cn > 1 else (97, 131)) * 255).astype(dt)
            for interp in (0, 1, 2):
                for border in (0, 1, 2, 3, 4):
                    assert_exact(port.remap(src, mx, my, interp, border, (9, 8, 7, 6)), ref.remap(src, mx, my, interp, border, (9, 8, 7, 6)), "remap planar")
                m12 = np.stack([rx, ry], -1)
                assert_exact(port.remap(src, m12, None, interp, 1), ref.remap(src, m12, None, interp, 1), "remap packed")
                xy, fr = ref.convertMaps(rx, ry)
                assert_exact(port.remap(src, xy, fr, interp, 1), ref.remap(src, xy, fr, interp, 1), "remap fixed")


def test_port_vs_reference_pyramids(ref, port, rng):
    for dt in (np.uint8, np.float32):
        for shape in ((97, 131), (64, 80), (5, 7), (2, 2), (1, 9), (33, 1), (40, 51, 3), (20, 22, 4)):
            src = (rng.random(shape) * 255).astype(dt)
            for b in (1, 2, 3, 4):
                if dt is np.uint8:
                    assert_exact(port.pyrDown(src, b), ref.pyrDown(src, b), "pyrDown u8")
                else:
                    assert_close(port.pyrDown(src, b), ref.pyrDown(src, b), atol=1e-4, what="pyrDown f32")
            assert_exact(port.pyrUp(src), ref.pyrUp(src), "pyrUp %s" % dt.__name__)


def test_port_vs_reference_box_filter(ref, port, rng):
    """cv::boxFilter / cv::blur: every sum type createBoxFilter picks (16-bit sums with the integer divide, int sums with the float scale of
    the SIMD body / the double scale of the scalar remainder, double sums for float images) -- bit for bit"""
    n = 0
    for (h, w), cn in [((37, 53), 1), ((64, 99), 3), ((50, 131), 4), ((1, 40), 1), ((33, 1), 3), ((240, 322), 1)]:
        shape = (h, w) if cn == 1 else (h, w, cn)
        u8 = rng.integers(0, 256, shape, dtype=np.uint8)
        f32 = (rng.random(shape, dtype=np.float32) * 255).astype(np.float32)
        wide = (f32 * np.exp2(rng.integers(-30, 30, shape)).astype(np.float32)).astype(np.float32)   # double sums that do round
        for ks in [(3, 3), (5, 5), (7, 3), (2, 4), (16, 16), (17, 17), (20, 20), (1, 1), (31, 9)]:
            for norm in (True, False):
                for border in (4, 1, 0, 2):
                    anchor = (-1, -1) if border != 1 else (ks[0] - 1, 0)
                    for img, dd in ((u8, -1), (u8, 5), (f32, -1), (wide, -1)):
                        a = ref.boxFilter(img, dd, ks, anchor, norm, border)
                        b = port.boxFilter(img, dd, ks, anchor, norm, border)
                        assert np.array_equal(a, b), "boxFilter %s dd=%d ks=%s norm=%d border=%d %s" % (img.dtype, dd, ks, norm, border, shape)
                        n += 1
    assert n > 1500
    assert np.array_equal(ref.blur(u8, (5, 5)), ref.boxFilter(u8, -1, (5, 5)))


def test_port_vs_reference_features(ref, port, rng):
    im = rand_u8(rng, 90, 120); tp = im[5:22, 9:32].copy()
    for m in range(6):
        a = ref.matchTemplate(im, tp, m)
        assert_close(port.matchTemplate(im, tp, m), a, atol=1e-3 * max(1.0, float(np.abs(a).max())), what="matchTemplate %d" % m)
    sm = _smooth(rng, 97, 131)
    for bs, ks in ((2, 3), (3, 3), (5, 5), (2, 1)):
        a = ref.cornerHarris(sm, bs, ks, 0.04)
        assert_close(port.cornerHarris(sm, bs, ks, 0.04), a, atol=3e-6 * float(np.abs(a).max()), what="cornerHarris")
        a = ref.cornerMinEigenVal(sm, bs, ks)
        assert_close(port.cornerMinEigenVal(sm, bs, ks), a, atol=3e-6 * float(np.abs(a).max()), what="cornerMinEigenVal")
    for harris in (True, False):
        for md in (0, 5, 10.5):
            a, _ = ref.goodFeaturesToTrack(sm, 200, 0.01, md, 3, 3, harris, 0.04)
            b, _ = port.goodFeaturesToTrack(sm, 200, 0.01, md, 3, 3, harris, 0.04)
            assert_exact(b, a, "goodFeaturesToTrack harris=%s md=%g" % (harris, md))
    wg, wd = ref.sift_pyramid(sm, 3, 1.6, True)
    pg, pd = port.sift_pyramid(sm, 3, 1.6, True)
    assert len(wg) == len(pg)
    for o in range(len(wg)):
        for i in range(6):
            assert_close(pg[o][i], wg[o][i], atol=1e-3, what="sift gauss")
        for i in range(5):
            assert_close(pd[o][i], wd[o][i], atol=1e-3, what="sift dog")


@pytest.mark.reference_library
def test_reference_reproduces_the_depth_cvtcolor_hashes(ref):
    """tests/kat_depth.py: the constants the GPU tests compare against were generated from this very library"""
    from kat_depth import KAT_DEPTH, kat_dcn, kat_hash, kat_input
    for (code, kind), want in sorted(KAT_DEPTH.items()):
        assert kat_hash(ref.cvtColor(kat_input(kind), code, kat_dcn(code))) == want, "reference hash changed: code %d on %s" % (code, kind)
