"""GPU: the host-pointer C ABI (cv_hal_* shaped and batched b200cv_host_*) gives the same bytes as the oracle."""
import ctypes

import numpy as np
import pytest

import opencv_b200 as C
from util import assert_close, assert_exact, rand_u8

pytestmark = pytest.mark.gpu
u8p = ctypes.POINTER(ctypes.c_ubyte)


def p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_hal_signatures(cvb, oracle, rng):
    L = cvb.lib()
    img = rand_u8(rng, 120, 161, 3)
    dst = np.empty_like(img)
    sz = ctypes.c_size_t
    rc = L.b200cv_hal_gaussianBlur(p(img), sz(img.strides[0]), p(dst), sz(dst.strides[0]), 161, 120, 0, 3, sz(0), sz(0), sz(0), sz(0), sz(5), sz(5),
                                   ctypes.c_double(0), ctypes.c_double(0), 4)
    assert rc == 0
    assert_exact(dst, oracle.GaussianBlur(img, (5, 5), 0), "hal gaussianBlur")
    # a ROI of a larger Mat (non-zero margins): the pixels around it are real and must be used -- equal to blurring the parent and cropping
    par = rand_u8(rng, 140, 181, 3)
    roi = par[7:7 + 120, 9:9 + 161]
    out = np.empty((120, 161, 3), np.uint8)
    rc = L.b200cv_hal_gaussianBlur(p(roi), sz(par.strides[0]), p(out), sz(out.strides[0]), 161, 120, 0, 3, sz(9), sz(7), sz(181 - 161 - 9), sz(140 - 120 - 7),
                                   sz(7), sz(7), ctypes.c_double(0), ctypes.c_double(0), 4)
    assert rc == 0
    assert_exact(out, oracle.GaussianBlur(par, (7, 7), 0)[7:127, 9:170], "hal gaussianBlur on a ROI with context")
    # ... unless the border is BORDER_ISOLATED: then the ROI is the image
    rc = L.b200cv_hal_gaussianBlur(p(roi), sz(par.strides[0]), p(out), sz(out.strides[0]), 161, 120, 0, 3, sz(9), sz(7), sz(11), sz(13),
                                   sz(7), sz(7), ctypes.c_double(0), ctypes.c_double(0), 4 | 16)
    assert rc == 0
    assert_exact(out, oracle.GaussianBlur(np.ascontiguousarray(roi), (7, 7), 0), "hal gaussianBlur, BORDER_ISOLATED")
    # in place
    tmp = img.copy()
    rc = L.b200cv_hal_gaussianBlur(p(tmp), sz(tmp.strides[0]), p(tmp), sz(tmp.strides[0]), 161, 120, 0, 3, sz(0), sz(0), sz(0), sz(0), sz(5), sz(5),
                                   ctypes.c_double(0), ctypes.c_double(0), 4)
    assert rc == 0
    assert_exact(tmp, oracle.GaussianBlur(img, (5, 5), 0), "hal gaussianBlur in place")
    gray = np.empty((120, 161), np.uint8)
    assert L.b200cv_hal_cvtBGRtoGray(p(img), sz(img.strides[0]), p(gray), sz(gray.strides[0]), 161, 120, 0, 3, ctypes.c_bool(False)) == 0
    assert_exact(gray, oracle.cvtColor(img, C.COLOR_BGR2GRAY, 1), "hal cvtBGRtoGray")
    hsv = np.empty_like(img)
    assert L.b200cv_hal_cvtBGRtoHSV(p(img), sz(img.strides[0]), p(hsv), sz(hsv.strides[0]), 161, 120, 0, 3, ctypes.c_bool(True), ctypes.c_bool(False),
                                    ctypes.c_bool(True)) == 0
    assert_exact(hsv, oracle.cvtColor(img, C.COLOR_RGB2HSV, 3), "hal cvtBGRtoHSV swapBlue")
    half = np.empty((60, 80, 3), np.uint8)
    assert L.b200cv_hal_resize(16, p(img[:, :160]), sz(img.strides[0]), 160, 120, p(half), sz(half.strides[0]), 80, 60, ctypes.c_double(0.5),
                               ctypes.c_double(0.5), 1) == 0
    assert_exact(half, oracle.resize(np.ascontiguousarray(img[:, :160]), (80, 60), 1), "hal resize")
    # filter context life cycle
    ctx = ctypes.c_void_p()
    ker = (rng.random((5, 5)).astype(np.float32)); ker /= ker.sum()
    assert L.b200cv_hal_filterInit(ctypes.byref(ctx), p(ker), sz(ker.strides[0]), 5, 5, 5, 161, 120, 16, 16, 4, ctypes.c_double(0), 2, 2,
                                   ctypes.c_bool(False), ctypes.c_bool(False)) == 0
    assert L.b200cv_hal_filter(ctx, p(img), sz(img.strides[0]), p(dst), sz(dst.strides[0]), 161, 120, 161, 120, 0, 0) == 0
    assert L.b200cv_hal_filterFree(ctx) == 0
    assert_close(dst, oracle.filter2D(img, -1, ker), atol=1, what="hal filter")


def test_host_batch_pipeline(cvb, oracle, rng):
    from opencv_b200 import hal
    batch = np.stack([rand_u8(rng, 480, 640, 3) for _ in range(40)])     # > one chunk: exercises all three pipeline streams
    src = hal.pinned_empty(batch.shape, np.uint8); src[...] = batch
    out = hal.GaussianBlur(src, (7, 7), 1.5)
    gray = hal.cvtColor(src, C.COLOR_BGR2GRAY)
    for i in (0, 13, 39):
        assert_exact(out[i], oracle.GaussianBlur(batch[i], (7, 7), 1.5), "batched host blur frame %d" % i)
        assert_exact(gray[i, :, :, 0], oracle.cvtColor(batch[i], C.COLOR_BGR2GRAY, 1), "batched host gray frame %d" % i)
    M = np.array([[0.9, 0.1, 5], [-0.1, 0.9, 7]])
    yy, xx = np.mgrid[0:200, 0:300].astype(np.float32)
    mx = (xx * 2.1 + 3).astype(np.float32); my = (yy * 2.3 + 5 * np.sin(xx / 17)).astype(np.float32)
    rm = hal.remap(batch[:3], mx, my, 2, 4)
    assert_exact(rm[2], oracle.remap(batch[2], mx, my, 2, 4), "host remap")
    bl = hal.blur(batch[:5], (11, 11))
    assert_exact(bl[4], oracle.blur(batch[4], (11, 11)), "host blur")
    w = hal.warpAffine(batch[:3], M, (640, 480))
    assert_exact(w[1], oracle.warpAffine(batch[1], M, (640, 480)), "host warpAffine")
    r = hal.matchTemplate(batch[0, :, :, 0].copy(), batch[0, 100:132, 200:232, 0].copy(), C.TM_CCORR_NORMED)
    assert np.unravel_index(r.argmax(), r.shape) == (100, 200)


def test_opencv_built_with_b200_hal(cvb, ref, rng):
    """oracle/_ref/libocvref_hal.so is the UNMODIFIED reference compiled with hal/b200cv_hal_replacement.hpp registered as its imgproc
    HAL (what -DOpenCV_HAL_DIR=<repo>/hal does): plain cv::resize / cv::cvtColor / cv::warpAffine / cv::sepFilter2D / cv::GaussianBlur
    calls on host cv::Mat data now run on the B200 and still return the reference's bytes."""
    from oracle.api import Oracle, available
    if not available("ref_hal"):
        pytest.skip("libocvref_hal.so not built (python oracle/build_ref.py --hal)")
    hal = Oracle("ref_hal")
    img = rand_u8(rng, 480, 640, 3)
    g = img[:, :, 0].copy()
    n0 = cvb.launch_count()
    assert_exact(hal.cvtColor(img, C.COLOR_BGR2YUV, 3), ref.cvtColor(img, C.COLOR_BGR2YUV, 3), "cv::cvtColor via HAL")
    n1 = cvb.launch_count()
    assert n1 > n0, "cv::cvtColor did not reach the B200 HAL"
    # 16-bit and float images reach the device too (cvtcolor_depth.cu) -- bit-exact incl. the float vector-body / scalar-tail split
    f3 = (rng.random((241, 323, 3), dtype=np.float32) * 1.2).astype(np.float32)
    w3 = rng.integers(0, 65536, (241, 323, 3), dtype=np.uint16)
    nb = cvb.launch_count()
    for src_img in (f3, w3):
        for code, dcn in ((C.COLOR_BGR2GRAY, 1), (C.COLOR_RGB2YCrCb, 3), (C.COLOR_YUV2BGR, 3), (C.COLOR_BGR2RGBA, 4), (C.COLOR_BGR2XYZ, 3)):
            assert_exact(hal.cvtColor(src_img, code, dcn), ref.cvtColor(src_img, code, dcn), "cv::cvtColor %s code %d via HAL" % (src_img.dtype, code))
    assert cvb.launch_count() - nb >= 10, "16-bit / float cv::cvtColor did not reach the B200 HAL"
    assert_exact(hal.resize(img, (320, 240), 1), ref.resize(img, (320, 240), 1), "cv::resize via HAL")
    assert_exact(hal.resize(img, (427, 321), 2), ref.resize(img, (427, 321), 2), "cv::resize CUBIC via HAL")
    M = np.array([[0.9, 0.1, 5], [-0.1, 0.9, 7]])
    assert_exact(hal.warpAffine(img, M, (640, 480), 1, 1), ref.warpAffine(img, M, (640, 480), 1, 1), "cv::warpAffine via HAL")
    if hal.has("pyr_down"):
        nb = cvb.launch_count()
        assert_exact(hal.pyrDown(img), ref.pyrDown(img), "cv::pyrDown via HAL (hal_ni_pyrdown)")
        assert cvb.launch_count() > nb, "cv::pyrDown did not reach the B200 HAL"
    if hal.has("box_filter"):
        nb = cvb.launch_count()
        assert_exact(hal.blur(img, (5, 5)), ref.blur(img, (5, 5)), "cv::blur via HAL (hal_ni_boxFilter)")
        assert_exact(hal.boxFilter(g, 5, (19, 19), (-1, -1), True, 1), ref.boxFilter(g, 5, (19, 19), (-1, -1), True, 1), "cv::boxFilter 8U->32F via HAL")
        assert cvb.launch_count() - nb >= 2, "cv::boxFilter did not reach the B200 HAL"
    if hal.has("remap"):
        yy, xx = np.mgrid[0:300, 0:400].astype(np.float32)
        mx = (xx * 1.5 + 10 * np.sin(yy / 20)).astype(np.float32); my = (yy * 1.55 - 8 + 5 * np.cos(xx / 30)).astype(np.float32)
        nb = cvb.launch_count()
        assert_exact(hal.remap(img, mx, my, 1, 1), ref.remap(img, mx, my, 1, 1), "cv::remap via HAL (hal_ni_remap32f)")
        assert cvb.launch_count() > nb, "cv::remap did not reach the B200 HAL"
    assert_exact(hal.GaussianBlur(img, (5, 5), 0), ref.GaussianBlur(img, (5, 5), 0), "cv::GaussianBlur (binomial HAL hook)")
    f = g.astype(np.float32)
    assert_close(hal.GaussianBlur(f, (7, 7), 1.5), ref.GaussianBlur(f, (7, 7), 1.5), atol=1e-4, what="cv::GaussianBlur f32 via HAL")
    assert_exact(hal.Sobel(g, 3, 1, 0, 3), ref.Sobel(g, 3, 1, 0, 3), "cv::Sobel via HAL")
    assert cvb.launch_count() - n1 >= 6
    # cornerHarris has no HAL hook of its own but its Sobel calls go through the seam
    a = ref.cornerHarris(g, 2, 3, 0.04)
    assert_close(hal.cornerHarris(g, 2, 3, 0.04), a, atol=3e-6 * float(np.abs(a).max()), what="cv::cornerHarris (Sobel via HAL)")


@pytest.mark.parametrize("inplace", [False, True])
def test_opencv_hal_roi_with_context(cvb, ref, rng, inplace):
    """Row a5 of the scope table (FilterEngine's wholeSize / ofs): a cv::Mat that is a ROI of a larger Mat, filtered by the UNMODIFIED reference
    built with the B200 HAL, must equal the stock reference -- the border rule applies at the PARENT's edges, the pixels around the ROI are real --
    and the call must have reached the device (launch counter).  ROIs in a corner (margins clipped by the parent), in the middle, flush with
    one side; 8-bit and float; in place."""
    from oracle.api import Oracle, available
    if not available("ref_hal"):
        pytest.skip("libocvref_hal.so not built (python oracle/build_ref.py --hal)")
    hal = Oracle("ref_hal")
    par8 = rand_u8(rng, 200, 260, 3)
    parf = (rng.random((200, 260)) * 255).astype(np.float32)
    for rect in ((0, 0, 100, 80), (31, 17, 160, 120), (100, 2, 160, 190), (3, 120, 250, 80)):
        for border in (4, 1, 0):
            cases = [(par8, 0, 5, 0.0), (parf, 0, 9, 2.0), (par8, 1, 7, 0.0), (par8, 2, 7, 1.6), (parf, 2, 11, 2.2), (par8, 3, 5, 0.0), (parf, 3, 5, 0.0), (parf, 4, 3, 0.0)]
            for par, op, k, sigma in cases:
                n0 = cvb.launch_count()
                got = hal.roi_filter(par, rect, op, k, sigma, border, inplace)
                assert cvb.launch_count() > n0, "ROI op %d did not reach the B200 HAL (rect %s border %d)" % (op, rect, border)
                want = ref.roi_filter(par, rect, op, k, sigma, border, inplace)
                what = "cv:: op %d k=%d on ROI %s of a %s parent, border %d, inplace %s" % (op, k, rect, par.dtype, border, inplace)
                if par.dtype == np.uint8:     # bit-exact in the reference's vector body; its scalar remainder columns (width mod 32) may round the other way
                    assert_close(got, want, atol=1, what=what)
                    assert (got != want).mean() < 5e-3, what + ": %d bytes differ" % int((got != want).sum())
                else:
                    assert_close(got, want, atol=1e-3, rtol=1e-5, what=what)


def test_cpp_host_mirror(cvb):
    """tests/cpp/test_host_api (compiled from tests/cpp/test_host_api.cpp against opencv_b200/host/b200cv.hpp) exercises
    Stream / Event / GpuMat / Filter::apply / free functions with cv:: argument order"""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(__file__), "cpp", "test_host_api")
    if not os.path.exists(exe):
        pytest.skip("tests/cpp/test_host_api not built")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


def test_cv_typed_surface_against_real_opencv_headers(cvb):
    """oracle/_ref/test_cv_surface: opencv_b200/host/b200cv_opencv.hpp compiled with -DB200CV_WITH_OPENCV against the reference's own headers and
    linked with the reference's core + imgproc (built by tests/cpp/build_cv_surface.py): cv::InputArray kinds MAT / CUDA_GPU_MAT /
    CUDA_HOST_MEM, createGaussianFilter(...)->apply(src, dst, stream) as in gpu-basics-similarity.cpp:392-404, each result checked against
    the cv:: call on the CPU inside the binary"""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(__file__), "..", "oracle", "_ref", "test_cv_surface")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/test_cv_surface not built (needs the reference's sources at build time)")
    # this tree's libraries, whatever run path the binary was linked with where oracle/_ref was built
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, LD_LIBRARY_PATH=os.pathsep.join([os.path.join(root, "opencv_b200", "lib"), os.path.join(root, "oracle", "_ref")] +
                                                           [p for p in [os.environ.get("LD_LIBRARY_PATH")] if p]))
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "cv surface ok" in r.stdout


def test_host_entries_from_concurrent_threads(cvb, oracle, rng):
    """OpenCV calls its HAL from many threads at once (parallel_for_ bodies, user threads): the host entries keep one context (streams + staging)
    per calling thread.  Eight threads, different image sizes and ops, repeated: every result equals the oracle's."""
    import threading
    from opencv_b200 import hal as H
    imgs = [rand_u8(rng, 200 + 17 * i, 300 + 13 * i, 3) for i in range(8)]
    M = np.array([[0.9, 0.1, 5], [-0.1, 0.9, 7]])
    want = [(oracle.GaussianBlur(im, (5, 5), 0), oracle.cvtColor(im, C.COLOR_BGR2YUV, 3), oracle.resize(im, (im.shape[1] // 2 + 3, im.shape[0] // 2 + 1), 1),
             oracle.warpAffine(im, M, (im.shape[1], im.shape[0]), 1, 1), oracle.matchTemplate(im[:, :, 0].copy(), im[20:36, 30:54, 0].copy(), 3)) for im in imgs]
    errors = []

    def work(i):
        try:
            im = imgs[i]
            for _ in range(12):
                got = (H.GaussianBlur(im, (5, 5), 0), H.cvtColor(im, C.COLOR_BGR2YUV, 3), H.resize(im, (im.shape[1] // 2 + 3, im.shape[0] // 2 + 1), interpolation=1),
                       H.warpAffine(im, M, (im.shape[1], im.shape[0]), 1, 1), H.matchTemplate(im[:, :, 0].copy(), im[20:36, 30:54, 0].copy(), 3))
                for k in range(4):
                    if not np.array_equal(got[k], want[i][k]):
                        errors.append("thread %d op %d differs" % (i, k))
                if not np.allclose(got[4], want[i][4], atol=1e-4):
                    errors.append("thread %d matchTemplate differs" % i)
        except Exception as e:      # noqa: BLE001 -- reported below
            errors.append("thread %d: %r" % (i, e))

    threads = [threading.Thread(target=work, args=(i,)) for i in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:5]
