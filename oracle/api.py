"""oracle/api.py -- numpy-level access to the two CPU oracles.  TEST INFRASTRUCTURE ONLY.

    Oracle("ref")   the UNMODIFIED reference built by oracle/build_ref.py  (oracle/_ref/libocvref.so, prefix ref_)
    Oracle("port")  the plain-C restatement in oracle/port/*.c            (oracle/_build/liboracle_port.so, prefix port_)

Both export the same C signatures (see oracle/ref_shim.cpp), so every test can run against either.
Nothing under opencv_b200/ imports this module.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_LIB = os.path.join(HERE, "_ref", "libocvref.so")
REF_HAL_LIB = os.path.join(HERE, "_ref", "libocvref_hal.so")   # the reference with hal/b200cv_hal_replacement.hpp registered (integration proof)
PORT_LIB = os.path.join(HERE, "_build", "liboracle_port.so")
B200_LIB = os.path.join(os.path.dirname(HERE), "opencv_b200", "lib", "libb200cv.so")

CV_8U, CV_16S, CV_32F = 0, 3, 5
_DEPTH = {np.dtype(np.uint8): CV_8U, np.dtype(np.uint16): 2, np.dtype(np.int16): CV_16S, np.dtype(np.float32): CV_32F}
_NP = {CV_8U: np.uint8, CV_16S: np.int16, CV_32F: np.float32}

vp, sz, dbl = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_double


def cvtype(a):
    cn = 1 if a.ndim == 2 else a.shape[2]
    return _DEPTH[a.dtype] + ((cn - 1) << 3)


def _p(a):
    return a.ctypes.data_as(vp)


def _path(kind):
    return {"ref": REF_LIB, "ref_hal": REF_HAL_LIB}.get(kind, PORT_LIB)


def available(kind):
    return os.path.exists(_path(kind))


def yuv_dst_shape(sw, sh, code):
    """(width, height, channels) of cv::cvtColor's destination for the subsampled-YUV codes (color.cpp:323-372)"""
    if 90 <= code <= 105:
        return sw, sh * 2 // 3, (4 if code in (94, 95, 96, 97, 102, 103, 104, 105) else 3)
    if code == 106:
        return sw, sh * 2 // 3, 1
    if 107 <= code <= 122:
        return sw, sh, (4 if code in (111, 112, 119, 120, 121, 122) else 3)
    if code in (123, 124):
        return sw, sh, 1
    if 127 <= code <= 134:
        return sw, sh * 3 // 2, 1
    if 143 <= code <= 154:
        return sw, sh, 2
    if 46 <= code <= 49 or 139 <= code <= 142:
        return sw, sh, (4 if code >= 139 else 3)
    raise ValueError("not a subsampled-YUV code: %d" % code)


class Oracle:
    def __init__(self, kind="ref"):
        self.kind = kind
        path = _path(kind)
        if not os.path.exists(path):
            raise FileNotFoundError("%s oracle not built: %s" % (kind, path))
        if kind == "ref_hal":
            # its libb200cv.so dependency resolves (by soname) to this tree's library loaded first, not to wherever the run path of the
            # reference build points
            ctypes.CDLL(B200_LIB)
        self.lib = ctypes.CDLL(path)
        self.pfx = "ref_" if kind in ("ref", "ref_hal") else "port_"

    def has(self, name):
        return hasattr(self.lib, self.pfx + name)

    def fn(self, name):
        return getattr(self.lib, self.pfx + name)

    @staticmethod
    def _ok(rc, what):
        if rc != 0:
            raise RuntimeError("oracle %s failed: %d" % (what, rc))

    # ---- helpers only the real reference has -------------------------------------------------------------
    def set_num_threads(self, n):
        return self.fn("set_num_threads")(int(n))

    def num_threads(self):
        return self.fn("get_num_threads")()

    def rng_fill(self, shape, dtype, seed, lo, hi):
        a = np.zeros(shape, dtype)
        h, w = shape[0], shape[1]
        self._ok(self.fn("rng_fill")(_p(a), sz(a.strides[0]), w, h, cvtype(a), ctypes.c_ulonglong(seed), dbl(lo), dbl(hi)), "rng_fill")
        return a

    def getGaussianKernel(self, n, sigma, ktype=np.float64):
        out = np.zeros(n, ktype)
        self._ok(self.fn("gaussian_kernel")(int(n), dbl(sigma), 6 if ktype == np.float64 else 5, _p(out)), "gaussian_kernel")
        return out

    def getRotationMatrix2D(self, center, angle, scale):
        m = np.zeros((2, 3), np.float64)
        self._ok(self.fn("get_rotation_matrix2d")(dbl(center[0]), dbl(center[1]), dbl(angle), dbl(scale), _p(m)), "rot")
        return m

    # ---- hot-path ops -----------------------------------------------------------------------------------------
    def GaussianBlur(self, src, ksize, sigmaX, sigmaY=0, borderType=4):
        src = np.ascontiguousarray(src)
        dst = np.empty_like(src)
        h, w = src.shape[:2]
        self._ok(self.fn("gaussian_blur")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, cvtype(src),
                                          int(ksize[0]), int(ksize[1]), dbl(sigmaX), dbl(sigmaY), int(borderType)), "GaussianBlur")
        return dst

    def _dst_like(self, src, ddepth):
        return np.empty(src.shape, _NP[ddepth] if ddepth is not None and ddepth >= 0 else src.dtype)

    def sepFilter2D(self, src, ddepth, kx, ky, anchor=(-1, -1), delta=0.0, borderType=4):
        src = np.ascontiguousarray(src)
        dst = self._dst_like(src, ddepth)
        kx = np.ascontiguousarray(kx, np.float32).reshape(-1)
        ky = np.ascontiguousarray(ky, np.float32).reshape(-1)
        h, w = src.shape[:2]
        self._ok(self.fn("sep_filter2d")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, cvtype(src),
                                         -1 if ddepth is None else int(ddepth), _p(kx), len(kx), _p(ky), len(ky),
                                         int(anchor[0]), int(anchor[1]), dbl(delta), int(borderType)), "sepFilter2D")
        return dst

    def filter2D(self, src, ddepth, kernel, anchor=(-1, -1), delta=0.0, borderType=4):
        src = np.ascontiguousarray(src)
        dst = self._dst_like(src, ddepth)
        k = np.ascontiguousarray(kernel, np.float32)
        h, w = src.shape[:2]
        self._ok(self.fn("filter2d")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, cvtype(src),
                                     -1 if ddepth is None else int(ddepth), _p(k), k.shape[1], k.shape[0],
                                     int(anchor[0]), int(anchor[1]), dbl(delta), int(borderType)), "filter2D")
        return dst

    def Sobel(self, src, ddepth, dx, dy, ksize=3, scale=1.0, delta=0.0, borderType=4):
        src = np.ascontiguousarray(src)
        dst = self._dst_like(src, ddepth)
        h, w = src.shape[:2]
        self._ok(self.fn("sobel")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, cvtype(src),
                                  -1 if ddepth is None else int(ddepth), int(dx), int(dy), int(ksize), dbl(scale), dbl(delta),
                                  int(borderType)), "Sobel")
        return dst

    def resize(self, src, dsize, interpolation=1):
        src = np.ascontiguousarray(src)
        dw, dh = dsize
        dst = np.empty((dh, dw) + src.shape[2:], src.dtype)
        sh, sw = src.shape[:2]
        self._ok(self.fn("resize")(_p(src), sz(src.strides[0]), sw, sh, _p(dst), sz(dst.strides[0]), dw, dh, cvtype(src),
                                   int(interpolation)), "resize")
        return dst

    def resize_fxfy(self, src, fx, fy, interpolation=1):
        """cv::resize(src, dst, Size(), fx, fy): only the real reference has it"""
        src = np.ascontiguousarray(src)
        sh, sw = src.shape[:2]
        dw, dh = int(round(sw * fx)), int(round(sh * fy))
        dst = np.empty((dh, dw) + src.shape[2:], src.dtype)
        self._ok(self.fn("resize_fxfy")(_p(src), sz(src.strides[0]), sw, sh, _p(dst), sz(dst.strides[0]), dw, dh, cvtype(src),
                                        int(interpolation), ctypes.c_double(fx), ctypes.c_double(fy)), "resize_fxfy")
        return dst

    def roi_filter(self, parent, rect, op, k, sigma=0.0, border=4, inplace=False):
        """op on parent(rect) as a cv::Mat ROI (0 GaussianBlur, 1 blur, 2 sepFilter2D, 3 filter2D, 4 Sobel); only the real reference has it"""
        parent = np.ascontiguousarray(parent)
        ph, pw = parent.shape[:2]
        rx, ry, rw, rh = rect
        dst = np.empty((rh, rw) + parent.shape[2:], parent.dtype)
        self._ok(self.fn("roi_filter")(_p(parent), sz(parent.strides[0]), pw, ph, cvtype(parent), rx, ry, rw, rh, _p(dst), sz(dst.strides[0]),
                                       int(op), int(k), dbl(sigma), int(border), int(bool(inplace))), "roi_filter")
        return dst

    def _warp(self, name, src, M, dsize, flags, borderMode, borderValue, dst0=None):
        src = np.ascontiguousarray(src)
        dw, dh = dsize
        dst = np.zeros((dh, dw) + src.shape[2:], src.dtype)
        if dst0 is not None:            # BORDER_TRANSPARENT: the destination's previous content shows through
            dst[...] = dst0
        sh, sw = src.shape[:2]
        M = np.ascontiguousarray(M, np.float64)
        bv = np.zeros(4, np.float64)
        bv[:len(np.atleast_1d(borderValue))] = np.atleast_1d(borderValue)
        self._ok(self.fn(name)(_p(src), sz(src.strides[0]), sw, sh, _p(dst), sz(dst.strides[0]), dw, dh, cvtype(src),
                               _p(M), int(flags), int(borderMode), _p(bv)), name)
        return dst

    def warpAffine(self, src, M, dsize, flags=1, borderMode=0, borderValue=0, dst=None):
        return self._warp("warp_affine", src, M, dsize, flags, borderMode, borderValue, dst)

    def warpPerspective(self, src, M, dsize, flags=1, borderMode=0, borderValue=0, dst=None):
        return self._warp("warp_perspective", src, M, dsize, flags, borderMode, borderValue, dst)

    def remap(self, src, map1, map2, interpolation, borderMode=0, borderValue=0, dst=None):
        src = np.ascontiguousarray(src); map1 = np.ascontiguousarray(map1)
        map2 = np.ascontiguousarray(map2) if map2 is not None else None
        dh, dw = map1.shape[:2]
        dst0 = dst
        dst = np.zeros((dh, dw) + src.shape[2:], src.dtype)
        if dst0 is not None:
            dst[...] = dst0
        sh, sw = src.shape[:2]
        bv = np.zeros(4, np.float64)
        bv[:len(np.atleast_1d(borderValue))] = np.atleast_1d(borderValue)
        self._ok(self.fn("remap")(_p(src), sz(src.strides[0]), sw, sh, cvtype(src), _p(dst), sz(dst.strides[0]), dw, dh,
                                  _p(map1), sz(map1.strides[0]), cvtype(map1), _p(map2) if map2 is not None else None,
                                  sz(map2.strides[0]) if map2 is not None else sz(0), cvtype(map2) if map2 is not None else 0,
                                  int(interpolation), int(borderMode), _p(bv)), "remap")
        return dst

    def convertMaps(self, mapx, mapy, nninterpolation=False):
        mapx = np.ascontiguousarray(mapx, np.float32); mapy = np.ascontiguousarray(mapy, np.float32)
        h, w = mapx.shape
        xy = np.zeros((h, w, 2), np.int16); fr = np.zeros((h, w), np.uint16)
        self._ok(self.fn("convert_maps")(_p(mapx), _p(mapy), w, h, _p(xy), _p(fr), int(bool(nninterpolation))), "convertMaps")
        return xy, fr

    def pyrDown(self, src, borderType=4):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dst = np.zeros(((h + 1) // 2, (w + 1) // 2) + src.shape[2:], src.dtype)
        self._ok(self.fn("pyr_down")(_p(src), sz(src.strides[0]), w, h, cvtype(src), _p(dst), sz(dst.strides[0]), int(borderType)), "pyrDown")
        return dst

    def pyrUp(self, src):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dst = np.zeros((h * 2, w * 2) + src.shape[2:], src.dtype)
        self._ok(self.fn("pyr_up")(_p(src), sz(src.strides[0]), w, h, cvtype(src), _p(dst), sz(dst.strides[0])), "pyrUp")
        return dst

    def boxFilter(self, src, ddepth, ksize, anchor=(-1, -1), normalize=True, borderType=4):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dd = {-1: src.dtype, 0: np.uint8, 5: np.float32}[int(ddepth)]
        dst = np.zeros(src.shape, dd)
        self._ok(self.fn("box_filter")(_p(src), sz(src.strides[0]), w, h, cvtype(src), _p(dst), sz(dst.strides[0]), int(ddepth),
                                       int(ksize[0]), int(ksize[1]), int(anchor[0]), int(anchor[1]), int(bool(normalize)), int(borderType)), "boxFilter")
        return dst

    def blur(self, src, ksize, anchor=(-1, -1), borderType=4):
        return self.boxFilter(src, -1, ksize, anchor, True, borderType)

    def cvtColor(self, src, code, dcn):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dst = np.empty((h, w) if dcn == 1 else (h, w, dcn), src.dtype)
        self._ok(self.fn("cvt_color")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, cvtype(src), cvtype(dst),
                                      int(code)), "cvtColor")
        return dst

    def cvtColorLab(self, src, code):
        """8-bit BGR / RGB <-> Lab: codes 44, 45, 74, 75 (to Lab) and 56, 57, 78, 79 (from Lab); <-> XYZ: 32-35.  The reference goes through cvtColor."""
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dst = np.zeros((h, w, 3), np.uint8)
        if self.kind != "port":
            return self.cvtColor(src, code, 3)
        if int(code) in (32, 33, 34, 35):
            self._ok(self.fn("cvt_color_xyz")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, src.shape[2], 3, int(code)), "cvtColor(XYZ)")
        elif int(code) in (44, 45, 74, 75):
            self._ok(self.fn("cvt_color_lab")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, src.shape[2], int(code)), "cvtColor(Lab)")
        else:
            self._ok(self.fn("cvt_color_lab_inv")(_p(src), sz(src.strides[0]), _p(dst), sz(dst.strides[0]), w, h, 3, int(code)), "cvtColor(Lab inverse)")
        return dst

    def cvtColorYUV(self, src, code):
        """subsampled YUV wire formats (codes 90-134): destination shape follows from the code"""
        src = np.ascontiguousarray(src)
        sh, sw = src.shape[:2]
        scn = 1 if src.ndim == 2 else src.shape[2]
        dw, dh, dcn = yuv_dst_shape(sw, sh, code)
        dst = np.zeros((dh, dw) if dcn == 1 else (dh, dw, dcn), np.uint8)
        self._ok(self.fn("cvt_color_yuv")(_p(src), sz(src.strides[0]), sw, sh, scn, _p(dst), sz(dst.strides[0]), dw, dh, dcn, int(code)), "cvtColor(YUV)")
        return dst

    def cvtColorTwoPlane(self, y, uv, code):
        y = np.ascontiguousarray(y); uv = np.ascontiguousarray(uv)
        h, w = y.shape[:2]
        dcn = 4 if int(code) in (94, 95, 96, 97) else 3
        dst = np.zeros((h, w, dcn), np.uint8)
        self._ok(self.fn("cvt_color_two_plane")(_p(y), sz(y.strides[0]), _p(uv), sz(uv.strides[0]), w, h, _p(dst), sz(dst.strides[0]), dcn, int(code)), "cvtColorTwoPlane")
        return dst

    def integral(self, src, with_sqsum=False):
        src = np.ascontiguousarray(src)
        h, w = src.shape
        s = np.zeros((h + 1, w + 1), np.int32)
        q = np.zeros((h + 1, w + 1), np.float64) if with_sqsum else None
        self._ok(self.fn("integral")(_p(src), sz(src.strides[0]), w, h, _p(s), sz(s.strides[0]), _p(q) if with_sqsum else None,
                                     sz(q.strides[0]) if with_sqsum else sz(0)), "integral")
        return (s, q) if with_sqsum else s

    def matchTemplate(self, image, templ, method):
        image = np.ascontiguousarray(image)
        templ = np.ascontiguousarray(templ)
        ih, iw = image.shape[:2]
        th, tw = templ.shape[:2]
        res = np.empty((ih - th + 1, iw - tw + 1), np.float32)
        self._ok(self.fn("match_template")(_p(image), sz(image.strides[0]), iw, ih, _p(templ), sz(templ.strides[0]), tw, th,
                                           cvtype(image), _p(res), sz(res.strides[0]), int(method)), "matchTemplate")
        return res

    def matchTemplateMasked(self, image, templ, method, mask):
        image = np.ascontiguousarray(image); templ = np.ascontiguousarray(templ); mask = np.ascontiguousarray(mask)
        ih, iw = image.shape[:2]
        th, tw = templ.shape[:2]
        res = np.empty((ih - th + 1, iw - tw + 1), np.float32)
        self._ok(self.fn("match_template_masked")(_p(image), sz(image.strides[0]), iw, ih, _p(templ), sz(templ.strides[0]), tw, th, cvtype(image),
                                                  _p(mask), sz(mask.strides[0]), cvtype(mask), _p(res), sz(res.strides[0]), int(method)), "matchTemplate(mask)")
        return res

    def cornerHarris(self, src, blockSize, ksize, k, borderType=4):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dst = np.empty((h, w), np.float32)
        self._ok(self.fn("corner_harris")(_p(src), sz(src.strides[0]), w, h, cvtype(src), _p(dst), sz(dst.strides[0]),
                                          int(blockSize), int(ksize), dbl(k), int(borderType)), "cornerHarris")
        return dst

    def cornerMinEigenVal(self, src, blockSize, ksize=3, borderType=4):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        dst = np.empty((h, w), np.float32)
        self._ok(self.fn("corner_min_eigen_val")(_p(src), sz(src.strides[0]), w, h, cvtype(src), _p(dst), sz(dst.strides[0]),
                                                 int(blockSize), int(ksize), int(borderType)), "cornerMinEigenVal")
        return dst

    def goodFeaturesToTrack(self, src, maxCorners, qualityLevel, minDistance, blockSize=3, gradientSize=3, useHarrisDetector=False,
                            k=0.04, max_out=100000):
        src = np.ascontiguousarray(src)
        h, w = src.shape[:2]
        pts = np.zeros((max_out, 2), np.float32)
        q = np.zeros(max_out, np.float32)
        n = ctypes.c_int(0)
        self._ok(self.fn("good_features_to_track")(_p(src), sz(src.strides[0]), w, h, cvtype(src), _p(pts), _p(q), int(max_out),
                                                   ctypes.byref(n), int(maxCorners), dbl(qualityLevel), dbl(minDistance),
                                                   int(blockSize), int(gradientSize), int(bool(useHarrisDetector)), dbl(k)), "gftt")
        cnt = min(n.value, max_out)
        return pts[:cnt].copy(), q[:cnt].copy()

    def sift_detect_and_compute(self, gray, nfeatures=0, nOctaveLayers=3, contrastThreshold=0.04, edgeThreshold=10, sigma=1.6, max_kp=200000,
                                precise_upscale=True, mask=None):
        """the reference's cv::SIFT::detectAndCompute (real reference only): (keypoints[n,5] = x, y, size, angle, response; octave[n]; desc[n,128]).
        precise_upscale=True is SIFT::create(..., enable_precise_upscale=true): the first-octave image sift_pyramid() builds."""
        gray = np.ascontiguousarray(gray)
        mask = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        h, w = gray.shape
        kp = np.zeros((max_kp, 6), np.float32); desc = np.zeros((max_kp, 128), np.float32); n = ctypes.c_int(0)
        self._ok(self.fn("sift_detect_and_compute")(_p(gray), sz(gray.strides[0]), w, h, int(nfeatures), int(nOctaveLayers), dbl(contrastThreshold),
                                                     dbl(edgeThreshold), dbl(sigma), int(bool(precise_upscale)),
                                                     _p(mask) if mask is not None else None, sz(mask.strides[0]) if mask is not None else sz(0),
                                                     int(max_kp), _p(kp), _p(desc), ctypes.byref(n)), "SIFT")
        m = min(n.value, max_kp)
        return kp[:m, :5].copy(), kp[:m, 5].copy().view(np.int32), desc[:m].copy()

    def sift_detect_from_pyramid(self, gauss, dog, nOctaveLayers=3, contrastThreshold=0.04, edgeThreshold=10, sigma=1.6, upscale=True, max_kp=200000,
                                 nfeatures=0):
        """port only: extrema + refinement + orientation on GIVEN pyramids ([octave][layer] lists as sift_pyramid returns) -> (kp[n,5], octave[n])"""
        no = len(gauss)
        dims = np.array([[g[0].shape[1], g[0].shape[0]] for g in gauss], np.int32).reshape(-1)
        G = np.concatenate([np.ascontiguousarray(l, np.float32).reshape(-1) for g in gauss for l in g])
        D = np.concatenate([np.ascontiguousarray(l, np.float32).reshape(-1) for d in dog for l in d])
        kp = np.zeros((max_kp, 6), np.float32); n = ctypes.c_int(0)
        self._ok(self.fn("sift_detect")(_p(G), _p(D), _p(dims), no, int(nOctaveLayers), dbl(contrastThreshold), dbl(edgeThreshold), dbl(sigma),
                                        -1 if upscale else 0, int(nfeatures), int(max_kp), _p(kp), ctypes.byref(n)), "sift_detect")
        m = min(n.value, max_kp)
        return kp[:m, :5].copy(), kp[:m, 5].copy().view(np.int32)

    def sift_descriptors_from_pyramid(self, gauss, kp, octave, nOctaveLayers=3, upscale=True):
        """port only: 128-float descriptors of given keypoints (kp[n,5], octave[n] as sift_detect_* return) on a GIVEN Gaussian pyramid"""
        no = len(gauss)
        dims = np.array([[g[0].shape[1], g[0].shape[0]] for g in gauss], np.int32).reshape(-1)
        G = np.concatenate([np.ascontiguousarray(l, np.float32).reshape(-1) for g in gauss for l in g])
        k6 = np.zeros((len(kp), 6), np.float32); k6[:, :5] = kp; k6[:, 5] = np.asarray(octave, np.int32).view(np.float32)
        desc = np.zeros((len(kp), 128), np.float32)
        self._ok(self.fn("sift_descriptors")(_p(G), _p(dims), no, int(nOctaveLayers), -1 if upscale else 0, _p(k6), len(kp), _p(desc)), "sift_descriptors")
        return desc

    def sift_pyramid(self, gray, nOctaveLayers=3, sigma=1.6, upscale=True):
        """returns (gauss list-of-lists [octave][layer], dog list-of-lists)"""
        gray = np.ascontiguousarray(gray)
        h, w = gray.shape
        ge, de, no = sz(0), sz(0), ctypes.c_int(0)
        f = self.fn("sift_pyramid")
        upscale = int(upscale)               # True / 1: precise first octave (warpAffine); 2: SIFT::create's default (resize); 0: no upscaling
        self._ok(f(_p(gray), sz(gray.strides[0]), w, h, int(nOctaveLayers), dbl(sigma), upscale, None, ctypes.byref(ge),
                   None, ctypes.byref(de), ctypes.byref(no), None), "sift_pyramid(query)")
        G = np.zeros(ge.value, np.float32)
        D = np.zeros(de.value, np.float32)
        dims = np.zeros(2 * no.value, np.int32)
        self._ok(f(_p(gray), sz(gray.strides[0]), w, h, int(nOctaveLayers), dbl(sigma), upscale, _p(G), ctypes.byref(ge),
                   _p(D), ctypes.byref(de), ctypes.byref(no), _p(dims)), "sift_pyramid")
        return unpack_pyramid(G, D, dims, no.value, nOctaveLayers)


def unpack_pyramid(G, D, dims, n_octaves, n_layers):
    gauss, dog = [], []
    go = do = 0
    for o in range(n_octaves):
        w, h = int(dims[2 * o]), int(dims[2 * o + 1])
        gl, dl = [], []
        for _ in range(n_layers + 3):
            gl.append(G[go:go + w * h].reshape(h, w)); go += w * h
        for _ in range(n_layers + 2):
            dl.append(D[do:do + w * h].reshape(h, w)); do += w * h
        gauss.append(gl); dog.append(dl)
    return gauss, dog
