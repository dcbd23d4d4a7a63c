"""ctypes binding of the CPU oracle of the camera frame -> level-0 working image step (ellc_ingest_oracle.cpp; test infrastructure
only: tests/ and tools/bench_ingest.py use it as the checker, the product never imports it)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libellc_ingest_oracle.so")
_SRC = [os.path.join(_HERE, "ellc_ingest_oracle.cpp"), os.path.join(_HERE, "ellc_ingest_oracle.h")]
_lib = None


def build(force=False):
    """Compile with tests/ingest_oracle/Makefile (also run by __graft_entry__.build())."""
    if force or not os.path.exists(_SO) or any(os.path.getmtime(p) > os.path.getmtime(_SO) for p in _SRC):
        subprocess.check_call(["make", "-C", _HERE, "clean", "all"], stdout=subprocess.DEVNULL)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


# ---- camera frame -> level-0 working image (frame::frame(VideoCapture), src/Frame.cpp:34-119) ----------------------------------
def _cam(img):
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape[:2]
    c = 1 if img.ndim == 2 else img.shape[2]
    return img, w, h, c


def _d(a, n):
    return np.ascontiguousarray(np.asarray(a, np.float64).reshape(n))


def bgr2gray(img):
    """cv::cvtColor(CV_BGR2GRAY) of OpenCV 3.0.0 (14-bit coefficients); a 1-channel image is returned as it is."""
    img, w, h, c = _cam(img)
    out = np.empty((h, w), np.uint8)
    lib().ellc_oracle_bgr2gray(_p(img), w, h, c, w * c, _p(out))
    return out


def undistort_map(K, dist, new_K, w, h):
    """initUndistortRectifyMap(K, dist, I, new_K, (w, h), CV_16SC2) -> (map_xy [h, w, 2] int16, map_frac [h, w] uint16)."""
    xy = np.empty((h, w, 2), np.int16); fr = np.empty((h, w), np.uint16)
    lib().ellc_oracle_undistort_map(_p(_d(K, 9)), _p(_d(dist, 5)), _p(_d(new_K, 9)), int(w), int(h), _p(xy), _p(fr))
    return xy, fr


def remap(gray, map_xy, map_frac):
    gray = np.ascontiguousarray(gray, np.uint8)
    map_xy = np.ascontiguousarray(map_xy, np.int16); map_frac = np.ascontiguousarray(map_frac, np.uint16)
    h, w = map_frac.shape
    out = np.empty((h, w), np.uint8)
    lib().ellc_oracle_remap_u8(_p(gray), gray.shape[1], gray.shape[0], _p(map_xy), _p(map_frac), w, h, _p(out))
    return out


def resize(gray, dw, dh):
    gray = np.ascontiguousarray(gray, np.uint8)
    out = np.empty((dh, dw), np.uint8)
    lib().ellc_oracle_resize_u8(_p(gray), gray.shape[1], gray.shape[0], _p(out), int(dw), int(dh))
    return out


def ingest(img, dw, dh, undistort=False, K=None, dist=None, new_K=None):
    """The reference's order: gray -> undistort (if set) -> resize to dw x dh."""
    img, w, h, c = _cam(img)
    out = np.empty((dh, dw), np.uint8)
    z9, z5 = np.zeros(9), np.zeros(5)
    lib().ellc_oracle_ingest(_p(img), w, h, c, w * c, 1 if undistort else 0, _p(_d(K if undistort else z9, 9)),
                             _p(_d(dist if undistort else z5, 5)), _p(_d(new_K if undistort else z9, 9)), _p(out), int(dw), int(dh))
    return out


def optimal_new_camera_matrix(K, dist, w, h, alpha):
    out = np.empty(9, np.float64)
    lib().ellc_oracle_optimal_new_camera_matrix(_p(_d(K, 9)), _p(_d(dist, 5)), int(w), int(h), C.c_double(alpha), _p(out))
    return out.reshape(3, 3)
