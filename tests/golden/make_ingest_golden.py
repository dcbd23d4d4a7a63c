"""Generates tests/golden/ingest_vectors.npz: camera frame -> level-0 working image, stage by stage, from cv2.

The reference builds its working image in frame::frame(VideoCapture) (src/Frame.cpp:34-119, SURVEY 3.1) in this order:
BGR -> gray (CV_BGR2GRAY), lens undistortion (getOptimalNewCameraMatrix + cv::undistort, FLAG_DO_UNDISTORTION), resize by
RESIZE_FACTOR (INTER_LINEAR).  Per case the file records:
  gray15      cv2.cvtColor(BGR2GRAY) of cv2 4.x (15-bit coefficients): only to quantify the gap to OpenCV 3.0.0's 14-bit form
  gray        OpenCV 3.0.0's CV_BGR2GRAY, (B*1868 + G*9617 + R*4899 + 8192) >> 14 (the reference pins 3.0.0)
  map_xy, map_frac   cv2.initUndistortRectifyMap(K, dist, I, new_K, size, CV_16SC2)          (undistorting cases)
  undist      cv2.remap(gray, map, INTER_LINEAR, BORDER_CONSTANT 0) == cv2.undistort(gray, K, dist, new_K)
  out         cv2.resize(undist or gray, working size, INTER_LINEAR): the composed pipeline in the reference order
  new_K_a{0,05,1}    cv2.getOptimalNewCameraMatrix(K, dist, size, alpha) for alpha 0, 0.5, 1
Inputs are regenerated from their seed by the tests (camera_image()); every array above DIGEST_BYTES is stored as the SHA-256 of
its bytes.  The generator also checks its numpy restatement of each stage (model_*) against cv2 on every case, so that the
arithmetic DESIGN.md section 9 states is the arithmetic cv2 runs.

    python tests/golden/make_ingest_golden.py
"""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "ingest_vectors.npz")
DIGEST_BYTES = 16384

# the reference's camera (src/ExternVariable.h:53-59: ORIG_FX / ORIG_FY at 1920x1080) with a seeded 5-coefficient distortion
FX, FY = 1642.405612, 1636.148027
DIST = np.array([0.12, -0.25, 0.001, -0.0005, 0.08])

# name: (camera w, h, channels, working w, h, undistort, alpha of new_K)
CASES = {
    "f4":        (192, 144, 3, 48, 36, 0, None),
    "f4_ud_a0":  (192, 144, 3, 48, 36, 1, 0.0),
    "f4_ud_a1":  (192, 144, 3, 48, 36, 1, 1.0),
    "f2":        (96, 72, 3, 48, 36, 0, None),
    "nonint":    (1280, 720, 3, 480, 270, 1, 1.0),
    "gray1_ud":  (160, 120, 1, 40, 30, 1, 0.0),
    "odd_ud":    (203, 151, 3, 51, 38, 1, 0.5),
}


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def camera_matrix(w, h):
    """The reference's focal lengths scaled to the camera width, principal point at the centre (plus a seeded offset)."""
    s = w / 1920.0
    return np.array([[FX * s, 0.0, w / 2.0 + 1.25], [0.0, FY * s, h / 2.0 - 0.75], [0.0, 0.0, 1.0]])


def camera_image(name):
    w, h, c = CASES[name][:3]
    rng = np.random.default_rng(sum(map(ord, name)))
    shape = (h, w, c) if c == 3 else (h, w)
    return rng.integers(0, 256, shape, dtype=np.uint8)


# ---- numpy restatement of each stage (OpenCV 3.0.0 arithmetic) -------------------------------------------------------------
def model_gray(img):
    if img.ndim == 2:
        return img.copy()
    b, g, r = (img[..., k].astype(np.int32) for k in range(3))
    return ((b * 1868 + g * 9617 + r * 4899 + 8192) >> 14).astype(np.uint8)


def inv3(a):
    """Matx33d::inv (Matx_FastInvOp<_Tp, 3>: cofactors over the determinant) in OpenCV's operation order."""
    d = a[0, 0] * (a[1, 1] * a[2, 2] - a[2, 1] * a[1, 2]) - a[0, 1] * (a[1, 0] * a[2, 2] - a[2, 0] * a[1, 2]) + \
        a[0, 2] * (a[1, 0] * a[2, 1] - a[2, 0] * a[1, 1])
    d = 1.0 / d
    b = np.empty((3, 3))
    b[0, 0] = (a[1, 1] * a[2, 2] - a[1, 2] * a[2, 1]) * d
    b[0, 1] = (a[0, 2] * a[2, 1] - a[0, 1] * a[2, 2]) * d
    b[0, 2] = (a[0, 1] * a[1, 2] - a[0, 2] * a[1, 1]) * d
    b[1, 0] = (a[1, 2] * a[2, 0] - a[1, 0] * a[2, 2]) * d
    b[1, 1] = (a[0, 0] * a[2, 2] - a[0, 2] * a[2, 0]) * d
    b[1, 2] = (a[0, 2] * a[1, 0] - a[0, 0] * a[1, 2]) * d
    b[2, 0] = (a[1, 0] * a[2, 1] - a[1, 1] * a[2, 0]) * d
    b[2, 1] = (a[0, 1] * a[2, 0] - a[0, 0] * a[2, 1]) * d
    b[2, 2] = (a[0, 0] * a[1, 1] - a[0, 1] * a[1, 0]) * d
    return b


def model_map(K, dist, newK, w, h):
    """initUndistortRectifyMap(..., CV_16SC2), incremental form (_x += ir[0] along a row) as OpenCV 3.0.0 writes it."""
    ir = inv3(newK).reshape(9)
    k1, k2, p1, p2, k3 = dist
    fx, fy, u0, v0 = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    i = np.arange(h, dtype=np.float64)[:, None]

    def run(c0, c1, c2):
        a = np.empty((h, w))
        a[:, :1] = i * c1 + c2
        a[:, 1:] = c0
        return np.add.accumulate(a, axis=1)                  # sequential left-to-right sums, as the loop adds them
    _x, _y, _w = run(ir[0], ir[1], ir[2]), run(ir[3], ir[4], ir[5]), run(ir[6], ir[7], ir[8])
    wi = 1.0 / _w
    x = _x * wi; y = _y * wi
    x2 = x * x; y2 = y * y
    r2 = x2 + y2; _2xy = 2 * x * y
    kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((0.0 * r2 + 0.0) * r2 + 0.0) * r2)
    u = fx * (x * kr + p1 * _2xy + p2 * (r2 + 2 * x2)) + u0
    v = fy * (y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy) + v0
    iu = np.clip(np.rint(u * 32), -2 ** 31, 2 ** 31 - 1).astype(np.int64)
    iv = np.clip(np.rint(v * 32), -2 ** 31, 2 ** 31 - 1).astype(np.int64)
    xy = np.stack([(iu >> 5).astype(np.int16), (iv >> 5).astype(np.int16)], axis=-1)
    frac = ((iv & 31) * 32 + (iu & 31)).astype(np.uint16)
    return xy, frac


def model_remap(src, xy, frac):
    """remap INTER_LINEAR / BORDER_CONSTANT 0 with a CV_16SC2 map: weights (32-a)(32-b)*32 ..., (sum + 2^14) >> 15."""
    h, w = src.shape
    x0 = xy[..., 0].astype(np.int64); y0 = xy[..., 1].astype(np.int64)
    a = (frac & 31).astype(np.int64); b = (frac >> 5).astype(np.int64)
    s = src.astype(np.int64)

    def tap(yy, xx):
        ok = (xx >= 0) & (xx < w) & (yy >= 0) & (yy < h)
        return np.where(ok, s[np.clip(yy, 0, h - 1), np.clip(xx, 0, w - 1)], 0)
    acc = tap(y0, x0) * (32 - a) * (32 - b) * 32 + tap(y0, x0 + 1) * a * (32 - b) * 32 + \
        tap(y0 + 1, x0) * (32 - a) * b * 32 + tap(y0 + 1, x0 + 1) * a * b * 32
    return np.clip((acc + (1 << 14)) >> 15, 0, 255).astype(np.uint8)


def resize_taps(ssize, dsize):
    """cv::resize INTER_LINEAR coefficient tables along one axis (resizeGeneric): float source coordinate, clamped borders,
    coefficients saturate_cast<short>(c * 2048).  Returns (i0, i1, a0, a1) per destination index."""
    scale = 1.0 / (dsize / ssize)
    i0 = np.empty(dsize, np.int64); a0 = np.empty(dsize, np.int64); a1 = np.empty(dsize, np.int64)
    for d in range(dsize):
        f = np.float32((d + 0.5) * scale - 0.5)
        s = int(np.floor(f))
        f = np.float32(f - np.float32(s))
        if s < 0:
            f, s = np.float32(0), 0
        if s + 1 >= ssize and s >= ssize - 1:
            f, s = np.float32(0), ssize - 1
        i0[d] = s
        a0[d] = int(np.rint(np.float32(np.float32(1) - f) * np.float32(2048)))
        a1[d] = int(np.rint(f * np.float32(2048)))
    return i0, np.minimum(i0 + 1, ssize - 1), a0, a1


def model_resize(src, dw, dh):
    """Horizontal S[x0]*a0 + S[x1]*a1; vertical ((b0*(h0>>4))>>16) + ((b1*(h1>>4))>>16) + 2) >> 2."""
    sh, sw = src.shape
    x0, x1, a0, a1 = resize_taps(sw, dw)
    y0, y1, b0, b1 = resize_taps(sh, dh)
    s = src.astype(np.int64)
    hr = s[:, x0] * a0 + s[:, x1] * a1
    h0, h1 = hr[y0], hr[y1]
    out = (((b0[:, None] * (h0 >> 4)) >> 16) + ((b1[:, None] * (h1 >> 4)) >> 16) + 2) >> 2
    return np.clip(out, 0, 255).astype(np.uint8)


def model_pipeline(img, dw, dh, undistort, K=None, dist=None, newK=None):
    g = model_gray(img)
    if undistort:
        xy, fr = model_map(K, dist, newK, g.shape[1], g.shape[0])
        g = model_remap(g, xy, fr)
    return model_resize(g, dw, dh)


def store(out, key, a):
    a = np.ascontiguousarray(a)
    if a.nbytes > DIGEST_BYTES:
        out[key + "_sha"] = np.array(digest(a))
    else:
        out[key] = a


def main():
    import cv2
    cv2.setNumThreads(1)
    out = {"dist": DIST, "cases": np.array(list(CASES))}
    for name, (w, h, c, dw, dh, ud, alpha) in CASES.items():
        img = camera_image(name)
        K = camera_matrix(w, h)
        store(out, f"{name}/input", img)
        out[f"{name}/K"] = K
        gray = model_gray(img)
        if c == 3:
            g15 = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
            store(out, f"{name}/gray15", g15)
            out[f"{name}/gray15_diff"] = np.array([int((g15 != gray).sum()), int(np.abs(g15.astype(int) - gray).max())])
        store(out, f"{name}/gray", gray)
        for a, tag in ((0.0, "a0"), (0.5, "a05"), (1.0, "a1")):
            nk, _ = cv2.getOptimalNewCameraMatrix(K, DIST, (w, h), a)
            out[f"{name}/new_K_{tag}"] = nk
        src = gray
        if ud:
            newK = cv2.getOptimalNewCameraMatrix(K, DIST, (w, h), alpha)[0]
            out[f"{name}/new_K"] = newK
            m1, m2 = cv2.initUndistortRectifyMap(K, DIST, None, newK, (w, h), cv2.CV_16SC2)
            xy, fr = model_map(K, DIST, newK, w, h)
            assert np.array_equal(xy, m1) and np.array_equal(fr, m2), name
            store(out, f"{name}/map_xy", m1)
            store(out, f"{name}/map_frac", m2)
            und = cv2.remap(gray, m1, m2, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
            assert np.array_equal(und, cv2.undistort(gray, K, DIST, None, newK)), name
            assert np.array_equal(und, model_remap(gray, xy, fr)), name
            store(out, f"{name}/undist", und)
            src = und
        res = cv2.resize(src, (dw, dh), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(res, model_resize(src, dw, dh)), name
        cv2.setUseOptimized(False)
        assert np.array_equal(res, cv2.resize(src, (dw, dh), interpolation=cv2.INTER_LINEAR)), name
        cv2.setUseOptimized(True)
        store(out, f"{name}/out", res)
    # gray-then-resize against resize-then-gray on the factor-4 case: the order matters
    img = camera_image("f4")
    a = cv2.resize(model_gray(img), (48, 36), interpolation=cv2.INTER_LINEAR)
    b = model_gray(cv2.resize(img, (48, 36), interpolation=cv2.INTER_LINEAR))
    out["order_diff_f4"] = np.array([int((a != b).sum()), a.size])
    out["source"] = np.array(f"cv2 {cv2.__version__}")
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, {k: v for k, v in out.items() if k.endswith("_diff") or k == "order_diff_f4"})


if __name__ == "__main__":
    main()
