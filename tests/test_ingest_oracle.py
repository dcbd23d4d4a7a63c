"""CPU: the oracle's restatement of the camera -> level-0 step (gray, undistortion, resize; frame::frame(VideoCapture)) against
the cv2 fixture tests/golden/ingest_vectors.npz, stage by stage and composed, and the host helper ellc_optimal_new_camera_matrix."""
import ctypes as C
import hashlib
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_ingest_golden as mk  # noqa: E402
from tests import ingest_oracle  # noqa: E402

G = np.load(os.path.join(HERE, "golden", "ingest_vectors.npz"))
CASES = list(mk.CASES)


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def same(key, got):
    """got equals the fixture entry `key`, stored either as the array or as the SHA-256 of its bytes."""
    if key in G:
        return np.array_equal(G[key], got) and G[key].dtype == got.dtype
    return str(G[key + "_sha"]) == digest(got)


def test_inputs_regenerate():
    for name in CASES:
        assert same(f"{name}/input", mk.camera_image(name)), name


@pytest.mark.parametrize("name", CASES)
def test_oracle_stages_equal_fixture(name):
    w, h, c, dw, dh, ud, _ = mk.CASES[name]
    img = mk.camera_image(name)
    gray = ingest_oracle.bgr2gray(img)
    assert same(f"{name}/gray", gray)
    src = gray
    if ud:
        xy, fr = ingest_oracle.undistort_map(G[f"{name}/K"], G["dist"], G[f"{name}/new_K"], w, h)
        assert same(f"{name}/map_xy", xy) and same(f"{name}/map_frac", fr)
        src = ingest_oracle.remap(gray, xy, fr)
        assert same(f"{name}/undist", src)
    assert same(f"{name}/out", ingest_oracle.resize(src, dw, dh))
    composed = ingest_oracle.ingest(img, dw, dh, bool(ud), G[f"{name}/K"], G["dist"], G[f"{name}/new_K"] if ud else None)
    assert same(f"{name}/out", composed)


def test_gray_14bit_against_cv2_15bit():
    """OpenCV 3.0.0's 14-bit CV_BGR2GRAY (what the reference runs) against cv2 4.x's 15-bit form: at most 1 level apart, on at
    most 0.5 % of the pixels."""
    for name in CASES:
        if mk.CASES[name][2] != 3:
            continue
        n_diff, max_diff = (int(v) for v in G[f"{name}/gray15_diff"])
        gray = ingest_oracle.bgr2gray(mk.camera_image(name))
        assert max_diff <= 1 and n_diff <= 0.005 * gray.size, (name, n_diff, max_diff)
        if f"{name}/gray15" in G:
            d = np.abs(G[f"{name}/gray15"].astype(int) - gray)
            assert d.max() <= 1 and int((d != 0).sum()) == n_diff


def test_order_matters():
    """Gray-then-resize and resize-then-gray differ: the step follows the reference's order (SURVEY 3.1)."""
    n, size = (int(v) for v in G["order_diff_f4"])
    assert n > 0.05 * size


@pytest.mark.parametrize("alpha,tag", [(0.0, "a0"), (0.5, "a05"), (1.0, "a1")])
def test_optimal_new_camera_matrix_matches_cv2(alpha, tag):
    from egomotion_with_local_loop_closures_b200 import capi
    for name in CASES:
        w, h = mk.CASES[name][:2]
        want = G[f"{name}/new_K_{tag}"]
        for got in (capi.optimal_new_camera_matrix(G[f"{name}/K"], G["dist"], w, h, alpha),
                    ingest_oracle.optimal_new_camera_matrix(G[f"{name}/K"], G["dist"], w, h, alpha)):
            assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max(), (name, got, want)


def test_optimal_new_camera_matrix_rejects_bad_input():
    from egomotion_with_local_loop_closures_b200 import capi
    out = np.zeros(9)
    K = np.ascontiguousarray(mk.camera_matrix(64, 48).reshape(9))
    d = np.ascontiguousarray(mk.DIST)
    L = capi.lib()
    assert L.ellc_optimal_new_camera_matrix(K.ctypes.data, d.ctypes.data, 1, 48, 0.0, out.ctypes.data) == -1
    assert L.ellc_optimal_new_camera_matrix(None, d.ctypes.data, 64, 48, 0.0, out.ctypes.data) == -1


def test_ingest_symbols_exported():
    from egomotion_with_local_loop_closures_b200 import capi
    L = capi.lib()
    for s in ("ellc_optimal_new_camera_matrix", "ellc_set_camera", "ellc_ingest_frames", "ellc_ingest_keyframe",
              "ellc_read_camera_tables"):
        assert s in capi.SYMBOLS and getattr(L, s) is not None
    assert C.sizeof(capi.Camera) == 208
