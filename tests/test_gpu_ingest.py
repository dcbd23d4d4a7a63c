"""GPU: camera images -> level-0 slot images on the device (ellc_set_camera / ellc_ingest_frames / ellc_ingest_keyframe) against
the cv2 fixture and the CPU oracle, bit for bit, and everything downstream of the slot against the plain upload path."""
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

pytestmark = pytest.mark.gpu

G = np.load(os.path.join(HERE, "golden", "ingest_vectors.npz"))


@pytest.fixture(scope="module")
def capi():
    import __graft_entry__ as g
    g.build()
    from egomotion_with_local_loop_closures_b200 import capi as m
    return m


def same(key, got):
    if key in G:
        return np.array_equal(G[key], got)
    return str(G[key + "_sha"]) == hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest()


def camera_for(capi, name):
    w, h, c, dw, dh, ud, _ = mk.CASES[name]
    return capi.make_camera(w, h, c, bool(ud), G[f"{name}/K"], G["dist"], G[f"{name}/new_K"] if ud else None)


def tracker(capi, w, h, **over):
    kw = dict(max_keyframes=2, max_frames=4)
    kw.update(over)
    return capi.Tracker(capi.default_config(w, h, **kw))


@pytest.mark.parametrize("name", list(mk.CASES))
def test_level0_equals_fixture_and_oracle(capi, name):
    w, h, c, dw, dh, ud, _ = mk.CASES[name]
    img = mk.camera_image(name)
    t = tracker(capi, dw, dh)
    t.set_camera(camera_for(capi, name))
    t.ingest_frames([1], [img])
    got = t.read_frame_level(1, 0)[0]
    assert same(f"{name}/out", got)
    assert np.array_equal(got, ingest_oracle.ingest(img, dw, dh, bool(ud), G[f"{name}/K"], G["dist"], G[f"{name}/new_K"] if ud else None))
    t.close()


@pytest.mark.parametrize("name", [n for n in mk.CASES if mk.CASES[n][5]])
def test_map_and_taps_equal_fixture(capi, name):
    """The CV_16SC2 map the device built, at the tap positions, is cv2's map there (the oracle's full map is pinned to the fixture
    by digest in the same test); the tap tables are cv::resize's."""
    w, h, c, dw, dh, ud, _ = mk.CASES[name]
    xy, fr = ingest_oracle.undistort_map(G[f"{name}/K"], G["dist"], G[f"{name}/new_K"], w, h)
    assert same(f"{name}/map_xy", xy) and same(f"{name}/map_frac", fr)
    t = tracker(capi, dw, dh)
    t.set_camera(camera_for(capi, name))
    tx, ty, mxy, mfr = t.read_camera_tables()
    x0, x1, _, _ = mk.resize_taps(w, dw)
    y0, y1, _, _ = mk.resize_taps(h, dh)
    assert np.array_equal(tx, np.stack([x0, x1], 1)) and np.array_equal(ty, np.stack([y0, y1], 1))
    rows, cols = ty.reshape(-1), tx.reshape(-1)
    assert np.array_equal(mxy, xy[rows][:, cols]) and np.array_equal(mfr, fr[rows][:, cols])
    t.close()


@pytest.mark.parametrize("undistort", [False, True])
def test_random_sweep_2560x1920_host_and_device(capi, undistort):
    """2560x1920 BGR camera -> 640x480: eight random frames, from host memory and from CUDA tensors, against the oracle."""
    import torch
    w, h, dw, dh = 2560, 1920, 640, 480
    K = mk.camera_matrix(w, h)
    newK = capi.optimal_new_camera_matrix(K, mk.DIST, w, h, 0.0)
    rng = np.random.default_rng(7 + undistort)
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(8)]
    t = tracker(capi, dw, dh, max_frames=16)
    t.set_camera(capi.make_camera(w, h, 3, undistort, K, mk.DIST, newK))
    t.ingest_frames(list(range(8)), imgs)
    t.ingest_frames(list(range(8, 16)), [torch.from_numpy(a).cuda() for a in imgs])
    for i, a in enumerate(imgs):
        host = t.read_frame_level(i, 0)[0]
        dev = t.read_frame_level(8 + i, 0)[0]
        assert np.array_equal(host, dev), i
        assert np.array_equal(host, ingest_oracle.ingest(a, dw, dh, undistort, K, mk.DIST, newK)), i
    t.close()


def camera_scene(w, h, F=4, seed=3):
    """A tracking case at w x h and its frames as F x F-upsampled BGR camera images (the channels differ slightly)."""
    from tests.helpers import make_case
    case = make_case(w, h, n_frames=3, seed=seed)
    rng = np.random.default_rng(seed)

    def cam(gray):
        big = np.kron(gray.astype(np.int16), np.ones((F, F), np.int16))
        bgr = np.stack([big + rng.integers(-3, 4, big.shape) for _ in range(3)], -1)
        return np.clip(bgr, 0, 255).astype(np.uint8)
    return case, cam(case["kf"]["image"]), [cam(f) for f in case["frames"]]


def test_prepared_slots_and_records_equal_the_upload_path(capi):
    """After ingestion the pyramids, gradients, masks, selection counts and track records equal those of ellc_upload_frame /
    ellc_upload_keyframe fed the oracle's level-0 image."""
    from tests.helpers import gpu_config
    case, kf_cam, fr_cam = camera_scene(320, 240)
    W, H = 1280, 960
    K = mk.camera_matrix(W, H)
    newK = capi.optimal_new_camera_matrix(K, mk.DIST, W, H, 1.0)
    kf = case["kf"]
    a = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=3))
    b = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=3))
    a.set_camera(capi.make_camera(W, H, 3, True, K, mk.DIST, newK))
    a.ingest_keyframe(0, kf_cam, kf["depth"], kf["var"])
    a.ingest_frames([0, 1, 2], fr_cam)
    b.upload_keyframe(0, ingest_oracle.ingest(kf_cam, 320, 240, True, K, mk.DIST, newK), kf["depth"], kf["var"])
    for i, f in enumerate(fr_cam):
        b.upload_frame(i, ingest_oracle.ingest(f, 320, 240, True, K, mk.DIST, newK))
    pairs = a.make_pairs([0, 0, 0], [0, 1, 2])
    ra, rb = a.track_batch(pairs), b.track_batch(pairs)
    assert ra.tobytes() == rb.tobytes()
    for level in range(4):
        for s in range(3):
            for x, y in zip(a.read_frame_level(s, level), b.read_frame_level(s, level)):
                assert np.array_equal(x, y), (level, s)
        ka, kb = a.read_keyframe_level(0, level), b.read_keyframe_level(0, level)
        assert np.array_equal(ka[0], kb[0]) and np.array_equal(ka[1], kb[1]) and ka[2] == kb[2], level
    assert int(ra["n_selected"][0][0]) > 0
    a.close(); b.close()


def test_pipelined_ingestion_equals_serial(capi):
    """Ingestion enqueued while a batch tracks -- into other slots, and into the slots that batch reads -- gives the records a
    serial run gives."""
    from tests.helpers import gpu_config
    case, kf_cam, fr_cam = camera_scene(320, 240, seed=5)
    W, H = 1280, 960
    K = mk.camera_matrix(W, H)
    newK = capi.optimal_new_camera_matrix(K, mk.DIST, W, H, 0.0)
    cam = capi.make_camera(W, H, 3, True, K, mk.DIST, newK)
    kf = case["kf"]
    n = 64
    frames_a = [fr_cam[i % 3] for i in range(n)]
    frames_b = [fr_cam[(i + 1) % 3] for i in range(n)]
    pairs_a = capi.Tracker.make_pairs([0] * n, list(range(n)))
    pairs_b = capi.Tracker.make_pairs([0] * n, list(range(n, 2 * n)))

    p = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=2 * n))
    p.set_camera(cam)
    p.ingest_keyframe(0, kf_cam, kf["depth"], kf["var"])
    p.ingest_frames(list(range(n)), frames_a)
    da = p.track_batch_async(pairs_a)
    p.ingest_frames(list(range(n, 2 * n)), frames_b)             # behind nothing: batch a reads other slots
    db = p.track_batch_async(pairs_b)
    p.ingest_frames(list(range(n)), frames_b)                    # slots batch a may still read: ordered behind it
    dc = p.track_batch_async(pairs_a)
    rc_pipe = p.results_download(dc, n)
    rb_pipe = p.results_download(db, n)
    ra_pipe = p.results_download(da, n)

    s = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=2 * n))
    s.set_camera(cam)
    s.ingest_keyframe(0, kf_cam, kf["depth"], kf["var"])
    s.ingest_frames(list(range(n)), frames_a)
    s.synchronize()
    ra = s.track_batch(pairs_a)
    s.ingest_frames(list(range(n, 2 * n)), frames_b)
    s.synchronize()
    rb = s.track_batch(pairs_b)
    assert ra_pipe.tobytes() == ra.tobytes() and rb_pipe.tobytes() == rb.tobytes() and rc_pipe.tobytes() == rb.tobytes()
    p.close(); s.close()


def test_error_codes(capi):
    L = capi.lib()
    t = tracker(capi, 48, 36)
    img = np.zeros((144, 192, 3), np.uint8)
    slots = np.array([0], np.int32)
    ptrs = (C.c_void_p * 1)(img.ctypes.data)
    assert L.ellc_ingest_frames(t._h, 1, slots.ctypes.data, ptrs, 0) == -3                 # no camera set
    assert L.ellc_read_camera_tables(t._h, None, None, None, None) == -3
    bad = [capi.make_camera(192, 144, 2), capi.make_camera(40, 144, 3), capi.make_camera(192, 144, 3, pitch=100),
           capi.make_camera(192, 144, 3, True, np.eye(3), mk.DIST, np.zeros((3, 3)))]
    for cam in bad:
        assert L.ellc_set_camera(t._h, C.byref(cam)) == -1
    assert L.ellc_set_camera(t._h, None) == -1
    t.set_camera(capi.make_camera(192, 144, 3))
    assert L.ellc_ingest_frames(t._h, 1, np.array([4], np.int32).ctypes.data, ptrs, 0) == -1  # slot out of range
    assert L.ellc_ingest_frames(t._h, 2, np.array([1, 1], np.int32).ctypes.data, (C.c_void_p * 2)(img.ctypes.data, img.ctypes.data), 0) == -1
    assert L.ellc_ingest_frames(t._h, 1, slots.ctypes.data, (C.c_void_p * 1)(None), 0) == -1  # null image
    assert L.ellc_ingest_frames(t._h, 1, slots.ctypes.data, ptrs, 2) == -1
    d = [np.zeros((36 >> l, 48 >> l), np.float32) for l in range(4)]
    dp = (C.c_void_p * 4)(*[a.ctypes.data for a in d])
    assert L.ellc_ingest_keyframe(t._h, 2, img.ctypes.data, 0, dp, dp) == -1                 # keyframe slot out of range
    assert L.ellc_ingest_keyframe(t._h, 0, None, 0, dp, dp) == -1
    assert L.ellc_ingest_frames(t._h, 1, slots.ctypes.data, ptrs, 0) == 0
    t.synchronize()
    t.close()
